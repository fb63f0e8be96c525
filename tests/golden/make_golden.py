#!/usr/bin/env python3
"""Generate the committed golden fixtures from the UNMODIFIED reference.

Needs the reference source tree (``THEIA_REFERENCE_ROOT``, see oracle/ref_loader.py):

    python tests/golden/make_golden.py

Writes
  tests/golden/reference_test_vectors.json -- the vectors the reference's own unit
      test holds (plugins/anomaly-detection/anomaly_detection_test.py:199-402).
  tests/golden/sql_cases.json -- the 12 (arguments, SQL text) cases of the reference's SQL-generation test
      (anomaly_detection_test.py:46-195).
  tests/golden/udf_cases.json -- seeded input series and the outputs of the
      reference UDFs ``calculate_ewma``, ``calculate_ewma_anomaly`` and
      ``calculate_dbscan_anomaly`` (anomaly_detection.py:146-212, 325-349) on them,
      called with ``decimal.Decimal`` elements as Spark hands them over
      (``Decimal(38,18)``, anomaly_detection.py:488).  scikit-learn here is 1.9.0
      (the reference pins 1.3.0); numpy 2.3.5.
  tests/golden/udf_cases_oracle_stddev.json -- heavy-tailed seeded series and the outputs of the same
      three reference UDFs when they are handed the oracle's own stddev_samp.

The fixtures travel to the GPU box; the reference tree does not.
"""
import json
import os
import sys
from decimal import Decimal

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle.ref_loader import load_reference_job, load_reference_test_vectors  # noqa: E402

EPS = 250000000


def series_bank():
    rng = np.random.default_rng(20240922)
    bank = []

    def add(tag, vals):
        bank.append((tag, [int(v) for v in vals]))

    lengths = [1, 2, 3, 4, 5, 8, 11, 12, 13, 24, 50, 100, 257]
    for n in lengths:
        base = float(np.exp(rng.uniform(np.log(1e6), np.log(1e10))))
        v = base + rng.normal(0, 1e-3 * base, n)
        spike = rng.random(n) < 0.05
        v = np.where(spike, v * rng.choice([0.1, 2.5, 12.0], n), v)
        add("typical_n%d" % n, np.maximum(np.rint(v), 1))
        add("small_n%d" % n, rng.integers(0, 1000, n))
        # exact-eps ties: a lattice with spacing eps, jittered by a few points
        lat = 4_000_000_000 + EPS * rng.integers(0, 6, n)
        add("ties_n%d" % n, lat)
        lat2 = 50_000_000_000 + EPS * rng.integers(0, 4, n) + rng.integers(0, 2, n)
        add("ties_big_n%d" % n, lat2)
        # two dense clusters and stragglers
        c = np.where(rng.random(n) < 0.5, 1_000_000_000, 9_000_000_000) + rng.integers(-EPS, EPS, n)
        add("clusters_n%d" % n, np.maximum(c, 0))
        # > 2^53: conversion to double rounds
        add("huge_n%d" % n, (1 << 62) + rng.integers(0, 1 << 40, n).astype(object) * 1024 + 1)
        add("const_n%d" % n, np.full(n, 4005277827))
    # near-threshold gaps around eps for the KD-tree regime
    for n in (12, 30):
        gaps = rng.choice([EPS - 1, EPS, EPS + 1, 3], n)
        add("gaps_n%d" % n, 1_000_000 + np.cumsum(gaps))
    return bank


def oracle_stddev_cases(ad):
    """Series with rare 300x spikes; the reference UDFs are handed the oracle's restatement of the job's stddev_samp."""
    from oracle import tad_oracle
    rng = np.random.default_rng(99)
    cases = []
    for n in (1, 2, 7, 11, 12, 40, 90):
        vals = [int(x) for x in np.maximum(np.rint(4e9 + rng.normal(0, 4e6, n) * rng.choice([1, 1, 1, 300], n)), 1)]
        dec = [Decimal(v) for v in vals]
        sd = tad_oracle.stddev_samp(vals)
        cases.append({"values": vals, "stddev": sd, "ewma": [float(e) for e in ad.calculate_ewma(dec)],
                      "ewma_flags": [bool(b) for b in ad.calculate_ewma_anomaly(dec, sd)],
                      "dbscan_flags": [bool(b) for b in ad.calculate_dbscan_anomaly(dec, sd)]})
    return cases


def main():
    ad = load_reference_job()
    with open(os.path.join(HERE, "reference_test_vectors.json"), "w") as f:
        json.dump(load_reference_test_vectors(), f)
    cases = []
    for tag, vals in series_bank():
        dec = [Decimal(v) for v in vals]
        x = np.array(vals, dtype=np.uint64).astype(np.float64)
        sd = float(np.std(x, ddof=1)) if len(vals) > 1 else None
        ewma = [float(e) for e in ad.calculate_ewma(dec)]
        ewma_flags = [bool(b) for b in ad.calculate_ewma_anomaly(dec, sd)]
        dbscan_flags = [bool(b) for b in ad.calculate_dbscan_anomaly(dec, sd)]
        cases.append({"tag": tag, "values": vals, "stddev_numpy": sd, "ewma": ewma,
                      "ewma_flags": ewma_flags, "dbscan_flags": dbscan_flags})
    with open(os.path.join(HERE, "udf_cases.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py",
                   "reference_commit": "bc06ff0afe05c984f2efc7a53e68e8f152914c3e",
                   "cases": cases}, f)
    print("wrote %d udf cases" % len(cases))
    cases = oracle_stddev_cases(ad)
    with open(os.path.join(HERE, "udf_cases_oracle_stddev.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py",
                   "reference_commit": "bc06ff0afe05c984f2efc7a53e68e8f152914c3e",
                   "cases": cases}, f)
    print("wrote %d oracle-stddev udf cases" % len(cases))
    # the reference's 12 SQL-generation cases (anomaly_detection_test.py:46-195): inputs + expected SQL text
    import importlib
    tmod = importlib.import_module("anomaly_detection_test")
    sql_cases = [{"args": list(inp), "sql": sql} for inp, sql in tmod.test_generate_sql_query.pytestmark[0].args[1]]
    with open(os.path.join(HERE, "sql_cases.json"), "w") as f:
        json.dump(sql_cases, f, indent=1)
    print("wrote %d sql cases" % len(sql_cases))


if __name__ == "__main__":
    main()

"""Pin the oracle: (i) the reference's own golden vectors
(plugins/anomaly-detection/anomaly_detection_test.py:199-402, committed as
tests/golden/reference_test_vectors.json), (ii) outputs of the unmodified reference UDFs on
seeded series (tests/golden/udf_cases.json, made by tests/golden/make_golden.py), and
(iii) outputs of the same UDFs on heavy-tailed series when handed the oracle's own stddev
(tests/golden/udf_cases_oracle_stddev.json, same generator)."""
import json
import os

import numpy as np
import pytest

from oracle import c_oracle, tad_oracle as o

G = os.path.join(os.path.dirname(__file__), "golden")
REF = json.load(open(os.path.join(G, "reference_test_vectors.json")))
CASES = json.load(open(os.path.join(G, "udf_cases.json")))["cases"]
SD_CASES = json.load(open(os.path.join(G, "udf_cases_oracle_stddev.json")))["cases"]


def test_reference_ewma_values_exact():
    # anomaly_detection_test.py:252-258 asserts == on the full list
    assert list(o.calculate_ewma(REF["throughput_list"])) == REF["expected_ewma_row_list"]
    calc, _, _ = c_oracle.ewma_series(REF["throughput_list"])
    assert list(calc) == REF["expected_ewma_row_list"]


def test_reference_ewma_flags():
    # :366-373, with the test's stddev constant
    flags = o.calculate_ewma_anomaly(REF["throughput_list"], REF["stddev"])
    assert list(flags) == REF["expected_anomaly_list_ewma"]
    assert list(np.flatnonzero(flags)) == [68, 69, 70]


def test_reference_dbscan_flags():
    # :394-402
    assert list(o.calculate_dbscan_anomaly(REF["throughput_list"])) == REF["expected_dbscan_anomaly_list"]
    assert list(c_oracle.dbscan_series(REF["throughput_list"])) == REF["expected_dbscan_anomaly_list"]


def test_reference_stddev_constant():
    # :286 stddev = 4.9198515356827E9 (14 significant digits of stddev_samp of the golden series)
    sd = o.stddev_samp(REF["throughput_list"])
    assert abs(sd - REF["stddev"]) / REF["stddev"] < 1e-13
    x = np.array(REF["throughput_list"], dtype=np.float64)
    assert abs(sd - np.std(x, ddof=1)) / sd < 1e-14
    # flags are unchanged when the oracle's own stddev replaces the constant
    assert list(o.calculate_ewma_anomaly(REF["throughput_list"], sd)) == REF["expected_anomaly_list_ewma"]


@pytest.mark.parametrize("case", CASES, ids=[c["tag"] for c in CASES])
def test_udf_cases(case):
    v = case["values"]
    assert list(o.calculate_ewma(v)) == case["ewma"]
    assert list(o.calculate_ewma_anomaly(v, case["stddev_numpy"])) == case["ewma_flags"]
    assert list(o.calculate_dbscan_anomaly(v)) == case["dbscan_flags"]
    sd = o.stddev_samp(v)
    if case["stddev_numpy"] is None:
        assert sd is None
    elif case["stddev_numpy"] > 0:
        assert abs(sd - case["stddev_numpy"]) / case["stddev_numpy"] < 1e-11


@pytest.mark.parametrize("case", CASES, ids=[c["tag"] for c in CASES])
def test_c_port_matches_python(case):
    v = case["values"]
    calc, flags, sd = c_oracle.ewma_series(v)
    assert list(calc) == case["ewma"]
    psd = o.stddev_samp(v)
    assert (psd is None and np.isnan(sd)) or psd == sd
    assert list(flags) == list(o.calculate_ewma_anomaly(v, psd))
    assert list(c_oracle.dbscan_series(v)) == case["dbscan_flags"]


def test_recorded_reference_udfs():
    for case in SD_CASES:
        vals = case["values"]
        sd = o.stddev_samp(vals)
        assert sd == case["stddev"]
        assert list(o.calculate_ewma(vals)) == case["ewma"]
        assert list(o.calculate_ewma_anomaly(vals, sd)) == case["ewma_flags"]
        assert list(o.calculate_dbscan_anomaly(vals)) == case["dbscan_flags"]

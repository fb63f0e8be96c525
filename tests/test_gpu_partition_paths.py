"""Parity of the single-GPU partition paths that the default engine does not take on small tables: the exact
(histogram + scan + scatter) partition, the optimistic partition falling back to it when its overflow list fills,
and host input that is copied in more than one chunk."""
import os

import pytest

from theia_b200 import synth
from tests.util import assert_same_rows, oracle_rows

pytestmark = pytest.mark.gpu

CHUNK_ROWS = 8 << 20          # host input is copied to the device in chunks of about this many rows


def _engine(**env):
    from theia_b200.engine import TadEngine
    os.environ.update(env)
    try:
        return TadEngine(device=0)
    finally:
        for k in env:
            del os.environ[k]


@pytest.fixture(scope="module")
def exact_engine():
    """Engine that always takes the exact partition (TAD_OPTIMISTIC=0)."""
    eng = _engine(TAD_OPTIMISTIC="0")
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def one_bucket_engine():
    """Engine forced to one hash bucket: one 4096-row slot, so the optimistic overflow list (2^20 rows for tables
    below 32M rows) fills on any table of more than ~1.05M rows."""
    eng = _engine(TAD_DEBUG_LOGB="0")
    yield eng
    eng.close()


def run_both(engine, table, algo, **kw):
    got, st = engine.run(table, algo=algo, tad_id="paths", **kw)
    want, ns, npts = oracle_rows(table, algo=algo, **kw)
    assert st["state"] == "COMPLETED", st
    assert st["series"] == ns and st["points"] == npts, (st, ns, npts)
    assert_same_rows(got, want, what="%s %s" % (algo, kw))
    return st


def ran_exact(st):
    """With host input only the exact partition records a scatter phase; the optimistic one scatters inside h2d."""
    return st["phase_ms"]["scatter"] > 0


@pytest.mark.parametrize("algo", ["EWMA", "DBSCAN"])
def test_exact_partition_ragged_duplicates(exact_engine, algo):
    t = synth.make_flows(3000, 30, seed=41, dup_frac=0.2, ragged=True)
    for emit_all in (False, True):
        st = run_both(exact_engine, t, algo, emit_all=emit_all)
        assert ran_exact(st)


@pytest.mark.parametrize("algo", ["EWMA", "DBSCAN"])
def test_exact_partition_spill(exact_engine, algo):
    t = synth.make_flows(40, 5000, seed=42, dup_frac=0.05, ragged=True)      # some connections > 4096 rows
    st = run_both(exact_engine, t, algo, emit_all=True)
    assert ran_exact(st)
    assert 0 < st["spill_rows"] < st["rows_kept"]


@pytest.mark.parametrize("algo", ["EWMA", "DBSCAN"])
def test_overflow_falls_back_to_exact(one_bucket_engine, algo):
    t = synth.make_flows(12000, 100, seed=43)
    assert len(t["value"]) > 4096 + (1 << 20)
    st = run_both(one_bucket_engine, t, algo)
    assert ran_exact(st)
    assert st["spill_rows"] == st["rows_kept"] == len(t["value"])


@pytest.fixture(scope="module")
def two_chunk_table():
    t = synth.make_flows(85000, 100, seed=44)
    assert len(t["value"]) > CHUNK_ROWS
    want, ns, npts = oracle_rows(t, algo="EWMA")
    return t, want, ns, npts


@pytest.mark.parametrize("which", ["default", "exact"])
def test_host_input_in_two_chunks(engine, exact_engine, two_chunk_table, which):
    t, want, ns, npts = two_chunk_table
    eng = engine if which == "default" else exact_engine
    got, st = eng.run(t, algo="EWMA", tad_id="chunks")
    assert st["state"] == "COMPLETED", st
    assert st["rows_kept"] == len(t["value"])
    assert st["series"] == ns and st["points"] == npts, (st, ns, npts)
    assert ran_exact(st) == (which == "exact")
    assert_same_rows(got, want, what="two chunks, %s engine" % which)

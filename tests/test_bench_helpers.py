"""bench.py's parity helpers on CPU: per-segment one-stage oracle answers combine into the whole table's answer, and the
comparison flags what it should."""
import copy
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from greengage_b200 import capi, tpch  # noqa: E402
from oracle import pyoracle as po  # noqa: E402


def _oracle(pages, threads=2):
    scan, part, pool = tpch.q1_plan(capi.TAB_LINEITEM_WIDE, capi.AGGSTAGE_PARTIAL)
    rows, secs, scanned = po.seqscan_agg_mt(scan, part, tpch.q1_final_agg(part), pool, pages, threads)
    return bench.q1_rows_from_oracle(rows), scanned


def test_segment_answers_combine_to_the_whole_tables_answer():
    whole, _, nr = tpch.synth_generate(tpch.synth_spec(capi.TAB_LINEITEM_WIDE, 60_000), nthreads=2)
    want, scanned = _oracle(whole)
    assert scanned == nr
    parts = []
    for seg in range(3):
        pages, _, _ = tpch.synth_generate(tpch.synth_spec(capi.TAB_LINEITEM_WIDE, 60_000, nsegs=3, seg=seg), nthreads=2)
        parts.append(_oracle(pages)[0])
    got = bench.q1_combine(parts)
    par = bench.q1_compare(got, want)
    assert par["ok"] and par["counts_equal"] and par["rows"] == 4 and par["max_rel_err"] < 1e-9


def test_compare_flags_a_wrong_count_and_a_wrong_sum():
    pages, _, _ = tpch.synth_generate(tpch.synth_spec(capi.TAB_LINEITEM_WIDE, 20_000), nthreads=2)
    want, _ = _oracle(pages)
    bad = copy.deepcopy(want)
    k = next(iter(bad))
    bad[k] = (bad[k][0], bad[k][1] + 1)
    assert not bench.q1_compare(bad, want)["ok"]
    bad = copy.deepcopy(want)
    bad[k][0][2] *= 1.00001
    assert not bench.q1_compare(bad, want)["ok"]
    bad = copy.deepcopy(want)
    del bad[k]
    assert not bench.q1_compare(bad, want)["ok"]


def test_slot_rows_decode_like_oracle_rows():
    import numpy as np
    f = lambda d: int(np.float64(d).view(np.int64))
    rows = [([65, 70, f(1.5), f(2.5), f(3.5), f(4.5), f(5.5), f(6.5), f(7.5), 42], [0] * 10, [0] * 10, [0] * 10)]
    got = bench.q1_rows_from_slots(rows)
    assert got == {(65, 70): ([1.5, 2.5, 3.5, 4.5, 5.5, 6.5, 7.5], 42)}


def test_cpulist_and_numa_lookup_degrade_quietly():
    assert bench._cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert bench._cpulist("") == set()
    # no GPU here: the lookup says so instead of raising, and bench.py then leaves the affinity alone
    assert bench.gpu_numa_cpus(0) is None or isinstance(bench.gpu_numa_cpus(0), tuple)


def test_a_failing_rjoin_child_costs_the_entry_not_the_run(monkeypatch):
    """rjoin_in_children: a child that exits with an error (here: no CUDA device) yields an error entry carrying the tail of its
    log; nothing raises, nothing hangs."""
    import time
    import types
    monkeypatch.setenv("MASTER_PORT", "29611")
    monkeypatch.setenv("GGB200_RJOIN_TIMEOUT", "120")
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")          # the child sees no device on a GPU machine either
    t0 = time.time()
    r = bench.rjoin_in_children(types.SimpleNamespace(rjoin_rows=2e6), 0, 1)
    assert "error" in r and "child exited" in r["error"] and time.time() - t0 < 110


def test_random_access_bound_needs_the_measured_rates(monkeypatch):
    monkeypatch.setattr(bench, "_random_rates", {"gather_g_per_s": 40.0, "cas_insert_g_per_s": 9.0, "atomic_pair_g_per_s": 18.0})
    b = bench.join_random_bound(3.7e9, 25e6, 16.9e9, 1e8, 2.77, 7.96, 6486.1)
    assert abs(b["build_bound_ms"] - (3.7e9 / 6486.1e9 * 1e3 + 25e6 / 9e9 * 1e3)) < 1e-9
    assert 0.9 < b["build_frac_of_bound"] < 1.3 and 0.5 < b["probe_frac_of_bound"] < 0.8
    monkeypatch.setattr(bench, "_random_rates", {"error": "no tool"})
    assert bench.join_random_bound(1, 1, 1, 1, 1.0, 1.0, 6486.1) is None

"""A CPU segment on the other side of a Motion: the rows of this engine's PARTIAL-stage Agg leave as the reference's tuple
chunks (GgExecSendTupleChunks) and the reference's own CvtChunksToTup reads them; rows the reference's SerializeTuple wrote —
as MemTuples and in the heap-tuple form — arrive at a Motion node (GgExecRecvTupleChunks) and the FINAL stage above it gives the
one-stage answer.  Host C of the product (gg_executor.c + gg_tupser.c) over the oracle-backed stand-in device library; the
reference side (memtuple.o, tupser.o, tupchunklist.o) ran when tests/golden/wire_kat.json was made (make_golden.py wire_kat):
the streams it read and what it read from them, and the streams it wrote."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from greengage_b200 import capi, executor as ex, tpch  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from _util import golden  # noqa: E402
from test_executor_multiseg import MockRel, build_mock  # noqa: E402

NSEG = 3
ROWS = 30_000
PARTIAL_CHUNK_SIZES = (8124, 64)            # segment 0's PARTIAL rows as this engine's tuple chunks
SENDER_CHUNK_SIZES = (48, 8124, 8124)       # every segment's rows as the reference's SerializeTuple writes them


def bind_mock(L):
    """the executor surface and the tuple-chunk entry points of the mock-linked host code"""
    L = ex.bind(L)
    L.mock_engine.restype = C.c_void_p
    L.mock_relation.restype = C.c_void_p
    L.mock_relation.argtypes = [C.c_void_p, C.c_uint64]
    L.GgExecSendTupleChunks.restype = C.c_int64
    L.GgExecSendTupleChunks.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_int64)]
    L.GgExecRecvTupleChunks.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    return L


@pytest.fixture(scope="module")
def mock(tmp_path_factory):
    L = bind_mock(C.CDLL(build_mock(str(tmp_path_factory.mktemp("mockwire")))))
    old = ex._lib
    ex._lib = L
    yield L
    ex._lib = old


def shard(seg):
    pages, _, _ = tpch.synth_generate(tpch.synth_spec(capi.TAB_LINEITEM_WIDE, ROWS, nsegs=NSEG, seg=seg), nthreads=1)
    return pages


def partial_chunks(L, eng, seg, max_chunk):
    """PARTIAL Agg <- SeqScan on one segment, its rows as tuple chunks"""
    scan, part, pool = tpch.q1_plan(capi.TAB_LINEITEM_WIDE, capi.AGGSTAGE_PARTIAL)
    b = ex.PlanBuilder()
    rel = MockRel(L, shard(seg))                       # keeps the pages alive while the plan runs
    x = ex.Executor(eng, pool, [rel], b.agg(b.seqscan(0, scan.desc, scan.qual), part))
    out = (C.c_uint8 * 65536)()
    n = C.c_int64(0)
    got = L.GgExecSendTupleChunks(x.state, max_chunk, out, len(out), C.byref(n))
    assert got > 0, L.GgExecLastError()
    rows = x.rows()                          # the same rows as slots: keys, sums, {N, sumX, sumX2} x 3, count
    x.end()
    return bytes(out[:got]), n.value, rows


def b2f(v):
    return np.int64(v).view(np.float64).item()


def test_partial_rows_leave_as_the_references_chunks_and_its_reader_reads_them(mock):
    """the stream is byte for byte the one the reference's CvtChunksToTup read, and what it read is these rows"""
    kat = golden("wire_kat.json")["partial"]
    eng = mock.mock_engine()
    for max_chunk in PARTIAL_CHUNK_SIZES:
        stream, n, rows = partial_chunks(mock, eng, 0, max_chunk)
        assert n == len(rows) == 4 and stream[-4:] == b"\x00\x00\x04\x00"          # ends with TC_END_OF_STREAM
        assert stream.hex() == kat[str(max_chunk)]["stream"], max_chunk
        for (v, nl, ty, ln), got in zip(rows, kat[str(max_chunk)]["read"], strict=True):
            assert got["form"] == 1 and got["nulls"] == [0] * 10                         # a MemTuple
            assert got["keys"] == [capi.unpack_str(v[0], ln[0]), capi.unpack_str(v[1], ln[1])]
            assert got["sums"] == v[2:6]                                                   # float8 sums: the same bits
            for k in range(3):
                assert got["arrays"][k] == [1, 0, 701, 3, 1] + v[6 + 3 * k:9 + 3 * k] and got["array_lens"][k] == 44
            assert got["count"] == v[15]


@pytest.mark.parametrize("form", ["ours", "ref-memtuple", "ref-heap"])
def test_rows_from_cpu_senders_arrive_at_the_motion_and_the_final_stage_combines_them(mock, form):
    eng = mock.mock_engine()
    if form == "ours":
        streams = [partial_chunks(mock, eng, seg, 8124 if seg else 80)[0][:-4] for seg in range(NSEG)]
    else:
        streams = [bytes.fromhex(h) for h in golden("wire_kat.json")["senders"][form]]
        assert len(streams) == NSEG
    wire = b"".join(streams) + b"\x00\x00\x04\x00"
    # the receiving slice: Agg(FINAL) <- Gather Motion <- [Agg(PARTIAL) <- SeqScan on the senders]
    scan, part, pool = tpch.q1_plan(capi.TAB_LINEITEM_WIDE, capi.AGGSTAGE_PARTIAL)
    fin = tpch.q1_final_agg(part)
    b = ex.PlanBuilder()
    plan = b.agg(b.motion(b.agg(b.seqscan(0, scan.desc, scan.qual), part), ex.MOTION_GATHER, [], 1), fin)
    rel0 = MockRel(mock, shard(0))
    x = ex.Executor(eng, pool, [rel0], plan)
    motion = mock.GgExecOuterPlanState(x.state)
    assert mock.GgExecNodeKind(motion) == b"motion"
    assert mock.GgExecRecvTupleChunks(motion, wire, len(wire)) == 0, mock.GgExecLastError()
    got = {(v[0], v[1]): v for v, nl, ty, ln in x.rows()}
    x.end()
    whole, _, _ = tpch.synth_generate(tpch.synth_spec(capi.TAB_LINEITEM_WIDE, ROWS), nthreads=1)
    s1, a1, p1 = tpch.q1_plan(capi.TAB_LINEITEM_WIDE)
    want, _, _ = po.seqscan_agg(s1, a1, p1, whole)
    assert len(got) == len(want) == 4
    for w in want:
        v = got[(w.key[0], w.key[1])]
        assert v[9] == w.agg[7].i
        for col in range(7):
            assert abs(b2f(v[2 + col]) - w.agg[col].f[0]) <= 1e-9 * abs(w.agg[col].f[0])


def test_a_truncated_stream_is_refused(mock):
    eng = mock.mock_engine()
    stream, n, rows = partial_chunks(mock, eng, 0, 8124)
    scan, part, pool = tpch.q1_plan(capi.TAB_LINEITEM_WIDE, capi.AGGSTAGE_PARTIAL)
    b = ex.PlanBuilder()
    plan = b.agg(b.motion(b.agg(b.seqscan(0, scan.desc, scan.qual), part), ex.MOTION_GATHER, [], 1), tpch.q1_final_agg(part))
    rel0 = MockRel(mock, shard(0))
    x = ex.Executor(eng, pool, [rel0], plan)
    motion = mock.GgExecOuterPlanState(x.state)
    assert mock.GgExecRecvTupleChunks(motion, stream[:-4], len(stream) - 4) != 0        # no end-of-stream chunk
    assert mock.GgExecRecvTupleChunks(motion, stream[:50], 50) != 0
    x.end()


def test_es_snapshot_is_handed_to_the_scans(mock):
    """EState.es_snapshot -> gg_engine_set_snapshot before the slice runs (the stand-in device library scans with the oracle's
    HeapTupleSatisfiesMVCC); without it the same pages are refused with the visibility code"""
    from _util import mvcc_snapshot, stamp_visibility
    pages, _, nr = tpch.synth_generate(tpch.synth_spec(capi.TAB_LINEITEM_NARROW, 20_000, seed=2), nthreads=1)
    pg, vis = stamp_visibility(pages, all_visible_every=3)
    scan, agg, pool = tpch.q1_plan(capi.TAB_LINEITEM_NARROW)
    snap = mvcc_snapshot()
    po.set_snapshot(snap)
    try:
        want, wsc, _ = po.seqscan_agg(scan, agg, pool, pg)
    finally:
        po.set_snapshot(None)
    assert wsc == sum(vis)
    eng = type("E", (), {"h": C.c_void_p(mock.mock_engine())})
    b = ex.PlanBuilder()
    rel = MockRel(mock, pg)
    x = ex.Executor(eng, pool, [rel], b.agg(b.seqscan(0, scan.desc, scan.qual), agg), snapshot=snap)
    rows = x.rows()
    x.end()
    assert sorted(v[-1] for v, nl, ty, ln in rows) == sorted(r.agg[7].i for r in want)
    x = ex.Executor(eng, pool, [rel], b.agg(b.seqscan(0, scan.desc, scan.qual), agg))
    with pytest.raises(ex.ExecError) as e:
        x.rows()
    x.end()
    assert e.value.code == -7

"""Generate the golden vectors under tests/golden/ from the REFERENCE ITSELF.  Run in the build container
(needs /root/reference and oracle/_ref/libggref.so, built by `make -C oracle/ref_build`).

  hash_kat.json     hash_any / hash_uint32 / hashint4 / hashint8 / hashfloat8 / hashbpchar / bpchareq and
                    cdbhash+jump-consistent-hash routing, computed by the reference's own hashfunc.o,
                    varchar.o and cdbhash.o
  heap_kat.json     tuples formed by the reference's heap_form_tuple (heaptuple.o) for rows with NULLs,
                    short and long varlenas, and what its heap_deform_tuple reads back
  float_kat.json    float8pl/mi/mul/div incl. overflow/underflow/div-by-zero ERRORs, float8 comparisons,
                    float8_accum / float8_combine / float8_avg, int8inc / int8pl overflow, date vs timestamp
  lineitem_q1.npz   the reference's own regression data (src/test/regress/data/lineitem_small.csv + lineitem.csv,
                    loaded into heap_lineitem by input/rpt_tpch.source:98-99), columns as arrays
  q1_expected.json  the reference's golden Q1 answer over that data (output/rpt_tpch.source:309-315)
  orders_tpch.npz   heap_orders of the same suite (order_small.csv + order.csv)
  tpch_join_expected.json  the reference's golden Q4 (semi join) and Q12 (inner join) answers over heap_orders/heap_lineitem
  onek.npz + onek_agg_expected.json  the suite's onek table (int4 columns) and the golden plain / hashed aggregates of aggregates.out
  aocs_kat.npz      append-only column-oriented (AOCS) column files written by the reference's datumstreamblock.o +
                    cdbappendonlystorageformat.o, what its reader returns for them, and CRC-32C known answers
  sort_golden.json  ORDER BY answers of expected/sort.out for the column types the Sort path takes, ASC/DESC, NULLS FIRST/LAST
  memtuple_kat.json MemTuples formed by the reference's memtuple.o (create_memtuple_binding / memtuple_form_to) for rows with
                    NULLs, short and long varlenas, > 32 attributes and tuples beyond the 2-byte-offset limit, the bindings
                    themselves, what memtuple_deform reads back, and the same rows as tuple chunks out of the reference's
                    tupser.o / tupchunklist.o (SerializeTuple, both the MemTuple and the heap-tuple form, several chunk sizes)
  numeric_kat.json  the reference's numeric.o: text -> on-disk digits (numeric_in), numeric_add / _sub / _mul results with their
                    display scales, numeric_cmp, and sum / avg (a fold of numeric_add; numeric_div(sum, N) as numeric_avg does)
  mvcc_kat.json     the reference's tqual.o + transam.o: HeapTupleSatisfiesMVCC of tuple headers against snapshots and
                    transaction status tables (oracle/ref_build/refwrap_tqual.c)
  join_j1j2.json    J1_TBL / J2_TBL of sql/join.sql and the golden inner / left / right / full equi-join tables of expected/join.out
  hash_random_kat.json  digests of the reference's hashes and routing of test_oracle_hash.py's 20000 random inputs
  aocs_random_kat.json  digests of the column files the reference writes for test_oracle_aocs.py's random columns, and of
                    what its reader returns for them
  wire_kat.json     tuple chunks exchanged with the reference's tupser.o / tupchunklist.o in test_executor_wire.py
"""
import ctypes as C
import json
import os
import random
import re
import struct
import sys
from datetime import date

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))             # the tests whose random inputs some fixtures answer for
from greengage_b200 import capi  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

REF = "/root/reference"
R = po.ref_lib()
assert R is not None, "build oracle/_ref first: make -C oracle/ref_build"
rng = random.Random(20260922)


def f2b(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


def hash_kat():
    out = {"hash_any": [], "hash_uint32": [], "hashint4": [], "hashint8": [], "hashfloat8": [], "hashbpchar": [],
           "bpchareq": [], "route": []}
    fixed = [b"", b"A", b"N", b"R", b"F", b"O", b"hello world!", b"0123456789ab", b"0123456789abc", b"x" * 23, b"y" * 24, b"z" * 25]
    for b in fixed + [bytes(rng.getrandbits(8) for _ in range(rng.randint(0, 64))) for _ in range(300)]:
        out["hash_any"].append([b.hex(), R.ref_hash_any(b, len(b))])
    for v in [0, 1, 42, 0xFFFFFFFF, 0x80000000] + [rng.getrandbits(32) for _ in range(200)]:
        out["hash_uint32"].append([v, R.ref_hash_uint32(v)])
    for v in [0, 1, -1, 2 ** 31 - 1, -2 ** 31] + [rng.getrandbits(32) - 2 ** 31 for _ in range(200)]:
        out["hashint4"].append([v, R.ref_hashint4(v)])
    for v in [0, 1, -1, 2 ** 63 - 1, -2 ** 63, 2 ** 32, -2 ** 32, 2 ** 31, -2 ** 31 - 1] + [rng.getrandbits(64) - 2 ** 63 for _ in range(300)]:
        out["hashint8"].append([str(v), R.ref_hashint8(v)])
    for x in [0.0, -0.0, 1.0, -1.0, 0.1, 1e300, -1e-300, float("inf"), float("-inf"), float("nan")] + [rng.uniform(-1e6, 1e6) for _ in range(200)]:
        out["hashfloat8"].append([str(f2b(x)), R.ref_hashfloat8(x)])
    strs = [b"A", b"A ", b"A   ", b" A", b"", b"   ", b"DELIVER IN PERSON        ", b"DELIVER IN PERSON", b"abc  def  "]
    strs += [bytes(rng.choice(b"ab ") for _ in range(rng.randint(0, 12))) for _ in range(200)]
    for s in strs:
        out["hashbpchar"].append([s.hex(), R.ref_hashbpchar(s, len(s))])
    for _ in range(300):
        a, b = rng.choice(strs), rng.choice(strs)
        out["bpchareq"].append([a.hex(), b.hex(), R.ref_bpchareq(a, len(a), b, len(b))])
    # routing: cdbhashinit/cdbhash/cdbhashreduce with real hash functions
    typs = [20, 23, 701, 1042]
    for _ in range(1500):
        nkeys = rng.randint(1, 3)
        nsegs = rng.choice([1, 2, 3, 4, 5, 7, 8, 16, 31, 64, 100, 1000])
        t, v, ln, nu = [], [], [], []
        for k in range(nkeys):
            ty = rng.choice(typs)
            isn = rng.random() < 0.1
            if ty == 20:
                val, l = rng.getrandbits(64) - 2 ** 63, 0
            elif ty == 23:
                val, l = rng.getrandbits(32) - 2 ** 31, 0
            elif ty == 701:
                val, l = f2b(rng.choice([0.0, -0.0, 1.5, rng.uniform(-1e9, 1e9)])), 0
            else:
                s = bytes(rng.choice(b"ANRFO") for _ in range(rng.randint(0, 8)))
                val, l = int.from_bytes(s.ljust(8, b"\0"), "little", signed=True), len(s)
            t.append(ty); v.append(val); ln.append(l); nu.append(1 if isn else 0)
        seg = R.ref_cdbhash_route((C.c_int32 * nkeys)(*t), (C.c_int64 * nkeys)(*v), (C.c_int32 * nkeys)(*ln),
                                  (C.c_int32 * nkeys)(*nu), nkeys, nsegs)
        out["route"].append({"typ": t, "val": [str(x) for x in v], "len": ln, "null": nu, "nsegs": nsegs, "seg": seg})
    json.dump(out, open(os.path.join(HERE, "hash_kat.json"), "w"))
    print("hash_kat.json", {k: len(v) for k, v in out.items()})


def heap_kat():
    """tuples formed by the reference's heap_form_tuple"""
    out = []
    descs = [("li_wide", capi.synth_tupdesc(capi.TAB_LINEITEM_WIDE)), ("orders", capi.synth_tupdesc(capi.TAB_ORDERS))]
    # a descriptor with nullable columns, a long varlena and odd alignments
    d = capi.gg_tupdesc()
    spec = [(23, 4, 'i', 1), (1042, -1, 'i', 0), (20, 8, 'd', 1), (1043, -1, 'i', 0), (701, 8, 'd', 1), (1082, 4, 'i', 1), (1043, -1, 'i', 0), (23, 4, 'i', 1), (20, 8, 'd', 1)]
    d.natts = len(spec)
    for i, (t, l, al, bv) in enumerate(spec):
        a = d.attrs[i]
        a.atttypid, a.attlen, a.attalign, a.attbyval, a.attnotnull, a.atttypmod = t, l, ord(al), bv, 0, -1
    descs.append(("mixed", d))
    for name, desc in descs:
        n = desc.natts
        for case in range(60):
            vals, lens, nulls, pyvals = (C.c_int64 * n)(), (C.c_int32 * n)(), (C.c_uint8 * n)(), []
            keep = []
            for i in range(n):
                a = desc.attrs[i]
                isnull = name == "mixed" and rng.random() < 0.25
                nulls[i] = 1 if isnull else 0
                if isnull:
                    pyvals.append(None)
                    continue
                if a.attlen == -1:
                    ln = rng.choice([0, 1, 2, 5, 25, 43, 126, 127, 200]) if name == "mixed" else rng.randint(1, 44)
                    s = bytes(rng.choice(b"abcdefg hij") for _ in range(ln))
                    buf = C.create_string_buffer(s, max(len(s), 1))
                    keep.append(buf)
                    vals[i] = C.addressof(buf)
                    lens[i] = len(s)
                    pyvals.append(s.hex())
                elif a.atttypid == 701:
                    x = rng.choice([0.0, 1.0, -2.5, rng.uniform(-1e5, 1e5)])
                    vals[i] = f2b(x)
                    pyvals.append(str(f2b(x)))
                elif a.attlen == 4:
                    x = rng.getrandbits(32) - 2 ** 31
                    vals[i] = x
                    pyvals.append(str(x))
                else:
                    x = rng.getrandbits(64) - 2 ** 63
                    vals[i] = x
                    pyvals.append(str(x))
            outbuf = (C.c_uint8 * 2048)()
            ln = R.ref_heap_form_tuple(n, desc.attrs, vals, lens, nulls, outbuf, 2048)
            tup = bytes(outbuf[:ln])
            dv, dn = (C.c_int64 * n)(), (C.c_uint8 * n)()
            tb = (C.c_uint8 * ln).from_buffer_copy(tup)
            R.ref_heap_deform_tuple(n, desc.attrs, tb, ln, dv, dn)
            out.append({"desc": name, "values": pyvals, "tuple": tup.hex(),
                        "deform": [str(dv[i]) for i in range(n)], "deform_null": [int(dn[i]) for i in range(n)]})
    meta = {}
    for name, desc in descs:
        meta[name] = [[desc.attrs[i].atttypid, desc.attrs[i].attlen, chr(desc.attrs[i].attalign), desc.attrs[i].attbyval] for i in range(desc.natts)]
    json.dump({"descs": meta, "cases": out}, open(os.path.join(HERE, "heap_kat.json"), "w"))
    print("heap_kat.json", len(out))


def memtuple_kat():
    """MemTuple + tuple-chunk goldens out of the reference's memtuple.o / tupser.o (oracle/ref_build/refwrap_motion.c)"""
    rng = random.Random(20260923)          # its own stream: the other fixtures do not change when this one is regenerated
    TY = {"int8": (20, 8, 'd', 1), "int4": (23, 4, 'i', 1), "int2": (21, 2, 's', 1), "bool": (16, 1, 'c', 1), "float8": (701, 8, 'd', 1),
          "date": (1082, 4, 'i', 1), "bpchar": (1042, -1, 'i', 0), "varchar": (1043, -1, 'i', 0), "text": (25, -1, 'i', 0), "f8arr": (1022, -1, 'd', 0)}
    descs = {
        "q1_partial": ["bpchar", "bpchar", "float8", "float8", "float8", "float8", "f8arr", "f8arr", "f8arr", "int8"],    # what a PARTIAL Q1 ships
        "ints4": ["int4", "int4", "date", "bpchar"],                                                                       # 4-byte column alignment
        "mixed": ["int4", "bpchar", "int8", "varchar", "float8", "date", "text", "int2", "bool", "int8", "int2", "bool"],
        "wide40": ["int4", "int8", "bool", "varchar", "int2"] * 8,                                                         # NULL bitmap beyond the free 4 bytes
        "strings": ["text", "int2", "text", "bool", "varchar"],
    }
    meta, cases = {}, []
    for name, cols in descs.items():
        n = len(cols)
        attrs = (capi.gg_attr * n)()
        for i, c in enumerate(cols):
            t, l, al, bv = TY[c]
            attrs[i].atttypid, attrs[i].attlen, attrs[i].attalign, attrs[i].attbyval, attrs[i].attnotnull, attrs[i].atttypmod = t, l, ord(al), bv, 0, -1
        meta[name] = {"cols": [list(TY[c]) for c in cols], "bind": {}}
        for large in (0, 1):
            o6, info = (C.c_int32 * (6 * n))(), (C.c_int32 * 2)()
            vs = R.ref_memtuple_binding(n, attrs, large, o6, info)
            meta[name]["bind"]["large" if large else "small"] = {"var_start": vs, "att": [list(o6[6 * i:6 * i + 6]) for i in range(n)]}
            meta[name]["column_align"], meta[name]["null_bitmap_extra"] = info[0], info[1]
        for case in range(40):
            pnull = rng.choice([0.0, 0.0, 0.15, 0.5, 0.9])
            big = name == "strings" and case % 8 == 0
            vals, lens, nulls, pyvals, keep = (C.c_int64 * n)(), (C.c_int32 * n)(), (C.c_uint8 * n)(), [], []
            for i, c in enumerate(cols):
                t, l, al, bv = TY[c]
                if rng.random() < pnull:
                    nulls[i] = 1
                    pyvals.append(None)
                    continue
                if l == -1:
                    if c == "f8arr":
                        pay = struct.pack("<iiIii3d", 1, 0, 701, 3, 1, float(rng.randint(0, 10 ** 6)), rng.uniform(-1e9, 1e9), rng.uniform(0, 1e12))
                    else:
                        ln = rng.choice([0, 1, 2, 7, 8, 9, 25, 125, 126, 127, 128, 300]) if not big else rng.choice([40000, 70000])
                        pay = bytes(rng.choice(b"abcdefg hij") for _ in range(ln))
                    buf = C.create_string_buffer(pay, max(len(pay), 1))
                    keep.append(buf)
                    vals[i], lens[i] = C.addressof(buf), len(pay)
                    pyvals.append(pay.hex() if len(pay) <= 400 else "x%d:%d" % (len(pay), pay[0]))
                    if len(pay) > 400:                      # long payloads are regenerated from (length, byte): keep them uniform
                        pay = bytes([pay[0]]) * len(pay)
                        buf = C.create_string_buffer(pay, len(pay))
                        keep.append(buf)
                        vals[i] = C.addressof(buf)
                elif c == "float8":
                    x = rng.choice([0.0, 1.0, -2.5, rng.uniform(-1e5, 1e5)])
                    vals[i] = f2b(x)
                    pyvals.append(str(f2b(x)))
                else:
                    bits = {8: 64, 4: 32, 2: 16, 1: 1}[l]
                    x = rng.getrandbits(bits) - (2 ** (bits - 1) if bits > 1 else 0)
                    vals[i] = x
                    pyvals.append(str(x))
            cap = 200000
            outbuf = (C.c_uint8 * cap)()
            ln = R.ref_memtuple_form(n, attrs, vals, lens, nulls, outbuf, cap)
            mt = bytes(outbuf[:ln])
            dv, dn = (C.c_int64 * n)(), (C.c_uint8 * n)()
            R.ref_memtuple_deform(n, attrs, (C.c_uint8 * ln).from_buffer_copy(mt), dv, dn)
            rec = {"desc": name, "values": pyvals, "deform": [str(dv[i]) for i in range(n)], "deform_null": [int(dn[i]) for i in range(n)]}
            if ln <= 4096:
                rec["memtuple"] = mt.hex()
            else:
                import hashlib
                rec["memtuple_len"], rec["memtuple_sha1"] = ln, hashlib.sha1(mt).hexdigest()
            if ln <= 4096:
                rec["chunks"] = {}
                for mc in (8124, 64, 16):
                    nch = C.c_int32(0)
                    cb = (C.c_uint8 * (4 * ln + 4096))()
                    t = R.ref_serialize_tuple(n, attrs, vals, lens, nulls, 0, mc, cb, len(cb), C.byref(nch))
                    rec["chunks"][str(mc)] = [bytes(cb[:t]).hex(), nch.value]
                nch = C.c_int32(0)
                cb = (C.c_uint8 * (4 * ln + 4096))()
                t = R.ref_serialize_tuple(n, attrs, vals, lens, nulls, 1, rng.choice([8124, 48]), cb, len(cb), C.byref(nch))
                rec["heap_chunks"] = bytes(cb[:t]).hex()
            cases.append(rec)
    json.dump({"descs": meta, "cases": cases}, open(os.path.join(HERE, "memtuple_kat.json"), "w"))
    print("memtuple_kat.json", len(cases))


def numeric_kat():
    """numeric goldens out of the reference's numeric.o (oracle/ref_build/refwrap_numeric.c)"""
    rng = random.Random(20260924)
    out = {"values": [], "binops": [], "cmp": [], "sumavg": []}
    buf, txt = (C.c_uint8 * 256)(), C.create_string_buffer(512)

    def rand_text(maxdigits=15, scales=(0, 1, 2, 2, 2, 3, 4, 6)):
        sc = rng.choice(scales)
        mag = rng.choice([0, 1, 7, 99, 100, 9999, 10000, rng.getrandbits(rng.randint(1, int(maxdigits * 3.3)))])
        return capi.numeric_text(mag * rng.choice([1, 1, -1]), sc)

    for t in ["0", "0.00", "1", "-1", "0.01", "-0.05", "12345.60", "9999999999999.99", "10000", "10000.0001", "0.0001", "123456789012345678"] + [rand_text(18, (0, 1, 2, 4, 9, 15, 20, 70)) for _ in range(300)]:
        n = R.ref_numeric_in(t.encode(), -1, buf, 256)
        out["values"].append([t, bytes(buf[4:n]).hex()])
    for _ in range(600):
        a, b, op = rand_text(), rand_text(), rng.choice("+-*")
        n = R.ref_numeric_binop(ord(op), a.encode(), b.encode(), txt, 512)
        assert n > 0
        out["binops"].append([op, a, b, txt.value.decode()])
        out["cmp"].append([a, b, R.ref_numeric_cmp(a.encode(), b.encode())])
    for _ in range(60):
        sc = rng.choice([0, 2, 2, 4, 6])
        vals = [capi.numeric_text(rng.randint(-10 ** rng.randint(1, 12), 10 ** rng.randint(1, 12)) if rng.random() < 0.9 else 0, sc) for _ in range(rng.choice([1, 2, 3, 10, 200]))]
        if rng.random() < 0.2:
            vals = [capi.numeric_text(rng.randint(0, 99), sc) for _ in vals]           # small sums: fractional averages
        acc = "0"
        for v in vals:
            R.ref_numeric_binop(ord("+"), acc.encode(), v.encode(), txt, 512)
            acc = txt.value.decode()
        R.ref_numeric_binop(ord("/"), acc.encode(), str(len(vals)).encode(), txt, 512)
        out["sumavg"].append({"values": vals, "sum": acc, "avg": txt.value.decode()})
    json.dump(out, open(os.path.join(HERE, "numeric_kat.json"), "w"))
    print("numeric_kat.json", {k: len(v) for k, v in out.items()})


def mvcc_kat():
    """HeapTupleSatisfiesMVCC out of the reference's tqual.o + transam.o (oracle/ref_build/refwrap_tqual.c): tuple headers with
    every combination of the hint and lock bits the rule reads, xmin / xmax drawn around the snapshot's xmin, xmax and xip
    (one xid universe crosses the 2^32 wrap), the scanning backend's own xid with command ids around curcid, and a random
    commit / abort / in-progress status per xid.  `unsupported` holds the headers the device refuses (multixact, combo cid,
    moved tuples, sub-committed or out-of-range status): no reference answer is recorded for those."""
    rng = random.Random(20260925)
    R.ref_heap_satisfies_mvcc.restype = C.c_int
    R.ref_heap_satisfies_mvcc.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p]
    R.ref_tqual_flush_cache.argtypes = [C.c_uint32]
    XC, XI, AC, AI, MULTI, LOCK, EXCL, KEYSHR, COMBO, MOVED_OFF, MOVED_IN = 0x100, 0x200, 0x400, 0x800, 0x1000, 0x80, 0x40, 0x10, 0x20, 0x4000, 0x8000
    snaps, cases, unsupported = [], [], []
    for si in range(48):
        base = 0xFFFFFFE0 if si % 6 == 5 else 4 * rng.randint(1, 10 ** 6)
        n = 64
        xid = lambda d: (base + d) & 0xFFFFFFFF
        ok = [d for d in range(n) if xid(d) >= 3]
        status = [rng.choice([0, 1, 1, 1, 2]) for _ in range(n)]
        lo = rng.randint(8, 30)
        hi = rng.randint(lo, 56)
        xip_d = sorted(rng.sample([d for d in range(lo, hi) if d in ok], min(rng.randint(0, 6), len([d for d in range(lo, hi) if d in ok])))) if hi > lo else []
        own_d = rng.choice([None, None] + [d for d in ok if d >= lo])
        if own_d is not None:
            status[own_d] = 0
        clog = bytearray((n + 3) // 4)
        for d, st in enumerate(status):
            clog[d >> 2] |= st << ((d & 3) * 2)
        snap = {"xmin": xid(lo) if xid(lo) >= 3 else 3, "xmax": xid(hi) if xid(hi) >= 3 else 3, "xip": [xid(d) for d in xip_d], "curcid": rng.randint(0, 6),
                "own_xid": xid(own_d) if own_d is not None else 0, "clog_base": base, "clog_n": n, "clog": bytes(clog).hex()}
        snaps.append(snap)
        xip_arr = (C.c_uint32 * max(1, len(snap["xip"])))(*snap["xip"])
        pick = lambda: rng.choice([xid(rng.choice(ok)), xid(rng.choice(ok)), snap["own_xid"] or xid(rng.choice(ok)), 2, 0, snap["xmin"], snap["xmax"]] + snap["xip"])
        for _ in range(70):
            infomask = 0x0002
            for bit, pr in ((XC, 0.35), (XI, 0.2), (AC, 0.3), (AI, 0.35), (LOCK, 0.08), (EXCL, 0.12), (KEYSHR, 0.08)):
                if rng.random() < pr:
                    infomask |= bit
            xmin, xmax, cid = pick(), pick(), rng.randint(0, 7)
            hdr = struct.pack("<IIIHHHHHB", xmin, xmax, cid, 0, 0, 1, 8, infomask, 24) + b"\0"
            R.ref_tqual_flush_cache(0x7FFFFFF0)
            vis = R.ref_heap_satisfies_mvcc(hdr, snap["xmin"], snap["xmax"], len(snap["xip"]), xip_arr, snap["curcid"], snap["own_xid"], base, n, bytes(clog))
            cases.append([si, infomask, xmin, xmax, cid, vis])
        for _ in range(8):
            infomask = 0x0002 | rng.choice([0, XC, AC, XC | AC])
            kind = rng.choice(["multi", "combo", "moved", "range"])
            xmin, xmax, cid = xid(rng.choice(ok)), xid(rng.choice(ok)), 1
            if kind == "multi":
                infomask = (infomask | MULTI) & ~(AI | LOCK)
            elif kind == "combo":
                if not snap["own_xid"]:
                    continue
                infomask = (infomask | COMBO) & ~XC
                xmin = snap["own_xid"]
            elif kind == "moved":
                infomask = (infomask | rng.choice([MOVED_OFF, MOVED_IN])) & ~XC
            elif kind == "range":
                infomask &= ~XC
                xmin = (base + n + rng.randint(0, 1000)) & 0xFFFFFFFF
                if xmin < 3 or xmin == snap["own_xid"]:
                    continue
            unsupported.append([si, infomask, xmin, xmax, cid, kind])
    json.dump({"snapshots": snaps, "cases": cases, "unsupported": unsupported}, open(os.path.join(HERE, "mvcc_kat.json"), "w"))
    print("mvcc_kat.json", len(snaps), "snapshots,", len(cases), "cases,", sum(c[5] for c in cases), "visible,", len(unsupported), "unsupported")


def float_kat():
    out = {"arith": [], "cmp": [], "accum": [], "combine": [], "avg": [], "int8inc": [], "int8pl": [], "date_ts": []}
    specials = [0.0, -0.0, 1.0, -1.0, 0.5, 1e308, -1e308, 1.7976931348623157e308, 4.9e-324, 1e-308, 1e-200, 1e200,
                float("inf"), float("-inf"), float("nan"), 3.14, 100.25, 0.07]
    vals = specials + [rng.uniform(-1e6, 1e6) for _ in range(40)]
    err = C.c_int32(0)
    for fn in ("pl", "mi", "mul", "div"):
        f = getattr(R, "ref_float8" + fn)
        for _ in range(400):
            a, b = rng.choice(vals), rng.choice(vals)
            r = f(a, b, C.byref(err))
            out["arith"].append([fn, str(f2b(a)), str(f2b(b)), int(err.value), str(f2b(r)) if not err.value else "0",
                                 R.ref_last_error().decode() if err.value and hasattr(R.ref_last_error, "restype") else ""])
    for _ in range(400):
        a, b = rng.choice(vals), rng.choice(vals)
        out["cmp"].append([str(f2b(a)), str(f2b(b)), R.ref_float8eq(a, b), R.ref_float8lt(a, b), R.ref_float8le(a, b), R.ref_btfloat8cmp(a, b)])
    for _ in range(100):
        st = (C.c_double * 3)(0.0, 0.0, 0.0)
        seq = [rng.choice([1.0, 2.5, 1e307, 1e308, -1e308, 1e154, 1e155, 3.0, float("inf")]) for _ in range(rng.randint(1, 6))]
        errs = []
        for x in seq:
            R.ref_float8_accum(st, x, C.byref(err))
            errs.append(int(err.value))
            if err.value:
                break
        out["accum"].append([[str(f2b(x)) for x in seq], errs, [str(f2b(st[i])) for i in range(3)]])
    for _ in range(100):
        a = (C.c_double * 3)(float(rng.randint(0, 5)), rng.choice(vals[:14]), abs(rng.choice(vals[:12])))
        b = (C.c_double * 3)(float(rng.randint(0, 5)), rng.choice(vals[:14]), abs(rng.choice(vals[:12])))
        a0 = [str(f2b(a[i])) for i in range(3)]
        R.ref_float8_combine(a, b, C.byref(err))
        out["combine"].append([a0, [str(f2b(b[i])) for i in range(3)], int(err.value), [str(f2b(a[i])) for i in range(3)]])
    isn = C.c_int32(0)
    for _ in range(60):
        st = (C.c_double * 3)(float(rng.choice([0, 1, 2, 7, 1000])), rng.choice(vals[:12]), 1.0)
        r = R.ref_float8_avg(st, C.byref(isn))
        out["avg"].append([[str(f2b(st[i])) for i in range(3)], int(isn.value), str(f2b(r))])
    for v in [0, 1, -1, 2 ** 63 - 2, 2 ** 63 - 1, -2 ** 63]:
        r = R.ref_int8inc(v, C.byref(err))
        out["int8inc"].append([str(v), int(err.value), str(r)])
    ints = [0, 1, -1, 2 ** 63 - 1, -2 ** 63, 2 ** 62, -2 ** 62, 12345]
    for a in ints:
        for b in ints:
            r = R.ref_int8pl(a, b, C.byref(err))
            out["int8pl"].append([str(a), str(b), int(err.value), str(r)])
    US = 86400000000
    dates = [0, 1, -1, -396, -504, 10957, -2921, 2 ** 31 - 1, -2 ** 31, 106751991, 106751992, -106751991, -106751992]
    tss = [0, -396 * US, -504 * US, -504 * US + 1, -504 * US - 1, 2 ** 63 - 1, -2 ** 63, 12345678901234]
    for op in range(6):
        for d in dates:
            for ts in tss:
                r = R.ref_date_cmp_timestamp(op, d, ts, C.byref(err))
                out["date_ts"].append([op, d, str(ts), int(err.value), int(r)])
    json.dump(out, open(os.path.join(HERE, "float_kat.json"), "w"))
    print("float_kat.json", {k: len(v) for k, v in out.items()})


def lineitem_fixture():
    rows = []
    for fn in ("lineitem_small.csv", "lineitem.csv"):      # load order of input/rpt_tpch.source:98-99
        for ln in open(os.path.join(REF, "src/test/regress/data", fn), encoding="latin1"):
            f = ln.rstrip("\n").split("|")
            if len(f) >= 16:
                rows.append(f[:16])
    epoch = date(2000, 1, 1)

    def d2i(s):
        y, m, d = map(int, s.split("-"))
        return (date(y, m, d) - epoch).days

    instr = sorted({r[13] for r in rows})
    modes = sorted({r[14] for r in rows})
    np.savez_compressed(
        os.path.join(HERE, "lineitem_q1.npz"),
        orderkey=np.array([int(r[0]) for r in rows], dtype=np.int64),
        partkey=np.array([int(r[1]) for r in rows], dtype=np.int32),
        suppkey=np.array([int(r[2]) for r in rows], dtype=np.int32),
        linenumber=np.array([int(r[3]) for r in rows], dtype=np.int32),
        quantity=np.array([float(r[4]) for r in rows]), extendedprice=np.array([float(r[5]) for r in rows]),
        discount=np.array([float(r[6]) for r in rows]), tax=np.array([float(r[7]) for r in rows]),
        returnflag=np.array([ord(r[8]) for r in rows], dtype=np.uint8),
        linestatus=np.array([ord(r[9]) for r in rows], dtype=np.uint8),
        shipdate=np.array([d2i(r[10]) for r in rows], dtype=np.int32),
        commitdate=np.array([d2i(r[11]) for r in rows], dtype=np.int32),
        receiptdate=np.array([d2i(r[12]) for r in rows], dtype=np.int32),
        shipinstruct=np.array([instr.index(r[13]) for r in rows], dtype=np.uint8),
        shipmode=np.array([modes.index(r[14]) for r in rows], dtype=np.uint8),
        comment_len=np.array([len(r[15].encode("latin1")) for r in rows], dtype=np.uint8),
        shipinstruct_names=np.array(instr), shipmode_names=np.array(modes))
    # the golden answer, parsed from the reference's expected output
    txt = open(os.path.join(REF, "src/test/regress/output/rpt_tpch.source")).read().splitlines()
    exp = []
    for i, ln in enumerate(txt):
        if "l_shipdate <= date '1998-12-01' - interval '108 day'" in ln and "heap_lineitem" in "\n".join(txt[i - 4:i]):
            j = i
            while not txt[j].startswith("----------+"):
                j += 1
            j += 1
            while txt[j].strip().startswith("mpph1"):
                f = [x.strip() for x in txt[j].split("|")]
                exp.append({"returnflag": f[1], "linestatus": f[2], "sum_qty": f[3], "sum_base_price": f[4],
                            "sum_disc_price": f[5], "sum_charge": f[6], "avg_qty": f[7], "avg_price": f[8],
                            "avg_disc": f[9], "count_order": int(f[10])})
                j += 1
            break
    assert len(exp) == 4, exp
    json.dump({"source": "src/test/regress/output/rpt_tpch.source:288-315", "interval_days": 108, "rows": exp,
               "nrows_loaded": len(rows)}, open(os.path.join(HERE, "q1_expected.json"), "w"), indent=1)
    print("lineitem_q1.npz", len(rows), "rows; q1_expected.json", exp[0])


def orders_fixture():
    """heap_orders as the reference loads it (order_small.csv + order.csv, input/rpt_tpch.source:92-93) and the golden
    answers of the two TPC-H queries of its regression suite that are a lineitem-orders hash join with an aggregate
    on top: Q4 (semi join, output/rpt_tpch.source 'mpph4') and Q12 (inner join, 'mpph12')."""
    rows = []
    for fn in ("order_small.csv", "order.csv"):
        for ln in open(os.path.join(REF, "src/test/regress/data", fn), encoding="latin1"):
            f = ln.rstrip("\n").split("|")
            if len(f) >= 9:
                rows.append(f[:9])
    epoch = date(2000, 1, 1)

    def d2i(s):
        y, m, d = map(int, s.split("-"))
        return (date(y, m, d) - epoch).days

    prios = sorted({r[5] for r in rows})
    np.savez_compressed(
        os.path.join(HERE, "orders_tpch.npz"),
        orderkey=np.array([int(r[0]) for r in rows], dtype=np.int64), custkey=np.array([int(r[1]) for r in rows], dtype=np.int32),
        orderstatus=np.array([ord(r[2]) for r in rows], dtype=np.uint8), totalprice=np.array([float(r[3]) for r in rows]),
        orderdate=np.array([d2i(r[4]) for r in rows], dtype=np.int32),
        orderpriority=np.array([prios.index(r[5]) for r in rows], dtype=np.uint8), orderpriority_names=np.array(prios),
        shippriority=np.array([int(r[7]) for r in rows], dtype=np.int32))
    txt = open(os.path.join(REF, "src/test/regress/output/rpt_tpch.source")).read().splitlines()

    def answer(tag, first_from):
        """rows of the first result block tagged `tag` whose query reads `first_from` (the heap_ tables)"""
        out = []
        for i, ln in enumerate(txt):
            if ln.strip().startswith("select  '%s'," % tag) and any(first_from in x for x in txt[i:i + 30]):
                j = i
                while not txt[j].startswith("----------+"):
                    j += 1
                j += 1
                while txt[j].strip().startswith(tag + " "):
                    out.append([x.strip() for x in txt[j].split("|")][1:])
                    j += 1
                return out
        raise AssertionError(tag)

    q4 = answer("mpph4", "heap_orders")
    q12 = answer("mpph12", "heap_orders")
    json.dump({"source": "src/test/regress/output/rpt_tpch.source (mpph4, mpph12 over heap_orders/heap_lineitem)",
               "q4": {"orderdate_from": d2i("1994-05-01"), "orderdate_to": d2i("1994-08-01"),
                      "rows": [{"orderpriority": r[0], "order_count": int(r[1])} for r in q4]},
               "q12": {"shipmodes": ["RAIL", "MAIL"], "receipt_from": d2i("1993-01-01"), "receipt_to": d2i("1994-01-01"),
                       "high_priorities": ["1-URGENT", "2-HIGH"],
                       "rows": [{"shipmode": r[0], "high_line_count": int(r[1]), "low_line_count": int(r[2])} for r in q12]},
               "norders_loaded": len(rows)}, open(os.path.join(HERE, "tpch_join_expected.json"), "w"), indent=1)
    print("orders_tpch.npz", len(rows), "rows; q4", q4, "q12", q12)


def join_j1j2_fixture():
    """J1_TBL / J2_TBL of the reference's join regression test (sql/join.sql:6-38: NULL keys, duplicate keys, keys only one
    side has) and its golden result tables for the equi-joins of every outer-join type (expected/join.out)."""
    sql = open(os.path.join(REF, "src/test/regress/sql/join.sql")).read().splitlines()

    def inserts(tab):
        rows = []
        for ln in sql:
            if ln.startswith("INSERT INTO %s VALUES (" % tab):
                vals = [v.strip() for v in ln[ln.index("(") + 1:ln.rindex(")")].split(",")]
                rows.append([None if v == "NULL" else (v.strip("'") if v.startswith("'") else int(v)) for v in vals])
        return rows

    out = open(os.path.join(REF, "src/test/regress/expected/join.out")).read().splitlines()

    def answer(from_clause):
        i = next(n for n, ln in enumerate(out) if ln.strip().startswith(from_clause))
        while not out[i].startswith("-----+"):
            i += 1
        cols = [c.strip() for c in out[i - 1].split("|")][1:]
        rows = []
        i += 1
        while not out[i].startswith("("):
            f = [x.strip() for x in out[i].split("|")][1:]
            rows.append([None if x == "" else (x if c == "t" else int(x)) for c, x in zip(cols, f)])
            i += 1
        assert out[i] == "(%d rows)" % len(rows), (from_clause, out[i], len(rows))
        return {"cols": cols, "rows": rows}

    q = {"inner": answer("FROM J1_TBL INNER JOIN J2_TBL USING (i);"),
         "inner_i_eq_k": answer("FROM J1_TBL JOIN J2_TBL ON (J1_TBL.i = J2_TBL.k);"),
         "left": answer("FROM J1_TBL LEFT OUTER JOIN J2_TBL USING (i)"),
         "right": answer("FROM J1_TBL RIGHT OUTER JOIN J2_TBL USING (i);"),
         "full": answer("FROM J1_TBL FULL OUTER JOIN J2_TBL USING (i)")}
    json.dump({"source": "src/test/regress/sql/join.sql:6-38 (tables), expected/join.out (answers)",
               "j1": inserts("J1_TBL"), "j2": inserts("J2_TBL"), "queries": q},
              open(os.path.join(HERE, "join_j1j2.json"), "w"), indent=1)
    print("join_j1j2.json", {k: len(v["rows"]) for k, v in q.items()})


def sort_fixture():
    """Golden ORDER BY answers of the reference's sort regression test (expected/sort.out): gpsort_alltypes columns of the
    types the Sort path takes (int8, char, date, float8, int4), ASC and DESC, and colltest's text COLLATE "C" with NULLS
    LAST / NULLS FIRST through a merging Gather Motion."""
    out = open(os.path.join(REF, "src/test/regress/expected/sort.out")).read().splitlines()
    epoch = date(2000, 1, 1)

    def block(query):
        i = out.index(query)
        while not out[i].startswith("---"):
            i += 1
        rows = []
        i += 1
        while not out[i].startswith("("):
            rows.append(out[i].strip())
            i += 1
        assert out[i] == "(%d rows)" % len(rows), (query, out[i])
        return rows

    conv = {"int8": int, "int4": int, "float8": float, "bpchar": str,
            "date": lambda x: (date(int(x[6:]), int(x[:2]), int(x[3:5])) - epoch).days}       # regression DateStyle: MM-DD-YYYY
    cols = {}
    for col, typ in (("col1", "int8"), ("col6", "bpchar"), ("col10", "date"), ("col12", "float8"), ("col14", "int4")):
        cols[col] = {"type": typ,
                     "asc": [conv[typ](x) for x in block("select %s from gpsort_alltypes order by %s asc;" % (col, col))],
                     "desc": [conv[typ](x) for x in block("select %s from gpsort_alltypes order by %s desc;" % (col, col))]}
    coll = {"nulls_last": [x or None for x in block('select * from colltest order by t COLLATE "C";')],
            "nulls_first": [x or None for x in block('select * from colltest order by t COLLATE "C" NULLS FIRST;')]}
    json.dump({"source": "src/test/regress/expected/sort.out (gpsort_alltypes, colltest)", "alltypes": cols, "colltest": coll},
              open(os.path.join(HERE, "sort_golden.json"), "w"), indent=1)
    print("sort_golden.json", {k: v["asc"] for k, v in cols.items()}, coll)


def onek_fixture():
    """onek of the reference's regression suite (data/onek.data, 1000 rows; the 13 int4 columns of sql/create_table.sql:18-34)
    and the golden aggregates over it in expected/aggregates.out: sum(four), max(four), count(four), and the hashed
    `select ten, count(*), sum(four) from onek group by ten`."""
    rows = [[int(x) for x in ln.split("\t")[:13]] for ln in open(os.path.join(REF, "src/test/regress/data/onek.data"))]
    np.savez_compressed(os.path.join(HERE, "onek.npz"), ints=np.array(rows, dtype=np.int32))
    out = open(os.path.join(REF, "src/test/regress/expected/aggregates.out")).read().splitlines()

    def block(query):
        i = out.index(query)
        while not out[i].startswith("---"):
            i += 1
        rows = []
        i += 1
        while not out[i].startswith("("):
            rows.append([int(x) for x in out[i].split("|")])
            i += 1
        return rows

    json.dump({"source": "src/test/regress/expected/aggregates.out:30-34,54-58,256-260,268-282",
               "columns": ["unique1", "unique2", "two", "four", "ten", "twenty", "hundred", "thousand", "twothousand", "fivethous",
                           "tenthous", "odd", "even"],
               "sum_four": block("SELECT sum(four) AS sum_1500 FROM onek;")[0][0],
               "max_four": block("SELECT max(four) AS max_3 FROM onek;")[0][0],
               "count_four": block("SELECT count(four) AS cnt_1000 FROM onek;")[0][0],
               "by_ten": block("select ten, count(*), sum(four) from onek")},
              open(os.path.join(HERE, "onek_agg_expected.json"), "w"), indent=1)
    print("onek.npz", len(rows), "rows")


AOCS_TYPES = [("int8", capi.INT8OID, 8, "d", 1), ("int4", capi.INT4OID, 4, "i", 1), ("float8", capi.FLOAT8OID, 8, "d", 1),
              ("date", capi.DATEOID, 4, "i", 1), ("bpchar1", capi.BPCHAROID, -1, "i", 0), ("text", capi.TEXTOID, -1, "i", 0)]


def aocs_attr(typid, attlen, align, byval):
    a = capi.gg_attr()
    a.atttypid, a.atttypmod, a.attlen, a.attalign, a.attbyval, a.attnotnull = typid, -1, attlen, ord(align), byval, 0
    return a


def aocs_kat():
    """Column files of an append-only column-oriented relation (compresstype=none) WRITTEN BY THE REFERENCE'S OWN
    datumstreamblock.o + cdbappendonlystorageformat.o (oracle/ref_build/refwrap_aocs.c), and what its block reader returns
    for them: per type x {no NULLs, 20 % NULLs} x {checksum on, off}, 8 KB blocks so every file has several."""
    g = np.random.default_rng(20260923)
    out = {"crc_inputs": g.integers(0, 256, 4096).astype(np.uint8)}
    lens_for_crc = [0, 1, 3, 8, 12, 13, 64, 1000, 4096]
    out["crc_lens"] = np.array(lens_for_crc, dtype=np.int32)
    out["crc_values"] = np.array([R.ref_aocs_crc32c(out["crc_inputs"].ctypes.data, ln) for ln in lens_for_crc], dtype=np.uint32)
    names = []
    for name, typid, attlen, align, byval in AOCS_TYPES:
        att = aocs_attr(typid, attlen, align, byval)
        n = {"bpchar1": 6000, "text": 1200}.get(name, 2500)
        if name == "float8":
            vals = [float(x) for x in np.concatenate([g.normal(size=n - 6) * 1e3, [0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324]])]
        elif name == "bpchar1":
            vals = [bytes([65 + int(x)]) for x in g.integers(0, 26, n)]
        elif name == "text":
            vals = [bytes(g.integers(97, 123, int(ln)).astype(np.uint8)) for ln in g.choice([0, 1, 5, 30, 125, 126, 127, 128, 300], n)]
        elif name == "int8":
            vals = [int(x) for x in g.integers(-2**62, 2**62, n)]
        else:
            vals = [int(x) for x in g.integers(-2**31, 2**31, n)]
        for nullfrac in (0.0, 0.2):
            nulls = (g.random(n) < nullfrac).astype(np.uint8) if nullfrac else None
            for cs in (1, 0):
                key = "%s_n%d_c%d" % (name, int(nullfrac * 10), cs)
                f = po.aocs_write_column(att, vals, nulls, blocksize=8192, checksum=bool(cs), first_rownum=1, ref=True)
                v, nl, fr, rc = po.aocs_read_column(att, f, n, checksum=bool(cs), ref=True)
                assert len(v) == n and len(rc) > 1
                names.append(key)
                out[key + "_file"], out[key + "_vals"], out[key + "_nulls"] = f, v, nl
                out[key + "_firstrows"], out[key + "_rowcounts"] = fr, rc
                if nulls is not None:
                    out[key + "_innulls"] = nulls
        if attlen == -1:
            out[name + "_inlens"] = np.array([len(b) for b in vals], dtype=np.int32)
            out[name + "_inbytes"] = np.frombuffer(b"".join(vals), dtype=np.uint8)
        elif name == "float8":
            out[name + "_in"] = np.array(vals, dtype=np.float64).view(np.int64)
        else:
            out[name + "_in"] = np.array(vals, dtype=np.int64)
    out["cases"] = np.array(names)
    np.savez_compressed(os.path.join(HERE, "aocs_kat.npz"), **out)
    print("aocs_kat.npz", len(names), "column files")


def hash_random_kat():
    """The reference's hash_any / hashint8 / cdbhash routing of the random inputs tests/test_oracle_hash.py draws
    (random.Random(7)), as SHA-256 digests of each output sequence: 20000 cases in a few bytes."""
    import test_oracle_hash as th
    from test_oracle_aocs import sha256
    out = {"cases": th.RANDOM_CASES}
    for name, fn in (("hash_any", R.ref_hash_any), ("hashint8", R.ref_hashint8), ("route", R.ref_cdbhash_route)):
        out[name] = sha256(th.random_hash_outputs(fn, name))
    json.dump(out, open(os.path.join(HERE, "hash_random_kat.json"), "w"), indent=1)
    print("hash_random_kat.json", out)


def aocs_random_kat():
    """Random column files the reference's own writer makes for tests/test_oracle_aocs.py's random inputs (np.random.default_rng(77),
    32 KB blocks), and what its own reader returns for them, as SHA-256 digests: the files are megabytes, the digests are not."""
    import test_oracle_aocs as ta
    out = []
    for name, nullfrac, a, vals, nulls in ta.random_columns():
        f = po.aocs_write_column(a, vals, nulls, ref=True)
        rv, rn, rf, rr = po.aocs_read_column(a, f, len(vals), ref=True)
        out.append({"type": name, "nullfrac": nullfrac, "rows": len(vals), "file_bytes": int(f.size), "file": ta.sha256(f),
                    "read": ta.sha256(rv, rn, rf, rr), "max_rows_per_block": int(rr.max())})
    json.dump(out, open(os.path.join(HERE, "aocs_random_kat.json"), "w"), indent=1)
    print("aocs_random_kat.json", len(out), "column files")


def wire_kat():
    """Tuple chunks across a Motion, as tests/test_executor_wire.py exchanges them with the reference's tupser.o / tupchunklist.o:
      partial  the PARTIAL-stage Q1 rows of segment 0 as the product's GgExecSendTupleChunks writes them (two chunk sizes), and
               what the reference's CvtChunksToTup reads from each tuple's chunks
      senders  every segment's rows written by the reference's SerializeTuple, as a MemTuple and as a heap tuple"""
    import tempfile
    import test_executor_wire as tw
    from greengage_b200 import executor as ex
    L = tw.bind_mock(C.CDLL(tw.build_mock(tempfile.mkdtemp())))
    old, ex._lib = ex._lib, L
    eng = L.mock_engine()
    # the PARTIAL Q1 row: two bpchar keys, four float8 sums, three float8[] {N, sumX, sumX2}, count
    wire = [(1042, -1, 'i', 0), (1042, -1, 'i', 0)] + [(701, 8, 'd', 1)] * 4 + [(1022, -1, 'd', 0)] * 3 + [(20, 8, 'd', 1)]
    attrs = (capi.gg_attr * len(wire))()
    for i, (t, l, al, bv) in enumerate(wire):
        attrs[i].atttypid, attrs[i].attlen, attrs[i].attalign, attrs[i].attbyval, attrs[i].atttypmod = t, l, ord(al), bv, -1
    out = {"partial": {}, "senders": {"ref-memtuple": [], "ref-heap": []}}
    for max_chunk in tw.PARTIAL_CHUNK_SIZES:
        stream, n, rows = tw.partial_chunks(L, eng, 0, max_chunk)
        read, pos = [], 0
        for _ in rows:
            end = pos                                   # one tuple's chunks: up to and including the WHOLE / PARTIAL_END chunk
            while True:
                size, typ = struct.unpack_from("<HH", stream, end)
                end += 4 + size
                if typ in (0, 3):
                    break
            vals, lens, nulls, sb = (C.c_int64 * 10)(), (C.c_int32 * 10)(), (C.c_uint8 * 10)(), (C.c_uint8 * 1024)()
            form = R.ref_deserialize_tuple(10, attrs, stream[pos:end], end - pos, vals, lens, nulls, sb, 1024)
            sbb = bytes(sb)
            read.append({"form": form, "nulls": list(nulls),
                         "keys": [sbb[vals[k]:vals[k] + lens[k]].decode() for k in range(2)],
                         "sums": list(vals[2:6]), "count": vals[9],
                         "arrays": [list(struct.unpack_from("<iiIii3q", sbb, vals[6 + k])) for k in range(3)],
                         "array_lens": list(lens[6:9])})
            pos = end
        assert pos == len(stream) - 4
        out["partial"][str(max_chunk)] = {"stream": stream.hex(), "read": read}
    for form in out["senders"]:
        for seg in range(tw.NSEG):
            _, _, rows = tw.partial_chunks(L, eng, seg, 8124)
            parts = []
            for v, nl, ty, ln in rows:
                keep = [C.create_string_buffer(capi.unpack_str(v[k], ln[k]).encode(), max(ln[k], 1)) for k in range(2)]
                arrs = [C.create_string_buffer(struct.pack("<iiIii3q", 1, 0, 701, 3, 1, *v[6 + 3 * k:9 + 3 * k]), 44) for k in range(3)]
                vals = (C.c_int64 * 10)(C.addressof(keep[0]), C.addressof(keep[1]), v[2], v[3], v[4], v[5],
                                        C.addressof(arrs[0]), C.addressof(arrs[1]), C.addressof(arrs[2]), v[15])
                lens = (C.c_int32 * 10)(ln[0], ln[1], 0, 0, 0, 0, 44, 44, 44, 0)
                buf, nch = (C.c_uint8 * 4096)(), C.c_int32(0)
                t = R.ref_serialize_tuple(10, attrs, vals, lens, (C.c_uint8 * 10)(), 1 if form == "ref-heap" else 0,
                                          tw.SENDER_CHUNK_SIZES[seg], buf, 4096, C.byref(nch))
                parts.append(bytes(buf[:t]))
            out["senders"][form].append(b"".join(parts).hex())
    ex._lib = old
    json.dump(out, open(os.path.join(HERE, "wire_kat.json"), "w"), indent=1)
    print("wire_kat.json", {k: len(v["stream"]) // 2 for k, v in out["partial"].items()})


if __name__ == "__main__":
    R.ref_last_error.restype = C.c_char_p
    if len(sys.argv) > 1:                  # only the named fixtures: python make_golden.py memtuple_kat
        for fn in sys.argv[1:]:
            globals()[fn]()
        sys.exit(0)
    hash_kat()
    heap_kat()
    float_kat()
    lineitem_fixture()
    orders_fixture()
    join_j1j2_fixture()
    sort_fixture()
    onek_fixture()
    aocs_kat()
    memtuple_kat()
    numeric_kat()
    mvcc_kat()
    hash_random_kat()
    aocs_random_kat()
    wire_kat()

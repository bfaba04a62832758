"""The oracle's hashing and segment routing against golden vectors computed by the reference's own
hashfunc.o / varchar.o / cdbhash.o (tests/golden/make_golden.py), value by value and, for 20000 random
inputs, as digests of what those objects returned.  The product's host-side routing (libgghost) is held to the
same vectors."""
import ctypes as C
import hashlib
import random

import numpy as np

from _util import golden
from greengage_b200 import capi
from oracle import pyoracle as po

K = golden("hash_kat.json")
L = po.lib()


def test_hash_any_golden():
    for hexs, want in K["hash_any"]:
        b = bytes.fromhex(hexs)
        assert L.or_hash_any(b, len(b)) == want
        assert capi.host_lib().gg_hash_any(b, len(b)) == want


def test_scalar_hashes_golden():
    for v, want in K["hash_uint32"]:
        assert L.or_hash_uint32(v) == want
    for v, want in K["hashint4"]:
        assert L.or_hashint4(v) == want
    for v, want in K["hashint8"]:
        assert L.or_hashint8(int(v)) == want
    for bits, want in K["hashfloat8"]:
        assert L.or_hashfloat8(C.c_double.from_buffer_copy(C.c_int64(int(bits))).value) == want


def test_known_answers_from_survey():
    # SURVEY.md §8c: values obtained from the reference's hashfunc.o
    assert L.or_hash_uint32(0) == 4022255791 and L.or_hash_uint32(1) == 2389907270 and L.or_hash_uint32(42) == 1509752520
    for s, want in ((b"A", 1656725486), (b"N", 1706742859), (b"R", 4055972430), (b"F", 1874189369), (b"O", 2962905310)):
        assert L.or_hash_any(s, 1) == want
    assert L.or_hashfloat8(1.0) == 376496956


def test_bpchar_golden():
    for hexs, want in K["hashbpchar"]:
        b = bytes.fromhex(hexs)
        assert L.or_hashbpchar(b, len(b)) == want
    for a, b, want in K["bpchareq"]:
        a, b = bytes.fromhex(a), bytes.fromhex(b)
        assert L.or_bpchareq(a, len(a), b, len(b)) == want


def test_routing_golden_oracle_and_product():
    H = capi.host_lib()
    for r in K["route"]:
        n = len(r["typ"])
        t = (C.c_int32 * n)(*r["typ"])
        v = (C.c_int64 * n)(*[int(x) for x in r["val"]])
        ln = (C.c_int32 * n)(*r["len"])
        nu = (C.c_int32 * n)(*r["null"])
        assert L.or_route_datums(t, v, ln, nu, n, r["nsegs"]) == r["seg"]
        assert H.gg_cdbhash_route(t, v, ln, nu, n, r["nsegs"]) == r["seg"]


RANDOM_CASES = 20000


def random_hash_outputs(fn, name):
    """fn's answers to the RANDOM_CASES inputs random.Random(7) draws, as an array: hash_any of 0..48 random bytes ("hash_any"),
    hashint8 of a random int8 ("hashint8"), or the segment a random int8 key routes to among 1..999 ("route")."""
    rng = random.Random(7)
    out = []
    for _ in range(RANDOM_CASES):
        n = rng.randint(0, 48)
        b = bytes(rng.getrandbits(8) for _ in range(n))
        v = rng.getrandbits(64) - (1 << 63)
        ns = rng.choice([1, 2, 3, 5, 8, 13, 64, 999])
        if name == "hash_any":
            out.append(fn(b, n))
        elif name == "hashint8":
            out.append(fn(v))
        else:
            t, vv, ln, nu = (C.c_int32 * 1)(20), (C.c_int64 * 1)(v), (C.c_int32 * 1)(0), (C.c_int32 * 1)(0)
            out.append(fn(t, vv, ln, nu, 1, ns))
    return np.array(out, dtype=np.int32 if name == "route" else np.uint32)


def test_against_reference_objects_when_built():
    """The oracle on RANDOM_CASES random inputs against what the reference's own hashfunc.o / cdbhash.o returned for them
    (tests/golden/hash_random_kat.json keeps a SHA-256 digest of each output sequence; make_golden.py hash_random_kat)."""
    kat = golden("hash_random_kat.json")
    assert kat["cases"] == RANDOM_CASES
    for name, fn in (("hash_any", L.or_hash_any), ("hashint8", L.or_hashint8), ("route", L.or_route_datums)):
        assert hashlib.sha256(random_hash_outputs(fn, name).tobytes()).hexdigest() == kat[name], name


def test_bulk_routing_of_aggregate_rows_matches_the_oracle():
    """greengage_b200.motion.route_rows_raw (one C call over a gg_aggrow array, what bench.py's Redistribute uses) against
    the oracle's cdbhash restatement, row by row: int, float8 (incl. -0), packed-string and NULL keys."""
    import ctypes as C
    import numpy as np
    from greengage_b200 import capi, motion
    from oracle import pyoracle as po
    rng = np.random.default_rng(31)
    n = 500
    rows = (capi.gg_aggrow * n)()
    typids = [capi.INT8OID, capi.BPCHAROID, capi.FLOAT8OID, capi.INT4OID]
    for r in rows:
        r.key[0] = int(rng.integers(-2**40, 2**40))
        s, ln = capi.pack_str("".join(rng.choice(list("ABCxyz"), int(rng.integers(0, 6)))))
        r.key[1], r.keylen[1] = s, ln
        f = float(rng.choice([0.0, -0.0, 1.5, -2.25, 1e300, float(rng.normal())]))
        r.key[2] = np.float64(f).view(np.int64).item()
        r.key[3] = int(rng.integers(-1000, 1000))
        for c in range(4):
            r.keyisnull[c] = int(rng.random() < 0.15)
    buf = np.frombuffer(rows, dtype=np.uint8)
    for nsegs in (1, 2, 3, 8, 64):
        got = motion.route_rows_raw(buf, n, typids, nsegs)
        t = (C.c_int32 * 4)(*typids)
        for i, r in enumerate(rows):
            v = (C.c_int64 * 4)(*[r.key[c] for c in range(4)])
            ln = (C.c_int32 * 4)(*[r.keylen[c] for c in range(4)])
            nn = (C.c_int32 * 4)(*[r.keyisnull[c] for c in range(4)])
            assert got[i] == po.lib().or_route_datums(t, v, ln, nn, 4, nsegs), (i, nsegs)

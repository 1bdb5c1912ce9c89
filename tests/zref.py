"""ctypes bindings used by the tests only.

  ref       -- the UNMODIFIED reference, oracle/_ref/libzopfli_ref.so (+ libref_seams.so wrappers)
  oracle    -- the plain-C restatement, oracle/_build/libzopfli_oracle.so
  Reference -- the reference's answers to the tests' calls, recorded in tests/golden/reference_answers.json,
               so that the comparisons run where the reference cannot be built
Neither is ever imported by the product package.
"""
from __future__ import annotations

import atexit
import ctypes as C
import hashlib
import json
import multiprocessing as mp
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")

u8p = C.POINTER(C.c_ubyte)
u16p = C.POINTER(C.c_uint16)


from zopfli_b200 import ZopfliOptions  # same 6-int layout, zopfli.h:33-64


def ensure_built(reference=False):
    """the oracle's libraries; with `reference`, also the reference's (oracle/Makefile builds them where its
    sources are readable)"""
    need = [os.path.join(ORACLE_DIR, "_build", "libzopfli_oracle.so")]
    if reference:
        need += [os.path.join(ORACLE_DIR, "_ref", "libzopfli_ref.so"),
                 os.path.join(ORACLE_DIR, "_ref", "libref_seams.so")]
    if not all(os.path.exists(p) for p in need):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "all" if reference else "oracle"])


def reference_built(ndebug=False):
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libzopfli_ref_ndebug.so" if ndebug else "libzopfli_ref.so"))


def _np_u8(b):
    a = np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else b
    # pad so that neither library can read past the end
    pad = np.zeros(len(a) + 16, dtype=np.uint8)
    pad[: len(a)] = a
    return pad


def _ptr(a, t):
    return a.ctypes.data_as(t)


class Ref:
    def __init__(self, ndebug=False):
        ensure_built(reference=True)
        name = "libzopfli_ref_ndebug.so" if ndebug else "libzopfli_ref.so"
        self.lib = C.CDLL(os.path.join(ORACLE_DIR, "_ref", name))
        self.seams = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libref_seams.so"))
        self.lib.ZopfliCompress.argtypes = [C.POINTER(ZopfliOptions), C.c_int, C.c_void_p, C.c_size_t,
                                            C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        self.lib.ZopfliCompress.restype = None
        self.lib.ZopfliDeflatePart.argtypes = [C.POINTER(ZopfliOptions), C.c_int, C.c_int, C.c_void_p,
                                               C.c_size_t, C.c_size_t, u8p, C.POINTER(C.c_void_p),
                                               C.POINTER(C.c_size_t)]
        self.lib.ZopfliDeflatePart.restype = None
        self.lib.ZopfliDeflate.argtypes = [C.POINTER(ZopfliOptions), C.c_int, C.c_int, C.c_void_p,
                                           C.c_size_t, u8p, C.POINTER(C.c_void_p),
                                           C.POINTER(C.c_size_t)]
        self.lib.ZopfliDeflate.restype = None
        self.libc = C.CDLL(None)
        self.libc.free.argtypes = [C.c_void_p]
        s = self.seams
        s.ref_lz77.restype = C.c_size_t
        s.ref_lz77.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_void_p,
                               C.c_void_p, C.c_size_t]
        s.ref_match_table.restype = None
        s.ref_match_table.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t] + [C.c_void_p] * 6
        s.ref_limited_match.restype = None
        s.ref_limited_match.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.c_void_p]
        s.ref_block_size.restype = C.c_double
        s.ref_block_size.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                     C.c_size_t, C.c_int]
        s.ref_block_split_lz77.restype = C.c_size_t
        s.ref_block_split_lz77.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                           C.c_void_p, C.c_size_t]
        s.ref_block_split.restype = C.c_size_t
        s.ref_block_split.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p,
                                      C.c_size_t]
        s.ref_length_limited.restype = C.c_int
        s.ref_length_limited.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        s.ref_entropy.restype = None
        s.ref_entropy.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        s.ref_optimize_rle.restype = None
        s.ref_optimize_rle.argtypes = [C.c_int, C.c_void_p]

    @staticmethod
    def options(numiterations=15, blocksplitting=1, blocksplittingmax=15):
        o = ZopfliOptions(0, 0, numiterations, blocksplitting, 0, blocksplittingmax)
        return o

    def compress(self, data: bytes, fmt=0, **kw) -> bytes:
        """ZopfliCompress; fmt 0 gzip, 1 zlib, 2 deflate (zopfli.h:70-74)."""
        o = self.options(**kw)
        a = _np_u8(data)
        out = C.c_void_p(None)
        n = C.c_size_t(0)
        self.lib.ZopfliCompress(C.byref(o), fmt, a.ctypes.data, len(data), C.byref(out), C.byref(n))
        res = C.string_at(out, n.value) if n.value else b""
        self.libc.free(out)
        return res

    def deflate_part(self, data: bytes, instart, inend, final=1, btype=2, **kw):
        o = self.options(**kw)
        a = _np_u8(data)
        out = C.c_void_p(None)
        n = C.c_size_t(0)
        bp = C.c_ubyte(0)
        self.lib.ZopfliDeflatePart(C.byref(o), btype, final, a.ctypes.data, instart, inend,
                                   C.byref(bp), C.byref(out), C.byref(n))
        res = C.string_at(out, n.value) if n.value else b""
        self.libc.free(out)
        return res, bp.value

    def lz77(self, data: bytes, instart, inend, mode=0, numiterations=15):
        a = _np_u8(data)
        cap = inend - instart + 16
        ll = np.zeros(cap, dtype=np.uint16)
        dd = np.zeros(cap, dtype=np.uint16)
        n = self.seams.ref_lz77(a.ctypes.data, instart, inend, mode, numiterations, ll.ctypes.data,
                                dd.ctypes.data, cap)
        return ll[:n].copy(), dd[:n].copy()

    def match_table(self, data: bytes, instart, inend, want_sublen=True):
        a = _np_u8(data)
        n = inend - instart
        ln = np.zeros(n, dtype=np.uint16)
        ds = np.zeros(n, dtype=np.uint16)
        sub = np.zeros((n, 259), dtype=np.uint16) if want_sublen else None
        same = np.zeros(n, dtype=np.uint16)
        hv = np.zeros(n, dtype=np.int32)
        hv2 = np.zeros(n, dtype=np.int32)
        self.seams.ref_match_table(a.ctypes.data, instart, inend, ln.ctypes.data, ds.ctypes.data,
                                   sub.ctypes.data if want_sublen else None, same.ctypes.data,
                                   hv.ctypes.data, hv2.ctypes.data)
        return ln, ds, sub, same, hv, hv2

    def limited_match(self, data, instart, inend, limits):
        a = _np_u8(data)
        n = inend - instart
        lim = np.ascontiguousarray(limits, dtype=np.uint16)
        ln = np.zeros(n, dtype=np.uint16)
        ds = np.zeros(n, dtype=np.uint16)
        self.seams.ref_limited_match(a.ctypes.data, instart, inend, lim.ctypes.data, ln.ctypes.data,
                                     ds.ctypes.data)
        return ln, ds

    def block_size(self, data, litlens, dists, lstart, lend, btype):
        a = _np_u8(data)
        ll = np.ascontiguousarray(litlens, dtype=np.uint16)
        dd = np.ascontiguousarray(dists, dtype=np.uint16)
        return self.seams.ref_block_size(a.ctypes.data, ll.ctypes.data, dd.ctypes.data, len(ll), lstart,
                                         lend, btype)

    def block_split_lz77(self, data, litlens, dists, maxblocks=15):
        a = _np_u8(data)
        ll = np.ascontiguousarray(litlens, dtype=np.uint16)
        dd = np.ascontiguousarray(dists, dtype=np.uint16)
        pts = np.zeros(64 + maxblocks, dtype=np.uint64)
        n = self.seams.ref_block_split_lz77(a.ctypes.data, ll.ctypes.data, dd.ctypes.data, len(ll),
                                            maxblocks, pts.ctypes.data, len(pts))
        return pts[:n].astype(np.int64)

    def block_split(self, data, instart, inend, maxblocks=15):
        a = _np_u8(data)
        pts = np.zeros(64 + maxblocks, dtype=np.uint64)
        n = self.seams.ref_block_split(a.ctypes.data, instart, inend, maxblocks, pts.ctypes.data, len(pts))
        return pts[:n].astype(np.int64)

    def length_limited(self, freq, maxbits):
        f = np.ascontiguousarray(freq, dtype=np.uint64)
        out = np.zeros(len(f), dtype=np.uint32)
        err = self.seams.ref_length_limited(f.ctypes.data, len(f), maxbits, out.ctypes.data)
        return err, out

    def entropy(self, counts):
        c = np.ascontiguousarray(counts, dtype=np.uint64)
        out = np.zeros(len(c), dtype=np.float64)
        self.seams.ref_entropy(c.ctypes.data, len(c), out.ctypes.data)
        return out

    def optimize_rle(self, counts):
        c = np.array(counts, dtype=np.uint64)
        self.seams.ref_optimize_rle(len(c), c.ctypes.data)
        return c


class ZoStore(C.Structure):
    _fields_ = [("litlens", u16p), ("dists", u16p), ("pos", C.POINTER(C.c_uint32)),
                ("size", C.c_size_t), ("cap", C.c_size_t)]


class Oracle:
    def __init__(self):
        ensure_built()
        L = self.lib = C.CDLL(os.path.join(ORACLE_DIR, "_build", "libzopfli_oracle.so"))
        L.zo_segment_new.restype = C.c_void_p
        L.zo_segment_new.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t]
        L.zo_segment_free.argtypes = [C.c_void_p]
        for f in ("zo_segment_hv", "zo_segment_same", "zo_segment_hv2"):
            getattr(L, f).restype = C.c_uint
            getattr(L, f).argtypes = [C.c_void_p, C.c_size_t]
        L.zo_find_longest_match.restype = None
        L.zo_find_longest_match.argtypes = [C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p,
                                            C.POINTER(C.c_uint16), C.POINTER(C.c_uint16)]
        for f in ("zo_lz77_greedy", "zo_lz77_optimal_fixed"):
            getattr(L, f).restype = None
            getattr(L, f).argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(ZoStore)]
        L.zo_lz77_optimal.restype = None
        L.zo_lz77_optimal.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(ZoStore)]
        L.zo_store_init.argtypes = [C.POINTER(ZoStore)]
        L.zo_store_free.argtypes = [C.POINTER(ZoStore)]
        L.zo_length_limited_code_lengths.restype = C.c_int
        L.zo_length_limited_code_lengths.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.zo_calculate_entropy.restype = None
        L.zo_calculate_entropy.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.zo_dynamic_block_size.restype = C.c_double
        L.zo_dynamic_block_size.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.zo_optimize_huffman_for_rle.restype = None
        L.zo_optimize_huffman_for_rle.argtypes = [C.c_int, C.c_void_p]

    def _store_call(self, fn, *args):
        st = ZoStore()
        self.lib.zo_store_init(C.byref(st))
        fn(*args, C.byref(st))
        n = st.size
        ll = np.ctypeslib.as_array(st.litlens, (n,)).copy() if n else np.zeros(0, np.uint16)
        dd = np.ctypeslib.as_array(st.dists, (n,)).copy() if n else np.zeros(0, np.uint16)
        self.lib.zo_store_free(C.byref(st))
        return ll, dd

    def lz77(self, data, instart, inend, mode=0, numiterations=15):
        a = _np_u8(data)
        if mode == 0:
            return self._store_call(self.lib.zo_lz77_optimal, a.ctypes.data, instart, inend, numiterations)
        if mode == 1:
            return self._store_call(self.lib.zo_lz77_optimal_fixed, a.ctypes.data, instart, inend)
        return self._store_call(self.lib.zo_lz77_greedy, a.ctypes.data, instart, inend)

    def match_table(self, data, instart, inend, want_sublen=True):
        a = _np_u8(data)
        n = inend - instart
        seg = self.lib.zo_segment_new(a.ctypes.data, instart, inend)
        ln = np.zeros(n, dtype=np.uint16)
        ds = np.zeros(n, dtype=np.uint16)
        sub = np.zeros((n, 259), dtype=np.uint16) if want_sublen else None
        same = np.zeros(n, dtype=np.uint16)
        hv = np.zeros(n, dtype=np.int32)
        hv2 = np.zeros(n, dtype=np.int32)
        tmp = np.zeros(259, dtype=np.uint16)
        d = C.c_uint16()
        l = C.c_uint16()
        for j in range(n):
            p = instart + j
            tmp[:] = 0
            self.lib.zo_find_longest_match(seg, p, 258, tmp.ctypes.data, C.byref(d), C.byref(l))
            ln[j], ds[j] = l.value, d.value
            if want_sublen and l.value >= 3:
                sub[j, 3:l.value + 1] = tmp[3:l.value + 1]
            same[j] = self.lib.zo_segment_same(seg, p)
            hv[j] = self.lib.zo_segment_hv(seg, p)
            hv2[j] = self.lib.zo_segment_hv2(seg, p)
        self.lib.zo_segment_free(seg)
        return ln, ds, sub, same, hv, hv2

    def limited_match(self, data, instart, inend, limits):
        a = _np_u8(data)
        n = inend - instart
        seg = self.lib.zo_segment_new(a.ctypes.data, instart, inend)
        ln = np.zeros(n, dtype=np.uint16)
        ds = np.zeros(n, dtype=np.uint16)
        d = C.c_uint16()
        l = C.c_uint16()
        for j in range(n):
            if limits[j] >= 3:
                self.lib.zo_find_longest_match(seg, instart + j, int(limits[j]), None, C.byref(d), C.byref(l))
                ln[j], ds[j] = l.value, d.value
        self.lib.zo_segment_free(seg)
        return ln, ds

    def length_limited(self, freq, maxbits):
        f = np.ascontiguousarray(freq, dtype=np.uint64)
        out = np.zeros(len(f), dtype=np.uint32)
        err = self.lib.zo_length_limited_code_lengths(f.ctypes.data, len(f), maxbits, out.ctypes.data)
        return err, out

    def entropy(self, counts):
        c = np.ascontiguousarray(counts, dtype=np.uint64)
        out = np.zeros(len(c), dtype=np.float64)
        self.lib.zo_calculate_entropy(c.ctypes.data, len(c), out.ctypes.data)
        return out

    def dynamic_block_size(self, llc, dc):
        a = np.ascontiguousarray(llc, dtype=np.uint64)
        b = np.ascontiguousarray(dc, dtype=np.uint64)
        return self.lib.zo_dynamic_block_size(a.ctypes.data, b.ctypes.data, None, None)

    def optimize_rle(self, counts):
        c = np.array(counts, dtype=np.uint64)
        self.lib.zo_optimize_huffman_for_rle(len(c), c.ctypes.data)
        return c


_LEN_SYM = None


def histogram(litlens, dists):
    """288+32 histogram of an LZ77 symbol list (no end symbol)."""
    global _LEN_SYM
    if _LEN_SYM is None:
        t = np.zeros(259, dtype=np.int64)
        base = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115,
                131, 163, 195, 227, 258]
        for s, b in enumerate(base):
            t[b:] = 257 + s
        _LEN_SYM = t
    ll = np.asarray(litlens).astype(np.int64)
    dd = np.asarray(dists).astype(np.int64)
    lit = dd == 0
    llc = np.bincount(ll[lit], minlength=288)[:288].astype(np.uint64)
    llc += np.bincount(_LEN_SYM[ll[~lit]], minlength=288)[:288].astype(np.uint64)
    d = dd[~lit]
    ds = np.where(d < 5, d - 1, 0)
    big = d >= 5
    x = (d[big] - 1)
    l = np.floor(np.log2(x)).astype(np.int64)
    ds[big] = 2 * l + ((x >> (l - 1)) & 1)
    dc = np.bincount(ds, minlength=32)[:32].astype(np.uint64)
    return llc, dc


# ---- the reference's answers, recorded ----
# The reference cannot be built everywhere the tests run (its sources are not part of this repository), so every
# call the tests make to it is answered from tests/golden/reference_answers.json.  Small answers are stored as
# they are; bytes and arrays longer than VERBATIM by length and SHA-256.  Where the oracle restatement computes
# the same function, a digest-only answer is the oracle's value after checking it against the digest, so the
# tests can keep using reference parses as inputs.  To record (where oracle/_ref is built):
#   ZOPFLI_B200_RECORD_REFERENCE=tests/golden/reference_answers.json python -m pytest tests ...
ANSWERS = os.path.join(ROOT, "tests", "golden", "reference_answers.json")
VERBATIM = 64
ORACLE_EQUIVALENT = ("lz77", "match_table", "limited_match", "length_limited", "entropy", "optimize_rle")
REF_METHODS = ORACLE_EQUIVALENT + ("compress", "deflate_part", "block_size", "block_split_lz77", "block_split")


def _sha(b):
    return hashlib.sha256(b).hexdigest()


def encode(x, digest=False):
    """JSON form of a value: small bytes / arrays as they are (unless `digest`), larger ones by digest"""
    if isinstance(x, (bytes, bytearray, memoryview)):
        x = bytes(x)
        return {"hex": x.hex()} if len(x) <= VERBATIM and not digest else {"bytes": len(x), "sha256": _sha(x)}
    if isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        if a.size <= VERBATIM and not digest:
            return {"dtype": a.dtype.str, "shape": list(a.shape), "data": a.tolist()}
        return {"dtype": a.dtype.str, "shape": list(a.shape), "sha256": _sha(a.tobytes())}
    if isinstance(x, tuple):
        return {"tuple": [encode(v, digest) for v in x]}
    if isinstance(x, list):
        return [encode(v, digest) for v in x]
    if isinstance(x, dict):
        return {"kw": {k: encode(v, digest) for k, v in sorted(x.items())}}
    if isinstance(x, np.integer):
        return int(x)
    if isinstance(x, np.floating):
        return float(x)
    return x


def _list_digest(values):
    return {"items": len(values), "sha256": _sha(json.dumps(encode(values, True), sort_keys=True).encode())}


class Recorded:
    """An answer of the reference known by its digest: equal to any value with the same digest."""

    def __init__(self, rec):
        self.rec = rec

    def __eq__(self, other):
        if "items" in self.rec:
            return isinstance(other, list) and _list_digest(other) == self.rec
        return encode(other, True) == self.rec

    def __len__(self):
        return self.rec["items"] if "items" in self.rec else self.rec["bytes"]

    def __repr__(self):
        return "<reference answer %s>" % json.dumps(self.rec)


def _decode(rec, computed=None, what=""):
    if isinstance(rec, list):
        return [_decode(r, None if computed is None else c, what) for r, c in
                zip(rec, computed if computed is not None else [None] * len(rec))]
    if not isinstance(rec, dict):
        return rec
    if "tuple" in rec:
        cs = computed if computed is not None else [None] * len(rec["tuple"])
        return tuple(_decode(r, c, what) for r, c in zip(rec["tuple"], cs))
    if "hex" in rec:
        return bytes.fromhex(rec["hex"])
    if "data" in rec:
        return np.array(rec["data"], dtype=np.dtype(rec["dtype"])).reshape(rec["shape"])
    if computed is None:
        return Recorded(rec)
    assert encode(computed, True) == rec, "the oracle restatement's %s differs from the reference's" % what
    return computed


def _live_call(args):
    method, a, kw = args
    return getattr(Ref(), method)(*a, **kw)


class Reference:
    """The reference's answers with the methods of `Ref`: recorded ones by default, the live library while
    recording (ZOPFLI_B200_RECORD_REFERENCE=<file>: the answers file plus the new answers is written there)."""

    def __init__(self):
        self.out = os.environ.get("ZOPFLI_B200_RECORD_REFERENCE")
        self.live = Ref() if self.out else None
        self.table = json.load(open(ANSWERS)) if os.path.exists(ANSWERS) else {}
        self._oracle = None
        if self.out:
            if os.path.exists(self.out):   # successive recording processes add to one file
                self.table.update(json.load(open(self.out)))
            atexit.register(self.save)

    def save(self):
        with open(self.out, "w") as f:
            f.write("{\n" + ",\n".join(json.dumps(k) + ": " + json.dumps(self.table[k], sort_keys=True, separators=(",", ":"))
                                      for k in sorted(self.table)) + "\n}\n")

    @property
    def oracle(self):
        if self._oracle is None:
            self._oracle = Oracle()
        return self._oracle

    @staticmethod
    def _key(method, args, kw):
        return method + ":" + _sha(json.dumps(encode((args, kw), True), sort_keys=True).encode())[:32]

    def _lookup(self, key):
        assert key in self.table, "no recorded reference answer for %s: record it where oracle/_ref is built" % key
        return self.table[key]

    def call(self, method, *args, **kw):
        key = self._key(method, args, kw)
        if self.live is not None:
            value = getattr(self.live, method)(*args, **kw)
            self.table[key] = encode(value)
            return value
        rec = self._lookup(key)
        computed = getattr(self.oracle, method)(*args, **kw) if method in ORACLE_EQUIVALENT and \
            _needs_digest_check(rec) else None
        return _decode(rec, computed, method)

    def many(self, method, calls):
        """[method(*c) for c in calls], recorded as one digest"""
        key = self._key("many/" + method, calls, {})
        if self.live is not None:
            values = [getattr(self.live, method)(*c) for c in calls]
            self.table[key] = _list_digest(values)
            return values
        rec = self._lookup(key)
        if method not in ORACLE_EQUIVALENT:
            return Recorded(rec)
        values = [getattr(self.oracle, method)(*c) for c in calls]
        assert _list_digest(values) == rec, "the oracle restatement's %s differs from the reference's" % method
        return values

    def map(self, method, calls, **kw):
        """[method(*c, **kw) for c in calls]: while recording in a process pool (the children never touch CUDA)"""
        if self.live is None:
            return [self.call(method, *c, **kw) for c in calls]
        with mp.get_context("fork").Pool(min(8, max(1, len(calls)))) as pool:
            values = pool.map(_live_call, [(method, c, kw) for c in calls])
        for c, v in zip(calls, values):
            self.table[self._key(method, c, kw)] = encode(v)
        return values

    def answer(self, name, args, live, digest=False):
        """an answer that needs more than one call: live(ref) computes it from the `Ref` library"""
        key = self._key(name, args, {})
        if self.live is not None:
            value = live(self.live)
            self.table[key] = _list_digest(value) if digest else encode(value)
            return value
        return _decode(self._lookup(key))

    def __getattr__(self, method):
        if method not in REF_METHODS:
            raise AttributeError(method)
        return lambda *a, **kw: self.call(method, *a, **kw)


def _needs_digest_check(rec):
    if isinstance(rec, list):
        return any(_needs_digest_check(r) for r in rec)
    if isinstance(rec, dict):
        if "tuple" in rec:
            return any(_needs_digest_check(r) for r in rec["tuple"])
        return "sha256" in rec
    return False


_reference = None


def reference() -> Reference:
    global _reference
    if _reference is None:
        _reference = Reference()
    return _reference

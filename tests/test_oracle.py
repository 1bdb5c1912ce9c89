"""Pins the plain-C restatement (oracle/zopfli_oracle.c) against the UNMODIFIED reference compiled
from the original project (oracle/_ref; its recorded answers, tests/golden/reference_answers.json), at the seams of SURVEY.md section 4:
  seam 3: per-position ZopfliFindLongestMatch (length, dist, sublen[3..length]) + hash state
  seam 2: ZopfliLZ77Store out of ZopfliLZ77Greedy / ZopfliLZ77Optimal / ZopfliLZ77OptimalFixed
plus the integer helpers the iterate loop drags in (katajainen.c, tree.c, deflate.c estimators).
Bit-exact everywhere (integer/byte work; the fp64 entropy must match to the last bit too).
"""
import os

import numpy as np
import pytest

import zref
from zopfli_b200 import corpus

TXT = corpus.synth_text(300000, 2)
CASES = [
    ("text-head", TXT, 0, 20000),
    ("text-mid", TXT, 100000, 125000),            # 32 KiB history in play
    ("collide", corpus.adv_collide(), 40000, 52000),  # chain cap + hash collisions
    ("chain", corpus.adv_chain(), 30000, 42000),
    ("runs", corpus.adv_runs(), 0, 40000),        # chain-2 switch, long-run shortcut
    ("longrun", corpus.adv_longrun(), 0, 150000),  # `same` saturates at 65535
    ("longrun-cut", corpus.adv_longrun(), 1000, 68000),  # block boundary inside a byte run
    ("random", corpus.random_bytes(3000), 0, 3000),
    ("foobar", corpus.go_case_foobar(), 0, 7013),
    ("binary", corpus.synth_binary(200000), 60000, 100000),
    ("tiny3", b"abcabcabc", 0, 9),
    ("tiny1", b"a", 0, 1),
    ("tail-repeat", b"xyz" * 200 + b"aaaa", 100, 604),
]


@pytest.mark.parametrize("name,data,s,e", CASES, ids=[c[0] for c in CASES])
def test_match_table_seam(ref, oracle, name, data, s, e):
    e2 = min(e, s + 12000)  # python-side loop over positions; keep it quick
    a = ref.match_table(data, s, e2)
    b = oracle.match_table(data, s, e2)
    for x, y, what in zip(a, b, ("length", "dist", "sublen", "same", "hv", "hv2")):
        if len(data) < 2 and what in ("hv", "hv2"):
            continue  # hash.c:139-143 warms up one byte fewer for a 1-byte range; key never used
        assert np.array_equal(x, y), what


@pytest.mark.parametrize("name,data,s,e", CASES[:6], ids=[c[0] for c in CASES[:6]])
def test_limited_walk_is_table_lookup(ref, oracle, name, data, s, e):
    """SURVEY App. A.3: FindLongestMatch(limit=L, sublen=NULL) == (L, sublen_full[L])."""
    e2 = min(e, s + 6000)
    ln, ds, sub, *_ = ref.match_table(data, s, e2)
    rng = np.random.default_rng(5)
    limits = np.where(ln >= 3, rng.integers(3, 259, len(ln)), 0)
    limits = np.minimum(limits, ln).astype(np.uint16)
    limits[limits < 3] = 0
    rl, rd = ref.limited_match(data, s, e2, limits)
    ol, od = oracle.limited_match(data, s, e2, limits)
    assert np.array_equal(rl, ol) and np.array_equal(rd, od)
    j = np.nonzero(limits >= 3)[0]
    assert np.array_equal(rl[j], limits[j])
    assert np.array_equal(rd[j], sub[j, limits[j]])


@pytest.mark.parametrize("name,data,s,e", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("mode,iters", [(2, 0), (3, 0), (1, 0), (0, 1), (0, 15)])
def test_store_seam(ref, oracle, name, data, s, e, mode, iters):
    a = ref.lz77(data, s, e, mode, iters)
    b = oracle.lz77(data, s, e, mode, iters)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    if s == 0 and len(a[0]):
        llc, dc = zref.histogram(*a)
        assert ref.block_size(data, a[0], a[1], 0, len(a[0]), 2) == oracle.dynamic_block_size(llc, dc)


def test_store_seam_50_iterations(ref, oracle):
    """randomisation + blended statistics active (squeeze.c:505-517)."""
    a = ref.lz77(TXT, 0, 40000, 0, 50)
    b = oracle.lz77(TXT, 0, 40000, 0, 50)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_length_limited_code_lengths(ref, oracle):
    rng = np.random.default_rng(0)
    calls = []
    for t in range(1500):
        n = int(rng.choice([19, 32, 288]))
        mb = 7 if n == 19 else 15
        k = int(rng.integers(0, n + 1))
        f = np.zeros(n, dtype=np.uint64)
        idx = rng.choice(n, k, replace=False)
        m = t % 5
        if m == 0:
            f[idx] = rng.integers(1, 4, k)
        elif m == 1:
            f[idx] = rng.integers(1, 100000, k)
        elif m == 2:
            f[idx] = (2 ** rng.integers(0, 18, k)).astype(np.uint64)
        elif m == 3:
            f[idx] = np.sort(rng.integers(1, 50, k))
        else:  # forces the 15-bit limit with many ties
            f[idx] = (1.5 ** rng.integers(0, 34, k)).astype(np.uint64) + rng.integers(0, 2, k).astype(np.uint64)
        calls.append((f, mb))
    for (f, mb), (e1, a) in zip(calls, ref.many("length_limited", calls)):
        e2, b = oracle.length_limited(f, mb)
        assert e1 == e2 and np.array_equal(a, b)


def test_entropy_and_rle(ref, oracle):
    rng = np.random.default_rng(1)
    calls = []
    for t in range(200):
        c = rng.integers(0, 5000, 288).astype(np.uint64)
        c[rng.random(288) < 0.3] = 0
        calls.append((c,))
    calls.append((np.zeros(32),))
    for (c,), want in zip(calls, ref.many("entropy", calls)):
        assert np.array_equal(want, oracle.entropy(c))
    calls = []
    for t in range(400):
        n = int(rng.choice([32, 288]))
        c = rng.integers(0, 30, n).astype(np.uint64)
        c[rng.random(n) < 0.4] = 0
        if t % 3 == 0:
            c = np.repeat(rng.integers(0, 9, n // 8 + 1), 8)[:n].astype(np.uint64)
        calls.append((c,))
    for (c,), want in zip(calls, ref.many("optimize_rle", calls)):
        assert np.array_equal(want, oracle.optimize_rle(c))


# ---- the integer formulation of the forward DP (k_iterate's "integer window", iterate.cuh) ----
# oracle/dp_int_model.c runs a sequential model of it next to the oracle's reference DP on every pass of
# ZopfliLZ77Optimal / OptimalFixed and counts positions whose cost or length_array entry differs.
INT_DP_CASES = [
    ("text", TXT, 32768, 300000, 5),
    ("text-fixed", TXT, 32768, 300000, 0),
    ("binary", corpus.synth_binary(300000, 4), 0, 300000, 8),
    ("binary-fixed", corpus.synth_binary(300000, 4), 0, 300000, 0),
    ("collide", corpus.adv_collide(), 0, len(corpus.adv_collide()), 4),
    ("runs", corpus.adv_runs(), 0, len(corpus.adv_runs()), 4),
    ("longrun-cut", corpus.adv_longrun(), 1000, 68000, 3),
    ("random", corpus.random_bytes(200000), 0, 200000, 3),
]


@pytest.mark.parametrize("name,data,s,e,iters", INT_DP_CASES, ids=[c[0] for c in INT_DP_CASES])
def test_integer_dp_model_equals_reference_dp(name, data, s, e, iters):
    import ctypes as C
    zref.ensure_built()
    path = os.path.join(zref.ORACLE_DIR, "_build", "libdp_int_model.so")
    if not os.path.exists(path):
        import subprocess
        subprocess.check_call(["make", "-s", "-C", zref.ORACLE_DIR, "oracle"])
    lib = C.CDLL(path)
    lib.zo_dp_int_check.restype = C.c_uint64
    lib.zo_dp_int_check.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p]
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    out = np.zeros(8, dtype=np.uint64)
    mism = lib.zo_dp_int_check(buf.ctypes.data, s, e, iters, out.ctypes.data)
    steps_total, steps_int = int(out[0]), int(out[1])
    assert mism == 0
    assert steps_total > 0
    if name in ("text", "random"):
        assert steps_int > 0.8 * steps_total   # the model really ran in the integer representation


@pytest.mark.slow
def test_integer_dp_model_on_the_bench_giant_master_block():
    """master block 85 of the C2 bench text holds the 969,128-position block (costs beyond 2^21, float ulp 0.25):
    15 DP passes of the model against the reference arithmetic, one block (no splitting)"""
    import ctypes as C
    zref.ensure_built()
    lib = C.CDLL(os.path.join(zref.ORACLE_DIR, "_build", "libdp_int_model.so"))
    lib.zo_dp_int_check.restype = C.c_uint64
    lib.zo_dp_int_check.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p]
    text = corpus.synth_text(86_000_000, 2)      # a prefix of the bench text (the generator is prefix-stable)
    a = 85 * 1_000_000
    buf = np.frombuffer(text[a - 32768:a + 1_000_000], dtype=np.uint8).copy()
    out = np.zeros(8, dtype=np.uint64)
    assert lib.zo_dp_int_check(buf.ctypes.data, 32768, 32768 + 1_000_000, 15, out.ctypes.data) == 0
    assert int(out[1]) > 0.95 * int(out[0])

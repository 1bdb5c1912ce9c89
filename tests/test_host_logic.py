"""Host-side logic of the product (block splitter, size estimators, emitter, containers, splice,
span sharding) against the UNMODIFIED reference's recorded answers -- runs without a GPU.

End-to-end cases link the PRODUCT's host sources against a mock engine that answers LZ77 parse
requests with the oracle (tests/hostmock/): whatever differs from the reference here is a host
bug, not a kernel bug.  The shipped libzopfli.so.1 contains no such path.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import zopfli_b200 as zb
import zref
from zopfli_b200 import corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TXT = corpus.synth_text(2200000, 2)


@pytest.fixture(scope="module")
def mock():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "hostmock")])
    return zb.Library(os.path.join(ROOT, "tests", "_build", "libzopfli_hostmock.so"))


@pytest.fixture(scope="module")
def host():
    """the real product library; only its GPU-free host seams are used in this file"""
    if not os.path.exists(zb.LIB_PATH):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "zopfli_b200", "csrc")])
    return zb.Library()


def test_library_exports_every_declared_symbol(host):
    import ctypes
    import re
    names = set()
    for h in ("zopfli.h", "zopfli_b200.h"):
        src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", h)).read(), flags=re.S)
        names |= set(re.findall(r"\b(Zopfli[A-Za-z0-9]+)\s*\(", src))
    assert names >= set(zb.EXPORTS)
    for n in sorted(names):
        assert hasattr(host.lib, n), n
    o = zb.ZopfliOptions()
    host.lib.ZopfliInitOptions(ctypes.byref(o))  # util.c:28-35
    assert (o.verbose, o.verbose_more, o.numiterations, o.blocksplitting, o.blocksplittinglast,
            o.blocksplittingmax) == (0, 0, 15, 1, 0, 15)
    assert ctypes.sizeof(zb.ZopfliOptions) == 24


def test_length_limited_host(ref, host):
    rng = np.random.default_rng(0)
    calls = []
    for t in range(600):
        n = int(rng.choice([19, 32, 288]))
        mb = 7 if n == 19 else 15
        f = np.zeros(n, np.uint32)
        k = int(rng.integers(0, n + 1))
        idx = rng.choice(n, k, replace=False)
        if t % 2:
            f[idx] = (1.5 ** rng.integers(0, 30, k)).astype(np.uint32) + rng.integers(0, 2, k).astype(np.uint32)
        else:
            f[idx] = rng.integers(1, 9, k)
        calls.append((f.astype(np.uint64), mb))
    for (f, mb), want in zip(calls, ref.many("length_limited", calls)):
        assert np.array_equal(want[1], host.host_length_limited(f.astype(np.uint32), mb)[1])


def test_split_and_block_sizes(ref, host):
    rng = np.random.default_rng(1)
    for data, s, e in [(TXT, 0, 1000000), (corpus.synth_binary(400000), 0, 400000), (corpus.adv_runs(), 0, 200000)]:
        ll, dd = ref.lz77(data, s, e, 3)
        for maxblocks in (15, 4, 0):
            assert np.array_equal(ref.block_split_lz77(data, ll, dd, maxblocks), host.host_block_split_lz77(ll, dd, maxblocks))
        calls = []
        for t in range(40):
            a = int(rng.integers(0, len(ll) - 1))
            b = int(rng.integers(a + 1, min(len(ll), a + 1 + int(rng.choice([50, 900, 5000, 100000]))) + 1))
            calls += [(data, ll, dd, a, b, bt) for bt in (0, 1, 2, -1)]
        assert [host.host_block_size(*c[1:]) for c in calls] == ref.many("block_size", calls)
    # small store: the `lz77->size > 1000` quirk of deflate.c:615 goes the other way
    ll, dd = ref.lz77(TXT, 2000, 3200, 3)
    assert len(ll) < 1000
    for a, b in [(0, len(ll)), (10, 200), (5, 6)]:
        assert ref.block_size(TXT, ll, dd, a, b, -1) == host.host_block_size(ll, dd, a, b, -1)


def test_emit_dynamic_block_matches_reference_stream(ref, host):
    """single block, no splitting: the reference's whole output is one AddLZ77Block call"""
    data = TXT[:30000]
    ll, dd = ref.lz77(data, 0, len(data), 0, 15)
    want, bp = ref.deflate_part(data, 0, len(data), final=1, blocksplitting=0)
    got, bits = host.host_emit_block(ll, dd, 0, len(ll), 2, 1)
    assert got == want and bits % 8 == bp


END_TO_END = [
    ("empty", b""), ("a", b"a"), ("ab", b"ab"), ("abc", b"abc"), ("foobar", corpus.go_case_foobar()),
    ("rand3000", corpus.random_bytes(3000)), ("text40k", TXT[:40000]), ("runs", corpus.adv_runs()[:60000]),
    ("mixed", corpus.mixed_small(50000)), ("zeros", b"\0" * 70000), ("rand70k", corpus.random_bytes(70000)),
    ("binary", corpus.synth_binary(120000)), ("len258", b"q" * 258), ("len259", b"q" * 259),
]


@pytest.mark.parametrize("name,data", END_TO_END, ids=[c[0] for c in END_TO_END])
def test_compress_all_formats(ref, mock, name, data):
    for fmt in (0, 1, 2):
        assert ref.compress(data, fmt) == mock.compress(data, fmt), fmt


def test_known_answers(mock):
    """oracle known answers recorded in SURVEY App. C"""
    assert mock.compress(b"", 0).hex() == "1f8b08000000000002030300" + "0000000000000000"
    assert mock.compress(b"", 1).hex() == "78da030000000001"
    assert mock.compress(b"", 2).hex() == "0300"
    assert mock.compress(b"a", 2).hex() == "4b0400"
    assert mock.compress(b"a", 1).hex() == "78da4b040000620062"
    assert mock.compress(b"a", 0).hex() == "1f8b08000000000002034b040043beb7e801000000"


def test_options_and_btypes(ref, mock):
    data = TXT[:60000]
    for kw in ({"numiterations": 1}, {"numiterations": 5, "blocksplittingmax": 3}, {"blocksplitting": 0},
               {"blocksplittingmax": 0, "numiterations": 2}):
        assert ref.compress(data, 2, **kw) == mock.compress(data, 2, **kw), kw
    for btype in (0, 1, 2):
        for final in (0, 1):
            a, abp = ref.deflate_part(data, 0, len(data), final=final, btype=btype, numiterations=3)
            b, bbp = mock.deflate_part(data, 0, len(data), final=final, btype=btype, numiterations=3)
            assert a == b and abp == bbp, (btype, final)
    big = corpus.random_bytes(140000)  # stored blocks split at 65535
    assert ref.deflate_part(big, 0, len(big), btype=0) == mock.deflate_part(big, 0, len(big), btype=0)


def chained_deflate_parts(lib, data, numiterations, parts):
    """ZopfliDeflatePart calls (btype, final, start, end) sharing one output buffer and bit pointer (deflate.h:50-53)"""
    import ctypes as C
    arr = np.frombuffer(data + b"\0" * 16, np.uint8)
    o = zb.ZopfliOptions(0, 0, numiterations, 1, 0, 15)
    out, n, bp = C.c_void_p(None), C.c_size_t(0), C.c_ubyte(0)
    for btype, final, s, e in parts:
        lib.ZopfliDeflatePart(C.byref(o), btype, final, arr.ctypes.data, s, e, C.byref(bp), C.byref(out), C.byref(n))
    return C.string_at(out, n.value), bp.value


def test_deflate_part_with_dictionary_and_chained_bp(ref, mock):
    data = TXT[:150000]
    a, abp = ref.deflate_part(data, 50000, 110000, final=1, numiterations=2)
    b, bbp = mock.deflate_part(data, 50000, 110000, final=1, numiterations=2)
    assert a == b and abp == bbp
    parts = [(2, 0, 0, 70000), (2, 1, 70000, 150000)]
    got = chained_deflate_parts(mock.lib, data, 2, parts)
    assert got == ref.answer("chained_deflate_parts", (data, 2, parts), lambda r: chained_deflate_parts(r.lib, data, 2, parts))
    import zlib
    assert zlib.decompress(got[0], -15) == data


def test_multi_master_block_and_spans(ref, mock):
    data = TXT  # 2.2 MB: three master blocks, last one partial
    want = ref.compress(data, 2, numiterations=1)
    assert mock.compress(data, 2, numiterations=1) == want
    # SURVEY 8(e): per-shard spans spliced by a bit-offset scan equal the single-call stream
    spans = [mock.deflate_span(data, m, m + 1, final=int(m == 2), numiterations=1) for m in range(3)]
    got, bp = mock.splice_spans(spans)
    assert got == want
    # stored blocks inside spans (random data -> stored), with a non-zero bit offset before them
    mix = TXT[:1000000] + corpus.random_bytes(300000)
    want = ref.compress(mix, 2, numiterations=1)
    spans = [mock.deflate_span(mix, m, m + 1, final=int(m == 1), numiterations=1) for m in range(2)]
    assert mock.splice_spans(spans)[0] == want


def test_two_lane_finalisation_order(ref, mock, monkeypatch):
    """Master blocks without a "giant" block are finalised while the giants' lane is still busy
    (driver.cpp stage C); the stream must not depend on which master block finishes first."""
    data = TXT
    want = ref.compress(data, 2, numiterations=1)
    for giant in (20000, 60000, 150000):   # different clean/dirty partitions of the master blocks
        monkeypatch.setenv("ZOPFLI_B200_GIANT", str(giant))
        assert mock.compress(data, 2, numiterations=1) == want, giant


def test_chunk_pipelines(ref, mock, monkeypatch):
    """Master blocks run as independent chunk pipelines on separate engine lanes and host threads
    (driver.cpp run_chunk); the output is the master blocks' pieces in order, whatever the chunking."""
    data = TXT + corpus.synth_binary(900000, 3)   # 4 master blocks
    want = ref.compress(data, 2, numiterations=1)
    for chunks in (1, 3, 4):
        monkeypatch.setenv("ZOPFLI_B200_FORCE_CHUNKS", str(chunks))
        monkeypatch.setenv("ZOPFLI_B200_GIANT", "60000")
        assert mock.compress(data, 2, numiterations=1) == want, chunks
    # a pipeline takes its master blocks in batches (bounded device memory on GiB inputs)
    monkeypatch.setenv("ZOPFLI_B200_FORCE_CHUNKS", "2")
    monkeypatch.setenv("ZOPFLI_B200_BATCH", "1")
    assert mock.compress(data, 2, numiterations=1) == want


def test_splice_many_small_parts_all_bit_phases(ref, mock):
    """Chains of tiny ZopfliDeflatePart calls (btype 0/1/2, sizes 0..70) into one buffer: every bit
    phase, pieces shorter than a byte, stored blocks right after partial bytes (driver.cpp splice)."""
    import zlib
    rng = np.random.default_rng(11)
    base = (TXT[:3000] + corpus.random_bytes(800) + b"a" * 300 + TXT[5000:7000])
    cuts = [0]
    while cuts[-1] < len(base):
        cuts.append(min(len(base), cuts[-1] + int(rng.integers(0, 70))))
    types = rng.integers(0, 3, len(cuts) - 1)
    parts = [(int(types[i]), int(i == len(cuts) - 2), cuts[i], cuts[i + 1]) for i in range(len(cuts) - 1)]
    got = chained_deflate_parts(mock.lib, base, 1, parts)
    assert got == ref.answer("chained_deflate_parts", (base, 1, parts), lambda r: chained_deflate_parts(r.lib, base, 1, parts))
    assert zlib.decompress(got[0], -15) == base


def test_nocopy_result_wrapper(mock):
    """compress_ptr_nocopy hands out the library's malloc()ed buffer itself; same bytes, explicit free."""
    data = TXT[:60000]
    a = np.frombuffer(data + b"\0" * 16, np.uint8)
    want = mock.compress(data, zb.ZOPFLI_FORMAT_ZLIB, numiterations=1)
    ob = mock.compress_ptr_nocopy(a.ctypes.data, len(data), zb.ZOPFLI_FORMAT_ZLIB, numiterations=1)
    assert len(ob) == len(want) and ob.tobytes() == want and bytes(ob.view[:16]) == want[:16]
    ob.close()
    ob.close()  # idempotent


@pytest.mark.parametrize("budget", [0, 200, 3000, 100000])
def test_batched_split_scheduler_matches_reference(ref, host, budget):
    """batched_split.hpp (speculative FindMinimum for every block, lockstep rounds, one to three
    levels of the nine-point recursion per round depending on `budget`) returns the reference's
    ZopfliBlockSplitLZ77 points (blocksplitter.c:215-273) for several stores at once."""
    rng = np.random.default_rng(5)
    stores = []
    datas = [TXT[:400000], corpus.synth_binary(300000, 7), corpus.mixed_small(90000), TXT[900000:960000],
             corpus.adv_runs()[:120000], TXT[1000000:1000500]]
    for d in datas:
        ll, dd = ref.lz77(d, 0, len(d), 0, 1)   # greedy store
        stores.append((d, ll, dd))
    for maxblocks in (15, 4, 0):
        got = host.host_batched_split([(ll, dd) for _, ll, dd in stores], maxblocks=maxblocks, budget=budget)
        for (d, ll, dd), g in zip(stores, got):
            want = ref.block_split_lz77(d, ll, dd, maxblocks=maxblocks)
            assert np.array_equal(g, want), (len(d), maxblocks, budget)


class Store(ctypes.Structure):  # lz77.h:44-62
    _fields_ = [("litlens", ctypes.POINTER(ctypes.c_ushort)), ("dists", ctypes.POINTER(ctypes.c_ushort)),
                ("size", ctypes.c_size_t), ("data", ctypes.c_void_p), ("pos", ctypes.c_void_p),
                ("ll_symbol", ctypes.c_void_p), ("d_symbol", ctypes.c_void_p), ("ll_counts", ctypes.c_void_p),
                ("d_counts", ctypes.c_void_p)]


def _entry_point_sizes(lib, st, ranges):
    """ZopfliCalculateBlockSize for btype 0, 1, 2 and ...AutoType of each range of the store `st`"""
    C = ctypes
    for f in (lib.ZopfliCalculateBlockSize, lib.ZopfliCalculateBlockSizeAutoType):
        f.restype = C.c_double
    lib.ZopfliCalculateBlockSize.argtypes = [C.POINTER(Store), C.c_size_t, C.c_size_t, C.c_int]
    lib.ZopfliCalculateBlockSizeAutoType.argtypes = [C.POINTER(Store), C.c_size_t, C.c_size_t]
    return [x for a, b in ranges for x in [lib.ZopfliCalculateBlockSize(C.byref(st), a, b, btype) for btype in (0, 1, 2)] +
            [lib.ZopfliCalculateBlockSizeAutoType(C.byref(st), a, b)]]


def _reference_store_sizes(r, data, ranges):
    """a store BUILT BY THE REFERENCE (ZopfliLZ77Greedy) priced by the reference"""
    C = ctypes

    class BlockState(C.Structure):  # lz77.h:86-97
        _fields_ = [("options", C.c_void_p), ("lmc", C.c_void_p), ("blockstart", C.c_size_t), ("blockend", C.c_size_t)]

    arr = np.frombuffer(data + b"\0" * 16, np.uint8)
    o = zb.ZopfliOptions(0, 0, 1, 1, 0, 15)
    st, bs = Store(), BlockState()
    r.lib.ZopfliInitLZ77Store(C.c_void_p(arr.ctypes.data), C.byref(st))
    r.lib.ZopfliInitBlockState(C.byref(o), C.c_size_t(0), C.c_size_t(len(data)), 0, C.byref(bs))
    r.lib.ZopfliAllocHash.restype = None
    hbuf = C.create_string_buffer(256)  # ZopfliHash (hash.h:29-47): a few pointers and ints
    r.lib.ZopfliAllocHash(C.c_size_t(32768), hbuf)
    r.lib.ZopfliLZ77Greedy(C.byref(bs), C.c_void_p(arr.ctypes.data), C.c_size_t(0), C.c_size_t(len(data)), C.byref(st), hbuf)
    assert st.size == ranges[0][1]
    sizes = _entry_point_sizes(r.lib, st, ranges)
    r.lib.ZopfliCleanHash(hbuf)
    r.lib.ZopfliCleanBlockState(C.byref(bs))
    r.lib.ZopfliCleanLZ77Store(C.byref(st))
    return sizes


def test_deflate_h_block_size_entry_points(ref, host):
    """ZopfliCalculateBlockSize / ...AutoType (deflate.h:79-86) take the reference's own ZopfliLZ77Store: the
    reference's greedy parse in the reference's store layout is priced as the reference prices the store it
    builds itself."""
    C = ctypes
    for data in (TXT[:90000], corpus.random_bytes(5000), TXT[:700], corpus.adv_runs()[:50000]):
        arr = np.frombuffer(data + b"\0" * 16, np.uint8)
        ll, dd = ref.lz77(data, 0, len(data), 2, 0)   # ZopfliLZ77Greedy
        n = len(ll)
        assert n > 0
        st = Store(ll.ctypes.data_as(C.POINTER(C.c_ushort)), dd.ctypes.data_as(C.POINTER(C.c_ushort)), n, arr.ctypes.data)
        rng = np.random.default_rng(n)
        ranges = [(0, n), (0, 0), (n // 3, n // 3 + 1), (n // 4, 3 * n // 4)] + \
                 [tuple(int(x) for x in sorted(rng.integers(0, n + 1, 2))) for _ in range(12)]
        want = ref.answer("reference_store_sizes", (data, ranges), lambda r: _reference_store_sizes(r, data, ranges),
                          digest=True)
        assert _entry_point_sizes(host.lib, st, ranges) == want, len(data)


def test_concurrent_calls_and_span_validation(ref, mock):
    """API-level state (engine lease, layout / timing globals, lazy CRC table) under concurrent callers,
    and ZopfliB200AppendSpan's rejection of truncated spans."""
    import threading
    inputs = [corpus.synth_text(60000, 21), corpus.synth_binary(50000), corpus.adv_runs()[:40000], b"", b"abc" * 3000,
              corpus.mixed_small(30000)]
    want = [ref.compress(d, i % 3, numiterations=2) for i, d in enumerate(inputs)]
    got = [None] * len(inputs)

    def work(i):
        got[i] = mock.compress(inputs[i], i % 3, numiterations=2)

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(inputs))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert got == want
    span = mock.deflate_span(inputs[0], 0, 1, final=1, numiterations=1)
    assert mock.splice_spans([span])[0] == ref.compress(inputs[0], 2, numiterations=1)
    for cut in (1, 9, len(span) - 1):
        with pytest.raises(ValueError):
            mock.splice_spans([span[:cut]])
    offs = mock.last_master_bit_offsets()
    assert len(offs) >= 2 and offs[0] == 0


def test_optimize_for_rle_restatement(ref, host):
    """The run-segmentation form of OptimizeHuffmanForRle (deflate_size.hpp) against the reference's
    scan (deflate.c:434-518) on histograms with plateaus, zero gaps and near-equal neighbours."""
    rng = np.random.default_rng(5)
    calls = []
    for t in range(3000):
        n = int(rng.choice([32, 288, 30, 19, 7, 1]))
        kind = t % 5
        if kind == 0:
            c = rng.integers(0, 6, n)
        elif kind == 1:
            c = np.repeat(rng.integers(0, 40, n), rng.integers(1, 9, n))[:n]
        elif kind == 2:
            c = (rng.integers(0, 3, n) == 0) * rng.integers(0, 2000, n)
        elif kind == 3:
            c = np.cumsum(rng.integers(-2, 3, n)).clip(0)
        else:
            c = rng.integers(0, 1 << int(rng.integers(1, 20)), n)
        c = np.asarray(c, np.uint32)
        if len(c) < n:
            c = np.pad(c, (0, n - len(c)))
        calls.append((c,))
    for t, ((c,), want) in enumerate(zip(calls, ref.many("optimize_rle", calls))):
        assert np.array_equal(want, host.host_optimize_rle(c)), (t, c.tolist())


def test_checksums_threaded_and_combined(mock):
    """CRC-32 / Adler-32 of the container trailers (gzip_container.c:27-81, zlib_container.c:29-48): the
    threaded versions with their exact combination rules against zlib, across the threading threshold."""
    import zlib
    rng = np.random.default_rng(8)
    for n in (0, 1, 5551, 5553, 70000, (4 << 20) - 1, (4 << 20) + 12345, 9000001):
        d = rng.integers(0, 256, n, dtype=np.uint8).tobytes() if n % 2 else bytes([255]) * n
        assert mock.adler32(d) == zlib.adler32(d), n
        a = np.frombuffer(d, np.uint8)
        assert mock.crc32(a.ctypes.data if n else 0, n) == zlib.crc32(d), n


def test_verbose_reports_match_the_reference(ref, tmp_path):
    """options.verbose: the split-point, tree-size and block-size reports (blocksplitter.c:148-180,
    deflate.c:718-744) come out byte for byte as the reference prints them; only the per-iteration lines
    of squeeze.c:493-495 are not mirrored (they would need every iteration's cost back from the device)."""
    script = tmp_path / "verb.py"
    script.write_text('''
import sys, ctypes as C, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import zopfli_b200 as zb, zref
from zopfli_b200 import corpus
d = corpus.synth_text(300000, 3) + corpus.random_bytes(40000) + corpus.synth_text(100000, 4)
if sys.argv[1] == "ref":
    r = zref.Ref(); o = r.options(numiterations=2); o.verbose = 1
    a = np.frombuffer(d, np.uint8); out = C.c_void_p(None); n = C.c_size_t(0)
    r.lib.ZopfliCompress(C.byref(o), 2, a.ctypes.data, len(d), C.byref(out), C.byref(n))
else:
    zb.Library(%r).compress(d, 2, numiterations=2, verbose=1)
''' % (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "_build", "libzopfli_hostmock.so")))

    def run(which):
        r = subprocess.run([sys.executable, str(script), which], capture_output=True, text=True, check=True)
        return [l for l in r.stderr.splitlines() if not l.startswith("Iteration")]
    want = ref.answer("verbose_stderr", ("synth_text(300000, 3) + random_bytes(40000) + synth_text(100000, 4)", 2),
                      lambda r: run("ref"))
    assert run("mock") == want and len(want) > 10

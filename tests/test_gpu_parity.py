"""Parity of the sm_100a path (through the C ABI of libzopfli.so.1) against the UNMODIFIED
reference's recorded answers (tests/golden/reference_answers.json), at the three seams of SURVEY.md section 4.  Integer / byte work: bit-exact, zero tolerance.
"""
import zlib

import numpy as np
import pytest

import zopfli_b200 as zb
import zref
from zopfli_b200 import corpus

pytestmark = pytest.mark.gpu

TXT = corpus.synth_text(2300000, 2)
SEAM_CASES = [
    ("text-head", TXT, 0, 20000),
    ("text-mid", TXT, 100000, 125000),
    ("collide", corpus.adv_collide(), 40000, 52000),
    ("chain", corpus.adv_chain(), 30000, 42000),
    ("runs", corpus.adv_runs(), 0, 40000),
    ("longrun", corpus.adv_longrun(), 0, 150000),
    ("longrun-cut", corpus.adv_longrun(), 1000, 68000),
    ("random", corpus.random_bytes(3000), 0, 3000),
    ("foobar", corpus.go_case_foobar(), 0, 7013),
    ("binary", corpus.synth_binary(200000), 60000, 100000),
    ("tiny3", b"abcabcabc", 0, 9),
    ("tiny1", b"a", 0, 1),
    ("tail-repeat", b"xyz" * 200 + b"aaaa", 100, 604),
]


@pytest.fixture(scope="module")
def lib():
    return zb.library()


@pytest.mark.parametrize("name,data,s,e", SEAM_CASES, ids=[c[0] for c in SEAM_CASES])
def test_match_table_seam(ref, lib, name, data, s, e):
    """seam 3: ZopfliFindLongestMatch per position incl. sublen and the hash state"""
    a = ref.match_table(data, s, e)
    b = lib.match_table(data, s, e)
    for x, y, what in zip(a, b, ("length", "dist", "sublen", "same", "hv", "hv2")):
        if what == "length":  # lengths below 3 mean "no match" either way (lz77.c:399-400)
            assert np.array_equal(np.where(x < 3, 0, x), np.where(y < 3, 0, y)), what
        elif what == "dist":
            m = a[0] >= 3
            assert np.array_equal(x[m], y[m]), what
        elif len(data) >= 3 or what not in ("hv", "hv2"):
            assert np.array_equal(x, y), what


@pytest.mark.parametrize("name,data,s,e", SEAM_CASES, ids=[c[0] for c in SEAM_CASES])
@pytest.mark.parametrize("mode,iters", [(2, 0), (1, 0), (0, 1), (0, 15)])
def test_store_seam(ref, lib, name, data, s, e, mode, iters):
    """seam 2: ZopfliLZ77Store out of Greedy / OptimalFixed / Optimal"""
    a = ref.lz77(data, s, e, mode, iters)
    b = lib.lz77(data, s, e, mode, iters)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_store_seam_50_iterations_and_batch(ref, lib):
    a = ref.lz77(TXT, 0, 40000, 0, 50)   # randomisation + blended statistics (squeeze.c:505-517)
    b = lib.lz77(TXT, 0, 40000, 0, 50)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    ranges = [(0, 30000), (30000, 31000), (31000, 90000), (90000, 90000), (90000, 140000)]
    res, cost = lib.lz77_batch(TXT, ranges, 0, 5)
    for (s, e), (ll, dd), c in zip(ranges, res, cost):
        r = ref.lz77(TXT, s, e, 0, 5)
        assert np.array_equal(r[0], ll) and np.array_equal(r[1], dd)
        if e > s:  # the device's per-iteration block size is exact (squeeze.c:492)
            llc, dc = zref.histogram(ll, dd)
            h = np.concatenate([llc, dc]).astype(np.uint32)
            assert lib.dynamic_block_bits(h, device=False) == int(c)
            assert ref.block_size(TXT[s:e], ll, dd, 0, len(ll), 2) == float(c)


def test_device_block_bits(lib):
    rng = np.random.default_rng(3)
    for t in range(40):
        h = np.zeros(320, np.uint32)
        k = int(rng.integers(1, 288))
        h[rng.choice(286, k, replace=False)] = (1.4 ** rng.integers(0, 30, k)).astype(np.uint32) + 1
        kd = int(rng.integers(0, 30))
        h[288 + rng.choice(30, kd, replace=False)] = rng.integers(1, 3000, kd)
        assert lib.dynamic_block_bits(h, device=True) == lib.dynamic_block_bits(h, device=False)


END_TO_END = [
    ("empty", b""), ("a", b"a"), ("ab", b"ab"), ("abc", b"abc"), ("foobar", corpus.go_case_foobar()),
    ("rand3000", corpus.random_bytes(3000)), ("text40k", TXT[:40000]), ("runs", corpus.adv_runs()),
    ("collide", corpus.adv_collide()), ("chain", corpus.adv_chain()), ("longrun", corpus.adv_longrun()),
    ("mixed", corpus.mixed_small(50000)), ("zeros", b"\0" * 70000), ("rand70k", corpus.random_bytes(70000)),
    ("binary", corpus.synth_binary(300000)), ("len258", b"q" * 258), ("len259", b"q" * 259),
    ("32767", TXT[:32767]), ("32768", TXT[:32768]), ("32769", TXT[:32769]),
]


@pytest.mark.parametrize("name,data", END_TO_END, ids=[c[0] for c in END_TO_END])
def test_compress_all_formats(ref, lib, name, data):
    """seam 1: final bytes of ZopfliCompress for gzip / zlib / raw deflate"""
    for fmt in (0, 1, 2):
        got = lib.compress(data, fmt)
        assert got == ref.compress(data, fmt), fmt
    assert zlib.decompress(lib.compress(data, 1)) == data


def test_master_block_boundaries(ref, lib):
    for n in (999999, 1000000, 1000001, 2000000, 2300000):
        data = TXT[:n]
        got = lib.compress(data, 2, numiterations=2)
        assert got == ref.compress(data, 2, numiterations=2), n
        assert zlib.decompress(got, -15) == data


def test_options_btypes_and_parts(ref, lib):
    data = TXT[:150000]
    for kw in ({"numiterations": 1}, {"numiterations": 5, "blocksplittingmax": 3}, {"blocksplitting": 0},
               {"blocksplittingmax": 0, "numiterations": 2}):
        assert ref.compress(data, 2, **kw) == lib.compress(data, 2, **kw), kw
    for btype in (0, 1, 2):
        a = ref.deflate_part(data, 0, 60000, final=1, btype=btype, numiterations=3)
        b = lib.deflate_part(data, 0, 60000, final=1, btype=btype, numiterations=3)
        assert a == b, btype
    a = ref.deflate_part(data, 50000, 110000, final=1, numiterations=2)
    b = lib.deflate_part(data, 50000, 110000, final=1, numiterations=2)
    assert a == b


def test_spans_splice_to_single_stream(ref, lib):
    data = TXT[:2300000]
    want = ref.compress(data, 2, numiterations=1)
    spans = [lib.deflate_span(data, m, m + 1, final=int(m == 2), numiterations=1) for m in range(3)]
    assert lib.splice_spans(spans)[0] == want


def test_full_size_properties(lib):
    """BASELINE-sized behaviour through size-independent properties: the stream inflates back to
    the input, and per-master-block spans splice to the same bytes as the one-shot call."""
    data = corpus.synth_text(8000000, 7)
    z = lib.compress(data, 2)
    assert zlib.decompress(z, -15) == data
    spans = [lib.deflate_span(data, m, min(m + 3, 8), final=int(m + 3 >= 8)) for m in range(0, 8, 3)]
    assert lib.splice_spans(spans)[0] == z


def test_nocopy_result_and_device_input(ref, lib):
    """compress_ptr_nocopy (the malloc()ed result itself) with a device-resident input copy."""
    import torch
    data = TXT[:1200000]
    host = torch.zeros(len(data) + 64, dtype=torch.uint8).pin_memory()
    host[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8)
    dev = host.cuda()
    want = ref.compress(data, 0, numiterations=2)
    for dptr in (None, dev.data_ptr()):
        ob = lib.compress_ptr_nocopy(host.data_ptr(), len(data), zb.ZOPFLI_FORMAT_GZIP, dev_ptr=dptr, numiterations=2)
        assert len(ob) == len(want) and ob.tobytes() == want
        ob.close()


def test_pipeline_shapes_give_one_stream(ref):
    """Chunk pipelines, the giant-block lane split and the host thread count are scheduling
    choices: every combination must produce the reference's bytes.  The switches are read once per
    process, hence subprocesses."""
    import os, subprocess, sys, tempfile
    data = TXT  # three master blocks
    want = ref.compress(data, 2, numiterations=2)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "in.bin")
        open(src, "wb").write(data)
        code = ("import sys; sys.path.insert(0, %r); import zopfli_b200 as zb; d = open(%r, 'rb').read(); "
                "open(sys.argv[1], 'wb').write(zb.compress(d, zb.ZOPFLI_FORMAT_DEFLATE, numiterations=2))" % (root, src))
        for i, env in enumerate([{"ZOPFLI_B200_FORCE_CHUNKS": "3", "ZOPFLI_B200_GIANT": "50000"},
                                 {"ZOPFLI_B200_FORCE_CHUNKS": "2", "ZOPFLI_B200_GIANT": "100000000"},
                                 {"ZOPFLI_B200_CONTEXTS": "1", "ZOPFLI_B200_THREADS": "3"}]):
            out = os.path.join(td, "out%d.bin" % i)
            subprocess.check_call([sys.executable, "-c", code, out], env=dict(os.environ, **env))
            assert open(out, "rb").read() == want, env


def test_reentrant_concurrent_calls(ref, lib):
    """The reference keeps no mutable globals (zopfli.h:82-88): concurrent calls on different inputs
    must not disturb each other.  Eight threads x different inputs x mixed formats / entry points,
    twice as many callers as engine contexts, all compared with the reference."""
    import threading
    inputs = [TXT[:300000], corpus.synth_binary(250000), corpus.adv_runs(), TXT[1000000:1250000],
              corpus.mixed_small(120000), TXT[500000:1700000], corpus.adv_collide(), b"", ]
    want, got, errs = {}, {}, []
    for i, d in enumerate(inputs):
        want[i] = (ref.compress(d, i % 3, numiterations=3), ref.deflate_part(d, 0, len(d) // 2, final=0, numiterations=2))

    def work(i):
        try:
            d = inputs[i]
            for _ in range(2):
                got[i] = (lib.compress(d, i % 3, numiterations=3), lib.deflate_part(d, 0, len(d) // 2, final=0, numiterations=2))
                if got[i] != want[i]:
                    errs.append(i)
        except Exception as e:  # pragma: no cover
            errs.append((i, repr(e)))

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(inputs))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    assert got == want


def test_verbose_output_matches_reference(ref, tmp_path):
    """options.verbose / verbose_more on a one-block input (so the order of the lines is fixed): the
    split-point, per-iteration (squeeze.c:493-495), tree-size and block-size lines on stderr are the
    reference's, byte for byte."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "verb.py"
    script.write_text('''
import sys, ctypes as C, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import zopfli_b200 as zb, zref
from zopfli_b200 import corpus
d = corpus.synth_text(120000, 3)
more = int(sys.argv[2])
def opts(o):
    o.verbose = 1; o.verbose_more = more; o.numiterations = 9; o.blocksplitting = 0
    return o
if sys.argv[1] == "ref":
    r = zref.Ref(); lib = r.lib; o = opts(r.options())
else:
    z = zb.library(); lib = z.lib; o = opts(z.options())
a = np.zeros(len(d) + 64, np.uint8); a[:len(d)] = np.frombuffer(d, np.uint8)
out = C.c_void_p(None); n = C.c_size_t(0)
lib.ZopfliCompress(C.byref(o), 2, C.c_void_p(a.ctypes.data), C.c_size_t(len(d)), C.byref(out), C.byref(n))
''' % (root, os.path.join(root, "tests")))

    def run(which, more):
        r = subprocess.run([sys.executable, str(script), which, str(more)], capture_output=True, text=True, check=True)
        return r.stderr.splitlines()
    for more in (0, 1):
        want = ref.answer("verbose_stderr", ("synth_text(120000, 3)", 9, more), lambda r: run("ref", more))
        assert run("b200", more) == want and any(l.startswith("Iteration") for l in want), more

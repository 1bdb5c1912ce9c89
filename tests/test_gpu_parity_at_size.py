"""Parity with the UNMODIFIED reference (its recorded answers) at the sizes bench.py runs:
BASELINE.json configs C2 (100 MB text, 15 iterations) and C4 (51 MB binary, 50 iterations).

The reference needs ~2 s of CPU per master block at 15 iterations, so the full inputs are covered by
SAMPLED master blocks compared through ZopfliDeflatePart (deflate.c:811-906; a master block is an
independent unit, deflate.c:908-931): the five master blocks that hold the LARGEST deflate blocks of
the C2 text (tools/find_giant_masters.py; master 85 holds the 969,128-position block whose DP chain is
the bench's critical path and whose costs cross 2^21) plus eight uniformly spread ones.  Zero tolerance:
byte-identical streams.
"""
import zlib

import numpy as np
import pytest

import zopfli_b200 as zb
from zopfli_b200 import corpus

pytestmark = pytest.mark.gpu

MB = 1000000
C2_BYTES = 100000000
C4_BYTES = 51220480
GIANT_MASTERS = [85, 84, 78, 42, 40]          # tools/find_giant_masters.py on synth_text(1e8, 2)
UNIFORM_MASTERS = [3, 15, 27, 39, 51, 63, 75, 99]


def _slices(data, masters):
    out = []
    for m in masters:
        a, b = m * MB, min(len(data), (m + 1) * MB)
        lo = max(0, a - 32768)  # only the 32 KiB window before the range can matter (squeeze.c:229-230)
        out.append((data[lo:b], a - lo, b - lo))
    return out


def _reference_parts(ref, parts, iters, final=1):
    return ref.map("deflate_part", parts, final=final, numiterations=iters)


@pytest.fixture(scope="module")
def lib():
    return zb.library()


@pytest.fixture(scope="module")
def c2():
    return corpus.synth_text(C2_BYTES, 2)


def test_c2_giant_and_sampled_master_blocks(ref, lib, c2):
    """C2 at 15 iterations: the master blocks holding the five largest blocks + eight sampled ones."""
    masters = GIANT_MASTERS + UNIFORM_MASTERS
    parts = _slices(c2, masters)
    want = _reference_parts(ref, parts, 15)
    lib.reset_stats()
    for m, (piece, s, e), w in zip(masters, parts, want):
        got = lib.deflate_part(piece, s, e, final=1, numiterations=15)   # (bytes, bp)
        assert got == w, "master block %d differs from the reference (%d vs %d bytes)" % (m, len(got[0]), len(w[0]))
        assert zlib.decompressobj(-15, zdict=piece[:s]).decompress(got[0]) == piece[s:e]  # the 32 KiB before the range is its dictionary
    st = lib.stats()
    assert st["max_block_positions"] >= 900000  # the giant blocks really went through k_iterate


def test_c2_whole_stream_contains_the_sampled_master_blocks(ref, lib, c2):
    """One ZopfliCompress of the first 45 master blocks (the batched pipelines, lanes and giants of the
    bench) == per-master-block reference spans, compared through the per-master bit offsets."""
    n = 45 * MB
    data = c2[:n]
    z = lib.compress(data, zb.ZOPFLI_FORMAT_DEFLATE, numiterations=15)
    assert zlib.decompress(z, -15) == data
    offs = lib.last_master_bit_offsets()
    assert len(offs) == 46 and offs[0] == 0
    masters = [0, 9, 40, 42, 43]
    parts = _slices(data, masters)
    bits = np.unpackbits(np.frombuffer(z, dtype=np.uint8), bitorder="little")
    want = _reference_parts(ref, parts, 15, final=0)  # BFINAL is set only on the stream's very last block
    for m, w in zip(masters, want):
        # the master block's bits, zero-padded to whole bytes, and its bit count mod 8: (bytes, bp) of ZopfliDeflatePart
        got = np.packbits(bits[offs[m]:offs[m + 1]], bitorder="little").tobytes(), int(offs[m + 1] - offs[m]) & 7
        assert got == w, "master block %d" % m


def test_c4_binary_50_iterations(ref, lib):
    """C4: redundant binary at numiterations=50 -- random restarts + blended statistics
    (squeeze.c:505-517) on full-size master blocks."""
    data = corpus.synth_binary(C4_BYTES, 4)
    masters = [7, 30]
    parts = _slices(data, masters)
    want = _reference_parts(ref, parts, 50)
    for m, (piece, s, e), w in zip(masters, parts, want):
        got = lib.deflate_part(piece, s, e, final=1, numiterations=50)
        assert got == w, "C4 master block %d differs from the reference" % m


def test_three_master_blocks_15_iterations_all_formats(ref, lib):
    data = corpus.synth_text(2300000, 2)
    for fmt in (zb.ZOPFLI_FORMAT_GZIP, zb.ZOPFLI_FORMAT_ZLIB, zb.ZOPFLI_FORMAT_DEFLATE):
        assert lib.compress(data, fmt, numiterations=15) == ref.compress(data, fmt, numiterations=15), fmt


def test_device_auto_type_bits_seam(ref, lib):
    """k_split_eval (the splitter's cost oracle) == ZopfliCalculateBlockSizeAutoType (deflate.c:610-621)
    on ranges of a greedy store, including the `lz77->size > 1000` switch (small and large stores)."""
    data = corpus.synth_text(400000, 5)
    rng = np.random.default_rng(11)
    for s, e in ((0, 300000), (1000, 4000)):
        ll, dd = ref.lz77(data, s, e, 2, 0)
        n = len(ll)
        a = rng.integers(0, n, 200)
        b = rng.integers(0, n + 1, 200)
        lo, hi = np.minimum(a, b), np.maximum(a, b)
        lo[0], hi[0] = 0, n
        got = lib.device_auto_type_bits(ll, dd, lo, hi)
        want = ref.many("block_size", [(data[s:e], ll, dd, int(lo[i]), int(hi[i]), -1) for i in range(len(lo))])
        assert [float(g) for g in got] == want, (s, e)


def test_one_block_larger_than_a_master_block(ref, lib):
    """ZopfliDeflatePart over 2.5 MB with block splitting off: ONE deflate block whose symbol counts pass
    the default 2^21-entry log table (the table grows on demand instead of aborting)."""
    data = corpus.synth_text(2500000, 9)
    for kw in ({"numiterations": 7, "blocksplitting": 0},):
        a = ref.deflate_part(data, 0, len(data), final=1, **kw)
        b = lib.deflate_part(data, 0, len(data), final=1, **kw)
        assert a == b, kw

"""The integer window of k_iterate's forward DP (zopfli_b200/csrc/iterate.cuh, DESIGN.md section 2): it has to
actually run (otherwise every parity test would only exercise the fp64 paths), and the fp64-only build of the
same call (ZOPFLI_B200_INTDP=0, read once per process) has to produce the same bytes as it and as the
reference (squeeze.c:217-309).  Integer / byte work: zero tolerance."""
import os
import subprocess
import sys

import pytest

import zopfli_b200 as zb
from zopfli_b200 import corpus

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = [
    ("text", lambda: corpus.synth_text(700000, 11), 6),      # long matches: integer general groups, ring joins
    ("binary", lambda: corpus.synth_binary(400000, 5), 8),   # byte runs: shortcut zones force the fp64 general path
    ("random4", lambda: bytes(b & 3 for b in corpus.random_bytes(300000)), 4),
]


@pytest.mark.parametrize("name,make,iters", CASES, ids=[c[0] for c in CASES])
def test_integer_window_runs_and_matches_fp64_and_reference(ref, name, make, iters):
    data = make()
    lib = zb.library()
    lib.reset_stats()
    got = lib.compress(data, zb.ZOPFLI_FORMAT_DEFLATE, numiterations=iters)
    st = lib.stats()
    assert st["iterate_steps"] > 0
    if name != "binary":
        assert st["int_steps"] > 0.5 * st["iterate_steps"], "the integer window did not run"
    assert got == ref.compress(data, zb.ZOPFLI_FORMAT_DEFLATE, numiterations=iters)
    # the same call with the integer window switched off, in a process of its own
    code = ("import sys, hashlib; sys.path.insert(0, %r); import zopfli_b200 as zb; from zopfli_b200 import corpus\n"
            "data = open(sys.argv[1], 'rb').read()\n"
            "lib = zb.library(); lib.reset_stats()\n"
            "out = lib.compress(data, zb.ZOPFLI_FORMAT_DEFLATE, numiterations=%d)\n"
            "assert lib.stats()['int_steps'] == 0\n"
            "print(hashlib.sha256(out).hexdigest())\n") % (ROOT, iters)
    import hashlib
    import tempfile
    with tempfile.NamedTemporaryFile(suffix=".bin") as f:
        f.write(data)
        f.flush()
        env = dict(os.environ, ZOPFLI_B200_INTDP="0")
        r = subprocess.run([sys.executable, "-c", code, f.name], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip().splitlines()[-1] == hashlib.sha256(got).hexdigest()

"""Golden vectors (reference-generated, tests/golden/make_golden.py) and the restated Go tests
(/root/reference/go/zopfli/zopfli_test.go:35-69: round trip + size bounds; the Go wrapper itself
cannot run here -- no Go toolchain)."""
import gzip
import hashlib
import json
import os

import pytest

import zopfli_b200 as zb
from zopfli_b200 import corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "zopfli_golden.json")))
import importlib.util
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
_mg = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(_mg)
FMT = {"gzip": 0, "zlib": 1, "deflate": 2}


def _check(lib_compress, name):
    data = _mg.CASES[name]()
    g = GOLD[name]
    assert len(data) == g["n"] and hashlib.sha256(data).hexdigest() == g["sha256"], "generator drifted"
    for key, want in g["streams"].items():
        fname, it = key.split("_i")
        z = lib_compress(data, FMT[fname], numiterations=int(it))
        if isinstance(want, str):
            assert z.hex() == want, key
        else:
            assert len(z) == want["len"] and hashlib.sha256(z).hexdigest() == want["sha256"], key


@pytest.mark.parametrize("name", sorted(GOLD))
def test_host_logic_matches_golden(name):
    """the product's host code over the oracle-backed mock engine (tests/hostmock) reproduces the committed vectors"""
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "hostmock")])
    _check(zb.Library(os.path.join(ROOT, "tests", "_build", "libzopfli_hostmock.so")).compress, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GOLD))
def test_product_matches_golden(name):
    _check(zb.library().compress, name)


@pytest.mark.gpu
def test_go_cases():
    lib = zb.library()
    z = lib.compress(corpus.go_case_foobar(), 0)     # zopfli_test.go:36-38: <= 500 bytes
    assert gzip.decompress(z) == corpus.go_case_foobar() and len(z) <= 500
    r = corpus.random_bytes(3000, 1)                 # zopfli_test.go:40-42: <= 3100 bytes
    z = lib.compress(r, 0)
    assert gzip.decompress(z) == r and len(z) <= 3100
    z = lib.compress(b"", 0)                         # zopfli_test.go:44-46: <= 20 bytes
    assert gzip.decompress(z) == b"" and len(z) <= 20

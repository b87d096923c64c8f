"""-m gpu: the C++ drop-in layer (include/spsparse/*.hpp over the C ABI).

(1) tests/cpp/host_layer_test.cpp: this repo's own C++ test of the template API.
(2) the REFERENCE's own gtest sources (tests/test_xiter.cpp, test_array.cpp, test_multiply_sparse.cpp),
    compiled UNMODIFIED against this repo's headers by `make -C oracle dropin` when SPSPARSE_REFERENCE names a
    checkout of the original spsparse (the sources stay there; the binaries go to oracle/_ref/).
"""
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(path, timeout=600):
    r = subprocess.run([path], capture_output=True, text=True, timeout=timeout)
    return r.returncode, r.stdout[-4000:] + r.stderr[-2000:]


def test_host_layer_cpp():
    exe = os.path.join(ROOT, "tests", "cpp", "_bin", "host_layer_test")
    if not os.path.exists(exe):
        pytest.skip("tests/cpp/_bin/host_layer_test not built (run __graft_entry__.build())")
    rc, out = run(exe)
    assert rc == 0 and "0 failure(s)" in out, out


@pytest.mark.parametrize("name", ["test_xiter", "test_array", "test_multiply_sparse"])
def test_reference_sources_against_our_headers(name):
    exe = os.path.join(ROOT, "oracle", "_ref", "dropin_" + name)
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/dropin_* not built (needs SPSPARSE_REFERENCE, a checkout of the original spsparse, at build time)")
    rc, out = run(exe)
    assert rc == 0 and " 0 failed" in out, out

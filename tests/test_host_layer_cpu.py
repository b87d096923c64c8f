"""CPU suite: the host-only part of the C++ template layer (include/spsparse/*.hpp).

(1) tests/cpp/host_only_test.cpp -- container, accessors, iterators, sorted joins, accumulators, error hook and the
    short-circuits of consolidate/multiply that return before any device work (SURVEY 8a rows a1, a2, a6, a8, a12).
(2) the REFERENCE's own tests/test_xiter.cpp, compiled unmodified against this repo's headers (oracle/_ref/dropin_test_xiter,
    built by `make -C oracle dropin` when SPSPARSE_REFERENCE names a checkout of it): joins are pure host code, so it runs without a GPU.
Everything that computes on the device is in test_gpu_dropin.py.
"""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_host_only_cpp():
    import __graft_entry__ as g
    exe = g.build_cpp_test("host_only_test")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "0 failure(s)" in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]


def test_reference_xiter_source_against_our_headers():
    exe = os.path.join(ROOT, "oracle", "_ref", "dropin_test_xiter")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/dropin_test_xiter not built (needs SPSPARSE_REFERENCE, a checkout of the original spsparse, at build time)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and " 0 failed" in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]

"""CPU suite: NetCDF I/O of COO arrays (SURVEY 8f rank 4; reference slib/spsparse/netcdf.hpp:23-138, tests/test_netcdf.cpp).

include/spsparse/netcdf.hpp runs here over the minimal classic-format netCDF of include/spsparse_b200/mini_netcdf/ (the image has
no netCDF library).  Three independent checks of that format code:
(1) tests/cpp/netcdf_test.cpp selftest: the reference's write / read(alloc) / read(no alloc) round trip and the API subset;
(2) the CDF-5 file ncio_spsparse writes, byte for byte against a file assembled HERE from the published grammar
    (header = magic numrecs dim_list gatt_list var_list, big-endian, 4-byte padding; CDF-5: 64-bit counts and offsets);
(3) scipy.io.netcdf_file -- an unrelated implementation of CDF-1/2 -- reads what the C++ writer wrote (classic, classic64)
    and the C++ reader reads what scipy wrote, record (unlimited) variables included.
(4) the REFERENCE's own tests/test_netcdf.cpp, compiled unmodified against these headers (oracle/_ref/dropin_test_netcdf).
"""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe():
    import __graft_entry__ as g
    return g.build_cpp_test("netcdf_test")


def run(exe, *args):
    r = subprocess.run([exe, *args], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r.stdout


def test_selftest(exe, tmp_path):
    out = run(exe, "selftest", str(tmp_path))
    assert "0 failure(s)" in out, out


# ---- (2) the CDF-5 grammar, restated --------------------------------------------------------------------------------------------
NC_DIMENSION, NC_VARIABLE, NC_ATTRIBUTE = 0x0A, 0x0B, 0x0C
NC_DOUBLE, NC_INT64, NC_UINT64 = 6, 10, 11


def pad4(b):
    return b + b"\0" * (-len(b) % 4)


def name5(s):
    return struct.pack(">q", len(s)) + pad4(s.encode())


def cdf5_spsparse(vname, shape, idx, val):
    """The file ncio_spsparse writes for one array (netcdf.hpp:93-106), as CDF-5 bytes."""
    n, rank = len(val), len(shape)
    dims = [(vname + ".size", n), (vname + ".rank", rank)]
    hdr = b"CDF\x05" + struct.pack(">q", 0)
    hdr += struct.pack(">iq", NC_DIMENSION, len(dims)) + b"".join(name5(nm) + struct.pack(">q", ln) for nm, ln in dims)
    hdr += struct.pack(">iq", 0, 0)                                                  # no global attributes
    shape_att = struct.pack(">iq", NC_ATTRIBUTE, 1) + name5("shape") + struct.pack(">iq", NC_UINT64, rank) + struct.pack(f">{rank}Q", *shape)
    absent = struct.pack(">iq", 0, 0)
    variables = [  # name, dimids, attribute list, type, vsize
        (vname + ".info", [], shape_att, NC_INT64, 8),
        (vname + ".indices", [0, 1], absent, NC_INT64, 8 * n * rank),
        (vname + ".vals", [0], absent, NC_DOUBLE, 8 * n),
    ]
    def var_header(nm, dimids, atts, typ, vsize, begin):
        return name5(nm) + struct.pack(">q", len(dimids)) + b"".join(struct.pack(">q", d) for d in dimids) + atts + struct.pack(">iqq", typ, vsize, begin)
    fixed = len(hdr) + 12 + sum(len(var_header(*v, 0)) for v in variables)
    begins, off = [], fixed
    for v in variables:
        begins.append(off)
        off += v[4]
    hdr += struct.pack(">iq", NC_VARIABLE, len(variables)) + b"".join(var_header(*v, b) for v, b in zip(variables, begins))
    assert len(hdr) == fixed
    data = struct.pack(">q", 0)                                                      # <v>.info: never written, reads as 0
    data += np.asarray(idx, dtype=">i8").reshape(n, rank).tobytes() + np.asarray(val, dtype=">f8").tobytes()
    return hdr + data


FIXED_IDX = [[1, 2], [3, 3], [4, 5], [1, 2], [0, 0]]
FIXED_VAL = [2.0, 6.0, 1.0, -0.25, 0.0]


def test_cdf5_file_byte_for_byte(exe, tmp_path):
    p = tmp_path / "arr1.nc"
    run(exe, "write", str(p))
    want = cdf5_spsparse("arr1", (5, 6), FIXED_IDX, FIXED_VAL)
    got = p.read_bytes()
    assert got == want, (len(got), len(want), next((i for i in range(min(len(got), len(want))) if got[i] != want[i]), None))


def test_reader_takes_a_file_assembled_from_the_grammar(exe, tmp_path):
    """... and the reverse: bytes assembled here (another array, rank 1) are read back by the C++ side."""
    p = tmp_path / "v.nc"
    p.write_bytes(cdf5_spsparse("v", (9,), [[8], [0], [3]], [1.5, -2.0, 1e300]))
    out = run(exe, "dump", str(p))
    assert "var v.indices int64 v.size v.rank\nvalues 8 0 3\n" in out and "var v.vals double v.size\nvalues 1.5 -2 1.0000000000000001e+300\n" in out, out


# ---- the Python mirror's reader / writer (spsparse_b200/ncio.py): the same files ---------------------------------------------------
def test_python_mirror_writes_the_same_bytes_and_reads_the_cpp_files(exe, tmp_path):
    from spsparse_b200 import ncio
    idx = [np.array([r for r, _ in FIXED_IDX]), np.array([c for _, c in FIXED_IDX])]
    p_py, p_cpp = tmp_path / "py.nc", tmp_path / "cpp.nc"
    ncio.write_spsparse(str(p_py), {"arr1": ((5, 6), idx, FIXED_VAL)})
    run(exe, "write", str(p_cpp))
    assert p_py.read_bytes() == p_cpp.read_bytes() == cdf5_spsparse("arr1", (5, 6), FIXED_IDX, FIXED_VAL)
    shape, ridx, rval = ncio.read_spsparse(str(p_cpp), "arr1")
    assert shape == (5, 6) and [x.tolist() for x in ridx] == [x.tolist() for x in idx] and rval.tolist() == FIXED_VAL
    # two arrays of different rank in one file, through the C++ reader
    rng = np.random.default_rng(3)
    n = 1000
    big = ((7000, 9000), [rng.integers(0, 7000, n), rng.integers(0, 9000, n)], rng.standard_normal(n))
    vec = ((50,), [rng.integers(0, 50, 7)], rng.standard_normal(7))
    p2 = tmp_path / "two.nc"
    ncio.write_spsparse(str(p2), {"M": big, "v": vec})
    for name, (shp, ix, vv) in (("M", big), ("v", vec)):
        s2, i2, v2 = ncio.read_spsparse(str(p2), name)
        assert s2 == shp and all(np.array_equal(a, b) for a, b in zip(i2, ix)) and np.array_equal(v2, vv)
    out = run(exe, "dump", str(p2))
    assert "var M.indices int64 M.size M.rank" in out and "var v.vals double v.size" in out
    assert "values " + " ".join(repr(float(x)) if False else f"{x:.17g}" for x in vec[2]) in out
    with pytest.raises(KeyError):
        ncio.read_spsparse(str(p2), "nope")
    bad = tmp_path / "bad.nc"
    bad.write_bytes(b"\x89HDF\r\n\x1a\n" + b"\0" * 64)
    with pytest.raises(ValueError, match="HDF5"):
        ncio.read_spsparse(str(bad), "M")


def test_python_mirror_reads_classic_files_from_scipy(tmp_path):
    """CDF-1 / CDF-2 files with the same variable names (int32 indices: the classic types), written by scipy."""
    from scipy.io import netcdf_file
    from spsparse_b200 import ncio
    for version in (1, 2):
        p = tmp_path / f"classic{version}.nc"
        with netcdf_file(str(p), "w", version=version) as f:
            f.createDimension("A.size", 4)
            f.createDimension("A.rank", 2)
            info = f.createVariable("A.info", "i4", ())
            info.shape_ = 0   # (scipy reserves the attribute name "shape"; written below through _attributes)
            info._attributes.clear()
            info._attributes["shape"] = np.array([10, 20], dtype=np.int32)
            ind = f.createVariable("A.indices", "i4", ("A.size", "A.rank")); ind[:] = np.array([[1, 2], [3, 4], [9, 19], [0, 0]], dtype=np.int32)
            vals = f.createVariable("A.vals", "f8", ("A.size",)); vals[:] = np.array([1.5, -2.0, 3.25, 0.0])
        shape, idx, val = ncio.read_spsparse(str(p), "A")
        assert shape == (10, 20) and idx[0].tolist() == [1, 3, 9, 0] and idx[1].tolist() == [2, 4, 19, 0] and val.tolist() == [1.5, -2.0, 3.25, 0.0]


# ---- (3) against scipy's netCDF-3 implementation ---------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt,version", [("classic", 1), ("classic64", 2)])
def test_scipy_reads_what_the_writer_wrote(exe, tmp_path, fmt, version):
    from scipy.io import netcdf_file
    p = tmp_path / f"{fmt}.nc"
    run(exe, "write-classic", str(p), fmt)
    assert p.read_bytes()[:4] == b"CDF" + bytes([version])
    with netcdf_file(str(p), "r", mmap=False) as f:
        assert f.version_byte == version
        assert dict(f.dimensions) == {"n": 5, "rank": 2}
        assert f.variables["indices"].data.tolist() == FIXED_IDX and f.variables["indices"].data.dtype == np.dtype(">i4")
        assert f.variables["vals"].data.tolist() == FIXED_VAL
        assert f.variables["tag"].data.tolist() == [-7, 300]
        assert f.variables["indices"]._attributes["shape"].tolist() == [5, 6]
        assert f.history == b"written by netcdf_test"


@pytest.mark.parametrize("version", [1, 2])
def test_reader_takes_what_scipy_wrote(exe, tmp_path, version):
    from scipy.io import netcdf_file
    p = tmp_path / f"scipy{version}.nc"
    rng = np.random.default_rng(5 + version)
    a = rng.integers(-1000, 1000, (4, 3)).astype(np.int32)
    b = rng.standard_normal(7)
    c = rng.integers(-100, 100, (5, 3)).astype(np.int16)    # record variable: 3 shorts per record, padded
    d = rng.standard_normal(5).astype(np.float32)          # second record variable
    with netcdf_file(str(p), "w", version=version) as f:
        f.createDimension("t", None)
        f.createDimension("y", 4)
        f.createDimension("x", 3)
        f.createDimension("m", 7)
        f.title = "from scipy"
        va = f.createVariable("a", "i4", ("y", "x")); va[:] = a; va.units = "counts"
        vb = f.createVariable("b", "f8", ("m",)); vb[:] = b
        vc = f.createVariable("c", "i2", ("t", "x")); vc[:] = c
        vd = f.createVariable("d", "f4", ("t",)); vd[:] = d
    out = run(exe, "dump", str(p))
    vals = {}
    lines = out.splitlines()
    for i, ln in enumerate(lines):
        if ln.startswith("var "):
            vals[ln.split()[1]] = (ln.split()[2:], np.array([float(x) for x in lines[i + 1].split()[1:]]))
    assert "dim t 5 1" in out and "dim y 4 0" in out
    assert vals["a"][0] == ["int", "y", "x"] and np.array_equal(vals["a"][1], a.ravel().astype(float))
    assert vals["b"][0] == ["double", "m"] and np.array_equal(vals["b"][1], b)
    assert vals["c"][0] == ["short", "t", "x"] and np.array_equal(vals["c"][1], c.ravel().astype(float))
    assert vals["d"][0] == ["float", "t"] and np.array_equal(vals["d"][1], d.astype(float))


def test_single_record_variable_is_not_padded(exe, tmp_path):
    """The classic format's special case: with exactly one record variable, records are packed without padding."""
    from scipy.io import netcdf_file
    p = tmp_path / "onerec.nc"
    c = np.arange(15, dtype=np.int16).reshape(5, 3) - 7
    with netcdf_file(str(p), "w", version=1) as f:
        f.createDimension("t", None)
        f.createDimension("x", 3)
        vc = f.createVariable("c", "i2", ("t", "x")); vc[:] = c
    out = run(exe, "dump", str(p))
    assert "values " + " ".join(str(int(x)) for x in c.ravel()) in out, out


# ---- (4) the reference's own test source -----------------------------------------------------------------------------------------
def test_reference_netcdf_test_against_our_headers(tmp_path):
    exe = os.path.join(ROOT, "oracle", "_ref", "dropin_test_netcdf")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/dropin_test_netcdf not built (needs SPSPARSE_REFERENCE, a checkout of the original spsparse, at build time)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120, cwd=str(tmp_path))
    assert r.returncode == 0 and " 0 failed" in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]

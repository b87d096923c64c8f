"""CPU: the reference arm of bench.py runs here (it times the reference's own CPU code) and must print exactly one
JSON line with the keys the driver reads; bench.py and the tools must at least parse."""
import ast
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-rows", "300", "--ref-procs", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "products/s" and d["higher_is_better"] is True and d["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d, k
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] == 2 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_scripts_parse():
    for rel in ["bench.py", "__graft_entry__.py"] + [os.path.join("tools", f) for f in sorted(os.listdir(os.path.join(ROOT, "tools"))) if f.endswith(".py")]:
        ast.parse(open(os.path.join(ROOT, rel)).read(), filename=rel)


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_clock_sampler_prefers_nvml_and_survives_failed_queries(monkeypatch):
    """bench.py's clocks line: NVML polled every 2 ms (fake module here), failed queries are missing samples, throttle
    reasons are collected; without NVML and without nvidia-smi the line carries nulls instead of failing."""
    import time
    import types
    bench = _bench()
    nv = types.ModuleType("pynvml")

    class NVMLError(Exception):
        pass
    calls = [0]

    def clock(h, t):
        calls[0] += 1
        if calls[0] % 4 == 0:
            raise NVMLError("transient")
        return 1900 + calls[0] % 2
    nv.NVMLError = NVMLError
    nv.nvmlInit = lambda: None
    nv.nvmlDeviceGetHandleByUUID = lambda u: ("uuid", u)
    nv.nvmlDeviceGetHandleByIndex = lambda i: ("index", i)
    nv.NVML_CLOCK_SM = 1
    nv.nvmlDeviceGetMaxClockInfo = lambda h, t: 1965
    nv.nvmlDeviceGetClockInfo = clock
    nv.nvmlDeviceGetCurrentClocksThrottleReasons = lambda h: 4 | 1   # sw_power_cap + gpu_idle (not reported)
    nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown = 8, 64
    nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap = 32, 4
    monkeypatch.setitem(sys.modules, "pynvml", nv)
    s = bench.ClockSampler(0, "GPU-1234")
    time.sleep(0.02)
    assert s.sm == []            # nothing is kept before the timed region begins
    s.begin()
    time.sleep(0.05)
    out = s.stop()
    assert out["samples"] >= 5 and out["source"].startswith("nvml") and 1900 <= out["sm_mhz"] <= 1901
    assert out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"]
    broken = types.ModuleType("pynvml")   # no NVML at all (no attributes): falls back to nvidia-smi, absent here too
    monkeypatch.setitem(sys.modules, "pynvml", broken)
    out = bench.ClockSampler(0, None).stop()
    assert out["samples"] == 0 and out["sm_mhz"] is None and out["reasons"] == []


def test_numa_binding_reads_sysfs_and_never_fails(monkeypatch):
    import builtins
    import io
    import types
    bench = _bench()
    props = types.SimpleNamespace(pci_domain_id=0, pci_bus_id=0x1B, pci_device_id=0)
    torch = types.SimpleNamespace(cuda=types.SimpleNamespace(get_device_properties=lambda i: props))
    have = os.sched_getaffinity(0)
    some = sorted(have)[: max(1, len(have) // 2)]
    files = {"/sys/bus/pci/devices/0000:1b:00.0/numa_node": "1\n",
             "/sys/devices/system/node/node1/cpulist": ",".join(str(c) for c in some) + ",100000-100003\n"}
    real = builtins.open
    monkeypatch.setattr(builtins, "open", lambda p, *a, **k: io.StringIO(files[p]) if p in files else real(p, *a, **k))
    try:
        out = bench.bind_to_gpu_numa_node(torch, 0)
        assert out["node"] == 1 and out["cpus"] == len(some) and os.sched_getaffinity(0) == set(some)
        assert out["bound"] == (set(some) != have)
    finally:
        os.sched_setaffinity(0, have)
    files["/sys/bus/pci/devices/0000:1b:00.0/numa_node"] = "-1\n"
    assert bench.bind_to_gpu_numa_node(torch, 0)["bound"] is False and os.sched_getaffinity(0) == have
    del files["/sys/bus/pci/devices/0000:1b:00.0/numa_node"]       # no such device in sysfs
    assert bench.bind_to_gpu_numa_node(torch, 0)["bound"] is False
    monkeypatch.setenv("SPB_NO_NUMA_BIND", "1")
    assert bench.bind_to_gpu_numa_node(torch, 0) == {"bound": False, "why": "SPB_NO_NUMA_BIND"}


def test_dump_outputs_writes_c_whole_or_as_a_fixed_sample(monkeypatch, tmp_path):
    """--dump-outputs: C's rows, columns and values as float64 .npy files; a small C whole, a large one at seeded
    positions in order -- the same positions in every run, and the same for all three arrays -- under 64 MB in all, at
    N = 1 and over the ranks of N = 8.  Host arrays stand in for the device memory of the result; every value encodes its
    row and column, so entries taken from different positions cannot pass."""
    import numpy as np
    import torch
    bench = _bench()
    rng = np.random.default_rng(3)
    n = bench.DUMP_ENTRIES + 1000
    row = np.sort(rng.integers(0, 1 << 20, n)).astype(np.int32)
    col = rng.integers(0, 1 << 20, n).astype(np.int32)
    arrays = [row, col, row * float(1 << 20) + col]

    class Result:
        def __init__(self, size):
            self.n = size

        def size(self):
            return self.n

        def device_ptrs(self):
            return (0, 1), 2

    def as_tensor(x, device=None):
        if isinstance(x, bench.DevView):
            iface = x.__cuda_array_interface__
            return torch.from_numpy(arrays[iface["data"][0]][:iface["shape"][0]])
        return torch.from_numpy(np.asarray(x))
    monkeypatch.setattr(torch, "as_tensor", as_tensor)
    for size, d in ((1000, "small"), (n, "a"), (n, "b")):
        bench.dump_result(torch, Result(size), str(tmp_path / d), 0, 1)
    names = ("C_row.npy", "C_col.npy", "C_val.npy")
    assert sorted(os.listdir(tmp_path / "a")) == sorted(names)
    for name, a in zip(names, arrays):
        small = np.load(tmp_path / "small" / name)
        assert small.dtype == np.float64 and np.array_equal(small, a[:1000])
        x, y = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert x.dtype == np.float64 and len(x) == bench.DUMP_ENTRIES and x.tobytes() == y.tobytes()
    r, c, v = (np.load(tmp_path / "a" / name) for name in names)
    assert np.array_equal(v, r * (1 << 20) + c) and np.isin(v, arrays[2]).all()    # whole entries of C
    assert np.all(np.diff(r) >= 0)                                                   # positions in order: rows stay sorted
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    for rank in range(8):                                                            # N = 8: every rank its own block
        bench.dump_result(torch, Result(n), str(tmp_path / "n8"), rank, 8)
    files = os.listdir(tmp_path / "n8")
    assert sorted(files) == sorted(f"{name[:-4]}.rank{rank}.npy" for name in names for rank in range(8))
    assert sum(os.path.getsize(tmp_path / "n8" / f) for f in files) <= 64 << 20

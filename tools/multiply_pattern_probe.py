"""Times spb_multiply_mm against spb_mm_pattern_run on three workloads, in one process:

    python tools/multiply_pattern_probe.py [--reps 10] [--warmup 2] [--out result.json]

- config 5 on one GPU: banded 10^8-row A * diag(w) * B from unsorted COO (the step a time stepper runs every step);
- config 3: regridding A * diag(s) * A^T, one values array passed for both operands;
- R-MAT scale 20, A * A (long rows: the hash bin).

For each workload: plan creation is timed once; then the two paths alternate, `warmup` times each untimed and `reps` times
each timed with CUDA events on the library's stream.  Both paths read the same device values.  Their outputs are compared on
the device: index arrays equal, values equal as bits.  The device name and power limit are read in the same process (query
only).  Prints one JSON object per workload; --out also writes them to a file."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class _View:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _device_info(torch):
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def _same_on_device(torch, R1, R2):
    """Shape equal, index arrays equal and values equal as bits."""
    n = R1.size()
    if n != R2.size() or tuple(R1.shape) != tuple(R2.shape) or R1.sort_order != R2.sort_order:
        return False
    (i1, v1), (i2, v2) = R1.device_ptrs(), R2.device_ptrs()
    if n == 0:
        return True
    ok = True
    for a, b in zip(i1, i2):
        ok = ok and torch.equal(torch.as_tensor(_View(a, n, "<i4"), device="cuda"), torch.as_tensor(_View(b, n, "<i4"), device="cuda"))
    return ok and torch.equal(torch.as_tensor(_View(v1, n, "<i8"), device="cuda"), torch.as_tensor(_View(v2, n, "<i8"), device="cuda"))


def probe(sp, torch, ctx, stream, name, args, reps, warmup):
    """args: (Cst, si, A, tA, sj, B, tB, sk)."""
    Cst, si, A, tA, sj, B, tB, sk = args
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    _, a_val = A.device_ptrs()
    _, b_val = B.device_ptrs()
    e0, e1 = ev(), ev()
    e0.record(stream)
    plan = sp.MultiplyPattern(ctx, Cst, si, A, tA, sj, B, tB, sk)
    e1.record(stream)
    e1.synchronize()
    t_create = e0.elapsed_time(e1)

    def fresh():
        return sp.multiply(ctx, Cst, si, A, tA, sj, B, tB, sk, stats=True)

    def planned():
        return plan.run(a_val, b_val, stats=True)

    R1, st_f = fresh()
    R2, st_p = planned()
    identical = _same_on_device(torch, R1, R2)
    R1.free(); R2.free()
    times = {"multiply": [], "plan_run": []}
    folds = []
    for rep in range(warmup + reps):
        for which, fn in (("multiply", fresh), ("plan_run", planned)):
            a, b = ev(), ev()
            a.record(stream)
            R, st = fn()
            b.record(stream)
            b.synchronize()
            R.free()
            if rep >= warmup:
                times[which].append(a.elapsed_time(b))
                if which == "plan_run":
                    folds.append((st.ms_fold_a, st.ms_fold_b, st.mm.ms_numeric))
    nnz_bound = plan.nnz_bound
    plan.free()
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    mid = lambda i: round(sorted(f[i] for f in folds)[len(folds) // 2], 3)  # noqa: E731
    return {
        "workload": name, "nnz_a": A.size(), "nnz_b": B.size(), "nnz_c": st_p.mm.nnz_c, "nnz_bound": nnz_bound,
        "products": st_p.mm.products, "rows_merge": st_p.mm.rows_merge, "rows_hash": st_p.mm.rows_hash,
        "fresh_rows_esc": st_f.rows_esc, "fresh_rows_hash": st_f.rows_hash,
        "fallback": bool(st_p.fallback), "bit_identical": bool(identical),
        "ms_plan_create": round(t_create, 3),
        "ms_multiply": {"median": round(med["multiply"], 3), "min": round(min(times["multiply"]), 3),
                        "max": round(max(times["multiply"]), 3)},
        "ms_plan_run": {"median": round(med["plan_run"], 3), "min": round(min(times["plan_run"]), 3),
                        "max": round(max(times["plan_run"]), 3)},
        "ms_plan_fold_a_median": mid(0), "ms_plan_fold_b_median": mid(1), "ms_plan_numeric_median": mid(2),
        "fresh_ms_numeric": round(st_f.ms_numeric, 3),
        "speedup_median": round(med["multiply"] / med["plan_run"], 2),
        "reps": reps, "warmup": warmup,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 5 or args.warmup < 1:
        ap.error("at least 5 timed reps after 1 warm-up")
    import torch
    if not torch.cuda.is_available():
        sys.exit("multiply_pattern_probe: needs a CUDA device")
    import spsparse_b200 as sp
    results = {"info": _device_info(torch), "runs": []}
    stream = torch.cuda.Stream()
    with sp.Context(0, stream.cuda_stream) as ctx:
        # config 5 on one GPU: bench.py's seeds and sizes, unsorted A and B
        m = 100_000_000
        A = sp.gen_banded(ctx, 0x5EED0005, m, 0, m)
        B = sp.gen_banded(ctx, 0x5EED0015, m, 0, m)
        w = sp.gen_vector(ctx, 0x5EED0025, m)
        results["runs"].append(probe(sp, torch, ctx, stream, "config5_banded_1e8_rows_A_diag_w_B",
                                     (1.0, None, A, ".", w, B, ".", None), args.reps, args.warmup))
        for x in (A, B, w):
            x.free()
        print(json.dumps(results["runs"][-1]), flush=True)
        # config 3: A * diag(s) * A^T with one values array for both operands
        ny, nx, gy, gx = 3200, 3125, 1000, 1000
        A = sp.gen_regrid(ctx, 0x5EED0003, ny, nx, gy, gx)
        s = sp.gen_vector(ctx, 0x5EED0013, gy * gx)
        results["runs"].append(probe(sp, torch, ctx, stream, "config3_regrid_A_diag_s_AT",
                                     (1.0, None, A, ".", s, A, "T", None), args.reps, args.warmup))
        for x in (A, s):
            x.free()
        print(json.dumps(results["runs"][-1]), flush=True)
        # R-MAT scale 20, A * A
        A = sp.gen_rmat(ctx, 0x5EED0004, 20, 4 << 20)
        results["runs"].append(probe(sp, torch, ctx, stream, "rmat20_A_A", (1.0, None, A, ".", None, A, ".", None),
                                     args.reps, args.warmup))
        A.free()
        print(json.dumps(results["runs"][-1]), flush=True)
    print(json.dumps(results["info"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)
    if not all(r["bit_identical"] for r in results["runs"]):
        sys.exit("multiply_pattern_probe: the plan's output differs from spb_multiply_mm's")


if __name__ == "__main__":
    main()

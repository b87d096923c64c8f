"""Times spb_consolidate against spb_consolidate_plan_run on the config 2 input (gen_dup_coo, 2*10^8 entries, with input
zeros) and on a config 5 block (gen_banded, 10^8 rows), in one process:

    python tools/consolidate_plan_probe.py [--reps 12] [--warmup 2] [--out result.json]

For each input: plan creation is timed once; then the two paths alternate, `warmup` times each untimed and `reps` times
each timed with CUDA events on the library's stream.  The outputs of both paths are compared on the device: index arrays
equal, values equal as bits.  The device name and power limit are read in the same process (query only).  Prints one
JSON object per input and a summary; --out also writes them to a file."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_PEAK = 6.5e12   # bytes/s: the device-to-device copy rate the byte model below is priced at (model only)


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
    """Index arrays equal and values equal as bits (NaN payloads included)."""
    n = R1.size()
    if n != R2.size() or R1.sort_order != R2.sort_order:
        return False
    (i1, v1), (i2, v2) = R1.device_ptrs(), R2.device_ptrs()
    ok = True
    for a, b in zip(i1, i2):
        ok = ok and torch.equal(torch.as_tensor(_View(a, n, "<i4"), device="cuda"), torch.as_tensor(_View(b, n, "<i4"), device="cuda"))
    return ok and torch.equal(torch.as_tensor(_View(v1, n, "<i8"), device="cuda"), torch.as_tensor(_View(v2, n, "<i8"), device="cuda"))


def probe(sp, torch, ctx, stream, name, A, reps, warmup):
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    n = A.size()
    _, val_ptr = A.device_ptrs()
    e0, e1 = ev(), ev()
    e0.record(stream)
    plan = sp.ConsolidatePlan(ctx, A, sp.ROW_MAJOR)
    e1.record(stream)
    e1.synchronize()
    t_create = e0.elapsed_time(e1)

    def fresh():
        return sp.consolidate(ctx, A, sp.ROW_MAJOR, sp.ADD, False, stats=True)

    def planned():
        return plan.run(val_ptr, sp.ADD, False, stats=True)

    # bit-identity at this size, before timing
    R1, st_f = fresh()
    R2, st_p = planned()
    identical = _same_on_device(torch, R1, R2)
    n_kept, n_out = st_p.n_kept, st_p.n_out
    R1.free(); R2.free()
    times = {"consolidate": [], "plan_run": []}
    plan_split = []
    for rep in range(warmup + reps):
        for which, fn in (("consolidate", fresh), ("plan_run", planned)):
            a, b = ev(), ev()
            a.record(stream)
            R, st = fn()
            b.record(stream)
            b.synchronize()
            R.free()
            if rep >= warmup:
                times[which].append(a.elapsed_time(b))
                if which == "plan_run":
                    plan_split.append((st.ms_sort, st.ms_reduce))
    plan.free()
    model_bytes = n * (4 + 8 + 8) + n_kept * (16 + 16) + n_out * 16
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {
        "input": name, "n": n, "n_runs": plan.n_runs, "n_kept": n_kept, "n_out": n_out,
        "bit_identical": bool(identical), "fresh_passes": st_f.passes, "fresh_digit_bits": st_f.digit_bits,
        "ms_plan_create": round(t_create, 3),
        "ms_consolidate": {"median": round(med["consolidate"], 3), "min": round(min(times["consolidate"]), 3),
                           "max": round(max(times["consolidate"]), 3)},
        "ms_plan_run": {"median": round(med["plan_run"], 3), "min": round(min(times["plan_run"]), 3),
                        "max": round(max(times["plan_run"]), 3)},
        "ms_plan_run_gather_median": round(sorted(s for s, _ in plan_split)[len(plan_split) // 2], 3),
        "ms_plan_run_reduce_median": round(sorted(r for _, r in plan_split)[len(plan_split) // 2], 3),
        "speedup_median": round(med["consolidate"] / med["plan_run"], 2),
        "model_bytes": model_bytes, "model_ms_at_copy_peak": round(model_bytes / COPY_PEAK * 1e3, 3),
        "reps": reps, "warmup": warmup,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 10 or args.warmup < 2:
        ap.error("at least 10 timed reps after 2 warm-ups")
    import torch
    if not torch.cuda.is_available():
        sys.exit("consolidate_plan_probe: needs a CUDA device")
    import spsparse_b200 as sp
    results = {"info": _device_info(torch), "runs": []}
    stream = torch.cuda.Stream()
    with sp.Context(0, stream.cuda_stream) as ctx:
        # config 2: 2*10^8 entries over 1.4*10^8 draws in 2^24 x 2^24, every 16th input an explicit zero
        A = sp.gen_dup_coo(ctx, 0x5EED0002, 0, 200_000_000, 140_000_000, 24, 16)
        results["runs"].append(probe(sp, torch, ctx, stream, "config2_dup_coo_2e8_zeros", A, args.reps, args.warmup))
        A.free()
        print(json.dumps(results["runs"][-1]), flush=True)
        # config 5: one banded operand, 10^8 rows x 5 entries
        A = sp.gen_banded(ctx, 0x5EED0005, 100_000_000, 0, 100_000_000)
        results["runs"].append(probe(sp, torch, ctx, stream, "config5_banded_1e8_rows", A, args.reps, args.warmup))
        A.free()
        print(json.dumps(results["runs"][-1]), flush=True)
    print(json.dumps(results["info"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)
    if not all(r["bit_identical"] for r in results["runs"]):
        sys.exit("consolidate_plan_probe: the plan's output differs from spb_consolidate's")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- headline benchmark of the spsparse hot path on B200.

One "step" = one pass of the whole hot path over one batch of synthetic input, here BASELINE
config 5 (the only config BASELINE.json defines at 1, 2, 4 AND 8 GPUs, so the same workload is
measured at every N):  C = A * diag(w) * B  with A, B pentadiagonal 10^8 x 10^8 given as
UNSORTED COO (scrambled insertion order, explicit zeros on the clamped edge diagonals), i.e.
    consolidate(A row block) + consolidate(B row shard) + [NCCL all-gather of B] + SpGEMM.
A is row-partitioned over the ranks, B is replicated once per step by the all-gather, every rank
emits its consolidated row block of C; no collective follows the multiply (strong scaling).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU code (oracle/_ref)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's C to DIR/*.npy

At N=1 the JSON line also carries, under "also", BASELINE config 2 (consolidate of a 200M-entry
COO) and config 3 (regridding SpGEMM), each with its own roofline fraction, and the CPU baseline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S5A, S5B, S5W = 0x5EED0005, 0x5EED0015, 0x5EED0025
S2 = 0x5EED0002
S3, S3S = 0x5EED0003, 0x5EED0013
METRIC = "spgemm_intermediate_products_per_sec"
UNIT = "products/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of one GPU DURING the timed region (B200_PROFILING.md's clocks line).

    Two sources run side by side: NVML polled from a thread every 2 ms (a timed region can be as short as 50 ms at
    8 GPUs, where a 100 ms `nvidia-smi -lms` loop returns nothing) and the recipe's `nvidia-smi` loop.  The NVML
    samples are reported when there are any, the nvidia-smi ones otherwise."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu, uuid=None):
        import threading
        self.p = self.f = self.thread = None
        self.sm, self.reasons, self.smax = [], set(), None
        self.live = threading.Event()   # set by begin(): samples before it are not kept (the sampler is started ahead of the
        self.halt = threading.Event()   # barrier in front of the timed region, so that starting it costs no rank any timed time)
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(uuid or gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:
                h = nv.nvmlDeviceGetHandleByUUID(uuid) if uuid else nv.nvmlDeviceGetHandleByIndex(gpu)
            except (nv.NVMLError, TypeError):
                h = nv.nvmlDeviceGetHandleByIndex(gpu)
            self.smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                    nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                    nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                    nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}

            def poll():
                while not self.halt.is_set():
                    if self.live.is_set():
                        try:
                            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                            for b, nm in bits.items():
                                if r & b:
                                    self.reasons.add(nm)
                        except Exception:  # noqa: BLE001 -- a failed query is a missing sample
                            pass
                    self.halt.wait(0.002)

            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001 -- no NVML: the nvidia-smi loop is the only source
            self.thread = None

    def _smi_samples(self):
        sm, smax, reasons = [], [], set()
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.p.kill()
        if self.f is not None:
            self.f.flush()
            self.f.seek(0)
            for line in self.f.read().splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); smax.append(float(c[2]))
                except ValueError:
                    continue
                for nm, v in zip(self.NAMES, c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            self.f.close()
            os.unlink(self.f.name)
        return sm, (max(smax) if smax else None), reasons

    def begin(self):
        """The timed region starts now."""
        self.live.set()
        return self

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self.thread is not None:
            self.halt.set()
            self.thread.join(timeout=2)
        sm, smax, reasons = self._smi_samples()
        if self.sm:
            out.update(sm_mhz=float(np.median(self.sm)), sm_max_mhz=self.smax, reasons=sorted(self.reasons | reasons),
                       samples=len(self.sm), source="nvml, 2 ms period")
        elif sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(smax), reasons=sorted(reasons), samples=len(sm),
                       source="nvidia-smi -lms 100")
        return out


def gpu_uuid(torch, local):
    """NVML name of the CUDA device `local` (CUDA_VISIBLE_DEVICES may renumber the devices; NVML never does)."""
    try:
        return "GPU-" + str(torch.cuda.get_device_properties(local).uuid)
    except Exception:  # noqa: BLE001
        return None


def bind_to_gpu_numa_node(torch, local):
    """Run this rank on the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of the end-to-end
    leg (first touch) and the threads that feed the copy engines are local to the GPU's PCIe root.  Returns what was
    done (reported under config.numa).  SPB_NO_NUMA_BIND=1 leaves the process where it is."""
    if os.environ.get("SPB_NO_NUMA_BIND"):
        return {"bound": False, "why": "SPB_NO_NUMA_BIND"}
    try:
        pr = torch.cuda.get_device_properties(local)
        dev = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{dev}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return {"bound": False, "why": "no NUMA information for the GPU", "pci": dev}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        have = os.sched_getaffinity(0)
        want = cpus & have
        if not want:
            return {"bound": False, "why": "none of the node's CPUs is available to this process", "node": node, "pci": dev}
        if want != have:
            os.sched_setaffinity(0, want)
        return {"bound": want != have, "node": node, "cpus": len(want), "cpus_before": len(have), "pci": dev}
    except Exception as e:  # noqa: BLE001 -- placement is an optimisation, never a reason to fail
        return {"bound": False, "why": repr(e)}


class DevView:
    """Zero-copy torch view of device memory owned by the library (for NCCL)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    # stdout must carry exactly ONE line (the JSON): NCCL and friends print banners to fd 1, so fd 1 is
    # pointed at stderr for the duration of the run and the line is written to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    import spsparse_b200 as sp

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()
    ctx = sp.Context(local, stream.cuda_stream)
    hbm, peak_src = peaks()
    m = args.rows
    from spsparse_b200.dist import row_range
    r0, r1 = row_range(m, rank, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def launches():
        import ctypes
        n = ctypes.c_uint64()
        ctx.lib.spb_ctx_launch_count(ctx.h, ctypes.byref(n))
        return n.value

    replicator = [None, False]  # (PeerReplicator or None, tried)

    def gather_b_prepare(Bc):
        """Library calls of the replication (main thread only: a context is not re-entrant): views of the
        consolidated shard's arrays and its row pointers."""
        n_local = Bc.size()
        (p0, p1), pv = Bc.device_ptrs()
        dptr = Bc.dense_ptr_range(r0, r1)  # row pointers of this rank's rows [r0, r1) only: O(shard), not O(m)
        local_ptr = torch.as_tensor(DevView(dptr, r1 - r0, "<i4"), device="cuda")
        cols = torch.as_tensor(DevView(p1, n_local, "<i4"), device="cuda")
        vals = torch.as_tensor(DevView(pv, n_local, "<f8"), device="cuda")
        return local_ptr, cols, vals

    def gather_b_start(shard, need=None):
        """Start replicating the row-sharded, consolidated B on every rank (spsparse_b200/dist.py), in
        compressed form: local row pointers of this rank's rows + column and value of every entry.
        Asynchronous, so that consolidate(A) overlaps the transfers."""
        from spsparse_b200 import dist as spd
        local_ptr, cols, vals = shard
        if not replicator[1]:
            replicator[1] = True
            if not os.environ.get("SPB_NO_PEER_COPY"):
                try:
                    replicator[0] = spd.PeerReplicator(rank, world, 5 * (r1 - r0), r1 - r0, torch.device("cuda", local))
                except Exception as e:  # noqa: BLE001 -- any failure: use the NCCL path
                    print(f"[bench] symmetric-memory replication unavailable ({e!r}); using NCCL all-gather", file=sys.stderr)
        if replicator[0] is not None:
            return replicator[0].start(local_ptr, cols, vals, None if os.environ.get("SPB_FULL_REPLICATE") else need)
        return spd.replicate_csr_start(local_ptr, cols, vals, rank, world)

    fetch_ms = []  # per step: (fetch kernel, whole side stream) in ms
    timeline = []  # per step: stream-event times (ms) between the phases of the hot path
    pulled = [None]  # rows of B this rank fetched in the last step (None: everything)
    # The row-partitioned multiply behind the C ABI (spb_rowpart_*): shards of B published / fetched through peer-mapped
    # memory by the library's own kernels, no host round trip inside a step.  SPB_LEGACY_DIST=1: the round-1 path
    # (torch symmetric memory + copy engines driven from Python, spsparse_b200/dist.py), kept for A/B runs.
    rowpart = [None]
    mode = {"fetch_all": bool(os.environ.get("SPB_FULL_REPLICATE"))}
    if not os.environ.get("SPB_LEGACY_DIST"):
        from spsparse_b200.dist import RowPartition
        rows_max = max(row_range(m, g, world)[1] - row_range(m, g, world)[0] for g in range(world))
        rowpart[0] = RowPartition(ctx, rank, world, m, 5 * rows_max + 16)

    def hot_path(A_raw, B_raw, w, before_a=None):
        """consolidate(B shard) -> [replicate B, overlapped with] consolidate(A block) -> SpGEMM.
        before_a: called before the first use of A (the end-to-end run makes the stream wait for A's upload there)."""
        from spsparse_b200 import dist as spd
        if rowpart[0] is not None:
            if before_a is not None:
                before_a()
            Cm, rs = rowpart[0].multiply(1.0, None, A_raw, w, B_raw, None, fetch_all=mode["fetch_all"])
            pulled[0] = int(rs.rows_fetched)
            spg = rs.mm.ms_total
            other = rs.ms_total - (rs.ms_consolidate_b + rs.ms_consolidate_a + rs.ms_fetch_wait + spg)
            timeline.append([rs.ms_consolidate_b, other, rs.ms_consolidate_a, rs.ms_fetch_wait, spg])
            fetch_ms.append((rs.ms_fetch, rs.ms_side_stream))
            return Cm, (rs.a, rs.b, rs.mm)   # views into rs (ctypes keeps it alive)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record(stream)
        Bc, sb = sp.consolidate(ctx, B_raw, sp.ROW_MAJOR, stats=True)
        ev[1].record(stream)
        pending = None
        if before_a is not None:
            before_a()
        if world > 1:
            # interval hull of the inner indices this rank's block of A references: only those rows of B are fetched.
            # (Starting the replication from a helper thread, so that its host round trips overlap consolidate(A), was
            # tried: kernels of the second stream then waited for the sort on one of the ranks; see profiles/r01_notes.md.)
            (_, a1), _ = A_raw.device_ptrs()
            lo, hi = torch.aminmax(torch.as_tensor(DevView(a1, A_raw.size(), "<i4"), device="cuda"))
            pending = gather_b_start(gather_b_prepare(Bc), (int(lo.item()), int(hi.item())))
        ev[2].record(stream)
        Ac, sa = sp.consolidate(ctx, A_raw, sp.ROW_MAJOR, stats=True)
        ev[3].record(stream)
        if pending:
            pulled[0] = pending.get("pulled_rows")
            ptr, cols, vals, total = spd.replicate_csr_finish(pending)  # library stream now waits for NCCL
            Bf = sp.CooArray.wrap_csr(ctx, (m, m), 0, ptr.data_ptr(), cols.data_ptr(), vals.data_ptr(), total)
        else:
            Bf = Bc
        ev[4].record(stream)
        Cm, st = sp.multiply_prepared(ctx, 1.0, None, Ac, 0, w, Bf, 0, None)
        ev[5].record(stream)
        stream.synchronize()
        timeline.append([ev[i].elapsed_time(ev[i + 1]) for i in range(5)])
        if Bf is not Bc:
            Bf.free()
            del pending, ptr, cols, vals
        Ac.free(); Bc.free()
        return Cm, (sa, sb, st)

    with torch.cuda.stream(stream):
        A_raw = sp.gen_banded(ctx, S5A, m, r0, r1)
        B_raw = sp.gen_banded(ctx, S5B, m, r0, r1)
        w = sp.gen_vector(ctx, S5W, m)
        ctx.sync()
        nA, nB = A_raw.size(), B_raw.size()

        # ---------------- device-resident timing (value) -----------------------------------------
        for _ in range(args.warmup):
            Cm, _ = hot_path(A_raw, B_raw, w)
            Cm.free()
        # the clock sampler (rank 0: an nvidia-smi child process and an NVML thread) is STARTED before the barrier: starting it
        # after the barrier delayed rank 0's first timed step by the fork + NVML initialisation (5 ... 130 ms measured), and at
        # N > 1 the other ranks -- whose clocks were already running -- spent that time waiting for rank 0's shard
        sampler = ClockSampler(local, gpu_uuid(torch, local)) if rank == 0 else None
        barrier()
        l0 = launches()
        if sampler:
            sampler.begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acc = []
        e0.record(stream)
        for k in range(args.steps):
            Cm, sts = hot_path(A_raw, B_raw, w)
            acc.append(sts)
            if k < args.steps - 1 or not args.dump_outputs:
                Cm.free()
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if sampler else None
        l1 = launches()
        if args.dump_outputs:
            dump_result(torch, Cm, args.dump_outputs, rank, world)
            Cm.free()
        # partition-independent fingerprints of C (one extra, untimed step): exact wrap-around checksum of the
        # index structure and the fp64 sum of the values -- equal at every N if the row blocks tile C correctly
        Cm, _ = hot_path(A_raw, B_raw, w)
        (c0, c1), cv = Cm.device_ptrs()
        nc = Cm.size()
        ti = torch.as_tensor(DevView(c0, nc, "<i4"), device="cuda").to(torch.int64)
        tk = torch.as_tensor(DevView(c1, nc, "<i4"), device="cuda").to(torch.int64)
        fp = torch.stack([(ti * 1000003 + tk).sum(), torch.tensor(nc, device="cuda")])
        vsum = torch.as_tensor(DevView(cv, nc, "<f8"), device="cuda").sum().reshape(1)
        if world > 1:
            dist.all_reduce(fp, op=dist.ReduceOp.SUM)
            dist.all_reduce(vsum, op=dist.ReduceOp.SUM)
        fingerprint = {"index_checksum": int(fp[0].item()), "nnz_c": int(fp[1].item()), "value_sum": float(vsum.item())}
        del ti, tk
        Cm.free()
        ms = e0.elapsed_time(e1) / args.steps
        # N > 1: the same step with ALL of B fetched by every rank (what a general, non-banded matrix needs: the
        # north-star's "B replicated once"), timed the same way, reported under also.full_replicate
        full_rep = None
        if world > 1 and rowpart[0] is not None and not mode["fetch_all"] and not args.no_also:
            mode["fetch_all"] = True
            n_tl = len(timeline)
            for _ in range(2):
                Cx, _ = hot_path(A_raw, B_raw, w); Cx.free()
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for _ in range(args.steps):
                Cx, fsts = hot_path(A_raw, B_raw, w); Cx.free()
            f1.record(stream)
            barrier()
            tf = torch.tensor([f0.elapsed_time(f1) / args.steps], dtype=torch.float64, device="cuda")
            dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            full_rep = {"ms_per_step": float(tf.item()), "rows_fetched_rank0": pulled[0],
                        "timeline_ms_rank0": dict(zip(["consolidate_b", "publish_and_gaps", "consolidate_a", "fetch_wait", "spgemm_incl_prepare"],
                                                      [float(x) for x in np.mean(np.array(timeline[n_tl + 2:]), axis=0)])),
                        "fetch_kernel_ms_rank0": float(np.mean([f[0] for f in fetch_ms[-args.steps:]]))}
            del timeline[n_tl:]
            mode["fetch_all"] = False
            Cx, _ = hot_path(A_raw, B_raw, w); Cx.free()   # pulled[0] back to what the headline run fetches
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        # every rank's own step time and phase times (the headline takes the maximum; the spread shows where a rank waits)
        per_rank = None
        if world > 1:
            mine = torch.tensor([ms] + [float(x) for x in np.mean(np.array(timeline[args.warmup:args.warmup + args.steps]), axis=0)],
                                dtype=torch.float64, device="cuda")
            allr = torch.zeros(world * mine.numel(), dtype=torch.float64, device="cuda")
            dist.all_gather_into_tensor(allr, mine)
            allr = allr.view(world, -1).cpu().numpy()
            per_rank = {"ms_per_step": [float(x) for x in allr[:, 0]],
                        "phases_ms": {k: [float(x) for x in allr[:, 1 + i]] for i, k in enumerate(
                            ["consolidate_b", "publish_and_gaps", "consolidate_a", "replicate_b_wait", "spgemm_incl_prepare"])}}
        sa, sb, st = acc[-1]
        cnt = torch.tensor([st.products, st.nnz_c, sa.n_out + sb.n_out, nA + nB], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        ms = float(t.item())
        F, nnzC, cons_out, cons_in = (float(x) for x in cnt.tolist())
        value = F / (ms * 1e-3)
        if full_rep is not None:
            full_rep["value"] = F / (full_rep["ms_per_step"] * 1e-3)
            full_rep["unit"] = UNIT

        # per-phase means on this rank
        ms_cons = float(np.mean([a.ms_total + b.ms_total for a, b, _ in acc]))
        ms_pass = float(np.mean([a.ms_pass for a, _, _ in acc]))
        ms_spgemm = float(np.mean([s.ms_symbolic + s.ms_numeric for _, _, s in acc]))
        ms_prep = float(np.mean([s.ms_prepare for _, _, s in acc]))
        pass_bytes = 32.0 * sa.n_kept  # one radix pass: read 8B key + 8B value, write both
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
        if os.path.exists(tp):  # dram__bytes_read+write of this kernel from an `ncu --set full` capture of this command
            tj = json.load(open(tp))
            tj = tj.get("k_radix_pass9" if sa.digit_bits == 9 else "k_radix_pass", tj if "dram_bytes_per_entry" in tj else None)
            if tj:
                traffic = tj["dram_bytes_per_entry"] * sa.n_kept
                traffic_src = (f"{tj['dram_bytes_per_entry']:.2f} B/entry measured by ncu ({tj['kernel']}, {tj['entries_per_launch']} entries/launch, "
                               f"{tj['report']})")
        pass_gbs = pass_bytes / (ms_pass * 1e-3) / 1e9 if ms_pass > 0 else 0.0
        spgemm_bytes = 16.0 * st.products + 56.0 * st.nnz_a + 16.0 * st.nnz_c + 16.0 * st.rows_a
        # BASELINE.md section 4: P = ceil(key bits / 8) passes of the MODEL, whatever the implementation runs
        cons_bytes = lambda s: s.n_in * (8 + 16) + 32.0 * s.n_kept * (-(-s.key_bits // 8)) + 16.0 * s.n_out  # noqa: E731

        # ---------------- end to end through the C ABI with HOST buffers (e2e) -----------------------
        e2e = None
        if not args.no_e2e:
            def pinned(n, dt):
                return torch.empty(max(int(n), 1), dtype=dt, pin_memory=True)
            hA = [pinned(nA, torch.int32), pinned(nA, torch.int32), pinned(nA, torch.float64)]
            hB = [pinned(nB, torch.int32), pinned(nB, torch.int32), pinned(nB, torch.float64)]
            wi, wv = w.to_host()
            A_raw.to_host(out=([hA[0].numpy()[:nA], hA[1].numpy()[:nA]], hA[2].numpy()[:nA]))
            B_raw.to_host(out=([hB[0].numpy()[:nB], hB[1].numpy()[:nB]], hB[2].numpy()[:nB]))
            # scalej: a rank only needs the entries of w whose index its block of A can reference (an index absent from a
            # scale vector excludes that term, multiply_sparse.hpp:79-92 -- and no entry of the block has such an index), so
            # it uploads that slice, not all 10^8 entries: found once from the host copy of the block's column indices
            jlo, jhi = (int(hA[1].numpy()[:nA].min()), int(hA[1].numpy()[:nA].max())) if nA else (0, -1)
            mW = jhi - jlo + 1
            hW = [pinned(mW, torch.int32), pinned(mW, torch.float64)]
            hW[0].numpy()[:mW] = wi[0][jlo:jhi + 1]; hW[1].numpy()[:mW] = wv[jlo:jhi + 1]
            ncap = int(st.nnz_c)
            hC = [pinned(ncap, torch.int32), pinned(ncap, torch.int32), pinned(ncap, torch.float64)]
            A_raw.free(); B_raw.free(); w.free()

            # Software pipeline over the steps (double-buffered device inputs): the H2D copies of step k+1 run on
            # a copy stream while step k computes, and the D2H copy of C(k) runs on a third stream while step k+1
            # computes.  PCIe is full duplex, so uploads and downloads overlap too.  Every step still moves all of
            # its inputs host->device and all of its result device->host inside the timed region.
            up, down_s = torch.cuda.Stream(), torch.cuda.Stream()
            dev_in = [[torch.empty(nA, dtype=torch.int32, device="cuda"), torch.empty(nA, dtype=torch.int32, device="cuda"),
                       torch.empty(nA, dtype=torch.float64, device="cuda"),
                       torch.empty(nB, dtype=torch.int32, device="cuda"), torch.empty(nB, dtype=torch.int32, device="cuda"),
                       torch.empty(nB, dtype=torch.float64, device="cuda"),
                       torch.empty(max(mW, 1), dtype=torch.int32, device="cuda"), torch.empty(max(mW, 1), dtype=torch.float64, device="cuda")]
                      for _ in range(2)]
            host_in = [hA[0][:nA], hA[1][:nA], hA[2][:nA], hB[0][:nB], hB[1][:nB], hB[2][:nB], hW[0][:max(mW, 1)], hW[1][:max(mW, 1)]]
            ready = [torch.cuda.Event(), torch.cuda.Event()]      # B and w of the slot are on the device
            ready_a = [torch.cuda.Event(), torch.cuda.Event()]    # ... and A (uploaded last: consolidate(B) starts under it)
            freed = [torch.cuda.Event(), torch.cuda.Event()]
            state = {"prev_c": None, "prev_done": None}

            def enqueue_upload(k):
                s_ = k % 2
                up.wait_event(freed[s_])
                with torch.cuda.stream(up):
                    for j in (3, 4, 5, 6, 7):
                        dev_in[s_][j].copy_(host_in[j], non_blocking=True)
                    ready[s_].record(up)
                    for j in (0, 1, 2):
                        dev_in[s_][j].copy_(host_in[j], non_blocking=True)
                    ready_a[s_].record(up)

            def run_steps(count):
                nc_last = 0
                for s_ in range(2):
                    freed[s_].record(stream)
                enqueue_upload(0)
                for k in range(count):
                    if k + 1 < count:
                        enqueue_upload(k + 1)
                    s_ = k % 2
                    stream.wait_event(ready[s_])
                    d = dev_in[s_]
                    a = sp.CooArray.wrap_device(ctx, (m, m), [d[0].data_ptr(), d[1].data_ptr()], d[2].data_ptr(), nA)
                    b = sp.CooArray.wrap_device(ctx, (m, m), [d[3].data_ptr(), d[4].data_ptr()], d[5].data_ptr(), nB)
                    ww = sp.CooArray.wrap_device(ctx, (m,), [d[6].data_ptr()], d[7].data_ptr(), mW, (0,))
                    Cm, _ = hot_path(a, b, ww, before_a=lambda: stream.wait_event(ready_a[s_]))
                    freed[s_].record(stream)
                    for x in (a, b, ww):
                        x.free()
                    n = Cm.size()
                    (c0, c1), cv = Cm.device_ptrs()
                    if state["prev_c"] is not None:   # the previous result has left the device: release it
                        state["prev_done"].synchronize()
                        state["prev_c"].free()
                    down_s.wait_stream(stream)
                    with torch.cuda.stream(down_s):
                        hC[0][:n].copy_(torch.as_tensor(DevView(c0, n, "<i4"), device="cuda"), non_blocking=True)
                        hC[1][:n].copy_(torch.as_tensor(DevView(c1, n, "<i4"), device="cuda"), non_blocking=True)
                        hC[2][:n].copy_(torch.as_tensor(DevView(cv, n, "<f8"), device="cuda"), non_blocking=True)
                        done = torch.cuda.Event()
                        done.record(down_s)
                    state["prev_c"], state["prev_done"] = Cm, done
                    nc_last = n
                state["prev_done"].synchronize()
                state["prev_c"].free()
                state["prev_c"] = None
                return nc_last

            run_steps(min(args.warmup, 3))
            barrier()
            e0.record(stream)
            nc = run_steps(args.steps)
            torch.cuda.synchronize()
            e1.record(stream)
            barrier()
            # the bytes that came back must be the same C the device-resident run produced
            with np.errstate(over="ignore"):
                hchk = int((hC[0].numpy()[:nc].astype(np.int64) * 1000003 + hC[1].numpy()[:nc]).sum())
            hv = torch.tensor([hchk, nc], dtype=torch.int64, device="cuda")
            if world > 1:
                dist.all_reduce(hv, op=dist.ReduceOp.SUM)
            e2e_ok = (int(hv[0].item()) == fingerprint["index_checksum"]) and (int(hv[1].item()) == fingerprint["nnz_c"])
            ems = e0.elapsed_time(e1) / args.steps
            t = torch.tensor([ems], dtype=torch.float64, device="cuda")
            b = torch.tensor([16.0 * nA + 16.0 * nB + 12.0 * mW, 16.0 * nc], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dist.all_reduce(b, op=dist.ReduceOp.SUM)
            e2e = {"value": F / (float(t.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(t.item()),
                   "h2d_bytes_per_step": float(b[0].item()), "d2h_bytes_per_step": float(b[1].item()),
                   "result_matches_device_run": bool(e2e_ok),
                   "api": "pinned host buffers -> async H2D -> spb_coo_wrap_device + spb_consolidate x2 + spb_multiply_mm_prepared -> async D2H; steps software-pipelined (upload of step k+1 and download of step k overlap step k's kernels)"}
            if rank == 0 and world == 1:
                e2e.update(e2e_other_apis(ctx, sp, torch, args, m, hA, hB, (wi[0], wv), nA, nB, fingerprint))
            del hA, hB, hC
        else:
            A_raw.free(); B_raw.free(); w.free()

        also, cpu = {}, None
        if rank == 0 and world == 1 and not args.no_also:
            also = also_configs(ctx, sp, torch, stream, args, hbm)
        if rank == 0 and full_rep is not None:
            also = dict(also, full_replicate=full_rep)
        if rank == 0 and world == 1 and e2e is not None:
            e2e["cpp_api"] = e2e_cpp_api(ctx, torch, args, m, fingerprint)
        if rank == 0 and world == 1 and not args.no_cpu:
            cpu = cpu_baseline(args)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "BASELINE config 5: banded 1e8-row triple product A*diag(w)*B from unsorted COO "
                                   "(consolidate A + consolidate B + replicate the needed rows of B + SpGEMM)" if m == 100_000_000 else
                                   f"REDUCED banded triple product, {m} rows (not the headline size)",
                       "rows": m, "nnz_a_raw": cons_in / 2, "nnz_c": nnzC, "products": F,
                       "partition": f"A rows / B rows split over {world} rank(s); each step every rank fetches, in compressed form (row pointers + cols + vals, 12 B/entry), the rows of B inside the interval hull of the inner indices its block of A references (rank 0 fetched {pulled[0] if pulled[0] is not None else m} of {m} rows; a block whose columns span everything fetches all of B = the plain replicate, SPB_FULL_REPLICATE=1 forces it and also.full_replicate times it): " + ("fetched by the library's own kernel with loads from the peers' memory (CUDA IPC over NVLink; spb_rowpart_multiply), no host round trip inside a step, overlapped with consolidate(A)" if rowpart[0] is not None else "pulled from the peers' symmetric memory over NVLink by copy engines (SPB_LEGACY_DIST path)"),
                       "l2": "inputs (>= 2 GB per rank) are far larger than the 126 MB L2; no flush needed",
                       "index_type": "int32", "value_type": "f64", "result_fingerprint": fingerprint, "numa_rank0": numa},
            "phases_rank0": {"ms_consolidate_a_plus_b": ms_cons, "ms_spgemm_symbolic_plus_numeric": ms_spgemm,
                             "ms_spgemm_prepare": ms_prep,
                             "consolidate_nnz_per_sec": (sa.n_out + sb.n_out) / (ms_cons * 1e-3),
                             "consolidate_entries_in_per_sec": (nA + nB) / (ms_cons * 1e-3),
                             "consolidate_model_frac": (cons_bytes(sa) + cons_bytes(sb)) / (ms_cons * 1e-3) / 1e9 / hbm,
                             "spgemm_products_per_sec": st.products / (ms_spgemm * 1e-3),
                             "spgemm_model_bytes": spgemm_bytes,
                             "spgemm_model_frac": spgemm_bytes / (ms_spgemm * 1e-3) / 1e9 / hbm,
                             "rows_merge": st.rows_merge, "rows_esc": st.rows_esc,
                             "timeline_ms": dict(zip(["consolidate_b", "publish_and_gaps" if rowpart[0] is not None else "replicate_b_launch", "consolidate_a", "replicate_b_wait",
                                                      "spgemm_incl_prepare"],
                                                     [float(x) for x in np.mean(np.array(timeline[args.warmup:args.warmup + args.steps]), axis=0)]))},
            "per_rank": per_rank,
            "roofline": {"bound": "hbm", "kernel": ("k_radix_pass9<false, BULK> (one 9-bit LSD scatter pass, key+value)" if sa.digit_bits == 9 else
                                                    "k_radix_pass<false, BULK> (one 8-bit LSD scatter pass, key+value)"),
                         "achieved": pass_gbs, "peak": hbm, "unit": "GB/s", "frac": pass_gbs / hbm,
                         "traffic": traffic, "traffic_source": traffic_src, "bytes_per_launch": pass_bytes, "ms_per_launch": ms_pass,
                         "peak_source": peak_src,
                         "note": ("9-bit digits: three passes over the 27-bit row part instead of four 8-bit ones (a 9-bit pass costs 10 % more "
                                  "than an 8-bit one, three of them less than four); tiles loaded by cp.async.bulk + mbarrier "
                                  "(profiles/r02_notes.md)") if sa.digit_bits == 9 else None,
                         # the other kernels of a consolidate with a time of their own in spb_consolidate_stats
                         "reduce_pass": kernel_roofline("k_reduce_warp<false> (duplicate-reduce, a warp per 256-entry tile, tile offsets from the in-row sort's head counts: "
                                                        "16 B per entry read, 16 B per output written)" if os.environ.get("SPB_REDUCE_WARP", "1") == "1" else
                                                        "k_reduce_by_key / k_reduce_warp<true> (SPB_REDUCE_WARP set: look-back variants)",
                                                        "k_reduce_warp", 16.0 * sa.n_kept + 16.0 * sa.n_out, sa.ms_reduce, hbm, sa.n_kept)},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(l1 - l0),
            "clocks": clocks,
            "also": also,
        }
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    ctx.sync()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_ENTRIES = 1 << 21   # 3 arrays x 8 B x 2^21 entries = 48 MB over all ranks, under the 64 MB a dump may take
DUMP_SEED = 0x5EED00D0


def dump_result(torch, Cm, out_dir, rank, world):
    """--dump-outputs: the C of the timed path's last step, as a caller receives it, written as <out_dir>/C_row.npy,
    C_col.npy and C_val.npy in float64 (int32 indices are exact in it).  At N > 1 every rank writes its own row block,
    with a .rank<r> suffix, and takes an equal share of the DUMP_ENTRIES entries.  A block larger than its share is
    sampled at positions drawn with a fixed seed, in order: the same positions for the same nnz, so two builds can be
    compared entry for entry."""
    os.makedirs(out_dir, exist_ok=True)
    nc = Cm.size()
    share = DUMP_ENTRIES // world
    (c0, c1), cv = Cm.device_ptrs()
    pos = None
    if nc > share:
        pos = torch.as_tensor(np.sort(np.random.default_rng(DUMP_SEED).choice(nc, share, replace=False)), device="cuda")
    suffix = f".rank{rank}" if world > 1 else ""
    for name, ptr, typestr in (("C_row", c0, "<i4"), ("C_col", c1, "<i4"), ("C_val", cv, "<f8")):
        if nc == 0:
            a = np.empty(0, np.float64)
        else:
            t = torch.as_tensor(DevView(ptr, nc, typestr), device="cuda")
            a = (t if pos is None else t[pos]).to(torch.float64).cpu().numpy()
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def e2e_other_apis(ctx, sp, torch, args, m, hA, hB, w_host, nA, nB, fingerprint):
    """The same step end to end through the entry points a user of the reference binds, with PAGEABLE host memory (what
    std::vector is), beside the pinned + pre-wrapped pipeline above:
      cabi_pageable  spb_coo_upload x3 -> spb_multiply_mm -> spb_coo_download, plain numpy arrays, nothing overlapped
                     across steps; the library moves pageable memory with worker threads through pinned staging buffers
      cpp_api        spsparse::multiply(C, 1.0, NULL, A, '.', &w, B, '.', NULL) on VectorCooArrays (include/spsparse/), a
                     C++ program of its own (tools/cpp/e2e_multiply.cpp) -- the reference's own entry point"""
    import ctypes
    out = {}
    F = fingerprint
    a = [np.array(t.numpy()[:nA]) for t in hA]          # pageable copies
    b = [np.array(t.numpy()[:nB]) for t in hB]
    wi, wv = np.ascontiguousarray(w_host[0]), np.ascontiguousarray(w_host[1])
    ms = []
    ok = True
    for it in range(1 + min(args.steps, 2)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dA = sp.CooArray.from_host(ctx, (m, m), a[:2], a[2])
        dB = sp.CooArray.from_host(ctx, (m, m), b[:2], b[2])
        dW = sp.CooArray.from_host(ctx, (m,), [wi], wv, (0,))
        Cm = sp.multiply(ctx, 1.0, None, dA, ".", dW, dB, ".", None)
        idx, val = Cm.to_host()
        dt = time.perf_counter() - t0
        for x in (dA, dB, dW, Cm):
            x.free()
        if it:
            ms.append(dt * 1e3)
        with np.errstate(over="ignore"):
            chk = int((idx[0].astype(np.int64) * 1000003 + idx[1]).sum())
        ok = ok and chk == F["index_checksum"] and len(val) == F["nnz_c"]
        del idx, val
    out["cabi_pageable"] = {"ms_per_step": float(np.mean(ms)), "value": 25.0 * m / (float(np.mean(ms)) * 1e-3), "unit": UNIT,
                            "h2d_bytes_per_step": 16.0 * nA + 16.0 * nB + 12.0 * m, "d2h_bytes_per_step": 16.0 * F["nnz_c"],
                            "result_matches_device_run": bool(ok), "steps": len(ms),
                            "api": "pageable numpy arrays -> spb_coo_upload x3 -> spb_multiply_mm (consolidates A and B itself) -> spb_coo_download; one step at a time"}
    del a, b
    return out


def e2e_cpp_api(ctx, torch, args, m, fingerprint):
    """The C++-API leg of the end-to-end measurement (see e2e_other_apis); run last: it needs the device memory this
    process has cached, which is handed back to the driver first."""
    import ctypes
    out = {}
    F = fingerprint
    exe = os.path.join(ROOT, "tests", "cpp", "_bin", "e2e_multiply")
    if os.path.exists(exe):
        rel = ctypes.c_uint64()
        ctx.lib.spb_ctx_trim(ctx.h, ctypes.byref(rel))   # the other process needs the device memory this one has cached
        torch.cuda.empty_cache()
        try:
            r = subprocess.run([exe, str(m), str(min(args.steps, 2)), "1"], capture_output=True, text=True, timeout=900,
                               env=dict(os.environ, SPSPARSE_B200_DEVICE=str(ctx.device)))
            j = json.loads(r.stdout.strip().splitlines()[-1])
            out["cpp_api"] = {"ms_per_step": j["ms_per_step"], "ms_best": j["ms_best"], "value": 25.0 * m / (j["ms_per_step"] * 1e-3), "unit": UNIT,
                              "h2d_bytes_per_step": j["h2d_bytes_per_step"], "d2h_bytes_per_step": j["d2h_bytes_per_step"],
                              "result_matches_device_run": (j["index_checksum"] - F["index_checksum"]) % (1 << 64) == 0 and j["nnz_c"] == F["nnz_c"],
                              "steps": min(args.steps, 2),
                              "api": "spsparse::multiply(C, 1.0, NULL, A, '.', &w, B, '.', NULL) on VectorCooArray<int,double,2> (std::vector storage), include/spsparse/; tools/cpp/e2e_multiply.cpp"}
        except Exception as e:  # noqa: BLE001 -- a missing leg is reported, not fatal
            out["cpp_api"] = {"unavailable": repr(e)[:300]}
    return out.get("cpp_api")


def kernel_roofline(kernel, key, algo_bytes, ms, hbm, units=None, unit_name=None):
    """Roofline sub-block of one config's dominant kernel: algorithmic bytes of a launch / its duration (CUDA events inside the
    library) against the measured copy peak, and -- when profiles/r02_ncu_traffic.json has a capture of that kernel -- the DRAM
    bytes ncu measured, scaled to this launch by the capture's bytes per unit."""
    blk = {"kernel": kernel, "bound": "hbm", "bytes_per_launch": float(algo_bytes), "ms_per_launch": float(ms),
           "achieved": float(algo_bytes) / (ms * 1e-3) / 1e9 if ms > 0 else 0.0, "peak": hbm, "unit": "GB/s", "traffic": None}
    blk["frac"] = blk["achieved"] / hbm
    tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp)).get(key)
        if tj and units is not None and "dram_bytes_per_" + (unit_name or "entry") in tj:
            blk["traffic"] = tj["dram_bytes_per_" + (unit_name or "entry")] * units
            blk["traffic_source"] = f"{tj['dram_bytes_per_' + (unit_name or 'entry')]:.2f} B per {unit_name or 'entry'} measured by ncu ({tj.get('report')})"
    return blk


def also_configs(ctx, sp, torch, stream, args, hbm):
    """BASELINE configs 2, 3 and 4 on one GPU (device-resident inputs, CUDA events on the library stream)."""
    out = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # ---- config 2: consolidate 200M entries, ~30% duplicates, 2^24 x 2^24 ----------------------------
    n, ub = args.cons_entries, int(args.cons_entries * 0.7)
    A = sp.gen_dup_coo(ctx, S2, 0, n, ub, 24, 0)
    ctx.sync()
    for _ in range(args.warmup):
        R = sp.consolidate(ctx, A, sp.ROW_MAJOR); R.free()
    sts = []
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(args.steps):
        R, st = sp.consolidate(ctx, A, sp.ROW_MAJOR, stats=True)
        sts.append(st)
        if _ == args.steps - 1:
            idx, val = R.to_host() if n <= 200_000_000 else (None, None)
        R.free()
    e1.record(stream)
    torch.cuda.synchronize()
    st = sts[-1]
    ms_k = float(np.mean([s.ms_total for s in sts]))
    model = n * (8.0 + 32.0 * (-(-st.key_bits // 8)) + 16.0) + 16.0 * st.n_out  # BASELINE.md section 4 (P = ceil(K/8))
    out["consolidate_config2"] = {
        "workload": f"BASELINE config 2: consolidate {n} unsorted COO entries, 2^24 x 2^24, ~30% duplicates",
        "n_in": n, "nnz_out": st.n_out, "passes": st.passes, "passes_model": -(-st.key_bits // 8), "key_bits": st.key_bits,
        "passes_note": "radix passes executed; when the column part of the key is two or more digits wide the passes cover the row part only and one in-row column sort (k_segment_sort) replaces the rest, so fewer bytes move than the model's P = ceil(K/8) passes assume",
        "ms_kernels": ms_k, "ms_sort": float(np.mean([s.ms_sort for s in sts])),
        "ms_reduce": float(np.mean([s.ms_reduce for s in sts])), "ms_pass": float(np.mean([s.ms_pass for s in sts])),
        "consolidate_nnz_per_sec": st.n_out / (ms_k * 1e-3), "entries_in_per_sec": n / (ms_k * 1e-3),
        "model_bytes": model, "model_frac": model / (ms_k * 1e-3) / 1e9 / hbm,
        "compulsory_frac": (16.0 * n + 16.0 * st.n_out) / (ms_k * 1e-3) / 1e9 / hbm,
        "pass_gbs": 32.0 * st.n_kept / (float(np.mean([s.ms_pass for s in sts])) * 1e-3) / 1e9,
        "first_entry": [int(idx[0][0]), int(idx[1][0])] if idx is not None else None,
        "sum_values": float(val.sum()) if val is not None else None,
        "roofline": kernel_roofline(f"k_radix_pass{'9' if st.digit_bits == 9 else ''}<false, BULK> ({st.passes - 1} of its {st.passes} scatter passes; pass 0 reads the caller's arrays)",
                                    "k_radix_pass9" if st.digit_bits == 9 else "k_radix_pass", 32.0 * st.n_kept,
                                    float(np.mean([s.ms_pass for s in sts])), hbm, st.n_kept),
        "roofline_reduce": kernel_roofline("k_reduce_warp<false> (16 B per entry read, 16 B per output written)", "k_reduce_warp",
                                           16.0 * st.n_kept + 16.0 * st.n_out, float(np.mean([s.ms_reduce for s in sts])), hbm, st.n_kept),
    }
    A.free()
    # ---- config 3: regridding SpGEMM  C = A diag(s) A^T, A = 1e7 x 1e6 ---------------------------------
    ny, nx, gy, gx = args.regrid
    A = sp.gen_regrid(ctx, S3, ny, nx, gy, gx)
    s = sp.gen_vector(ctx, S3S, gy * gx)
    Ar = sp.consolidate(ctx, A, sp.ROW_MAJOR)   # op(A) rows
    Bt = sp.consolidate(ctx, A, sp.COL_MAJOR)   # op(B) = A^T bucketed by its inner index (= column of A)
    for _ in range(args.warmup):
        Cm, st = sp.multiply_prepared(ctx, 1.0, None, Ar, 0, s, Bt, 1, None); Cm.free()
    sts = []
    for _ in range(args.steps):
        Cm, st = sp.multiply_prepared(ctx, 1.0, None, Ar, 0, s, Bt, 1, None)
        sts.append(st); Cm.free()
    ms_k = float(np.mean([x.ms_symbolic + x.ms_numeric for x in sts]))
    model = 16.0 * st.products + 56.0 * st.nnz_a + 16.0 * st.nnz_c + 16.0 * st.rows_a
    out["spgemm_config3"] = {
        "workload": f"BASELINE config 3: regridding A*diag(s)*A^T, A {ny * nx} x {gy * gx}, 4 nnz/row",
        "products": st.products, "nnz_a": st.nnz_a, "nnz_c": st.nnz_c, "rows_merge": st.rows_merge, "rows_esc": st.rows_esc,
        "ms_symbolic": float(np.mean([x.ms_symbolic for x in sts])), "ms_numeric": float(np.mean([x.ms_numeric for x in sts])),
        "ms_prepare": float(np.mean([x.ms_prepare for x in sts])),
        "products_per_sec": st.products / (ms_k * 1e-3), "nnz_c_per_sec": st.nnz_c / (ms_k * 1e-3),
        "model_bytes": model, "model_frac": model / (ms_k * 1e-3) / 1e9 / hbm,
        "compulsory_frac": (12.0 * st.nnz_a + 12.0 * st.nnz_b + 8.0 * gy * gx + 16.0 * st.nnz_c) / (ms_k * 1e-3) / 1e9 / hbm,
        "roofline": kernel_roofline("k_merge_numeric<4, 16> (register k-way merge, numeric pass: 12 B per product read, 16 B per output written)",
                                    "k_merge_numeric", 12.0 * st.products + 16.0 * st.nnz_c,
                                    float(np.mean([x.ms_merge_numeric for x in sts])), hbm, st.nnz_c, "output"),
    }
    for x in (A, s, Ar, Bt):
        x.free()
    # ---- config 4: R-MAT A*A, full multiply() incl. its consolidations (skewed rows: all three bins in use) -----
    def mm_model(st):
        return 16.0 * st.products + 56.0 * st.nnz_a + 16.0 * st.nnz_c + 16.0 * st.rows_a

    def kernel_ms(sts):
        keys = ("ms_merge_count", "ms_hash_count", "ms_esc", "ms_merge_numeric", "ms_hash_emit", "ms_hash_splits", "ms_hash_numeric")
        return {k: float(np.mean([getattr(x, k) for x in sts])) for k in keys}

    # (a) the member of the family whose product fits one array (scale 20), in ONE multiply() call -- as in round 1
    sc = args.rmat_scale
    A = sp.gen_rmat(ctx, 0x5EED0004, sc, 4 << sc)
    for _ in range(max(1, args.warmup - 1)):
        Cm, st = sp.multiply(ctx, 1.0, None, A, ".", None, A, ".", None, stats=True); Cm.free()
    sts = []
    for _ in range(args.steps):
        Cm, st = sp.multiply(ctx, 1.0, None, A, ".", None, A, ".", None, stats=True)
        sts.append(st); Cm.free()
    ms_k = float(np.mean([x.ms_symbolic + x.ms_numeric for x in sts]))
    model = mm_model(st)
    out[f"spgemm_config4_scale{sc}"] = {
        "workload": f"BASELINE config 4 family: R-MAT scale {sc} (a,b,c,d = .57,.19,.19,.05; edge factor 4) A*A in one multiply() call",
        "products": st.products, "products_hash": st.products_hash, "products_esc": st.products_esc, "nnz_a": st.nnz_a, "nnz_c": st.nnz_c,
        "rows_merge": st.rows_merge, "rows_hash": st.rows_hash, "rows_esc": st.rows_esc,
        "ms_symbolic": float(np.mean([x.ms_symbolic for x in sts])),
        "ms_numeric": float(np.mean([x.ms_numeric for x in sts])), "ms_prepare_incl_consolidate": float(np.mean([x.ms_prepare for x in sts])),
        "ms_kernels": kernel_ms(sts),
        "products_per_sec": st.products / (ms_k * 1e-3), "model_bytes": model, "model_frac": model / (ms_k * 1e-3) / 1e9 / hbm,
        "roofline": kernel_roofline("k_hash_numeric<256, 2560, 4096> (shared-memory hash accumulators: 12 B per product read, 20 B per output written)",
                                    "k_hash_numeric", 12.0 * st.products_hash + 20.0 * st.nnz_c,
                                    float(np.mean([x.ms_hash_numeric for x in sts])), hbm, st.products_hash, "product"),
        "roofline_symbolic": kernel_roofline("k_hash_symbolic (one bitmap pass: 4 B per product read, 4 B per output written)",
                                             "k_hash_symbolic", 4.0 * st.products_hash + 4.0 * st.nnz_c,
                                             float(np.mean([x.ms_hash_count for x in sts])), hbm, st.products_hash, "product"),
    }
    A.free()
    # (b) config 4 AS NAMED: 2^24 rows.  Its product (5.6e10 outputs) fits no single array -- VectorCooArray offsets are int
    # (algorithm.hpp:419) and 16 B x nnzC is 0.9 TB -- so it is formed in row panels (spb_mm_plan_*: the A-row loop of the
    # reference carries no state between rows, multiply_sparse.hpp:192-246); every panel's rows of C are produced in full
    # on the device and released.  Timed: symbolic + numeric of every panel of one sweep (CUDA events inside the library)
    # and the wall clock of the sweep.
    scn = args.rmat_scale_named
    if scn:
        A = sp.gen_rmat(ctx, 0x5EED0004, scn, 4 << scn)
        ctx.sync()
        t0 = time.perf_counter()
        plan = sp.MultiplyPlan(ctx, 1.0, None, A, ".", None, A, ".", None, max_products_per_panel=args.panel_products)
        ctx.sync()
        plan_s = time.perf_counter() - t0
        A.free()
        sweeps = []
        for sweep in range(2):     # one warm-up sweep, one timed one (seconds each)
            ctx.sync()
            t0 = time.perf_counter()
            sts = []
            for p in range(plan.n_panels):
                Cp, st = plan.panel(p, stats=True)
                sts.append(st)
                Cp.free()
            ctx.sync()
            sweeps.append((time.perf_counter() - t0, sts))
        wall_s, sts = min(sweeps[1:], key=lambda x: x[0])

        class Tot:
            pass
        tot = Tot()
        for k in ("products", "products_hash", "products_esc", "nnz_c", "rows_merge", "rows_hash", "rows_esc", "rows_a"):
            setattr(tot, k, int(sum(getattr(x, k) for x in sts)))
        tot.nnz_a = int(sum(x.nnz_a for x in sts))
        ms_k = float(sum(x.ms_symbolic + x.ms_numeric for x in sts))
        model = mm_model(tot)
        kms = {k: float(sum(getattr(x, k) for x in sts)) for k in ("ms_merge_count", "ms_hash_count", "ms_esc", "ms_merge_numeric",
                                                                    "ms_hash_emit", "ms_hash_splits", "ms_hash_numeric", "ms_prepare")}
        out["spgemm_config4"] = {
            "workload": f"BASELINE config 4 as named: R-MAT 2^{scn} rows (a,b,c,d = .57,.19,.19,.05; edge factor 4, {4 << scn} raw edges, duplicates kept) A*A, "
                        f"formed in {plan.n_panels} row panels of <= {args.panel_products} intermediate products (spb_mm_plan_*)",
            "products": tot.products, "products_hash": tot.products_hash, "products_esc": tot.products_esc, "nnz_a": tot.nnz_a, "nnz_c": tot.nnz_c,
            "rows_merge": tot.rows_merge, "rows_hash": tot.rows_hash, "rows_esc": tot.rows_esc, "panels": plan.n_panels,
            "ms_symbolic_plus_numeric_all_panels": ms_k, "ms_sweep_wall": wall_s * 1e3, "ms_plan_incl_consolidate": plan_s * 1e3,
            "ms_kernels_all_panels": kms,
            "products_per_sec": tot.products / (ms_k * 1e-3), "products_per_sec_wall": tot.products / wall_s,
            "model_bytes": model, "model_frac": model / (ms_k * 1e-3) / 1e9 / hbm,
            "parity": "tests/test_gpu_full_size.py::test_config4_as_named_scale24_row_panels: an unbiased 1/64 sample of the rows of this product, bit for bit (structure, order, values) against the CPU oracle",
        }
        plan.free()
    return out


# ------------------------------------------------------------------------------------------------
def ref_impl():
    from oracle import oracle as O
    r = O.reference()
    return (r, "reference") if r is not None else (O.port(), "port")


def banded_sample(n):
    from oracle import oracle as O
    from spsparse_b200 import gen
    a, b, w = gen.banded(S5A, n, 0, n), gen.banded(S5B, n, 0, n), gen.vector(S5W, n)
    return O.Coo(*a), O.Coo(*b), O.Coo(w[0], w[1], w[2], (0,))


def cpu_baseline(args):
    """The reference's own CPU code on bounded samples of the same workload families (rank 0, N=1), as BASELINE.md section 5
    lays out: consolidate on a prefix of the config-2 input (the whole 2*10^8-entry input with --cpu-full, ~3 min); multiply
    on members of the banded family at two sizes with the fitted power law (the reference visits every row x column pair and
    re-scans scalej per pair, so full size is unreachable -- said, not extrapolated silently); and the row-wise CPU oracle
    (reference semantics, NOT the reference's algorithm) on a larger member, labelled as such."""
    from oracle import oracle as O
    impl, kind = ref_impl()
    sizes = [args.cpu_rows, 2 * args.cpu_rows] if args.cpu_full else [args.cpu_rows // 2, args.cpu_rows]
    runs = []
    for n in sizes:
        A, B, W = banded_sample(n)
        t0 = time.perf_counter()
        if kind == "reference":
            out, st = impl.multiply_mm(1.0, None, A, ".", W, B, ".", None, want_stats=True)
            sec = st["seconds"]
        else:
            out = impl.multiply_mm(1.0, None, A, ".", W, B, ".", None)
            sec = time.perf_counter() - t0
        runs.append({"rows": n, "seconds": sec, "products": banded_products(n), "products_per_sec": banded_products(n) / sec,
                     "row_col_pairs_per_sec": float(n) * n / sec, "nnz_c": out.n})
    expo = float(np.log(runs[-1]["seconds"] / runs[0]["seconds"]) / np.log(runs[-1]["rows"] / runs[0]["rows"]))
    n, sec, F = runs[-1]["rows"], runs[-1]["seconds"], runs[-1]["products"]
    res = {"value": F / sec, "unit": UNIT, "cores": 1, "kind": kind, "host_cores": os.cpu_count(),
           "sample": f"{n}x{n} member of the banded family: multiply(C,1,NULL,A,'.',&w,B,'.',NULL) took {sec:.2f} s single-threaded (the "
                     f"reference has no threads); every row x column pair is merge-joined (multiply_sparse.hpp:192-246) and each join "
                     f"re-scans scalej from its start (:223-228): measured time ~ rows^{expo:.2f} between {runs[0]['rows']} and {n} rows, so the "
                     f"full 1e8-row config is unreachable and products/s falls with the row count",
           "seconds": sec, "nnz_c": runs[-1]["nnz_c"], "multiply_runs": runs, "fitted_exponent": expo}
    # consolidate beside it (linearithmic, so this one extrapolates honestly)
    nc = 200_000_000 if args.cpu_full else args.cpu_cons_entries
    a = O.port().gen_dup_coo(S2, 0, nc, 140_000_000 if nc == 200_000_000 else int(nc * 0.7), 24, 0)
    if kind == "reference":
        sec, nout, vsum = impl.consolidate_timed(a, (0, 1))
    else:
        t0 = time.perf_counter(); r = impl.consolidate(a, (0, 1)); nout, vsum = r.n, float(r.val.sum()); sec = time.perf_counter() - t0
    res["consolidate"] = {"nnz_per_sec": nout / sec, "entries_in_per_sec": nc / sec, "seconds": sec, "nnz_out": nout, "sum_values": vsum,
                          "sample": ("the whole config-2 input" if nc == 200_000_000 else f"first {nc} entries of the config-2 generator") +
                                    ", consolidate(ret, A, {0,1}), " + ("genuine reference" if kind == "reference" else "oracle port")}
    del a
    # the row-wise CPU oracle: same results as the reference wherever the reference can run, linear in the products
    no = 20_000_000 if args.cpu_full else args.cpu_oracle_rows
    A, B, W = banded_sample(no)
    t0 = time.perf_counter()
    out = O.port().multiply_mm(1.0, None, A, ".", W, B, ".", None)
    sec = time.perf_counter() - t0
    res["row_wise_oracle"] = {"rows": no, "seconds": sec, "products_per_sec": banded_products(no) / sec, "nnz_c": out.n,
                              "note": "reference-semantics CPU oracle (row-wise Gustavson, oracle/spsparse_oracle.c), NOT the reference's "
                                      "algorithm; includes its consolidations of A and B; 1 core"}
    return res


def banded_products(n):
    # row i of A has entries at j in [i-2,i+2] within range; each j contributes the in-range length of B row j
    i = np.arange(n)
    lo, hi = np.maximum(i - 2, 0), np.minimum(i + 2, n - 1)
    blen = hi - lo + 1
    c = np.concatenate([[0], np.cumsum(blen)])
    return int((c[hi + 1] - c[lo]).sum())


_REF_JOB = {}


def _ref_row_block(blk):
    """Worker of the reference arm: the reference's multiply on one contiguous block of A's rows (forked, so the
    sample and the loaded library are inherited)."""
    impl, A, B, W, bounds = _REF_JOB["impl"], _REF_JOB["A"], _REF_JOB["B"], _REF_JOB["W"], _REF_JOB["bounds"]
    from oracle import oracle as O
    lo, hi = bounds[blk], bounds[blk + 1]
    pick = (A.idx[0] >= lo) & (A.idx[0] < hi)
    Ab = O.Coo(A.shape, [A.idx[0][pick], A.idx[1][pick]], A.val[pick])
    t0 = time.perf_counter()
    out = impl.multiply_mm(1.0, None, Ab, ".", W, B, ".", None)
    return time.perf_counter() - t0, out.n


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import multiprocessing as mp
    impl, kind = ref_impl()
    n = args.ref_rows
    A, B, W = banded_sample(n)
    F = banded_products(n)
    # The reference has no threads.  "All the host threads it can use" = what a user with a multi-core host would do with
    # it: independent processes on contiguous row blocks of A (the split this repo uses across GPUs), whole B in each.
    procs = max(1, min(os.cpu_count() or 1, args.ref_procs if args.ref_procs > 0 else (os.cpu_count() or 1)))
    _REF_JOB.update(impl=impl, A=A, B=B, W=W, bounds=[n * b // procs for b in range(procs + 1)])
    times = []
    ctxmp = mp.get_context("fork")
    pool = ctxmp.Pool(procs) if procs > 1 else None   # created once, outside the timed steps
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        if pool is None:
            _ref_row_block(0)
        else:
            pool.map(_ref_row_block, range(procs))
        sec = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(sec)
    if pool is not None:
        pool.close(); pool.join()
    sec = float(np.mean(times))
    value = F / sec
    sample = (f"{n}x{n} member of the banded family (the reference's multiply visits every row x column pair and re-scans scalej per pair: "
              f"rows^2..rows^3 work, 1e8 rows is unreachable), full call incl. its internal consolidations; the reference is "
              f"single-threaded, so {procs} independent processes each multiply one contiguous block of A's rows by the whole B "
              f"(wall clock around all of them; the worker processes are started once, before the timed steps)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "BASELINE config 5 family (banded A*diag(w)*B), bounded sample", "rows": n, "products": F},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample, "host_cores": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the headline, of the pinned end-to-end pipeline and of "
                                                       "'also' configs 2, 3 and 4 (one call); the pageable C-ABI and C++-API end-to-end legs "
                                                       "(seconds per step) time min(steps, 2), reported as their own 'steps', and config 4 "
                                                       "as named times one sweep of its row panels")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows of the banded problem (headline: 1e8)")
    ap.add_argument("--cons-entries", type=int, default=200_000_000)
    ap.add_argument("--regrid", type=int, nargs=4, default=[3200, 3125, 1000, 1000])
    ap.add_argument("--rmat-scale", type=int, default=20, help="member of the config-4 family run in one multiply() call")
    ap.add_argument("--rmat-scale-named", type=int, default=24, help="config 4 as named (row panels); 0 = skip")
    ap.add_argument("--panel-products", type=int, default=1 << 30, help="intermediate products per row panel")
    ap.add_argument("--cpu-rows", type=int, default=3000)
    ap.add_argument("--cpu-cons-entries", type=int, default=30_000_000)
    ap.add_argument("--cpu-oracle-rows", type=int, default=2_000_000)
    ap.add_argument("--cpu-full", action="store_true", help="CPU baselines at BASELINE.md section 5's full sizes (minutes)")
    ap.add_argument("--ref-rows", type=int, default=2000)
    ap.add_argument("--ref-procs", type=int, default=0, help="processes of the reference arm (0 = all host cores)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-only", action="store_true", help="only the CPU baselines (with --cpu-full: BASELINE.md section 5's full sizes), no GPU work")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step to DIR/*.npy (float64, at most 64 MB: "
                                                          "a fixed, seeded sample of a larger result)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        print(f"note: warmup {args.warmup} < 3 breaks the timing rules", file=sys.stderr)
    if args.impl == "reference":
        return run_reference(args)
    if args.cpu_only:
        print(json.dumps({"cpu_baseline": cpu_baseline(args)}))
        return None
    return run_ours(args)


if __name__ == "__main__":
    main()

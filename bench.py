#!/usr/bin/env python
"""bench.py -- candidate x point scoring throughput on B200 (BASELINE.json metric).

A "step" = one pass of the hot path (K2 score, + the NCCL all-reduce of the per-candidate counts
when sharded) over config c3: 4096 candidates (1024 planes/spheres/cylinders/cones) x 16 Mi points
per GPU (point-range shards; weak scaling: every rank holds its own 16 Mi-point shard).

  value      G candidate.point evals/s, whole job, inputs resident in HBM (device-timed)
  e2e        same metric through the public call with HOST buffers: every step uploads the cloud
             (pinned host -> device), the candidates, scores, and reads the counts back
  roofline   the tiled score kernel against the FP32 roofline (the path is FP32-ALU bound)
  cpu_baseline  the CPU restatement of the reference (oracle/) on a bounded sample

`--impl reference` times the CPU restatement of RANSAC.jl's scorecandidate loop instead (Julia is
not installed in this image, so the Julia package itself cannot run; see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_EVAL = {"plane": 13, "sphere": 16, "cylinder": 27, "cone": 38}  # SURVEY.md 8(d)
MIX_FLOPS = 23.5
NCU_FULL = "profiles/r2f_kernels_ncu_full.json"  # the committed `ncu --set full` capture roofline.traffic is read from


def ncu_traffic(cands: int, points: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the score kernels of one step, from the committed ncu
    capture of the same command -- only if that capture is of THIS configuration; None otherwise."""
    try:
        d = json.load(open(os.path.join(ROOT, NCU_FULL)))
        if d["config"]["candidates"] == cands and d["config"]["points"] == points:
            return float(d["traffic_bytes_per_step"])
    except Exception:
        pass
    return None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=16 << 20, help="points per GPU")
    ap.add_argument("--cands", type=int, default=4096)
    ap.add_argument("--cpu-sample", type=int, default=0, help="override the CPU sample (points)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cull", action="store_true", help="skip the informational culled-scoring leg")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--ransac", default="c4,c5",
                    help="comma list of scenes (c2, c4, c5; 'none') on which end-to-end ransac() is also timed, at every N "
                         "(sharded storage + the library's NCCL at N > 1; extra JSON key `ransac`): c4 = the 10 M-point "
                         "CAD-like scene BASELINE.json's second headline is quoted on, c5 = the 100 M-point LiDAR-like scan")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaled c3 leg at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed calls returned in their last step to DIR/<name>.npy (float32 / float64): the "
                         "per-candidate counts and, for every --ransac scene, the extracted shapes, their inlier totals and "
                         "(at N = 1) the shape each point of a fixed strided sample went to")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML polled every 10 ms from a
    thread (the timed region is ~0.2 s, shorter than nvidia-smi's start-up), nvidia-smi as a fallback."""

    BAD = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
    NOTED = {"sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.index = index
        self.sm, self.pw, self.reasons = [], [], set()
        self.mx = None
        self._stop = threading.Event()
        self.t = None
        self.source = None
        self.period = float(os.environ.get("BENCH_CLOCK_PERIOD_MS", "10")) / 1e3

    def _nvml_loop(self, nv, h):
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.pw.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in {**self.BAD, **self.NOTED}.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.period <= 0:
            return
        try:
            import pynvml as nv

            nv.nvmlInit()
            vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
            ent = vis[self.index] if self.index < len(vis) else str(self.index)
            if ent.isdigit():
                h = nv.nvmlDeviceGetHandleByIndex(int(ent))
            elif ent.startswith("GPU-"):
                h = nv.nvmlDeviceGetHandleByUUID(ent)
            else:  # by PCI bus id of the CUDA device, robust against any other enumeration
                import torch

                bus = torch.cuda.get_device_properties(self.index).pci_bus_id
                h = nv.nvmlDeviceGetHandleByIndex(next(i for i in range(nv.nvmlDeviceGetCount())
                                                       if nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(i)).bus == bus))
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.source = f"nvml, {self.period * 1e3:.0f} ms period"
            self.t = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.t.start()
            return
        except Exception:
            pass
        try:  # fallback: nvidia-smi loop
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 50"

            def rd():
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for line in self.proc.stdout:
                    r = [x.strip() for x in line.split(",")]
                    try:
                        self.sm.append(float(r[0])), self.pw.append(float(r[2]))
                        self.mx = float(r[1])
                        for nme, v in zip(names, r[3:7]):
                            if v.lower().startswith("active"):
                                self.reasons.add(nme)
                    except Exception:
                        pass

            self.t = threading.Thread(target=rd, daemon=True)
            self.t.start()
        except Exception:
            self.source = None

    def stop(self):
        self._stop.set()
        if getattr(self, "proc", None):
            self.proc.terminate()
        if self.t:
            self.t.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["no clock samples"], "samples": 0, "source": self.source}
        return {"sm_mhz": float(np.median(self.sm)), "sm_min_mhz": float(min(self.sm)), "sm_max_mhz": self.mx,
                "power_w_max": max(self.pw) if self.pw else None, "samples": len(self.sm), "reasons": sorted(self.reasons),
                "source": self.source}


def make_workload(points: int, ncands: int, rank: int):
    from ransac_jl_b200 import scenes

    sc = scenes.scene_mixed(3 + 1000 * rank, points)
    # candidates are identical on every rank: generated from rank 0's primitives
    sc0 = sc if rank == 0 else scenes.Scene(None, None, None, scenes.scene_mixed(3, 1024).primitives)
    cands = scenes.perturbed_candidates(sc0, ncands // 4, seed=7)
    return sc, cands


def cpu_baseline(sc, cands, params, budget_pts: int, ncand: int = 64):
    """CPU restatement of the reference (oracle/) on a bounded sample of the same workload."""
    from oracle import ransac_oracle as O
    from tests.helpers import oracle_params, to_oracle_shape

    op = oracle_params(params)
    try:
        from oracle import c_oracle
        have_c = c_oracle.available()
    except Exception:
        have_c = False
    n = min(budget_pts, len(sc.vertices))
    P = sc.vertices[:n].astype(np.float64)
    N = sc.normals[:n].astype(np.float64)
    step = max(1, len(cands) // ncand)
    sample = cands[::step]
    t0 = time.perf_counter()
    if have_c:
        counts, cores = c_oracle.score_counts(sample, P, N, op, nthreads=os.cpu_count() or 1)  # all host threads, explicitly
    else:
        cores = 1
        counts = np.array([int(O.compatibles(to_oracle_shape(sh), P, N, op).sum()) for sh in sample], np.int32)
    dt = time.perf_counter() - t0
    ev = len(sample) * n
    single = None
    if have_c:  # the reference is single-threaded: the same code on ONE thread, on 1/16 of the points
        n1 = max(1, n // 16)
        t1 = time.perf_counter()
        c_oracle.score_counts(sample, P[:n1], N[:n1], op, nthreads=1)
        single = len(sample) * n1 / (time.perf_counter() - t1) / 1e9
    return {"_counts": counts, "_step": step, "_n": n,
            "value": ev / dt / 1e9, "unit": "G evals/s", "cores": cores, "kind": "port", "single_thread_value": single,
            "sample": f"{len(sample)} candidates (every {step}th, all four types) x first {n} points of the workload; "
                      f"{'C (OpenMP)' if have_c else 'NumPy'} float64 restatement of RANSAC.jl compatibles*, {dt:.2f} s"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm for the path (restated, see module doc)."""
    if rank != 0:
        return
    import ransac_jl_b200  # noqa: F401 (host-side types only; nothing below touches the GPU)
    from ransac_jl_b200 import params as RP

    pts = args.cpu_sample or (2 << 20)
    sc, cands = make_workload(pts, args.cands, 0)
    params = RP.ransacparameters()
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_baseline(sc, cands, params, pts, ncand=128)
        r = {k: v for k, v in r.items() if not k.startswith("_")}
        if i >= args.warmup:
            vals.append(r)
    v = float(np.mean([x["value"] for x in vals]))
    ms = float(np.mean([len(cands[:: max(1, len(cands) // 128)]) * pts / (x["value"] * 1e9) * 1e3 for x in vals]))
    out = {
        "impl": "reference", "metric": "candidate_point_evals_per_s", "value": v, "unit": "G evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"c3 candidate-scoring microbench, bounded CPU sample: {vals[-1]['sample']}"},
        "cpu_baseline": dict(vals[-1], value=v),
        "e2e": {"value": v, "unit": "G evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "Julia is not installed in this image: the timed code is the CPU restatement of RANSAC.jl's scorecandidate loop (oracle/), not the Julia package",
    }
    print(json.dumps(out))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist

    import ransac_jl_b200 as R
    from ransac_jl_b200._lib import lib
    import ctypes as C

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    if world > 1:  # the library's own NCCL communicator: torch.distributed only carries its 128-byte id
        from ransac_jl_b200 import shard

        shard.init_comm(R.Context.get(local))

    sc, cands = make_workload(args.points, args.cands, rank)
    params = R.ransacparameters()
    cp = R.to_c(params)
    Cn = len(cands)
    n = len(sc.vertices)

    # ---- resident arm: cloud + candidates in HBM --------------------------------------------
    pc = R.RANSACCloud(sc.vertices, sc.normals, [np.zeros(0, np.int64)], device=local)
    arr = R.pack_cands(cands)
    d_cands = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
    d_counts = torch.zeros(Cn, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)  # a real (non-default) stream: its handle is what the C ABI gets
    torch.cuda.set_stream(stream)

    def step_resident(cloud=None):
        cloud = cloud or pc
        rc = lib.rsc_score_dev(cloud.handle, C.byref(cp), d_cands.data_ptr(), Cn, -1, d_counts.data_ptr(), stream.cuda_stream)
        pc.ctx.check(rc)
        if world > 1:  # ncclAllReduce(int32, sum) of the per-candidate counts, enqueued by the library on the same stream
            pc.ctx.check(lib.rsc_ctx_allreduce(pc.ctx.h, d_counts.data_ptr(), Cn, stream.cuda_stream))

    if world > 1:
        dist.barrier()  # first barrier = lazy NCCL set-up: keep it out of the neighbourhood of the timed region
    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    t_a = torch.cuda.Event(enable_timing=True)
    t_b = torch.cuda.Event(enable_timing=True)
    t_a.record()
    for a, b in evs:
        a.record()
        step_resident()
        b.record()
    t_b.record()
    torch.cuda.synchronize()
    counts_host = d_counts.cpu().numpy()  # the counts of the last timed step
    if world > 1:
        dist.barrier()
    total_ms = t_a.elapsed_time(t_b)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([total_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    evals_per_step = float(Cn) * n * world
    value = evals_per_step / (ms_per_step * 1e-3) / 1e9

    # kernel-only time of the tiled score kernel (CUDA events recorded by the library on the same
    # stream around that launch alone), averaged over a few extra steps
    kms, guard = [], 0
    for _ in range(3):
        step_resident()
        k, guard = _last_kernel(pc)
        kms.append(k)
    kernel_ms = float(np.mean(kms))

    # ---- e2e arm: host buffers through the public call -----------------------------------------
    e2e = None
    if not args.no_e2e:
        xyz = torch.from_numpy(sc.vertices).pin_memory()
        nrm = torch.from_numpy(sc.normals).pin_memory()
        counts_h = np.zeros(Cn, dtype=np.int32)

        def step_e2e():
            # the public host-buffer calls: upload this step's cloud, upload + score the candidates,
            # read the counts back (device buffers of the cloud handle are reused, not re-allocated)
            pc.ctx.check(lib.rsc_cloud_update(pc.handle, xyz.data_ptr(), nrm.data_ptr(), n))
            pc.ctx.check(lib.rsc_score(pc.handle, C.byref(cp), arr, Cn, -1, counts_h.ctypes.data, None))

        for _ in range(max(1, min(args.warmup, 2))):
            step_e2e()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
            if world > 1:
                tt = torch.from_numpy(counts_h).to(dev)
                dist.all_reduce(tt)
                counts_h[:] = tt.cpu().numpy()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        if world == 1:
            assert np.array_equal(counts_h, counts_host), "e2e and resident arms disagree"
        e2e = {"value": evals_per_step / (dt / args.steps) / 1e9, "unit": "G evals/s",
               "h2d_bytes_per_step": int(2 * n * 12 + Cn * 64 + Cn * 16), "d2h_bytes_per_step": int(Cn * 4 + 4),
               "ms_per_step": dt / args.steps * 1e3}

    # ---- strong-scaled c3 (SURVEY 8d: "shards N/G per GPU"): the SAME total of points, 1/N of them per GPU ----
    strong = None
    if world > 1 and not args.no_strong:
        n_s = (n // world) // 2048 * 2048
        pcs = R.RANSACCloud(sc.vertices[:n_s], sc.normals[:n_s], [np.zeros(0, np.int64)], device=local)
        for _ in range(args.warmup):
            step_resident(pcs)
        torch.cuda.synchronize()
        dist.barrier()
        s_a, s_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_a.record()
        for _ in range(args.steps):
            step_resident(pcs)
        s_b.record()
        torch.cuda.synchronize()
        dist.barrier()
        ts = torch.tensor([s_a.elapsed_time(s_b)], device=dev)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        ms_s = float(ts.item()) / args.steps
        ks = []
        for _ in range(3):
            step_resident(pcs)
            ks.append(_last_kernel(pcs)[0])
        strong = {"scaling": "strong", "points_total": int(n_s * world), "points_per_gpu": int(n_s), "candidates": Cn,
                  "ms_per_step": ms_s, "value": float(Cn) * n_s * world / (ms_s * 1e-3) / 1e9, "unit": "G evals/s",
                  "score_kernels_ms": float(np.mean(ks)),
                  "note": "same step as the headline (rsc_score_dev + the library's ncclAllReduce of the counts), "
                          "max over ranks; compare with the 1-GPU headline value for the strong-scaling efficiency"}
        pcs.close()

    # ---- end-to-end ransac() at this N (all ranks take part) ----
    ransac_out = None
    extracted = {}  # scene -> what ransac() returned in the last timed run
    scenes_req = [s for s in args.ransac.split(",") if s and s != "none"]
    if scenes_req:
        # free the microbenchmark's device buffers first (c5 needs 2.4 GB per replica at N = 1)
        keep_for_rank0 = (sc, cands)
        from tools import ransac_e2e

        ransac_out = {}
        for which in scenes_req:
            try:
                ransac_out[which], extracted[which] = ransac_e2e.run(which, rank, world, local, dist if world > 1 else None,
                                                                     cpu_loop=not args.no_cpu, reps=args.steps,
                                                                     return_extracted=True)
            except Exception as e:  # informational keys: never lose the headline line
                ransac_out[which] = {"error": repr(e)}
                if world > 1:
                    break  # the ranks may no longer be in step

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_max = (clocks or {}).get("sm_max_mhz") or peaks.get("sm_max_mhz") or 1965.0
    nsm = torch.cuda.get_device_properties(local).multi_processor_count
    fp32_peak = nsm * 128 * 2 * sm_max * 1e6 / 1e12
    ach = MIX_FLOPS * Cn * n / (kernel_ms * 1e-3) / 1e12
    fma_chain = None  # measured FP32 peak of this very GPU: scalar FFMA chains (tools/fp32_peak.cu, ~1 s)
    try:
        pk = subprocess.run([os.path.join(ROOT, "tools", "fp32_peak")], capture_output=True, text=True, timeout=120)  # rank 0 = device 0
        fma_chain = float(json.loads(pk.stdout.strip().splitlines()[-1])["ffma_scalar_tflops"])
    except Exception:
        pass
    roofline = {
        "bound": "fp32", "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak,
        # dram__bytes_read.sum + dram__bytes_write.sum of the score kernels of one step, read from the committed
        # `ncu --set full` capture (same command and configuration; null for any other configuration)
        "traffic": ncu_traffic(Cn, n), "traffic_source": NCU_FULL, "algorithmic_bytes": 4 * 24.125 * n,
        "peak_source": f"derived: {nsm} SMs x 128 FP32 lanes x 2 x {sm_max:.0f} MHz (MEASURED_PEAKS.json has no FP32 entry; "
                       "the path uses no tensor cores and is not HBM bound)",
        "peak_measured_fma_chain": fma_chain, "frac_of_measured_fma_chain": (ach / fma_chain) if fma_chain else None,
        "kernel": "rsc::score_kernel<T,K,MINB,U,MASKS> x5 (one launch per column type: plane, sphere, cylinder, cone, wide cone; "
                  "side by side on forked streams; kernel_ms = CUDA events around the launches)", "kernel_ms": kernel_ms,
        "algorithmic_flops_per_eval": MIX_FLOPS,
        "hbm_gbs_algorithmic": (Cn / 512) * 24.125 * n / (kernel_ms * 1e-3) / 1e9,
        "hbm_peak_gbs": peaks.get("hbm_gbs"),
    }
    out = {
        "metric": "candidate_point_evals_per_s", "value": value, "unit": "G evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"c3 candidate-scoring microbench: {Cn} candidates (4 shape types x {Cn // 4}) x "
                               f"{n} points per GPU, whole-cloud scoring, counts only",
                   "points_per_gpu": n, "candidates": Cn, "parallelism": f"point-range shards x{world}, "
                   "int32 count all-reduce (NCCL)" if world > 1 else "single GPU",
                   "l2": "inputs (403 MB of points per pass) exceed the 126 MB L2; no flush needed"},
        # per step: compile_kernel, 5 x score_kernel (plane, sphere, cylinder, cone, wide cone), fixup_scan_kernel,
        # fixup_pair_kernel, select_counts_kernel
        "e2e": e2e, "gpu_launches": 9 * args.steps, "clocks": clocks, "roofline": roofline,
        "fp64_guard_pairs_per_step": int(guard),
    }
    # K4 (refit over the whole shard, HBM bound): mask kernel time -> GB/s of algorithmic bytes
    try:
        ex = R.refit(cands[0], pc, params)
        st4 = pc.ctx.stats()
        ms20, nin = C.c_double(), C.c_int64()
        cand0 = cands[0].to_cand()
        pc.ctx.check(lib.rsc_debug_refit_mask_ms(pc.handle, C.byref(cp), C.byref(cand0), 20, C.byref(ms20), C.byref(nin)))
        assert nin.value == len(ex.inpoints)
        out["refit"] = {"kernel": "rsc::extract_mask_kernel<T>", "points": n, "inliers": int(len(ex.inpoints)),
                        "kernel_ms": ms20.value, "achieved_gbs": 24.125 * n / (ms20.value * 1e-3) / 1e9,
                        "kernel_ms_single_launch_event_pair": st4.refit_mask_ms,
                        "timing": "20 back-to-back launches between one CUDA-event pair (a pair around ONE ~70 us launch reads "
                                  "10-20 us high: that was the 64 us (ncu) vs 86 us (events) gap of round 1); the 403 MB cloud "
                                  "exceeds the 126 MB L2, so repeats do not hit in cache",
                        "peak_gbs": peaks.get("hbm_gbs"), "bound": "hbm", "algorithmic_bytes_per_point": 24.125}
    except Exception as e:  # informational key only
        out["refit"] = {"error": repr(e)}
    # counts + packed bitmasks variant (SURVEY 8d), device resident: 4096 x 4 Mi points -> 2 GiB of masks
    if world == 1:
        try:
            out["masks_variant"] = time_masks_variant(R, lib, C, torch, sc, cands, params, local, dev)
        except Exception as e:  # informational key only
            out["masks_variant"] = {"error": repr(e)}
    if strong is not None:
        out["strong"] = strong
    if ransac_out is not None:
        out["ransac"] = ransac_out
    if not args.no_cpu and world == 1:
        # ~10 s of CPU work: 512 candidates (every 8th) x all points of rank 0's shard of the same workload
        cb = cpu_baseline(sc, cands, params, args.cpu_sample or len(sc.vertices), ncand=512)
        # the oracle's counts of those candidates against the device's, on the same points: parity at the
        # full c3 size (the device counted all 4096 candidates over all points in the timed steps above)
        if cb["_n"] == n:
            want, got = np.asarray(cb["_counts"]), counts_host[:: cb["_step"]]
            out["parity_checked"] = {"cands": int(len(want)), "points": int(n), "mismatches": int((want != got).sum()),
                                     "max_abs_count_diff": int(np.abs(want.astype(np.int64) - got).max()),
                                     "checker": "oracle/oracle.c::orc_score (float64 restatement of compatibles*)"}
        out["cpu_baseline"] = {k: v for k, v in cb.items() if not k.startswith("_")}
    # informational, last (nothing measured above depends on it): the same counts through Morton-tile culling
    # (rsc_score_culled, DESIGN.md section 3).  Never the headline: the reference evaluates every pair.
    if world == 1 and not args.no_cull:
        try:
            out["culled_variant"] = time_culled_variant(R, pc, cands, params)
        except Exception as e:
            out["culled_variant"] = {"error": repr(e)}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, counts_host, extracted, world)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(dirname, counts, extracted, world, sample=1 << 20):
    """--dump-outputs: the per-candidate counts of the last timed step and, per ransac() scene, the extracted shapes
    (rows: type, outwards, p[7]) and their inlier totals.  The full inlier lists (up to 10^8 indices) are represented
    by a strided sample of about `sample` point indices 0, s, 2s, ...: the extraction order of the shape that took
    each one, -1 if none.  Rank 0 holds only its own point range at N > 1, so the sample is written at N = 1 only."""
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "score_counts.npy"), counts.astype(np.float64))
    for which, ex in extracted.items():
        cands = [e.shape.to_cand() for e in ex]
        shapes = np.array([[c.type, c.outwards, *c.p] for c in cands], np.float64).reshape(len(cands), 9)
        np.save(os.path.join(dirname, f"ransac_{which}_shapes.npy"), shapes)
        np.save(os.path.join(dirname, f"ransac_{which}_inliers.npy"), np.array([e.total for e in ex], np.float64))
        if world == 1:
            from tools.ransac_e2e import SCENES

            n = SCENES[which][0]
            step = max(1, n // sample)
            label = np.full((n + step - 1) // step, -1, np.float32)
            for k, e in enumerate(ex):
                label[e.inpoints[e.inpoints % step == 0] // step] = k
            np.save(os.path.join(dirname, f"ransac_{which}_sampled_point_shape.npy"), label)


def time_culled_variant(R, pc, cands, params, reps=3):
    """rsc_score_culled on the resident cloud of the headline workload; counts checked against the dense path."""
    pc.build_cells(11)
    dense, _ = R.score_counts(pc, cands, -1, params)
    got, info = R.score_counts_culled(pc, cands, params)  # builds the Morton copy + tile spheres
    ms = []
    for _ in range(reps):
        got, info = R.score_counts_culled(pc, cands, params)
        ms.append(info["kernel_ms"])
    evals = len(cands) * pc.size
    return {"kernel": "rsc::cull_score_kernel", "kernel_ms": min(ms), "equal_counts": bool(np.array_equal(got, dense)),
            "pairs_total": info["pairs_total"], "pairs_survived": info["pairs_survived"],
            "surviving_fraction": info["pairs_survived"] / max(1, info["pairs_total"]),
            "G_evals_s_reference_equivalent": evals / (min(ms) * 1e-3) / 1e9,
            "note": "skips (candidate, 128-point Morton tile) pairs that provably hold no compatible point; same counts"}


def time_masks_variant(R, lib, C, torch, sc, cands, params, local, dev, npts=4 << 20):
    """rsc_score_dev_masks: counts + candidate-major inlier bitmasks written to device memory."""
    n = min(npts, len(sc.vertices))
    pc = R.RANSACCloud(sc.vertices[:n], sc.normals[:n], [np.zeros(0, np.int64)], device=local)
    cp = R.to_c(params)
    Cn = len(cands)
    arr = R.pack_cands(cands)
    d_cands = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
    d_counts = torch.zeros(Cn, dtype=torch.int32, device=dev)
    words = (n + 31) // 32
    d_masks = torch.empty((Cn, words), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    best = None
    for it in range(4):
        ev[0].record()
        pc.ctx.check(lib.rsc_score_dev_masks(pc.handle, C.byref(cp), d_cands.data_ptr(), Cn, -1, d_counts.data_ptr(),
                                             d_masks.data_ptr(), st.cuda_stream))
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1])
        best = ms if best is None or ms < best else best
    # popcount of the masks must equal the counts (sample of candidates)
    sel = list(range(0, Cn, 257))
    pop = [int(np.unpackbits(d_masks[i].cpu().numpy().view(np.uint8)).sum()) for i in sel]
    ok = pop == [int(d_counts[i].item()) for i in sel]
    pc.close()
    return {"points": n, "candidates": Cn, "ms_per_step": best, "G_evals_s": Cn * n / best / 1e6, "mask_bytes": int(Cn * words * 4),
            "popcount_equals_counts": bool(ok)}


def _last_kernel(pc):
    import ctypes as C

    from ransac_jl_b200._lib import lib

    ms, gp = C.c_double(), C.c_int64()
    pc.ctx.check(lib.rsc_ctx_last_kernel(pc.ctx.h, C.byref(ms), C.byref(gp)))
    return ms.value, gp.value


if __name__ == "__main__":
    main()

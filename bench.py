#!/usr/bin/env python
"""Benchmark of the NeuralRecon-W per-ray training hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl nrw|reference] [--precision bf16x3|bf16|bf16x6]
                    [--dump-outputs DIR]

A "step" = one full training step over one batch of 8192 synthetic posed-camera rays x 128 samples
(BASELINE config C2 "brandenburg_gate config, 8192 rays x 128 samples"): voxel-guided hierarchical
sampling -> background NeRF -> SDF value/normal -> colour net -> NeuS compositing -> loss -> backward
(hand-derived second order) -> [NCCL all-reduce] -> clip(0.99) -> Adam.  Prints ONE JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "neuralrecon-w_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

# algorithmic FLOP per sample (2*MAC, forward) of the three MLPs (SURVEY.md 8 / BASELINE.md 3)
F_SDF, F_COL, F_NERF = 4195328, 1170688, 1318912
DEFAULT_PRECISION = "mixed"      # headline precision policy: 3-product forward (outputs 1e-4), plain-bf16 backward GEMMs (DESIGN.md 6a;
                                 # evidence: tests/test_gpu_precision_policy.py, profiles/r2_precision_study.json)
WORKLOADS = {
    "C3": dict(n_samples=64, n_importance=64, up_sample_steps=4, n_outside=4, rays=8192, fine=True, boundary_samples=10, sample_range=16,
               name="brandenburg_gate config + appearance embedding + surface-guided fine sampling (SDF-derived octree traced every step, "
                    "16-voxel window, 10 boundary samples): 8192 rays x 138 samples"),
    "C5": dict(dim=512, name="sdf_extract.sh marching-cubes grid: batched SDF query of the dense 512^3 lattice (134,217,728 points)"),
    "C2": dict(n_samples=64, n_importance=64, up_sample_steps=4, n_outside=4, rays=8192,
               name="brandenburg_gate config, synthetic ray cache, 8192 rays x 128 samples (64 coarse + 64 importance, 4 up-sample rounds, 4 outside)"),
    "C1": dict(n_samples=64, n_importance=16, up_sample_steps=2, n_outside=4, rays=1024,
               name="400x400 synthetic pinhole camera, 1024-ray batch, 64 coarse + 16 importance samples"),
}


def flop_per_ray(w):
    """W_ray = F*[(n_s + (k-1) n_i/k) + 6 S] + 3 C S + 3 N T  (SURVEY.md 8d)."""
    k = w["up_sample_steps"]
    n_new = w["n_importance"] // k
    S = w["n_samples"] + k * n_new + (w.get("boundary_samples", 0) if w.get("fine") else 0)
    T = S + w["n_outside"]
    evals = w["n_samples"] + (k - 1) * n_new
    return F_SDF * (evals + 6 * S) + 3 * F_COL * S + 3 * F_NERF * T


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line), read
    in-process through NVML every 100 ms.  (A looping `nvidia-smi --query-gpu` child was measured to stall kernel
    launches for seconds on boxes without persistence mode, so it is only the fallback, at a 1 s period.)"""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.sm, self.mx, self.reasons, self.power = index, [], [], set(), []
        self.stop_flag, self.thread, self.proc, self.source = threading.Event(), None, None, None

    def _nvml_loop(self, nv, h):
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)      # board power, W
                except Exception:
                    pass
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                for name, bit in self.BITS:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def _smi_loop(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                self.sm.append(float(f[0])); self.mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            self.source = "nvml"
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "1000"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._smi_loop, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        time.sleep(0.12)
        self.stop_flag.set()
        if self.proc is not None:
            self.proc.terminate()
        self.thread.join(timeout=2.0)
        sm, pw = sorted(self.sm), sorted(self.power)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
               "reasons": sorted(self.reasons), "samples": len(sm), "source": self.source}
        if pw:
            out["power_w"] = {"median": pw[len(pw) // 2], "max": pw[-1]}
        return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1409.5), d.get("hbm_gbs", 6576.7), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(out_dir, arrays):
    """--dump-outputs: what the last timed step computed, as out_dir/<name>.npy (float32), so that two builds run with the
    same arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


DUMP_SAMPLE = 1 << 22      # C5 volume entries written by --dump-outputs (16 MB of the 512 MB volume, a fixed seeded sample)


# ----------------------------------------------------------------------------------------------
def _ref_cfg(workload):
    from oracle import synth

    w = WORKLOADS[workload]
    return synth.PathConfig(n_samples=w["n_samples"], n_importance=w["n_importance"], up_sample_steps=w["up_sample_steps"],
                            n_outside=w["n_outside"], perturb=1.0)


def reference_kind():
    """"reference": the UNMODIFIED reference (oracle/_ref = verbatim copy made by oracle/fetch_ref.py, or /root/reference);
    "port": the pinned restatement oracle/neuconw_port.py (only when no reference copy travelled to this box)."""
    from oracle import ref_runner

    return "reference" if ref_runner.available() else "port"


def make_reference_stepper(workload, device):
    """Returns (kind, step(batch)) running one full training step of the reference on `device`:
    zero_grad -> NeuconWRenderer.render -> NeuconWLoss -> backward -> clip_grad_norm_(0.99) -> Adam(eps=1e-7)."""
    from oracle import synth

    cfg = _ref_cfg(workload)
    if reference_kind() == "reference":
        from oracle import ref_runner

        r = ref_runner.RefRunner(cfg, synth.make_params(seed=0), device=device)
        return "reference", cfg, (lambda b: r.train_step(b, perturb_overwrite=-1))
    from oracle import neuconw_port as port

    P = {k: v.to(device) for k, v in synth.make_params(seed=0).items()}
    return "port", cfg, (lambda b: port.train_step(P, cfg, b, perturb_overwrite=-1)[1])


def cpu_reference(workload, n_rays_cpu, steps, warmup, threads):
    """The reference's own PyTorch CPU path timed on the host cores: one full training step per sample batch."""
    from oracle import synth

    torch.set_num_threads(threads)
    kind, cfg, step = make_reference_stepper(workload, "cpu")
    batch = synth.make_rays(n_rays_cpu, cfg, seed=1)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        step(batch)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return n_rays_cpu / dt, dt, kind


def torch_gpu_reference(workload, n_rays, steps, warmup, device):
    """The reference's stock torch.nn / cuBLAS fp32 path on THIS GPU (the '>= 4x' denominator of BASELINE.json),
    at the full batch of the workload when it fits in HBM (halved on OOM until it does)."""
    from oracle import synth

    kind, cfg, step = make_reference_stepper(workload, device)
    while True:
        try:
            batch = {k: v.to(device) for k, v in synth.make_rays(n_rays, cfg, seed=1).items()}
            for _ in range(warmup):
                step(batch)
            torch.cuda.synchronize()
            break
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            n_rays //= 2
            if n_rays < 64:
                raise
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        step(batch)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / steps
    return n_rays / (ms * 1e-3), ms, n_rays, kind


DTYPES = {"bf16": "bf16", "bf16x3": "bf16 (3-product split, fp32 accumulate)", "bf16x6": "bf16 (6-product split, fp32 accumulate)",
          "mixed": "bf16 (3-product split forward, plain bf16 backward, fp32 accumulate)"}
NCU_TRAFFIC = os.path.join(ROOT, "profiles", "gemm_traffic.json")   # written from the round's `ncu --set full` capture


def roofline_from_timing(L, out5, n_steps, ms_step, alg_flop_step, peak_tf, peak_src, workload=None):
    """roofline of the dominant kernel family from the live CUDA-event timing of EVERY tcgen05 GEMM launch."""
    k_ms, k_flop, k_mma, k_n, k_bytes = (out5[i] / n_steps for i in range(5))
    achieved = k_flop / (k_ms * 1e-3) / 1e12
    traffic = src = kernel = None
    if os.path.isfile(NCU_TRAFFIC):
        t = json.load(open(NCU_TRAFFIC))
        t = t.get(workload, t) if workload else t
        traffic, src = t.get("dram_bytes_per_launch"), t.get("source")
        kernel = t.get("kernel")
    return {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
            "traffic": traffic, "traffic_source": src, "peak_source": peak_src,
            "kernel": "sdf_fused_kernel (fused forward-only SDF chain: encoding + 8 tcgen05 layers + head)" if workload == "C5" else
                      "gemm_tc2_kernel / gemm_tc_kernel / sdf_fused_kernel (tcgen05 GEMM of every dense layer; the sampler's forward-only chains fused)",
            "traffic_kernel": kernel,
            "launches_per_step": k_n, "kernel_ms_per_step": k_ms, "share_of_step": k_ms / ms_step,
            "algorithmic_tflop_per_step_in_kernel": k_flop / 1e12,
            "algorithmic_hbm_gb_per_step_in_kernel": k_bytes / 1e9,
            "algorithmic_hbm_gbs_in_kernel": k_bytes / (k_ms * 1e-3) / 1e9,
            "mma_tflops_incl_split_products": k_mma / (k_ms * 1e-3) / 1e12,
            "mma_frac_of_peak": k_mma / (k_ms * 1e-3) / 1e12 / peak_tf,
            "step_level": {"algorithmic_tflop_per_step": alg_flop_step / 1e12, "achieved": alg_flop_step / (ms_step * 1e-3) / 1e12,
                           "frac": alg_flop_step / (ms_step * 1e-3) / 1e12 / peak_tf}}


def bench_c5(args, rank, world, local):
    """BASELINE config 5: the SDF half of extract_mesh (utils/visualization.py:36-107) on the dense dim^3 lattice.
    A step = one full lattice.  metric: SDF queries/s."""
    import ctypes as C

    w = WORKLOADS["C5"]
    dim = args.dim or w["dim"]
    n = dim ** 3
    config = {"workload": w["name"] if dim == 512 else f"dense {dim}^3 SDF lattice", "grid_dim": dim, "queries_per_step": n,
              "chunk_rows": args.chunk_rows, "parallelism": f"dp{world} (get_local_split slices + all_gather)" if world > 1 else "single",
              "l2": f"each step streams {n * 16 / 1e9:.1f} GB of points+SDF and GBs of inter-layer activations: far beyond the 126 MB L2"}
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import ref_runner, synth
        from oracle.make_golden import build_reference

        threads = min(os.cpu_count() or 1, 64)
        torch.set_num_threads(threads)
        m = build_reference(synth.PathConfig(), synth.make_params(seed=0))
        chunk, n_chunks = 102144, 2                           # scripts/sdf_extract.sh:15 --chunk 102144
        pts = (torch.rand(chunk, 1, 3) * 2 - 1)
        times = []
        with torch.no_grad():
            for it in range(max(0, args.warmup) + max(1, args.steps)):
                t0 = time.perf_counter()
                for _ in range(n_chunks):
                    m["renderer"].sdf(pts)
                if it >= max(0, args.warmup):
                    times.append(time.perf_counter() - t0)
        dt = sum(times) / len(times)
        qps = chunk * n_chunks / dt
        print(json.dumps({"impl": "reference", "metric": "SDF grid queries/sec", "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
                          "steps": max(1, args.steps), "warmup": max(0, args.warmup), "ms_per_step": dt * 1e3, "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "reference",
                                           "sample": f"{n_chunks} chunks of {chunk} points through the UNMODIFIED reference NeuconWRenderer.sdf (torch CPU fp32)"},
                          "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    assert torch.cuda.is_available(), "bench.py --impl nrw needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from nrw import _lib
    from nrw.mesh import sdf_volume
    from nrw.train import TrainSystem

    L = _lib.lib()
    sysm = TrainSystem(device, precision=args.precision, chunk_rows=args.chunk_rows, world_size=world, seed=66)
    host_out = torch.empty(n, dtype=torch.float32).pin_memory() if rank == 0 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(k, e2e):
        for _ in range(k):
            vol, _, _ = sdf_volume(sysm.renderer, dim, chunk=1 << 20)
            if e2e and rank == 0:
                host_out.copy_(vol.reshape(-1), non_blocking=True)     # what marching cubes consumes on the host
            if e2e:
                torch.cuda.synchronize()
        return vol

    run(max(args.warmup, 1) if dim >= 512 else max(args.warmup, 3), False)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = L.nrw_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); e0.record(); vol = run(args.steps, False); e1.record(); barrier()
    if args.dump_outputs and rank == 0:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
        dump_outputs(args.dump_outputs, {"sdf_volume_sample": vol.reshape(-1)[idx.to(device)]})
    launches = (L.nrw_launch_count() - l0) // max(args.steps, 1)
    ms = e0.elapsed_time(e1) / args.steps
    clk = clocks.stop() if rank == 0 else None
    barrier(); e0.record(); run(args.steps, True); e1.record(); barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    L.nrw_gemm_timing(1, None)
    run(1, False)
    torch.cuda.synchronize()
    out5 = (C.c_double * 5)()
    L.nrw_gemm_timing(0, out5)
    barrier()
    if rank == 0:
        peak_tf, peak_hbm, peak_src = peaks()
        # one rank evaluates n/world queries; the roofline object describes rank 0's kernels
        roof = roofline_from_timing(L, out5, 1, ms, F_SDF_VALUE * n / world, peak_tf, peak_src, workload="C5")
        line = {"metric": "SDF grid queries/sec", "value": n / (ms * 1e-3), "unit": "queries/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": DTYPES[args.precision], "data": "synthetic", "config": config, "precision_mode": args.precision,
                "clocks": clk, "gpu_launches": int(launches),
                "sdf_min_max": [float(vol.min()), float(vol.max())],
                "e2e": {"value": n / (ms_e2e * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": 24,
                        "d2h_bytes_per_step": n * 4, "ms_per_step": ms_e2e,
                        "note": "input = the lattice description (origin, radius, dim); output = the full SDF volume copied to pinned host memory"},
                "roofline": roof}
        if not args.no_torch_gpu_ref:
            try:
                from oracle import synth
                from oracle.make_golden import build_reference
                m = build_reference(synth.PathConfig(), synth.make_params(seed=0))
                m["neuconw"].to(device)
                chunk = 102144
                pts = (torch.rand(chunk, 1, 3, device=device) * 2 - 1)
                with torch.no_grad():
                    for _ in range(3):
                        m["renderer"].sdf(pts).cpu()
                    torch.cuda.synchronize()
                    e0.record()
                    for _ in range(20):
                        m["renderer"].sdf(pts).detach().cpu()            # utils/visualization.py:78-79: per-chunk .cpu()
                    e1.record()
                    torch.cuda.synchronize()
                rms = e0.elapsed_time(e1) / 20
                gref = {"value": chunk / (rms * 1e-3), "unit": "queries/s", "kind": "reference",
                        "sample": f"20 chunks of {chunk} points (scripts/sdf_extract.sh chunk) through the UNMODIFIED reference NeuconWRenderer.sdf "
                                  "on this GPU incl. the per-chunk .cpu() of utils/visualization.py:79",
                        "speedup_of_this_arm": line["value"] / (chunk / (rms * 1e-3)),
                        "e2e_speedup_of_this_arm": line["e2e"]["value"] / (chunk / (rms * 1e-3))}
                line["reference_torch_gpu"] = gref
                line["roofline"]["reference_torch_gpu"] = gref
            except Exception as e:  # noqa
                line["reference_torch_gpu"] = {"error": str(e)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


F_SDF_VALUE = 4195328 - 2 * 512 * 512     # value-only query: lin8 reduces to its sdf row (512 MACs), not 513 x 512


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="nrw", choices=["nrw", "reference"])
    ap.add_argument("--precision", default=os.environ.get("NRW_PRECISION", DEFAULT_PRECISION), choices=["bf16x3", "mixed", "bf16", "bf16x6"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--rays", type=int, default=0)
    ap.add_argument("--dim", type=int, default=0)
    ap.add_argument("--chunk_rows", type=int, default=int(os.environ.get("NRW_CHUNK_ROWS", 262144)))
    ap.add_argument("--cpu_rays", type=int, default=512)
    ap.add_argument("--cache_rays", type=int, default=1 << 21, help="rows of the synthetic device-resident ray cache")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_torch_gpu_ref", action="store_true")
    ap.add_argument("--no_other_modes", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32, < 64 MB in all)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.workload == "C5":
        return bench_c5(args, rank, world, local)
    w = dict(WORKLOADS[args.workload])
    if args.rays:
        w["rays"] = args.rays
    k = w["up_sample_steps"]
    fine = bool(w.get("fine"))
    S = w["n_samples"] + k * (w["n_importance"] // k) + (w.get("boundary_samples", 0) if fine else 0)
    config = {"workload": w["name"], "rays_per_gpu": w["rays"], "samples_per_ray": S, "outside_samples": w["n_outside"],
              "batch_source": f"fresh batch every step from a device-resident synthetic ray cache ({args.cache_rays} rows, reference layout "
                              "rays[n,12]/rgbs[n,3]; on-GPU permutation gather + RAY_MASK_LIST filter inside the timed region)",
              "l2": "per-step working set (>= 4 GB of chunk activations) far exceeds the 126 MB L2; no flush needed",
              "parallelism": f"dp{world}" if world > 1 else "single"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        threads = min(os.cpu_count() or 1, 64)   # beyond ~64 threads MKL on these layer sizes slows down
        rps, dt, kind = cpu_reference(args.workload, args.cpu_rays, max(1, args.steps), max(0, args.warmup), threads)
        src = {"reference": "UNMODIFIED reference NeuconWRenderer.render + NeuconWLoss + backward + clip + Adam (oracle/_ref, torch CPU fp32)",
               "port": "oracle/neuconw_port.py restatement (no reference copy on this box), torch CPU fp32"}[kind]
        line = {"impl": "reference", "metric": "training rays/sec", "value": rps, "unit": "rays/s", "n_gpus": args.gpus,
                "steps": max(1, args.steps), "warmup": max(0, args.warmup), "ms_per_step": dt * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": rps, "unit": "rays/s", "cores": threads, "kind": kind,
                                 "sample": f"{args.cpu_rays} of the {w['rays']} rays x {S} samples per step; {src}"},
                "e2e": {"value": rps, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ product arm
    assert torch.cuda.is_available(), "bench.py --impl nrw needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    import ctypes as C
    from nrw import _lib
    from nrw.raycache import RayCache, synthetic_cache
    from nrw.synthetic import install_synthetic_scene, make_ray_batch
    from nrw.train import TrainSystem

    L = _lib.lib()
    R = w["rays"]

    def make_system(precision):
        sysm = TrainSystem(device, n_samples=w["n_samples"], n_importance=w["n_importance"], up_sample_steps=k,
                           n_outside=w["n_outside"], precision=precision, chunk_rows=args.chunk_rows,
                           batch_size=R, world_size=world, seed=66)
        info = None
        if fine:      # config C3: SDF-derived octree (octree_update, neuconw_system.py:268-312) -> surface-guided fine sampling
            import nrw.octree as noct
            r = sysm.renderer
            install_synthetic_scene(r)
            r.octree_data = r.get_octree(device)
            scale = float(r.octree_data["scale"])
            train_level = int(math.ceil(math.log2(2 * scale / 0.02)))          # NeuconWSystem.surface_level, TRAIN_VOXEL_SIZE
            r.sample_range, r.boundary_samples = w["sample_range"], w["boundary_samples"]
            fo = noct.octree_update(r, train_level, 0.0)
            info = {"coarse_level": int(r.octree_data["level"]), "fine_level": int(fo["level"]), "fine_voxel": float(fo["voxel_size"]),
                    "fine_leaf_voxels": int(fo["spc_data"]["pyramid"][0, int(fo["level"])])}
        return sysm, info

    sysm, fine_info = make_system(args.precision)
    if fine_info:
        config["fine_octree"] = fine_info
    c_rays, c_rgbs = synthetic_cache(args.cache_rays, n_images=256, seed=1 + rank)   # this rank's shard
    cache = RayCache(c_rays, c_rgbs, batch_size=R, device=device, seed=100 + rank)
    hosts = [make_ray_batch(R, seed=1 + rank + 17 * i, pin=True) for i in range(4)]    # pinned host batches (e2e arm)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(n, from_host):
        last = None
        for i in range(n):
            if from_host:
                b = {kk: v.to(device, non_blocking=True) for kk, v in hosts[i % len(hosts)].items()}
            else:
                b = cache.next_batch()
            loss = sysm.training_step(b)
            last = loss.item() if from_host else loss      # e2e: device->host read of the step's loss
        return last

    def timed(n, from_host):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        l0 = L.nrw_launch_count()
        barrier(); e0.record(); loss = run(n, from_host); e1.record(); barrier()
        return e0.elapsed_time(e1) / n, clocks.stop() if rank == 0 else None, (L.nrw_launch_count() - l0) // max(n, 1), loss

    warm = max(args.warmup, 3)
    run(warm, False)
    ms, clk, launches, loss = timed(args.steps, False)
    if args.dump_outputs and rank == 0:     # the step's loss, the parameters it updated and the gradient it applied
        eng = sysm.renderer.engine
        dump_outputs(args.dump_outputs, {"loss": loss.reshape(1), "params_flat": eng.flat, "grad_flat": eng.last_flat_grad,
                                         "embedding_a": sysm.embedding_a.weight})
    run(1, True)
    ms_e2e, clk2, _, _ = timed(args.steps, True)
    t = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    # ---- roofline of the dominant kernel: CUDA events around EVERY tcgen05 GEMM launch of two more steps.
    # Every rank runs them (the step holds the gradient all-reduce); only rank 0's kernel times are reported. ----
    L.nrw_gemm_timing(1, None)
    sysm.stage_events = []
    run(2, False)
    torch.cuda.synchronize()
    out5 = (C.c_double * 5)()
    L.nrw_gemm_timing(0, out5)
    # ---- where the step goes, per rank (CUDA events TrainSystem records in-stream at its stage boundaries, same two steps):
    # compute = forward + backward up to the all-reduce; reduce = the two NCCL all-reduces INCLUDING the wait for the slowest rank
    # (so min over ranks = the collective itself, and max over ranks of compute = what weak scaling is bounded by). ----
    ev, sysm.stage_events = sysm.stage_events, None
    acc = {}
    for (n0, a0), (n1, a1) in zip(ev, ev[1:]):
        if n1 != "start":
            acc[n1] = acc.get(n1, 0.0) + a0.elapsed_time(a1) / 2
    st = torch.tensor([acc.get("forward", 0.0) + acc.get("backward", 0.0), acc.get("reduce", 0.0), acc.get("optimizer", 0.0)],
                      device=device, dtype=torch.float64)
    st_all = [torch.zeros_like(st) for _ in range(world)]
    if world > 1:
        dist.all_gather(st_all, st)
    else:
        st_all = [st]
    stages = {"compute_ms_per_rank": [round(float(x[0]), 3) for x in st_all], "reduce_ms_per_rank": [round(float(x[1]), 3) for x in st_all],
              "optimizer_ms_per_rank": [round(float(x[2]), 3) for x in st_all],
              "note": "2 steps after the timed region with per-launch GEMM events on; reduce includes waiting for the slowest rank "
                      "(min over ranks = the NCCL all-reduces themselves)"}
    trace_share = None
    if fine and rank == 0:      # share of the step spent tracing the SDF-derived octree (K1a)
        r = sysm.renderer
        rays = cache.next_batch()["rays"]
        ro = ((rays[:, 0:3] - r.origin.to(device).float()) / r.radius).float().contiguous()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(20):
            r.get_near_far_sdf(r.fine_octree_data, ro, rays[:, 3:6].contiguous(), rays[:, 6:7] / r.radius, rays[:, 7:8] / r.radius)
        e1.record(); torch.cuda.synchronize()
        trace_share = {"octree_trace_ms_per_step": e0.elapsed_time(e1) / 20, "share_of_step": e0.elapsed_time(e1) / 20 / ms}
        r = rays = ro = None        # do not keep the first system (and its activation slots) alive through these locals
    barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    h2d = sum(v.numel() * v.element_size() for v in hosts[0].values())
    flops_step = flop_per_ray(w) * R
    peak_tf, peak_hbm, peak_src = peaks()
    line = {"metric": "training rays/sec", "value": R * world / (ms * 1e-3), "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPES[args.precision],
            "data": "synthetic", "config": config, "precision_mode": args.precision, "loss": float(loss),
            "forward_slots": list(getattr(sysm.renderer.engine, "slots", ())),
            "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": R * world / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e, "clocks": clk2},
            "roofline": roofline_from_timing(L, out5, 2, ms, flops_step, peak_tf, peak_src)}
    line["stages"] = stages
    if trace_share:
        line["octree_trace"] = trace_share
    if world == 1:
        import gc
        dev_batch = {kk: v.to(device) for kk, v in hosts[0].items()}
        if not args.no_other_modes:
            others = {}
            for mode in ("bf16x3", "mixed", "bf16"):
                if mode == args.precision:
                    continue
                try:
                    sysm = None                      # free the previous system's 90 GB of activation slots first
                    gc.collect()
                    torch.cuda.empty_cache()
                    sysm, _ = make_system(mode)
                    for _ in range(3):
                        sysm.training_step(cache.next_batch())
                    m, _, _, _ = timed(args.steps, False)
                    others[mode] = {"value": R / (m * 1e-3), "unit": "rays/s", "ms_per_step": m, "dtype": DTYPES[mode],
                                    "forward_slots": list(getattr(sysm.renderer.engine, "slots", ()))}
                except Exception as e:  # noqa
                    others[mode] = {"error": str(e)[:200]}
            line["other_precision_modes"] = others
        sysm = None
        gc.collect()
        torch.cuda.empty_cache()
        if not args.no_torch_gpu_ref and not fine:
            try:
                rps, rms, n_ref, kind = torch_gpu_reference(args.workload, R, 20, 5, device)
                gref = {"value": rps, "unit": "rays/s", "ms_per_step": rms, "kind": kind, "rays": n_ref, "steps": 20, "warmup": 5,
                        "speedup_of_this_arm": line["value"] / rps, "e2e_speedup_of_this_arm": line["e2e"]["value"] / rps,
                        "sample": f"{n_ref} rays x {S} samples per step, full training step of the "
                                  f"{'UNMODIFIED reference (oracle/_ref)' if kind == 'reference' else 'restated port'} on this GPU (stock torch fp32 / cuBLAS)"}
                line["reference_torch_gpu"] = gref
                line["roofline"]["reference_torch_gpu"] = gref       # kept by the driver with the roofline object
            except Exception as e:  # noqa
                line["reference_torch_gpu"] = {"error": str(e)[:200]}
            gc.collect()
            torch.cuda.empty_cache()
        if not args.no_cpu_baseline and not fine:
            threads = min(os.cpu_count() or 1, 64)   # beyond ~64 threads MKL on these layer sizes slows down
            rps, dt, kind = cpu_reference(args.workload, args.cpu_rays, 2, 1, threads)
            line["cpu_baseline"] = {"value": rps, "unit": "rays/s", "cores": threads, "kind": kind,
                                    "sample": f"{args.cpu_rays} of the {R} rays x {S} samples per step, 1 warm-up + 2 timed full training steps "
                                              f"({'UNMODIFIED reference, oracle/_ref' if kind == 'reference' else 'restated port'}, torch CPU fp32)"}
            if "reference_torch_gpu" in line and "value" in line["reference_torch_gpu"]:
                line["cpu_baseline"]["gpu_reference"] = line["reference_torch_gpu"]
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py - headline benchmark of the B200 Grad-Shafranov hot path.

Default workload (BASELINE.json configs[2], the configuration the metric is quoted on): a UQ sweep of
independent ITER-like 129x129 FREE-BOUNDARY H-mode equilibria with perturbed coil currents, plasma current and
pedestal parameters (SURVEY.md 8d config 3) - `FusionKernel.solve_free_boundary(coils, max_outer_iter=20, tol=1e-4)`
of the reference for every sample, i.e. the outer loop of fusion_kernel_free_boundary.py:623-739 (coil
Green's-function flux on the wall, SI mu0) around the Picard + multigrid inner solve.  `--batch` equilibria PER GPU
(weak scaling; 4096 at N=1 is the named configuration) or in TOTAL with `--scaling strong` (4096 over N GPUs is
the north_star target).  One "step" = one complete batched solve.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--workload free_boundary|fixed_boundary|slab]
                    [--scaling weak|strong] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = converged equilibria/s with the per-sample inputs already resident in
HBM; `e2e` = the same metric through the public host API (BatchedFusionKernel.solve_free_boundary: host arrays in,
staged through pinned memory; every flux map, current density and summary row back into pinned host memory).
`roofline` is for the dominant kernel (k_picard_resident), timed live with CUDA events on its stream
(gsb_timing); `plasma_wall` times the same sweep with the plasma's own wall flux M @ (J dA) inside the loop and
carries the FP64-tensor roofline of that GEMM against a cuBLAS DGEMM measured in the same run; `fixed_boundary` is
round 1's headline workload (one Picard solve per sample, vacuum-field wall) for continuity.  `cpu_baseline` /
`--impl reference` time the NumPy port of the reference's CPU path (oracle/gs_oracle.py - the reference itself is
Python and cannot travel to the GPU box) on all host cores the way the reference runs sweeps
(tools/parallel_gen_iter.py: a process pool).  `parity_checked` = samples of this very run compared with the
oracle (psi rel-L2 <= 1e-9, outer iterations equal, Picard iterations +-1 per inner solve).

`--workload slab` is BASELINE configs[4]: ONE 4097^2 multigrid_solve, slab-decomposed over the N ranks (strong
scaling), GLUPS per V-cycle against the 261 B/point HBM roofline.

`--dump-outputs DIR` writes, after the timed steps, what the timed path returned in its last step (rank 0) as
DIR/<name>.npy in float64: psi, j_phi, psi_ext, summary, fb_summary of the batch (fixed_boundary: psi, j_phi,
summary; slab: the owned psi rows and residual_linf, cycles, converged).  The inputs are seeded, so two builds run
with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID = 129
COIL_SCALE = 1.0e6  # config currents are MA; the reference's SI-mu0 coil flux wants amperes (tests/golden/make_golden.py)
# Measured constants of the dominant kernel from this round's committed ncu --set full capture (profiles/);
# None until a capture of the current kernel exists.
# r2 captures (profiles/r2_picard_resident.md) of ONE k_picard_resident launch = one 4096-sample fixed-boundary sweep,
# 367 540 Picard iterations, final code of the round: DRAM 2.55 GB read + 38.42 GB written (135.8 GB before the J plane
# was dropped from the per-CTA workspace), FP64 pipe 26.3 % active.
TRAFFIC_NCU_PER_ITER = 40.97e9 / 367540.0    # DRAM bytes per Picard iteration (workspace write-back dominates)
DP_WARP_INSTR_PER_ITER = 151.3e3             # FP64 warp instructions per Picard iteration (pipe-active cycles x 4 / 2)
NCU_SOURCE = "profiles/r2_picard_resident.md"
ITER_COILS = [(3.5, 3.0, -1.0), (8.0, 3.0, 4.0), (9.5, 0.0, 6.0), (8.0, -3.0, 4.0), (3.5, -3.0, -1.0),
              (9.5, 3.0, 3.0), (2.1, 0.0, 0.0)]
PSI_TOL = 1e-9
BYTES_PER_POINT_ITER = 350.0  # SURVEY.md 8d: 261 (V-cycle, all levels) + 89 (topology, source, relax, residual)
DUMP_BYTES = 60_000_000  # --dump-outputs stays below 64 MB, .npy headers included
DUMP_SEED = 0


def base_config(n: int = GRID) -> dict:
    """validation/iter_config.json of the reference, H-mode profiles, n x n grid."""
    return {
        "reactor_name": "ITER-Like-Demo", "grid_resolution": [n, n],
        "dimensions": {"R_min": 2.0, "R_max": 10.0, "Z_min": -4.0, "Z_max": 4.0},
        "physics": {"plasma_current_target": 15.0, "vacuum_permeability": 1.0, "profiles": {"mode": "h-mode"}},
        "coils": [{"name": f"C{i}", "r": r, "z": z, "current": c} for i, (r, z, c) in enumerate(ITER_COILS)],
        "solver": {"max_iterations": 500, "convergence_threshold": 1e-4, "relaxation_factor": 0.1},
    }


def uq_inputs(batch: int, seed0: int = 2026):
    """Per-sample perturbations (SURVEY.md 8d config 3; tools/parallel_gen_iter.py:96-101)."""
    base = np.array([c[2] for c in ITER_COILS])
    cc = np.empty((batch, len(base)))
    ip = np.empty(batch)
    ped = np.empty((batch, 4))
    for k in range(batch):
        rng = np.random.default_rng(seed0 + k)
        cc[k] = base * rng.uniform(0.85, 1.15, size=len(base))
        ip[k] = 15.0 * rng.uniform(0.8, 1.2)
        ped[k] = [0.92 * rng.uniform(0.97, 1.03), 0.05 * rng.uniform(0.9, 1.1), 1.0 * rng.uniform(0.9, 1.1),
                  0.3 * rng.uniform(0.9, 1.1)]
    return cc, ip, ped


def workload_text(workload: str, grid: int, batch: int, scaling: str) -> str:
    per = "per GPU" if scaling == "weak" else "in total, sharded over the GPUs"
    if workload == "free_boundary":
        return (f"UQ sweep of {batch} independent ITER-like {grid}x{grid} free-boundary H-mode equilibria {per} "
                "(BASELINE configs[2]): solve_free_boundary(max_outer_iter=20, tol=1e-4) per sample - SI coil flux on "
                "the wall, Picard+multigrid inner solves; coil currents x U(0.85,1.15), Ip x U(0.8,1.2), pedestal "
                "params +-3-10 %")
    return (f"UQ sweep of {batch} independent ITER-like {grid}x{grid} H-mode equilibria {per} (one solve_equilibrium "
            "per sample, vacuum-field wall; round 1's headline); coil currents x U(0.85,1.15), Ip x U(0.8,1.2), "
            "pedestal params +-3-10 %")


def static_config(args, batch_per_gpu: int, total: int) -> dict:
    """The workload description: identical in the B200 arm and in the reference arm (run-dependent numbers live in
    `stats`, the reference arm's bounded sample in `cpu_baseline.sample`)."""
    n_pts = args.grid ** 2
    return {"workload": workload_text(args.workload, args.grid, args.batch, args.scaling),
            "grid": [args.grid, args.grid], "batch_per_gpu": batch_per_gpu, "global_batch": total,
            "method": "picard+multigrid(3,3,omega=1.6)", "tol": 1e-4,
            "l2_policy": f"working set {3 * batch_per_gpu * n_pts * 8 / 2 ** 20:.0f} MiB of fields per step exceeds the "
                         "126 MB L2" if batch_per_gpu * n_pts * 8 > 126e6 else
                         "working set fits L2 (small --batch run; not the headline configuration)"}


# ------------------------------------------------------------------------------------ CPU arm
def _cpu_one(args):
    cfg, cc, ip, ped, workload, keep = args
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gs_oracle as G
    scale = COIL_SCALE if workload == "free_boundary" else 1.0
    for coil, cur in zip(cfg["coils"], cc):
        coil["current"] = float(cur) * scale
    cfg["physics"]["plasma_current_target"] = float(ip)
    pd = dict(zip(("ped_top", "ped_width", "ped_height", "core_alpha"), (float(v) for v in ped)))
    cfg["physics"]["profiles"] = {"mode": "h-mode", "p_prime": pd, "ff_prime": dict(pd)}
    prob = G.PicardProblem(cfg)
    if workload == "free_boundary":
        pos = [(c["r"], c["z"]) for c in cfg["coils"]]
        r = G.free_boundary_solve(prob, pos, [c["current"] for c in cfg["coils"]], [1] * len(pos), max_outer_iter=20,
                                  tol=1e-4)
        out = {"outer": r["outer_iterations"], "inner": list(r["inner_iterations"]), "converged": r["final_diff"] < 1e-4}
    else:
        r = G.picard_solve(prob)
        out = {"outer": 1, "inner": [r["iterations"]], "converged": bool(r["converged"])}
    if keep:
        out["psi"] = np.array(prob.Psi)
    return out


def cpu_sweep(n_samples: int, cores: int, seed0: int, workload: str, grid: int = GRID, keep: int = 0, pool=None):
    """Time `n_samples` oracle solves on a `cores`-process pool; returns (eq/s, seconds, per-sample results)."""
    import multiprocessing as mp
    cc, ip, ped = uq_inputs(n_samples, seed0)
    jobs = [(base_config(grid), cc[k], ip[k], ped[k], workload, k < keep) for k in range(n_samples)]
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores)
        pool.map(_cpu_one, [j[:5] + (False,) for j in jobs[:cores]])  # warm the workers (imports, page-in)
    try:
        t0 = time.perf_counter()
        out = pool.map(_cpu_one, jobs)
        dt = time.perf_counter() - t0
    finally:
        if own:
            pool.close()
            pool.join()
    return n_samples / dt, dt, out


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if args.workload == "slab":
        print(json.dumps({"impl": "reference", "unavailable": "the slab workload has no CPU arm in bench.py "
                          "(tests/golden/make_golden.py mg_4097 times the reference's multigrid_solve: minutes per solve)"}))
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    n = max(cores, 2)  # one sample per core and step: K steps stay within a few minutes (3.6 s per free-boundary sample)
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    pool = mp.get_context("fork").Pool(cores)
    times, rates = [], []
    try:
        for s in range(max(args.warmup, 1)):  # warm-up steps: imports, page-in, first-touch of every worker
            cpu_sweep(min(n, cores), cores, 2026, args.workload, args.grid, pool=pool)
        for s in range(args.steps):
            rate, dt, _ = cpu_sweep(n, cores, 2026 + 1000 * s, args.workload, args.grid, pool=pool)
            times.append(dt)
            rates.append(rate)
    finally:
        pool.close()
        pool.join()
    value = float(np.mean(rates))
    if args.scaling == "strong":
        total, per_gpu = args.batch, -(-args.batch // max(world, 1))
    else:
        total, per_gpu = world * args.batch, args.batch
    line = {
        "impl": "reference", "metric": "converged_equilibria_per_s", "value": value, "unit": "equilibria/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config(args, per_gpu, total),
        "cpu_baseline": {"value": value, "unit": "equilibria/s", "cores": cores, "kind": "port",
                         "sample": f"each step solves a bounded sample of {n} of the equilibria on a {cores}-process pool "
                                   "(NumPy port of the reference's solve_free_boundary / solve_equilibrium; the reference "
                                   "is Python and cannot travel to the GPU box)"},
        "e2e": {"value": value, "unit": "equilibria/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU arm
class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled DURING the timed region.  Uses NVML in-process (a query costs
    microseconds); spawning nvidia-smi every 200 ms stalls the driver long enough to distort the
    host-driven e2e leg.  Falls back to nvidia-smi only if NVML is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        bits = [getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
        return [str(sm), str(mx)] + ["Active" if (r & b) else "Not Active" for b in bits]

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self.samples.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                    parts = [p.strip() for p in out.strip().split(",")]
                    if len(parts) >= 6:
                        self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.05 if self.nvml is not None else 0.5)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy kernel)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(out_dir: str, fields: dict, scalars: dict | None = None) -> None:
    """Write device tensors that share a leading axis (the equilibria of a batch, or the rows of a slab) as
    <out_dir>/<name>.npy, float64.  When together they exceed DUMP_BYTES, every field keeps the same sorted sample of
    that axis, drawn with DUMP_SEED, so runs with the same arguments stay comparable entry for entry.  `scalars` are
    written as 0-d arrays."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = next(iter(fields.values())).shape[0]
    per_entry = sum(t.element_size() * t.numel() // n for t in fields.values())
    keep = min(n, DUMP_BYTES // per_entry)
    if keep < 1:
        raise SystemExit(f"bench.py: one entry of the outputs ({per_entry} B) exceeds the --dump-outputs budget")
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, keep, replace=False))
    for name, t in fields.items():
        a = t.index_select(0, torch.as_tensor(idx, device=t.device)).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64, copy=False))
    for name, v in (scalars or {}).items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


class _Dist:
    """torch.distributed plumbing (one process per GPU under torchrun); no data-path collective is used by the
    batch workloads - only the barrier and the reductions of the timing / convergence scalars."""

    def __init__(self):
        import torch
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product path)")
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{self.local}"))
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, v: float, op: str) -> float:
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([v], device=f"cuda:{self.local}", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def timed(self, fn, steps, launch_count):
        """K steps bracketed by barrier + synchronize on both sides, CUDA events, MAX over ranks."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = launch_count()
        e0.record()
        last = None
        for _ in range(steps):
            last = fn()
        e1.record()
        self.barrier()
        return self.reduce(e0.elapsed_time(e1), "max"), launch_count() - l0, last

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def dgemm_peak_tflops(torch, local: int) -> float:
    """cuBLAS DGEMM 8192^3 on this box, best of 3 (the FP64 tensor-pipe peak the wall GEMM is compared with)."""
    n = 8192
    a = torch.randn((n, n), dtype=torch.float64, device=f"cuda:{local}")
    b = torch.randn((n, n), dtype=torch.float64, device=f"cuda:{local}")
    best = 0.0
    torch.matmul(a, b)
    torch.cuda.synchronize()
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def run_gpu_arm(args) -> None:
    import torch
    import scpn_fusion_core_b200 as pkg
    from scpn_fusion_core_b200 import _device as D
    from scpn_fusion_core_b200 import _lib
    from scpn_fusion_core_b200.fusion_kernel import shard_range

    dd = _Dist()
    world, rank, local = dd.world, dd.rank, dd.local
    free_boundary = args.workload == "free_boundary"
    if args.scaling == "strong":
        lo, hi = shard_range(args.batch, world, rank)
    else:
        lo, hi = rank * args.batch, (rank + 1) * args.batch
    B = hi - lo
    if B < 1:
        raise SystemExit("bench.py: fewer equilibria than ranks")
    total = args.batch if args.scaling == "strong" else world * args.batch
    cfg = base_config(args.grid)
    bk = pkg.BatchedFusionKernel(cfg, device=local)
    # strong scaling: sample k of the ONE sweep is seeded 2026 + k whatever the rank layout.  Weak scaling: every GPU
    # solves the named 4096-sample sweep (seeds 2026 .. 2026 + B - 1), so per-GPU work is identical by construction and
    # a straggler (one sample in ~8000 of a longer seed range does not converge within 500 Picard iterations and keeps
    # a single SM busy for every remaining outer iteration) cannot masquerade as a scaling loss.
    cc, ip, ped = uq_inputs(B, 2026 + (lo if args.scaling == "strong" else 0))
    ped8 = np.concatenate([ped, ped], axis=1)
    mu0 = cfg["physics"]["vacuum_permeability"]
    w_fixed = (mu0 * cc) / (2.0 * np.pi)      # calculate_vacuum_field weights (fusion_kernel.py:245-249)
    cc_si = cc * COIL_SCALE                   # I * turns (turns = 1), SI amperes
    dev_in = lambda a: D.to_device(a, local)
    w_dev, wsi_dev, ip_dev, ped_dev = dev_in(w_fixed), dev_in(cc_si), dev_in(ip), dev_in(ped8)
    psi_buf = D.empty((B, args.grid, args.grid), local)
    j_buf = D.empty((B, args.grid, args.grid), local)
    pinned = bk.pinned_outputs(B)
    ctx = bk._context(B)

    def step_fb(plasma_wall=False):
        return bk.solve_free_boundary_device(wsi_dev, ip_dev, ped_dev, psi_out=psi_buf, jphi_out=j_buf,
                                             max_outer_iter=20, tol=1e-4, plasma_wall=plasma_wall)

    def step_fixed():
        return bk.solve_device(w_dev, ip_dev, ped_dev, psi_out=psi_buf, jphi_out=j_buf)

    def step_e2e():
        # the public batched entry point: host arrays in (staged through pinned memory by the API), flux maps, current
        # densities and summary rows out into pinned host memory; everything inside the timed region
        if free_boundary:
            return bk.solve_free_boundary(cc_si, ip, ped, ped, max_outer_iter=20, tol=1e-4, out=pinned)
        return bk.solve(cc, ip, ped, ped, out=pinned)

    step_resident = step_fb if free_boundary else step_fixed
    warm = max(args.warmup, 3)
    for _ in range(warm):
        last = step_resident()
    sampler = ClockSampler(local)
    sampler.start()
    ms, launches, last = dd.timed(step_resident, args.steps, _lib.launch_count)
    if args.dump_outputs and rank == 0:  # before the legs below reuse psi_buf / j_buf
        dump_outputs(args.dump_outputs, last)
    summ = last["summary"].cpu().numpy()
    if free_boundary:
        fbs = last["fb_summary"].cpu().numpy()
        conv_mask = (summ[:, 1] > 0.5) & (fbs[:, 3] > 0.5)
        iters = fbs[:, 2]
        outer = fbs[:, 0]
    else:
        conv_mask = summ[:, 1] > 0.5
        iters = summ[:, 0]
        outer = np.ones(B)
    psi_check = last["psi"][:4].cpu().numpy()
    n_conv = int(dd.reduce(float(conv_mask.sum()), "sum"))
    it_sum_all = dd.reduce(float(iters.sum()), "sum")
    for _ in range(2):
        step_e2e()
    ms_e2e, _, last_e2e = dd.timed(step_e2e, args.steps, _lib.launch_count)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    clocks = sampler.summary()

    # ---- dominant kernel: k_picard_resident, CUDA events on its stream inside the library (gsb_timing) ----
    n_pts = args.grid ** 2
    n_int = (args.grid - 2) ** 2
    peak, peak_src = measured_peak_hbm()
    out4 = (4 * _lib.c_double)()
    reps = max(1, min(args.steps, 3))
    if free_boundary:
        _lib.check(ctx.lib.gsb_timing(ctx.handle, 1, None, 1))
        l0 = _lib.launch_count()
        for _ in range(reps):
            rr = step_fb()
        torch.cuda.synchronize()
        launches_one = (_lib.launch_count() - l0) / reps
        _lib.check(ctx.lib.gsb_timing(ctx.handle, 0, out4, 1))
        k_ms_total, k_launches = out4[0] / reps, out4[1] / reps
        it_sum = float(rr["fb_summary"].cpu().numpy()[:, 2].sum())
        resident = launches_one < 10 * max(outer.max(), 1)
    else:
        k_times = []
        for _ in range(reps):
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            l0 = _lib.launch_count()
            rr = bk.solve_device(w_dev, ip_dev, ped_dev, psi_out=psi_buf, jphi_out=j_buf, events=ev)
            torch.cuda.synchronize()
            launches_one = _lib.launch_count() - l0
            k_times.append(ev[0].elapsed_time(ev[1]))
        k_ms_total, k_launches = float(np.mean(k_times)), 1.0
        it_sum = float(rr["summary"].cpu().numpy()[:, 0].sum())
        resident = launches_one <= 3
    alg_bytes = BYTES_PER_POINT_ITER * n_pts * it_sum            # per step (all launches of the kernel in one step)
    achieved = alg_bytes / (k_ms_total * 1e-3) / 1e9
    roof = {"bound": "hbm",
            "kernel": "k_picard_resident (persistent: one CTA per equilibrium, psi resident in shared memory for the "
                      "whole inner solve)" if resident else "streaming Picard launch sequence (grid does not fit one SM)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "traffic": (TRAFFIC_NCU_PER_ITER * it_sum / max(k_launches, 1.0) if resident else None),
            "traffic_source": NCU_SOURCE + " (ncu dram__bytes_read.sum + dram__bytes_write.sum per Picard iteration x the "
                              "live iteration count, per launch)",
            "launch_ms": k_ms_total / max(k_launches, 1.0), "launches_per_step": k_launches,
            "algorithmic_bytes_per_launch": alg_bytes / max(k_launches, 1.0),
            "algorithmic_bytes_note": f"{BYTES_PER_POINT_ITER:.0f} B per grid point per Picard iteration x {n_pts} points x "
                                      f"{it_sum:.0f} Picard iterations per step (sum over the batch and the outer "
                                      "iterations); psi never leaves shared memory during an inner solve, so frac may "
                                      "exceed 1 - the kernel is FP64-issue bound, not HBM bound: see fp64",
            "share_of_step": k_ms_total / (ms / args.steps)}
    if resident and clocks.get("sm_mhz"):
        dp_rate = DP_WARP_INSTR_PER_ITER * 32.0 * it_sum / (k_ms_total * 1e-3)          # FP64 thread instructions / s
        dp_peak = ctx_num_sms(torch, local) * 64.0 * clocks["sm_mhz"] * 1e6             # 64 FP64 lanes / SM / clk
        roof["fp64"] = {"achieved": dp_rate / 1e12, "peak": dp_peak / 1e12, "unit": "T FP64 instr/s (DADD/DMUL/DFMA issue)",
                        "frac": dp_rate / dp_peak,
                        "source": f"{DP_WARP_INSTR_PER_ITER:.0f} FP64 warp instructions per Picard iteration ({NCU_SOURCE}) x "
                                  "the live iteration count; peak = SMs x 64 lanes x the sampled SM clock"}

    line_extra = {}
    # ---- plasma-wall variant: the lane-C wall term as one DMMA GEMM per outer iteration, with its own roofline ----
    if free_boundary and not args.no_extras:
        step_fb(True)
        torch.cuda.synchronize()
        ms_pw, _, last_pw = dd.timed(lambda: step_fb(True), reps, _lib.launch_count)
        fpw = last_pw["fb_summary"].cpu().numpy()
        _lib.check(ctx.lib.gsb_timing(ctx.handle, 1, None, 1))
        for _ in range(reps):
            step_fb(True)
        torch.cuda.synchronize()
        _lib.check(ctx.lib.gsb_timing(ctx.handle, 0, out4, 1))
        g_ms, g_n = out4[2] / reps, out4[3] / reps
        n_wall = 2 * args.grid + 2 * (args.grid - 2)
        flops = 2.0 * n_wall * n_int * B
        dgemm = dgemm_peak_tflops(torch, local) if rank == 0 else 0.0
        g_tf = flops * g_n / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
        conv_pw = int(dd.reduce(float(((fpw[:, 3] > 0.5) & (last_pw["summary"].cpu().numpy()[:, 1] > 0.5)).sum()), "sum"))
        line_extra["plasma_wall"] = {
            "value": conv_pw * reps / (ms_pw * 1e-3), "unit": "equilibria/s", "ms_per_step": ms_pw / reps,
            "converged": conv_pw, "outer_iterations_max": int(fpw[:, 0].max()),
            "what": "same sweep with wall = coil flux + M @ (J_phi dA) from the second outer iteration on (lane-C term, "
                    "jax_free_boundary_predictive.py:443-498; parity unpinned: NumPy restatement only)",
            "roofline_gemm": {"bound": "tensor", "kernel": "k_wall_gemm_big (mma.sync.m8n8k4.f64 = DMMA; tcgen05 has no "
                              "FP64 kind)", "achieved": g_tf, "peak": dgemm, "unit": "TFLOP/s",
                              "frac": g_tf / dgemm if dgemm else None,
                              "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (torch.matmul f64, best of 3)",
                              "launch_ms": g_ms / max(g_n, 1.0), "launches_per_step": g_n,
                              "shape": [B, n_wall, n_int], "flops_per_launch": flops}}
    # ---- round 1's headline workload for continuity ----
    if free_boundary and not args.no_extras:
        for _ in range(2):
            step_fixed()
        ms_fx, _, last_fx = dd.timed(step_fixed, reps, _lib.launch_count)
        sfx = last_fx["summary"].cpu().numpy()
        conv_fx = int(dd.reduce(float((sfx[:, 1] > 0.5).sum()), "sum"))
        line_extra["fixed_boundary"] = {"value": conv_fx * reps / (ms_fx * 1e-3), "unit": "equilibria/s",
                                        "ms_per_step": ms_fx / reps, "converged": conv_fx,
                                        "picard_iterations_mean": float(sfx[:, 0].mean()),
                                        "what": "round 1's headline: one solve_equilibrium per sample, vacuum-field wall"}
    # ---- secondary: the HBM-streaming smoother (what a V-cycle's smoothing uses on grids that do not fit an SM) ----
    st = D.stream_ptr()

    def time_smooth(fuse, sweeps, n_rep):
        _lib.check(ctx.lib.gsb_smooth_ex(ctx.handle, D.ptr(psi_buf), D.ptr(j_buf), B, 1.6, sweeps, 0, fuse, st))
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(n_rep):
            _lib.check(ctx.lib.gsb_smooth_ex(ctx.handle, D.ptr(psi_buf), D.ptr(j_buf), B, 1.6, sweeps, 0, fuse, st))
        f1.record()
        torch.cuda.synchronize()
        return f0.elapsed_time(f1) / n_rep

    if not args.no_extras:
        s_ms = time_smooth(3, 6, 5) / 2.0        # per launch (3 sweeps each); two launches per call, back to back
        c_ms = time_smooth(0, 3, 10) / 6.0       # per colour-pass launch
        s_bytes = 24.0 * n_int * B * 3           # 24 B/LUP per sweep (SURVEY 8d) x 3 sweeps per launch
        line_extra["roofline_streaming_smoother"] = {
            "bound": "hbm", "kernel": "k_sweep_warp<6> (3 RB-SOR sweeps = 6 colour passes per pass over HBM, whole batch, "
                                      "warp-autonomous temporal blocking)",
            "achieved": s_bytes / (s_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": s_bytes / (s_ms * 1e-3) / 1e9 / peak, "launch_ms": s_ms, "algorithmic_bytes_per_launch": s_bytes,
            "glups": (n_int * B * 3) / (s_ms * 1e-3) / 1e9,
            "per_colour_pass_kernel": {"kernel": "k_smooth_colour", "achieved": 12.0 * n_int * B / (c_ms * 1e-3) / 1e9,
                                       "frac": 12.0 * n_int * B / (c_ms * 1e-3) / 1e9 / peak, "launch_ms": c_ms,
                                       "algorithmic_bytes_per_launch": 12.0 * n_int * B}}

    if rank == 0:
        value = n_conv * args.steps / (ms * 1e-3)      # CONVERGED equilibria per second, whole job
        e2e = n_conv * args.steps / (ms_e2e * 1e-3)
        h2d = int((cc.size + ip.size + ped8.size) * 8)
        d2h = int(2 * B * n_pts * 8 + B * 16 * 8 + (B * 4 * 8 if free_boundary else 0))
        line = {
            "metric": "converged_equilibria_per_s", "value": value, "unit": "equilibria/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": static_config(args, B, total),
            "stats": {"converged": n_conv, "unconverged": total - n_conv,
                      "picard_iterations_mean": float(iters.mean()), "picard_iterations_max": int(iters.max()),
                      "outer_iterations_max": int(outer.max())},
            "e2e": {"value": e2e, "unit": "equilibria/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": ("BatchedFusionKernel.solve_free_boundary" if free_boundary else "BatchedFusionKernel.solve") +
                           "(host arrays, out=pinned_outputs(B)): inputs staged host -> device, psi AND J_phi of every "
                           "equilibrium plus the summary rows device -> pinned host, all inside the timed region"},
            "gpu_launches": int(launches),
            "glups_per_vcycle": 8.0 * n_int * it_sum_all * args.steps / (ms * 1e-3) / 1e9,
            "roofline": roof,
            "clocks": clocks,
        }
        line.update(line_extra)
        cores = os.cpu_count() or 1
        if not args.no_cpu_baseline:
            n = (2 if free_boundary else 4) * max(cores, 2)
            rate, dt, res = cpu_sweep(n, cores, 2026, args.workload, args.grid, keep=4 if lo == 0 else 0)
            its = [sum(r["inner"]) for r in res]
            line["cpu_baseline"] = {"value": rate, "unit": "equilibria/s", "cores": cores, "kind": "port",
                                    "sample": f"{n} of the {total} equilibria, {cores}-process pool, {dt:.1f} s "
                                              f"(NumPy port of the reference CPU path; Picard iterations per sample "
                                              f"{min(its)}-{max(its)})"}
            # parity of THIS run's output: the oracle solved the first samples of rank 0's batch on the same seeds
            checked = 0
            for k, r in enumerate(res[:4]):
                if "psi" not in r:
                    continue
                err = float(np.linalg.norm(psi_check[k] - r["psi"]) / np.linalg.norm(r["psi"]))
                ok = err <= PSI_TOL and int(outer[k]) == r["outer"] and abs(int(iters[k]) - sum(r["inner"])) <= r["outer"]
                if not ok:
                    raise SystemExit(f"bench.py: parity check failed on sample {k}: rel_l2={err:.3e}, outer "
                                     f"{int(outer[k])} vs {r['outer']}, Picard iterations {int(iters[k])} vs {sum(r['inner'])}")
                checked += 1
            line["parity_checked"] = checked
            line["parity_tolerance"] = "psi rel-L2 <= 1e-9, outer iterations equal, Picard iterations +-1 per inner solve"
        print(json.dumps(line), flush=True)
    dd.close()


def ctx_num_sms(torch, local: int) -> int:
    return int(torch.cuda.get_device_properties(local).multi_processor_count)


# ------------------------------------------------------------------------------------ slab workload
def run_slab(args) -> None:
    """BASELINE configs[4]: ONE n x n multigrid_solve (bench_gpu_gs_solver._problem source, psi_bc = 0, tol 1e-8,
    omega 1, 3/3, min_grid 5), Z-row slabs over the ranks; halos over NVLink peer memory when N > 1."""
    import torch
    from scpn_fusion_core_b200 import _lib
    from scpn_fusion_core_b200.slab import CudaSlabOps, SlabComm, SlabMultigrid

    dd = _Dist()
    world, rank, local = dd.world, dd.rank, dd.local
    n = args.grid if args.grid > 129 else 4097
    comm = SlabComm(rank, world)
    mgs = SlabMultigrid(n, n, 4.0, 8.0, -4.0, 4.0, comm, CudaSlabOps(local))
    peer = False
    if world > 1 and not args.slab_nccl:
        peer = comm.enable_peer_halo(local, mgs.halo * n)
        if peer and not args.slab_nccl_gather:
            comm.enable_peer_gather(local, mgs.gathered["nz"] * mgs.gathered["nr"])
    g0, g1 = mgs.owned_rows()
    z = torch.linspace(-4.0, 4.0, n, dtype=torch.float64, device=f"cuda:{local}")[g0:g1, None]
    r = torch.linspace(4.0, 8.0, n, dtype=torch.float64, device=f"cuda:{local}")[None, :]
    src = -torch.exp(-((r - 6.0) ** 2 + z ** 2) / 0.5)
    bc = torch.zeros_like(src)

    def step():
        return mgs.solve(src, bc, tol=1e-8, max_cycles=50)

    for _ in range(max(args.warmup, 3)):
        out = step()
    sampler = ClockSampler(local)
    sampler.start()
    ms, launches, out = dd.timed(step, args.steps, _lib.launch_count)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    psi, res, cycles, conv = out
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"psi": psi}, {"residual_linf": res, "cycles": cycles, "converged": conv})
    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        n_int = (n - 2) ** 2
        per_cycle_ms = ms / args.steps / cycles
        glups = 8.0 * n_int / (per_cycle_ms * 1e-3) / 1e9
        achieved = 261.0 * n * n / (per_cycle_ms * 1e-3) / 1e9
        line = {"metric": "glups_per_vcycle", "value": glups, "unit": "GLUPS", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"one {n}x{n} multigrid_solve (BASELINE configs[4]): V-cycles (3,3), omega 1.0, "
                                       f"tol 1e-8, Z-row slabs over {world} GPU(s)", "grid": [n, n], "cycles": int(cycles),
                           "converged": bool(conv), "residual_linf": float(res),
                           "halo_transport": "NVLink peer memory (gsb_halo_push/recv, CUDA IPC)" if peer else
                                             ("NCCL point-to-point" if world > 1 else "none"),
                           "coarse_gather": ("NVLink peer memory (gsb_gather_push/wait)" if comm.gather is not None else
                                             ("NCCL all-gather" if world > 1 else "none")),
                           "cuda_graph": bool(mgs.used_graph), "l2_policy": f"{n * n * 8 / 2 ** 20:.0f} MiB per field exceeds L2"},
                "ms_per_vcycle": per_cycle_ms, "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "kernel": "one multigrid V-cycle, all levels (k_sweep_warp<6>, "
                             "k_residual_restrict, k_prolong_add, resident tail)", "achieved": achieved, "peak": peak * world,
                             "unit": "GB/s", "frac": achieved / (peak * world), "peak_source": peak_src + f" x {world} GPUs",
                             "traffic": None, "algorithmic_bytes_per_launch": 261.0 * n * n,
                             "algorithmic_bytes_note": "261 B per fine-grid point per V-cycle (SURVEY.md 8d)"},
                "e2e": {"value": glups, "unit": "GLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8,
                        "api": "SlabMultigrid.solve with device-resident owned rows; the host reads the residual scalar "
                               "every cycle (inside the timed region)"},
                "clocks": sampler.summary()}
        print(json.dumps(line), flush=True)
    comm.disable_peer_gather()
    if peer:
        comm.disable_peer_halo()
    dd.close()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096, help="equilibria per GPU (weak) or in total (strong)")
    ap.add_argument("--grid", type=int, default=GRID)
    ap.add_argument("--workload", default="free_boundary", choices=["free_boundary", "fixed_boundary", "slab"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the plasma-wall / fixed-boundary / smoother legs")
    ap.add_argument("--slab-nccl", action="store_true", help="slab workload: NCCL point-to-point halos instead of peer memory")
    ap.add_argument("--slab-nccl-gather", action="store_true", help="slab workload: NCCL all-gather of the coarse level (no multi-rank graph)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last step as DIR/<name>.npy (float64, rank 0; a "
                         "fixed, seeded sample of the equilibria or rows when the whole would exceed 60 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path, not of --impl reference")
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "slab":
        run_slab(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()

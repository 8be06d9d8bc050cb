"""Throughput of the batched shape-optimising free-boundary loop (BatchedFusionKernel.solve_free_boundary with
optimize_shape=True, gsb_free_boundary_shape_solve) on one GPU.

Workload: bench.py's ITER-like H-mode UQ sweep (coil currents x U(0.85,1.15) in SI amperes, Ip x U(0.8,1.2), pedestal
+-3-10 %), re-fitting the seven coil currents every outer iteration to 8 isoflux control points around the plasma with
alpha = 1e-10 and a 6 MA limit on PF1 (20 MA on the others), max_outer_iter=20, tol=1e-4.  Batches of 1024 and 4096 at
65^2 and 129^2.  Reports, per size:
  * converged equilibria per second and the outer-iteration histogram (device events around the device entry);
  * the shape step's cost, two ways, at a fixed outer count (tol=0, 4 outer iterations): the device time of its own
    launches (k_shape_target, k_shape_fit, the coil-flux rewrite k_coil_flux; torch.profiler, separate pass) as a share
    of all device time; and the wall-time difference between optimize_shape True and False (alternated), which also
    holds the extra inner Picard iterations that the changing coil flux causes (the Picard counts of both are listed);
  * the per-equilibrium host path (FusionKernel.solve_free_boundary(optimize_shape=True): psi to NumPy and
    scipy lsq_linear every outer iteration) on 16 samples, and the speed-up at the same grid.
The card name and power limit are read in the same run.  Prints one JSON object; --out also writes it to a file.
Usage: python tools/bench_shape_sweep.py [--out FILE] [--grids 65,129] [--batches 1024,4096] [--host-samples 16]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import scpn_fusion_core_b200 as pkg  # noqa: E402
from scpn_fusion_core_b200 import _device as D  # noqa: E402

TH = np.linspace(0.0, 2.0 * np.pi, 9)[:-1] + 0.3
POINTS = np.column_stack([6.0 + 1.9 * np.cos(TH), 2.6 * np.sin(TH)])  # inside the 2..10 x -4..4 box
LIMITS = np.array([6.0e6, 20e6, 20e6, 20e6, 20e6, 20e6, 20e6])
ALPHA = 1e-10


def card() -> dict:
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, torch):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1) / 1e3


def run_size(n: int, B: int, torch) -> dict:
    cfg = bench.base_config(n)
    bk = pkg.BatchedFusionKernel(cfg)
    cc, ip, ped = bench.uq_inputs(B)
    cc = cc * 1.0e6
    ped8 = np.concatenate([ped, ped], axis=1)
    ip_d, ped_d = D.to_device(ip, bk.device), D.to_device(ped8, bk.device)
    shape = dict(optimize_shape=True, target_points=POINTS, current_limits=LIMITS, tikhonov_alpha=ALPHA)

    def sweep(max_outer, tol, with_shape):
        if with_shape:
            return bk.solve_free_boundary_device(None, ip_d, ped_d, max_outer_iter=max_outer, tol=tol,
                                                 currents=D.to_device(cc, bk.device), **shape)
        return bk.solve_free_boundary_device(D.to_device(cc, bk.device), ip_d, ped_d, max_outer_iter=max_outer,
                                             tol=tol)  # one turn per coil: w = I

    sweep(2, 0.0, True)  # warm-up: context, Green's tables, factor, every kernel
    sweep(2, 0.0, False)
    r, sec = timed(lambda: sweep(20, 1e-4, True), torch)
    fb = r["fb_summary"].cpu().numpy()
    so = r["shape_out"].cpu().numpy()
    P = POINTS.shape[0]
    outer = fb[:, 0].astype(int)
    conv = int((fb[:, 3] > 0.5).sum())
    res = {"grid": n, "batch": B, "seconds": sec, "converged": conv, "converged_eq_per_s": conv / sec,
           "eq_per_s": B / sec, "outer_iterations_histogram": {int(k): int(v) for k, v in zip(*np.unique(outer, return_counts=True))},
           "picard_iterations_mean_per_outer": float(np.mean(fb[:, 2] / outer)),
           "active_bounds_histogram": {int(k): int(v) for k, v in zip(*np.unique(so[:, 2 * P + 2].astype(int), return_counts=True))},
           "fit_fallbacks": int(so[:, 2 * P + 3].sum())}
    # shape-step cost at a fixed outer count, both variants alternated
    on, off, pic = [], [], {}
    for _ in range(2):
        r1, s1 = timed(lambda: sweep(4, 0.0, True), torch)
        r0, s0 = timed(lambda: sweep(4, 0.0, False), torch)
        on.append(s1)
        off.append(s0)
        pic = {"shape": float(r1["fb_summary"][:, 2].mean()), "plain": float(r0["fb_summary"][:, 2].mean())}
    t_on, t_off = min(on), min(off)
    res["fixed_4_outer"] = {"seconds_shape": on, "seconds_plain": off, "picard_iterations_mean": pic,
                            "wall_difference_ms_per_outer": (t_on - t_off) / 4 * 1e3,
                            "wall_difference_share": (t_on - t_off) / t_on}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sweep(4, 0.0, True)
        torch.cuda.synchronize()
    dev = {}
    for e in prof.key_averages():
        us = float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
        if us > 0:
            dev[e.key] = us
    total = sum(dev.values())
    step = {k: v for k, v in dev.items() if "k_shape_target" in k or "k_shape_fit" in k or "k_coil_flux" in k}
    res["fixed_4_outer"]["profiled"] = {
        "device_ms_total": total / 1e3, "shape_step_device_ms": sum(step.values()) / 1e3,
        "shape_step_device_share": sum(step.values()) / total,
        "shape_step_ms_per_outer": sum(step.values()) / 4e3,
        "kernels_ms": {k: v / 1e3 for k, v in sorted(dev.items(), key=lambda kv: -kv[1])[:12]}}
    return res


def host_path(n: int, samples: int, torch) -> dict:
    cfg = bench.base_config(n)
    cc, ip, ped = bench.uq_inputs(samples)
    t_total, outer = 0.0, []
    for k in range(samples + 1):  # sample 0 twice: the first call builds the context and tables
        j = max(k - 1, 0)
        c = json.loads(json.dumps(cfg))
        c["physics"]["plasma_current_target"] = float(ip[j])
        pd = dict(zip(("ped_top", "ped_width", "ped_height", "core_alpha"), (float(v) for v in ped[j])))
        c["physics"]["profiles"] = {"mode": "h-mode", "p_prime": pd, "ff_prime": dict(pd)}
        kern = pkg.FusionKernel(c)
        coils = kern.build_coilset_from_config()
        coils.currents = cc[j] * 1.0e6
        coils.target_flux_points, coils.current_limits = POINTS, LIMITS
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = kern.solve_free_boundary(coils, max_outer_iter=20, tol=1e-4, optimize_shape=True, tikhonov_alpha=ALPHA)
        torch.cuda.synchronize()
        if k:
            t_total += time.perf_counter() - t0
            outer.append(int(r["outer_iterations"]))
    return {"grid": n, "samples": samples, "seconds": t_total, "eq_per_s": samples / t_total,
            "outer_iterations": outer}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--grids", default="65,129")
    ap.add_argument("--batches", default="1024,4096")
    ap.add_argument("--host-samples", type=int, default=16)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_shape_sweep.py measures the GPU path: no CUDA device visible")
    out = {"card": card(), "workload": __doc__.split("\n\n")[0], "points": POINTS.tolist(), "limits": LIMITS.tolist(),
           "alpha": ALPHA, "batched": [], "host_path": []}
    for n in [int(v) for v in args.grids.split(",")]:
        for B in [int(v) for v in args.batches.split(",")]:
            out["batched"].append(run_size(n, B, torch))
            print(json.dumps(out["batched"][-1]), file=sys.stderr, flush=True)
        h = host_path(n, args.host_samples, torch)
        best = max(b["eq_per_s"] for b in out["batched"] if b["grid"] == n)
        h["speedup_of_best_batched_eq_per_s"] = best / h["eq_per_s"]
        out["host_path"].append(h)
        print(json.dumps(h), file=sys.stderr, flush=True)
    out["card_after"] = card()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

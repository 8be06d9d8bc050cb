"""Cost of the batched wall-contour boundary reconstruction (gsb_boundary_flux;
BatchedFusionKernel.solve_free_boundary(reconstruct_boundary=True) and reconstruct_boundary_flux_from_coils) on one GPU.

Workload: bench.py's 4096-sample ITER-like H-mode UQ sweep on 129^2 (coil currents x U(0.85,1.15) in SI amperes, one turn
per coil, Ip x U(0.8,1.2), pedestal +-3-10 %), max_outer_iter=20, tol=1e-4, with the 512-point wall contour, a 4-point
limiter, an axis point and two X-points.  Reports:
  * the C entry's CUDA-event time on the sweep's final currents and psi (wall-contour target), shared and per-sample
    axis / X-points, median of repeated launches;
  * the end-to-end wall time of solve_free_boundary with reconstruct_boundary on and off (alternated, host arrays in
    and out, as bench.py's end-to-end leg);
  * the one-sample host path (FusionKernel.reconstruct_boundary_flux_from_coils) on the same geometry for comparison.
The card name and power limit are read in the same run.  Prints one JSON object; --out also writes it to a file.
Usage: python tools/bench_boundary_sweep.py [--out FILE] [--batch 4096] [--grid 129] [--repeats 3]"""
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
from scpn_fusion_core_b200.free_boundary import _wall_contour  # noqa: E402

LIMITER = np.array([[3.9, -4.6], [8.6, -4.6], [8.6, 4.6], [3.9, 4.6]])
AXIS = np.array([6.2, 0.0])
XPTS = np.array([[5.0, -3.4], [5.0, 3.4]])


def card() -> dict:
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--grid", type=int, default=129)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--host-samples", type=int, default=64)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_boundary_sweep.py measures the GPU path: no CUDA device visible")
    out = {"card": card(), "workload": __doc__.split("Reports:")[0].strip(),
           "grid": args.grid, "batch": args.batch}
    cfg = bench.base_config(args.grid)
    bk = pkg.BatchedFusionKernel(cfg)
    B = args.batch
    cc, ip, ped = bench.uq_inputs(B)
    cc = cc * 1.0e6
    geo = dict(limiter_points=LIMITER, axis_point=AXIS, x_points=XPTS)

    def e2e(on: bool):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=20, tol=1e-4, reconstruct_boundary=on,
                                   **(geo if on else {}))
        torch.cuda.synchronize()
        return r, time.perf_counter() - t0

    e2e(False)  # warm-up: context, tables, every kernel
    r_on, _ = e2e(True)
    t_on, t_off = [], []
    for _ in range(args.repeats):
        t_off.append(e2e(False)[1])
        t_on.append(e2e(True)[1])
    vb = r_on["vacuum_boundary_abs_error"]
    out["end_to_end"] = {"seconds_off": t_off, "seconds_on": t_on,
                         "median_difference_ms": (float(np.median(t_on)) - float(np.median(t_off))) * 1e3,
                         "converged": int(np.count_nonzero(r_on["fb_converged"])),
                         "vacuum_boundary_abs_error_max": float(np.max(vb)),
                         "vacuum_boundary_abs_error_median": float(np.median(vb))}
    # the entry alone, on the sweep's final state (plain loop: the wall ring of psi is the target)
    kw = dict(max_outer_iter=20, tol=1e-4)
    dev = bk.solve_free_boundary_device(D.to_device(cc, bk.device), D.to_device(ip, bk.device),
                                        D.to_device(np.concatenate([ped, ped], axis=1), bk.device), **kw)
    pts = _wall_contour(bk)[0]
    cur = D.to_device(cc, bk.device)
    rng = np.random.default_rng(1)
    per = dict(limiter_points=LIMITER, axis_point=AXIS + rng.normal(0.0, 0.05, (B, 2)),
               x_points=XPTS[None] + rng.normal(0.0, 0.05, (B, 2, 2)))
    out["entry"] = {}
    for name, g in (("shared_points", geo), ("per_sample_points", per)):
        ms = []
        for k in range(10):
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            bk.reconstruct_boundary_flux_device(cur, boundary_points=pts, target_field=dev["psi"], events=ev, **g)
            torch.cuda.synchronize()
            if k:
                ms.append(ev[0].elapsed_time(ev[1]))
        out["entry"][name] = {"ms_median": float(np.median(ms)), "ms_min": float(np.min(ms)),
                              "samples_per_s": B / (float(np.median(ms)) / 1e3), "boundary_points": int(len(pts)),
                              "limiter_points": 4, "x_points": 2}
    # one sample at a time on the host path of FusionKernel
    k1 = pkg.FusionKernel(cfg)
    coils = k1.build_coilset_from_config()
    n = min(args.host_samples, B)
    coils.currents = cc[0].copy()
    k1.reconstruct_boundary_flux_from_coils(coils, boundary_points=pts, target_flux=np.zeros(len(pts)), **geo)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in range(n):
        coils.currents = cc[b].copy()
        k1.reconstruct_boundary_flux_from_coils(coils, boundary_points=pts, target_flux=np.zeros(len(pts)), **geo)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    out["host_one_sample"] = {"samples": n, "seconds": sec, "samples_per_s": n / sec,
                              "speedup_of_entry_shared": out["entry"]["shared_points"]["samples_per_s"] / (n / sec)}
    out["card_after"] = card()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

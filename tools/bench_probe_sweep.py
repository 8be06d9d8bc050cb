"""Throughput of the batched magnetic-probe current reconstruction
(BatchedFusionKernel.reconstruct_coil_currents_from_magnetic_probes, gsb_probe_reconstruct) on one GPU.

Workload: the ITER-like configuration of bench.py (seven coils, 129^2 grid), a synthetic diagnostic set of 32 flux loops
and 64 B probes (alternating R and Z) on two ellipses around the plasma, sigma 1e-3 on every row, alpha = 1e-10 and a
6 MA limit on PF1 (20 MA on the others, as tools/bench_shape_sweep.py).  Each sample's true currents and its prior are
two independent draws of bench.py's UQ coil currents (x U(0.85,1.15), SI amperes); its measurements are the response
of the true currents plus Gaussian noise of that sigma.  Batches of 4096 and 65536.  Reports, per batch:
  * the device time of the C entry (CUDA events around gsb_probe_reconstruct, inputs already on the device; median of
    the repeats) and fits per second;
  * the end-to-end time of the public method (response matrix, host-to-device and device-to-host copies, host
    checks; median of the repeats) and fits per second;
  * the kernel split of one call of the public method (torch.profiler, separate pass);
  * the active-bound histogram and the number of failed fits.
Then the one-sample host path (FusionKernel.reconstruct_coil_currents_from_magnetic_probes: device response matrix,
scipy lsq_linear(method="trf")) on 64 samples, its agreement with the batched currents, and the speed-up of the batched
end-to-end rate over it.  The card name and power limit are read in the same run.  Prints one JSON object; --out also
writes it to a file.
Usage: python tools/bench_probe_sweep.py [--out FILE] [--batches 4096,65536] [--repeats 20] [--host-samples 64]"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
import scpn_fusion_core_b200 as pkg  # noqa: E402
from bench_shape_sweep import LIMITS, card  # noqa: E402
from scpn_fusion_core_b200 import _device as D  # noqa: E402

GRID = 129
ALPHA = 1e-10
SIGMA = 1e-3
_TF = np.linspace(0.0, 2.0 * np.pi, 33)[:-1] + 0.05
FLUX_POINTS = np.column_stack([6.0 + 3.4 * np.cos(_TF), 4.6 * np.sin(_TF)])
_TB = np.linspace(0.0, 2.0 * np.pi, 65)[:-1] + 0.02
B_POINTS = np.column_stack([6.0 + 3.1 * np.cos(_TB), 4.2 * np.sin(_TB)])
B_DIRS = ["R" if i % 2 == 0 else "Z" for i in range(len(_TB))]
GEOMETRY = dict(flux_points=FLUX_POINTS, b_probe_points=B_POINTS, b_probe_directions=B_DIRS)


def problem(bk, B: int):
    from scpn_fusion_core_b200.free_boundary import build_magnetic_probe_response_matrix
    coils = pkg.CoilSet(positions=[(c["r"], c["z"]) for c in bk.cfg["coils"]],
                        currents=np.array([c["current"] for c in bk.cfg["coils"]]), turns=[1] * len(bk.cfg["coils"]))
    R = build_magnetic_probe_response_matrix(bk, coils, **GEOMETRY)
    truth = bench.uq_inputs(B)[0] * 1.0e6
    prior = bench.uq_inputs(B, seed0=1_000_000)[0] * 1.0e6
    meas = truth @ R.T + np.random.default_rng(5).normal(scale=SIGMA, size=(B, R.shape[0]))
    nf = len(FLUX_POINTS)
    kw = dict(GEOMETRY, flux_measurements=meas[:, :nf], b_probe_measurements=meas[:, nf:],
              measurement_sigma=np.full(R.shape[0], SIGMA), tikhonov_alpha=ALPHA, coil_currents=prior,
              current_limits=LIMITS)
    return R, meas, prior, kw


def run_batch(bk, B: int, repeats: int, torch) -> dict:
    R, meas, prior, kw = problem(bk, B)
    sg = kw["measurement_sigma"]
    meas_d, prior_d = D.to_device(meas, bk.device), D.to_device(prior, bk.device)
    ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def device_call():
        return bk.reconstruct_coil_currents_device(R, meas_d, prior_d, measurement_sigma=sg, tikhonov_alpha=ALPHA,
                                                   current_limits=LIMITS, events=ev)

    bk.reconstruct_coil_currents_from_magnetic_probes(**kw)  # warm-up: module load, allocator, every kernel
    device_call()
    torch.cuda.synchronize()
    dev_s = []
    for _ in range(repeats):
        out = device_call()
        torch.cuda.synchronize()
        dev_s.append(ev[0].elapsed_time(ev[1]) / 1e3)
    e2e_s, res = [], None
    for _ in range(max(repeats // 4, 3)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = bk.reconstruct_coil_currents_from_magnetic_probes(**kw)
        torch.cuda.synchronize()
        e2e_s.append(time.perf_counter() - t0)
    np.testing.assert_array_equal(res["coil_currents"], out["currents"].cpu().numpy())
    t_dev, t_e2e = float(np.median(dev_s)), float(np.median(e2e_s))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        bk.reconstruct_coil_currents_from_magnetic_probes(**kw)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        us = float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
        if us > 0:
            kern[e.key] = us / 1e3
    ab = res["active_bounds"]
    return {"batch": B, "rows": int(R.shape[0]), "coils": int(R.shape[1]),
            "device_seconds_median": t_dev, "device_seconds": dev_s, "device_fits_per_s": B / t_dev,
            "e2e_seconds_median": t_e2e, "e2e_seconds": e2e_s, "e2e_fits_per_s": B / t_e2e,
            "profiled_kernels_ms": dict(sorted(kern.items(), key=lambda kv: -kv[1])[:12]),
            "active_bounds_histogram": {int(k): int(v) for k, v in zip(*np.unique(ab, return_counts=True))},
            "weighted_residual_rms_median": float(np.median(res["weighted_residual_rms"])),
            "response_rank": res["response_rank"], "response_condition": res["response_condition"]}, res, kw


def host_path(kw, batched: dict, samples: int, torch) -> dict:
    kern = pkg.FusionKernel(bench.base_config(GRID))
    coils = kern.build_coilset_from_config()
    coils.current_limits = LIMITS
    nf = len(FLUX_POINTS)
    t_total, rel = 0.0, 0.0
    for k in range(samples + 1):  # sample 0 twice: the first call loads the library and warms the allocator
        j = max(k - 1, 0)
        coils.currents = kw["coil_currents"][j].copy()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = kern.reconstruct_coil_currents_from_magnetic_probes(
            coils, flux_points=FLUX_POINTS, flux_measurements=kw["flux_measurements"][j], b_probe_points=B_POINTS,
            b_probe_directions=B_DIRS, b_probe_measurements=kw["b_probe_measurements"][j],
            measurement_sigma=kw["measurement_sigma"], tikhonov_alpha=ALPHA)
        torch.cuda.synchronize()
        if k:
            t_total += time.perf_counter() - t0
            x = batched["coil_currents"][j]
            rel = max(rel, float(np.max(np.abs(x - r["coil_currents"])) / np.max(np.abs(x))))
    return {"samples": samples, "seconds": t_total, "fits_per_s": samples / t_total,
            "max_abs_current_difference_over_max_current_vs_batched": rel}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--batches", default="4096,65536")
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--host-samples", type=int, default=64)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_probe_sweep.py measures the GPU path: no CUDA device visible")
    out = {"card": card(), "workload": __doc__.split("\n\n")[1], "grid": GRID, "alpha": ALPHA, "sigma": SIGMA,
           "limits": LIMITS.tolist(), "flux_points": FLUX_POINTS.tolist(), "b_probe_points": B_POINTS.tolist(),
           "b_probe_directions": B_DIRS, "batched": []}
    bk = pkg.BatchedFusionKernel(bench.base_config(GRID))
    first = None
    for B in [int(v) for v in args.batches.split(",")]:
        row, res, kw = run_batch(bk, B, args.repeats, torch)
        out["batched"].append(row)
        first = first or (res, kw)
        print(json.dumps(row), file=sys.stderr, flush=True)
    h = host_path(first[1], first[0], args.host_samples, torch)
    h["speedup_of_best_batched_e2e_fits_per_s"] = max(b["e2e_fits_per_s"] for b in out["batched"]) / h["fits_per_s"]
    out["host_path"] = h
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

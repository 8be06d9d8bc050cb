"""a18: batched plasma->wall Green's-function contraction wall[b][w] = sum_s M[w][s] * (J[b][s]*dA)
(jax_free_boundary_predictive.py:498) as an FP64 tensor-core GEMM (k_wall_gemm_sk, stream-K DMMA); compared
with cuBLAS DGEMM on the same shape and with cuBLAS 8192^3 (the FP64 tensor peak measured on this box).
Usage: python tools/bench_wall_gemm.py [n B]...   (default: the headline shape and a set of ragged shapes)"""
import json, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from scpn_fusion_core_b200 import _device as D, _lib

args = [int(v) for v in sys.argv[1:]]
shapes = list(zip(args[0::2], args[1::2])) or [(129, 4096), (129, 512), (129, 130), (129, 3), (65, 4096), (33, 300),
                                                (257, 1024), (17, 64), (40, 77)]

def timeit(fn, reps=5):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps

a = torch.randn((8192, 8192), dtype=torch.float64, device="cuda"); b = torch.randn((8192, 8192), dtype=torch.float64, device="cuda")
ms_big = timeit(lambda: torch.matmul(a, b), 3)
peak = 2 * 8192 ** 3 / ms_big / 1e9
del a, b
out = {"cublas_dgemm_8192_tflops": peak, "shapes": []}
for n, B in shapes:
    nzz = n if n != 40 else 52  # one non-square grid
    R = np.linspace(2.0, 10.0, n); Z = np.linspace(-4.0, 4.0, nzz)
    ctx = D.get_context(nzz, n, R, Z, float(R[1] - R[0]), float(Z[1] - Z[0]), B, 0)
    nw, ni = 2 * n + 2 * (nzz - 2), (nzz - 2) * (n - 2)
    M = D.empty((nw, ni), 0)
    st = D.stream_ptr()
    _lib.check(ctx.lib.gsb_wall_matrix(ctx.handle, 4e-7 * np.pi, D.ptr(M), st))
    J = torch.randn((B, nzz, n), dtype=torch.float64, device="cuda")
    wall = D.empty((B, nw), 0)
    dA = float((R[1] - R[0]) * (Z[1] - Z[0]))
    run = lambda: _lib.check(ctx.lib.gsb_wall_flux(ctx.handle, D.ptr(M), D.ptr(J), dA, D.ptr(wall), B, st))
    flops = 2.0 * B * nw * ni
    ms = timeit(run)
    X = (J[:, 1:-1, 1:-1].reshape(B, ni) * dA).contiguous()
    ref = X @ M.T
    err = float((wall - ref).abs().max() / ref.abs().max())
    run(); torch.cuda.synchronize(); w2 = wall.clone(); run(); torch.cuda.synchronize()
    ms_cublas = timeit(lambda: torch.matmul(X, M.T))
    rec = {"grid": [nzz, n], "batch": B, "shape_BxNwxK": [B, nw, ni], "ms": ms, "tflops": flops / ms / 1e9,
           "cublas_same_shape_ms": ms_cublas, "cublas_same_shape_tflops": flops / ms_cublas / 1e9,
           "vs_cublas_same_shape": ms_cublas / ms, "frac_of_dgemm_peak": flops / ms / 1e9 / peak,
           "rel_err_vs_cublas": err, "deterministic": bool(torch.equal(w2, wall))}
    out["shapes"].append(rec)
    print(json.dumps(rec), flush=True)
    assert err < 1e-12, err
    del M, J, wall, X, ref
print(json.dumps(out))

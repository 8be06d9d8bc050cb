// gsb_internal.cuh - shared internals of libgsb200 (not part of the ABI).
//
// Conventions
//   * fields are float64, C-order [b][iz][ir]; `n` = nz*nr is the per-equilibrium stride
//   * element-wise arithmetic follows the reference's NumPy operand order and is kept
//     free of FMA contraction (dmul/dadd/dsub wrappers) so that results are bit-identical
//     to NumPy wherever NumPy's own result is defined by IEEE +,-,*,/ alone
//   * divisions by per-level / per-column constants use the Markstein sequence
//     q = a*y; r = fma(-b,q,a); q' = fma(r,y,q) with y = RN(1/b) at 3 FP64 issue slots instead of ~25.
//     What is proven: r is exact, and before its final rounding q' equals a/b + (a/b - q)*d with
//     d = b*y - 1, |d| <= 2^-53 and |a/b - q| < 1.5 ulp, i.e. the exact quotient perturbed by less than
//     1.7e-16 ulp; so q' == RN(a/b) unless a/b lies that close to a rounding boundary.  A quotient of two
//     binary64 numbers can come as close as 2^-54 ulp to a midpoint, so for a given divisor a handful of
//     the 2^52 possible significands of `a` may round the other way (1 ulp): about 2^-51 per division,
//     never seen in 2e8 random operand pairs nor in any parity test, and 7 orders of magnitude inside the
//     1e-9 tolerance.  Exact for power-of-two divisors (d = 0).
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/gsb200.h"

namespace gsb {

// ---------------------------------------------------------------- errors / launch count
void set_error(const std::string &msg);
extern std::atomic<long long> g_launches;
constexpr int kMaxDevices = 64;

#define GSB_CUDA(call)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (call);                                                                \
    if (_e != cudaSuccess) {                                                                \
      gsb::set_error(std::string(#call) + ": " + cudaGetErrorString(_e));                   \
      return GSB_ECUDA;                                                                     \
    }                                                                                       \
  } while (0)

#define GSB_LAUNCH_CHECK()                                                                  \
  do {                                                                                      \
    gsb::g_launches.fetch_add(1, std::memory_order_relaxed);                                \
    cudaError_t _e = cudaGetLastError();                                                    \
    if (_e != cudaSuccess) {                                                                \
      gsb::set_error(std::string("kernel launch: ") + cudaGetErrorString(_e));              \
      return GSB_ECUDA;                                                                     \
    }                                                                                       \
  } while (0)

#define GSB_REQUIRE(cond, msg)                                                              \
  do {                                                                                      \
    if (!(cond)) {                                                                          \
      gsb::set_error(msg);                                                                  \
      return GSB_EINVAL;                                                                    \
    }                                                                                       \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) attribute: opt a kernel in
// once per device, not once per process (one process may drive several GPUs, and from several threads).
#define GSB_SMEM_OPT_IN(kernel, bytes)                                                      \
  do {                                                                                      \
    static std::atomic<bool> _done[gsb::kMaxDevices];                                       \
    int _dev = 0;                                                                           \
    GSB_CUDA(cudaGetDevice(&_dev));                                                         \
    if (_dev < 0 || _dev >= gsb::kMaxDevices || !_done[_dev].load(std::memory_order_acquire)) { \
      GSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
      if (_dev >= 0 && _dev < gsb::kMaxDevices) _done[_dev].store(true, std::memory_order_release); \
    }                                                                                       \
  } while (0)

// ---------------------------------------------------------------- exact FP64 helpers
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
// a / b with y = RN(1/b) precomputed: q = a*y; r = fma(-b,q,a); q' = fma(r,y,q).  Equals the IEEE
// quotient except for the ~2^-51 fraction of dividends whose exact quotient sits within 1.7e-16 ulp of
// a rounding boundary (see the header of this file); finite operands, no overflow / subnormal quotient.
// A non-finite q (inf/NaN input or overflow) is returned as is, which is the IEEE result as well
// (+-inf keeps its sign, NaN stays NaN) - branch free.
__device__ __forceinline__ double ddiv_y(double a, double b, double y) {
  const double q = __dmul_rn(a, y);
  const double r = __fma_rn(-b, q, a);
  const double q2 = __fma_rn(r, y, q);
  return (fabs(q) < INFINITY) ? q2 : q;
}

constexpr double kCap = 1.0e250;  // fusion_kernel_numerics.py:16
__device__ __forceinline__ double sanitize(double v) {
  if (isnan(v)) return 0.0;
  if (isinf(v)) return v > 0 ? kCap : -kCap;
  return fmin(fmax(v, -kCap), kCap);
}
__device__ __forceinline__ double clip_cap(double v) {
  // np.clip propagates NaN
  if (isnan(v)) return v;
  return fmin(fmax(v, -kCap), kCap);
}

// ---------------------------------------------------------------- level geometry
// One multigrid level, passed by value to kernels.  Column tables live in device memory.
struct LevelGeom {
  int nz, nr;
  double dr, dz;
  double dr2, dz2, two_dr;              // residual denominators (multigrid_solve.py:243-245)
  double inv_dr2, inv_dz2, inv_two_dr;  // their correctly rounded reciprocals
  double a_ns, a_c, inv_a_c;            // multigrid_solve.py:188-189
  const double *a_e;                    // [nr] 1/dr2 - 1/(2 R dr)   (interior columns)
  const double *a_w;                    // [nr] 1/dr2 + 1/(2 R dr)
  const double *r_safe;                 // [nr] max(R, 1e-10)
  const double *inv_r_safe;             // [nr]
};

struct HostLevel {
  int nz = 0, nr = 0;
  double dr = 0, dz = 0;
  std::vector<double> r_row, a_e, a_w, r_safe, inv_r_safe;
  double a_ns = 0, a_c = 0;
};

// multigrid_solve.py:289-312 level recursion; r_row per level by the reference's
// full-weighting of r_grid (interior rows).
std::vector<HostLevel> plan_levels(int nz, int nr, const double *r_row, double dr, double dz,
                                   int min_grid);

// ---------------------------------------------------------------- stencil point functions
// RB-SOR / Gauss-Seidel update, NumPy operand order (multigrid_solve.py:196-205)
__device__ __forceinline__ double sor_point(const LevelGeom &g, double ae, double aw, double E,
                                            double W, double S, double N, double src, double old,
                                            double omega, double omw) {
  double acc = dadd(dmul(ae, E), dmul(aw, W));
  acc = dadd(acc, dmul(g.a_ns, S));
  acc = dadd(acc, dmul(g.a_ns, N));
  acc = dsub(acc, src);
  const double gs = ddiv_y(acc, g.a_c, g.inv_a_c);
  return dadd(dmul(omw, old), dmul(omega, gs));
}

// L psi = (E - 2C + W)/dr2 - ((E - W)/(2dr))/R + (N - 2C + S)/dz2   (multigrid_solve.py:243-247)
__device__ __forceinline__ double gs_apply_v(const LevelGeom &g, double rs, double inv_rs, double C, double E,
                                             double W, double S, double N) {
  const double twoC = dmul(2.0, C);
  const double d2r = ddiv_y(dadd(dsub(E, twoC), W), g.dr2, g.inv_dr2);
  const double d1r = ddiv_y(dsub(E, W), g.two_dr, g.inv_two_dr);
  const double d2z = ddiv_y(dadd(dsub(N, twoC), S), g.dz2, g.inv_dz2);
  return dadd(dsub(d2r, ddiv_y(d1r, rs, inv_rs)), d2z);
}
__device__ __forceinline__ double gs_apply(const LevelGeom &g, int ir, double C, double E, double W,
                                           double S, double N) {
  return gs_apply_v(g, g.r_safe[ir], g.inv_r_safe[ir], C, E, W, S, N);
}

// 9-point full weighting (multigrid_solve.py:76-91), reference operand order
__device__ __forceinline__ double fw9(double c, double s, double n, double w, double e, double sw,
                                      double se, double nw, double ne) {
  const double t2 = dmul(2.0, dadd(dadd(dadd(s, n), w), e));
  const double t1 = dadd(dadd(dadd(sw, se), nw), ne);
  return dmul(dadd(dadd(dmul(4.0, c), t2), t1), 0.0625);  // /16 is exact scaling
}

// ---------------------------------------------------------------- block reductions
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Deterministic block-wide sum (fixed tree); result valid in thread 0.  `sh` >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double *sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    v = lane < nw ? sh[lane] : 0.0;
    v = warp_sum(v);
  }
  return v;
}
__device__ __forceinline__ double block_max(double v, double *sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    v = lane < nw ? sh[lane] : -INFINITY;
    v = warp_max(v);
  }
  return v;
}
// (value, index) extremum with first-occurrence tie-break (np.argmax / np.argmin order).
struct ValIdx {
  double v;
  int i;
};
template <bool MAX>
__device__ __forceinline__ ValIdx better(ValIdx a, ValIdx b) {
  if (b.i < 0) return a;
  if (a.i < 0) return b;
  bool take_b = MAX ? (b.v > a.v) : (b.v < a.v);
  if (b.v == a.v) take_b = b.i < a.i;
  return take_b ? b : a;
}
template <bool MAX>
__device__ __forceinline__ ValIdx warp_arg(ValIdx x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ValIdx y;
    y.v = __shfl_xor_sync(0xffffffffu, x.v, o);
    y.i = __shfl_xor_sync(0xffffffffu, x.i, o);
    x = better<MAX>(x, y);
  }
  return x;
}
template <bool MAX>
__device__ __forceinline__ ValIdx block_arg(ValIdx x, double *shv, int *shi) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
  x = warp_arg<MAX>(x);
  __syncthreads();
  if (lane == 0) {
    shv[w] = x.v;
    shi[w] = x.i;
  }
  __syncthreads();
  if (w == 0) {
    if (lane < nw) {
      x.v = shv[lane];
      x.i = shi[lane];
    } else {
      x.v = 0.0;
      x.i = -1;
    }
    x = warp_arg<MAX>(x);
  }
  return x;
}

// glibc 2.39 hypot (sysdeps/ieee754/dbl-64/e_hypot.c, non-FMA kernel) restated with
// IEEE +,-,*,/,sqrt only, so np.hypot is reproduced bit-for-bit (checked on 2e6 pairs).
__device__ __forceinline__ double hypot_kernel(double ax, double ay) {
  double h = __dsqrt_rn(dadd(dmul(ax, ax), dmul(ay, ay)));
  double t1, t2;
  if (h <= dmul(2.0, ay)) {
    double delta = dsub(h, ay);
    t1 = dmul(ax, dsub(dmul(2.0, delta), ax));
    t2 = dmul(dsub(delta, dmul(2.0, dsub(ax, ay))), delta);
  } else {
    double delta = dsub(h, ax);
    t1 = dmul(dmul(2.0, delta), dsub(ax, dmul(2.0, ay)));
    t2 = dadd(dmul(dsub(dmul(4.0, delta), ay), ay), dmul(delta, delta));
  }
  return dsub(h, __ddiv_rn(dadd(t1, t2), dmul(2.0, h)));
}
static __device__ __noinline__ double hypot_glibc_slow(double x, double y) {
  if (isinf(x) || isinf(y)) return INFINITY;
  if (isnan(x) || isnan(y)) return dadd(x, y);
  x = fabs(x);
  y = fabs(y);
  double ax = x < y ? y : x;
  double ay = x < y ? x : y;
  if (ax > 0x1p+511) {  // LARGE_VAL: scale both inputs down
    if (ay <= dmul(ax, 0x1p-54)) return dadd(ax, ay);
    return dmul(hypot_kernel(dmul(ax, 0x1p-600), dmul(ay, 0x1p-600)), 0x1p+600);
  }
  if (ay < 0x1p-459) {  // TINY_VAL: scale both inputs up
    if (ax >= dmul(ay, 0x1p+54)) return dadd(ax, ay);
    return dmul(hypot_kernel(dmul(ax, 0x1p+600), dmul(ay, 0x1p+600)), 0x1p-600);
  }
  if (ax >= dmul(ay, 0x1p+54)) return dadd(ax, ay);
  return hypot_kernel(ax, ay);
}
__device__ __forceinline__ double hypot_glibc(double x, double y) {
  const double fx = fabs(x), fy = fabs(y);
  const double ax = fx < fy ? fy : fx;
  const double ay = fx < fy ? fx : fy;
  // common case (no scaling, no shortcut, nothing non-finite: NaN fails every comparison)
  if (ax <= 0x1p+511 && ay >= 0x1p-459 && ax < dmul(ay, 0x1p+54)) return hypot_kernel(ax, ay);
  return hypot_glibc_slow(x, y);
}
__device__ __forceinline__ double sanitize_fast(double v) {
  return (fabs(v) <= kCap) ? v : sanitize(v);  // identity for in-range finite values (the common case)
}

}  // namespace gsb

// ---------------------------------------------------------------- context
struct gsb_level_dev {
  gsb::LevelGeom g;
  double *tables = nullptr;  // one allocation: a_e | a_w | r_safe | inv_r_safe
  double *d = nullptr;       // coarse right-hand side  [batch_cap][n]   (levels >= 1)
  double *e = nullptr;       // coarse correction       [batch_cap][n]   (levels >= 1)
  double *alt = nullptr;     // ping-pong partner of the level's solution for out-of-place fused sweeps (lazy)
};

struct gsb_picard_ws;  // defined in gsb_picard.cu

struct gsb_ctx {
  int device = 0;
  int nz = 0, nr = 0;
  size_t n = 0;
  int batch_cap = 0;
  double dr = 0, dz = 0;
  std::vector<double> r_row, z_axis;
  int planned_min_grid = -1;
  int res_l0 = -1;          // first level of the shared-memory-resident V-cycle tail (n_levels = none)
  double *split_src = nullptr;  // [batch_cap][2*nz*hw] level-0 rhs in colour-split layout
  double *x_alt = nullptr;      // [batch_cap][n] level-0 ping-pong partner for out-of-place fused sweeps (lazy)
  int num_sms = 148;
  std::vector<gsb_level_dev> levels;
  double *z_dev = nullptr;  // [nz]
  double *r_dev = nullptr;  // [nr]
  // scratch for reductions / mg_solve
  double *red = nullptr;    // [batch_cap][red_stride] reduction partials
  int red_stride = 0;       // doubles per equilibrium: >= kRedStride, larger for small batch_cap (big grids)
  int *active = nullptr;    // [batch_cap]
  int *counter = nullptr;   // device counter
  int *h_counter = nullptr; // pinned host mirror
  double *mg_bc = nullptr;  // wall ring copy for mg_solve [batch_cap][ring]
  gsb_picard_ws *picard = nullptr;
  int picard_last_iters = 0;
  cudaStream_t gstream = nullptr;  // private capture-capable stream of the streaming Picard loop
  cudaEvent_t gevent = nullptr;
  // optional per-kernel-class timing of gsb_free_boundary_solve (gsb_timing): CUDA events on the launching stream
  bool timing = false;
  double timing_acc[4] = {0, 0, 0, 0};  // inner Picard solves: ms, count; wall GEMMs: ms, count
  // lane-C wall indices
  int n_wall = 0, n_int = 0;
  double *gemm_ws = nullptr;  // stream-K partial tiles of the wall GEMM (grow-only)
  size_t gemm_ws_bytes = 0;
  // free-boundary outer loop workspace, sized for batch_cap on first use (no allocation in steady state)
  double *fb_old = nullptr, *fb_part = nullptr, *fb_wall = nullptr;
  int *fb_ints = nullptr;
  // shape-optimising outer loop (gsb_free_boundary_shape_solve): factor, stencil, weights (grow-only)
  double *fb_shape = nullptr;
  size_t fb_shape_bytes = 0;
};

namespace gsb {
constexpr int kRedStride = 64;  // doubles of reduction scratch per equilibrium
int ensure_plan(gsb_ctx *ctx, int min_grid);
__host__ __device__ inline int ring_size(int nz, int nr) { return 2 * nr + 2 * nz; }
// V-cycle on device (gsb_mg.cu); `active` may be NULL.
int vcycle_launch(gsb_ctx *ctx, double *psi, size_t psi_stride, const double *src, int batch,
                  double omega, int pre, int post, const int *active, cudaStream_t st);
int smooth_launch(const LevelGeom &g, double *psi, size_t stride, const double *src, size_t sstride,
                  int batch, double omega, int sweeps, int clip, const int *active, cudaStream_t st);
// temporally blocked sweeps (gsb_sweep.cu): `sweeps` (1..3) full RB-SOR sweeps in one pass over HBM
int sweep_fused_launch(const LevelGeom &g, const double *in, size_t istride, double *out, size_t ostride,
                       const double *src, size_t sstride, int batch, double omega, int sweeps, int par_off,
                       int num_sms, const int *active, cudaStream_t st);
void sweep_fused_plan(int nz, int nr, int batch, int nst, int num_sms, int *strip_cols, int *band_rows,
                      int *n_strips, int *n_bands);
// n_sweeps sweeps of level `g` starting from `cur` (in place when one tile per equilibrium covers the
// grid, otherwise ping-pong with `alt`); *result receives the buffer that holds the outcome.
int smooth_fused(gsb_ctx *ctx, const LevelGeom &g, double *cur, double *alt, size_t stride, const double *src,
                 size_t sstride, int batch, double omega, int n_sweeps, const int *active, cudaStream_t st,
                 double **result);
// fused residual + full weighting, one residual evaluation per fine point (gsb_mg.cu; odd fine sizes only)
int residual_restrict_tiled_launch(const LevelGeom &g, const double *psi, size_t pstride, const double *src,
                                   size_t sstride, double *dc, size_t dstride, int nzc, int nrc, int roff, int ci0,
                                   int ci1, int zero_rest, int split_out, int batch, const int *active,
                                   cudaStream_t st);
constexpr int kJacobiFused = 5;  // Jacobi steps per pass of the temporally blocked kernel (gsb_sweep.cu)
int jacobi_fused_launch(const LevelGeom &g, const double *in, double *out, const double *src, int batch, int num_sms,
                        const int *active, cudaStream_t st);
int jacobi_steps_launch(gsb_ctx *ctx, double *psi, double *tmp, const double *src, int n_steps, int batch,
                        const int *active, cudaStream_t st);
int jacobi_launch(const LevelGeom &g, const double *psi, const double *src, double *out, int batch,
                  const int *active, cudaStream_t st);
int ring_apply_launch(double *f, size_t stride, const double *ring, int nz, int nr, int batch, const int *active,
                      cudaStream_t st);
int ring_save_launch(const double *f, size_t stride, double *ring, int nz, int nr, int batch,
                     cudaStream_t st);
int residual_norms_launch(gsb_ctx *ctx, const LevelGeom &g, const double *psi, size_t pstride,
                          const double *src, size_t sstride, double *linf, double *rms, int batch,
                          const int *active, cudaStream_t st);
// The seam between the batched free-boundary loop (gsb_picard.cu) and its shape step (gsb_fit.cu), kept out of the
// library's exports.  free_boundary_loop runs the shape step `sh` after every inner solve unless sh is NULL.
#pragma GCC visibility push(hidden)
struct ShapeStep;
int free_boundary_check(gsb_ctx *ctx, const gsb_free_boundary_params *fb, int batch);
int free_boundary_loop(gsb_ctx *ctx, const gsb_picard_params *p, const gsb_free_boundary_params *fb, const ShapeStep *sh,
                       double *psi_dev, double *psi_ext_dev, const double *wall_m_dev, const double *ip_dev,
                       const double *prof_dev, double *jphi_dev, double *summary_dev, double *fb_summary_dev, int batch,
                       void *stream);
int shape_step_launch(gsb_ctx *ctx, const ShapeStep &sh, const double *psi, double *psi_ext, const int *mask, int batch,
                      cudaStream_t st);
#pragma GCC visibility pop
}  // namespace gsb

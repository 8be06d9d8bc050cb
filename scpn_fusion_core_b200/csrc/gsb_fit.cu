// gsb_fit.cu - bounded least-squares current fits: the shape step of the batched free-boundary loop and the
// magnetic-probe current reconstruction.  Each factors its fit matrix once per call (k_shape_factor) and then fits
// one sample per warp (fit_warp: bounded-variable least squares).
#include "gsb_internal.cuh"

#include <algorithm>

namespace gsb {

// ---------------------------------------------------------------------------- shape step of the outer loop
// (optimize_shape=True, fusion_kernel_free_boundary.py:664-701).  The fit matrix A = [M^T; sqrt(alpha) I] is the same
// for the whole batch, so it is factored once per call (A = Q R, k_shape_factor) and every equilibrium then solves
// the n x n bounded problem min |R x - Q1^T t| (Q1 = the first P rows of Q), whose minimiser is that of
// |M^T x - t|^2 + alpha |x|^2.
constexpr int kShapeMaxCoils = 32;
constexpr int kShapeMaxPoints = 1024;
constexpr int kShapeWarps = 4;  // equilibria per k_shape_fit CTA

// Householder QR of A ((P+n) x n, column-major in `a`; overwritten by the reflectors) in one CTA.  Writes
// R [n][n] (row-major), Q1 [P][n] and *deficient = 1 when |R_ii| <= n eps max|R_jj| for some i.
__global__ void __launch_bounds__(1024)
k_shape_factor(const double *__restrict__ mmat, int n, int P, double sqrt_alpha, double *__restrict__ a,
               double *__restrict__ q, double *__restrict__ rmat, double *__restrict__ q1, int *__restrict__ deficient) {
  __shared__ double sh[32];
  __shared__ double diag[kShapeMaxCoils], beta[kShapeMaxCoils];
  const int m = P + n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  for (int idx = tid; idx < m * n; idx += blockDim.x) {
    const int j = idx / m, i = idx - j * m;
    a[idx] = i < P ? mmat[(size_t)j * P + i] : (i - P == j ? sqrt_alpha : 0.0);
    q[idx] = i == j ? 1.0 : 0.0;  // [I_n; 0]
  }
  __syncthreads();
  for (int k = 0; k < n; ++k) {
    double *col = a + (size_t)k * m;
    double s = 0.0;
    for (int i = k + tid; i < m; i += blockDim.x) s += col[i] * col[i];
    s = block_sum(s, sh);
    if (tid == 0) {
      const double sigma = sqrt(s), x0 = col[k];
      const double al = x0 >= 0.0 ? -sigma : sigma;
      diag[k] = al;
      beta[k] = sigma > 0.0 ? 1.0 / (sigma * (sigma + fabs(x0))) : 0.0;
      col[k] = x0 - al;  // the reflector v (rows k..m-1) stays in the column
    }
    __syncthreads();
    for (int j = k + 1 + warp; j < n; j += nwarps) {
      double *cj = a + (size_t)j * m;
      double d = 0.0;
      for (int i = k + lane; i < m; i += 32) d += col[i] * cj[i];
      const double f = beta[k] * warp_sum(d);
      for (int i = k + lane; i < m; i += 32) cj[i] -= f * col[i];
    }
    __syncthreads();
  }
  // Q [I_n; 0] = H_0 ... H_{n-1} [I_n; 0], applied right to left
  for (int k = n - 1; k >= 0; --k) {
    const double *col = a + (size_t)k * m;
    for (int j = warp; j < n; j += nwarps) {
      double *cj = q + (size_t)j * m;
      double d = 0.0;
      for (int i = k + lane; i < m; i += 32) d += col[i] * cj[i];
      const double f = beta[k] * warp_sum(d);
      for (int i = k + lane; i < m; i += 32) cj[i] -= f * col[i];
    }
    __syncthreads();
  }
  for (int idx = tid; idx < P * n; idx += blockDim.x) {
    const int p = idx / n, j = idx - p * n;
    q1[idx] = q[(size_t)j * m + p];
  }
  for (int idx = tid; idx < n * n; idx += blockDim.x) {
    const int i = idx / n, j = idx - i * n;
    rmat[idx] = i == j ? diag[i] : (i < j ? a[(size_t)j * m + i] : 0.0);
  }
  if (tid == 0) {
    double mx = 0.0;
    bool bad = false;
    for (int i = 0; i < n; ++i) {
      bad = bad || !isfinite(diag[i]);
      mx = fmax(mx, fabs(diag[i]));
    }
    for (int i = 0; i < n; ++i) bad = bad || !(fabs(diag[i]) > (double)n * 2.220446049250313e-16 * mx);
    *deficient = bad ? 1 : 0;
  }
}

// NumPy's pairwise summation (np.add.reduce of a contiguous float64 buffer) for n <= 128 * 2^D, in its order
__device__ __forceinline__ double np_pairwise_leaf(const double *a, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r = dadd(r, a[i]);
    return r;
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = dadd(r[j], a[i + j]);
  double res = dadd(dadd(dadd(r[0], r[1]), dadd(r[2], r[3])), dadd(dadd(r[4], r[5]), dadd(r[6], r[7])));
  for (; i < n; ++i) res = dadd(res, a[i]);
  return res;
}
// (each split leaves at most n/2 + 8 elements, so D = 4 covers kShapeMaxPoints = 1024: 1024 -> 520 -> 268 -> 142 -> 79)
template <int D>
__device__ __forceinline__ double np_pairwise_dev(const double *a, int n) {
  if constexpr (D == 0) {
    return np_pairwise_leaf(a, n);
  } else {
    if (n <= 128) return np_pairwise_leaf(a, n);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return dadd(np_pairwise_dev<D - 1>(a, n2), np_pairwise_dev<D - 1>(a + n2, n - n2));
  }
}

__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Shape target of every active equilibrium into out[b][0:P]: the explicit values, or (isoflux) np.mean of the
// bilinear samples interp_psi (:562-581) of the new Psi, every sample in the reference's operand order:
// ((1-tr)(1-tz)) p00 + (tr(1-tz)) p01 + ((1-tr)tz) p10 + (tr tz) p11, weights and corner index from the host.
__global__ void __launch_bounds__(256)
k_shape_target(const double *__restrict__ psi, size_t n, int nr, const double *__restrict__ wts,
               const int *__restrict__ corner, int P, const double *__restrict__ explicit_t, double *__restrict__ out,
               const int *__restrict__ mask) {
  __shared__ double smp[kShapeMaxPoints];
  __shared__ double mean;
  const int b = blockIdx.x;
  if (!mask[b]) return;
  double *o = out + (size_t)b * (2 * P + 4);
  if (explicit_t) {
    for (int p = threadIdx.x; p < P; p += blockDim.x) o[p] = explicit_t[(size_t)b * P + p];
    return;
  }
  const double *f = psi + (size_t)b * n;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    const double *c = f + corner[p];
    const double *w = wts + 4 * p;
    smp[p] = dadd(dadd(dadd(dmul(w[0], c[0]), dmul(w[1], c[1])), dmul(w[2], c[nr])), dmul(w[3], c[nr + 1]));
  }
  __syncthreads();
  if (threadIdx.x == 0) mean = __ddiv_rn(np_pairwise_dev<4>(smp, P), (double)P);
  __syncthreads();
  for (int p = threadIdx.x; p < P; p += blockDim.x) o[p] = mean;
}

struct ShapeFitArgs {
  const double *rmat;   // [n][n]
  const double *q1;     // [P][n]
  const double *mmat;   // [n][P]
  const double *lim;    // [n] or NULL
  const double *turns;  // [n]
  const int *mask;
  double *currents;     // [B][n] in: prior, out: fit
  double *w;            // [B][n] out: currents * turns
  double *out;          // [B][2P+4]
  int n, P, batch, max_iter;
};

// min |R_F z - d| over the free columns F (lanes with free=1) of the warp's R, d = c - R_B x_B.  Householder QR of the
// n x |F| matrix with lane = row, then back substitution.  Returns z of this lane's coil (free lanes only).
__device__ double shape_free_solve(const double *rs, double *ws, double *zs, int n, bool free_j, double c,
                                   double x) {
  const int lane = threadIdx.x & 31;
  const unsigned fm = __ballot_sync(0xffffffffu, free_j);
  const int f = __popc(fm);
  double d = c;
  int q = 0;
  for (int jj = 0; jj < n; ++jj) {
    const double xj = __shfl_sync(0xffffffffu, x, jj);
    const double rij = lane < n ? rs[lane * n + jj] : 0.0;
    if ((fm >> jj) & 1u) {
      ws[q * 32 + lane] = rij;
      ++q;
    } else {
      d -= rij * xj;
    }
  }
  __syncwarp();
  const bool row = lane < n;
  for (int k = 0; k < f; ++k) {
    const double wk = (row && lane >= k) ? ws[k * 32 + lane] : 0.0;
    const double sigma = sqrt(warp_sum(wk * wk));
    const double x0 = __shfl_sync(0xffffffffu, wk, k);
    const double al = x0 >= 0.0 ? -sigma : sigma;
    const double v = lane == k ? x0 - al : wk;
    const double beta = sigma > 0.0 ? 1.0 / (sigma * (sigma + fabs(x0))) : 0.0;
    for (int jj = k + 1; jj < f; ++jj) {
      const double wj = (row && lane >= k) ? ws[jj * 32 + lane] : 0.0;
      const double dd = warp_sum(v * wj);
      if (row && lane >= k) ws[jj * 32 + lane] = wj - beta * dd * v;
    }
    const double dd = warp_sum(v * ((row && lane >= k) ? d : 0.0));
    if (row && lane >= k) d -= beta * dd * v;
    if (lane == k) ws[k * 32 + k] = al;
    __syncwarp();
  }
  for (int k = f - 1; k >= 0; --k) {
    const double zk = __shfl_sync(0xffffffffu, d, k) / ws[k * 32 + k];
    if (lane < k) d -= ws[k * 32 + lane] * zk;
    if (lane == 0) zs[k] = zk;
  }
  __syncwarp();
  const double z = free_j ? zs[__popc(fm & ((1u << lane) - 1u))] : 0.0;
  __syncwarp();
  return z;
}

// Bounded-variable least squares (Stark & Parker 1995, the algorithm of lsq_linear(method="bvls")) on the n x n
// problem min |R x - c| within [lo, hi], one warp, lane = coil (lanes >= n: coil = false).  rs = R [n][n] row-major;
// ws [32*32] and zs [32] are the warp's scratch.  Writes this lane's x and returns false when more than max_iter
// free-set solves would be needed (x is then unusable).  Called by whole warps only.
__device__ __forceinline__ bool bvls_warp(const double *rs, double *ws, double *zs, int n, bool coil, double lo,
                                          double hi, double c, int max_iter, double &x_out) {
  const int lane = threadIdx.x & 31;
  double cmax = coil ? fabs(c) : 0.0, rmax = 0.0;
  for (int i = 0; i < n; ++i) rmax = fmax(rmax, coil ? fabs(rs[i * n + lane]) : 0.0);
  cmax = warp_max(cmax);
  rmax = warp_max(rmax);
  bool fallback = false;
  int bnd = 0;  // -1 at lo, +1 at hi, 0 free
  double x = 0.0;
  int iters = 0;
  // start (as scipy's bvls): solve on the free set, put violators on their bounds, repeat until feasible
  while (true) {
    const bool fr = coil && bnd == 0;
    if (!__any_sync(0xffffffffu, fr)) break;
    const double z = shape_free_solve(rs, ws, zs, n, fr, c, x);
    ++iters;
    const bool below = fr && z < lo, above = fr && z > hi;
    if (below) x = lo, bnd = -1;
    if (above) x = hi, bnd = 1;
    if (fr && !below && !above) x = z;
    if (!__any_sync(0xffffffffu, below || above)) break;
  }
  bool excluded = false;  // just freed and pushed straight back out: not a candidate until the next free step
  while (!fallback) {
    // g = R^T (R x - c); lane = row for r, lane = column for g
    double r = -c;
    for (int j = 0; j < n; ++j) {
      const double xj = __shfl_sync(0xffffffffu, x, j);
      if (coil) r += rs[lane * n + j] * xj;
    }
    double gj = 0.0;
    for (int i = 0; i < n; ++i) {
      const double ri = __shfl_sync(0xffffffffu, r, i);
      if (coil) gj += rs[i * n + lane] * ri;
    }
    const double xmax = warp_max(coil ? fabs(x) : 0.0);
    const double thresh = 64.0 * n * 2.220446049250313e-16 * rmax * (rmax * xmax + cmax);
    const double cand = (coil && bnd != 0 && !excluded) ? gj * (double)bnd : -INFINITY;
    double best = warp_max(cand);
    if (!(best > thresh)) break;  // KKT: no bound variable wants to move inwards
    const int t = __ffs(__ballot_sync(0xffffffffu, cand == best)) - 1;
    const int bnd_t = __shfl_sync(0xffffffffu, bnd, t);
    if (lane == t) bnd = 0;
    bool first = true;
    while (true) {
      if (++iters > max_iter) {
        fallback = true;
        break;
      }
      const bool fr = coil && bnd == 0;
      const double z = shape_free_solve(rs, ws, zs, n, fr, c, x);
      const bool below = fr && z < lo, above = fr && z > hi;
      double step = (below || above) ? ((below ? lo : hi) - x) / (z - x) : INFINITY;
      const double smin = warp_min_d(step);
      if (smin == INFINITY) {
        if (fr) x = z;
        excluded = false;
        break;
      }
      const int i = __ffs(__ballot_sync(0xffffffffu, step == smin)) - 1;
      const int side_i = __shfl_sync(0xffffffffu, below ? -1 : 1, i);
      // The freed variable leaves at once through the bound it came from: its inward gradient was rounding, so put
      // it back and try the next candidate.  Leaving through the OPPOSITE bound is an ordinary step (it moves there).
      if (first && i == t && side_i == bnd_t) {
        if (lane == t) bnd = bnd_t, excluded = true;
        break;
      }
      first = false;
      if (fr) x = fmin(fmax(x + smin * (z - x), lo), hi);
      if (lane == i) x = below ? lo : hi, bnd = below ? -1 : 1;
    }
  }
  x_out = x;
  return !fallback;
}

// min |R x - c| within [-lim, lim] for one warp, lane = coil: bvls_warp unless c is not finite, clip(prior, -lim, lim)
// when that fails (returns true).  x is 0 on lanes >= n; zs[0:32] receives the warp's x.  Called by whole warps only.
__device__ __forceinline__ bool fit_warp(const double *rs, double *ws, double *zs, int n, double lim, double prior,
                                         double c, bool finite, int max_iter, double &x) {
  const int lane = threadIdx.x & 31;
  const bool coil = lane < n;
  const double lo = -lim, hi = lim;
  x = 0.0;
  const bool failed = !finite || !bvls_warp(rs, ws, zs, n, coil, lo, hi, c, max_iter, x);
  if (failed) x = fmin(fmax(prior, lo), hi);
  if (!coil) x = 0.0;
  zs[lane] = x;
  __syncwarp();
  return failed;
}

// One warp per active equilibrium, lane = coil: c = Q1^T t, then fit_warp on min |R x - c| within +-limits; then the
// fit diagnostics and the coil weights x * turns.  A non-finite target or more than max_iter free-set solves keeps
// clip(prior, -lim, lim).
__global__ void __launch_bounds__(32 * kShapeWarps) k_shape_fit(ShapeFitArgs g) {
  __shared__ double rs[kShapeMaxCoils * kShapeMaxCoils];
  __shared__ double ws_all[kShapeWarps][32 * 32];
  __shared__ double zs_all[kShapeWarps][32];
  const int n = g.n, P = g.P;
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) rs[i] = g.rmat[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kShapeWarps + warp;
  if (b >= g.batch || !g.mask[b]) return;
  double *ws = ws_all[warp], *zs = zs_all[warp];
  double *o = g.out + (size_t)b * (2 * P + 4);
  const bool coil = lane < n;
  const double lim = (coil && g.lim) ? g.lim[lane] : INFINITY;
  const double prior = coil ? g.currents[(size_t)b * n + lane] : 0.0;
  double c = 0.0;
  bool finite = true;
  for (int p = 0; p < P; ++p) {
    const double t = o[p];
    finite = finite && isfinite(t);
    if (coil) c += g.q1[(size_t)p * n + lane] * t;
  }
  double x;
  const bool fallback = fit_warp(rs, ws, zs, n, lim, prior, c, finite, g.max_iter, x);
  if (coil) {
    g.currents[(size_t)b * n + lane] = x;
    g.w[(size_t)b * n + lane] = dmul(x, g.turns[lane]);
  }
  double ss = 0.0, mx = 0.0;
  for (int p = lane; p < P; p += 32) {
    double a = 0.0;
    for (int j = 0; j < n; ++j) a += g.mmat[(size_t)j * P + p] * zs[j];
    o[P + p] = a;
    const double r = a - o[p];
    ss += r * r;
    const double ar = fabs(r);
    mx = (ar > mx || ar != ar) && mx == mx ? ar : mx;  // NaN sticks, as in np.max
  }
  ss = warp_sum(ss);
  for (int off = 16; off > 0; off >>= 1) {
    const double y = __shfl_xor_sync(0xffffffffu, mx, off);
    mx = (y > mx || y != y) && mx == mx ? y : mx;
  }
  const int active = __popc(__ballot_sync(0xffffffffu, coil && g.lim && fabs(fabs(x) - lim) <= 1e-8));
  if (lane == 0) {
    o[2 * P] = sqrt(ss / (double)P);
    o[2 * P + 1] = mx;
    o[2 * P + 2] = (double)active;
    o[2 * P + 3] = fallback ? 1.0 : 0.0;
  }
}

// w[b][c] = currents[b][c] * turns[c] for the whole batch (I * turns, fusion_kernel_free_boundary.py:88-92)
__global__ void k_shape_weights(const double *__restrict__ cur, const double *__restrict__ turns, int n, int total,
                                double *__restrict__ w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) w[i] = dmul(cur[i], turns[i % n]);
}

// ---------------------------------------------------------------------------- magnetic-probe current reconstruction
// (reconstruct_coil_currents_from_magnetic_probes, fusion_kernel_free_boundary.py:370-488).  A = [diag(w) R_p;
// sqrt(alpha) I] is geometry only, so k_shape_factor factors it once per call (its M^T is diag(w) R_p) and every sample
// solves min |R x - c| with c = Q1^T (w o meas) + Q2^T (sqrt(alpha) prior), whose minimiser is that of
// |A x - [w o meas; sqrt(alpha) prior]|.
struct ProbeFitArgs {
  const double *rmat;    // [n][n]
  const double *q1;      // [m][n]
  const double *q;       // Q of k_shape_factor, column-major [(m+n)][n]: rows m..m+n-1 are Q2
  const double *resp_t;  // [n][m] unweighted response, transposed
  const double *w;       // [m] 1/sigma
  const double *lim;     // [n] or NULL
  const double *meas;    // [B][m]
  const double *prior;   // [B][n]
  double *currents;      // [B][n]
  double *residual;      // [B][m] R_p x - meas
  double *wresidual;     // [B][m] residual * w
  double *stats;         // [B][4] residual_rms, weighted_residual_rms, active bounds, failed
  double sqrt_alpha;
  int n, m, batch, max_iter;
};

// One warp per sample, lane = coil.  A non-finite right-hand side or more than max_iter free-set solves sets the
// failure flag and leaves clip(prior, -lim, lim) as the currents.
__global__ void __launch_bounds__(32 * kShapeWarps) k_probe_fit(ProbeFitArgs g) {
  __shared__ double rs[kShapeMaxCoils * kShapeMaxCoils];
  __shared__ double ws_all[kShapeWarps][32 * 32];
  __shared__ double zs_all[kShapeWarps][32];
  const int n = g.n, m = g.m;
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) rs[i] = g.rmat[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kShapeWarps + warp;
  if (b >= g.batch) return;
  double *ws = ws_all[warp], *zs = zs_all[warp];
  const double *mb = g.meas + (size_t)b * m;
  const bool coil = lane < n;
  const double lim = (coil && g.lim) ? g.lim[lane] : INFINITY;
  const double prior = coil ? g.prior[(size_t)b * n + lane] : 0.0;
  // c = Q1^T (w o meas) + Q2^T (sqrt(alpha) prior), rows in order; the measurement rows arrive 32 at a time
  double c = 0.0;
  for (int i0 = 0; i0 < m; i0 += 32) {
    const double v = i0 + lane < m ? dmul(mb[i0 + lane], g.w[i0 + lane]) : 0.0;
    const int cnt = min(32, m - i0);
    for (int r = 0; r < cnt; ++r) {
      const double t = __shfl_sync(0xffffffffu, v, r);
      if (coil) c += g.q1[(size_t)(i0 + r) * n + lane] * t;
    }
  }
  if (g.sqrt_alpha > 0.0) {  // alpha = 0: the reference drops the prior rows
    const double v = dmul(g.sqrt_alpha, prior);
    const double *q2 = g.q + (size_t)lane * (m + n) + m;
    for (int k = 0; k < n; ++k) {
      const double t = __shfl_sync(0xffffffffu, v, k);
      if (coil) c += q2[k] * t;
    }
  }
  const bool finite = __all_sync(0xffffffffu, !coil || isfinite(c));
  double x;
  const bool failed = fit_warp(rs, ws, zs, n, lim, prior, c, finite, g.max_iter, x);
  if (coil) g.currents[(size_t)b * n + lane] = x;
  double ss = 0.0, wss = 0.0;
  for (int i = lane; i < m; i += 32) {
    double a = 0.0;
    for (int j = 0; j < n; ++j) a += g.resp_t[(size_t)j * m + i] * zs[j];
    const double r = a - mb[i], wr = dmul(r, g.w[i]);
    g.residual[(size_t)b * m + i] = r;
    g.wresidual[(size_t)b * m + i] = wr;
    ss += r * r;
    wss += wr * wr;
  }
  ss = warp_sum(ss);
  wss = warp_sum(wss);
  // np.isclose(x, -lim) | np.isclose(x, lim): |x - b| <= 1e-8 + 1e-5 |b|, never true for an infinite bound
  const double tol = 1e-8 + 1e-5 * lim;
  const int active =
      __popc(__ballot_sync(0xffffffffu, coil && g.lim && (fabs(x + lim) <= tol || fabs(x - lim) <= tol)));
  if (lane == 0) {
    double *s = g.stats + (size_t)b * 4;
    s[0] = sqrt(ss / (double)m);
    s[1] = sqrt(wss / (double)m);
    s[2] = (double)active;
    s[3] = failed ? 1.0 : 0.0;
  }
}

// The shape step of gsb_free_boundary_shape_solve (device workspace laid out by that entry)
struct ShapeStep {
  ShapeFitArgs fit;
  const double *wts;      // [P][4] bilinear weights
  const int *corner;      // [P] flat index of the lower-left corner
  const double *target;   // NULL (isoflux) or [B][P]
  const double *green;    // [n][nz][nr] si==1 tables
};

// Target from the new Psi, current fit, coil flux of the new currents (fusion_kernel_free_boundary.py:664-701)
int shape_step_launch(gsb_ctx *ctx, const ShapeStep &sh, const double *psi, double *psi_ext, const int *mask,
                      int batch, cudaStream_t st) {
  k_shape_target<<<batch, 256, 0, st>>>(psi, ctx->n, ctx->nr, sh.wts, sh.corner, sh.fit.P, sh.target, sh.fit.out, mask);
  GSB_LAUNCH_CHECK();
  ShapeFitArgs a = sh.fit;
  a.mask = mask;
  k_shape_fit<<<(batch + kShapeWarps - 1) / kShapeWarps, 32 * kShapeWarps, 0, st>>>(a);
  GSB_LAUNCH_CHECK();
  // whole batch: retired equilibria keep their currents and recompute the same bits
  return gsb_coil_flux(ctx, sh.green, a.w, a.n, 1, psi_ext, batch, st);
}

// Device workspace of k_shape_factor for an (m + n) x n fit matrix: A, Q [(m+n)][n] column-major | R [n][n] |
// Q1 [m][n] | the rank flag in one double
struct FitFactor {
  double *a, *q, *r, *q1;
  int *flag;
  static size_t doubles(size_t m, size_t n) { return 2 * (m + n) * n + n * n + m * n + 1; }
  FitFactor(double *base, size_t m, size_t n)
      : a(base), q(a + (m + n) * n), r(q + (m + n) * n), q1(r + n * n), flag((int *)(q1 + m * n)) {}
};

// Factors [M^T; sqrt(alpha) I] (mmat = M [n][m]) into f and waits for the rank flag (read into h_flag): GSB_EINVAL
// with `msg` when the factor is rank deficient
static int fit_factor(const FitFactor &f, const double *mmat, int n, int m, double sqrt_alpha, int *h_flag,
                      const char *msg, cudaStream_t st) {
  k_shape_factor<<<1, 1024, 0, st>>>(mmat, n, m, sqrt_alpha, f.a, f.q, f.r, f.q1, f.flag);
  GSB_LAUNCH_CHECK();
  GSB_CUDA(cudaMemcpyAsync(h_flag, f.flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  GSB_CUDA(cudaStreamSynchronize(st));
  GSB_REQUIRE(*h_flag == 0, msg);
  return GSB_OK;
}

// tikhonov_alpha and current_limits ([n] or NULL), checked as both fits' references check them
static int check_alpha_limits(double alpha, const double *limits, int n) {
  GSB_REQUIRE(std::isfinite(alpha) && alpha >= 0.0, "tikhonov_alpha must be finite and non-negative.");
  if (limits)
    for (int j = 0; j < n; ++j)
      GSB_REQUIRE(std::isfinite(limits[j]) && limits[j] > 0.0,
                  "current_limits must contain finite positive values only.");
  return GSB_OK;
}

}  // namespace gsb

using namespace gsb;

extern "C" {

int gsb_free_boundary_shape_solve(gsb_ctx *ctx, const gsb_picard_params *p, const gsb_free_boundary_params *fb,
                                  const gsb_shape_params *sp, const double *green_dev, const int *turns_host,
                                  double *currents_dev, const double *target_dev, double *shape_out_dev,
                                  double *psi_dev, double *psi_ext_dev, const double *wall_m_dev,
                                  const double *ip_dev, const double *prof_dev, double *jphi_dev, double *summary_dev,
                                  double *fb_summary_dev, int batch, void *stream) {
  // every argument is checked here, before the first launch
  GSB_REQUIRE(ctx && p && fb && sp && green_dev && turns_host && currents_dev && shape_out_dev && psi_dev &&
                  psi_ext_dev && ip_dev && jphi_dev && summary_dev && fb_summary_dev,
              "gsb_free_boundary_shape_solve: NULL argument");
  int rc = free_boundary_check(ctx, fb, batch);
  if (rc) return rc;
  const int nc = sp->n_coils, P = sp->n_points;
  GSB_REQUIRE(nc >= 1 && nc <= kShapeMaxCoils, "optimize_shape supports 1 to 32 coils on the device.");
  GSB_REQUIRE(P >= 1 && P <= kShapeMaxPoints, "optimize_shape supports 1 to 1024 target points on the device.");
  GSB_REQUIRE(sp->coil_rz && sp->points, "gsb_free_boundary_shape_solve: NULL coil or point coordinates");
  GSB_REQUIRE(sp->isoflux || target_dev, "gsb_free_boundary_shape_solve: explicit targets need target_dev");
  rc = check_alpha_limits(sp->alpha, sp->limits, nc);
  if (rc) return rc;
  GSB_REQUIRE((int)ctx->z_axis.size() == ctx->nz, "gsb_free_boundary_shape_solve: context was created without a z axis");
  for (int c = 0; c < nc; ++c) {
    GSB_REQUIRE(std::isfinite(sp->coil_rz[2 * c]) && std::isfinite(sp->coil_rz[2 * c + 1]) && sp->coil_rz[2 * c] > 0.0,
                "source coil coordinates must be finite with R_src > 0.");
    GSB_REQUIRE(turns_host[c] >= 1, "turns must be positive integers.");
  }
  for (int q = 0; q < P; ++q)
    GSB_REQUIRE(std::isfinite(sp->points[2 * q]) && std::isfinite(sp->points[2 * q + 1]) && sp->points[2 * q] > 0.0,
                "target_flux_points must be finite with positive radii.");
  GSB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  // bilinear stencil of interp_psi (:562-581) on the host: searchsorted (side='left'), clamps, weights in its order
  const int nz = ctx->nz, nr = ctx->nr;
  std::vector<double> host(4 * (size_t)P + 2 * (size_t)nc);
  double *h_w = host.data(), *h_lim = h_w + 4 * (size_t)P, *h_turns = h_lim + nc;
  std::vector<int> corner(P);
  for (int q = 0; q < P; ++q) {
    const double R = sp->points[2 * q], Z = sp->points[2 * q + 1];
    int ir = (int)(std::lower_bound(ctx->r_row.begin(), ctx->r_row.end(), R) - ctx->r_row.begin()) - 1;
    int iz = (int)(std::lower_bound(ctx->z_axis.begin(), ctx->z_axis.end(), Z) - ctx->z_axis.begin()) - 1;
    ir = std::min(std::max(ir, 0), nr - 2);
    iz = std::min(std::max(iz, 0), nz - 2);
    volatile double tr = std::min(std::max((R - ctx->r_row[ir]) / ctx->dr, 0.0), 1.0);
    volatile double tz = std::min(std::max((Z - ctx->z_axis[iz]) / ctx->dz, 0.0), 1.0);
    volatile double ur = 1.0 - tr, uz = 1.0 - tz;
    h_w[4 * q] = ur * uz;
    h_w[4 * q + 1] = tr * uz;
    h_w[4 * q + 2] = ur * tz;
    h_w[4 * q + 3] = tr * tz;
    corner[q] = iz * nr + ir;
  }
  for (int c = 0; c < nc; ++c) {
    h_lim[c] = sp->limits ? sp->limits[c] : 0.0;
    h_turns[c] = (double)turns_host[c];
  }
  // device workspace (grow-only): M [nc][P] | factor | host block | w [cap][nc] | corner [P] ints
  const size_t factor_n = FitFactor::doubles(P, nc);
  const size_t nd = (size_t)nc * P + factor_n + host.size() + (size_t)ctx->batch_cap * nc;
  const size_t bytes = nd * sizeof(double) + (size_t)P * sizeof(int);
  if (ctx->fb_shape_bytes < bytes) {
    if (ctx->fb_shape) cudaFree(ctx->fb_shape);
    ctx->fb_shape = nullptr;
    ctx->fb_shape_bytes = 0;
    GSB_CUDA(cudaMalloc(&ctx->fb_shape, bytes));
    ctx->fb_shape_bytes = bytes;
  }
  double *d_m = ctx->fb_shape, *d_host = d_m + (size_t)nc * P + factor_n, *d_w = d_host + host.size();
  const FitFactor f(d_m + (size_t)nc * P, P, nc);
  int *d_corner = (int *)(ctx->fb_shape + nd);
  GSB_CUDA(cudaMemcpyAsync(d_host, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  GSB_CUDA(cudaMemcpyAsync(d_corner, corner.data(), P * sizeof(int), cudaMemcpyHostToDevice, st));
  rc = gsb_mutual_matrix(sp->coil_rz, turns_host, nc, sp->points, P, d_m, stream);
  if (rc) return rc;
  rc = fit_factor(f, d_m, nc, P, std::sqrt(sp->alpha), ctx->h_counter,
                  "the shape fit [M^T; sqrt(tikhonov_alpha) I] is rank deficient: use tikhonov_alpha > 0 or more "
                  "independent target points", st);
  if (rc) return rc;
  // starting coil flux
  const int total = batch * nc;
  k_shape_weights<<<(total + 255) / 256, 256, 0, st>>>(currents_dev, d_host + 4 * (size_t)P + nc, nc, total, d_w);
  GSB_LAUNCH_CHECK();
  rc = gsb_coil_flux(ctx, green_dev, d_w, nc, 1, psi_ext_dev, batch, stream);
  if (rc) return rc;
  ShapeStep sh{};
  sh.fit.rmat = f.r;
  sh.fit.q1 = f.q1;
  sh.fit.mmat = d_m;
  sh.fit.lim = sp->limits ? d_host + 4 * (size_t)P : nullptr;
  sh.fit.turns = d_host + 4 * (size_t)P + nc;
  sh.fit.currents = currents_dev;
  sh.fit.w = d_w;
  sh.fit.out = shape_out_dev;
  sh.fit.n = nc;
  sh.fit.P = P;
  sh.fit.batch = batch;
  sh.fit.max_iter = 3 * nc + 10;
  sh.wts = d_host;
  sh.corner = d_corner;
  sh.target = sp->isoflux ? nullptr : target_dev;
  sh.green = green_dev;
  return free_boundary_loop(ctx, p, fb, &sh, psi_dev, psi_ext_dev, wall_m_dev, ip_dev, prof_dev, jphi_dev,
                            summary_dev, fb_summary_dev, batch, stream);
}

int gsb_probe_reconstruct(const gsb_probe_params *pp, const double *meas_dev, const double *prior_dev,
                          double *currents_dev, double *residual_dev, double *wresidual_dev, double *stats_dev,
                          void *work_dev, long long *work_bytes, int batch, void *stream) {
  // every argument is checked here, before the first launch
  GSB_REQUIRE(pp && work_bytes, "gsb_probe_reconstruct: NULL argument");
  const int n = pp->n_coils, m = pp->n_rows;
  GSB_REQUIRE(n >= 1 && n <= kShapeMaxCoils, "probe reconstruction supports 1 to 32 coils on the device.");
  GSB_REQUIRE(m >= 1 && m <= kShapeMaxPoints, "probe reconstruction supports 1 to 1024 measurements on the device.");
  // workspace: host block {diag(w) R_p transposed [n][m] | R_p transposed [n][m] | w [m] | limits [n]} | factor
  const size_t mn = (size_t)m * n, host_n = 2 * mn + m + n;
  const size_t need = (host_n + FitFactor::doubles(m, n)) * sizeof(double);
  if (!work_dev) {
    *work_bytes = (long long)need;
    return GSB_OK;
  }
  GSB_REQUIRE(*work_bytes >= (long long)need, "gsb_probe_reconstruct: workspace too small");
  GSB_REQUIRE(meas_dev && prior_dev && currents_dev && residual_dev && wresidual_dev && stats_dev && pp->response,
              "gsb_probe_reconstruct: NULL argument");
  GSB_REQUIRE(batch >= 1, "gsb_probe_reconstruct: batch must be >= 1");
  GSB_REQUIRE(pp->max_iter >= 0, "gsb_probe_reconstruct: max_iter must be >= 0");
  int rc = check_alpha_limits(pp->alpha, pp->limits, n);
  if (rc) return rc;
  for (size_t k = 0; k < mn; ++k)
    GSB_REQUIRE(std::isfinite(pp->response[k]), "Magnetic probe response matrix contains non-finite entries.");
  if (pp->sigma)
    for (int i = 0; i < m; ++i)
      GSB_REQUIRE(std::isfinite(pp->sigma[i]) && pp->sigma[i] > 0.0,
                  "measurement_sigma must contain finite positive values only.");
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<double> host(host_n);
  double *h_a = host.data(), *h_r = h_a + mn, *h_w = h_r + mn, *h_lim = h_w + m;
  for (int i = 0; i < m; ++i) {
    const double w = pp->sigma ? 1.0 / pp->sigma[i] : 1.0;
    h_w[i] = w;
    for (int j = 0; j < n; ++j) {
      const double r = pp->response[(size_t)i * n + j];
      h_a[(size_t)j * m + i] = r * w;  // resp * w[:, None]
      h_r[(size_t)j * m + i] = r;
    }
  }
  for (int j = 0; j < n; ++j) h_lim[j] = pp->limits ? pp->limits[j] : 0.0;
  double *d_host = (double *)work_dev;
  const FitFactor f(d_host + host_n, m, n);
  GSB_CUDA(cudaMemcpyAsync(d_host, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  const double sqrt_alpha = std::sqrt(pp->alpha);
  int deficient = 0;
  rc = fit_factor(f, d_host, n, m, sqrt_alpha, &deficient,
                  "the probe fit [diag(w) R; sqrt(tikhonov_alpha) I] is rank deficient: use tikhonov_alpha > 0 or more "
                  "independent measurements", st);
  if (rc) return rc;
  ProbeFitArgs a{};
  a.rmat = f.r;
  a.q1 = f.q1;
  a.q = f.q;
  a.resp_t = d_host + mn;
  a.w = d_host + 2 * mn;
  a.lim = pp->limits ? d_host + 2 * mn + m : nullptr;
  a.meas = meas_dev;
  a.prior = prior_dev;
  a.currents = currents_dev;
  a.residual = residual_dev;
  a.wresidual = wresidual_dev;
  a.stats = stats_dev;
  a.sqrt_alpha = sqrt_alpha;
  a.n = n;
  a.m = m;
  a.batch = batch;
  a.max_iter = pp->max_iter > 0 ? pp->max_iter : 3 * n + 10;
  k_probe_fit<<<(batch + kShapeWarps - 1) / kShapeWarps, 32 * kShapeWarps, 0, st>>>(a);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

}  // extern "C"

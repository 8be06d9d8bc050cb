// gsb_mg.cu - streaming multigrid kernels for the toroidal Delta* operator (SURVEY.md 8a: a1-a9).
//
// "Streaming" = every pass reads/writes HBM (through L2); used for every level of grids that do
// not fit one SM's shared memory and as the general path.  One thread per updated point,
// batch in gridDim.z.  Arithmetic keeps NumPy's operand order (bit-identical results).
#include "gsb_internal.cuh"
#include "gsb_resident.cuh"

namespace gsb {

// ------------------------------------------------------------------------------------------
// a1/a2  red-black SOR colour pass  (multigrid_solve.py:193-206)
//   gs = (a_e*E + a_w*W + a_ns*S + a_ns*N - src) / a_c ;  psi = (1-w)*psi + w*gs
// ------------------------------------------------------------------------------------------
template <bool CLIP>
__global__ void __launch_bounds__(256)
k_smooth_colour(LevelGeom g, double *__restrict__ psi, size_t pstride,
                const double *__restrict__ src, size_t sstride, int parity, double omega,
                double omw, const int *__restrict__ active) {
  const int b = blockIdx.z;
  if (active && !active[b]) return;
  const int iz = 1 + blockIdx.y * blockDim.y + threadIdx.y;
  if (iz >= g.nz - 1) return;
  const int j0 = (((iz + 1) & 1) == parity) ? 1 : 2;
  const int ir = j0 + 2 * (blockIdx.x * blockDim.x + threadIdx.x);
  if (ir >= g.nr - 1) return;
  double *p = psi + (size_t)b * pstride + (size_t)iz * g.nr + ir;
  const double s = src[(size_t)b * sstride + (size_t)iz * g.nr + ir];
  double v = sor_point(g, g.a_e[ir], g.a_w[ir], p[1], p[-1], p[-g.nr], p[g.nr], s, p[0], omega, omw);
  if (CLIP) v = clip_cap(v);
  p[0] = v;
}

static dim3 colour_block(const LevelGeom &g) {
  const int half = (g.nr - 2 + 1) / 2;
  int bx = 1;
  while (bx < half && bx < 32) bx <<= 1;
  int by = 256 / bx;
  const int rows = g.nz - 2;
  while (by > 1 && by / 2 >= rows) by >>= 1;
  return dim3(bx, by, 1);
}

int smooth_launch(const LevelGeom &g, double *psi, size_t stride, const double *src, size_t sstride,
                  int batch, double omega, int sweeps, int clip, const int *active,
                  cudaStream_t st) {
  if (g.nz < 3 || g.nr < 3 || sweeps <= 0 || batch <= 0) return GSB_OK;
  const dim3 blk = colour_block(g);
  const int half = (g.nr - 2 + 1) / 2;
  const dim3 grd((half + blk.x - 1) / blk.x, (g.nz - 2 + blk.y - 1) / blk.y, batch);
  const double omw = 1.0 - omega;
  for (int s = 0; s < sweeps; ++s)
    for (int parity = 0; parity < 2; ++parity) {
      if (clip)
        k_smooth_colour<true><<<grd, blk, 0, st>>>(g, psi, stride, src, sstride, parity, omega, omw, active);
      else
        k_smooth_colour<false><<<grd, blk, 0, st>>>(g, psi, stride, src, sstride, parity, omega, omw, active);
      GSB_LAUNCH_CHECK();
    }
  return GSB_OK;
}

// Fused sweeps with the tile plan of gsb_sweep.cu.  Single tile per equilibrium: in place.
// Otherwise out of place, ping-pong between `cur` and `alt`.
int smooth_fused(gsb_ctx *ctx, const LevelGeom &g, double *cur, double *alt, size_t stride, const double *src,
                 size_t sstride, int batch, double omega, int n_sweeps, const int *active, cudaStream_t st,
                 double **result) {
  *result = cur;
  if (g.nz < 3 || g.nr < 3 || n_sweeps <= 0 || batch <= 0) return GSB_OK;
  int remaining = n_sweeps;
  while (remaining > 0) {
    const int s = std::min(remaining, 3);
    int sc, br, ns, nb;
    sweep_fused_plan(g.nz, g.nr, batch, 2 * s, ctx->num_sms, &sc, &br, &ns, &nb);
    const bool inplace = (ns == 1 && nb == 1);
    double *dst = inplace ? *result : (*result == cur ? alt : cur);
    GSB_REQUIRE(dst != nullptr, "smooth_fused: out-of-place sweep needs an alternate buffer");
    int rc = sweep_fused_launch(g, *result, stride, dst, stride, src, sstride, batch, omega, s, 0, ctx->num_sms, active, st);
    if (rc) return rc;
    *result = dst;
    remaining -= s;
  }
  return GSB_OK;
}

// ------------------------------------------------------------------------------------------
// a3  Jacobi step  (fusion_kernel_iterative_solver.py:54-95): sanitised inputs, clipped output
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_jacobi(LevelGeom g, const double *__restrict__ psi, const double *__restrict__ src,
         double *__restrict__ out, const int *__restrict__ active) {
  const int b = blockIdx.z;
  if (active && !active[b]) return;
  const int ir = blockIdx.x * blockDim.x + threadIdx.x;
  const int iz = blockIdx.y * blockDim.y + threadIdx.y;
  if (ir >= g.nr || iz >= g.nz) return;
  const size_t n = (size_t)g.nz * g.nr;
  const double *p = psi + b * n + (size_t)iz * g.nr + ir;
  double v;
  if (iz == 0 || ir == 0 || iz == g.nz - 1 || ir == g.nr - 1) {
    v = sanitize(p[0]);
  } else {
    const double E = sanitize(p[1]), W = sanitize(p[-1]);
    const double S = sanitize(p[-g.nr]), N = sanitize(p[g.nr]);
    const double s = sanitize(src[b * n + (size_t)iz * g.nr + ir]);
    double acc = dadd(dmul(g.a_e[ir], E), dmul(g.a_w[ir], W));
    acc = dadd(acc, dmul(g.a_ns, S));
    acc = dadd(acc, dmul(g.a_ns, N));
    acc = dsub(acc, s);
    v = clip_cap(ddiv_y(acc, g.a_c, g.inv_a_c));
  }
  out[b * n + (size_t)iz * g.nr + ir] = v;
}

__global__ void __launch_bounds__(256)
k_copy_masked(const double *__restrict__ src, double *__restrict__ dst, size_t n, const int *__restrict__ active) {
  const int b = blockIdx.y;
  if (!active[b]) return;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dst[(size_t)b * n + i] = src[(size_t)b * n + i];
}

int jacobi_launch(const LevelGeom &g, const double *psi, const double *src, double *out, int batch,
                  const int *active, cudaStream_t st) {
  const dim3 blk(32, 8, 1);
  const dim3 grd((g.nr + 31) / 32, (g.nz + 7) / 8, batch);
  k_jacobi<<<grd, blk, 0, st>>>(g, psi, src, out, active);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// n_steps Jacobi steps, result in psi_dev; tmp_dev is the ping-pong partner.  Groups of kJacobiFused steps run in
// one pass over HBM (k_jacobi_warp), the rest one step per launch.
int jacobi_steps_launch(gsb_ctx *ctx, double *psi, double *tmp, const double *src, int n_steps, int batch,
                        const int *active, cudaStream_t st) {
  const LevelGeom &g = ctx->levels[0].g;
  const size_t bytes = (size_t)batch * ctx->n * sizeof(double);
  double *cur = psi, *oth = tmp;
  const bool fused_ok = g.nz >= 3 && g.nr >= 3;
  int left = n_steps;
  while (left > 0) {
    int rc;
    if (fused_ok && left >= kJacobiFused) {
      rc = jacobi_fused_launch(g, cur, oth, src, batch, ctx->num_sms, active, st);
      left -= kJacobiFused;
    } else {
      rc = jacobi_launch(g, cur, src, oth, batch, active, st);
      left -= 1;
    }
    if (rc) return rc;
    std::swap(cur, oth);
  }
  if (cur != psi) {
    // inactive equilibria were never written in `tmp`: copy only through a kernel that honours the mask
    if (active) {
      const int blocks = (int)std::min<size_t>((ctx->n + 255) / 256, 64);
      k_copy_masked<<<dim3(blocks, batch), 256, 0, st>>>(cur, psi, ctx->n, active);
      GSB_LAUNCH_CHECK();
    } else {
      GSB_CUDA(cudaMemcpyAsync(psi, cur, bytes, cudaMemcpyDeviceToDevice, st));
    }
  }
  return GSB_OK;
}


// ------------------------------------------------------------------------------------------
// a4  residual / operator  (multigrid_solve.py:236-249)
//   L psi = (E - 2C + W)/dr2 - ((E - W)/(2dr))/R + (N - 2C + S)/dz2
// ------------------------------------------------------------------------------------------
template <bool WITH_SRC>
__global__ void __launch_bounds__(256)
k_residual(LevelGeom g, const double *__restrict__ psi, const double *__restrict__ src,
           double *__restrict__ out) {
  const int b = blockIdx.z;
  const int ir = blockIdx.x * blockDim.x + threadIdx.x;
  const int iz = blockIdx.y * blockDim.y + threadIdx.y;
  if (ir >= g.nr || iz >= g.nz) return;
  const size_t n = (size_t)g.nz * g.nr;
  const size_t o = b * n + (size_t)iz * g.nr + ir;
  double v = 0.0;
  if (iz > 0 && ir > 0 && iz < g.nz - 1 && ir < g.nr - 1) {
    const double *p = psi + o;
    v = gs_apply(g, ir, p[0], p[1], p[-1], p[-g.nr], p[g.nr]);
    if (WITH_SRC) v = dsub(v, src[o]);
  }
  out[o] = v;
}

// a5: per-equilibrium interior max|r| and sum r^2; grid (P, batch); partials -> red[b][2p..]
__global__ void __launch_bounds__(256)
k_residual_norm_partials(LevelGeom g, const double *__restrict__ psi, size_t pstride,
                         const double *__restrict__ src, size_t sstride, double *__restrict__ red,
                         int red_stride, const int *__restrict__ active) {
  __shared__ double sh[32];
  const int b = blockIdx.y, P = gridDim.x, p = blockIdx.x;
  if (active && !active[b]) return;
  const int rows = g.nz - 2, cols = g.nr - 2;
  const int r0 = (int)((long long)rows * p / P), r1 = (int)((long long)rows * (p + 1) / P);
  double mx = 0.0, sq = 0.0;
  const double *base = psi + (size_t)b * pstride;
  const double *sb = src + (size_t)b * sstride;
  // rows of the block's band one at a time, threads across the columns (no integer division per point)
  for (int iz = 1 + r0; iz < 1 + r1; ++iz)
    for (int ir = 1 + threadIdx.x; ir <= cols; ir += blockDim.x) {
      const double *q = base + (size_t)iz * g.nr + ir;
      double r = dsub(gs_apply(g, ir, q[0], q[1], q[-1], q[-g.nr], q[g.nr]), sb[(size_t)iz * g.nr + ir]);
      // NaN must survive the max (np.max propagates NaN)
      const double a = fabs(r);
      mx = (isnan(a) || isnan(mx)) ? NAN : fmax(mx, a);
      sq += r * r;
    }
  const bool anynan = __syncthreads_or(isnan(mx));
  double m = block_max(isnan(mx) ? 0.0 : mx, sh);
  double s = block_sum(sq, sh);
  if (threadIdx.x == 0) {
    red[(size_t)b * red_stride + 2 * p] = anynan ? NAN : m;
    red[(size_t)b * red_stride + 2 * p + 1] = s;
  }
}

__global__ void __launch_bounds__(128)
k_residual_norm_final(const double *__restrict__ red, int red_stride, int P, double n_int,
                      double *__restrict__ linf, double *__restrict__ rms, int batch,
                      const int *__restrict__ active) {
  // one CTA per equilibrium: fixed-tree reduction of the P partial (max, sum) pairs
  __shared__ double sh[32];
  const int b = blockIdx.x;
  if (b >= batch) return;
  if (active && !active[b]) return;
  double m = 0.0, s = 0.0;
  int nan = 0;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    const double v = red[(size_t)b * red_stride + 2 * p];
    if (isnan(v)) nan = 1;
    m = fmax(m, v);
    s += red[(size_t)b * red_stride + 2 * p + 1];
  }
  nan = __syncthreads_or(nan);
  m = block_max(m, sh);
  __syncthreads();
  s = block_sum(s, sh);
  if (threadIdx.x == 0) {
    if (linf) linf[b] = nan ? NAN : m;
    if (rms) rms[b] = (n_int > 0) ? sqrt(s / n_int) : 0.0;
  }
}

static int norm_partials(const LevelGeom &g, int red_stride) {
  const long long pts = (long long)(g.nz - 2) * (g.nr - 2);
  int P = (int)((pts + 4095) / 4096);
  if (P < 1) P = 1;
  if (P > red_stride / 2) P = red_stride / 2;
  if (P > 2048) P = 2048;
  if (P > g.nz - 2) P = g.nz - 2 > 0 ? g.nz - 2 : 1;
  return P;
}

int residual_norms_launch(gsb_ctx *ctx, const LevelGeom &g, const double *psi, size_t pstride,
                          const double *src, size_t sstride, double *linf, double *rms, int batch,
                          const int *active, cudaStream_t st) {
  if (g.nz < 3 || g.nr < 3) {
    if (linf) GSB_CUDA(cudaMemsetAsync(linf, 0, batch * sizeof(double), st));
    if (rms) GSB_CUDA(cudaMemsetAsync(rms, 0, batch * sizeof(double), st));
    return GSB_OK;
  }
  const int P = norm_partials(g, ctx->red_stride);
  k_residual_norm_partials<<<dim3(P, batch), 256, 0, st>>>(g, psi, pstride, src, sstride, ctx->red, ctx->red_stride, active);
  GSB_LAUNCH_CHECK();
  k_residual_norm_final<<<batch, 128, 0, st>>>(
      ctx->red, ctx->red_stride, P, (double)(g.nz - 2) * (double)(g.nr - 2), linf, rms, batch, active);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// ------------------------------------------------------------------------------------------
// a6  full-weighting restriction (multigrid_solve.py:57-99), generic shapes
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_restrict(const double *__restrict__ fine, double *__restrict__ coarse, int nzf, int nrf, int nzc,
           int nrc) {
  const int b = blockIdx.z;
  const int J = blockIdx.x * blockDim.x + threadIdx.x;
  const int I = blockIdx.y * blockDim.y + threadIdx.y;
  if (I >= nzc || J >= nrc) return;
  const double *f = fine + (size_t)b * nzf * nrf;
  double v;
  // wall injection; later assignments win at the corners (rows first, then columns)
  if (J == 0)
    v = f[(size_t)(2 * I) * nrf];
  else if (J == nrc - 1)
    v = f[(size_t)(2 * I) * nrf + (nrf - 1)];
  else if (I == 0)
    v = f[2 * J];
  else if (I == nzc - 1)
    v = f[(size_t)(nzf - 1) * nrf + 2 * J];
  else {
    const double *c = f + (size_t)(2 * I) * nrf + 2 * J;
    v = fw9(c[0], c[-nrf], c[nrf], c[-1], c[1], c[-nrf - 1], c[-nrf + 1], c[nrf - 1], c[nrf + 1]);
  }
  coarse[(size_t)b * nzc * nrc + (size_t)I * nrc + J] = v;
}

// fused: coarse rhs = restrict( -(L psi - src) ), wall = 0   (multigrid_solve.py:303-306)
__global__ void __launch_bounds__(256)
k_residual_restrict(LevelGeom g, const double *__restrict__ psi, size_t pstride,
                    const double *__restrict__ src, size_t sstride, double *__restrict__ dc, int nzc,
                    int nrc, int split_out, const int *__restrict__ active) {
  const int b = blockIdx.z;
  if (active && !active[b]) return;
  const int J = blockIdx.x * blockDim.x + threadIdx.x;
  const int I = blockIdx.y * blockDim.y + threadIdx.y;
  if (I >= nzc || J >= nrc) return;
  double v = 0.0;
  if (I > 0 && J > 0 && I < nzc - 1 && J < nrc - 1) {
    const double *pb = psi + (size_t)b * pstride;
    const double *sb = src + (size_t)b * sstride;
    double d[3][3];
#pragma unroll
    for (int a = -1; a <= 1; ++a)
#pragma unroll
      for (int c = -1; c <= 1; ++c) {
        const int iz = 2 * I + a, ir = 2 * J + c;
        const double *q = pb + (size_t)iz * g.nr + ir;
        const double r = dsub(gs_apply(g, ir, q[0], q[1], q[-1], q[-g.nr], q[g.nr]),
                              sb[(size_t)iz * g.nr + ir]);
        d[a + 1][c + 1] = -r;
      }
    v = fw9(d[1][1], d[0][1], d[2][1], d[1][0], d[1][2], d[0][0], d[0][2], d[2][0], d[2][2]);
  }
  if (split_out) {  // colour-split layout consumed by the resident kernel (gsb_resident.cuh)
    const int hwc = (nrc + 1) / 2;
    dc[(size_t)b * 2 * nzc * hwc + ((((I + J) & 1) * nzc + I) * hwc + (J >> 1))] = v;
  } else {
    dc[((size_t)b * nzc + I) * nrc + J] = v;
  }
}

// Tiled form of the same operator for odd fine widths (2^k+1 grids, every slab level): a CTA owns 8 x 32 coarse
// points, evaluates each of the 17 x 65 fine residuals under them ONCE into shared memory (the per-point kernel
// above evaluates every residual 2.25 times) and then applies the 9-point weights.  `roff` = fine row of coarse
// row 0 (slab arrays carry halo rows); rows [ci0, ci1) of dc are computed, the others are zeroed if zero_rest.
struct RRTiledArgs {
  LevelGeom g;
  const double *psi, *src;
  double *dc;
  size_t pstride, sstride, dstride;
  int nzc, nrc, roff, ci0, ci1, row_base, zero_rest, split_out;
  const int *active;
};
constexpr int kRRTI = 8, kRRTJ = 32, kRRFR = 2 * kRRTI + 1, kRRFC = 2 * kRRTJ + 1;
__global__ void __launch_bounds__(256) k_residual_restrict_tiled(const RRTiledArgs a) {
  __shared__ double sr[kRRFR][kRRFC + 1];
  const int b = blockIdx.z;
  if (a.active && !a.active[b]) return;
  const LevelGeom &g = a.g;
  const int J0 = blockIdx.x * kRRTJ, I0 = a.row_base + blockIdx.y * kRRTI;
  const double *pb = a.psi + (size_t)b * a.pstride;
  const double *sb = a.src + (size_t)b * a.sstride;
  const int i_lo = max(I0, a.ci0), i_hi = min(I0 + kRRTI, a.ci1);  // coarse rows of this tile that are computed
  const int iz_lo = 2 * i_lo + a.roff - 1, iz_hi = 2 * (i_hi - 1) + a.roff + 1;
  for (int idx = threadIdx.x; idx < kRRFR * kRRFC; idx += blockDim.x) {
    const int fr = idx / kRRFC, fc = idx - fr * kRRFC;
    const int iz = 2 * I0 + a.roff - 1 + fr, ir = 2 * J0 - 1 + fc;
    double v = 0.0;
    if (i_lo < i_hi && iz >= iz_lo && iz <= iz_hi && ir >= 1 && ir <= g.nr - 2) {
      const double *q = pb + (size_t)iz * g.nr + ir;
      v = -dsub(gs_apply(g, ir, q[0], q[1], q[-1], q[-g.nr], q[g.nr]), sb[(size_t)iz * g.nr + ir]);
    }
    sr[fr][fc] = v;
  }
  __syncthreads();
  const int tj = threadIdx.x & (kRRTJ - 1), ti = threadIdx.x / kRRTJ;
  const int I = I0 + ti, J = J0 + tj;
  if (I >= a.nzc || J >= a.nrc) return;
  double v = 0.0;
  const bool row_on = I >= a.ci0 && I < a.ci1;
  if (row_on && J > 0 && J < a.nrc - 1) {
    const int r = 2 * ti + 1, c = 2 * tj + 1;
    v = fw9(sr[r][c], sr[r - 1][c], sr[r + 1][c], sr[r][c - 1], sr[r][c + 1], sr[r - 1][c - 1], sr[r - 1][c + 1],
            sr[r + 1][c - 1], sr[r + 1][c + 1]);
  } else if (!row_on && !a.zero_rest) {
    return;
  }
  if (a.split_out) {
    const int hwc = (a.nrc + 1) / 2;
    a.dc[(size_t)b * a.dstride + ((((I + J) & 1) * a.nzc + I) * hwc + (J >> 1))] = v;
  } else {
    a.dc[(size_t)b * a.dstride + (size_t)I * a.nrc + J] = v;
  }
}

int residual_restrict_tiled_launch(const LevelGeom &g, const double *psi, size_t pstride, const double *src,
                                   size_t sstride, double *dc, size_t dstride, int nzc, int nrc, int roff, int ci0,
                                   int ci1, int zero_rest, int split_out, int batch, const int *active,
                                   cudaStream_t st) {
  RRTiledArgs a{g, psi, src, dc, pstride, sstride, dstride, nzc, nrc, roff, ci0, ci1, zero_rest ? 0 : ci0, zero_rest,
                split_out, active};
  const int rows = zero_rest ? nzc : ci1 - ci0;
  if (rows <= 0 || nrc <= 0) return GSB_OK;
  k_residual_restrict_tiled<<<dim3((nrc + kRRTJ - 1) / kRRTJ, (rows + kRRTI - 1) / kRRTI, batch), 256, 0, st>>>(a);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// ------------------------------------------------------------------------------------------
// a7  bilinear prolongation (multigrid_solve.py:102-145) incl. its slicing limits
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool prolong_value(const double *__restrict__ c, int nzc, int nrc,
                                              int nzf, int nrf, int iz, int ir, double &out) {
  const int kz = min(nzc, (nzf + 1) / 2), kr = min(nrc, (nrf + 1) / 2);
  const int hend = min(2 * (nrc - 1), nrf - 1), vend = min(2 * (nzc - 1), nzf - 1);
  const bool ze = (iz & 1) == 0, re = (ir & 1) == 0;
  const bool zok = ze ? (iz / 2 < kz) : (iz < vend);
  const bool rok = re ? (ir / 2 < kr) : (ir < hend);
  if (!(zok && rok)) {
    out = 0.0;
    return false;
  }
  const int I = iz >> 1, J = ir >> 1;
  const double *p = c + (size_t)I * nrc + J;
  if (ze && re)
    out = p[0];
  else if (ze)
    out = dmul(0.5, dadd(p[0], p[1]));
  else if (re)
    out = dmul(0.5, dadd(p[0], p[nrc]));
  else
    out = dmul(0.25, dadd(dadd(dadd(p[0], p[nrc]), p[1]), p[nrc + 1]));
  return true;
}

__global__ void __launch_bounds__(256)
k_prolong(const double *__restrict__ coarse, double *__restrict__ fine, int nzc, int nrc, int nzf,
          int nrf) {
  const int b = blockIdx.z;
  const int ir = blockIdx.x * blockDim.x + threadIdx.x;
  const int iz = blockIdx.y * blockDim.y + threadIdx.y;
  if (iz >= nzf || ir >= nrf) return;
  double v;
  prolong_value(coarse + (size_t)b * nzc * nrc, nzc, nrc, nzf, nrf, iz, ir, v);
  fine[(size_t)b * nzf * nrf + (size_t)iz * nrf + ir] = v;
}

// psi += P e on the interior (the wall correction is exactly zero: coarse walls are zero)
__global__ void __launch_bounds__(256)
k_prolong_add(const double *__restrict__ ec, int nzc, int nrc, double *__restrict__ psi,
              size_t pstride, int nzf, int nrf, const int *__restrict__ active) {
  const int b = blockIdx.z;
  if (active && !active[b]) return;
  const int ir = 1 + blockIdx.x * blockDim.x + threadIdx.x;
  const int iz0 = 1 + 4 * (blockIdx.y * blockDim.y + threadIdx.y);  // four rows per thread: four fine loads in flight
  if (iz0 >= nzf - 1 || ir >= nrf - 1) return;
  double *p = psi + (size_t)b * pstride + (size_t)iz0 * nrf + ir;
  const double *c = ec + (size_t)b * nzc * nrc;
  double old[4], v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) old[k] = (iz0 + k < nzf - 1) ? p[(size_t)k * nrf] : 0.0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    v[k] = 0.0;
    if (iz0 + k < nzf - 1) prolong_value(c, nzc, nrc, nzf, nrf, iz0 + k, ir, v[k]);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (iz0 + k < nzf - 1) p[(size_t)k * nrf] = dadd(old[k], v[k]);
}

// ------------------------------------------------------------------------------------------
// base level: all sweeps of a tiny grid in shared memory, one CTA per equilibrium
// (multigrid_solve.py:292-293: 50 sweeps when min_grid >= nz or nr)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_base_solve(LevelGeom g, double *__restrict__ x, size_t xstride, const double *__restrict__ rhs,
             size_t rstride, int zero_init, double omega, double omw, int sweeps,
             const int *__restrict__ active) {
  extern __shared__ double sm[];
  const int b = blockIdx.x;
  if (active && !active[b]) return;
  const int n = g.nz * g.nr;
  double *sx = sm, *ss = sm + n;
  double *xb = x + (size_t)b * xstride;
  const double *rb = rhs + (size_t)b * rstride;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    sx[i] = zero_init ? 0.0 : xb[i];
    ss[i] = rb[i];
  }
  __syncthreads();
  const int rows = g.nz - 2, half = (g.nr - 2 + 1) / 2;
  for (int s = 0; s < sweeps; ++s)
    for (int parity = 0; parity < 2; ++parity) {
      for (int idx = threadIdx.x; idx < rows * half; idx += blockDim.x) {
        const int iz = 1 + idx / half;
        const int j0 = (((iz + 1) & 1) == parity) ? 1 : 2;
        const int ir = j0 + 2 * (idx % half);
        if (ir < g.nr - 1) {
          double *p = sx + iz * g.nr + ir;
          p[0] = sor_point(g, g.a_e[ir], g.a_w[ir], p[1], p[-1], p[-g.nr], p[g.nr],
                           ss[iz * g.nr + ir], p[0], omega, omw);
        }
      }
      __syncthreads();
    }
  for (int i = threadIdx.x; i < n; i += blockDim.x) xb[i] = sx[i];
}

constexpr int kBaseSmemMax = 96 * 1024;

static int base_solve_launch(const LevelGeom &g, double *x, size_t xstride, const double *rhs,
                             size_t rstride, int zero_init, int batch, double omega, int sweeps,
                             const int *active, cudaStream_t st) {
  if (g.nz < 3 || g.nr < 3) {
    if (zero_init) GSB_CUDA(cudaMemsetAsync(x, 0, (size_t)batch * xstride * sizeof(double), st));
    return GSB_OK;
  }
  const size_t smem = 2 * (size_t)g.nz * g.nr * sizeof(double);
  if (smem > (size_t)kBaseSmemMax) {  // unusual aspect ratios: plain streaming sweeps
    if (zero_init) GSB_CUDA(cudaMemsetAsync(x, 0, (size_t)batch * xstride * sizeof(double), st));
    return smooth_launch(g, x, xstride, rhs, rstride, batch, omega, sweeps, 0, active, st);
  }
  GSB_SMEM_OPT_IN(k_base_solve, kBaseSmemMax);
  k_base_solve<<<batch, 128, smem, st>>>(g, x, xstride, rhs, rstride, zero_init, omega, 1.0 - omega, sweeps, active);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// ------------------------------------------------------------------------------------------
// shared-memory-resident V-cycle tail: one CTA per equilibrium (gsb_resident.cuh)
// ------------------------------------------------------------------------------------------
bool build_rplan(const gsb_ctx *ctx, int l0, int extra_doubles, RPlan *out) {
  const int L = (int)ctx->levels.size();
  if (l0 < 0 || l0 >= L || L - l0 > kResMaxLevels) return false;
  int off = 0;
  out->nlev = L - l0;
  for (int l = l0; l < L; ++l) {
    RLevel &r = out->lev[l - l0];
    const LevelGeom &g = ctx->levels[l].g;
    r.nz = g.nz;
    r.nr = g.nr;
    r.hw = (g.nr + 1) / 2;
    r.nk = g.nr / 2;
    r.g = g;
    const int T = kResThreads;
    const int rows = std::max(r.nz - 2, 0);
    r.lk = 0;
    while ((1 << r.lk) < r.nk) ++r.lk;
    r.nch = std::max(1, std::min(rows, T >> r.lk));
    r.rpc = rows > 0 ? (rows + r.nch - 1) / r.nch : 0;
    if (r.rpc > 1 && (r.rpc & 1)) {  // even chunks keep the row-parity pattern uniform across a warp
      r.rpc += 1;
      r.nch = (rows + r.rpc - 1) / r.rpc;
    }
    if (l == l0 && r.rpc > kResMaxRun) return false;  // the finest level prefetches a whole run's rhs into registers
    const int ncj = std::max(r.nr - 2, 1);
    r.lj = 0;
    while ((1 << r.lj) < ncj) ++r.lj;
    r.cch = std::max(1, std::min(rows, T >> r.lj));
    r.crpc = rows > 0 ? (rows + r.cch - 1) / r.cch : 0;
    const int planes = 2 * r.nz * r.hw;
    r.x_off = off;
    off += planes;
    if (l > l0) {
      r.d_off = off;
      off += planes;
    } else {
      r.d_off = -1;
    }
  }
  for (int l = l0; l < L; ++l) {  // column tables of the coarse levels live in shared memory too
    RLevel &r = out->lev[l - l0];
    r.t_off = -1;
    if (l > l0) {
      r.t_off = off;
      off += 2 * r.nr;
    }
  }
  out->pool_doubles = off;
  return (size_t)(off + res_stage_doubles(out->nlev) + extra_doubles) * sizeof(double) <= (size_t)kResSmemMax;
}

// dense [nz][nr] -> colour-split [2][nz][hw]
__global__ void __launch_bounds__(256)
k_dense_to_split(const double *__restrict__ in, size_t istride, double *__restrict__ out, int nz, int nr,
                 const int *__restrict__ active) {
  const int b = blockIdx.y;
  if (active && !active[b]) return;
  const int hw = (nr + 1) / 2;
  const double *f = in + (size_t)b * istride;
  double *o = out + (size_t)b * 2 * nz * hw;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nz * nr; i += gridDim.x * blockDim.x) {
    const int iz = i / nr, ir = i - iz * nr;
    o[split_index(nz, hw, iz, ir)] = f[i];
  }
}

// x: dense [b][nz][nr] (stride xstride) of the finest resident level; rhs: colour-split global.
__global__ void __launch_bounds__(kResThreads, 1)
k_vcycle_resident(const __grid_constant__ RPlan plan, double *__restrict__ x, size_t xstride, const double *__restrict__ rhs,
                  int zero_init, int batch, double omega, int pre, int post,
                  const int *__restrict__ active) {
  const int lev_off = res_stage(plan);
  const RLevel &F = res_level(lev_off, 0);
  const int planes = 2 * F.nz * F.hw;
  for (int b = blockIdx.x; b < batch; b += gridDim.x) {
    if (active && !active[b]) continue;
    double *xb = x + (size_t)b * xstride;
    if (zero_init)
      res_zero_off(F.x_off, planes);
    else
      res_load_dense(xb, F.x_off, F.nz, F.nr, F.hw);
    __syncthreads();
    res_vcycle(lev_off, plan.nlev, rhs + (size_t)b * planes, omega, pre, post);
    __syncthreads();
    res_store_dense(xb, F.x_off, F.nz, F.nr, F.hw);
    __syncthreads();
  }
}

static int resident_launch(gsb_ctx *ctx, int l0, double *x, size_t xstride, const double *rhs_split,
                           int zero_init, int batch, double omega, int pre, int post, const int *active,
                           cudaStream_t st) {
  RPlan plan;
  if (!build_rplan(ctx, l0, 0, &plan)) {
    set_error("resident_launch: plan does not fit shared memory");
    return GSB_EINVAL;
  }
  GSB_SMEM_OPT_IN(k_vcycle_resident, kResSmemMax);
  const size_t smem = (size_t)(plan.pool_doubles + res_stage_doubles(plan.nlev)) * sizeof(double);
  const int grid = std::min(batch, ctx->num_sms);
  k_vcycle_resident<<<grid, kResThreads, smem, st>>>(plan, x, xstride, rhs_split, zero_init, batch, omega, pre, post, active);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// ------------------------------------------------------------------------------------------
// a8  V-cycle driver (multigrid_solve.py:252-335), recursion unrolled over the planned levels.
// Levels [0, res_l0) stream through HBM; levels [res_l0, L) run inside k_vcycle_resident.
// ------------------------------------------------------------------------------------------
int vcycle_launch(gsb_ctx *ctx, double *psi, size_t psi_stride, const double *src, int batch,
                  double omega, int pre, int post, const int *active, cudaStream_t st) {
  const int L = (int)ctx->levels.size();
  const int l0 = ctx->res_l0;
  const dim3 blk(32, 8, 1);
  auto X = [&](int l) { return l == 0 ? psi : ctx->levels[l].e; };
  auto XS = [&](int l) { return l == 0 ? psi_stride : (size_t)ctx->levels[l].g.nz * ctx->levels[l].g.nr; };
  auto S = [&](int l) { return l == 0 ? src : (const double *)ctx->levels[l].d; };
  auto SS = [&](int l) { return l == 0 ? ctx->n : (size_t)ctx->levels[l].g.nz * ctx->levels[l].g.nr; };
  const int top = std::min(l0, L - 1);  // levels [0, top) are smoothed by streaming kernels
  // ping-pong partners for out-of-place fused sweeps (multi-tile levels), allocated on first use
  auto ALT = [&](int l, double **out) -> int {
    const LevelGeom &g = ctx->levels[l].g;
    int sc, br, ns, nb;
    sweep_fused_plan(g.nz, g.nr, batch, 6, ctx->num_sms, &sc, &br, &ns, &nb);
    *out = nullptr;
    if (ns == 1 && nb == 1) return GSB_OK;
    double **slot = l == 0 ? &ctx->x_alt : &ctx->levels[l].alt;
    if (!*slot) GSB_CUDA(cudaMalloc(slot, (size_t)ctx->batch_cap * XS(l) * sizeof(double)));
    *out = *slot;
    return GSB_OK;
  };
  std::vector<double *> curv(L, nullptr);  // buffer holding each streaming level's solution after pre-smoothing
  for (int l = 0; l < top; ++l) {
    const LevelGeom &g = ctx->levels[l].g;
    const LevelGeom &c = ctx->levels[l + 1].g;
    double *alt = nullptr;
    int rc = ALT(l, &alt);
    if (rc) return rc;
    if (alt && l == 0 && psi_stride != ctx->n) alt = nullptr;  // foreign stride: fall back to per-colour passes
    double *cur = X(l);
    {
      int sc, br, ns, nb;
      sweep_fused_plan(g.nz, g.nr, batch, 6, ctx->num_sms, &sc, &br, &ns, &nb);
      if ((ns == 1 && nb == 1) || alt)
        rc = smooth_fused(ctx, g, X(l), alt, XS(l), S(l), SS(l), batch, omega, pre, active, st, &cur);
      else
        rc = smooth_launch(g, X(l), XS(l), S(l), SS(l), batch, omega, pre, 0, active, st);
    }
    if (rc) return rc;
    curv[l] = cur;
    const dim3 grd((c.nr + 31) / 32, (c.nz + 7) / 8, batch);
    const int split = (l + 1 == l0) ? 1 : 0;
    if ((g.nz & 1) && (g.nr & 1) && c.nz >= 3 && c.nr >= 3 && (long long)g.nz * g.nr >= 4096) {
      // odd sizes (coarse point (I,J) sits on fine (2I,2J)): every fine residual is evaluated once per tile
      const size_t ds = split ? (size_t)2 * c.nz * ((c.nr + 1) / 2) : (size_t)c.nz * c.nr;
      rc = residual_restrict_tiled_launch(g, cur, XS(l), S(l), SS(l), ctx->levels[l + 1].d, ds, c.nz, c.nr, 0, 1, c.nz - 1,
                                          1, split, batch, active, st);
      if (rc) return rc;
    } else {
      k_residual_restrict<<<grd, blk, 0, st>>>(g, cur, XS(l), S(l), SS(l), ctx->levels[l + 1].d, c.nz, c.nr, split, active);
      GSB_LAUNCH_CHECK();
    }
    if (l + 1 < L - 1 && l + 1 != l0)  // resident / base solve zero-initialise on chip
      GSB_CUDA(cudaMemsetAsync(ctx->levels[l + 1].e, 0, (size_t)batch * c.nz * c.nr * sizeof(double), st));
  }
  if (l0 < L) {
    int rc;
    if (l0 == 0) {
      const LevelGeom &g = ctx->levels[0].g;
      const int blocks = std::min((g.nz * g.nr + 255) / 256, 32);
      k_dense_to_split<<<dim3(blocks, batch), 256, 0, st>>>(src, ctx->n, ctx->split_src, g.nz, g.nr, active);
      GSB_LAUNCH_CHECK();
      rc = resident_launch(ctx, 0, psi, psi_stride, ctx->split_src, 0, batch, omega, pre, post, active, st);
    } else {
      rc = resident_launch(ctx, l0, ctx->levels[l0].e, XS(l0), ctx->levels[l0].d, 1, batch, omega, pre, post, active, st);
    }
    if (rc) return rc;
  } else {
    const LevelGeom &g = ctx->levels[L - 1].g;
    int rc = base_solve_launch(g, X(L - 1), XS(L - 1), S(L - 1), SS(L - 1), L > 1 ? 1 : 0, batch, omega, 50, active, st);
    if (rc) return rc;
  }
  for (int l = top - 1; l >= 0; --l) {
    const LevelGeom &g = ctx->levels[l].g;
    const LevelGeom &c = ctx->levels[l + 1].g;
    double *cur = curv[l] ? curv[l] : X(l);
    if (g.nz > 2 && g.nr > 2) {
      const dim3 grd((g.nr - 2 + 31) / 32, (g.nz - 2 + 31) / 32, batch);  // 32 x 8 threads, four rows each
      k_prolong_add<<<grd, blk, 0, st>>>(ctx->levels[l + 1].e, c.nz, c.nr, cur, XS(l), g.nz, g.nr, active);
      GSB_LAUNCH_CHECK();
    }
    int rc;
    double *fin = cur;
    double *partner = (cur == X(l)) ? (l == 0 ? ctx->x_alt : ctx->levels[l].alt) : X(l);
    int sc, br, ns, nb;
    sweep_fused_plan(g.nz, g.nr, batch, 6, ctx->num_sms, &sc, &br, &ns, &nb);
    const bool single = (ns == 1 && nb == 1);
    if (single || (partner && !(l == 0 && psi_stride != ctx->n)))
      rc = smooth_fused(ctx, g, cur, partner, XS(l), S(l), SS(l), batch, omega, post, active, st, &fin);
    else
      rc = smooth_launch(g, cur, XS(l), S(l), SS(l), batch, omega, post, 0, active, st);
    if (rc) return rc;
    if (fin != X(l))  // odd number of out-of-place launches: bring the result home
      GSB_CUDA(cudaMemcpyAsync(X(l), fin, (size_t)batch * XS(l) * sizeof(double), cudaMemcpyDeviceToDevice, st));
  }
  return GSB_OK;
}

// wall ring helpers -----------------------------------------------------------------------
// ring layout: [row 0 (nr)] [row nz-1 (nr)] [col 0 (nz)] [col nr-1 (nz)]
__global__ void k_ring_save(const double *__restrict__ f, size_t stride, double *__restrict__ ring,
                            int nz, int nr) {
  const int b = blockIdx.y, rs = 2 * nr + 2 * nz;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rs) return;
  const double *fb = f + (size_t)b * stride;
  double v;
  if (i < nr) v = fb[i];
  else if (i < 2 * nr) v = fb[(size_t)(nz - 1) * nr + (i - nr)];
  else if (i < 2 * nr + nz) v = fb[(size_t)(i - 2 * nr) * nr];
  else v = fb[(size_t)(i - 2 * nr - nz) * nr + nr - 1];
  ring[(size_t)b * rs + i] = v;
}
__global__ void k_ring_apply(double *__restrict__ f, size_t stride, const double *__restrict__ ring,
                             int nz, int nr, const int *__restrict__ active) {
  const int b = blockIdx.y, rs = 2 * nr + 2 * nz;
  if (active && !active[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rs) return;
  double *fb = f + (size_t)b * stride;
  const double v = ring[(size_t)b * rs + i];
  // same precedence as the reference (rows then columns): skip row entries at the corners
  if (i < nr) { if (i > 0 && i < nr - 1) fb[i] = v; }
  else if (i < 2 * nr) { const int j = i - nr; if (j > 0 && j < nr - 1) fb[(size_t)(nz - 1) * nr + j] = v; }
  else if (i < 2 * nr + nz) fb[(size_t)(i - 2 * nr) * nr] = v;
  else fb[(size_t)(i - 2 * nr - nz) * nr + nr - 1] = v;
}

int ring_apply_launch(double *f, size_t stride, const double *ring, int nz, int nr, int batch, const int *active,
                      cudaStream_t st) {
  const int rs = ring_size(nz, nr);
  k_ring_apply<<<dim3((rs + 255) / 256, batch), 256, 0, st>>>(f, stride, ring, nz, nr, active);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int ring_save_launch(const double *f, size_t stride, double *ring, int nz, int nr, int batch,
                     cudaStream_t st) {
  const int rs = ring_size(nz, nr);
  k_ring_save<<<dim3((rs + 255) / 256, batch), 256, 0, st>>>(f, stride, ring, nz, nr);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

__global__ void k_mg_decide(const double *__restrict__ res, double tol, int cycle, int max_cycles,
                            int *__restrict__ active, int *__restrict__ cycles,
                            int *__restrict__ converged, int *__restrict__ counter, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  if (!active[b]) return;
  const bool conv = res[b] < tol;
  cycles[b] = cycle;
  converged[b] = conv ? 1 : 0;
  if (conv || cycle >= max_cycles) active[b] = 0;
  else atomicAdd(counter, 1);
}

__global__ void k_fill_int(int *p, int v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace gsb

using namespace gsb;

namespace gsb { int picard_phase_read(long long *out64, int reset); }
static bool omega_ok(double w) { return std::isfinite(w) && w >= 1.0 && w < 2.0; }

extern "C" {

// debug: per-phase clock64 totals of CTA 0 of k_vcycle_resident (zeros unless built with
// -DGSB_PHASE_TIMING); reset!=0 clears the counters after reading.
int gsb_debug_phase_cycles(long long *out64, int reset) {
#ifdef GSB_PHASE_TIMING
  if (out64) GSB_CUDA(cudaMemcpyFromSymbol(out64, g_phase, 64 * sizeof(long long)));
  if (reset) {
    long long z[64] = {0};
    GSB_CUDA(cudaMemcpyToSymbol(g_phase, z, sizeof(z)));
  }
#else
  if (out64)
    for (int i = 0; i < 64; ++i) out64[i] = 0;
  (void)reset;
#endif
  return picard_phase_read(out64, reset);  // the Picard translation unit has its own counters
}

int gsb_smooth_ex(gsb_ctx *ctx, double *psi_dev, const double *src_dev, int batch, double omega,
                  int n_sweeps, int clip, int fuse, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && src_dev, "gsb_smooth: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_smooth: batch outside [1, batch_cap]");
  GSB_REQUIRE(omega_ok(omega), "omega must be finite and satisfy 1.0 <= omega < 2.0");
  GSB_REQUIRE(fuse >= 0 && fuse <= 3, "gsb_smooth_ex: fuse must be 0 (one launch per colour pass) or 1..3");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, ctx->planned_min_grid < 0 ? 5 : ctx->planned_min_grid);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const LevelGeom &g = ctx->levels[0].g;
  if (clip || fuse == 0 || g.nz < 3 || g.nr < 3)
    return smooth_launch(g, psi_dev, ctx->n, src_dev, ctx->n, batch, omega, n_sweeps, clip, nullptr, st);
  double *cur = psi_dev;
  int remaining = n_sweeps;
  while (remaining > 0) {
    const int s = std::min(remaining, fuse);
    int sc, br, ns, nb;
    sweep_fused_plan(g.nz, g.nr, batch, 2 * s, ctx->num_sms, &sc, &br, &ns, &nb);
    double *dst = cur;
    if (!(ns == 1 && nb == 1)) {
      if (!ctx->x_alt) GSB_CUDA(cudaMalloc(&ctx->x_alt, (size_t)ctx->batch_cap * ctx->n * sizeof(double)));
      dst = (cur == psi_dev) ? ctx->x_alt : psi_dev;
    }
    rc = sweep_fused_launch(g, cur, ctx->n, dst, ctx->n, src_dev, ctx->n, batch, omega, s, 0, ctx->num_sms, nullptr, st);
    if (rc) return rc;
    cur = dst;
    remaining -= s;
  }
  if (cur != psi_dev)
    GSB_CUDA(cudaMemcpyAsync(psi_dev, cur, (size_t)batch * ctx->n * sizeof(double), cudaMemcpyDeviceToDevice, st));
  return GSB_OK;
}

int gsb_smooth(gsb_ctx *ctx, double *psi_dev, const double *src_dev, int batch, double omega,
               int n_sweeps, int clip, void *stream) {
  return gsb_smooth_ex(ctx, psi_dev, src_dev, batch, omega, n_sweeps, clip, 3, stream);
}

int gsb_jacobi(gsb_ctx *ctx, const double *psi_dev, const double *src_dev, double *out_dev,
               int batch, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && src_dev && out_dev, "gsb_jacobi: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_jacobi: batch outside [1, batch_cap]");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, ctx->planned_min_grid < 0 ? 5 : ctx->planned_min_grid);
  if (rc) return rc;
  return jacobi_launch(ctx->levels[0].g, psi_dev, src_dev, out_dev, batch, nullptr, (cudaStream_t)stream);
}

int gsb_jacobi_steps(gsb_ctx *ctx, double *psi_dev, const double *src_dev, double *tmp_dev, int n_steps, int batch,
                     void *stream) {
  GSB_REQUIRE(ctx && psi_dev && src_dev && tmp_dev, "gsb_jacobi_steps: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_jacobi_steps: batch outside [1, batch_cap]");
  GSB_REQUIRE(n_steps >= 0, "gsb_jacobi_steps: n_steps must be >= 0");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, ctx->planned_min_grid < 0 ? 5 : ctx->planned_min_grid);
  if (rc) return rc;
  return jacobi_steps_launch(ctx, psi_dev, tmp_dev, src_dev, n_steps, batch, nullptr, (cudaStream_t)stream);
}

static int residual_common(gsb_ctx *ctx, const double *psi, const double *src, double *out, int batch,
                           void *stream, bool with_src) {
  GSB_REQUIRE(ctx && psi && out && (src || !with_src), "gsb_residual: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_residual: batch outside [1, batch_cap]");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, ctx->planned_min_grid < 0 ? 5 : ctx->planned_min_grid);
  if (rc) return rc;
  const LevelGeom &g = ctx->levels[0].g;
  const dim3 blk(32, 8, 1), grd((g.nr + 31) / 32, (g.nz + 7) / 8, batch);
  if (with_src)
    k_residual<true><<<grd, blk, 0, (cudaStream_t)stream>>>(g, psi, src, out);
  else
    k_residual<false><<<grd, blk, 0, (cudaStream_t)stream>>>(g, psi, nullptr, out);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_residual(gsb_ctx *ctx, const double *psi_dev, const double *src_dev, double *res_dev,
                 int batch, void *stream) {
  return residual_common(ctx, psi_dev, src_dev, res_dev, batch, stream, true);
}

int gsb_apply_operator(gsb_ctx *ctx, const double *v_dev, double *out_dev, int batch, void *stream) {
  return residual_common(ctx, v_dev, nullptr, out_dev, batch, stream, false);
}

int gsb_residual_norms(gsb_ctx *ctx, const double *psi_dev, const double *src_dev, double *linf_dev,
                       double *rms_dev, int batch, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && src_dev, "gsb_residual_norms: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_residual_norms: batch outside [1, batch_cap]");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, ctx->planned_min_grid < 0 ? 5 : ctx->planned_min_grid);
  if (rc) return rc;
  return residual_norms_launch(ctx, ctx->levels[0].g, psi_dev, ctx->n, src_dev, ctx->n, linf_dev,
                               rms_dev, batch, nullptr, (cudaStream_t)stream);
}

int gsb_restrict_full_weight(const double *fine_dev, double *coarse_dev, int nz_f, int nr_f,
                             int batch, void *stream) {
  GSB_REQUIRE(fine_dev && coarse_dev, "gsb_restrict_full_weight: NULL argument");
  GSB_REQUIRE(nz_f >= 1 && nr_f >= 1 && batch >= 1 && batch <= 65535, "gsb_restrict_full_weight: bad shape");
  const int nzc = (nz_f + 1) / 2, nrc = (nr_f + 1) / 2;
  const dim3 blk(32, 8, 1), grd((nrc + 31) / 32, (nzc + 7) / 8, batch);
  k_restrict<<<grd, blk, 0, (cudaStream_t)stream>>>(fine_dev, coarse_dev, nz_f, nr_f, nzc, nrc);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_prolong_bilinear(const double *coarse_dev, double *fine_dev, int nz_c, int nr_c, int nz_f,
                         int nr_f, int batch, void *stream) {
  GSB_REQUIRE(coarse_dev && fine_dev, "gsb_prolong_bilinear: NULL argument");
  GSB_REQUIRE(nz_c >= 1 && nr_c >= 1 && nz_f >= 1 && nr_f >= 1 && batch >= 1 && batch <= 65535,
              "gsb_prolong_bilinear: bad shape");
  const dim3 blk(32, 8, 1), grd((nr_f + 31) / 32, (nz_f + 7) / 8, batch);
  k_prolong<<<grd, blk, 0, (cudaStream_t)stream>>>(coarse_dev, fine_dev, nz_c, nr_c, nz_f, nr_f);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_vcycle(gsb_ctx *ctx, double *psi_dev, const double *src_dev, int batch, double omega, int pre,
               int post, int min_grid, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && src_dev, "gsb_vcycle: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_vcycle: batch outside [1, batch_cap]");
  GSB_REQUIRE(omega_ok(omega), "omega must be finite and satisfy 1.0 <= omega < 2.0");
  GSB_REQUIRE(pre >= 0 && post >= 0, "gsb_vcycle: negative sweep count");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, min_grid);
  if (rc) return rc;
  return vcycle_launch(ctx, psi_dev, ctx->n, src_dev, batch, omega, pre, post, nullptr, (cudaStream_t)stream);
}

int gsb_mg_solve(gsb_ctx *ctx, const double *src_dev, double *psi_dev, int batch, double tol,
                 int max_cycles, double omega, int pre, int post, int min_grid, double *res_dev,
                 int *cycles_dev, int *converged_dev, void *stream) {
  GSB_REQUIRE(ctx && src_dev && psi_dev && res_dev && cycles_dev && converged_dev, "gsb_mg_solve: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_mg_solve: batch outside [1, batch_cap]");
  GSB_REQUIRE(std::isfinite(tol) && tol > 0.0, "tol must be finite and > 0.");
  GSB_REQUIRE(max_cycles >= 1, "max_cycles must be >= 1.");
  GSB_REQUIRE(omega_ok(omega), "omega must be finite and satisfy 1.0 <= omega < 2.0");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, min_grid);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const LevelGeom &g = ctx->levels[0].g;
  const int rs = ring_size(g.nz, g.nr);
  k_ring_save<<<dim3((rs + 255) / 256, batch), 256, 0, st>>>(psi_dev, ctx->n, ctx->mg_bc, g.nz, g.nr);
  GSB_LAUNCH_CHECK();
  k_fill_int<<<(batch + 255) / 256, 256, 0, st>>>(ctx->active, 1, batch);
  GSB_LAUNCH_CHECK();
  // cycle 0: residual of the initial state (multigrid_solve.py:444-445)
  for (int cycle = 0;; ++cycle) {
    rc = residual_norms_launch(ctx, g, psi_dev, ctx->n, src_dev, ctx->n, res_dev, nullptr, batch, ctx->active, st);
    if (rc) return rc;
    GSB_CUDA(cudaMemsetAsync(ctx->counter, 0, sizeof(int), st));
    k_mg_decide<<<(batch + 127) / 128, 128, 0, st>>>(res_dev, tol, cycle, max_cycles, ctx->active, cycles_dev, converged_dev, ctx->counter, batch);
    GSB_LAUNCH_CHECK();
    GSB_CUDA(cudaMemcpyAsync(ctx->h_counter, ctx->counter, sizeof(int), cudaMemcpyDeviceToHost, st));
    GSB_CUDA(cudaStreamSynchronize(st));
    if (ctx->h_counter[0] == 0) break;
    rc = vcycle_launch(ctx, psi_dev, ctx->n, src_dev, batch, omega, pre, post, ctx->active, st);
    if (rc) return rc;
    k_ring_apply<<<dim3((rs + 255) / 256, batch), 256, 0, st>>>(psi_dev, ctx->n, ctx->mg_bc, g.nz, g.nr, ctx->active);
    GSB_LAUNCH_CHECK();
  }
  return GSB_OK;
}

}  // extern "C"

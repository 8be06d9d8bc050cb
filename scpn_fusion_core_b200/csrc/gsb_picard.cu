// gsb_picard.cu - the batched Picard outer loop (SURVEY.md 8a: a10-a14) on device.
//
// One launch sequence advances EVERY active equilibrium of the batch by one Picard iteration:
//   T   k_topo          argmax psi, min psi, masked first-min of hypot(grad psi)   (a10, a11)
//   TS  k_xpoint_saddle optional 16-candidate Hessian saddle filter               (a11)
//   TF  k_topo_final    psi_axis / psi_boundary scalars (+ limiter fallback)       (:505)
//   S1  k_source_raw    psi_N, profiles, J_raw, deterministic partial sums         (a12)
//   S2  k_source_scale  J = J_raw*Ip/I ; Source = (-mu0*R)*J
//   E   elliptic step   copy + V-cycle | SOR sweep | Jacobi                         (a8/a2/a3)
//   R   k_relax         wall BC, NaN flag, mean|dpsi|, under-relaxation, GS residual (a13, a5)
//   D   k_decide        history, best-state tracking, convergence, buffer rotation  (a13)
// Per-equilibrium state lives in device arrays; the host only polls an active counter.
#include "gsb_internal.cuh"
#include "gsb_resident.cuh"

#include <algorithm>
#include <cstdlib>

constexpr int kPT = 32;  // max partial blocks per equilibrium
constexpr int kTW = 8;   // doubles per topo partial
constexpr int kRW = 4;   // doubles per relax partial
constexpr int kSadChunk = 4096;   // masked points per CTA of the saddle candidate kernel
constexpr int kSadChunksMax = 64; // -> up to 262144 masked points per equilibrium

struct PicardState {  // SoA, device pointers, [batch_cap] each
  int *active, *status, *iter, *cur, *best, *nxt, *xsel, *seed_active;
  double *diff_best, *gs_best, *gs_last, *diff_last, *scale;
  double *axbnd;  // [b][2]
  double *topo;   // [b][8]: iz_ax, ir_ax, psi_ax, iz_x, ir_x, psi_x, found, psi_min
};

struct Bufs {
  double *p[3];
};

struct gsb_picard_ws {
  int cap = 0;
  double *buf1 = nullptr, *buf2 = nullptr, *W = nullptr, *source = nullptr, *ring = nullptr;
  double *tpart = nullptr, *spart = nullptr, *rpart = nullptr;
  double *seedJ = nullptr, *cf = nullptr, *mr = nullptr;
  int *rowmask = nullptr;
  int *mrows = nullptr;        // compact list of the masked (divertor) rows
  int n_mrows = 0;
  int cand_chunks = 0;
  double *cand = nullptr;      // [cap][kSadChunks][16][2] per-chunk smallest |grad psi| candidates (value, flat index)
  int *ints = nullptr;
  double *dbls = nullptr;
  PicardState s{};
  // cached host-side parameters the device tables were built for
  double mu0 = NAN, z_min = NAN, r_min = NAN, r_max = NAN;
  double seed_sum = 0.0;
  // private per-CTA workspace of the persistent resident solve: [grid][5 * 2*nz*hw] (colour-split)
  double *res_ws = nullptr;
  int res_grid = 0;
  // Anderson mixing (method 3), allocated on first use: iterate / residual rings [cap][and_slots][n], Gram partials,
  // coefficients, fallback flags
  double *and_psi = nullptr, *and_res = nullptr, *and_part = nullptr, *and_alpha = nullptr;
  int *and_fb = nullptr;
  int and_slots = 0;
};

namespace gsb {

struct GradGeom {
  double dz, dr, two_dz, two_dr, inv_dz, inv_dr, inv_two_dz, inv_two_dr;
};

// np.gradient semantics (2nd-order centred interior, 1st-order one-sided edges), uniform spacing
__device__ __forceinline__ void grad_point(const double *__restrict__ f, int nz, int nr, int iz,
                                           int ir, const GradGeom &gg, double &gz, double &gr) {
  const double *p = f + (size_t)iz * nr + ir;
  if (iz == 0)
    gz = ddiv_y(dsub(p[nr], p[0]), gg.dz, gg.inv_dz);
  else if (iz == nz - 1)
    gz = ddiv_y(dsub(p[0], p[-nr]), gg.dz, gg.inv_dz);
  else
    gz = ddiv_y(dsub(p[nr], p[-nr]), gg.two_dz, gg.inv_two_dz);
  if (ir == 0)
    gr = ddiv_y(dsub(p[1], p[0]), gg.dr, gg.inv_dr);
  else if (ir == nr - 1)
    gr = ddiv_y(dsub(p[0], p[-1]), gg.dr, gg.inv_dr);
  else
    gr = ddiv_y(dsub(p[1], p[-1]), gg.two_dr, gg.inv_two_dr);
}

static GradGeom make_grad_geom(double dz, double dr) {
  GradGeom g;
  volatile double tz = 2.0 * dz, tr = 2.0 * dr;
  g.dz = dz;
  g.dr = dr;
  g.two_dz = tz;
  g.two_dr = tr;
  g.inv_dz = 1.0 / dz;
  g.inv_dr = 1.0 / dr;
  g.inv_two_dz = 1.0 / tz;
  g.inv_two_dr = 1.0 / tr;
  return g;
}

// ---------------------------------------------------------------------------- T
__global__ void __launch_bounds__(256)
k_topo(Bufs bufs, const int *__restrict__ cur, size_t n, int nz, int nr, GradGeom gg,
       const int *__restrict__ rowmask, double *__restrict__ tpart, const int *__restrict__ active) {
  __shared__ double shv[32];
  __shared__ int shi[32];
  const int b = blockIdx.y, P = gridDim.x, p = blockIdx.x;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  const int r0 = (int)((long long)nz * p / P), r1 = (int)((long long)nz * (p + 1) / P);
  ValIdx mx{0.0, -1}, mb{0.0, -1};
  double mn = INFINITY;
  // the block's band as one flat index range, (row, column) carried along without a division per point: every thread
  // is busy whatever nr is (a column-strided row loop leaves ONE thread working in its last trip at nr = 2^k + 1),
  // and a thread meets its points in increasing flat index
  {
    const int step = blockDim.x, sq = step / nr, sm = step - sq * nr;
    int iz = r0 + (int)threadIdx.x / nr, ir = (int)threadIdx.x - ((int)threadIdx.x / nr) * nr;
    const int end = r1 * nr;
#pragma unroll 2
    for (int flat = r0 * nr + (int)threadIdx.x; flat < end; flat += step) {
      const double v = f[flat];
      if (mx.i < 0 || v > mx.v) mx = ValIdx{v, flat};  // strict >: the first maximum of this thread's sequence stays
      mn = fmin(mn, v);
      if (rowmask[iz] != 0) {
        double gz, gr;
        grad_point(f, nz, nr, iz, ir, gg, gz, gr);
        const double bm = hypot_glibc(gr, gz);
        if (isfinite(bm) && (mb.i < 0 || bm < mb.v)) mb = ValIdx{bm, flat};
      }
      ir += sm;
      iz += sq;
      if (ir >= nr) {
        ir -= nr;
        ++iz;
      }
    }
  }
  mx = block_arg<true>(mx, shv, shi);
  __syncthreads();
  mb = block_arg<false>(mb, shv, shi);
  __syncthreads();
  const double mnb = -block_max(-mn, shv);
  if (threadIdx.x == 0) {
    double *o = tpart + ((size_t)b * kPT + p) * kTW;
    o[0] = mx.v;
    o[1] = (double)mx.i;
    o[2] = mb.v;
    o[3] = (double)mb.i;
    o[4] = mnb;
  }
}

// ---------------------------------------------------------------------------- TS
// fusion_kernel.py:295-337: among the (up to) 16 smallest masked |grad psi| keep true saddles
// (Hessian determinant < 0, interior only) and take the one with the smallest |grad psi|.
__global__ void __launch_bounds__(256)
k_xpoint_saddle(Bufs bufs, const int *__restrict__ cur, size_t n, int nz, int nr, GradGeom gg,
                double dr2, double dz2, double four_drdz, const int *__restrict__ rowmask,
                int *__restrict__ xsel, const int *__restrict__ active) {
  __shared__ double shv[32];
  __shared__ int shi[32];
  __shared__ double prev_v;
  __shared__ int prev_i, best_i;
  __shared__ double best_v;
  const int b = blockIdx.x;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  if (threadIdx.x == 0) {
    prev_v = -1.0;
    prev_i = -1;
    best_i = -1;
    best_v = INFINITY;
  }
  __syncthreads();
  for (int round = 0; round < 16; ++round) {
    const double pv = prev_v;
    const int pi = prev_i;
    ValIdx mb{0.0, -1};
    for (int flat = threadIdx.x; flat < nz * nr; flat += blockDim.x) {
      const int iz = flat / nr, ir = flat - iz * nr;
      if (!rowmask[iz]) continue;
      double gz, gr;
      grad_point(f, nz, nr, iz, ir, gg, gz, gr);
      const double bm = hypot_glibc(gr, gz);
      if (!isfinite(bm)) continue;
      // strictly after (pv, pi) in (value, index) lexicographic order
      if (bm < pv || (bm == pv && flat <= pi)) continue;
      mb = better<false>(mb, ValIdx{bm, flat});
    }
    mb = block_arg<false>(mb, shv, shi);
    if (threadIdx.x == 0) {
      prev_v = mb.v;
      prev_i = mb.i;
      if (mb.i >= 0) {
        const int iz = mb.i / nr, ir = mb.i - iz * nr;
        if (iz > 0 && iz < nz - 1 && ir > 0 && ir < nr - 1) {
          const double *q = f + mb.i;
          const double c2 = dmul(2.0, q[0]);
          const double d2r = __ddiv_rn(dadd(dsub(q[1], c2), q[-1]), dr2);
          const double d2z = __ddiv_rn(dadd(dsub(q[nr], c2), q[-nr]), dz2);
          const double drz = __ddiv_rn(
              dadd(dsub(dsub(q[nr + 1], q[nr - 1]), q[-nr + 1]), q[-nr - 1]), four_drdz);
          const double det = dsub(dmul(d2r, d2z), dmul(drz, drz));
          if (isfinite(det) && det < 0.0 && mb.v < best_v) {
            best_v = mb.v;
            best_i = mb.i;
          }
        }
      }
    }
    __syncthreads();
    if (prev_i < 0) break;
  }
  if (threadIdx.x == 0) xsel[b] = best_i;
}

// Two-kernel replacement of k_xpoint_saddle for large grids: |grad psi| is evaluated ONCE per masked
// point.  A: every CTA stages a chunk of masked points' |grad psi| in shared memory and extracts the
// chunk's 16 smallest in (value, flat index) order (16 block-wide argmin rounds over shared memory,
// the winner is replaced by +inf).  B: one CTA per equilibrium merges the chunk winners into the
// global 16 smallest (the same lexicographic order, so ties resolve like the single-CTA kernel) and
// applies the Hessian saddle test of fusion_kernel.py:295-337.
__global__ void __launch_bounds__(256)
k_saddle_cand(Bufs bufs, const int *__restrict__ cur, size_t n, int nz, int nr, GradGeom gg,
              const int *__restrict__ mrows, int n_mrows, int nchunks, double *__restrict__ cand,
              const int *__restrict__ active) {
  __shared__ double sv[kSadChunk];
  __shared__ double shv[32];
  __shared__ int shi[32];
  __shared__ int s_sel;
  const int b = blockIdx.y, c = blockIdx.x;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  const long long total = (long long)n_mrows * nr;
  const long long i0 = (long long)c * kSadChunk;
  const int cnt = (int)max(0LL, min((long long)kSadChunk, total - i0));
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
    const long long idx = i0 + i;
    const int mr = (int)(idx / nr), ir = (int)(idx - (long long)mr * nr);
    const int iz = mrows[mr];
    double gz, gr;
    grad_point(f, nz, nr, iz, ir, gg, gz, gr);
    const double bm = hypot_glibc(gr, gz);
    sv[i] = isfinite(bm) ? bm : INFINITY;
  }
  __syncthreads();
  double *o = cand + (((size_t)b * nchunks + c) * 16) * 2;
  for (int round = 0; round < 16; ++round) {
    ValIdx m{0.0, -1};
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const double v = sv[i];
      if (v < INFINITY && (m.i < 0 || v < m.v)) m = ValIdx{v, i};  // strided ascending i: first minimum wins
    }
    m = block_arg<false>(m, shv, shi);
    if (threadIdx.x == 0) {
      s_sel = m.i;
      if (m.i >= 0) {
        const long long idx = i0 + m.i;
        const int mr = (int)(idx / nr), ir = (int)(idx - (long long)mr * nr);
        o[2 * round] = m.v;
        o[2 * round + 1] = (double)(mrows[mr] * nr + ir);
        sv[m.i] = INFINITY;
      } else {
        o[2 * round] = INFINITY;
        o[2 * round + 1] = -1.0;
      }
    }
    __syncthreads();
    if (s_sel < 0) {  // chunk exhausted: fill the rest
      for (int r = round + 1 + threadIdx.x; r < 16; r += blockDim.x) {
        o[2 * r] = INFINITY;
        o[2 * r + 1] = -1.0;
      }
      break;
    }
  }
}

__global__ void __launch_bounds__(256)
k_saddle_pick(Bufs bufs, const int *__restrict__ cur, size_t n, int nz, int nr, double dr2, double dz2,
              double four_drdz, int nchunks, double *__restrict__ cand, int *__restrict__ xsel,
              const int *__restrict__ active) {
  __shared__ double shv[32];
  __shared__ int shi[32];
  __shared__ int s_sel;
  __shared__ double best_v;
  __shared__ int best_i;
  const int b = blockIdx.x;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  double *cv = cand + (size_t)b * nchunks * 32;
  const int ncand = nchunks * 16;
  if (threadIdx.x == 0) {
    best_v = INFINITY;
    best_i = -1;
  }
  __syncthreads();
  for (int round = 0; round < 16; ++round) {
    // global (value, flat index) minimum of the remaining candidates
    double mv = INFINITY;
    int mf = -1, mslot = -1;
    for (int i = threadIdx.x; i < ncand; i += blockDim.x) {
      const double v = cv[2 * i];
      const int fl = (int)cv[2 * i + 1];
      if (fl < 0) continue;
      if (mslot < 0 || v < mv || (v == mv && fl < mf)) mv = v, mf = fl, mslot = i;
    }
    // reduce on (value, flat): block_arg breaks ties on the index field -> carry the flat index there
    ValIdx m = block_arg<false>(ValIdx{mv, mf}, shv, shi);
    if (threadIdx.x == 0) s_sel = m.i;
    __syncthreads();
    const int sel = s_sel;
    if (sel < 0) break;
    if (mf == sel && mslot >= 0) cv[2 * mslot + 1] = -1.0;  // the owning thread retires the winner (flat indices are unique)
    if (threadIdx.x == 0) {
      const int iz = sel / nr, ir = sel - iz * nr;
      if (iz > 0 && iz < nz - 1 && ir > 0 && ir < nr - 1) {
        const double *q = f + sel;
        const double c2 = dmul(2.0, q[0]);
        const double d2r = __ddiv_rn(dadd(dsub(q[1], c2), q[-1]), dr2);
        const double d2z = __ddiv_rn(dadd(dsub(q[nr], c2), q[-nr]), dz2);
        const double drz = __ddiv_rn(dadd(dsub(dsub(q[nr + 1], q[nr - 1]), q[-nr + 1]), q[-nr - 1]), four_drdz);
        const double det = dsub(dmul(d2r, d2z), dmul(drz, drz));
        if (isfinite(det) && det < 0.0 && m.v < best_v) {
          best_v = m.v;
          best_i = sel;
        }
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) xsel[b] = best_i;
}

// ---------------------------------------------------------------------------- TF
__global__ void k_topo_final(Bufs bufs, const int *__restrict__ cur, size_t n, int nr, int P,
                             const double *__restrict__ tpart, const int *__restrict__ xsel,
                             double *__restrict__ topo, double *__restrict__ axbnd, int limiter,
                             int batch, const int *__restrict__ active) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  ValIdx mx{0.0, -1}, mb{0.0, -1};
  double mn = INFINITY;
  for (int p = 0; p < P; ++p) {
    const double *o = tpart + ((size_t)b * kPT + p) * kTW;
    mx = better<true>(mx, ValIdx{o[0], (int)o[1]});
    mb = better<false>(mb, ValIdx{o[2], (int)o[3]});
    mn = fmin(mn, o[4]);
  }
  double psi_ax = mx.v;
  if (fabs(psi_ax) < 1e-6) psi_ax = 1e-6;  // fusion_kernel.py:353
  int xi = mb.i;
  if (xsel && xsel[b] >= 0) xi = xsel[b];
  double psi_x, found;
  int izx = 0, irx = 0;
  if (xi >= 0) {
    psi_x = f[xi];
    izx = xi / nr;
    irx = xi - izx * nr;
    found = 1.0;
  } else {  // no divertor rows / nothing finite: ((0,0), min psi)  (fusion_kernel.py:339-340)
    psi_x = mn;
    found = 0.0;
  }
  double *t = topo + (size_t)b * 8;
  t[0] = (double)(mx.i / nr);
  t[1] = (double)(mx.i % nr);
  t[2] = psi_ax;
  t[3] = (double)izx;
  t[4] = (double)irx;
  t[5] = psi_x;
  t[6] = found;
  t[7] = mn;
  if (axbnd) {
    double pb = psi_x;
    if (limiter && fabs(dsub(psi_ax, pb)) < 0.1) pb = dmul(psi_ax, 0.1);  // newton_solver.py:505
    axbnd[2 * b] = psi_ax;
    axbnd[2 * b + 1] = pb;
  }
}

// ---------------------------------------------------------------------------- S1 / S2
struct ProfileDev {
  int hmode;
  double p[4], f[4];
};

// mtanh profile (fusion_kernel.py:380-389) with the two per-equilibrium divisors pre-inverted
// (Markstein division, see gsb_internal.cuh)
struct MtanhK {
  double top, width, half_h, alpha, inv_top, inv_width;
};
__device__ __forceinline__ MtanhK mtanh_k(const double *q) {
  MtanhK m;
  m.top = q[0], m.width = q[1], m.half_h = dmul(0.5, q[2]), m.alpha = q[3];
  m.inv_top = __ddiv_rn(1.0, q[0]);
  m.inv_width = __ddiv_rn(1.0, q[1]);
  return m;
}
// tanh(y) for |y| <= 20 as (1 - u)/(1 + u), u = exp(-2y): Cody-Waite reduction, degree-13 Taylor
// polynomial on |r| <= ln2/2 (truncation 4e-18 relative), exponent add, then a Newton-refined
// reciprocal.  Absolute error <= 4e-16 over the range (np.tanh itself is only accurate to ~1 ulp of
// a result that is then added to 1.0), ~30 instructions instead of ~90 for the library tanh().
__device__ __forceinline__ double tanh_lean(double y) {
  const double x = -2.0 * y;  // exact
  const int k = __double2int_rn(x * 1.4426950408889634074);
  const double kf = (double)k;
  double r = __fma_rn(-kf, 6.93147180369123816490e-01, x);
  r = __fma_rn(-kf, 1.90821492927058770002e-10, r);
  // Estrin evaluation of sum_{i<=13} r^i / i!: dependency depth 5 instead of 13 Horner steps (the
  // evaluation is latency bound with 4 warps per scheduler)
  const double r2 = r * r, r4 = r2 * r2, r8 = r4 * r4;
  const double a0 = __fma_rn(r, 1.0, 1.0);
  const double a1 = __fma_rn(r, 1.6666666666666666e-01, 0.5);
  const double a2 = __fma_rn(r, 8.333333333333333e-03, 4.1666666666666664e-02);
  const double a3 = __fma_rn(r, 1.984126984126984e-04, 1.388888888888889e-03);
  const double a4 = __fma_rn(r, 2.7557319223985893e-06, 2.48015873015873e-05);
  const double a5 = __fma_rn(r, 2.505210838544172e-08, 2.755731922398589e-07);
  const double a6 = __fma_rn(r, 1.6059043836821613e-10, 2.08767569878681e-09);
  const double b0 = __fma_rn(a1, r2, a0), b1 = __fma_rn(a3, r2, a2), b2 = __fma_rn(a5, r2, a4);
  const double d0 = __fma_rn(b1, r4, b0), d1 = __fma_rn(a6, r4, b2);
  const double p = __fma_rn(d1, r8, d0);
  const double u = __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));  // |k| <= 58: no over/underflow
  const double d = 1.0 + u, n = 1.0 - u;
  double y0;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(d));
  const double e = __fma_rn(-d, y0, 1.0);
  y0 = __fma_rn(y0, e, y0);  // one Newton step (>= 40 bits); the residual correction below finishes the quotient
  const double q = n * y0;
  return __fma_rn(__fma_rn(-d, q, n), y0, q);
}
__device__ __forceinline__ double mtanh_res(double x, const MtanhK &m) {
  double y = ddiv_yf(dsub(m.top, x), m.width, m.inv_width);
  y = fmin(fmax(y, -20.0), 20.0);
  const double ped = dmul(m.half_h, dadd(1.0, tanh_lean(y)));
  double core = 0.0;
  if (x < m.top) {
    const double t = ddiv_yf(x, m.top, m.inv_top);
    core = fmax(0.0, dsub(1.0, dmul(t, t)));
  }
  return dadd(ped, dmul(m.alpha, core));
}

__global__ void __launch_bounds__(256)
k_source_raw(Bufs bufs, const int *__restrict__ cur, size_t n, int nz, int nr,
             const double *__restrict__ axbnd, ProfileDev prof, const double *__restrict__ prof_dev,
             const double *__restrict__ rrow, const double *__restrict__ cf,
             double *__restrict__ jraw, double *__restrict__ spart, const int *__restrict__ active) {
  __shared__ double sh[32];
  const int b = blockIdx.y, P = gridDim.x, p = blockIdx.x;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  const double psi_ax = axbnd[2 * b];
  double denom = dsub(axbnd[2 * b + 1], psi_ax);
  if (fabs(denom) < 1e-9) denom = 1e-9;
  const double inv_denom = __ddiv_rn(1.0, denom);
  double pp[4], pf[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    pp[i] = prof_dev ? prof_dev[(size_t)b * 8 + i] : prof.p[i];
    pf[i] = prof_dev ? prof_dev[(size_t)b * 8 + 4 + i] : prof.f[i];
  }
  // the same profile evaluation as the resident kernel (lean tanh, pre-inverted divisors, one evaluation when
  // p' and FF' share their parameters): both Picard paths see identical profile values
  const MtanhK mkp = mtanh_k(pp), mkf = mtanh_k(pf);
  const bool same_prof = pp[0] == pf[0] && pp[1] == pf[1] && pp[2] == pf[2] && pp[3] == pf[3];
  const int r0 = (int)((long long)nz * p / P), r1 = (int)((long long)nz * (p + 1) / P);
  double acc = 0.0;
  // the block's band as one flat index range with the column carried along (every thread busy whatever nr is)
  const int step = blockDim.x, sm = step % nr;
  int ir = (int)threadIdx.x % nr;
#pragma unroll 2
  for (size_t o = (size_t)r0 * nr + threadIdx.x; o < (size_t)r1 * nr; o += step, ir = (ir + sm >= nr) ? ir + sm - nr : ir + sm) {
      const double pn = ddiv_yf(dsub(f[o], psi_ax), denom, inv_denom);
      const bool in = (pn >= 0.0) && (pn < 1.0);
      double pr = 0.0, ff = 0.0;
      if (in) {
        if (prof.hmode) {
          pr = mtanh_res(pn, mkp);
          ff = same_prof ? pr : mtanh_res(pn, mkf);
        } else {
          pr = dsub(1.0, pn);
          ff = pr;
        }
      }
      // J_raw = 0.5*(R*p) + 0.5*((1/(mu0 R))*ff)      (fusion_kernel.py:430-434)
      const double j = dadd(dmul(0.5, dmul(rrow[ir], pr)), dmul(0.5, dmul(cf[ir], ff)));
      jraw[(size_t)b * n + o] = j;
      acc += j;
    }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) spart[(size_t)b * kPT + p] = acc;
}

__global__ void __launch_bounds__(256)
k_source_scale(size_t n, int nz, int nr, double dr, double dz, const double *__restrict__ ip,
               const double *__restrict__ spart, int P, const double *__restrict__ mr,
               double *__restrict__ jphi, double *__restrict__ source, double *__restrict__ scale_out,
               const int *__restrict__ active) {
  const int b = blockIdx.y, p = blockIdx.x;
  if (active && !active[b]) return;
  double s = 0.0;
  for (int q = 0; q < P; ++q) s += spart[(size_t)b * kPT + q];
  const double icur = dmul(dmul(s, dr), dz);  // float(np.sum(J_raw)) * dR * dZ
  const bool ok = fabs(icur) > 1e-9;
  const double sc = ok ? __ddiv_rn(ip[b], icur) : 0.0;
  if (scale_out && p == 0 && threadIdx.x == 0) scale_out[b] = sc;
  const int r0 = (int)((long long)nz * p / gridDim.x), r1 = (int)((long long)nz * (p + 1) / gridDim.x);
  // the block's band as one flat index range, four elements per trip with their loads issued together; the column
  // index is carried along (no division per point, every thread busy whatever nr is)
  const int step = blockDim.x, sm = step % nr;
  int ir = (int)threadIdx.x % nr;
  const size_t base = (size_t)b * n, end = (size_t)r1 * nr;
  for (size_t o = (size_t)r0 * nr + threadIdx.x; o < end; o += (size_t)4 * step) {
    double jv[4];
    int irk[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      irk[k] = ir;
      ir = (ir + sm >= nr) ? ir + sm - nr : ir + sm;
      jv[k] = (o + (size_t)k * step < end) ? jphi[base + o + (size_t)k * step] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (o + (size_t)k * step < end) {
        const double j = ok ? dmul(jv[k], sc) : 0.0;
        jphi[base + o + (size_t)k * step] = j;
        if (source) source[base + o + (size_t)k * step] = dmul(mr[irk[k]], j);  // (-mu0*R)*J
      }
  }
}

// ---------------------------------------------------------------------------- E helpers
__global__ void __launch_bounds__(256)
k_copy_from_cur(Bufs bufs, const int *__restrict__ cur, size_t n, double *__restrict__ dst,
                int do_sanitize, const int *__restrict__ active) {
  const int b = blockIdx.y;
  if (active && !active[b]) return;
  const double *f = bufs.p[cur ? cur[b] : 0] + (size_t)b * n;
  double *d = dst + (size_t)b * n;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {  // four independent loads in flight per thread
    const double v0 = f[i], v1 = f[i + stride], v2 = f[i + 2 * stride], v3 = f[i + 3 * stride];
    d[i] = do_sanitize ? sanitize(v0) : v0;
    d[i + stride] = do_sanitize ? sanitize(v1) : v1;
    d[i + 2 * stride] = do_sanitize ? sanitize(v2) : v2;
    d[i + 3 * stride] = do_sanitize ? sanitize(v3) : v3;
  }
  for (; i < n; i += stride) d[i] = do_sanitize ? sanitize(f[i]) : f[i];
}

__global__ void __launch_bounds__(256)
k_jacobi_from_cur(LevelGeom g, Bufs bufs, const int *__restrict__ cur, const double *__restrict__ src,
                  double *__restrict__ out, const int *__restrict__ active) {
  const int b = blockIdx.z;
  if (active && !active[b]) return;
  const int ir = blockIdx.x * blockDim.x + threadIdx.x;
  const int iz = blockIdx.y * blockDim.y + threadIdx.y;
  if (ir >= g.nr || iz >= g.nz) return;
  const size_t n = (size_t)g.nz * g.nr;
  const double *p = bufs.p[cur[b]] + b * n + (size_t)iz * g.nr + ir;
  double v;
  if (iz == 0 || ir == 0 || iz == g.nz - 1 || ir == g.nr - 1) {
    v = sanitize(p[0]);
  } else {
    double acc = dadd(dmul(g.a_e[ir], sanitize(p[1])), dmul(g.a_w[ir], sanitize(p[-1])));
    acc = dadd(acc, dmul(g.a_ns, sanitize(p[-g.nr])));
    acc = dadd(acc, dmul(g.a_ns, sanitize(p[g.nr])));
    acc = dsub(acc, sanitize(src[b * n + (size_t)iz * g.nr + ir]));
    v = clip_cap(ddiv_y(acc, g.a_c, g.inv_a_c));
  }
  out[b * n + (size_t)iz * g.nr + ir] = v;
}

// ---------------------------------------------------------------------------- R
// ring layout as in gsb_mg.cu: [row0][row nz-1][col0][col nr-1]
__device__ __forceinline__ double wall_or(const double *__restrict__ W, const double *__restrict__ ring,
                                          int nz, int nr, int iz, int ir) {
  if (ir == 0) return ring[2 * nr + iz];
  if (ir == nr - 1) return ring[2 * nr + nz + iz];
  if (iz == 0) return ring[ir];
  if (iz == nz - 1) return ring[nr + ir];
  return W[(size_t)iz * nr + ir];
}

// A WARP owns 30 columns x a band of rows (32 lanes = the 30 columns plus one halo column on either side, whose
// lanes only form the relaxed value for their neighbours); a lane keeps its column and walks down the band with a
// three-row register window of the RELAXED iterate, so a point costs three global loads (psi, Psi_new of the row
// entering the window, the source) and one store, and the east / west neighbours of the residual stencil are warp
// shuffles with no edge cases.  The wall ring has been written into Psi_new beforehand (ring_apply_launch), so the
// row loop has no wall logic at all.  r2's first version (column chunk x band, wall handling and warp-edge loads in
// the loop) ran 214 instructions per point at 16 warps per SM; this one runs ~70.
constexpr int kRxCols = 30;  // owned columns per warp
struct RelaxPlan {
  int n_cw, n_rb, P;  // column warps, row bands, partial blocks (4 warps each) per equilibrium
};
static RelaxPlan relax_plan(int nz, int nr, int batch, int num_sms) {
  RelaxPlan r;
  r.n_cw = (std::max(nr - 1, 1) + kRxCols - 1) / kRxCols;  // columns 1 .. nr-1 in runs of 30; column 0 rides with the first
  const long long want = 64LL * num_sms;               // a few waves of resident warps: the kernel is load-latency bound
  const long long have = (long long)r.n_cw * batch;
  r.n_rb = (int)std::max<long long>(1, std::min<long long>((want + have - 1) / have, nz / 16));
  r.P = std::min((r.n_cw * r.n_rb + 3) / 4, kPT);
  return r;
}
__global__ void __launch_bounds__(128)
k_relax(LevelGeom g, Bufs bufs, const int *__restrict__ cur, const int *__restrict__ nxt,
        const double *__restrict__ Wall, const double *__restrict__ srcall, double alpha, double oma,
        double *__restrict__ rpart, const int *__restrict__ active, RelaxPlan rp) {
  __shared__ double sh[4][4];
  const int b = blockIdx.y;
  if (active && !active[b]) return;
  const int nz = g.nz, nr = g.nr;
  const size_t n = (size_t)nz * nr;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double dsum = 0.0, rmax = 0.0, rsq = 0.0;
  int bad = 0;
  constexpr int G = 4;  // rows per group: the loads of a whole group are in flight before the first use
  const int tiles = rp.n_cw * rp.n_rb;
  for (int tile = blockIdx.x * 4 + wid; tile < tiles; tile += rp.P * 4) {
    const int band = tile / rp.n_cw, cw = tile - band * rp.n_cw;
    const int col = cw * kRxCols + lane;
    const int jc = min(col, nr - 1);  // clamped: every lane loads from a valid address
    const bool owned = col < nr && ((lane >= 1 && lane <= kRxCols) || col == 0);
    const bool res_col = owned && col >= 1 && col <= nr - 2;
    const int z0 = (int)((long long)nz * band / rp.n_rb), z1 = (int)((long long)nz * (band + 1) / rp.n_rb);
    const double *fcol = bufs.p[cur[b]] + b * n + jc;
    const double *wcol = Wall + b * n + jc;
    const double *scol = srcall + b * n + jc;
    double *ocol = bufs.p[nxt[b]] + b * n + jc;
    const double rs = res_col ? g.r_safe[col] : 1.0, irs = res_col ? g.inv_r_safe[col] : 1.0;
    // window: relaxed values (1-a)*Psi + a*Psi_new (newton_solver.py:536) of rows iz-1, iz; (Psi_new, Psi) of row iz
    const size_t om = (size_t)max(z0 - 1, 0) * nr, o0 = (size_t)z0 * nr;
    double c_m = dadd(dmul(oma, fcol[om]), dmul(alpha, wcol[om]));
    double wn_0 = wcol[o0], old_0 = fcol[o0];
    double c_0 = dadd(dmul(oma, old_0), dmul(alpha, wn_0));
    for (int zb = z0; zb < z1; zb += G) {
      double wnv[G], oldv[G], sv[G];
#pragma unroll
      for (int u = 0; u < G; ++u) {  // row zb+u+1 enters the window; clamped rows are loaded and never used
        const size_t on_ = (size_t)min(zb + u + 1, nz - 1) * nr, oc = (size_t)min(zb + u, nz - 1) * nr;
        wnv[u] = wcol[on_];
        oldv[u] = fcol[on_];
        sv[u] = scol[oc];
      }
#pragma unroll
      for (int u = 0; u < G; ++u) {
        const int iz = zb + u;
        if (iz < z1) {  // warp-uniform
          const double c_p = dadd(dmul(oma, oldv[u]), dmul(alpha, wnv[u]));
          if (owned) {
            if (!(fabs(wn_0) <= 1.79769313486231570815e308)) bad = 1;  // NaN or +-inf in Psi_new
            dsum += fabs(dsub(wn_0, old_0));
            ocol[(size_t)iz * nr] = c_0;
          }
          const double c_w = __shfl_up_sync(0xffffffffu, c_0, 1), c_e = __shfl_down_sync(0xffffffffu, c_0, 1);
          if (res_col && iz > 0 && iz < nz - 1) {
            const double r = dsub(gs_apply_v(g, rs, irs, c_0, c_e, c_w, c_m, c_p), sv[u]);
            rmax = fmax(rmax, fabs(r));
            rsq += r * r;
          }
          c_m = c_0;
          c_0 = c_p;
          wn_0 = wnv[u];
          old_0 = oldv[u];
        }
      }
    }
  }
  dsum = warp_sum(dsum);
  rmax = warp_max(rmax);
  rsq = warp_sum(rsq);
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) {
    sh[wid][0] = dsum;
    sh[wid][1] = bad ? 1.0 : 0.0;
    sh[wid][2] = rmax;
    sh[wid][3] = rsq;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double *o = rpart + ((size_t)b * kPT + blockIdx.x) * kRW;
    o[0] = ((sh[0][0] + sh[1][0]) + sh[2][0]) + sh[3][0];
    o[1] = (sh[0][1] + sh[1][1] + sh[2][1] + sh[3][1]) > 0.0 ? 1.0 : 0.0;
    o[2] = fmax(fmax(sh[0][2], sh[1][2]), fmax(sh[2][2], sh[3][2]));
    o[3] = ((sh[0][3] + sh[1][3]) + sh[2][3]) + sh[3][3];
  }
}

// ---------------------------------------------------------------------------- D
__global__ void k_decide(PicardState s, const double *__restrict__ rpart, int P, double n_all,
                         double n_int, double tol, int need_gs, double gs_tol, int max_iter,
                         double *__restrict__ hist, double *__restrict__ gs_hist,
                         int *__restrict__ counter, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  if (!s.active[b]) return;
  double dsum = 0.0, rmax = 0.0, rsq = 0.0;
  bool bad = false;
  for (int p = 0; p < P; ++p) {
    const double *o = rpart + ((size_t)b * kPT + p) * kRW;
    dsum += o[0];
    bad = bad || (o[1] != 0.0);
    rmax = fmax(rmax, o[2]);
    rsq += o[3];
  }
  const int k = s.iter[b];
  if (bad) {  // NaN/Inf in Psi_new: revert to the best state and stop (newton_solver.py:518-532)
    s.status[b] = 3;
    s.iter[b] = k + 1;
    s.active[b] = 0;
    s.cur[b] = s.best[b];
    return;
  }
  const double diff = dsum / n_all;
  const double gs = (rmax > 0.0 && n_int > 0.0) ? sqrt(rsq / n_int) : 0.0;
  if (hist) hist[(size_t)b * max_iter + k] = diff;
  if (gs_hist) gs_hist[(size_t)b * max_iter + k] = gs;
  s.diff_last[b] = diff;
  s.gs_last[b] = gs;
  if (gs < s.gs_best[b]) s.gs_best[b] = gs;
  const int newcur = s.nxt[b];
  int best = s.best[b];
  if (diff < s.diff_best[b]) {
    s.diff_best[b] = diff;
    best = newcur;
  }
  s.cur[b] = newcur;
  s.best[b] = best;
  s.nxt[b] = (newcur == best) ? (newcur + 1) % 3 : 3 - newcur - best;
  s.iter[b] = k + 1;
  const bool conv = (diff < tol) && (!need_gs || gs < gs_tol);
  if (conv) {
    s.status[b] = 1;
    s.active[b] = 0;
  } else if (k + 1 >= max_iter) {
    s.status[b] = 2;
    s.active[b] = 0;
  } else {
    atomicAdd(counter, 1);
  }
}

// ---------------------------------------------------------------------------- A  (solver_method "anderson")
// Anderson mixing of the relaxed Picard iterates (fusion_kernel_iterative_solver.py:248-314, called from
// fusion_kernel_newton_solver.py:539-550): every iteration pushes (Psi_relaxed, Psi_new - Psi_relaxed) into a ring of
// `m` slots; on iterations k = 3, 6, 9, ... the iterate is replaced by sum_j alpha_j Psi_j over the last
// mk = min(m, k+1) entries, alpha from the 1e-10-regularised normal equations of the residual differences, walls reset
// to the boundary map, and the GS residual of the iteration is taken of the MIXED state.  Every active equilibrium of a
// solve is at the same iteration, but the decision "is this a mixing iteration" is taken on the device from s.iter so
// that the launch sequence stays iteration-independent (CUDA-graph replay).
// Not bit-identical to NumPy by construction: the reference forms the Gram matrix with BLAS (dF.T @ dF) and solves it
// with LAPACK gesv, whose summation orders are not specified; here fixed trees + partial-pivot LU.
constexpr int kAndMax = 8;                                           // largest supported mixing depth
constexpr int kAndEnt = (kAndMax - 1) * kAndMax / 2 + (kAndMax - 1); // upper-triangular Gram entries + rhs
constexpr int kAndPB = 16;                                           // partial blocks per equilibrium

__device__ __forceinline__ bool and_mix_iter(int k) { return k >= 3 && k % 3 == 0; }  // len(history) >= 3 and k % 3 == 0
__device__ __forceinline__ int and_mk(int m, int k) { return min(m, k + 1); }

struct AndersonBufs {
  double *psi, *res;   // [batch_cap][slots][n] rings
  double *part;        // [batch_cap][kAndPB][kAndEnt]
  double *alpha;       // [batch_cap][kAndMax]
  int *fallback;       // [batch_cap] 1: the mixed iterate is the latest iterate (LinAlgError / |sum alpha| < 1e-12 / mk < 2)
  int m, slots;
};

__global__ void __launch_bounds__(256)
k_and_push(AndersonBufs a, Bufs bufs, const int *__restrict__ nxt, const int *__restrict__ iter,
           const double *__restrict__ Wall, const double *__restrict__ ringall, int nz, int nr,
           const int *__restrict__ active) {
  const int b = blockIdx.y;
  if (!active[b] || a.m < 2) return;
  const size_t n = (size_t)nz * nr;
  const int slot = iter[b] % a.slots;
  const double *rel = bufs.p[nxt[b]] + b * n;
  const double *W = Wall + b * n;
  const double *ring = ringall + (size_t)b * ring_size(nz, nr);
  double *hp = a.psi + ((size_t)b * a.slots + slot) * n, *hr = a.res + ((size_t)b * a.slots + slot) * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int iz = (int)(i / nr), ir = (int)(i - (size_t)iz * nr);
    const double r = rel[i];
    hp[i] = r;
    hr[i] = dsub(wall_or(W, ring, nz, nr, iz, ir), r);  // Psi_new - Psi (relaxed), newton_solver.py:542
  }
}

__global__ void __launch_bounds__(256)
k_and_gram(AndersonBufs a, const int *__restrict__ iter, size_t n, const int *__restrict__ active) {
  __shared__ double sh[32];
  const int b = blockIdx.y;
  if (!active[b]) return;
  const int k = iter[b];
  if (!and_mix_iter(k)) return;
  const int mk = and_mk(a.m, k);
  if (mk < 2) return;
  const int d = mk - 1;
  const double *col[kAndMax];
#pragma unroll
  for (int j = 0; j < kAndMax; ++j) {
    const int slot = (k - mk + 1 + min(j, mk - 1)) % a.slots;  // oldest first; unused columns alias the last one
    col[j] = a.res + ((size_t)b * a.slots + slot) * n;
  }
  double acc[kAndEnt];
#pragma unroll
  for (int e = 0; e < kAndEnt; ++e) acc[e] = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    double r[kAndMax], df[kAndMax - 1];
#pragma unroll
    for (int j = 0; j < kAndMax; ++j) r[j] = j < mk ? col[j][i] : 0.0;
    const double last = col[kAndMax - 1][i];  // aliases column mk-1
#pragma unroll
    for (int j = 0; j < kAndMax - 1; ++j) df[j] = j < d ? dsub(r[j + 1], r[j]) : 0.0;  // np.diff(F, axis=1)
    int e = 0;
#pragma unroll
    for (int p = 0; p < kAndMax - 1; ++p)
#pragma unroll
      for (int q = p; q < kAndMax - 1; ++q, ++e) acc[e] += df[p] * df[q];
#pragma unroll
    for (int p = 0; p < kAndMax - 1; ++p, ++e) acc[e] += df[p] * last;
  }
  double *o = a.part + ((size_t)b * kAndPB + blockIdx.x) * kAndEnt;
#pragma unroll
  for (int e = 0; e < kAndEnt; ++e) {
    const double v = block_sum(acc[e], sh);
    if (threadIdx.x == 0) o[e] = v;
  }
}

// One thread per equilibrium: Gram assembly, + 1e-10 I, LU with partial pivoting (first largest |a_ik|, as idamax),
// gamma, alpha (fusion_kernel_iterative_solver.py:289-303, np.sum restated for <= 8 values).
__global__ void k_and_solve(AndersonBufs a, const int *__restrict__ iter, int n_part, int batch,
                            const int *__restrict__ active) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch || !active[b]) return;
  const int k = iter[b];
  if (!and_mix_iter(k)) return;
  const int mk = and_mk(a.m, k);
  if (mk < 2) {
    a.fallback[b] = 1;
    return;
  }
  const int d = mk - 1;
  double ent[kAndEnt];
  for (int e = 0; e < kAndEnt; ++e) {
    double v = 0.0;
    for (int p = 0; p < n_part; ++p) v += a.part[((size_t)b * kAndPB + p) * kAndEnt + e];
    ent[e] = v;
  }
  double A[kAndMax - 1][kAndMax - 1], x[kAndMax - 1];
  int e = 0;
  for (int p = 0; p < kAndMax - 1; ++p)
    for (int q = p; q < kAndMax - 1; ++q, ++e)
      if (q < d) A[p][q] = A[q][p] = ent[e];
  for (int p = 0; p < kAndMax - 1; ++p, ++e)
    if (p < d) x[p] = ent[e];
  for (int p = 0; p < d; ++p) A[p][p] = dadd(A[p][p], 1e-10);
  bool singular = false;
  for (int c = 0; c < d && !singular; ++c) {
    int piv = c;
    double best = fabs(A[c][c]);
    for (int r = c + 1; r < d; ++r)
      if (fabs(A[r][c]) > best) {
        best = fabs(A[r][c]);
        piv = r;
      }
    if (A[piv][c] == 0.0) {
      singular = true;  // gesv info > 0 -> numpy raises LinAlgError
      break;
    }
    if (piv != c) {
      for (int q = 0; q < d; ++q) {
        const double t = A[c][q];
        A[c][q] = A[piv][q];
        A[piv][q] = t;
      }
      const double t = x[c];
      x[c] = x[piv];
      x[piv] = t;
    }
    const double rp = 1.0 / A[c][c];
    for (int r = c + 1; r < d; ++r) {
      const double l = A[r][c] * rp;
      for (int q = c + 1; q < d; ++q) A[r][q] -= l * A[c][q];
      x[r] -= l * x[c];
    }
  }
  int fb = singular ? 1 : 0;
  double al[kAndMax];
  if (!singular) {
    for (int r = d - 1; r >= 0; --r) {
      double v = x[r];
      for (int q = r + 1; q < d; ++q) v -= A[r][q] * x[q];
      x[r] = v / A[r][r];
    }
    double gs = 0.0;
    for (int j = 0; j < d; ++j) gs = dadd(gs, x[j]);  // np.sum of < 8 values: left to right from 0
    for (int j = 0; j < d; ++j) al[j] = dsub(0.0, x[j]);
    al[d] = dsub(1.0, gs);
    double tot;
    if (mk < 8) {
      tot = 0.0;
      for (int j = 0; j < mk; ++j) tot = dadd(tot, al[j]);
    } else {  // np.sum of exactly 8 values: eight accumulators combined as a tree
      tot = dadd(dadd(dadd(al[0], al[1]), dadd(al[2], al[3])), dadd(dadd(al[4], al[5]), dadd(al[6], al[7])));
    }
    if (fabs(tot) < 1e-12) fb = 1;  // (a NaN sum compares false here as in the reference and mixes NaN through)
    if (!fb)
      for (int j = 0; j < mk; ++j) a.alpha[(size_t)b * kAndMax + j] = __ddiv_rn(al[j], tot);
  }
  a.fallback[b] = fb;
}

// mixed = sum_j alpha_j Psi_j (accumulated from zeros in history order, :306-312), walls <- boundary map
// (_apply_boundary_conditions); the fallback keeps the relaxed iterate and only resets its walls.
__global__ void __launch_bounds__(256)
k_and_mix(AndersonBufs a, Bufs bufs, const int *__restrict__ nxt, const int *__restrict__ iter,
          const double *__restrict__ ringall, int nz, int nr, const int *__restrict__ active) {
  const int b = blockIdx.y;
  if (!active[b]) return;
  const int k = iter[b];
  if (!and_mix_iter(k)) return;
  const size_t n = (size_t)nz * nr;
  const int mk = and_mk(a.m, k);
  const bool fb = a.fallback[b] != 0;
  const double *ring = ringall + (size_t)b * ring_size(nz, nr);
  double *out = bufs.p[nxt[b]] + b * n;
  const double *col[kAndMax];
  double al[kAndMax];
#pragma unroll
  for (int j = 0; j < kAndMax; ++j) {
    const int slot = (k - mk + 1 + min(j, max(mk - 1, 0))) % a.slots;
    col[j] = a.psi + ((size_t)b * a.slots + slot) * n;
    al[j] = (!fb && j < mk) ? a.alpha[(size_t)b * kAndMax + j] : 0.0;
  }
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int iz = (int)(i / nr), ir = (int)(i - (size_t)iz * nr);
    if (iz == 0 || iz == nz - 1 || ir == 0 || ir == nr - 1) {
      out[i] = wall_or(nullptr, ring, nz, nr, iz, ir);
    } else if (!fb) {
      double v = 0.0;
#pragma unroll
      for (int j = 0; j < kAndMax; ++j)
        if (j < mk) v = dadd(v, dmul(al[j], col[j][i]));
      out[i] = v;
    }
  }
}

// GS residual statistics of the mixed iterate (newton_solver.py:552 sees self.Psi AFTER the mixing step): overwrites
// the (max |r|, sum r^2) entries k_relax left for the relaxed iterate, in the same P partial slots k_decide adds up.
__global__ void __launch_bounds__(256)
k_and_gs(LevelGeom g, Bufs bufs, const int *__restrict__ nxt, const int *__restrict__ iter,
         const double *__restrict__ srcall, double *__restrict__ rpart, const int *__restrict__ active) {
  __shared__ double sh[32];
  const int b = blockIdx.y, p = blockIdx.x;
  if (!active[b] || !and_mix_iter(iter[b])) return;
  const int nz = g.nz, nr = g.nr;
  const size_t n = (size_t)nz * nr;
  const double *f = bufs.p[nxt[b]] + b * n;
  const double *src = srcall + b * n;
  const size_t n_in = (size_t)(nz - 2) * (nr - 2);
  double rmax = 0.0, rsq = 0.0;
  for (size_t q = (size_t)p * blockDim.x + threadIdx.x; q < n_in; q += (size_t)gridDim.x * blockDim.x) {
    const int iz = 1 + (int)(q / (nr - 2)), ir = 1 + (int)(q % (nr - 2));
    const size_t o = (size_t)iz * nr + ir;
    const double r = dsub(gs_apply(g, ir, f[o], f[o + 1], f[o - 1], f[o - nr], f[o + nr]), src[o]);
    rmax = fmax(rmax, fabs(r));
    rsq += r * r;
  }
  rmax = block_max(rmax, sh);
  __syncthreads();
  rsq = block_sum(rsq, sh);
  if (threadIdx.x == 0) {
    double *o = rpart + ((size_t)b * kPT + p) * kRW;
    o[2] = rmax;
    o[3] = rsq;
  }
}

__global__ void k_picard_init(PicardState s, int batch, int best0, const double *__restrict__ ip,
                              int seed, const int *__restrict__ mask) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const int on = mask ? (mask[b] != 0) : 1;  // masked-out equilibria are left untouched by the whole solve
  s.active[b] = on;
  s.status[b] = 0;
  s.iter[b] = 0;
  s.cur[b] = 0;
  s.best[b] = best0;
  s.nxt[b] = 1;
  s.xsel[b] = -1;
  s.seed_active[b] = (on && seed && fabs(ip[b]) >= 1e-12) ? 1 : 0;
  s.diff_best[b] = 1e9;
  s.gs_best[b] = INFINITY;
  s.gs_last[b] = INFINITY;
  s.diff_last[b] = 0.0;
  s.scale[b] = 0.0;
}

// seed source: Source0 = (-mu0 R) * (seedJ * Ip/I_seed)   (fusion_kernel_iterative_solver.py:400-408)
__global__ void __launch_bounds__(256)
k_seed_source(size_t n, int nr, const double *__restrict__ seedJ, double seed_sum_drdz,
              const double *__restrict__ ip, const double *__restrict__ mr,
              double *__restrict__ jphi, double *__restrict__ source,
              const int *__restrict__ seed_active) {
  const int b = blockIdx.y;
  if (!seed_active[b]) return;
  const double sc = seed_sum_drdz > 0.0 ? __ddiv_rn(ip[b], seed_sum_drdz) : 1.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const double j = dmul(seedJ[i], sc);
    jphi[(size_t)b * n + i] = j;
    source[(size_t)b * n + i] = dmul(mr[i % nr], j);
  }
}

__global__ void __launch_bounds__(256)
k_finalize(Bufs bufs, PicardState s, size_t n, double *__restrict__ summary, int batch,
           const int *__restrict__ mask) {
  const int b = blockIdx.y;
  if (mask && !mask[b]) return;
  const int c = s.cur[b];
  if (c != 0) {
    const double *f = bufs.p[c] + (size_t)b * n;
    double *d = bufs.p[0] + (size_t)b * n;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
      d[i] = f[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && summary) {
    double *o = summary + (size_t)b * 16;
    const double *t = s.topo + (size_t)b * 8;
    o[0] = (double)s.iter[b];
    o[1] = s.status[b] == 1 ? 1.0 : 0.0;
    o[2] = s.diff_best[b];
    o[3] = s.gs_last[b];
    o[4] = s.gs_best[b];
    o[5] = (double)s.status[b];
    o[6] = s.axbnd[2 * b];
    o[7] = s.axbnd[2 * b + 1];
    o[8] = t[0];
    o[9] = t[1];
    o[10] = t[3];
    o[11] = t[4];
    o[12] = s.diff_last[b];
    o[13] = t[6];
    o[14] = s.scale[b];
    o[15] = 0.0;
  }
}

// compute_b_field (fusion_kernel.py:450-456)
__global__ void __launch_bounds__(256)
k_bfield(const double *__restrict__ psi, int nz, int nr, GradGeom gg, const double *__restrict__ rrow,
         double *__restrict__ br, double *__restrict__ bz) {
  const int b = blockIdx.z;
  const int ir = blockIdx.x * blockDim.x + threadIdx.x;
  const int iz = blockIdx.y * blockDim.y + threadIdx.y;
  if (ir >= nr || iz >= nz) return;
  const size_t n = (size_t)nz * nr;
  double gz, gr;
  grad_point(psi + b * n, nz, nr, iz, ir, gg, gz, gr);
  const double rs = fmax(rrow[ir], 1e-6);
  const double inv = __ddiv_rn(1.0, rs);
  br[b * n + (size_t)iz * nr + ir] = dmul(-inv, gz);
  bz[b * n + (size_t)iz * nr + ir] = dmul(inv, gr);
}


// ============================================================================================
// Persistent shared-memory-resident Picard solve: ONE CTA runs the COMPLETE solve of one
// equilibrium (seed, every Picard iteration, V-cycles, convergence logic) and then fetches the
// next one.  psi lives in the colour-split shared-memory planes (gsb_resident.cuh) for the whole
// solve; the only per-iteration global traffic is the CTA's private, L2-resident workspace
// (previous iterate, J, right-hand side - all in the same colour-split layout).  No host polling,
// no launch per phase, and an equilibrium stops the moment it converges instead of waiting for the
// slowest of the batch.
//
// Element-wise phases walk the "slots" e = iz*hw + k (column pair 2k, 2k+1 of row iz) with stride
// blockDim.x: x(iz,2k) = plane[iz&1][e], x(iz,2k+1) = plane[(iz+1)&1][e], so both planes are read
// and written unit-stride and (iz, k) are tracked incrementally (no integer division in loops).
// ============================================================================================
struct PicardResArgs {
  double *psi;              // [B][n] in: initial flux, out: solution
  const double *bc;         // [B][n] boundary map (wall ring read)
  const double *ip;         // [B]
  const double *prof_dev;   // NULL or [B][8]
  double *jphi;             // [B][n] out
  double *summary;          // [B][16] out
  double *hist, *gs_hist;   // NULL or [B][max_iter]
  double *ws_psi;           // [grid][3][2*nz*hw]  iterate rotation (cur / next / best), colour-split
  double *ws_src;           // [grid][2*nz*hw]     J_raw, then the right-hand side (rescaled in place), colour-split
  const double *seedJ, *cf, *mr, *rrow;
  const int *rowmask;
  double seed_sum_drdz;
  int batch, max_iter, seed, saddle, need_gs, external;
  double tol, gs_tol, alpha, oma, omega;
  double dr, dz, dr2, dz2, four_drdz;
  GradGeom gg;
  ProfileDev prof;
  int scratch_off;          // pool offset (doubles) of 96 doubles of reduction / broadcast scratch
  int tplane_off;           // pool offset of a spare half plane (Jacobi seed)
  const int *order;         // NULL, or the compacted list of equilibria to solve (free-boundary outer loop)
  const int *n_order;       // device count of entries in `order`
};

__device__ __forceinline__ double pl(int xo, int nz, int hw, int iz, int ir) {
  return res_pool[xo + split_index(nz, hw, iz, ir)];
}

// np.gradient on the resident planes (same arithmetic as grad_point); generic accessor, used by the
// saddle filter only
__device__ __forceinline__ void grad_planes(int xo, int nz, int nr, int hw, int iz, int ir, const GradGeom &gg,
                                            double &gz, double &gr) {
  const double c = pl(xo, nz, hw, iz, ir);
  if (iz == 0)
    gz = ddiv_y(dsub(pl(xo, nz, hw, 1, ir), c), gg.dz, gg.inv_dz);
  else if (iz == nz - 1)
    gz = ddiv_y(dsub(c, pl(xo, nz, hw, iz - 1, ir)), gg.dz, gg.inv_dz);
  else
    gz = ddiv_y(dsub(pl(xo, nz, hw, iz + 1, ir), pl(xo, nz, hw, iz - 1, ir)), gg.two_dz, gg.inv_two_dz);
  if (ir == 0)
    gr = ddiv_y(dsub(pl(xo, nz, hw, iz, 1), c), gg.dr, gg.inv_dr);
  else if (ir == nr - 1)
    gr = ddiv_y(dsub(c, pl(xo, nz, hw, iz, ir - 1)), gg.dr, gg.inv_dr);
  else
    gr = ddiv_y(dsub(pl(xo, nz, hw, iz, ir + 1), pl(xo, nz, hw, iz, ir - 1)), gg.two_dr, gg.inv_two_dr);
}

// |grad psi| of one point from its own value and its four neighbours (np.gradient semantics:
// centred differences inside, one-sided first-order differences on the edges), np.hypot
__device__ __forceinline__ double grad_mag(const GradGeom &gg, double c, double up, double down, double left,
                                           double right, bool z_lo, bool z_hi, bool r_lo, bool r_hi) {
  double gz, gr;
  if (z_lo)
    gz = ddiv_yf(dsub(up, c), gg.dz, gg.inv_dz);
  else if (z_hi)
    gz = ddiv_yf(dsub(c, down), gg.dz, gg.inv_dz);
  else
    gz = ddiv_yf(dsub(up, down), gg.two_dz, gg.inv_two_dz);
  if (r_lo)
    gr = ddiv_yf(dsub(right, c), gg.dr, gg.inv_dr);
  else if (r_hi)
    gr = ddiv_yf(dsub(c, left), gg.dr, gg.inv_dr);
  else
    gr = ddiv_yf(dsub(right, left), gg.two_dr, gg.inv_two_dr);
  return hypot_glibc(gr, gz);
}

// J_raw of one point from its flux value (fusion_kernel.py:394-434): the per-point form of the S1 loop of the
// resident kernel (same operations in the same order, so the two agree bit for bit).  Used to rebuild J_phi for the
// output from the iterate the last source update saw - J is never stored per iteration.
struct JrawK {
  double psi_ax, denom, inv_denom;
  bool hmode, same_prof;
  MtanhK mkp, mkf;
};
__device__ __forceinline__ double jraw_point(const JrawK &K, double v, double r, double cfv) {
  const double pn = ddiv_yf(dsub(v, K.psi_ax), K.denom, K.inv_denom);
  double pr = 0.0, ff = 0.0;
  if (pn >= 0.0 && pn < 1.0) {
    if (K.hmode) {
      pr = mtanh_res(pn, K.mkp);
      ff = K.same_prof ? pr : mtanh_res(pn, K.mkf);
    } else {
      pr = ff = dsub(1.0, pn);
    }
  }
  return dadd(dmul(0.5, dmul(r, pr)), dmul(0.5, dmul(cfv, ff)));
}

// block-wide broadcast of a value computed by thread 0 (through the scratch area)
__device__ __forceinline__ double bcast_d(double v, int slot_off) {
  __syncthreads();
  if (threadIdx.x == 0) res_pool[slot_off] = v;
  __syncthreads();
  return res_pool[slot_off];
}

__global__ void __launch_bounds__(kResThreads, 1)
k_picard_resident(const __grid_constant__ RPlan plan, const __grid_constant__ PicardResArgs a) {
  const int lev_off = res_stage(plan);
  int nz, nr, hw, xo, f_lk, f_nch, f_rpc, f_nk;
  ResK rk;
  {
    const RLevel &F = res_level(lev_off, 0);
    nz = F.nz, nr = F.nr, hw = F.hw, xo = F.x_off, f_lk = F.lk, f_nch = F.nch, f_rpc = F.rpc, f_nk = F.nk;
    rk = res_load_resk(F.g);
  }
  const double *tab_ae = plan.lev[0].g.a_e;  // a_e | a_w (global)
  const double *tab_rs = plan.lev[0].g.r_safe, *tab_irs = plan.lev[0].g.inv_r_safe;
  const double a_ns0 = plan.lev[0].g.a_ns, a_c0 = plan.lev[0].g.a_c, inv_a_c0 = plan.lev[0].g.inv_a_c;
  const int n = nz * nr, ps = nz * hw, planes = 2 * ps, nslot = ps;
  const int tid = threadIdx.x, T = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  const int step_z = T / hw, step_k = T - step_z * hw;
  const int iz_first = tid / hw, k_first = tid - iz_first * hw;
  double *sh = res_pool + a.scratch_off;            // 32 doubles reduction scratch
  int *shi = reinterpret_cast<int *>(sh + 32);       // 32 ints (16 doubles)
  const int bslot = a.scratch_off + 48;              // broadcast slots
  double *wpsi = a.ws_psi + (size_t)blockIdx.x * 3 * planes;
  double *wsrc = a.ws_src + (size_t)blockIdx.x * planes;
  const double n_all = (double)n, n_int = (double)(nz - 2) * (double)(nr - 2);
  const bool odd_nr = (nr & 1) != 0;  // then slot k = hw-1 holds only the (even) wall column

// slot loop: e = tid, tid+T, ... ; (iz, k) tracked incrementally; pa/pb = plane offsets (without the
// pool base) of the even / odd column of the slot; has_odd = the odd column exists
#define GSB_SLOT_LOOP_BEGIN()                                                  \
  for (int e = tid, iz = iz_first, k = k_first; e < nslot; e += T) {          \
    const int par_ = iz & 1;                                                   \
    const int pa = par_ * ps + e, pb = (1 - par_) * ps + e;                    \
    const bool has_odd = odd_nr ? (k < hw - 1) : true;
#define GSB_SLOT_LOOP_END()                                                    \
    k += step_k;                                                               \
    iz += step_z;                                                              \
    if (k >= hw) {                                                             \
      k -= hw;                                                                 \
      ++iz;                                                                    \
    }                                                                          \
  }

  // static striding (a dynamic work queue was measured 10-25 % SLOWER: see profiles/r1_v5_summary.md)
  const int n_work = a.order ? min(*a.n_order, a.batch) : a.batch;
  for (int wi = blockIdx.x; wi < n_work; wi += gridDim.x) {
    const int b = a.order ? a.order[wi] : wi;
    const double *bc = a.bc + (size_t)b * n;
    const double ipb = a.ip[b];
    double pp[4], pf[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      pp[i] = a.prof_dev ? a.prof_dev[(size_t)b * 8 + i] : a.prof.p[i];
      pf[i] = a.prof_dev ? a.prof_dev[(size_t)b * 8 + 4 + i] : a.prof.f[i];
    }
    const MtanhK mkp = mtanh_k(pp), mkf = mtanh_k(pf);
    const bool same_prof = pp[0] == pf[0] && pp[1] == pf[1] && pp[2] == pf[2] && pp[3] == pf[3];
    // ---- initial flux -> planes; pre-seed copy is the initial "best" state (newton_solver.py:484)
    __syncthreads();
    res_load_dense(a.psi + (size_t)b * n, xo, nz, nr, hw);
    int cur = 0, best = 0, nxt = 1;
    const bool do_seed = a.seed && fabs(ipb) >= 1e-12;
    const double seed_sc = a.seed_sum_drdz > 0.0 ? __ddiv_rn(ipb, a.seed_sum_drdz) : 1.0;
    __syncthreads();
    if (a.seed) {
      for (int i = tid; i < planes; i += T) wpsi[2 * planes + i] = res_pool[xo + i];
      best = 2;
    }

    // ---- seed: Gaussian source scaled to Ip, 50 sanitised/clipped Jacobi steps (iterative_solver.py:384-410)
    if (do_seed) {
      const double sc = seed_sc;
      for (int iz = warp; iz < nz; iz += nw)
        for (int ir = lane; ir < nr; ir += 32) {
          const double j = dmul(a.seedJ[iz * nr + ir], sc);
          wsrc[split_index(nz, hw, iz, ir)] = dmul(a.mr[ir], j);
        }
      __syncthreads();
      int p0 = xo, p1 = xo + ps, pt = a.tplane_off;  // colour-0 plane, colour-1 plane, spare
      for (int step = 0; step < 50; ++step) {
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          // new colour-c values from the OLD other colour; colour 0 goes to the spare plane,
          // colour 1 is then updated in place from the old colour-0 plane
          const int src_plane = c == 0 ? p0 : p1;
          const int oth_plane = c == 0 ? p1 : p0;
          const int dst_plane = c == 0 ? pt : p1;
          // slot walk (e = iz*hw + k over all 512 threads: every trip but the last is full; a warp-per-row loop
          // leaves 31 of 32 lanes idle in the third trip of a 65-slot row), four slots per batch so that the four
          // right-hand-side loads (L2) are in flight before the first use
          int o = tid, iz = iz_first, k = k_first;
          while (o < nslot) {
            int vo[4], vz[4], vk[4];
            double vf[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              vo[u] = o, vz[u] = iz, vk[u] = k;
              const int s = (c + iz) & 1;
              const int ir = 2 * k + s;
              const bool interior = o < nslot && ir < nr && iz > 0 && iz < nz - 1 && ir > 0 && ir < nr - 1;
              vf[u] = interior ? __ldcg(wsrc + c * ps + o) : 0.0;
              o += T, k += step_k, iz += step_z;
              if (k >= hw) k -= hw, ++iz;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int oo = vo[u], zz = vz[u];
              const int s = (c + zz) & 1;
              const int ir = 2 * vk[u] + s;
              if (oo < nslot && ir < nr) {
                double v;
                if (zz == 0 || zz == nz - 1 || ir == 0 || ir == nr - 1) {
                  v = sanitize_fast(res_pool[src_plane + oo]);
                } else {
                  const double cc = sanitize_fast(res_pool[oth_plane + oo]);
                  const double side = sanitize_fast(res_pool[oth_plane + oo - 1 + 2 * s]);
                  const double S = sanitize_fast(res_pool[oth_plane + oo - hw]), N = sanitize_fast(res_pool[oth_plane + oo + hw]);
                  const double f = sanitize_fast(vf[u]);
                  double acc = dadd(dmul(__ldg(tab_ae + ir), s ? side : cc), dmul(__ldg(tab_ae + nr + ir), s ? cc : side));
                  acc = dadd(acc, dmul(a_ns0, S));
                  acc = dadd(acc, dmul(a_ns0, N));
                  acc = dsub(acc, f);
                  v = clip_cap(ddiv_y(acc, a_c0, inv_a_c0));
                }
                res_pool[dst_plane + oo] = v;
              }
            }
          }
          __syncthreads();
        }
        const int t = p0;  // the spare plane now holds colour 0
        p0 = pt;
        pt = t;
      }
      // 50 swaps: colour 0 is back in its home plane
    }
    if (a.external && !do_seed) {  // no seed ran: the loop's source is identically zero (J_phi = 0)
      for (int i = tid; i < planes; i += T) wsrc[i] = 0.0;
    }
    // current iterate -> workspace slot `cur`
    __syncthreads();
    for (int i = tid; i < planes; i += T) wpsi[(size_t)cur * planes + i] = res_pool[xo + i];
    __syncthreads();

    int status = 0, iters = 0;
    // J_phi is rebuilt for the output from (iterate slot, axis/boundary flux, scale) of the LAST source update
    int j_slot = -1;
    bool j_ok = false;
    double diff_best = 1e9, gs_best = INFINITY, gs_last = INFINITY, diff_last = 0.0, scale = 0.0;
    double psi_ax = 0.0, psi_b = 0.0, t_izax = 0, t_irax = 0, t_izx = 0, t_irx = 0, t_found = 0;

    for (int kit = 0; kit < a.max_iter; ++kit) {
      GSB_PHASE_BEGIN();
      // ---- T: topology on the resident planes (a10, a11)
      ValIdx mx{0.0, -1}, mb{0.0, -1};
      double mn = INFINITY;
      GSB_SLOT_LOOP_BEGIN()
        const int flat = iz * nr + 2 * k;
        const double ve = res_pool[xo + pa];
        const double vo = has_odd ? res_pool[xo + pb] : ve;
        // a thread visits flat indices in increasing order, so a strict > keeps the first maximum
        if (ve > mx.v || mx.i < 0) mx = ValIdx{ve, flat};
        mn = fmin(mn, ve);
        if (has_odd) {
          if (vo > mx.v) mx = ValIdx{vo, flat + 1};
          mn = fmin(mn, vo);
        }
        if (__ldg(a.rowmask + iz) != 0) {
          const bool z_lo = iz == 0, z_hi = iz == nz - 1;
          // even column 2k: vertical neighbours and the odd columns either side live in plane pb
          {
            const double up = z_hi ? 0.0 : res_pool[xo + pb + hw], down = z_lo ? 0.0 : res_pool[xo + pb - hw];
            const double left = k > 0 ? res_pool[xo + pb - 1] : 0.0;
            const double bm = grad_mag(a.gg, ve, up, down, left, vo, z_lo, z_hi, k == 0, !has_odd);
            if (isfinite(bm)) mb = better<false>(mb, ValIdx{bm, flat});
          }
          if (has_odd) {  // odd column 2k+1: neighbours in plane pa
            const bool r_hi = 2 * k + 1 == nr - 1;
            const double up = z_hi ? 0.0 : res_pool[xo + pa + hw], down = z_lo ? 0.0 : res_pool[xo + pa - hw];
            const double right = r_hi ? 0.0 : res_pool[xo + pa + 1];
            const double bm = grad_mag(a.gg, vo, up, down, ve, right, z_lo, z_hi, false, r_hi);
            if (isfinite(bm)) mb = better<false>(mb, ValIdx{bm, flat + 1});
          }
        }
      GSB_SLOT_LOOP_END()
      mx = block_arg<true>(mx, sh, shi);
      __syncthreads();
      mb = block_arg<false>(mb, sh, shi);
      __syncthreads();
      mn = -block_max(-mn, sh);
      int xi = mb.i;  // valid in thread 0
      if (a.saddle) {
        // fusion_kernel.py:295-337: up to 16 smallest masked |grad psi|, keep Hessian saddles
        double prev_v = -1.0, best_v = INFINITY;
        int prev_i = -1, best_i = -1;
        for (int round = 0; round < 16; ++round) {
          ValIdx c{0.0, -1};
          for (int iz = warp; iz < nz; iz += nw) {
            if (!a.rowmask[iz]) continue;
            for (int ir = lane; ir < nr; ir += 32) {
              const int flat = iz * nr + ir;
              double gz, gr;
              grad_planes(xo, nz, nr, hw, iz, ir, a.gg, gz, gr);
              const double bm = hypot_glibc(gr, gz);
              if (!isfinite(bm)) continue;
              if (bm < prev_v || (bm == prev_v && flat <= prev_i)) continue;
              c = better<false>(c, ValIdx{bm, flat});
            }
          }
          __syncthreads();
          c = block_arg<false>(c, sh, shi);
          // broadcast the pick
          if (threadIdx.x == 0) {
            res_pool[bslot] = c.v;
            res_pool[bslot + 1] = (double)c.i;
          }
          __syncthreads();
          prev_v = res_pool[bslot];
          prev_i = (int)res_pool[bslot + 1];
          __syncthreads();
          if (prev_i < 0) break;
          const int iz = prev_i / nr, ir = prev_i - iz * nr;
          if (iz > 0 && iz < nz - 1 && ir > 0 && ir < nr - 1) {
            const double q0 = pl(xo, nz, hw, iz, ir), c2 = dmul(2.0, q0);
            const double d2r = __ddiv_rn(dadd(dsub(pl(xo, nz, hw, iz, ir + 1), c2), pl(xo, nz, hw, iz, ir - 1)), a.dr2);
            const double d2z = __ddiv_rn(dadd(dsub(pl(xo, nz, hw, iz + 1, ir), c2), pl(xo, nz, hw, iz - 1, ir)), a.dz2);
            const double drz = __ddiv_rn(dadd(dsub(dsub(pl(xo, nz, hw, iz + 1, ir + 1), pl(xo, nz, hw, iz + 1, ir - 1)),
                                                   pl(xo, nz, hw, iz - 1, ir + 1)),
                                              pl(xo, nz, hw, iz - 1, ir - 1)),
                                         a.four_drdz);
            const double det = dsub(dmul(d2r, d2z), dmul(drz, drz));
            if (isfinite(det) && det < 0.0 && prev_v < best_v) {
              best_v = prev_v;
              best_i = prev_i;
            }
          }
        }
        if (best_i >= 0) xi = best_i;
      }
      // ---- TF: psi_axis / psi_boundary (thread 0), broadcast
      if (threadIdx.x == 0) {
        double pax = mx.v;
        if (fabs(pax) < 1e-6) pax = 1e-6;
        double px;
        double fx = 0.0, izx = 0.0, irx = 0.0;
        if (xi >= 0) {
          const int iz = xi / nr, ir = xi - iz * nr;
          px = pl(xo, nz, hw, iz, ir);
          fx = 1.0;
          izx = iz;
          irx = ir;
        } else {
          px = mn;
        }
        double pb = px;
        if (fabs(dsub(pax, pb)) < 0.1) pb = dmul(pax, 0.1);
        res_pool[bslot] = pax;
        res_pool[bslot + 1] = pb;
        res_pool[bslot + 2] = (double)(mx.i / nr);
        res_pool[bslot + 3] = (double)(mx.i % nr);
        res_pool[bslot + 4] = izx;
        res_pool[bslot + 5] = irx;
        res_pool[bslot + 6] = fx;
      }
      __syncthreads();
      psi_ax = res_pool[bslot];
      psi_b = res_pool[bslot + 1];
      t_izax = res_pool[bslot + 2];
      t_irax = res_pool[bslot + 3];
      t_izx = res_pool[bslot + 4];
      t_irx = res_pool[bslot + 5];
      t_found = res_pool[bslot + 6];
      __syncthreads();
      GSB_PHASE(48);  // topology

      if (!a.external) {  // external_profile_mode keeps the seed's J_phi / source (newton_solver.py:509)
      // ---- S1: J_raw(psi) + deterministic block sum (a12)
      double denom = dsub(psi_b, psi_ax);
      if (fabs(denom) < 1e-9) denom = 1e-9;
      const double inv_denom = __ddiv_rn(1.0, denom);
      const bool hmode = a.prof.hmode != 0;
      j_slot = cur;  // the planes hold a copy of wpsi[cur]
      double acc = 0.0;
      GSB_SLOT_LOOP_BEGIN()
        const double pn_e = ddiv_yf(dsub(res_pool[xo + pa], psi_ax), denom, inv_denom);
        const double pn_o = has_odd ? ddiv_yf(dsub(res_pool[xo + pb], psi_ax), denom, inv_denom) : -1.0;
        const bool in_e = pn_e >= 0.0 && pn_e < 1.0, in_o = pn_o >= 0.0 && pn_o < 1.0;
        double pr_e = 0.0, ff_e = 0.0, pr_o = 0.0, ff_o = 0.0;
        if (in_e || in_o) {
          // both points in straight-line code (two independent chains); out-of-plasma results are discarded
          if (hmode) {
            const double te = mtanh_res(pn_e, mkp), to = mtanh_res(pn_o, mkp);
            double fe = te, fo = to;
            if (!same_prof) {
              fe = mtanh_res(pn_e, mkf);
              fo = mtanh_res(pn_o, mkf);
            }
            pr_e = in_e ? te : 0.0, ff_e = in_e ? fe : 0.0;
            pr_o = in_o ? to : 0.0, ff_o = in_o ? fo : 0.0;
          } else {
            pr_e = ff_e = in_e ? dsub(1.0, pn_e) : 0.0;
            pr_o = ff_o = in_o ? dsub(1.0, pn_o) : 0.0;
          }
        }
        // J_raw = 0.5*(R*p) + 0.5*((1/(mu0 R))*ff)      (fusion_kernel.py:430-434)
        const double je = dadd(dmul(0.5, dmul(__ldg(a.rrow + 2 * k), pr_e)), dmul(0.5, dmul(__ldg(a.cf + 2 * k), ff_e)));
        __stcg(wsrc + pa, je);  // J_raw parks in the right-hand-side plane until S2 rescales it in place
        acc += je;
        if (has_odd) {
          const double jo = dadd(dmul(0.5, dmul(__ldg(a.rrow + 2 * k + 1), pr_o)), dmul(0.5, dmul(__ldg(a.cf + 2 * k + 1), ff_o)));
          __stcg(wsrc + pb, jo);
          acc += jo;
        }
      GSB_SLOT_LOOP_END()
      acc = block_sum(acc, sh);
      const double jsum = bcast_d(acc, bslot + 8);
      // ---- S2: J = J_raw * Ip/I ; Source = (-mu0 R) J   (split layout)
      const double icur = dmul(dmul(jsum, a.dr), a.dz);
      const bool ok = fabs(icur) > 1e-9;
      scale = ok ? __ddiv_rn(ipb, icur) : 0.0;
      j_ok = ok;
      {  // batches of four slots: all loads of a batch are in flight before the first use
        int e = tid, iz = iz_first, k = k_first;
        while (e < nslot) {
          double vje[4], vjo[4];
          int vpa[4], vpb[4], vk[4];
          bool vok[4], vho[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int par_ = iz & 1;
            vok[u] = e < nslot;
            vpa[u] = par_ * ps + e, vpb[u] = (1 - par_) * ps + e, vk[u] = k;
            vho[u] = odd_nr ? (k < hw - 1) : true;
            vje[u] = vok[u] ? __ldcg(wsrc + vpa[u]) : 0.0;
            vjo[u] = (vok[u] && vho[u]) ? __ldcg(wsrc + vpb[u]) : 0.0;
            e += T, k += step_k, iz += step_z;
            if (k >= hw) k -= hw, ++iz;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (vok[u]) {
              const double je = ok ? dmul(vje[u], scale) : 0.0;
              __stcg(wsrc + vpa[u], dmul(__ldg(a.mr + 2 * vk[u]), je));
              if (vho[u]) {
                const double jo = ok ? dmul(vjo[u], scale) : 0.0;
                __stcg(wsrc + vpb[u], dmul(__ldg(a.mr + 2 * vk[u] + 1), jo));
              }
            }
          }
        }
      }
      }  // !external
      __syncthreads();
      GSB_PHASE(49);  // source

      // ---- E: one V-cycle on the planes (they hold a copy of the current iterate)
      res_vcycle(lev_off, plan.nlev, wsrc, a.omega, 3, 3);
      __syncthreads();
      GSB_PHASE(50);  // V-cycle

      // ---- R: wall BC, NaN flag, mean|dpsi|, under-relaxation (in place)
      const double *old = wpsi + (size_t)cur * planes;
      double *out = wpsi + (size_t)nxt * planes;
      double dsum = 0.0;
      int bad = 0;
      {  // batches of four slots (see S2)
        int e = tid, iz = iz_first, k = k_first;
        while (e < nslot) {
          double voe[4], voo[4];
          int vpa[4], vpb[4], vk[4], vz[4];
          bool vok[4], vho[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int par_ = iz & 1;
            vok[u] = e < nslot;
            vpa[u] = par_ * ps + e, vpb[u] = (1 - par_) * ps + e, vk[u] = k, vz[u] = iz;
            vho[u] = odd_nr ? (k < hw - 1) : true;
            voe[u] = vok[u] ? __ldcg(old + vpa[u]) : 0.0;
            voo[u] = (vok[u] && vho[u]) ? __ldcg(old + vpb[u]) : 0.0;
            e += T, k += step_k, iz += step_z;
            if (k >= hw) k -= hw, ++iz;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (vok[u]) {
              const bool zwall = vz[u] == 0 || vz[u] == nz - 1;
              {
                const bool wall = zwall || vk[u] == 0 || !vho[u];  // column 0, or the lone even wall column nr-1
                const double wn = wall ? bc[vz[u] * nr + 2 * vk[u]] : res_pool[xo + vpa[u]];
                const double ov = voe[u];
                if (!(fabs(wn) <= 1.79769313486231570815e308)) bad = 1;  // NaN or +-inf
                dsum += fabs(dsub(wn, ov));
                const double c = dadd(dmul(a.oma, ov), dmul(a.alpha, wn));
                res_pool[xo + vpa[u]] = c;
                __stcg(out + vpa[u], c);
              }
              if (vho[u]) {
                const bool wall = zwall || (2 * vk[u] + 1 == nr - 1);
                const double wn = wall ? bc[vz[u] * nr + 2 * vk[u] + 1] : res_pool[xo + vpb[u]];
                const double ov = voo[u];
                if (!(fabs(wn) <= 1.79769313486231570815e308)) bad = 1;
                dsum += fabs(dsub(wn, ov));
                const double c = dadd(dmul(a.oma, ov), dmul(a.alpha, wn));
                res_pool[xo + vpb[u]] = c;
                __stcg(out + vpb[u], c);
              }
            }
          }
        }
      }
      const int anybad = __syncthreads_or(bad);
      GSB_PHASE(51);  // relax + diff
      // ---- G: GS residual of the relaxed iterate (compute_gs_residual_rms): thread <-> (k slot,
      // row chunk) of level 0, both columns of the slot, register window sliding down the rows
      double rmax = 0.0, rsq = 0.0;
      {
        const int k = tid & ((1 << f_lk) - 1), ch = tid >> f_lk;
        const int z0 = 1 + ch * f_rpc;
        const int z1 = min(z0 + f_rpc, nz - 1);
        if (ch < f_nch && k < f_nk && z0 < z1) {
          const int ce = 2 * k, co = 2 * k + 1;
          const bool e_in = ce >= 1 && ce <= nr - 2, o_in = co <= nr - 2;
          const double rs_e = __ldg(tab_rs + ce), irs_e = __ldg(tab_irs + ce);
          const double rs_o = o_in ? __ldg(tab_rs + co) : 1.0, irs_o = o_in ? __ldg(tab_irs + co) : 1.0;
          int e = z0 * hw + k;
          int par = z0 & 1;
          double ev_m = res_pool[xo + (1 - par) * ps + e - hw], od_m = res_pool[xo + par * ps + e - hw];
          double ev_0 = res_pool[xo + par * ps + e], od_0 = res_pool[xo + (1 - par) * ps + e];
          for (int iz = z0; iz < z1; ++iz) {
            const int pa = par * ps + e, pb = (1 - par) * ps + e;
            // row iz+1: the even column sits in plane 1-par, the odd column in plane par
            const double ev_p = res_pool[xo + pb + hw], od_p = res_pool[xo + pa + hw];
            if (e_in) {
              const double w = res_pool[xo + pb - 1];
              const double r = dsub(res_lx(rk, rs_e, irs_e, ev_0, od_0, w, ev_m, ev_p), __ldcg(wsrc + pa));
              rmax = fmax(rmax, fabs(r));
              rsq += r * r;
            }
            if (o_in) {
              const double ee = res_pool[xo + pa + 1];
              const double r = dsub(res_lx(rk, rs_o, irs_o, od_0, ee, ev_0, od_m, od_p), __ldcg(wsrc + pb));
              rmax = fmax(rmax, fabs(r));
              rsq += r * r;
            }
            ev_m = ev_0, ev_0 = ev_p;
            od_m = od_0, od_0 = od_p;
            e += hw;
            par ^= 1;
          }
        }
      }
      dsum = block_sum(dsum, sh);
      __syncthreads();
      rmax = block_max(rmax, sh);
      __syncthreads();
      rsq = block_sum(rsq, sh);
      // ---- D: decide (thread 0), broadcast
      if (threadIdx.x == 0) {
        double code = 0.0;  // 0 continue, 1 converged, 2 max-iter, 3 diverged
        double dbest = diff_best, gbest = gs_best, dl = diff_last, gl = gs_last;
        double improved = 0.0;
        if (anybad) {
          code = 3.0;
        } else {
          const double diff = dsum / n_all;
          const double gs = (rmax > 0.0 && n_int > 0.0) ? sqrt(rsq / n_int) : 0.0;
          if (a.hist) a.hist[(size_t)b * a.max_iter + kit] = diff;
          if (a.gs_hist) a.gs_hist[(size_t)b * a.max_iter + kit] = gs;
          dl = diff;
          gl = gs;
          if (gs < gbest) gbest = gs;
          if (diff < dbest) {
            dbest = diff;
            improved = 1.0;
          }
          if (diff < a.tol && (!a.need_gs || gs < a.gs_tol))
            code = 1.0;
          else if (kit + 1 >= a.max_iter)
            code = 2.0;
        }
        res_pool[bslot] = code;
        res_pool[bslot + 1] = dbest;
        res_pool[bslot + 2] = gbest;
        res_pool[bslot + 3] = dl;
        res_pool[bslot + 4] = gl;
        res_pool[bslot + 5] = improved;
      }
      __syncthreads();
      const int code = (int)res_pool[bslot];
      diff_best = res_pool[bslot + 1];
      gs_best = res_pool[bslot + 2];
      diff_last = res_pool[bslot + 3];
      gs_last = res_pool[bslot + 4];
      const bool improved = res_pool[bslot + 5] != 0.0;
      __syncthreads();
      iters = kit + 1;
      GSB_PHASE(52);  // GS residual + decide
      if (blockIdx.x == 0 && threadIdx.x == 0) GSB_PHASE_COUNT(53);
      if (code == 3) {  // revert to the best state (newton_solver.py:518-532)
        status = 3;
        cur = best;
        break;
      }
      const int newcur = nxt;
      if (improved) best = newcur;
      cur = newcur;
      // next slot: the lowest one that holds neither the current nor the best iterate (while every
      // iteration improves, best == cur and the solve ping-pongs between two slots only: the third
      // stays out of the L2 working set)
      nxt = (cur == best) ? (cur == 0 ? 1 : 0) : 3 - cur - best;
      if (code != 0) {
        status = code;
        break;
      }
    }

    // ---- results: colour-split workspace -> dense outputs
    {
      const double *fin = wpsi + (size_t)cur * planes;
      const double *jsrc = wpsi + (size_t)(j_slot >= 0 ? j_slot : 0) * planes;
      JrawK jk;  // psi_ax / psi_b still hold the values the last source update used
      jk.psi_ax = psi_ax;
      jk.denom = dsub(psi_b, psi_ax);
      if (fabs(jk.denom) < 1e-9) jk.denom = 1e-9;
      jk.inv_denom = __ddiv_rn(1.0, jk.denom);
      jk.hmode = a.prof.hmode != 0, jk.same_prof = same_prof, jk.mkp = mkp, jk.mkf = mkf;
      double *po = a.psi + (size_t)b * n;
      double *jo = a.jphi + (size_t)b * n;
      for (int iz = warp; iz < nz; iz += nw)
        for (int ir = lane; ir < nr; ir += 32) {
          const int o = split_index(nz, hw, iz, ir);
          po[iz * nr + ir] = fin[o];
          double j;
          if (j_slot >= 0)  // J_raw(psi of the last source update) * Ip/I, exactly as S1 / S2 formed it
            j = j_ok ? dmul(jraw_point(jk, __ldcg(jsrc + o), __ldg(a.rrow + ir), __ldg(a.cf + ir)), scale) : 0.0;
          else              // no source update ran (external_profile_mode): the seed's J_phi, or zero without a seed
            j = do_seed ? dmul(a.seedJ[iz * nr + ir], seed_sc) : 0.0;
          jo[iz * nr + ir] = j;
        }
      if (threadIdx.x == 0 && a.summary) {
        double *o = a.summary + (size_t)b * 16;
        o[0] = (double)iters;
        o[1] = status == 1 ? 1.0 : 0.0;
        o[2] = diff_best;
        o[3] = gs_last;
        o[4] = gs_best;
        o[5] = (double)status;
        o[6] = psi_ax;
        o[7] = psi_b;
        o[8] = t_izax;
        o[9] = t_irax;
        o[10] = t_izx;
        o[11] = t_irx;
        o[12] = diff_last;
        o[13] = t_found;
        o[14] = scale;
        o[15] = 0.0;
      }
    }
    __syncthreads();
  }
#undef GSB_SLOT_LOOP_BEGIN
#undef GSB_SLOT_LOOP_END
}

// ---------------------------------------------------------------------------- free-boundary outer loop
// fb_summary rows: [outer_iterations, final_diff, inner Picard iterations summed over the outer iterations, converged]
__global__ void k_fb_init(int *__restrict__ mask, int *__restrict__ order, int *__restrict__ n_order,
                          double *__restrict__ fbsum, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) *n_order = batch;
  if (b >= batch) return;
  mask[b] = 1;
  order[b] = b;
  fbsum[4 * b] = 0.0;
  fbsum[4 * b + 1] = INFINITY;
  fbsum[4 * b + 2] = 0.0;
  fbsum[4 * b + 3] = 0.0;
}

// index of wall point (iz, ir) in the C-order ring enumeration of wall_coord() (gsb_green.cu)
__device__ __forceinline__ int wall_index(int nz, int nr, int iz, int ir) {
  if (iz == 0) return ir;
  if (iz == nz - 1) return nr + 2 * (nz - 2) + ir;
  return nr + 2 * (iz - 1) + (ir ? 1 : 0);
}

// wall ring of psi <- ext ring (+ plasma wall flux); old <- psi
__global__ void __launch_bounds__(256)
k_fb_prepare(double *__restrict__ psi, const double *__restrict__ ext, const double *__restrict__ wall,
             double *__restrict__ old, size_t n, int nz, int nr, int nwall, const int *__restrict__ mask) {
  const int b = blockIdx.y;
  if (!mask[b]) return;
  double *f = psi + (size_t)b * n;
  const double *e = ext + (size_t)b * n;
  double *o = old + (size_t)b * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int iz = (int)(i / nr), ir = (int)(i - (size_t)iz * nr);
    double v = f[i];
    if (iz == 0 || ir == 0 || iz == nz - 1 || ir == nr - 1) {
      v = e[i];
      if (wall) v = dadd(v, wall[(size_t)b * nwall + wall_index(nz, nr, iz, ir)]);
      f[i] = v;
    }
    o[i] = v;
  }
}

// partial max |psi - old| (NaN wins like np.max)
__global__ void __launch_bounds__(256)
k_fb_diff(const double *__restrict__ psi, const double *__restrict__ old, size_t n, double *__restrict__ part,
          const int *__restrict__ mask) {
  __shared__ double sh[32];
  const int b = blockIdx.y, P = gridDim.x, p = blockIdx.x;
  if (!mask[b]) return;
  const size_t i0 = n * p / P, i1 = n * (p + 1) / P;
  const double *f = psi + (size_t)b * n, *o = old + (size_t)b * n;
  double m = 0.0;
  int bad = 0;
  for (size_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
    const double d = fabs(dsub(f[i], o[i]));
    if (d != d) bad = 1;
    m = fmax(m, d);
  }
  const int anybad = __syncthreads_or(bad);
  m = block_max(m, sh);
  if (threadIdx.x == 0) {
    part[((size_t)b * kPT + p) * 2] = m;
    part[((size_t)b * kPT + p) * 2 + 1] = anybad ? 1.0 : 0.0;
  }
}

// One CTA: per-equilibrium outer-loop decision, then an ORDERED compaction of the still-active equilibria
// (deterministic work list -> deterministic CTA assignment in the next resident launch).
__global__ void __launch_bounds__(1024)
k_fb_decide(const double *__restrict__ part, int P, double tol, int outer, const double *__restrict__ summary,
            double *__restrict__ fbsum, int *__restrict__ mask, int *__restrict__ order, int *__restrict__ n_order,
            int batch) {
  __shared__ int wsum[32];
  __shared__ int base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int b0 = 0; b0 < batch; b0 += blockDim.x) {
    const int b = b0 + tid;
    int keep = 0;
    if (b < batch && mask[b]) {
      double m = 0.0;
      bool bad = false;
      for (int q = 0; q < P; ++q) {
        m = fmax(m, part[((size_t)b * kPT + q) * 2]);
        bad = bad || part[((size_t)b * kPT + q) * 2 + 1] != 0.0;
      }
      const double diff = bad ? NAN : m;
      fbsum[4 * b] = (double)(outer + 1);
      fbsum[4 * b + 1] = diff;
      fbsum[4 * b + 2] += summary[(size_t)b * 16];  // Picard iterations of this outer iteration
      const bool conv = diff < tol;
      fbsum[4 * b + 3] = conv ? 1.0 : 0.0;
      keep = conv ? 0 : 1;
      mask[b] = keep;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    const int pos_in_warp = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) wsum[warp] = __popc(bal);
    __syncthreads();
    int off = base;
    for (int w = 0; w < warp; ++w) off += wsum[w];
    if (keep) order[off + pos_in_warp] = b;
    __syncthreads();
    if (tid == 0) {
      int t = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += wsum[w];
      base += t;
    }
    __syncthreads();
  }
  if (tid == 0) *n_order = base;
}

}  // namespace gsb

using namespace gsb;

// numpy's pairwise summation for a contiguous float64 buffer (used for the seed integral)
static double np_pairwise_sum(const double *a, size_t n) {
  if (n < 8) {
    double r = 0.0;
    for (size_t i = 0; i < n; ++i) r += a[i];
    return r;
  }
  if (n <= 128) {
    volatile double r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    size_t i;
    for (i = 8; i < n - (n % 8); i += 8)
      for (int j = 0; j < 8; ++j) r[j] = r[j] + a[i + j];
    volatile double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res = res + a[i];
    return res;
  }
  size_t n2 = n / 2;
  n2 -= n2 % 8;
  volatile double s1 = np_pairwise_sum(a, n2);
  volatile double s2 = np_pairwise_sum(a + n2, n - n2);
  return s1 + s2;
}

static int picard_ws_ensure(gsb_ctx *ctx, const gsb_picard_params *p) {
  if (!ctx->picard) {
    auto *w = new gsb_picard_ws();
    ctx->picard = w;
    w->cap = ctx->batch_cap;
    const size_t N = ctx->n * (size_t)w->cap * sizeof(double);
    GSB_CUDA(cudaMalloc(&w->buf1, N));
    GSB_CUDA(cudaMalloc(&w->buf2, N));
    GSB_CUDA(cudaMalloc(&w->W, N));
    GSB_CUDA(cudaMalloc(&w->source, N));
    GSB_CUDA(cudaMalloc(&w->ring, (size_t)w->cap * ring_size(ctx->nz, ctx->nr) * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->tpart, (size_t)w->cap * kPT * kTW * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->spart, (size_t)w->cap * kPT * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->rpart, (size_t)w->cap * kPT * kRW * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->seedJ, ctx->n * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->cf, ctx->nr * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->mr, ctx->nr * sizeof(double)));
    GSB_CUDA(cudaMalloc(&w->rowmask, ctx->nz * sizeof(int)));
    GSB_CUDA(cudaMalloc(&w->mrows, ctx->nz * sizeof(int)));
    GSB_CUDA(cudaMalloc(&w->ints, (size_t)w->cap * 8 * sizeof(int)));
    GSB_CUDA(cudaMalloc(&w->dbls, (size_t)w->cap * (5 + 2 + 8) * sizeof(double)));
    const size_t c = w->cap;
    PicardState &s = w->s;
    s.active = w->ints;
    s.status = w->ints + c;
    s.iter = w->ints + 2 * c;
    s.cur = w->ints + 3 * c;
    s.best = w->ints + 4 * c;
    s.nxt = w->ints + 5 * c;
    s.xsel = w->ints + 6 * c;
    s.seed_active = w->ints + 7 * c;
    s.diff_best = w->dbls;
    s.gs_best = w->dbls + c;
    s.gs_last = w->dbls + 2 * c;
    s.diff_last = w->dbls + 3 * c;
    s.scale = w->dbls + 4 * c;
    s.axbnd = w->dbls + 5 * c;
    s.topo = w->dbls + 7 * c;
  }
  gsb_picard_ws *w = ctx->picard;
  const bool same = (w->mu0 == p->mu0) && (w->z_min == p->z_min) && (w->r_min == p->r_min) && (w->r_max == p->r_max);
  if (!same) {
    const int nz = ctx->nz, nr = ctx->nr;
    GSB_REQUIRE((int)ctx->z_axis.size() == nz, "gsb_picard_solve: context was created without a z axis");
    std::vector<double> cf(nr), mr(nr), seed(ctx->n);
    std::vector<int> mask(nz);
    for (int j = 0; j < nr; ++j) {
      volatile double m = p->mu0 * ctx->r_row[j];
      cf[j] = 1.0 / m;                    // 1.0 / (mu0 * RR)
      volatile double nm = -p->mu0;
      mr[j] = nm * ctx->r_row[j];         // (-mu0) * RR
    }
    volatile double half_zmin = p->z_min * 0.5;
    for (int i = 0; i < nz; ++i) mask[i] = (half_zmin > ctx->z_axis[i]) ? 1 : 0;
    volatile double rc = (p->r_min + p->r_max) / 2.0;
    for (int i = 0; i < nz; ++i)
      for (int j = 0; j < nr; ++j) {
        volatile double a = ctx->r_row[j] - rc;
        volatile double a2 = a * a;
        volatile double z2 = ctx->z_axis[i] * ctx->z_axis[i];
        volatile double d = a2 + z2;
        volatile double arg = -d;
        volatile double arg2 = arg / 2.0;
        seed[(size_t)i * nr + j] = std::exp(arg2);
      }
    w->seed_sum = np_pairwise_sum(seed.data(), seed.size());
    GSB_CUDA(cudaMemcpy(w->cf, cf.data(), nr * sizeof(double), cudaMemcpyHostToDevice));
    GSB_CUDA(cudaMemcpy(w->mr, mr.data(), nr * sizeof(double), cudaMemcpyHostToDevice));
    GSB_CUDA(cudaMemcpy(w->rowmask, mask.data(), nz * sizeof(int), cudaMemcpyHostToDevice));
    {
      std::vector<int> rows;
      for (int i = 0; i < nz; ++i)
        if (mask[i]) rows.push_back(i);
      w->n_mrows = (int)rows.size();
      if (!rows.empty()) GSB_CUDA(cudaMemcpy(w->mrows, rows.data(), rows.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    GSB_CUDA(cudaMemcpy(w->seedJ, seed.data(), seed.size() * sizeof(double), cudaMemcpyHostToDevice));
    w->mu0 = p->mu0;
    w->z_min = p->z_min;
    w->r_min = p->r_min;
    w->r_max = p->r_max;
  }
  return GSB_OK;
}

static int partials_for(int nz, int nr) {
  long long pts = (long long)nz * nr;
  int P = (int)((pts + 4095) / 4096);
  if (P < 1) P = 1;
  if (P > 8) P = 8;  // the per-equilibrium final kernels (k_topo_final, k_source_scale) walk the partials serially
  if (P > nz) P = nz;
  return P;
}

static ProfileDev to_dev(const gsb_profile &q) {
  ProfileDev d;
  d.hmode = q.hmode;
  for (int i = 0; i < 4; ++i) {
    d.p[i] = q.ped_p[i];
    d.f[i] = q.ped_ff[i];
  }
  return d;
}

// X-point saddle filter for the streaming path: two-kernel candidate selection when the masked region
// fits kSadChunksMax chunks, the single-CTA kernel otherwise.
static int saddle_launch(gsb_ctx *ctx, Bufs bufs, const int *cur, int batch, const GradGeom &gg, double dr2,
                         double dz2, double four_drdz, int *xsel, const int *active, cudaStream_t st) {
  gsb_picard_ws *w = ctx->picard;
  const long long total = (long long)w->n_mrows * ctx->nr;
  const int nchunks = (int)((total + kSadChunk - 1) / kSadChunk);
  if (nchunks < 1 || nchunks > kSadChunksMax) {
    k_xpoint_saddle<<<batch, 256, 0, st>>>(bufs, cur, ctx->n, ctx->nz, ctx->nr, gg, dr2, dz2, four_drdz, w->rowmask, xsel, active);
    GSB_LAUNCH_CHECK();
    return GSB_OK;
  }
  if (!w->cand || w->cand_chunks < nchunks) {
    if (w->cand) cudaFree(w->cand);
    w->cand = nullptr;
    GSB_CUDA(cudaMalloc(&w->cand, (size_t)w->cap * nchunks * 32 * sizeof(double)));
    w->cand_chunks = nchunks;
  }
  k_saddle_cand<<<dim3(nchunks, batch), 256, 0, st>>>(bufs, cur, ctx->n, ctx->nz, ctx->nr, gg, w->mrows, w->n_mrows, nchunks, w->cand, active);
  GSB_LAUNCH_CHECK();
  k_saddle_pick<<<batch, 256, 0, st>>>(bufs, cur, ctx->n, ctx->nz, ctx->nr, dr2, dz2, four_drdz, nchunks, w->cand, xsel, active);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// Persistent resident solve (k_picard_resident).  Returns GSB_ESTATE (without setting an error) when
// one equilibrium's V-cycle hierarchy does not fit the shared memory of an SM.
namespace gsb {
int picard_phase_read(long long *out64, int reset) {
#ifdef GSB_PHASE_TIMING
  long long tmp[64];
  GSB_CUDA(cudaMemcpyFromSymbol(tmp, g_phase, sizeof(tmp)));
  if (out64)
    for (int i = 0; i < 64; ++i) out64[i] += tmp[i];
  if (reset) {
    long long z[64] = {0};
    GSB_CUDA(cudaMemcpyToSymbol(g_phase, z, sizeof(z)));
  }
#else
  (void)out64;
  (void)reset;
#endif
  return GSB_OK;
}
}  // namespace gsb

static int picard_resident_launch(gsb_ctx *ctx, const gsb_picard_params *p, double *psi_dev, const double *bc_dev,
                                  const double *ip_dev, const double *prof_dev, double *jphi_dev,
                                  double *summary_dev, double *hist_dev, double *gs_hist_dev, int batch,
                                  const int *order_dev, const int *n_order_dev, cudaStream_t st) {
  constexpr int kScratch = 96;
  RPlan plan;
  if (!build_rplan(ctx, 0, kScratch, &plan) || plan.nlev < 2) return GSB_ESTATE;
  const int nz = ctx->nz, nr = ctx->nr, hw = (nr + 1) / 2;
  // the Jacobi seed borrows the (then idle) planes of the first coarse level as its spare half plane
  const RLevel &c1 = plan.lev[1];
  if (4 * c1.nz * c1.hw < nz * hw) return GSB_ESTATE;
  gsb_picard_ws *w = ctx->picard;
  const size_t planes = (size_t)2 * nz * hw, per_cta = 4 * planes;  // three iterate slots + the right-hand side
  const int grid = std::min(batch, ctx->num_sms);
  if (w->res_grid < grid) {
    if (w->res_ws) cudaFree(w->res_ws);
    w->res_ws = nullptr;
    w->res_grid = 0;
    GSB_CUDA(cudaMalloc(&w->res_ws, (size_t)ctx->num_sms * per_cta * sizeof(double)));
    w->res_grid = ctx->num_sms;
  }
  PicardResArgs a{};
  a.psi = psi_dev;
  a.bc = bc_dev;
  a.ip = ip_dev;
  a.prof_dev = prof_dev;
  a.jphi = jphi_dev;
  a.summary = summary_dev;
  a.hist = hist_dev;
  a.gs_hist = gs_hist_dev;
  a.ws_psi = w->res_ws;
  a.ws_src = w->res_ws + (size_t)w->res_grid * 3 * planes;
  a.seedJ = w->seedJ;
  a.cf = w->cf;
  a.mr = w->mr;
  a.rrow = ctx->r_dev;
  a.rowmask = w->rowmask;
  {
    volatile double ssum = w->seed_sum * ctx->dr;
    volatile double ssum2 = ssum * ctx->dz;
    a.seed_sum_drdz = ssum2;
  }
  a.batch = batch;
  a.max_iter = p->max_iterations;
  a.seed = p->seed;
  a.saddle = p->saddle;
  a.need_gs = p->require_gs_residual;
  a.external = p->external_profile;
  a.tol = p->tol;
  a.gs_tol = p->gs_tol;
  a.alpha = p->alpha;
  a.oma = 1.0 - p->alpha;
  a.omega = p->omega;
  a.dr = ctx->dr;
  a.dz = ctx->dz;
  {
    volatile double dr2 = ctx->dr * ctx->dr, dz2 = ctx->dz * ctx->dz, f1 = 4.0 * ctx->dr, f2 = f1 * ctx->dz;
    a.dr2 = dr2;
    a.dz2 = dz2;
    a.four_drdz = f2;
  }
  a.gg = make_grad_geom(ctx->dz, ctx->dr);
  a.prof = to_dev(p->prof);
  a.scratch_off = plan.pool_doubles + res_stage_doubles(plan.nlev);
  a.tplane_off = c1.x_off;
  a.order = order_dev;
  a.n_order = n_order_dev;
  GSB_SMEM_OPT_IN(k_picard_resident, kResSmemMax);
  const size_t smem = (size_t)(a.scratch_off + kScratch) * sizeof(double);
  k_picard_resident<<<grid, kResThreads, smem, st>>>(plan, a);
  GSB_LAUNCH_CHECK();
  ctx->picard_last_iters = p->max_iterations;  // upper bound: the count lives in summary_dev
  return GSB_OK;
}

extern "C" {

void gsb_picard_ws_free(gsb_ctx *ctx) {
  gsb_picard_ws *w = ctx->picard;
  if (!w) return;
  void *ptrs[] = {w->buf1, w->buf2, w->W, w->source, w->ring, w->tpart, w->spart, w->rpart,
                  w->seedJ, w->cf, w->mr, w->rowmask, w->ints, w->dbls, w->res_ws, w->mrows, w->cand,
                  w->and_psi, w->and_res, w->and_part, w->and_alpha, w->and_fb};
  for (void *q : ptrs)
    if (q) cudaFree(q);
  delete w;
  ctx->picard = nullptr;
}

int gsb_topology(gsb_ctx *ctx, const double *psi_dev, int batch, double z_min, int saddle,
                 double *out_dev, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && out_dev, "gsb_topology: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_topology: batch outside [1, batch_cap]");
  GSB_CUDA(cudaSetDevice(ctx->device));
  gsb_picard_params p{};
  p.mu0 = 1.0;
  p.z_min = z_min;
  p.r_min = ctx->r_row.front();
  p.r_max = ctx->r_row.back();
  if (ctx->picard) {  // keep cached tables unless z_min changed
    p.mu0 = std::isnan(ctx->picard->mu0) ? 1.0 : ctx->picard->mu0;
    p.r_min = std::isnan(ctx->picard->r_min) ? p.r_min : ctx->picard->r_min;
    p.r_max = std::isnan(ctx->picard->r_max) ? p.r_max : ctx->picard->r_max;
  }
  int rc = picard_ws_ensure(ctx, &p);
  if (rc) return rc;
  gsb_picard_ws *w = ctx->picard;
  cudaStream_t st = (cudaStream_t)stream;
  Bufs bufs{{const_cast<double *>(psi_dev), nullptr, nullptr}};
  const int P = partials_for(ctx->nz, ctx->nr);
  const GradGeom gg = make_grad_geom(ctx->dz, ctx->dr);
  k_topo<<<dim3(P, batch), 256, 0, st>>>(bufs, nullptr, ctx->n, ctx->nz, ctx->nr, gg, w->rowmask, w->tpart, nullptr);
  GSB_LAUNCH_CHECK();
  if (saddle) {
    volatile double dr2 = ctx->dr * ctx->dr, dz2 = ctx->dz * ctx->dz, f1 = 4.0 * ctx->dr, f2 = f1 * ctx->dz;
    rc = saddle_launch(ctx, bufs, nullptr, batch, gg, dr2, dz2, f2, w->s.xsel, nullptr, st);
    if (rc) return rc;
  }
  k_topo_final<<<(batch + 127) / 128, 128, 0, st>>>(bufs, nullptr, ctx->n, ctx->nr, P, w->tpart,
                                                    saddle ? w->s.xsel : nullptr, out_dev, nullptr, 0, batch, nullptr);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_plasma_source(gsb_ctx *ctx, const double *psi_dev, const double *axis_bnd_dev,
                      const double *ip_dev, double mu0, const gsb_profile *prof,
                      const double *prof_dev, double *jphi_dev, int batch, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && axis_bnd_dev && ip_dev && prof && jphi_dev, "gsb_plasma_source: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_plasma_source: batch outside [1, batch_cap]");
  GSB_CUDA(cudaSetDevice(ctx->device));
  gsb_picard_params p{};
  p.mu0 = mu0;
  p.z_min = ctx->z_axis.empty() ? 0.0 : ctx->z_axis.front();
  p.r_min = ctx->r_row.front();
  p.r_max = ctx->r_row.back();
  if (ctx->picard && !std::isnan(ctx->picard->z_min)) {
    p.z_min = ctx->picard->z_min;
    p.r_min = ctx->picard->r_min;
    p.r_max = ctx->picard->r_max;
  }
  int rc = picard_ws_ensure(ctx, &p);
  if (rc) return rc;
  gsb_picard_ws *w = ctx->picard;
  cudaStream_t st = (cudaStream_t)stream;
  Bufs bufs{{const_cast<double *>(psi_dev), nullptr, nullptr}};
  const int P = partials_for(ctx->nz, ctx->nr);
  k_source_raw<<<dim3(P, batch), 256, 0, st>>>(bufs, nullptr, ctx->n, ctx->nz, ctx->nr, axis_bnd_dev, to_dev(*prof),
                                               prof_dev, ctx->r_dev, w->cf, jphi_dev, w->spart, nullptr);
  GSB_LAUNCH_CHECK();
  k_source_scale<<<dim3(P, batch), 256, 0, st>>>(ctx->n, ctx->nz, ctx->nr, ctx->dr, ctx->dz, ip_dev, w->spart, P, w->mr,
                                                 jphi_dev, nullptr, nullptr, nullptr);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_b_field(gsb_ctx *ctx, const double *psi_dev, double *br_dev, double *bz_dev, int batch, void *stream) {
  GSB_REQUIRE(ctx && psi_dev && br_dev && bz_dev, "gsb_b_field: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= 65535, "gsb_b_field: bad batch");
  GSB_CUDA(cudaSetDevice(ctx->device));
  const dim3 blk(32, 8, 1), grd((ctx->nr + 31) / 32, (ctx->nz + 7) / 8, batch);
  k_bfield<<<grd, blk, 0, (cudaStream_t)stream>>>(psi_dev, ctx->nz, ctx->nr, make_grad_geom(ctx->dz, ctx->dr), ctx->r_dev, br_dev, bz_dev);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_picard_last_launched_iterations(gsb_ctx *ctx) { return ctx ? ctx->picard_last_iters : 0; }

// The batched Picard solve behind gsb_picard_solve and the free-boundary outer loop.  mask_dev / order_dev /
// n_order_dev (all NULL, or all set and consistent: mask[b] != 0 <=> b is one of the first *n_order entries of
// order) restrict the solve to a subset of the batch; everything else is left untouched.
static int picard_solve_impl(gsb_ctx *ctx, const gsb_picard_params *p, double *psi_dev, const double *bc_dev,
                             const double *ip_dev, const double *prof_dev, double *jphi_dev, double *summary_dev,
                             double *hist_dev, double *gs_hist_dev, int batch, const int *mask_dev,
                             const int *order_dev, const int *n_order_dev, void *stream) {
  GSB_REQUIRE(ctx && p && psi_dev && bc_dev && ip_dev && jphi_dev && summary_dev, "gsb_picard_solve: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap, "gsb_picard_solve: batch outside [1, batch_cap]");
  GSB_REQUIRE(p->max_iterations >= 1, "gsb_picard_solve: max_iterations must be >= 1");
  GSB_REQUIRE(p->method >= 0 && p->method <= 3, "gsb_picard_solve: unknown method");
  GSB_REQUIRE(p->method != 3 || (p->anderson_depth >= 0 && p->anderson_depth <= kAndMax),
              "gsb_picard_solve: anderson_depth outside [0, 8]");
  GSB_REQUIRE(std::isfinite(p->omega) && p->omega >= 1.0 && p->omega < 2.0,
              "omega must be finite and satisfy 1.0 <= omega < 2.0");
  GSB_REQUIRE(!p->require_gs_residual || p->gs_tol > 0.0, "solver.gs_residual_threshold must be > 0");
  GSB_CUDA(cudaSetDevice(ctx->device));
  int rc = ensure_plan(ctx, 5);
  if (rc) return rc;
  rc = picard_ws_ensure(ctx, p);
  if (rc) return rc;
  gsb_picard_ws *w = ctx->picard;
  cudaStream_t st = (cudaStream_t)stream;
  const int nz = ctx->nz, nr = ctx->nr;
  const size_t n = ctx->n;
  const LevelGeom &g = ctx->levels[0].g;
  Bufs bufs{{psi_dev, w->buf1, w->buf2}};
  PicardState &s = w->s;
  const int P = partials_for(nz, nr);
  const GradGeom gg = make_grad_geom(ctx->dz, ctx->dr);
  if (p->method == 0 && !std::getenv("GSB_PICARD_STREAMING")) {
    rc = picard_resident_launch(ctx, p, psi_dev, bc_dev, ip_dev, prof_dev, jphi_dev, summary_dev, hist_dev,
                                gs_hist_dev, batch, order_dev, n_order_dev, st);
    if (rc != GSB_ESTATE) return rc;  // GSB_ESTATE: one equilibrium does not fit an SM -> streaming path
  }
  const int copy_blocks = (int)std::min<size_t>((n + 255) / 256, 64);
  const ProfileDev prof = to_dev(p->prof);

  // The loop below is ~12 launches per Picard iteration and a single equilibrium is launch-latency bound on it
  // (257^2: 22 us per launch), so blocks of `check_every` iterations are replayed from a CUDA graph.  Graph
  // capture is not allowed on the legacy default stream (what torch hands over by default): the whole solve runs
  // on a private non-blocking stream ordered after / before the caller's stream by events.
  const bool use_graph = !std::getenv("GSB_NO_GRAPH");
  cudaStream_t caller = st;
  if (use_graph) {
    if (!ctx->gstream) {
      GSB_CUDA(cudaStreamCreateWithFlags(&ctx->gstream, cudaStreamNonBlocking));
      GSB_CUDA(cudaEventCreateWithFlags(&ctx->gevent, cudaEventDisableTiming));
    }
    GSB_CUDA(cudaEventRecord(ctx->gevent, caller));
    GSB_CUDA(cudaStreamWaitEvent(ctx->gstream, ctx->gevent, 0));
    st = ctx->gstream;
  }

  k_picard_init<<<(batch + 127) / 128, 128, 0, st>>>(s, batch, p->seed ? 2 : 0, ip_dev, p->seed, mask_dev);
  GSB_LAUNCH_CHECK();
  rc = ring_save_launch(bc_dev, n, w->ring, nz, nr, batch, st);
  if (rc) return rc;
  if (p->external_profile) {  // equilibria whose seed does not run keep J_phi = 0 and a zero source
    GSB_REQUIRE(mask_dev == nullptr, "external_profile_mode is not combined with a masked (free-boundary batch) solve");
    GSB_CUDA(cudaMemsetAsync(jphi_dev, 0, (size_t)batch * n * sizeof(double), st));
    GSB_CUDA(cudaMemsetAsync(w->source, 0, (size_t)batch * n * sizeof(double), st));
  }
  if (p->seed) {
    // Psi_best = Psi.copy() is taken BEFORE seeding (newton_solver.py:484,496)
    GSB_CUDA(cudaMemcpyAsync(w->buf2, psi_dev, (size_t)batch * n * sizeof(double), cudaMemcpyDeviceToDevice, st));
    volatile double ssum = w->seed_sum * ctx->dr;
    volatile double ssum2 = ssum * ctx->dz;
    k_seed_source<<<dim3(copy_blocks, batch), 256, 0, st>>>(n, nr, w->seedJ, ssum2, ip_dev, w->mr, jphi_dev, w->source, s.seed_active);
    GSB_LAUNCH_CHECK();
    // 50 Jacobi steps, ping-pong psi <-> W (five steps per pass over HBM, gsb_sweep.cu: k_jacobi_warp)
    rc = jacobi_steps_launch(ctx, psi_dev, w->W, w->source, 50, batch, s.seed_active, st);
    if (rc) return rc;
  }

  AndersonBufs mixb{};
  if (p->method == 3) {  // depth < 2 never mixes (mk < 2): the "mixed" iterate is the relaxed one with its walls reset
    mixb.m = p->anderson_depth;
    mixb.slots = std::max(mixb.m, 1);
    if (mixb.m >= 2 && w->and_slots < mixb.slots) {
      if (w->and_psi) cudaFree(w->and_psi);
      if (w->and_res) cudaFree(w->and_res);
      w->and_psi = w->and_res = nullptr;
      w->and_slots = 0;
      const size_t bytes = (size_t)w->cap * mixb.slots * n * sizeof(double);
      GSB_CUDA(cudaMalloc(&w->and_psi, bytes));
      GSB_CUDA(cudaMalloc(&w->and_res, bytes));
      w->and_slots = mixb.slots;
    }
    if (!w->and_part) {
      GSB_CUDA(cudaMalloc(&w->and_part, (size_t)w->cap * kAndPB * kAndEnt * sizeof(double)));
      GSB_CUDA(cudaMalloc(&w->and_alpha, (size_t)w->cap * kAndMax * sizeof(double)));
      GSB_CUDA(cudaMalloc(&w->and_fb, (size_t)w->cap * sizeof(int)));
    }
    mixb.psi = w->and_psi;
    mixb.res = w->and_res;
    mixb.part = w->and_part;
    mixb.alpha = w->and_alpha;
    mixb.fallback = w->and_fb;
  }
  const double oma = 1.0 - p->alpha;
  const RelaxPlan rplan = relax_plan(nz, nr, batch, ctx->num_sms);
  const int check_every = p->check_every > 0 ? p->check_every : 8;
  volatile double dr2 = ctx->dr * ctx->dr, dz2 = ctx->dz * ctx->dz, f1 = 4.0 * ctx->dr, f2 = f1 * ctx->dz;
  // one Picard iteration of every active equilibrium; `poll`: reset the active counter before the decision and
  // copy it to the host afterwards.  Nothing in here depends on the host-side iteration number.
  auto issue_iteration = [&](bool poll) -> int {
    k_topo<<<dim3(P, batch), 256, 0, st>>>(bufs, s.cur, n, nz, nr, gg, w->rowmask, w->tpart, s.active);
    GSB_LAUNCH_CHECK();
    if (p->saddle) {
      int r2 = saddle_launch(ctx, bufs, s.cur, batch, gg, dr2, dz2, f2, s.xsel, s.active, st);
      if (r2) return r2;
    }
    k_topo_final<<<(batch + 127) / 128, 128, 0, st>>>(bufs, s.cur, n, nr, P, w->tpart, p->saddle ? s.xsel : nullptr,
                                                      s.topo, s.axbnd, 1, batch, s.active);
    GSB_LAUNCH_CHECK();
    if (!p->external_profile) {
      k_source_raw<<<dim3(P, batch), 256, 0, st>>>(bufs, s.cur, n, nz, nr, s.axbnd, prof, prof_dev, ctx->r_dev, w->cf,
                                                   jphi_dev, w->spart, s.active);
      GSB_LAUNCH_CHECK();
      k_source_scale<<<dim3(P, batch), 256, 0, st>>>(n, nz, nr, ctx->dr, ctx->dz, ip_dev, w->spart, P, w->mr, jphi_dev,
                                                     w->source, s.scale, s.active);
      GSB_LAUNCH_CHECK();
    }
    if (p->method == 0) {
      k_copy_from_cur<<<dim3(copy_blocks, batch), 256, 0, st>>>(bufs, s.cur, n, w->W, 0, s.active);
      GSB_LAUNCH_CHECK();
      int r2 = vcycle_launch(ctx, w->W, n, w->source, batch, p->omega, 3, 3, s.active, st);
      if (r2) return r2;
    } else if (p->method == 1 || p->method == 3) {  // "anderson" uses the SOR sweep (iterative_solver.py:376)
      k_copy_from_cur<<<dim3(copy_blocks, batch), 256, 0, st>>>(bufs, s.cur, n, w->W, 1, s.active);
      GSB_LAUNCH_CHECK();
      int r2 = smooth_launch(g, w->W, n, w->source, n, batch, p->omega, 1, 1, s.active, st);
      if (r2) return r2;
    } else {
      const dim3 blk(32, 8, 1), grd((nr + 31) / 32, (nz + 7) / 8, batch);
      k_jacobi_from_cur<<<grd, blk, 0, st>>>(g, bufs, s.cur, w->source, w->W, s.active);
      GSB_LAUNCH_CHECK();
    }
    {  // Psi_new's wall = the boundary map (copy_wall, newton_solver.py:514 via _elliptic_solve): written into W
      int r2 = ring_apply_launch(w->W, n, w->ring, nz, nr, batch, s.active, st);
      if (r2) return r2;
    }
    k_relax<<<dim3(rplan.P, batch), 128, 0, st>>>(g, bufs, s.cur, s.nxt, w->W, w->source, p->alpha, oma, w->rpart, s.active,
                                                  rplan);
    GSB_LAUNCH_CHECK();
    if (p->method == 3) {  // every kernel decides on the device whether this is a mixing iteration
      const int blocks = (int)std::min<size_t>((n + 255) / 256, 256);
      k_and_push<<<dim3(blocks, batch), 256, 0, st>>>(mixb, bufs, s.nxt, s.iter, w->W, w->ring, nz, nr, s.active);
      GSB_LAUNCH_CHECK();
      if (mixb.m >= 2) {
        k_and_gram<<<dim3(kAndPB, batch), 256, 0, st>>>(mixb, s.iter, n, s.active);
        GSB_LAUNCH_CHECK();
      }
      k_and_solve<<<(batch + 63) / 64, 64, 0, st>>>(mixb, s.iter, kAndPB, batch, s.active);
      GSB_LAUNCH_CHECK();
      k_and_mix<<<dim3(blocks, batch), 256, 0, st>>>(mixb, bufs, s.nxt, s.iter, w->ring, nz, nr, s.active);
      GSB_LAUNCH_CHECK();
      k_and_gs<<<dim3(rplan.P, batch), 256, 0, st>>>(g, bufs, s.nxt, s.iter, w->source, w->rpart, s.active);
      GSB_LAUNCH_CHECK();
    }
    if (poll) GSB_CUDA(cudaMemsetAsync(ctx->counter, 0, sizeof(int), st));
    k_decide<<<(batch + 127) / 128, 128, 0, st>>>(s, w->rpart, rplan.P, (double)n, (double)(nz - 2) * (double)(nr - 2), p->tol,
                                                  p->require_gs_residual, p->gs_tol, p->max_iterations, hist_dev,
                                                  gs_hist_dev, ctx->counter, batch);
    GSB_LAUNCH_CHECK();
    if (poll) GSB_CUDA(cudaMemcpyAsync(ctx->h_counter, ctx->counter, sizeof(int), cudaMemcpyDeviceToHost, st));
    return GSB_OK;
  };
  int k = 0;
  bool done = false;
  // first block eagerly: it performs every lazy allocation / attribute opt-in of the sequence (none is allowed
  // while a stream is being captured)
  while (k < p->max_iterations && !done) {
    const bool poll = ((k + 1) % check_every == 0) || (k + 1 == p->max_iterations);
    rc = issue_iteration(poll);
    if (rc) return rc;
    ++k;
    if (poll) {
      GSB_CUDA(cudaStreamSynchronize(st));
      done = ctx->h_counter[0] == 0;
      break;
    }
  }
  if (use_graph && !done && k < p->max_iterations) {
    // later blocks: one graph of `check_every` iterations.  An equilibrium that reaches max_iterations inside a
    // block simply turns inactive (k_decide), so whole blocks are always safe to replay.
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    const long long l0 = g_launches.load();
    GSB_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    for (int j = 0; j < check_every && rc == GSB_OK; ++j) rc = issue_iteration(j + 1 == check_every);
    cudaError_t ce = cudaStreamEndCapture(st, &graph);
    const long long per_block = g_launches.load() - l0;
    if (rc == GSB_OK && ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (rc) return rc;
    GSB_CUDA(ce);
    g_launches.fetch_sub(per_block);  // the captured launches did not run
    while (k < p->max_iterations && !done) {
      ce = cudaGraphLaunch(exec, st);
      if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
      if (ce != cudaSuccess) break;
      g_launches.fetch_add(per_block);
      k += check_every;
      done = ctx->h_counter[0] == 0;
    }
    cudaGraphExecDestroy(exec);
    GSB_CUDA(ce);
    if (k > p->max_iterations) k = p->max_iterations;
  } else {
    while (k < p->max_iterations && !done) {
      const bool poll = ((k + 1) % check_every == 0) || (k + 1 == p->max_iterations);
      rc = issue_iteration(poll);
      if (rc) return rc;
      ++k;
      if (poll) {
        GSB_CUDA(cudaStreamSynchronize(st));
        done = ctx->h_counter[0] == 0;
      }
    }
  }
  ctx->picard_last_iters = k;
  k_finalize<<<dim3(copy_blocks, batch), 256, 0, st>>>(bufs, s, n, summary_dev, batch, mask_dev);
  GSB_LAUNCH_CHECK();
  if (use_graph) {  // the caller's stream continues after the private one
    GSB_CUDA(cudaEventRecord(ctx->gevent, st));
    GSB_CUDA(cudaStreamWaitEvent(caller, ctx->gevent, 0));
  }
  return GSB_OK;
}

int gsb_picard_solve(gsb_ctx *ctx, const gsb_picard_params *p, double *psi_dev, const double *bc_dev,
                     const double *ip_dev, const double *prof_dev, double *jphi_dev, double *summary_dev,
                     double *hist_dev, double *gs_hist_dev, int batch, void *stream) {
  return picard_solve_impl(ctx, p, psi_dev, bc_dev, ip_dev, prof_dev, jphi_dev, summary_dev, hist_dev, gs_hist_dev,
                           batch, nullptr, nullptr, nullptr, stream);
}

}  // extern "C"

namespace gsb {

// ---------------------------------------------------------------------------------------------------------
// Batched free-boundary outer loop (solve_free_boundary, fusion_kernel_free_boundary.py:623-739) on device:
//   per outer iteration, for every equilibrium that has not converged yet:
//     wall ring of Psi <- coil flux ring [+ plasma wall flux M @ (J dA)]      (:652-655; lane C :498)
//     Psi_old <- Psi                                                          (:658)
//     warm-started, re-seeded Picard solve with that boundary map            (:659-662)
//     diff = max |Psi - Psi_old|; stop this equilibrium when diff < tol       (:708-711)
// The host only reads one counter per OUTER iteration.
// ---------------------------------------------------------------------------------------------------------
int free_boundary_loop(gsb_ctx *ctx, const gsb_picard_params *p, const gsb_free_boundary_params *fb, const ShapeStep *sh,
                       double *psi_dev, double *psi_ext_dev, const double *wall_m_dev, const double *ip_dev,
                       const double *prof_dev, double *jphi_dev, double *summary_dev, double *fb_summary_dev, int batch,
                       void *stream) {
  GSB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = ctx->n;
  const int nz = ctx->nz, nr = ctx->nr, nw = ctx->n_wall;
  // workspace: previous iterate, masks / work list, reduction partials, plasma wall flux
  const size_t cap = (size_t)ctx->batch_cap;
  if (!ctx->fb_old) GSB_CUDA(cudaMalloc(&ctx->fb_old, cap * n * sizeof(double)));
  if (!ctx->fb_part) GSB_CUDA(cudaMalloc(&ctx->fb_part, cap * kPT * 2 * sizeof(double)));
  if (!ctx->fb_ints) GSB_CUDA(cudaMalloc(&ctx->fb_ints, (2 * cap + 2) * sizeof(int)));
  if (wall_m_dev && !ctx->fb_wall) GSB_CUDA(cudaMalloc(&ctx->fb_wall, cap * nw * sizeof(double)));
  double *old = ctx->fb_old, *part = ctx->fb_part, *wall = wall_m_dev ? ctx->fb_wall : nullptr;
  int *mask = ctx->fb_ints, *order = ctx->fb_ints + batch, *n_order = ctx->fb_ints + 2 * batch;
  const int P = partials_for(nz, nr);
  const int blocks = (int)std::min<size_t>((n + 255) / 256, 64);
  int rc = GSB_OK;
  k_fb_init<<<(batch + 255) / 256, 256, 0, st>>>(mask, order, n_order, fb_summary_dev, batch);
  GSB_LAUNCH_CHECK();
  const double dA = ctx->dr * ctx->dz;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  if (ctx->timing)
    for (auto &e : ev) GSB_CUDA(cudaEventCreate(&e));
  int outer = 0;
  for (; outer < fb->max_outer_iter; ++outer) {
    const bool with_wall = wall_m_dev && (outer > 0 || fb->warm_j);
    if (with_wall) {
      if (ctx->timing) cudaEventRecord(ev[2], st);
      rc = gsb_wall_flux(ctx, wall_m_dev, jphi_dev, dA, wall, batch, stream);
      if (rc) break;
      if (ctx->timing) cudaEventRecord(ev[3], st);
    }
    k_fb_prepare<<<dim3(blocks, batch), 256, 0, st>>>(psi_dev, psi_ext_dev, with_wall ? wall : nullptr, old, n, nz, nr, nw, mask);
    GSB_LAUNCH_CHECK();
    if (ctx->timing) cudaEventRecord(ev[0], st);
    rc = picard_solve_impl(ctx, p, psi_dev, psi_dev /* the ring of psi IS the boundary map */, ip_dev, prof_dev, jphi_dev,
                           summary_dev, nullptr, nullptr, batch, mask, order, n_order, stream);
    if (rc) break;
    if (ctx->timing) cudaEventRecord(ev[1], st);
    if (sh) {  // before the decision, so an equilibrium that converges in this iteration still gets its currents
               // updated (as the reference)
      rc = shape_step_launch(ctx, *sh, psi_dev, psi_ext_dev, mask, batch, st);
      if (rc) break;
    }
    k_fb_diff<<<dim3(P, batch), 256, 0, st>>>(psi_dev, old, n, part, mask);
    GSB_LAUNCH_CHECK();
    k_fb_decide<<<1, 1024, 0, st>>>(part, P, fb->tol, outer, summary_dev, fb_summary_dev, mask, order, n_order, batch);
    GSB_LAUNCH_CHECK();
    GSB_CUDA(cudaMemcpyAsync(ctx->h_counter, n_order, sizeof(int), cudaMemcpyDeviceToHost, st));
    GSB_CUDA(cudaStreamSynchronize(st));
    if (ctx->timing) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ev[0], ev[1]) == cudaSuccess) ctx->timing_acc[0] += ms, ctx->timing_acc[1] += 1.0;
      if (with_wall && cudaEventElapsedTime(&ms, ev[2], ev[3]) == cudaSuccess) ctx->timing_acc[2] += ms, ctx->timing_acc[3] += 1.0;
    }
    if (ctx->h_counter[0] == 0) {
      ++outer;
      break;
    }
  }
  for (auto &e : ev)
    if (e) cudaEventDestroy(e);
  return rc;
}

int free_boundary_check(gsb_ctx *ctx, const gsb_free_boundary_params *fb, int batch) {
  GSB_REQUIRE(batch >= 1 && batch <= ctx->batch_cap && batch <= 65535, "gsb_free_boundary_solve: batch outside [1, min(batch_cap, 65535)]");
  GSB_REQUIRE(fb->max_outer_iter >= 1, "max_outer_iter must be >= 1.");
  GSB_REQUIRE(std::isfinite(fb->tol) && fb->tol >= 0.0, "tol must be finite and >= 0.");
  GSB_REQUIRE(ctx->nz >= 3 && ctx->nr >= 3, "gsb_free_boundary_solve: grid has no interior");
  return GSB_OK;
}

}  // namespace gsb

extern "C" {

int gsb_free_boundary_solve(gsb_ctx *ctx, const gsb_picard_params *p, const gsb_free_boundary_params *fb,
                            double *psi_dev, const double *psi_ext_dev, const double *wall_m_dev,
                            const double *ip_dev, const double *prof_dev, double *jphi_dev, double *summary_dev,
                            double *fb_summary_dev, int batch, void *stream) {
  GSB_REQUIRE(ctx && p && fb && psi_dev && psi_ext_dev && ip_dev && jphi_dev && summary_dev && fb_summary_dev,
              "gsb_free_boundary_solve: NULL argument");
  const int rc = free_boundary_check(ctx, fb, batch);
  if (rc) return rc;
  // without a shape step the loop only reads psi_ext
  return free_boundary_loop(ctx, p, fb, nullptr, psi_dev, const_cast<double *>(psi_ext_dev), wall_m_dev, ip_dev,
                            prof_dev, jphi_dev, summary_dev, fb_summary_dev, batch, stream);
}

int gsb_timing(gsb_ctx *ctx, int enable, double *out4, int reset) {
  GSB_REQUIRE(ctx, "gsb_timing: NULL context");
  ctx->timing = enable != 0;
  if (out4)
    for (int i = 0; i < 4; ++i) out4[i] = ctx->timing_acc[i];
  if (reset)
    for (double &v : ctx->timing_acc) v = 0.0;
  return GSB_OK;
}

}  // extern "C"

// gsb_resident.cuh - shared-memory-resident multigrid: one CTA owns one equilibrium and runs a
// whole V-cycle (all levels) without touching HBM.
//
// Layout ("colour-split"): a level field x[nz][nr] is kept as two planes, one per red/black
// colour c = (iz+ir)&1, each [nz][hw] with hw = (nr+1)/2 and element (iz, k) <-> ir = 2k + s,
// s = ir&1.  With it every operand of a colour pass is unit-stride across the lanes of a warp
// (no bank conflicts on 64-bit accesses):
//   point (iz, k) of colour p, s = (p+iz)&1:   S,N = Q[iz-1][k], Q[iz+1][k]   (Q = other colour)
//                                              s=0: W = Q[iz][k-1], E = Q[iz][k]
//                                              s=1: W = Q[iz][k],   E = Q[iz][k+1]
// Equivalently, with e = iz*hw + k the "slot" of the column pair (2k, 2k+1) in row iz:
//   x(iz, 2k)   = plane[iz&1][e]          x(iz, 2k+1) = plane[(iz+1)&1][e]
// Every operator maps a thread to one k slot (one column pair) and a run of consecutive rows and
// slides a register window down the run: a smoother update costs 3 shared loads + 1 store (+ the
// right-hand side).  All passes of a smoothing phase run inside one call so the per-thread setup
// (slot map, stencil coefficients) is paid once.  Arithmetic is the same operand order as the
// streaming kernels (bit-identical results).
#pragma once

#include "gsb_internal.cuh"

namespace gsb {

constexpr int kResThreads = 512;  // threads of a resident CTA (one CTA per SM): 16 warps at 128 registers
constexpr int kResMaxLevels = 12;
constexpr int kResSmemMax = 232448;  // 227 KB opt-in dynamic shared memory per CTA on sm_100

struct RLevel {
  int nz, nr, hw, nk;  // hw = (nr+1)/2 ; nk = nr/2 interior k slots
  int x_off;           // doubles offset of the solution planes [2][nz][hw] in the pool
  int d_off;           // doubles offset of the right-hand-side planes (levels after the first)
  int t_off;           // doubles offset of a shared-memory copy of a_e|a_w (2*nr) or -1
  // thread -> (k slot, row chunk) maps, precomputed on the host (no integer division on device)
  int lk;              // log2 of the padded slot count for k in [0, nk)
  int nch, rpc;        // row chunks over the nz-2 interior rows, rows per chunk
  int lj;              // log2 of the padded slot count for coarse columns J in [1, nrc-2] (restriction INTO this level)
  int cch, crpc;       // chunks over this level's interior rows when it is the coarse side
  LevelGeom g;
};
struct RPlan {
  int nlev;
  int pool_doubles;  // planes + tables; the staged level descriptors follow
  RLevel lev[kResMaxLevels];
};
static_assert(sizeof(RLevel) % 8 == 0, "RLevel is staged to shared memory in 8-byte words");
inline int res_stage_doubles(int nlev) { return nlev * (int)(sizeof(RLevel) / 8); }

// The one dynamic shared-memory array of the resident kernels.  Every access is written as
// res_pool[integer offset] so that it compiles to LDS/STS: a generic-address load from shared
// memory costs ~150 cycles instead of ~30 (measured).
extern __shared__ double res_pool[];

__device__ __forceinline__ const RLevel &res_level(int lev_off, int l) {
  return reinterpret_cast<const RLevel *>(res_pool + lev_off)[l];
}

// Optional in-kernel phase timing (build with -DGSB_PHASE_TIMING): CTA 0 accumulates clock64()
// deltas per phase into g_phase[]; read back with gsb_debug_phase_cycles().
#ifdef GSB_PHASE_TIMING
__device__ long long g_phase[64];
#define GSB_PHASE_BEGIN() long long _pt = clock64()
#define GSB_PHASE(idx)                                      \
  do {                                                      \
    if (blockIdx.x == 0 && threadIdx.x == 0) {              \
      const long long _now = clock64();                     \
      g_phase[(idx)] += _now - _pt;                         \
      _pt = _now;                                           \
    }                                                       \
  } while (0)
#define GSB_PHASE_COUNT(idx) g_phase[(idx)] += 1
#else
#define GSB_PHASE_BEGIN() do {} while (0)
#define GSB_PHASE(idx) do {} while (0)
#define GSB_PHASE_COUNT(idx) do {} while (0)
#endif

__device__ __forceinline__ int split_index(int nz, int hw, int iz, int ir) {
  return (((iz + ir) & 1) * nz + iz) * hw + (ir >> 1);
}

// a / b with y = RN(1/b): the Markstein sequence without ddiv_y's non-finite guard.  Identical to
// ddiv_y (and to IEEE a/b) whenever the quotient is finite; a non-finite quotient comes out as NaN
// instead of +-inf, which every caller treats the same way (non-finite => diverged).
__device__ __forceinline__ double ddiv_yf(double a, double b, double y) {
  const double q = __dmul_rn(a, y);
  const double r = __fma_rn(-b, q, a);
  return __fma_rn(r, y, q);
}

// dense global [nz][nr] -> planes (warp per row segment, no integer division)
__device__ __forceinline__ void res_load_dense(const double *__restrict__ g, int xo, int nz, int nr,
                                               int hw) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int iz = warp; iz < nz; iz += nw) {
    const double *row = g + (size_t)iz * nr;
    for (int ir = lane; ir < nr; ir += 32) res_pool[xo + (((iz + ir) & 1) * nz + iz) * hw + (ir >> 1)] = row[ir];
  }
}
__device__ __forceinline__ void res_store_dense(double *__restrict__ g, int xo, int nz, int nr, int hw) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int iz = warp; iz < nz; iz += nw) {
    double *row = g + (size_t)iz * nr;
    for (int ir = lane; ir < nr; ir += 32) row[ir] = res_pool[xo + (((iz + ir) & 1) * nz + iz) * hw + (ir >> 1)];
  }
}

// Per-level smoother constants held in registers (never re-read from shared memory).
struct SorK {
  double a_ns, a_c, inv_a_c, omega, omw;
};

// One RB-SOR update (multigrid_solve.py:196-205, NumPy operand order).  S = ir&1 of the updated
// point: its (W, E) neighbours are (side, c_cur) for S = 0 and (c_cur, side) for S = 1.
template <int S>
__device__ __forceinline__ double res_update(const SorK &c, double ae, double aw, double side, double c_prev,
                                             double c_cur, double c_next, double rhs, double old) {
  double acc = dadd(dmul(ae, S ? side : c_cur), dmul(aw, S ? c_cur : side));
  acc = dadd(acc, dmul(c.a_ns, c_prev));
  acc = dadd(acc, dmul(c.a_ns, c_next));
  acc = dsub(acc, rhs);
  const double gs = ddiv_yf(acc, c.a_c, c.inv_a_c);
  return dadd(dmul(c.omw, old), dmul(c.omega, gs));
}

// `cnt` consecutive rows of one k slot in one colour pass, right-hand side in the pool.  po/qo: pool
// offsets of P[z0][k] / Q[z0][k]; ro: pool offset of the rhs.  Row z0 has S = S0 and
// coefficients/predicate A; rows alternate A, B.
template <int S0>
__device__ __forceinline__ void res_smooth_run(int po, int qo, int ro, int hw, int cnt, double aeA, double awA, bool okA,
                                               double aeB, double awB, bool okB, const SorK &c) {
  constexpr int dA = S0 ? 1 : -1, dB = S0 ? -1 : 1;
  double c_prev = res_pool[qo - hw], c_cur = res_pool[qo];
  int i = 0;
  for (; i + 4 <= cnt; i += 4) {
    const double r0 = res_pool[ro], r1 = res_pool[ro + hw], r2 = res_pool[ro + 2 * hw], r3 = res_pool[ro + 3 * hw];
    ro += 4 * hw;
    const int q1 = qo + hw, q2 = q1 + hw, q3 = q2 + hw, q4 = q3 + hw;
    const int p1 = po + hw, p2 = p1 + hw, p3 = p2 + hw;
    const double c1 = res_pool[q1], c2 = res_pool[q2], c3 = res_pool[q3], c4 = res_pool[q4];
    const double s0 = res_pool[qo + dA], s1 = res_pool[q1 + dB], s2 = res_pool[q2 + dA], s3 = res_pool[q3 + dB];
    const double o0 = res_pool[po], o1 = res_pool[p1], o2 = res_pool[p2], o3 = res_pool[p3];
    const double v0 = res_update<S0>(c, aeA, awA, s0, c_prev, c_cur, c1, r0, o0);
    const double v1 = res_update<1 - S0>(c, aeB, awB, s1, c_cur, c1, c2, r1, o1);
    const double v2 = res_update<S0>(c, aeA, awA, s2, c1, c2, c3, r2, o2);
    const double v3 = res_update<1 - S0>(c, aeB, awB, s3, c2, c3, c4, r3, o3);
    if (okA) {
      res_pool[po] = v0;
      res_pool[p2] = v2;
    }
    if (okB) {
      res_pool[p1] = v1;
      res_pool[p3] = v3;
    }
    c_prev = c3;
    c_cur = c4;
    po = p3 + hw;
    qo = q4;
  }
  for (int t = 0; i < cnt; ++i, ++t) {  // tail (< 4 rows): alternate A, B
    const double c1 = res_pool[qo + hw];
    const double rv = res_pool[ro];
    if ((t & 1) == 0) {
      const double v = res_update<S0>(c, aeA, awA, res_pool[qo + dA], c_prev, c_cur, c1, rv, res_pool[po]);
      if (okA) res_pool[po] = v;
    } else {
      const double v = res_update<1 - S0>(c, aeB, awB, res_pool[qo + dB], c_prev, c_cur, c1, rv, res_pool[po]);
      if (okB) res_pool[po] = v;
    }
    c_prev = c_cur;
    c_cur = c1;
    po += hw;
    qo += hw;
    ro += hw;
  }
}

// The same pass with the right-hand side of ALL rows of the run (at most kResMaxRun) already in
// registers: the caller issues those global loads a whole pass ahead, so their L2 latency hides
// behind the previous pass.  Fully unrolled over groups of four rows (compile-time register indices).
constexpr int kResMaxRun = 16;  // rows per thread on the finest level
template <int S0>
__device__ __forceinline__ void res_smooth_run_pref(int po, int qo, int hw, int cnt, double aeA, double awA, bool okA,
                                                    double aeB, double awB, bool okB, const SorK &c,
                                                    const double (&r)[kResMaxRun]) {
  constexpr int dA = S0 ? 1 : -1, dB = S0 ? -1 : 1;
  double c_prev = res_pool[qo - hw], c_cur = res_pool[qo];
#pragma unroll
  for (int g = 0; g < kResMaxRun / 4; ++g) {
    if (4 * g + 4 <= cnt) {
      const int q1 = qo + hw, q2 = q1 + hw, q3 = q2 + hw, q4 = q3 + hw;
      const int p1 = po + hw, p2 = p1 + hw, p3 = p2 + hw;
      const double c1 = res_pool[q1], c2 = res_pool[q2], c3 = res_pool[q3], c4 = res_pool[q4];
      const double s0 = res_pool[qo + dA], s1 = res_pool[q1 + dB], s2 = res_pool[q2 + dA], s3 = res_pool[q3 + dB];
      const double o0 = res_pool[po], o1 = res_pool[p1], o2 = res_pool[p2], o3 = res_pool[p3];
      const double v0 = res_update<S0>(c, aeA, awA, s0, c_prev, c_cur, c1, r[4 * g], o0);
      const double v1 = res_update<1 - S0>(c, aeB, awB, s1, c_cur, c1, c2, r[4 * g + 1], o1);
      const double v2 = res_update<S0>(c, aeA, awA, s2, c1, c2, c3, r[4 * g + 2], o2);
      const double v3 = res_update<1 - S0>(c, aeB, awB, s3, c2, c3, c4, r[4 * g + 3], o3);
      if (okA) {
        res_pool[po] = v0;
        res_pool[p2] = v2;
      }
      if (okB) {
        res_pool[p1] = v1;
        res_pool[p3] = v3;
      }
      c_prev = c3;
      c_cur = c4;
      po = p3 + hw;
      qo = q4;
    } else if (4 * g < cnt) {
#pragma unroll
      for (int t = 0; t < 3; ++t) {  // tail (< 4 rows): alternate A, B
        if (4 * g + t < cnt) {
          const double c1 = res_pool[qo + hw];
          if ((t & 1) == 0) {
            const double v = res_update<S0>(c, aeA, awA, res_pool[qo + dA], c_prev, c_cur, c1, r[4 * g + t], res_pool[po]);
            if (okA) res_pool[po] = v;
          } else {
            const double v = res_update<1 - S0>(c, aeB, awB, res_pool[qo + dB], c_prev, c_cur, c1, r[4 * g + t], res_pool[po]);
            if (okB) res_pool[po] = v;
          }
          c_prev = c_cur;
          c_cur = c1;
          po += hw;
          qo += hw;
        }
      }
    }
  }
}

// `npass` colour passes (parity = (first + pass) & 1) of RB-SOR on the resident planes of level l.
// GR: the right-hand side (colour-split) and the coefficient tables live in global memory (the
// finest resident level); otherwise both are in the pool.  Ends with a barrier.
template <bool GR>
__device__ __noinline__ void res_smooth(int lev_off, int l, const double *__restrict__ rhs_g, int first, int npass,
                                        double omega, double omw) {
  int nz, nr, hw, nk, x_off, d_off, t_off, lk, nch, rpc;
  SorK c;
  const double *tab;
  {
    const RLevel &L = res_level(lev_off, l);
    nz = L.nz, nr = L.nr, hw = L.hw, nk = L.nk, x_off = L.x_off, d_off = L.d_off, t_off = L.t_off;
    lk = L.lk, nch = L.nch, rpc = L.rpc;
    c.a_ns = L.g.a_ns, c.a_c = L.g.a_c, c.inv_a_c = L.g.inv_a_c, c.omega = omega, c.omw = omw;
    tab = L.g.a_e;  // a_e | a_w, one allocation
  }
  const int tid = threadIdx.x;
  const int k = tid & ((1 << lk) - 1), ch = tid >> lk;
  const int z0 = 1 + ch * rpc;
  const int z1 = min(z0 + rpc, nz - 1);
  const bool active = (ch < nch) && (k < nk) && (z0 < z1);
  const int ir0 = 2 * k, ir1 = 2 * k + 1;
  double ae0 = 0.0, aw0 = 0.0, ae1 = 0.0, aw1 = 0.0;
  if (active) {
    if (GR) {
      ae0 = __ldg(tab + ir0);
      aw0 = __ldg(tab + nr + ir0);
      if (ir1 < nr) {
        ae1 = __ldg(tab + ir1);
        aw1 = __ldg(tab + nr + ir1);
      }
    } else {
      ae0 = res_pool[t_off + ir0];
      aw0 = res_pool[t_off + nr + ir0];
      if (ir1 < nr) {
        ae1 = res_pool[t_off + ir1];
        aw1 = res_pool[t_off + nr + ir1];
      }
    }
  }
  // k = 0 with S = 0 is the wall column: its `side` read at k-1 stays inside the pool (row >= 1)
  const bool ok0 = ir0 >= 1 && ir0 <= nr - 2, ok1 = ir1 <= nr - 2;
  const int o = z0 * hw + k, ps = nz * hw;
  const int cnt = z1 - z0;
  // every __syncthreads() below is reached by all threads of the CTA (inactive ones skip the work)
  if (rpc == 1) {
    // coarse levels: one row per thread, S varies across the warp -> runtime selects
    for (int pass = 0; pass < npass; ++pass) {
      if (active) {
        const int par = (first + pass) & 1;
        const int P = x_off + par * ps + o, Q = x_off + (1 - par) * ps + o;
        const int s = (par + z0) & 1;
        const double cc = res_pool[Q], side = res_pool[Q - 1 + 2 * s];
        const double rv = GR ? __ldcg(rhs_g + par * ps + o) : res_pool[d_off + par * ps + o];
        double acc = dadd(dmul(s ? ae1 : ae0, s ? side : cc), dmul(s ? aw1 : aw0, s ? cc : side));
        acc = dadd(acc, dmul(c.a_ns, res_pool[Q - hw]));
        acc = dadd(acc, dmul(c.a_ns, res_pool[Q + hw]));
        acc = dsub(acc, rv);
        const double gs = ddiv_yf(acc, c.a_c, c.inv_a_c);
        const double v = dadd(dmul(c.omw, res_pool[P]), dmul(c.omega, gs));
        if (s ? ok1 : ok0) res_pool[P] = v;
      }
      __syncthreads();
    }
    return;
  }
  // rpc is even -> z0 is odd -> S of the first row is uniform over the CTA: (par + 1) & 1
  if (GR) {
    // finest level: rhs in global (L2) memory; the whole run's rhs is fetched one pass ahead
    double r[kResMaxRun];
    auto fetch = [&](int par) {
      const double *rg = rhs_g + par * ps + o;
#pragma unroll
      for (int t = 0; t < kResMaxRun; ++t) r[t] = (t < cnt) ? __ldcg(rg + t * hw) : 0.0;
    };
    if (active) fetch(first & 1);
    for (int pass = 0; pass < npass; ++pass) {
      if (active) {
        const int par = (first + pass) & 1;
        const int P = x_off + par * ps + o, Q = x_off + (1 - par) * ps + o;
        if ((par + z0) & 1)
          res_smooth_run_pref<1>(P, Q, hw, cnt, ae1, aw1, ok1, ae0, aw0, ok0, c, r);
        else
          res_smooth_run_pref<0>(P, Q, hw, cnt, ae0, aw0, ok0, ae1, aw1, ok1, c, r);
        if (pass + 1 < npass) fetch(1 - par);
      }
      __syncthreads();
    }
  } else {
    for (int pass = 0; pass < npass; ++pass) {
      if (active) {
        const int par = (first + pass) & 1;
        const int P = x_off + par * ps + o, Q = x_off + (1 - par) * ps + o;
        const int ro = d_off + par * ps + o;
        if ((par + z0) & 1)
          res_smooth_run<1>(P, Q, ro, hw, cnt, ae1, aw1, ok1, ae0, aw0, ok0, c);
        else
          res_smooth_run<0>(P, Q, ro, hw, cnt, ae0, aw0, ok0, ae1, aw1, ok1, c);
      }
      __syncthreads();
    }
  }
}

// L x at one point (multigrid_solve.py:243-247), level constants in registers.
struct ResK {
  double dr2, dz2, two_dr, inv_dr2, inv_dz2, inv_two_dr;
};
__device__ __forceinline__ double res_lx(const ResK &g, double rs, double inv_rs, double C, double E, double W, double S,
                                         double N) {
  const double twoC = dmul(2.0, C);
  const double d2r = ddiv_yf(dadd(dsub(E, twoC), W), g.dr2, g.inv_dr2);
  const double d1r = ddiv_yf(dsub(E, W), g.two_dr, g.inv_two_dr);
  const double d2z = ddiv_yf(dadd(dsub(N, twoC), S), g.dz2, g.inv_dz2);
  return dadd(dsub(d2r, ddiv_yf(d1r, rs, inv_rs)), d2z);
}
__device__ __forceinline__ ResK res_load_resk(const LevelGeom &g) {
  ResK k;
  k.dr2 = g.dr2, k.dz2 = g.dz2, k.two_dr = g.two_dr, k.inv_dr2 = g.inv_dr2, k.inv_dz2 = g.inv_dz2,
  k.inv_two_dr = g.inv_two_dr;
  return k;
}

struct Row5 {
  double v0, v1, v2, v3, v4;
};
struct Row3 {
  double a, b, c;
};

// d_coarse = restrict_full_weight( -(L x - rhs) ) on the coarse interior (coarse wall unused).
// Thread <-> coarse column J and a chunk of coarse rows; marches over fine rows keeping the three
// residuals of each of the last fine rows (columns 2J-1, 2J, 2J+1) in registers.
template <bool GR>
__device__ __noinline__ void res_residual_restrict(int lev_off, int l, const double *__restrict__ rhs_g) {
  int nz, hw, xo, fd_off, cnz, cnr, chw, cd_off, lj, cch, crpc;
  ResK g;
  const double *ts, *ti;
  {
    const RLevel &L = res_level(lev_off, l);
    const RLevel &C = res_level(lev_off, l + 1);
    nz = L.nz, hw = L.hw, xo = L.x_off, fd_off = L.d_off;
    cnz = C.nz, cnr = C.nr, chw = C.hw, cd_off = C.d_off, lj = C.lj, cch = C.cch, crpc = C.crpc;
    g = res_load_resk(L.g);
    ts = L.g.r_safe, ti = L.g.inv_r_safe;
  }
  const int tid = threadIdx.x;
  const int J = 1 + (tid & ((1 << lj) - 1)), ch = tid >> lj;
  const int I0 = 1 + ch * crpc;
  const int I1 = min(I0 + crpc, cnz - 1);
  if (!(ch >= cch || J > cnr - 2 || I0 >= I1)) {
  // fine columns 2J-2 .. 2J+2 : even ones (k = J-1, J, J+1) live in plane (iz&1), odd ones
  // (k = J-1, J) in plane ((iz+1)&1)
  const int irm = 2 * J - 1, ir0 = 2 * J, irp = 2 * J + 1;
  const double rsm = ts[irm], rs0 = ts[ir0], rsp = ts[irp], ism = ti[irm], is0 = ti[ir0], isp = ti[irp];
  const int ps = nz * hw;
  const int last = 2 * (I1 - 1) + 1;  // last fine row whose residual is needed
  auto load_row = [&](int iz) -> Row5 {  // x(iz, 2J-2 .. 2J+2)
    const int e = iz * hw + J;
    const int pe = xo + (iz & 1) * ps + e;
    const int po = xo + ((iz + 1) & 1) * ps + e;
    Row5 r;
    r.v0 = res_pool[pe - 1];
    r.v1 = res_pool[po - 1];
    r.v2 = res_pool[pe];
    r.v3 = res_pool[po];
    r.v4 = res_pool[pe + 1];
    return r;
  };
  auto load_rhs = [&](int iz) -> Row3 {  // rhs(iz, 2J-1 .. 2J+1)
    const int e = iz * hw + J;
    const int pe = (iz & 1) * ps + e;
    const int po = ((iz + 1) & 1) * ps + e;
    Row3 r;
    if (GR) {
      r.a = rhs_g[po - 1];
      r.b = rhs_g[pe];
      r.c = rhs_g[po];
    } else {
      r.a = res_pool[fd_off + po - 1];
      r.b = res_pool[fd_off + pe];
      r.c = res_pool[fd_off + po];
    }
    return r;
  };
  int iz = 2 * I0 - 1;
  Row5 xm = load_row(iz - 1), x0 = load_row(iz);
  Row3 f = load_rhs(iz);
  auto res_row = [&]() -> Row3 {  // negated residuals of fine row iz, then slide the window down
    const Row5 xp = load_row(iz + 1);
    const Row3 fc = f;
    if (iz < last) f = load_rhs(iz + 1);  // one row ahead (global latency)
    Row3 r;
    r.a = -dsub(res_lx(g, rsm, ism, x0.v1, x0.v2, x0.v0, xm.v1, xp.v1), fc.a);
    r.b = -dsub(res_lx(g, rs0, is0, x0.v2, x0.v3, x0.v1, xm.v2, xp.v2), fc.b);
    r.c = -dsub(res_lx(g, rsp, isp, x0.v3, x0.v4, x0.v2, xm.v3, xp.v3), fc.c);
    xm = x0;
    x0 = xp;
    ++iz;
    return r;
  };
  Row3 rA = res_row();
  const int cps = cnz * chw;
  int cpar = (I0 + J) & 1;
  int co = cd_off + cpar * cps + I0 * chw + (J >> 1);
  for (int I = I0; I < I1; ++I) {
    const Row3 rB = res_row();
    const Row3 rC = res_row();
    res_pool[co] = fw9(rB.b, rA.b, rC.b, rB.a, rB.c, rA.a, rA.c, rC.a, rC.c);
    rA = rC;
    co += chw + (cpar ? -cps : cps);  // next coarse row: the plane parity flips
    cpar ^= 1;
  }
  }  // active
}

// x_fine += P e_coarse on the fine interior (prolongate_bilinear, multigrid_solve.py:102-145).
// Thread <-> fine k slot (columns 2k, 2k+1 <-> coarse columns k, k+1) and a chunk of fine rows.
static __device__ __noinline__ void res_prolong_add(int lev_off, int l) {
  int nz, nr, hw, nk, xo, lk, nch, rpc, nzc, nrc, hwc, eo;
  {
    const RLevel &L = res_level(lev_off, l);
    const RLevel &C = res_level(lev_off, l + 1);
    nz = L.nz, nr = L.nr, hw = L.hw, nk = L.nk, xo = L.x_off, lk = L.lk, nch = L.nch, rpc = L.rpc;
    nzc = C.nz, nrc = C.nr, hwc = C.hw, eo = C.x_off;
  }
  const int kz = min(nzc, (nz + 1) / 2), kr = min(nrc, (nr + 1) / 2);
  const int hend = min(2 * (nrc - 1), nr - 1), vend = min(2 * (nzc - 1), nz - 1);
  const int tid = threadIdx.x;
  const int k = tid & ((1 << lk) - 1), ch = tid >> lk;
  const int z0 = 1 + ch * rpc;
  const int z1 = min(z0 + rpc, nz - 1);
  if (!(ch >= nch || k >= nk || z0 >= z1)) {
  const int ire = 2 * k, iro = 2 * k + 1;
  const bool e_ok = ire >= 1 && ire <= nr - 2 && k < kr;
  const bool o_ok = iro <= nr - 2 && iro < hend;
  const bool has_b = k + 1 < nrc;
  const int ps = nz * hw, cps = nzc * hwc;
  // coarse (I, k) and (I, k+1): planes ((I+k)&1) and ((I+k+1)&1), slots k>>1 and (k+1)>>1
  auto coarse_pair = [&](int I, double &a, double &b) {
    const int par = (I + k) & 1;
    a = res_pool[eo + par * cps + I * hwc + (k >> 1)];
    b = has_b ? res_pool[eo + (1 - par) * cps + I * hwc + ((k + 1) >> 1)] : 0.0;
  };
  double a = 0.0, b = 0.0, c = 0.0, d = 0.0;
  if ((z0 >> 1) < nzc) coarse_pair(z0 >> 1, a, b);
  for (int iz = z0; iz < z1; ++iz) {
    const bool ze = (iz & 1) == 0;
    const bool row_ok = ze ? ((iz >> 1) < kz) : (iz < vend);
    double ve, vo;
    if (ze) {  // coincident row: (a, b) is coarse row iz/2
      ve = a;
      vo = dmul(0.5, dadd(a, b));
    } else {  // between coarse rows I and I+1
      const int I = iz >> 1;
      if (I + 1 < nzc) coarse_pair(I + 1, c, d);
      ve = dmul(0.5, dadd(a, c));
      vo = dmul(0.25, dadd(dadd(dadd(a, c), b), d));
    }
    if (row_ok) {
      const int e = iz * hw + k;
      if (e_ok) {
        const int p = xo + (iz & 1) * ps + e;  // even column: colour = iz&1
        res_pool[p] = dadd(res_pool[p], ve);
      }
      if (o_ok) {
        const int p = xo + ((iz + 1) & 1) * ps + e;
        res_pool[p] = dadd(res_pool[p], vo);
      }
    }
    if (!ze) {  // the next (even) row coincides with coarse row I+1
      a = c;
      b = d;
    }
  }
  }  // active
}

// Smoother column tables a_e | a_w (nr each): the coarse resident levels keep a copy in the pool so
// per-pass coefficient fetches cost a shared-memory load, not an L2 round trip.  The level
// descriptors themselves are copied to shared memory as well: with ~2.4 KB of kernel parameters the
// per-pass constant-bank reads miss the constant cache.  Returns the pool offset of the descriptors.
__device__ __forceinline__ int res_stage(const RPlan &plan) {
  const int lev_off = plan.pool_doubles;
  const int words = plan.nlev * (int)(sizeof(RLevel) / 8);
  const unsigned long long *src = reinterpret_cast<const unsigned long long *>(&plan.lev[0]);
  unsigned long long *dst = reinterpret_cast<unsigned long long *>(res_pool + lev_off);
  for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
  for (int l = 0; l < plan.nlev; ++l) {
    const RLevel &R = plan.lev[l];
    if (R.t_off < 0) continue;
    for (int i = threadIdx.x; i < 2 * R.nr; i += blockDim.x) res_pool[R.t_off + i] = R.g.a_e[i];
  }
  __syncthreads();
  return lev_off;
}

// Base level with at most 3x3 interior points and a zero wall: 50 sweeps by ONE warp, one lane per
// point, values in registers, neighbours through warp shuffles (no barriers, no shared-memory round
// trips).  Absent points of smaller grids behave as the zero wall.  Same point arithmetic.
static __device__ __noinline__ void res_base_small(int lev_off, int l, double omega, double omw, int sweeps) {
  if (threadIdx.x < 32) {
    const RLevel &B = res_level(lev_off, l);
    const int lane = threadIdx.x;
    const int nz = B.nz, nr = B.nr, hw = B.hw;
    SorK c;
    c.a_ns = B.g.a_ns, c.a_c = B.g.a_c, c.inv_a_c = B.g.inv_a_c, c.omega = omega, c.omw = omw;
    const int i = lane / 3, j = lane - 3 * i;  // interior point (1+i, 1+j)
    const bool on = lane < 9 && (1 + i) <= nz - 2 && (1 + j) <= nr - 2;
    const double ae = on ? res_pool[B.t_off + 1 + j] : 0.0, aw = on ? res_pool[B.t_off + nr + 1 + j] : 0.0;
    const double f = on ? res_pool[B.d_off + split_index(nz, hw, 1 + i, 1 + j)] : 0.0;
    const int x_idx = B.x_off + split_index(nz, hw, 1 + i, 1 + j);
    const int par = (i + j) & 1;
    const bool hasE = on && j < 2, hasW = on && j > 0, hasN = on && i < 2, hasS = on && i > 0;
    double v = 0.0;
    for (int s = 0; s < sweeps; ++s) {
#pragma unroll
      for (int parity = 0; parity < 2; ++parity) {
        const double e = __shfl_sync(0xffffffffu, v, (lane + 1) & 31);
        const double w = __shfl_sync(0xffffffffu, v, (lane + 31) & 31);
        const double n = __shfl_sync(0xffffffffu, v, (lane + 3) & 31);
        const double so = __shfl_sync(0xffffffffu, v, (lane + 29) & 31);
        // S = 1 form of res_update: (W, E) = (c_cur, side)
        const double nv = res_update<1>(c, ae, aw, hasE ? e : 0.0, hasS ? so : 0.0, hasW ? w : 0.0, hasN ? n : 0.0, f, v);
        if (on && par == parity) v = nv;
      }
    }
    if (on) res_pool[x_idx] = v;
  }
  __syncthreads();
}

__device__ __forceinline__ void res_zero_off(int off, int count) {
  for (int i = threadIdx.x; i < count; i += blockDim.x) res_pool[off + i] = 0.0;
}

// One V-cycle over the `nlev` resident levels staged at `lev_off` (multigrid_solve.py:252-335).
// The finest resident level's planes must already be in the pool; its right-hand side `rhs0` is in
// global memory (split layout).  Ends with all threads synchronised.
__device__ __forceinline__ void res_vcycle(int lev_off, int nlev, const double *__restrict__ rhs0, double omega,
                                           int pre, int post) {
  const double omw = 1.0 - omega;
  const int L = nlev;
  GSB_PHASE_BEGIN();
  for (int l = 0; l < L - 1; ++l) {
    int fnz, fnr, cnz, cnr, cx, chw;
    {
      const RLevel &F = res_level(lev_off, l);
      const RLevel &C = res_level(lev_off, l + 1);
      fnz = F.nz, fnr = F.nr, cnz = C.nz, cnr = C.nr, cx = C.x_off, chw = C.hw;
    }
    if (fnz > 2 && fnr > 2) {
      if (l == 0)
        res_smooth<true>(lev_off, l, rhs0, 0, 2 * pre, omega, omw);
      else
        res_smooth<false>(lev_off, l, nullptr, 0, 2 * pre, omega, omw);
    }
    GSB_PHASE(4 * l + 0);  // pre-smooth
    res_zero_off(cx, 2 * cnz * chw);
    if (cnz > 2 && cnr > 2) {
      if (l == 0)
        res_residual_restrict<true>(lev_off, l, rhs0);
      else
        res_residual_restrict<false>(lev_off, l, nullptr);
    }
    __syncthreads();
    GSB_PHASE(4 * l + 1);  // residual + restriction
  }
  {
    int bnz, bnr;
    {
      const RLevel &B = res_level(lev_off, L - 1);
      bnz = B.nz, bnr = B.nr;
    }
    if (bnz > 2 && bnr > 2) {
      if (L > 1 && bnz <= 5 && bnr <= 5)
        res_base_small(lev_off, L - 1, omega, omw, 50);
      else if (L == 1)
        res_smooth<true>(lev_off, 0, rhs0, 0, 100, omega, omw);
      else
        res_smooth<false>(lev_off, L - 1, nullptr, 0, 100, omega, omw);
    }
    GSB_PHASE(4 * (L - 1) + 0);  // base solve
  }
  for (int l = L - 2; l >= 0; --l) {
    int fnz, fnr;
    {
      const RLevel &F = res_level(lev_off, l);
      fnz = F.nz, fnr = F.nr;
    }
    if (fnz > 2 && fnr > 2) {
      res_prolong_add(lev_off, l);
      __syncthreads();
      GSB_PHASE(4 * l + 2);  // prolongation
      if (l == 0)
        res_smooth<true>(lev_off, l, rhs0, 0, 2 * post, omega, omw);
      else
        res_smooth<false>(lev_off, l, nullptr, 0, 2 * post, omega, omw);
      GSB_PHASE(4 * l + 3);  // post-smooth
    }
  }
}

// host: resident plan for levels [l0, end) of ctx; returns false if it does not fit one SM
bool build_rplan(const gsb_ctx *ctx, int l0, int extra_doubles, RPlan *out);

}  // namespace gsb

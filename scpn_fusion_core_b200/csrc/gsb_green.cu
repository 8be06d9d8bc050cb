// gsb_green.cu - Green's-function boundary pieces (SURVEY.md 8a: a15, a16, a18).
//
//  * Cephes ellpk/ellpe in device FP64 (what scipy.special.ellipk/ellipe wrap)
//  * coil -> grid unit tables, batched coil-flux accumulation
//  * coil -> points mutual matrix
//  * lane-C plasma -> wall response matrix and its batched contraction on the FP64 tensor pipe
#include "gsb_internal.cuh"

#include <cstdlib>

namespace gsb {

__constant__ double c_ellpk_P[11] = {
    1.37982864606273237150e-4, 2.28025724005875567385e-3, 7.97404013220415179367e-3,
    9.85821379021226008714e-3, 6.87489687449949877925e-3, 6.18901033637687613229e-3,
    8.79078273952743772254e-3, 1.49380448916805252718e-2, 3.08851465246711995998e-2,
    9.65735902811690126535e-2, 1.38629436111989062502e0};
__constant__ double c_ellpk_Q[11] = {
    2.94078955048598507511e-5, 9.14184723865917226571e-4, 5.94058303753167793257e-3,
    1.54850516649762399335e-2, 2.39089602715924892727e-2, 3.01204715227604046988e-2,
    3.73774314173823228969e-2, 4.88280347570998239232e-2, 7.03124996963957469739e-2,
    1.24999999999870820058e-1, 4.99999999999999999821e-1};
__constant__ double c_ellpe_P[11] = {
    1.53552577301013293365e-4, 2.50888492163602060990e-3, 8.68786816565889628429e-3,
    1.07350949056076193403e-2, 7.77395492516787092951e-3, 7.58395289413514708519e-3,
    1.15688436810574127319e-2, 2.18317996015557253103e-2, 5.68051945617860553470e-2,
    4.43147180560990850618e-1, 1.00000000000000000299e0};
__constant__ double c_ellpe_Q[10] = {
    3.27954898576485872656e-5, 1.00962792679356715133e-3, 6.50609489976927491433e-3,
    1.68862163993311317300e-2, 2.61769742454493659583e-2, 3.34833904888224918614e-2,
    4.27180926518931511717e-2, 5.85936634471101055642e-2, 9.37499997197644278445e-2,
    2.49999999999888314361e-1};

template <int N>
__device__ __forceinline__ double polevl(double x, const double *c) {
  double a = c[0];
#pragma unroll
  for (int i = 1; i < N; ++i) a = dadd(dmul(a, x), c[i]);
  return a;
}
// Cephes ellpk(x), x = 1-m in (MACHEP, 1]:  P(x) - log(x) Q(x)
__device__ __forceinline__ double ellpk_x(double x) {
  return dsub(polevl<11>(x, c_ellpk_P), dmul(log(x), polevl<11>(x, c_ellpk_Q)));
}
// Cephes ellpe(m): x = 1-m;  P(x) - log(x) (x Q(x))
__device__ __forceinline__ double ellpe_x(double x) {
  return dsub(polevl<11>(x, c_ellpe_P), dmul(log(x), dmul(x, polevl<10>(x, c_ellpe_Q))));
}

__device__ __forceinline__ double clipd(double v, double lo, double hi) {
  return fmin(fmax(v, lo), hi);
}

// fusion_kernel.py:236-249: sqrt(R Rc) and ((2-k2)K - 2E)/k with k2 clipped to [1e-12, 1-1e-12]
__device__ __forceinline__ void green_lane_a(double R, double Z, double Rc, double Zc, double &sq,
                                             double &term) {
  const double dZ = dsub(Z, Zc);
  const double rp = dadd(R, Rc);
  const double den = dadd(dmul(rp, rp), dmul(dZ, dZ));
  double k2 = __ddiv_rn(dmul(dmul(4.0, R), Rc), den);
  k2 = clipd(k2, 1e-12, 1.0 - 1e-12);
  const double x = dsub(1.0, k2);
  const double K = ellpk_x(x), E = ellpe_x(x);
  sq = __dsqrt_rn(dmul(R, Rc));
  const double k = __dsqrt_rn(k2);
  term = __ddiv_rn(dsub(dmul(dsub(2.0, k2), K), dmul(2.0, E)), k);
}

// fusion_kernel_free_boundary.py:58-80 (SI, self point -> 0)
__device__ __forceinline__ double green_si(double Ro, double Zo, double Rs, double Zs) {
  const double dr = dsub(Ro, Rs), dz = dsub(Zo, Zs);
  const bool self = dadd(dmul(dr, dr), dmul(dz, dz)) < 1e-24;
  const double rp = dadd(Ro, Rs);
  const double den = dadd(dmul(rp, rp), dmul(dz, dz));
  double k2 = den > 1e-30 ? __ddiv_rn(dmul(dmul(4.0, Ro), Rs), fmax(den, 1e-30)) : 0.0;
  k2 = clipd(k2, 1e-12, 1.0 - 1e-12);
  const double k = __dsqrt_rn(k2);
  const double x = dsub(1.0, k2);
  const double K = ellpk_x(x), E = ellpe_x(x);
  // _MU0 / (2 pi) * sqrt(R_obs R_src), _MU0 = 4e-7*pi
  const double mu0 = 4e-7 * 3.141592653589793;
  const double pref = dmul(__ddiv_rn(mu0, 2.0 * 3.141592653589793), __dsqrt_rn(dmul(Ro, Rs)));
  const double flux = __ddiv_rn(dmul(pref, dsub(dmul(dsub(2.0, k2), K), dmul(2.0, E))), k);
  return self ? 0.0 : flux;
}

// jax_free_boundary_gs.py:70-86 with jax_equilibrium_solver.py:50-123 (lane C)
__device__ __forceinline__ double green_lane_c(double R, double Z, double Rc, double Zc, double pref) {
  const double Rs = fmax(R, 1e-6);
  const double rp = dadd(Rs, Rc), dz = dsub(Z, Zc);
  const double den = dadd(dmul(rp, rp), dmul(dz, dz));
  const double k2 = clipd(__ddiv_rn(dmul(dmul(4.0, Rs), Rc), fmax(den, 1e-30)), 1e-9, 0.999999);
  const double k = __dsqrt_rn(k2);
  const double x = clipd(dsub(1.0, k2), 1.0e-16, 1.0);
  const double lx = log(x);
  const double K = dsub(polevl<11>(x, c_ellpk_P), dmul(lx, polevl<11>(x, c_ellpk_Q)));
  const double E = dsub(polevl<11>(x, c_ellpe_P), dmul(dmul(x, lx), polevl<10>(x, c_ellpe_Q)));
  const double two_k = __ddiv_rn(2.0, k);
  const double v = dmul(dmul(pref, __dsqrt_rn(dmul(Rs, Rc))),
                        dsub(dmul(dsub(two_k, k), K), dmul(two_k, E)));
  return isfinite(v) ? v : 0.0;
}

__global__ void __launch_bounds__(256)
k_green_table(const double *__restrict__ rrow, const double *__restrict__ zax, int nz, int nr,
              const double *__restrict__ coil_rz, int si, double *__restrict__ g) {
  const int c = blockIdx.y;
  const size_t n = (size_t)nz * nr;
  const double Rc = coil_rz[2 * c], Zc = coil_rz[2 * c + 1];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int iz = (int)(i / nr), ir = (int)(i - (size_t)iz * nr);
    if (si) {
      g[(size_t)c * n + i] = green_si(rrow[ir], zax[iz], Rc, Zc);
    } else {
      double sq, term;
      green_lane_a(rrow[ir], zax[iz], Rc, Zc, sq, term);
      g[((size_t)c * 2) * n + i] = sq;
      g[((size_t)c * 2 + 1) * n + i] = term;
    }
  }
}

// psi[b] = sum_c ... accumulated in coil order starting from 0.0 (Psi_vac += ...)
__global__ void __launch_bounds__(256)
k_coil_flux(const double *__restrict__ g, const double *__restrict__ w, int n_coils, size_t n, int si,
            double *__restrict__ psi) {
  const int b = blockIdx.y;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (int c = 0; c < n_coils; ++c) {
      const double wc = w[(size_t)b * n_coils + c];
      if (si)
        acc = dadd(acc, dmul(wc, g[(size_t)c * n + i]));
      else
        acc = dadd(acc, dmul(dmul(wc, g[((size_t)c * 2) * n + i]), g[((size_t)c * 2 + 1) * n + i]));
    }
    psi[(size_t)b * n + i] = acc;
  }
}

__global__ void k_mutual(const double *__restrict__ coil_rz, const int *__restrict__ turns,
                         const double *__restrict__ obs, int n_pts, double *__restrict__ m) {
  const int c = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pts) return;
  const double gval = green_si(obs[2 * i], obs[2 * i + 1], coil_rz[2 * c], coil_rz[2 * c + 1]);
  m[(size_t)c * n_pts + i] = dmul((double)turns[c], gval);
}

// wall ring / interior enumerations in C order (jax_free_boundary_predictive.py:166-180)
__device__ __forceinline__ void wall_coord(int w, int nz, int nr, int &iz, int &ir) {
  if (w < nr) {
    iz = 0;
    ir = w;
  } else if (w >= nr + 2 * (nz - 2)) {
    iz = nz - 1;
    ir = w - (nr + 2 * (nz - 2));
  } else {
    const int t = w - nr;
    iz = 1 + t / 2;
    ir = (t & 1) ? nr - 1 : 0;
  }
}

__global__ void __launch_bounds__(256)
k_wall_matrix(const double *__restrict__ rrow, const double *__restrict__ zax, int nz, int nr,
              double pref, double *__restrict__ m) {
  const int nint = (nz - 2) * (nr - 2);
  const int w = blockIdx.y;
  int wz, wr;
  wall_coord(w, nz, nr, wz, wr);
  const double Rw = rrow[wr], Zw = zax[wz];
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < nint; s += gridDim.x * blockDim.x) {
    const int iz = 1 + s / (nr - 2), ir = 1 + s % (nr - 2);
    m[(size_t)w * nint + s] = green_lane_c(Rw, Zw, rrow[ir], zax[iz], pref);
  }
}

// ------------------------------------------------------------------------------------------
// a18  wall[b][w] = sum_s M[w][s] * (J[b][interior s] * dA)
// C[B x Nw] = X[B x K] * M^T[K x Nw] on the FP64 tensor pipe: mma.sync m8n8k4 f64 (SASS DMMA.8x8x4, the only
// native FP64 MMA shape on sm_100a - the m16n8k{4,8,16} forms compile to sequences of it; tcgen05 has no
// FP64 kind).  The pipe retires one DMMA (512 flop) per ~4 cycles per SM, i.e. 128 flop/clk/SM - the same
// rate as 64 DFMA lanes - so the kernel is about keeping that one pipe fed without bubbles:
//   * persistent stream-K: the (output tile, K tile) space is linearised and cut into gridDim.x equal runs,
//     one CTA per SM, so every SM issues DMMAs from the first to the last cycle (no wave quantisation:
//     256 output tiles of 128x64 over 296 CTA slots cost the previous kernel 14 %).  A tile that is cut
//     writes partial sums; k_wall_reduce adds them in a fixed order (deterministic, no atomics);
//   * CTA tile 128(b) x 128(w) x 16(k), 16 warps of 32x32 (4x4 accumulator fragments: 8 LDS.64 feed 16 DMMA);
//   * operands keep their global K-contiguous layout in shared memory, rows padded to 20 doubles: fragment
//     loads (row = lane/4, k = lane%4) and the 8-byte cp.async fills (16 consecutive k per row) are both
//     bank-conflict free;
//   * 4-stage cp.async pipeline (zero-fill for the ragged last chunk of every grid row and for rows beyond
//     the batch / the wall) with full / empty mbarriers per stage instead of a CTA barrier per K tile
//     (the alternatives measured against this configuration: profiles/r2_wall_gemm.md);
//   * the interior gather is fused into the X-tile addressing: K is walked as (interior row, 16-column
//     chunk), so a K tile never straddles a grid row and needs no per-element index arithmetic; dA is
//     applied to the accumulators.
// ------------------------------------------------------------------------------------------
// Tile configuration: BM(b) x BN(w) x BK, NST cp.async stages, (BM/32) x (BN/32) warps of 32x32, CPS CTAs per SM.
template <int BM_, int BN_, int BK_, int NST_, int CPS_>
struct GemmCfg {
  static constexpr int BM = BM_, BN = BN_, BK = BK_, NST = NST_, CPS = CPS_;
  static constexpr int LD = BK + 4;  // row pitch in doubles: (4*row + k) mod 16 distinct over a half warp -> no bank conflicts
  static constexpr int THREADS = (BM / 32) * (BN / 32) * 32;
  static constexpr int WN = BN / 32;  // warps along w
  static constexpr int STAGE = (BM + BN) * LD;
  static constexpr int SMEM = NST * STAGE * (int)sizeof(double) + 2 * NST * 8;  // + full / empty mbarriers
  static constexpr int RP = THREADS / BK;  // rows filled per loader pass
};

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}
// mbarrier helpers (shared::cta, 32-bit shared addresses)
__device__ __forceinline__ void mbar_init(unsigned bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on `bar` when all cp.async issued so far by this thread have landed (counts as one of the expected arrivals)
__device__ __forceinline__ void mbar_arrive_on_cp_async(unsigned bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}

struct WallGemmArgs {
  const double *M, *J;
  double *out;    // [B][Nw]
  double *part;   // [tile][max_parts][BM*BN] partial sums of tiles cut by the stream-K schedule
  int nz, nr, batch, nwall, nint;
  int ntk;        // K tiles per output tile
  int nwt;        // output tiles along w
  long long total, spc;  // linearised (tile, K tile) steps; steps per CTA
  int max_parts;
  double dA;
};

template <class C>
__global__ void __launch_bounds__(C::THREADS, C::CPS) k_wall_gemm_sk(const WallGemmArgs a) {
  extern __shared__ double gsm[];
  constexpr int BM = C::BM, BN = C::BN, BK = C::BK, LD = C::LD, NST = C::NST, RP = C::RP;
  constexpr int XQ = BM / RP, MQ = BN / RP;  // loader passes per tile
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wb = (warp / C::WN) * 32, ww = (warp % C::WN) * 32;
  const int gid = lane >> 2, tig = lane & 3;
  const int lk = tid % BK, lr = tid / BK;  // loader role: column lk of rows lr, lr+RP, ...
  const int ncol = a.nr - 2, cpr = (ncol + BK - 1) / BK;
  const size_t n = (size_t)a.nz * a.nr;
  const long long s_begin = (long long)blockIdx.x * a.spc, s_end = min(a.total, s_begin + a.spc);
  long long s = s_begin;
  // mbarrier pipeline: full[st] completes when all THREADS loaders' copies of a K tile have landed in stage st,
  // empty[st] when all warps have finished reading it.  A warp refills a stage only one whole K tile after it
  // read it, so warps may drift apart by up to a tile instead of meeting at a CTA barrier every K tile.
  const unsigned bar_full = (unsigned)__cvta_generic_to_shared(gsm + NST * C::STAGE), bar_empty = bar_full + NST * 8;
  unsigned it = 0;  // K tiles consumed by this CTA so far (stage = it % NST, phase parity = (it / NST) & 1)
  if (tid == 0)
    for (int st = 0; st < NST; ++st) mbar_init(bar_full + 8 * st, C::THREADS), mbar_init(bar_empty + 8 * st, C::THREADS / 32);
  __syncthreads();
  while (s < s_end) {
    const int tile = (int)(s / a.ntk), k_lo = (int)(s - (long long)tile * a.ntk);
    const int k_hi = (int)min((long long)a.ntk, k_lo + (s_end - s));
    const int nk = k_hi - k_lo;
    const int b0 = (tile / a.nwt) * BM, w0 = (tile % a.nwt) * BN;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    // Loader, kept lean on purpose: every non-DMMA instruction in this loop costs tensor-pipe time (measured:
    // 40 integer instructions per K tile = 7 %, tools/ubench/dmma_pipe.cu).  Per thread and segment: XQ + MQ
    // byte pointers fixed for the whole segment; per K tile one CTA-uniform byte offset per operand.  Rows
    // beyond the batch / the wall are clamped to the last valid row (their results are never stored), so only
    // the ragged last 16-column chunk of a grid row needs a zero fill, and only on the M side: the X element
    // it meets is the (finite) wall column of J.
    const char *jq[XQ], *mq[MQ];
#pragma unroll
    for (int q = 0; q < XQ; ++q)
      jq[q] = reinterpret_cast<const char *>(a.J + (size_t)min(b0 + lr + RP * q, a.batch - 1) * n + a.nr + 1 + lk);
#pragma unroll
    for (int q = 0; q < MQ; ++q)
      mq[q] = reinterpret_cast<const char *>(a.M + (size_t)min(w0 + lr + RP * q, a.nwall - 1) * a.nint + lk);
    const unsigned s_thread = (unsigned)__cvta_generic_to_shared(gsm + lr * LD + lk);
    int t_row = k_lo / cpr, t_chunk = k_lo - t_row * cpr;  // position of the NEXT K tile to be issued
    auto issue = [&](int stage) {
      const int c0 = t_chunk * BK;
      const bool kok = c0 + lk < ncol;
      const size_t to_j = ((size_t)t_row * a.nr + c0) * sizeof(double);
      const size_t to_m = kok ? ((size_t)t_row * ncol + c0) * sizeof(double) : 0;
      const int msz = kok ? 8 : 0;  // src-size 0: the 8 destination bytes are zero-filled
      const unsigned sx = s_thread + stage * (C::STAGE * (int)sizeof(double));
      const unsigned smm = sx + BM * LD * (int)sizeof(double);
#pragma unroll
      for (int q = 0; q < XQ; ++q)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sx + q * (RP * LD * 8)), "l"(jq[q] + to_j) : "memory");
#pragma unroll
      for (int q = 0; q < MQ; ++q)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smm + q * (RP * LD * 8)), "l"(mq[q] + to_m), "r"(msz)
                     : "memory");
      if (++t_chunk == cpr) t_chunk = 0, ++t_row;
    };
    auto produce = [&](unsigned j) {  // fill stage j % NST with the next K tile (tile number j of this CTA)
      const unsigned sj = j % NST;
      if (j >= (unsigned)NST) mbar_wait(bar_empty + 8 * sj, ((j / NST) & 1) ^ 1);  // its previous tile has been read by all
      issue((int)sj);
      mbar_arrive_on_cp_async(bar_full + 8 * sj);
    };
#pragma unroll
    for (int st = 0; st < NST - 2; ++st)
      if (st < nk) produce(it + st);
    for (int i = 0; i < nk; ++i) {
      const int stage = (int)((it + i) % NST);
      if (i + NST - 2 < nk) produce(it + i + NST - 2);
      mbar_wait(bar_full + 8 * stage, ((it + i) / NST) & 1);
      const double *sX = gsm + stage * C::STAGE, *sM = sX + BM * LD;
#pragma unroll
      for (int ks = 0; ks < BK; ks += 4) {
        double af[4], bf[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) af[u] = sX[(wb + u * 8 + gid) * LD + ks + tig];  // A[row = gid][k = tig]
#pragma unroll
        for (int u = 0; u < 4; ++u) bf[u] = sM[(ww + u * 8 + gid) * LD + ks + tig];  // B[k = tig][col = gid]
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) dmma884(acc[u][v][0], acc[u][v][1], af[u], bf[v]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_empty + 8 * stage);
    }
    it += nk;
    // C fragment: row = gid, cols = 2*tig, 2*tig + 1
    const bool whole = (k_lo == 0 && k_hi == a.ntk);
    if (whole) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const int b = b0 + wb + u * 8 + gid, w = w0 + ww + v * 8 + 2 * tig;
          if (b < a.batch) {
            if (w < a.nwall) a.out[(size_t)b * a.nwall + w] = acc[u][v][0] * a.dA;
            if (w + 1 < a.nwall) a.out[(size_t)b * a.nwall + w + 1] = acc[u][v][1] * a.dA;
          }
        }
    } else {
      const int c_first = (int)(((long long)tile * a.ntk) / a.spc);
      double *pp = a.part + ((size_t)tile * a.max_parts + (blockIdx.x - c_first)) * (BM * BN);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const int lb = wb + u * 8 + gid, lw = ww + v * 8 + 2 * tig;
          *reinterpret_cast<double2 *>(pp + lb * BN + lw) = make_double2(acc[u][v][0], acc[u][v][1]);
        }
    }
    s += nk;
  }
}

// fixed-order sum of the partial tiles (tiles solved by a single CTA were written directly)
__global__ void __launch_bounds__(256) k_wall_reduce(const WallGemmArgs a, int BM, int BN) {
  const int tile = blockIdx.y;
  const int c_first = (int)(((long long)tile * a.ntk) / a.spc);
  const int c_last = (int)(((long long)(tile + 1) * a.ntk - 1) / a.spc);
  const int np = c_last - c_first + 1;
  if (np == 1) return;
  const int b0 = (tile / a.nwt) * BM, w0 = (tile % a.nwt) * BN;
  const double *pp = a.part + (size_t)tile * a.max_parts * (BM * BN);
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < BM * BN; e += gridDim.x * blockDim.x) {
    const int b = b0 + e / BN, w = w0 + e % BN;
    if (b >= a.batch || w >= a.nwall) continue;
    double sum = pp[e];
    for (int p = 1; p < np; ++p) sum += pp[(size_t)p * (BM * BN) + e];
    a.out[(size_t)b * a.nwall + w] = sum * a.dA;
  }
}

__global__ void k_wall_scatter(const double *__restrict__ wall, double *__restrict__ bc, int nz, int nr,
                               int nwall, int accumulate) {
  const int b = blockIdx.y;
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nwall) return;
  int iz, ir;
  wall_coord(w, nz, nr, iz, ir);
  double *p = bc + (size_t)b * nz * nr + (size_t)iz * nr + ir;
  const double v = wall[(size_t)b * nwall + w];
  p[0] = accumulate ? p[0] + v : v;
}

}  // namespace gsb

using namespace gsb;

template <class C>
static int wall_gemm_launch(gsb_ctx *ctx, WallGemmArgs a, cudaStream_t st) {
  const int cpr = (ctx->nr - 2 + C::BK - 1) / C::BK;
  a.ntk = (ctx->nz - 2) * cpr;
  a.nwt = (a.nwall + C::BN - 1) / C::BN;
  const int n_tiles = ((a.batch + C::BM - 1) / C::BM) * a.nwt;
  a.total = (long long)n_tiles * a.ntk;
  const int grid = (int)std::min<long long>((long long)ctx->num_sms * C::CPS, a.total);
  a.spc = (a.total + grid - 1) / grid;
  a.max_parts = (int)((a.ntk + a.spc - 1) / a.spc) + 1;
  const size_t need = (size_t)n_tiles * a.max_parts * C::BM * C::BN * sizeof(double);
  if (ctx->gemm_ws_bytes < need) {  // grow-only workspace: no allocation in steady state
    if (ctx->gemm_ws) GSB_CUDA(cudaFree(ctx->gemm_ws));
    ctx->gemm_ws = nullptr;
    ctx->gemm_ws_bytes = 0;
    GSB_CUDA(cudaMalloc(&ctx->gemm_ws, need));
    ctx->gemm_ws_bytes = need;
  }
  a.part = ctx->gemm_ws;
  GSB_SMEM_OPT_IN(k_wall_gemm_sk<C>, C::SMEM);
  k_wall_gemm_sk<C><<<grid, C::THREADS, C::SMEM, st>>>(a);
  GSB_LAUNCH_CHECK();
  if (a.spc % a.ntk != 0) {  // the runs do not end on tile boundaries: some tiles are cut
    k_wall_reduce<<<dim3(16, n_tiles), 256, 0, st>>>(a, C::BM, C::BN);
    GSB_LAUNCH_CHECK();
  }
  return GSB_OK;
}

extern "C" {

int gsb_green_table(gsb_ctx *ctx, const double *coil_rz, int n_coils, int si, double *g_dev, void *stream) {
  GSB_REQUIRE(ctx && coil_rz && g_dev, "gsb_green_table: NULL argument");
  GSB_REQUIRE(n_coils >= 1 && n_coils <= 65535, "gsb_green_table: bad coil count");
  GSB_REQUIRE((int)ctx->z_axis.size() == ctx->nz, "gsb_green_table: context was created without a z axis");
  GSB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  double *crz = nullptr;
  GSB_CUDA(cudaMalloc(&crz, 2 * n_coils * sizeof(double)));
  cudaError_t e = cudaMemcpyAsync(crz, coil_rz, 2 * n_coils * sizeof(double), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    const int blocks = (int)std::min<size_t>((ctx->n + 255) / 256, 1024);
    k_green_table<<<dim3(blocks, n_coils), 256, 0, st>>>(ctx->r_dev, ctx->z_dev, ctx->nz, ctx->nr, crz, si, g_dev);
    g_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(crz);
  if (e != cudaSuccess) {
    set_error(std::string("gsb_green_table: ") + cudaGetErrorString(e));
    return GSB_ECUDA;
  }
  return GSB_OK;
}

int gsb_coil_flux(gsb_ctx *ctx, const double *g_dev, const double *w_dev, int n_coils, int si,
                  double *psi_dev, int batch, void *stream) {
  GSB_REQUIRE(ctx && g_dev && w_dev && psi_dev, "gsb_coil_flux: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= 65535 && n_coils >= 1, "gsb_coil_flux: bad sizes");
  GSB_CUDA(cudaSetDevice(ctx->device));
  const int blocks = (int)std::min<size_t>((ctx->n + 255) / 256, 256);
  k_coil_flux<<<dim3(blocks, batch), 256, 0, (cudaStream_t)stream>>>(g_dev, w_dev, n_coils, ctx->n, si, psi_dev);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_mutual_matrix(const double *coil_rz, const int *turns, int n_coils, const double *obs_rz, int n_pts,
                      double *m_dev, void *stream) {
  GSB_REQUIRE(coil_rz && turns && obs_rz && m_dev, "gsb_mutual_matrix: NULL argument");
  GSB_REQUIRE(n_coils >= 1 && n_coils <= 65535 && n_pts >= 1, "gsb_mutual_matrix: bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  double *crz = nullptr, *obs = nullptr;
  int *tr = nullptr;
  cudaError_t e = cudaMalloc(&crz, 2 * n_coils * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&obs, 2 * (size_t)n_pts * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&tr, n_coils * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpyAsync(crz, coil_rz, 2 * n_coils * sizeof(double), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(obs, obs_rz, 2 * (size_t)n_pts * sizeof(double), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(tr, turns, n_coils * sizeof(int), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    k_mutual<<<dim3((n_pts + 127) / 128, n_coils), 128, 0, st>>>(crz, tr, obs, n_pts, m_dev);
    g_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(crz);
  cudaFree(obs);
  cudaFree(tr);
  if (e != cudaSuccess) {
    set_error(std::string("gsb_mutual_matrix: ") + cudaGetErrorString(e));
    return GSB_ECUDA;
  }
  return GSB_OK;
}

int gsb_wall_matrix(gsb_ctx *ctx, double mu0, double *m_dev, void *stream) {
  GSB_REQUIRE(ctx && m_dev, "gsb_wall_matrix: NULL argument");
  GSB_REQUIRE((int)ctx->z_axis.size() == ctx->nz, "gsb_wall_matrix: context was created without a z axis");
  GSB_REQUIRE(ctx->nz >= 3 && ctx->nr >= 3, "gsb_wall_matrix: grid has no interior");
  GSB_CUDA(cudaSetDevice(ctx->device));
  volatile double pref = mu0 * 1.0;
  volatile double pref2 = pref / (2.0 * 3.141592653589793);
  const int blocks = std::min((ctx->n_int + 255) / 256, 64);
  k_wall_matrix<<<dim3(blocks, ctx->n_wall), 256, 0, (cudaStream_t)stream>>>(ctx->r_dev, ctx->z_dev, ctx->nz, ctx->nr, pref2, m_dev);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

int gsb_wall_flux(gsb_ctx *ctx, const double *m_dev, const double *jphi_dev, double dA, double *wall_dev,
                  int batch, void *stream) {
  GSB_REQUIRE(ctx && m_dev && jphi_dev && wall_dev, "gsb_wall_flux: NULL argument");
  GSB_REQUIRE(batch >= 1, "gsb_wall_flux: bad batch");
  GSB_REQUIRE(ctx->nz >= 3 && ctx->nr >= 3, "gsb_wall_flux: grid has no interior");
  GSB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  WallGemmArgs a{};
  a.M = m_dev;
  a.J = jphi_dev;
  a.out = wall_dev;
  a.nz = ctx->nz, a.nr = ctx->nr, a.batch = batch, a.nwall = ctx->n_wall, a.nint = ctx->n_int;
  a.dA = dA;
  // 128x128x16 tiles, 4 stages, one CTA per SM: the fastest of the configurations in profiles/r2_wall_gemm.md
  return wall_gemm_launch<GemmCfg<128, 128, 16, 4, 1>>(ctx, a, st);
}

int gsb_wall_scatter(gsb_ctx *ctx, const double *wall_dev, double *bc_dev, int accumulate, int batch, void *stream) {
  GSB_REQUIRE(ctx && wall_dev && bc_dev, "gsb_wall_scatter: NULL argument");
  GSB_REQUIRE(batch >= 1 && batch <= 65535, "gsb_wall_scatter: bad batch");
  GSB_CUDA(cudaSetDevice(ctx->device));
  k_wall_scatter<<<dim3((ctx->n_wall + 127) / 128, batch), 128, 0, (cudaStream_t)stream>>>(
      wall_dev, bc_dev, ctx->nz, ctx->nr, ctx->n_wall, accumulate);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

}  // extern "C"

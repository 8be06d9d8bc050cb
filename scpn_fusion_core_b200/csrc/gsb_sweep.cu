// gsb_sweep.cu - temporally blocked streaming RB-SOR: S full sweeps (2S colour passes) of mg_smooth
// (multigrid_solve.py:148-208) in ONE pass over HBM; and the same for T Jacobi steps (k_jacobi_warp, the Picard seed).
//
// The per-colour streaming kernel (k_smooth_colour) moves psi twice and the source once per
// colour pass: 48 B of DRAM traffic per point per sweep for 24 algorithmic bytes.  Here every WARP
// owns a 64-column strip of one row band of one equilibrium and marches down the rows on its own:
// no CTA barrier anywhere, only __syncwarp; lane k holds the column pair (2k, 2k+1).  Colour pass t
// (= stage t) works two rows behind pass t-1, so the 2S stages of a step are mutually independent:
//   stage t at row r = i - 2t reads rows r-1, r, r+1: pass t-1 finished r+1 one step earlier, and
//   pass t+1 (row r-2) touches nothing stage t reads;
// a lane therefore gathers the operands of all 2S stages, computes 2S independent updates (ILP = 2S
// hides the FP64 latency) and hands them on, once per row step.
// Strips/bands overlap by 2S columns/rows; the overlap is recomputed (an update is valid t+1 points
// inside the tile edge after pass t) and only tile interiors are written, so with more than one
// tile per equilibrium the sweep is out of place (neighbours read each other's interiors).
// The body, sweep_warp_body_rc, carries the lane's own values in registers; the shared-memory ring (rows as two half
// rows, even / odd columns, filled by cp.async) is the landing zone of the row copies and the neighbour mailbox.
// Arithmetic: the same operand order as sor_point (bit-identical results).  History and captures, including the form
// that read every operand from the ring (bit-identical, 1.4-1.7x slower): profiles/r2_sweep_icache.md.
#include "gsb_internal.cuh"

namespace gsb {

constexpr int kSwCols = 64;  // columns per warp strip (2 per lane)
constexpr int kSwWPC = 4;    // warps per CTA (independent of each other)

struct SweepArgs {
  int nz, nr;               // array shape (local rows incl. halo rows in slab mode)
  int par_off;              // added to the local row index for the colour parity (global row offset)
  int band_rows, n_strips, n_bands;  // tile plan
  const double *in;
  double *out;
  const double *src;
  size_t istride, ostride, sstride;
  const double *a_e, *a_w;  // [nr] column tables
  double a_ns, a_c, inv_a_c, omega, omw;
  const int *active;
};

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// 32-bit shared-window accesses (the ring addresses rotate through registers, so the compiler could not prove the
// address space of a generic pointer).  asm volatile keeps the program order of ring reads and writes.
__device__ __forceinline__ double lds64(unsigned a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts64_if(bool p, unsigned a, double v) {  // predicated store, no branch
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, 0;\n\t@p st.shared.f64 [%0], %1;\n\t}" ::"r"(a), "d"(v), "r"((int)p));
}
__device__ __forceinline__ void cp_async8s(unsigned s, const void *gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}

// One warp, one tile, register-carried (the "register blocking" of the smoother).  P0 = (zl + par_off + cl) & 1 of the
// tile, hoisted into a template parameter by the dispatching kernel below, keeps every colour parity in the unrolled
// loop body a compile-time constant.  A lane owns the column pair (2k, 2k+1) of the strip, and of the five neighbours
// of an update only ONE belongs to another lane (west of the even column / east of the odd one); everything else the
// same lane produced itself a few steps earlier:
//   stage t at step qi updates (row q = qi - 2t, half hx):   K_t(qi) := the point's value afterwards (V, or O if masked)
//     N     = (q+1, hx)    = K_{t-1}(qi-1)        S = (q-1, hx) = K_{t-1}(qi-3)
//     own W/E = (q, 1-hx)  = K_{t-1}(qi-2)        O = (q, hx)   = K_{t-2}(qi-4)      F = source(q, hx) = F_{t-2}(qi-4)
//   stage 0 reads fresh input: a(qi) = in(qi+1, hx) and b(qi) = in(qi, hx) cover every input point exactly once, and
//     its own W/E = a(qi-1), S = a(qi-2);  stage 1's O = a(qi-3).
// With the step loop unrolled by 4 every carried value has a fixed register name (index = step & 3), so the ring in
// shared memory is only the landing zone of the asynchronous row copies and the mailbox for the one neighbour value:
// 10 shared loads + 5 stores per step instead of the 42 + 6 of reading every operand from the ring (which ran the
// shared-memory pipe at 74 %, profiles/r2_sweep_icache.md), and finished rows go from registers straight to global
// memory.  The loop is unrolled by 4 steps, not over the whole 16-row ring period (that body missed the instruction
// cache), so the sixteen slot addresses live in sixteen registers that rotate by UNR after every loop body.
template <int NST, int P0>
__device__ __forceinline__ void sweep_warp_body_rc(const SweepArgs &a, double *ring, int lane, int zl,
                                                   int zh, int z0, int z1, int cl, int wb, int c0, int c1,
                                                   const double *gin, const double *gsrc, double *gout) {
  constexpr int NRING = 16;
  constexpr int PF = NRING - 2 * NST;
  constexpr int UNR = 4;
  constexpr int L = NST - 1;  // last stage
  constexpr unsigned SLOT = 64 * 8, HALF = 32 * 8, SRC = NRING * SLOT;
  const int nr = a.nr;
  const int xe = 2 * lane, xo = 2 * lane + 1;
  const bool have_e = xe < wb, have_o = xo < wb;
  const bool upd_e = xe >= 1 && xe <= wb - 2, upd_o = xo <= wb - 2;
  const bool wr_e = have_e && cl + xe >= c0 && cl + xe < c1, wr_o = have_o && cl + xo >= c0 && cl + xo < c1;
  const double ae_e = have_e ? a.a_e[cl + xe] : 0.0, aw_e = have_e ? a.a_w[cl + xe] : 0.0;
  const double ae_o = have_o ? a.a_e[cl + xo] : 0.0, aw_o = have_o ? a.a_w[cl + xo] : 0.0;
  const double a_ns = a.a_ns, a_c = a.a_c, inv_a_c = a.inv_a_c, omega = a.omega, omw = a.omw;
  const unsigned rb = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)lane * 8u;
  const int nrows = zh - zl;
  const size_t rowb = (size_t)nr * sizeof(double);

  auto load_row = [&](bool row_ok, unsigned sa, const char *pr, const char *sr) {
    if (row_ok) {
      if (have_e) {
        cp_async8s(sa, pr);
        cp_async8s(sa + SRC, sr);
      }
      if (have_o) {
        cp_async8s(sa + HALF, pr + 8);
        cp_async8s(sa + SRC + HALF, sr + 8);
      }
    }
    cp_async_commit();
  };
  const char *pin = (const char *)(gin + (size_t)zl * nr + cl + xe);
  const char *psr = (const char *)(gsrc + (size_t)zl * nr + cl + xe);
#pragma unroll
  for (int q = 0; q < PF; ++q) load_row(q < nrows, rb + q * SLOT, pin + q * rowb, psr + q * rowb);
  pin += (size_t)PF * rowb;  // the row step qi = 0 prefetches
  psr += (size_t)PF * rowb;
  cp_async_wait<PF - 2>();  // rows 0 and 1 have landed
  __syncwarp();

  unsigned A[NRING];  // A[i]: slot of relative row base - 11 + i
#pragma unroll
  for (int i = 0; i < NRING; ++i) A[i] = rb + ((i + 5) & (NRING - 1)) * SLOT;
  char *pout = (char *)(gout + cl + xe) + ((ptrdiff_t)zl - 2 * L) * (ptrdiff_t)rowb;  // row written at step 0
  const unsigned w_lo = (unsigned)(z0 - zl + 2 * L), w_n = (unsigned)(z1 - z0);
  const unsigned q_hi = (unsigned)(nrows - 3);
  const int q_end = (nrows - 1) + 2 * L;  // the last loaded row leaves the last stage at this step
  double K[NST][UNR], Fc[NST][UNR], A4[UNR];
#pragma unroll
  for (int t = 0; t < NST; ++t)
#pragma unroll
    for (int i = 0; i < UNR; ++i) K[t][i] = Fc[t][i] = 0.0;
#pragma unroll
  for (int i = 0; i < UNR; ++i) A4[i] = 0.0;
  // a(-1) = in(0, 1 - P0): the half of row 0 that no step loads (a(qi) covers rows >= 1, b(0) the other half of row 0)
  A4[UNR - 1] = lds64(rb + (1 - P0) * HALF);

  for (int base = 0; base <= q_end; base += UNR) {
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int qi = base + u;
      if (qi <= q_end) {
        constexpr int M = UNR - 1;
        double Wv[NST], Ev[NST], Sv[NST], Nv[NST], Ov[NST], Fv[NST], own[NST];
        // ---- shared-memory reads: the neighbour lane's value for every stage, fresh input for stage 0, sources
#pragma unroll
        for (int t = 0; t < NST; ++t) {
          const int hx = (t + u + P0) & 1;
          const unsigned row = A[(11 + u - 2 * t) & (NRING - 1)];
          const double nb = lds64(hx ? row + 8 : row + HALF - 8);  // east of the odd column / west of the even one
          if (t == 0) {
            Ov[0] = lds64(row + hx * HALF);                                        // b(qi)
            Nv[0] = lds64(A[(12 + u) & (NRING - 1)] + hx * HALF);                  // a(qi)
            own[0] = A4[(u - 1) & M];
            Sv[0] = A4[(u - 2) & M];
            Fv[0] = lds64(row + hx * HALF + SRC);
          } else {
            Nv[t] = K[t - 1][(u - 1) & M];
            own[t] = K[t - 1][(u - 2) & M];
            Sv[t] = K[t - 1][(u - 3) & M];
            if (t == 1) {
              Ov[1] = A4[(u - 3) & M];
              Fv[1] = lds64(row + hx * HALF + SRC);
            } else {
              Ov[t] = K[t - 2][u & M];
              Fv[t] = Fc[t - 2][u & M];
            }
          }
          Wv[t] = hx ? own[t] : nb;
          Ev[t] = hx ? nb : own[t];
        }
        A4[u & M] = Nv[0];
        // ---- 2S independent updates
        double Kn[NST];
#pragma unroll
        for (int t = NST - 1; t >= 0; --t) {  // last stage first: stage t+2 has consumed K[t][u] before stage t renews it
          const int hx = (t + u + P0) & 1;
          double acc = dadd(dmul(hx ? ae_o : ae_e, Ev[t]), dmul(hx ? aw_o : aw_e, Wv[t]));
          acc = dadd(acc, dmul(a_ns, Sv[t]));
          acc = dadd(acc, dmul(a_ns, Nv[t]));
          acc = dsub(acc, Fv[t]);
          const double qq = __dmul_rn(acc, inv_a_c);
          const double gs = __fma_rn(__fma_rn(-a_c, qq, acc), inv_a_c, qq);  // acc / a_c (Markstein sequence, gsb_internal.cuh)
          const double V = dadd(dmul(omw, Ov[t]), dmul(omega, gs));
          const bool on = ((unsigned)(qi - 2 * t - 1) <= q_hi) && (hx ? upd_o : upd_e);
          Kn[t] = on ? V : Ov[t];
          if (t < L) sts64_if(on, A[(11 + u - 2 * t) & (NRING - 1)] + hx * HALF, V);  // mailbox for the neighbour lane
        }
#pragma unroll
        for (int t = 0; t < NST; ++t) {
          K[t][u & M] = Kn[t];
          Fc[t][u & M] = Fv[t];
        }
        load_row(qi + PF < nrows, A[(11 + u + PF) & (NRING - 1)], pin, psr);
        pin += rowb;
        psr += rowb;
        cp_async_wait<PF - 2>();  // row qi+2 has landed (stage 0 of the next step reads it)
        __syncwarp();
        // ---- relative row qi - 2L is final: both halves are in registers
        if ((unsigned)qi - w_lo < w_n) {
          const int hxl = (L + u + P0) & 1;
          const double ve = hxl ? own[L] : Kn[L], vo = hxl ? Kn[L] : own[L];
          if (wr_e) *(double *)pout = ve;
          if (wr_o) *(double *)(pout + 8) = vo;
        }
        pout += rowb;
      }
    }
    unsigned hd[UNR];
#pragma unroll
    for (int i = 0; i < UNR; ++i) hd[i] = A[i];
#pragma unroll
    for (int i = 0; i + UNR < NRING; ++i) A[i] = A[i + UNR];
#pragma unroll
    for (int i = 0; i < UNR; ++i) A[NRING - UNR + i] = hd[i];
  }
  if (gout != gin) {
    for (int w = z0; w < z1; ++w) {
      if (w >= zl + 1 && w <= zh - 2) continue;
      const double *irow = gin + (size_t)w * nr + cl;
      double *orow = gout + (size_t)w * nr + cl;
      if (wr_e) orow[xe] = irow[xe];
      if (wr_o) orow[xo] = irow[xo];
    }
  }
}

template <int NST>
__global__ void __launch_bounds__(32 * kSwWPC) k_sweep_warp(const SweepArgs a) {
  constexpr int NRING = 16;
  constexpr int STEP = kSwCols - 2 * NST;  // interior columns per strip (even)
  extern __shared__ double sw_pool[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  // per warp: psi ring [NRING][2][32] followed by the source ring [NRING][2][32].  (Edge lanes read one element
  // outside their half row - the neighbouring half row of the same slot - and never use it.)
  double *ring = sw_pool + wid * (2 * NRING * kSwCols);
  const int b = blockIdx.z;
  if (a.active && !a.active[b]) return;
  // (strip, band) tiles are numbered linearly and dealt four to a CTA, so CTAs are full whatever the strip count
  // (257 columns = 5 strips used to leave 3 of every 8 warp slots empty)
  const int tile = blockIdx.x * kSwWPC + wid;
  if (tile >= a.n_strips * a.n_bands) return;  // warps never synchronise with each other
  const int band = tile / a.n_strips, strip = tile - band * a.n_strips;
  const int nz = a.nz, nr = a.nr;
  // tile: interior rows [z0,z1) x cols [c0,c1); loaded rows [zl,zh) x cols [cl,ch)
  const int z0 = band * a.band_rows, z1 = min(nz, z0 + a.band_rows);
  const int c0 = strip * STEP, c1 = (a.n_strips == 1) ? nr : min(nr, c0 + STEP);  // one strip: nr <= 64
  const int zl = max(0, z0 - NST), zh = min(nz, z1 + NST);
  const int cl = max(0, c0 - NST), ch = min(nr, cl + kSwCols);  // cl is even (STEP and NST are)
  const int wb = ch - cl;
  const double *gin = a.in + (size_t)b * a.istride;
  const double *gsrc = a.src + (size_t)b * a.sstride;
  double *gout = a.out + (size_t)b * a.ostride;
  if ((zl + a.par_off + cl) & 1)
    sweep_warp_body_rc<NST, 1>(a, ring, lane, zl, zh, z0, z1, cl, wb, c0, c1, gin, gsrc, gout);
  else
    sweep_warp_body_rc<NST, 0>(a, ring, lane, zl, zh, z0, z1, cl, wb, c0, c1, gin, gsrc, gout);
}

// ------------------------------------------------------------------------------------------
// Temporally blocked Jacobi: T steps of _jacobi_step (fusion_kernel_iterative_solver.py:54-95; sanitised inputs, clipped
// output, walls = sanitised copy) in ONE pass over HBM, register-carried like sweep_warp_body_rc.  The Picard seed is 50
// of these steps per solve; one step per launch (k_jacobi) moved 24 B per point per step at 1.25 TB/s.
//   stage t at step qi produces level t+1 of row q = qi - 2t, both of the lane's columns:
//     N = K_{t-1}(qi-1), C = K_{t-1}(qi-2) (the row itself: O of a masked point, E of the even / W of the odd column),
//     S = K_{t-1}(qi-3), source = F_{t-1}(qi-2); west of the even column / east of the odd one come from the neighbour
//     lanes through the shared-memory ring (mailbox), which stage t then overwrites with its own level.
//   Carried values of the inner stages are kept SANITISED (what the next step's _sanitize_numeric_array makes of them);
//   the last stage writes its raw result (np.clip propagates NaN).
// Branch-free forms of sanitize / clip_cap (gsb_internal.cuh): same results, no slow-path code in the unrolled body.
__device__ __forceinline__ double sanitize_bf(double v) {  // NaN -> 0, +-inf and out-of-range -> +-cap
  const double r = (fabs(v) <= kCap) ? v : copysign(kCap, v);
  return (v != v) ? 0.0 : r;
}
__device__ __forceinline__ double clip_cap_bf(double v) {  // np.clip: NaN stays NaN
  return (fabs(v) <= kCap || v != v) ? v : copysign(kCap, v);
}

template <int T>
__device__ __forceinline__ void jacobi_warp_body(const SweepArgs &a, double *ring, int lane, int zl, int zh, int z0,
                                                 int z1, int cl, int wb, int c0, int c1, const double *gin,
                                                 const double *gsrc, double *gout) {
  constexpr int NRING = 16;
  constexpr int PF = 5;  // rows qi-2(T-1) .. qi+PF live: 2T-1+PF <= 16
  static_assert(2 * T - 1 + PF <= NRING && T >= 1, "ring too small");
  constexpr int UNR = 4, M = UNR - 1;
  constexpr int L = T - 1;
  constexpr unsigned SLOT = 64 * 8, HALF = 32 * 8, SRC = NRING * SLOT;
  const int nr = a.nr;
  const int xe = 2 * lane, xo = 2 * lane + 1;
  const bool have_e = xe < wb, have_o = xo < wb;
  const bool upd_e = xe >= 1 && xe <= wb - 2, upd_o = xo <= wb - 2;
  const bool wr_e = have_e && cl + xe >= c0 && cl + xe < c1, wr_o = have_o && cl + xo >= c0 && cl + xo < c1;
  const double ae_e = have_e ? a.a_e[cl + xe] : 0.0, aw_e = have_e ? a.a_w[cl + xe] : 0.0;
  const double ae_o = have_o ? a.a_e[cl + xo] : 0.0, aw_o = have_o ? a.a_w[cl + xo] : 0.0;
  const double a_ns = a.a_ns, a_c = a.a_c, inv_a_c = a.inv_a_c;
  const unsigned rb = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)lane * 8u;
  const int nrows = zh - zl;
  const size_t rowb = (size_t)nr * sizeof(double);

  auto load_row = [&](bool row_ok, unsigned sa, const char *pr, const char *sr) {
    if (row_ok) {
      if (have_e) {
        cp_async8s(sa, pr);
        cp_async8s(sa + SRC, sr);
      }
      if (have_o) {
        cp_async8s(sa + HALF, pr + 8);
        cp_async8s(sa + SRC + HALF, sr + 8);
      }
    }
    cp_async_commit();
  };
  const char *pin = (const char *)(gin + (size_t)zl * nr + cl + xe);
  const char *psr = (const char *)(gsrc + (size_t)zl * nr + cl + xe);
#pragma unroll
  for (int q = 0; q < PF; ++q) load_row(q < nrows, rb + q * SLOT, pin + q * rowb, psr + q * rowb);
  pin += (size_t)PF * rowb;
  psr += (size_t)PF * rowb;
  cp_async_wait<PF - 2>();  // rows 0 and 1 have landed
  __syncwarp();

  unsigned A[NRING];  // A[i]: slot of relative row base - 11 + i
#pragma unroll
  for (int i = 0; i < NRING; ++i) A[i] = rb + ((i + 5) & (NRING - 1)) * SLOT;
  char *pout = (char *)(gout + cl + xe) + ((ptrdiff_t)zl - 2 * L) * (ptrdiff_t)rowb;  // row written at step 0
  const unsigned w_lo = (unsigned)(z0 - zl + 2 * L), w_n = (unsigned)(z1 - z0);
  const unsigned q_hi = (unsigned)(nrows - 3);
  const int q_end = (nrows - 1) + 2 * L;
  // level-t values of the lane's two columns for the last four rows stage t handled, and their sources
  // (the last stage's values are not carried: nothing consumes them; sources are consumed two steps later only)
  constexpr int TC = T > 1 ? T - 1 : 1;
  double Ke[TC][UNR], Ko[TC][UNR], Fe[TC][2], Fo[TC][2], Ae[UNR], Ao[UNR];
#pragma unroll
  for (int t = 0; t < TC; ++t) {
#pragma unroll
    for (int i = 0; i < UNR; ++i) Ke[t][i] = Ko[t][i] = 0.0;
    Fe[t][0] = Fe[t][1] = Fo[t][0] = Fo[t][1] = 0.0;
  }
#pragma unroll
  for (int i = 0; i < UNR; ++i) Ae[i] = Ao[i] = 0.0;
  Ae[UNR - 1] = sanitize_bf(lds64(rb));  // a(-1) = in(0, .): stage 0 sees row 0 as "the row itself" at step 0
  Ao[UNR - 1] = sanitize_bf(lds64(rb + HALF));

  for (int base = 0; base <= q_end; base += UNR) {
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int qi = base + u;
      if (qi <= q_end) {
        double nbW[T], nbE[T];
        // ---- shared-memory reads: neighbour lanes' values of every stage's row, fresh input row qi+1, source row qi
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const unsigned row = A[(11 + u - 2 * t) & (NRING - 1)];
          nbW[t] = lds64(row + HALF - 8);  // lane-1's odd column
          nbE[t] = lds64(row + 8);         // lane+1's even column
        }
        nbW[0] = sanitize_bf(nbW[0]);  // stage 0 reads raw input; the mailbox values of later stages are sanitised
        nbE[0] = sanitize_bf(nbE[0]);
        const unsigned row0 = A[(11 + u) & (NRING - 1)], row1 = A[(12 + u) & (NRING - 1)];
        const double a_e_new = sanitize_bf(lds64(row1)), a_o_new = sanitize_bf(lds64(row1 + HALF));
        const double f_e_new = sanitize_bf(lds64(row0 + SRC)), f_o_new = sanitize_bf(lds64(row0 + SRC + HALF));
        __syncwarp();  // every lane has read the mailbox rows before any lane overwrites them below
        double Kne[T], Kno[T], Fne[T], Fno[T];
#pragma unroll
        for (int t = T - 1; t >= 0; --t) {
          double Ce, Co, Se, So, Ne, No, fe, fo;
          if (t == 0) {
            Ne = a_e_new;
            No = a_o_new;
            Ce = Ae[(u - 1) & M];
            Co = Ao[(u - 1) & M];
            Se = Ae[(u - 2) & M];
            So = Ao[(u - 2) & M];
            fe = f_e_new;
            fo = f_o_new;
          } else {
            Ne = Ke[t - 1][(u - 1) & M];
            No = Ko[t - 1][(u - 1) & M];
            Ce = Ke[t - 1][(u - 2) & M];
            Co = Ko[t - 1][(u - 2) & M];
            Se = Ke[t - 1][(u - 3) & M];
            So = Ko[t - 1][(u - 3) & M];
            fe = Fe[t - 1][u & 1];  // written two steps ago
            fo = Fo[t - 1][u & 1];
          }
          // even column: E = own odd column, W = neighbour; odd column: W = own even column, E = neighbour
          double acc = dadd(dmul(ae_e, Co), dmul(aw_e, nbW[t]));
          acc = dadd(acc, dmul(a_ns, Se));
          acc = dadd(acc, dmul(a_ns, Ne));
          acc = dsub(acc, fe);
          const double qe = ddiv_y(acc, a_c, inv_a_c);
          acc = dadd(dmul(ae_o, nbE[t]), dmul(aw_o, Ce));
          acc = dadd(acc, dmul(a_ns, So));
          acc = dadd(acc, dmul(a_ns, No));
          acc = dsub(acc, fo);
          const double qo = ddiv_y(acc, a_c, inv_a_c);
          const bool on_row = (unsigned)(qi - 2 * t - 1) <= q_hi;
          // inner level: clip, then what the next step's sanitiser makes of it (= sanitize of the quotient); the last
          // level keeps np.clip's NaN.  Masked points copy the (already sanitised) value of the level below.
          const double ve = t < L ? sanitize_bf(qe) : clip_cap_bf(qe), vo = t < L ? sanitize_bf(qo) : clip_cap_bf(qo);
          const double ke = (on_row && upd_e) ? ve : Ce, ko = (on_row && upd_o) ? vo : Co;
          if (t < L) {  // mailbox for the neighbour lanes
            const bool row_in = (unsigned)(qi - 2 * t) < (unsigned)nrows;
            const unsigned row = A[(11 + u - 2 * t) & (NRING - 1)];
            sts64_if(row_in && have_e, row, ke);
            sts64_if(row_in && have_o, row + HALF, ko);
          }
          Kne[t] = ke;
          Kno[t] = ko;
          Fne[t] = fe;
          Fno[t] = fo;
        }
#pragma unroll
        for (int t = 0; t < L; ++t) {
          Ke[t][u & M] = Kne[t];
          Ko[t][u & M] = Kno[t];
          Fe[t][u & 1] = Fne[t];
          Fo[t][u & 1] = Fno[t];
        }
        Ae[u & M] = a_e_new;
        Ao[u & M] = a_o_new;
        load_row(qi + PF < nrows, A[(11 + u + PF) & (NRING - 1)], pin, psr);
        pin += rowb;
        psr += rowb;
        cp_async_wait<PF - 2>();  // row qi+2 has landed (the next step reads it as its fresh row)
        __syncwarp();
        if ((unsigned)qi - w_lo < w_n) {  // relative row qi - 2L has passed the last stage
          if (wr_e) *(double *)pout = Kne[L];
          if (wr_o) *(double *)(pout + 8) = Kno[L];
        }
        pout += rowb;
      }
    }
    unsigned hd[UNR];
#pragma unroll
    for (int i = 0; i < UNR; ++i) hd[i] = A[i];
#pragma unroll
    for (int i = 0; i + UNR < NRING; ++i) A[i] = A[i + UNR];
#pragma unroll
    for (int i = 0; i < UNR; ++i) A[NRING - UNR + i] = hd[i];
  }
}

template <int T>
__global__ void __launch_bounds__(32 * kSwWPC, 3) k_jacobi_warp(const SweepArgs a) {
  constexpr int NRING = 16;
  constexpr int STEP = kSwCols - 2 * T;  // interior columns per strip
  extern __shared__ double sw_pool[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double *ring = sw_pool + wid * (2 * NRING * kSwCols);
  const int b = blockIdx.z;
  if (a.active && !a.active[b]) return;
  const int tile = blockIdx.x * kSwWPC + wid;
  if (tile >= a.n_strips * a.n_bands) return;
  const int band = tile / a.n_strips, strip = tile - band * a.n_strips;
  const int nz = a.nz, nr = a.nr;
  const int z0 = band * a.band_rows, z1 = min(nz, z0 + a.band_rows);
  const int c0 = strip * STEP, c1 = (a.n_strips == 1) ? nr : min(nr, c0 + STEP);
  const int zl = max(0, z0 - T), zh = min(nz, z1 + T);
  const int cl = max(0, c0 - T), ch = min(nr, cl + kSwCols);
  jacobi_warp_body<T>(a, ring, lane, zl, zh, z0, z1, cl, ch - cl, c0, c1, a.in + (size_t)b * a.istride,
                      a.src + (size_t)b * a.sstride, a.out + (size_t)b * a.ostride);
}

static size_t sweep_smem_bytes() {
  const int nring = 16;
  return (size_t)(kSwWPC * 2 * nring * kSwCols) * sizeof(double);
}

// Tile plan: strips of (64 - 2*NST) interior columns (one strip when the row fits 64 columns); row
// bands sized so that the grid has enough warps to fill the GPU when the batch alone does not.
void sweep_fused_plan(int nz, int nr, int batch, int nst, int num_sms, int *strip_cols, int *band_rows,
                      int *n_strips, int *n_bands) {
  const int step = kSwCols - 2 * nst;
  if (nr <= kSwCols) {
    *strip_cols = nr;
    *n_strips = 1;
  } else {
    *strip_cols = step;
    *n_strips = (nr + step - 1) / step;
  }
  const long long warps = (long long)*n_strips * batch;
  const long long want = 24LL * num_sms;
  int bands = 1;
  // a warp marches down its band row by row, ~1 us per row step when it is alone on its SM (measured on
  // 257^2..1025^2 single grids: 45 us per launch with 32-row bands, whatever the level): a level that cannot fill
  // the GPU is latency bound, so its bands shrink down to 8 rows - the 2*nst halo rows recomputed per band are
  // free there, and the results do not depend on the tiling.  (A cost model that also avoided band counts just
  // past a wave boundary was measured and made things worse: full SMs are throughput bound, r2_streaming_picard.md.)
  if (warps < want) bands = (int)std::min<long long>((want + warps - 1) / warps, std::max(1, nz / 8));
  const int br = (nz + bands - 1) / bands;
  *band_rows = br;
  *n_bands = (nz + br - 1) / br;
}

// S = sweeps (1..3) fused sweeps; in == out is allowed only for a single tile per equilibrium.
int sweep_fused_launch(const LevelGeom &g, const double *in, size_t istride, double *out, size_t ostride,
                       const double *src, size_t sstride, int batch, double omega, int sweeps, int par_off,
                       int num_sms, const int *active, cudaStream_t st) {
  if (g.nz < 3 || g.nr < 3 || sweeps <= 0 || batch <= 0) return GSB_OK;
  GSB_REQUIRE(sweeps <= 3, "sweep_fused_launch: at most 3 fused sweeps");
  const int nst = 2 * sweeps;
  SweepArgs a{};
  a.nz = g.nz;
  a.nr = g.nr;
  a.par_off = par_off;
  int ns, nb;
  int sc;
  sweep_fused_plan(g.nz, g.nr, batch, nst, num_sms, &sc, &a.band_rows, &ns, &nb);
  a.n_strips = ns;
  a.n_bands = nb;
  GSB_REQUIRE(in != out || (ns == 1 && nb == 1), "sweep_fused_launch: in-place needs a single tile per equilibrium");
  a.in = in;
  a.out = out;
  a.src = src;
  a.istride = istride;
  a.ostride = ostride;
  a.sstride = sstride;
  a.a_e = g.a_e;
  a.a_w = g.a_w;
  a.a_ns = g.a_ns;
  a.a_c = g.a_c;
  a.inv_a_c = g.inv_a_c;
  a.omega = omega;
  a.omw = 1.0 - omega;
  a.active = active;
  const size_t smem = sweep_smem_bytes();
  const dim3 grd((ns * nb + kSwWPC - 1) / kSwWPC, 1, batch), blk(32 * kSwWPC, 1, 1);
  // one GSB_SMEM_OPT_IN per kernel: each expansion remembers on its own that its attribute is set
  if (nst == 2) {
    GSB_SMEM_OPT_IN(k_sweep_warp<2>, smem);
    k_sweep_warp<2><<<grd, blk, smem, st>>>(a);
  } else if (nst == 4) {
    GSB_SMEM_OPT_IN(k_sweep_warp<4>, smem);
    k_sweep_warp<4><<<grd, blk, smem, st>>>(a);
  } else {
    GSB_SMEM_OPT_IN(k_sweep_warp<6>, smem);
    k_sweep_warp<6><<<grd, blk, smem, st>>>(a);
  }
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

// T = 5 Jacobi steps per pass over HBM, out of place (in != out).
int jacobi_fused_launch(const LevelGeom &g, const double *in, double *out, const double *src, int batch, int num_sms,
                        const int *active, cudaStream_t st) {
  constexpr int T = kJacobiFused;
  GSB_REQUIRE(in != out, "jacobi_fused_launch: out of place only");
  if (batch <= 0) return GSB_OK;
  SweepArgs a{};
  a.nz = g.nz;
  a.nr = g.nr;
  int ns, nb, sc;  // T halo rows / columns per side, like a sweep of T stages
  sweep_fused_plan(g.nz, g.nr, batch, T, num_sms, &sc, &a.band_rows, &ns, &nb);
  a.n_strips = ns;
  a.n_bands = nb;
  a.in = in;
  a.out = out;
  a.src = src;
  a.istride = a.ostride = a.sstride = (size_t)g.nz * g.nr;
  a.a_e = g.a_e;
  a.a_w = g.a_w;
  a.a_ns = g.a_ns;
  a.a_c = g.a_c;
  a.inv_a_c = g.inv_a_c;
  a.active = active;
  const size_t smem = sweep_smem_bytes();
  const dim3 grd((ns * nb + kSwWPC - 1) / kSwWPC, 1, batch), blk(32 * kSwWPC, 1, 1);
  GSB_SMEM_OPT_IN(k_jacobi_warp<T>, smem);
  k_jacobi_warp<T><<<grd, blk, smem, st>>>(a);
  GSB_LAUNCH_CHECK();
  return GSB_OK;
}

}  // namespace gsb

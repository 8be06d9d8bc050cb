/* gsb200.h - C ABI of libgsb200.so: the B200-native Grad-Shafranov hot path.
 *
 * Two groups of entry points (reference paths are relative to the reference root):
 *
 *  A. The reference's own native ABI, verbatim: the six symbols its ctypes bridge
 *     binds (src/scpn_fusion/hpc/hpc_bridge.py:190-250) and its C++ solver exports
 *     (src/scpn_fusion/hpc/solver.cpp:200-335).  HOST pointers, row-major [iz][ir]
 *     float64, size == nz*nr.  libgsb200.so can be handed to the reference through
 *     SCPN_SOLVER_LIB unchanged (INTEGRATION.md section 1).
 *
 *  B. The device API (gsb_*): what the Python host mirror of the reference's
 *     solver surface (scpn_fusion_core_b200/) calls.  All `*_dev` arguments are
 *     DEVICE pointers (e.g. torch.Tensor.data_ptr()), dense C-order float64
 *     [batch][nz][nr] unless stated; `stream` is a cudaStream_t passed as void*
 *     (NULL = legacy default stream).  No exceptions cross the ABI: functions
 *     return GSB_OK (0) or a negative GSB_E* code; gsb_last_error() gives the text.
 *     Nothing here falls back to the CPU: without a CUDA device every call that
 *     would compute returns GSB_ENODEV.
 *
 * Plain C types only; no torch / CUDA types in any signature.
 */
#ifndef GSB200_H
#define GSB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSB_ABI_VERSION 1

enum {
  GSB_OK = 0,
  GSB_EINVAL = -1,  /* bad argument (NULL pointer, shape, omega outside [1,2), ...) */
  GSB_ENODEV = -2,  /* no usable CUDA device */
  GSB_ECUDA = -3,   /* a CUDA runtime call failed; see gsb_last_error() */
  GSB_ENOMEM = -4,
  GSB_ESTATE = -5   /* call sequence error (e.g. Picard state not set) */
};

/* ------------------------------------------------------------------------- */
/* A. reference native ABI (solver.cpp:200-335 / hpc_bridge.py:190-250)      */
/* ------------------------------------------------------------------------- */

/* solver.cpp:205 - NULL if nr<2 || nz<2 || rmin>=rmax || zmin>=zmax (or no GPU). */
void *create_solver(int nr, int nz, double rmin, double rmax, double zmin, double zmax);
/* solver.cpp:226 - constant Dirichlet wall value; NULL handle ignored. */
void set_boundary_dirichlet(void *solver_ptr, double boundary_value);
/* solver.cpp:243 - max(iterations,1) RB-SOR sweeps at omega=1.8 of
 * source = -1.0*R*j; psi persists in the handle across calls (warm start). */
void run_step(void *solver_ptr, const double *j_array, double *psi_array, int size, int iterations);
/* solver.cpp:273 - sweeps until max|delta psi| <= tol; omega clamped to [0.1,1.99];
 * returns sweeps done (>=1), 0 on invalid input. */
int run_step_converged(void *solver_ptr, const double *j_array, double *psi_array, int size,
                       int max_iterations, double omega, double tolerance, double *final_delta_out);
/* solver.cpp:325,331 */
void destroy_solver(void *solver_ptr);
void delete_solver(void *solver_ptr);

/* ------------------------------------------------------------------------- */
/* B. device API                                                             */
/* ------------------------------------------------------------------------- */

typedef struct gsb_ctx gsb_ctx;

int gsb_abi_version(void);
const char *gsb_last_error(void);
/* Number of visible CUDA devices (0 without a GPU; never fails). */
int gsb_device_count(void);
/* Count of kernels launched by this library in this process (bench.py's gpu_launches). */
long long gsb_launch_count(void);

/* Debug: clock64() totals per V-cycle phase of CTA 0 of the shared-memory-resident kernel
 * (index 4*level + {0 pre-smooth, 1 residual+restrict, 2 prolong, 3 post-smooth}; the base level
 * uses slot 0).  All zeros unless the library was built with -DGSB_PHASE_TIMING. out64: 64 values. */
int gsb_debug_phase_cycles(long long *out64, int reset);

/* Host-only planning helper (works without a GPU): level sizes of the V-cycle
 * the reference would run on (nz,nr) with `min_grid` (multigrid_solve.py:292,
 * coarse size (n+1)//2).  Writes up to `cap` (nz,nr) pairs, returns the number of
 * levels including the base level. */
int gsb_plan_levels(int nz, int nr, int min_grid, int *nz_out, int *nr_out, int cap);
/* Host-only: per-level interior-row R values and stencil columns exactly as the
 * reference derives them (restrict_full_weight of r_grid, multigrid_solve.py:307;
 * a_e/a_w, :186-187).  out arrays hold nr_level doubles (walls = 0). */
int gsb_plan_level_tables(int nz, int nr, const double *r_row, double dr, double dz, int min_grid,
                          int level, double *r_out, double *a_e_out, double *a_w_out,
                          double *scalars_out /* dr,dz,a_ns,a_c */);

/* Context: one grid geometry + workspace for up to batch_cap equilibria on one
 * device.  r_row: HOST array of nr R-coordinates (an interior row of the
 * reference's r_grid); dr,dz: the spacings exactly as the calling entry point
 * computes them (SURVEY.md App.A item 1).  z_axis may be NULL when only the
 * multigrid entry points are used. */
int gsb_create(gsb_ctx **out, int nz, int nr, const double *r_row, const double *z_axis, double dr,
               double dz, int batch_cap, int device);
void gsb_destroy(gsb_ctx *ctx);

/* --- multigrid operators (multigrid_solve.py) ---------------------------- */

/* a1/a2: n_sweeps in-place red-black SOR sweeps (mg_smooth, multigrid_solve.py:148-208).
 * clip!=0 adds the +-1e250 clamp of _sor_step (fusion_kernel_iterative_solver.py:158). */
int gsb_smooth(gsb_ctx *ctx, double *psi_dev, const double *src_dev, int batch, double omega,
               int n_sweeps, int clip, void *stream);
/* Same, choosing the kernel: fuse = 0 launches one kernel per colour pass (48 B of DRAM traffic per
 * point per sweep); fuse = 1..3 runs that many sweeps per pass over HBM with the temporally blocked
 * kernel of gsb_sweep.cu (24 B per point per pass; identical results).  gsb_smooth uses fuse = 3. */
int gsb_smooth_ex(gsb_ctx *ctx, double *psi_dev, const double *src_dev, int batch, double omega,
                  int n_sweeps, int clip, int fuse, void *stream);
/* a3: out-of-place toroidal Jacobi step with sanitise+clip (_jacobi_step, :54-95). */
int gsb_jacobi(gsb_ctx *ctx, const double *psi_dev, const double *src_dev, double *out_dev,
               int batch, void *stream);
/* a3 repeated: n_steps Jacobi steps in place (result in psi_dev; tmp_dev [batch][nz][nr] is scratch) - the Picard
 * seed's 50 steps (_seed_plasma, fusion_kernel_iterative_solver.py:410-415).  Groups of 5 steps run in one pass over
 * HBM (temporally blocked, register-carried kernel); results are bit-identical to n_steps calls of gsb_jacobi. */
int gsb_jacobi_steps(gsb_ctx *ctx, double *psi_dev, const double *src_dev, double *tmp_dev, int n_steps,
                     int batch, void *stream);
/* a4: r = L*psi - src on the interior, 0 on the wall (mg_residual, :211-249). */
int gsb_residual(gsb_ctx *ctx, const double *psi_dev, const double *src_dev, double *res_dev,
                 int batch, void *stream);
/* a4: L*v (apply_gs_operator, fusion_kernel_solver_runtime.py:54-68). */
int gsb_apply_operator(gsb_ctx *ctx, const double *v_dev, double *out_dev, int batch, void *stream);
/* a5: per-equilibrium interior max|r| and RMS (residual_linf :338; compute_gs_residual_rms). */
int gsb_residual_norms(gsb_ctx *ctx, const double *psi_dev, const double *src_dev,
                       double *linf_dev, double *rms_dev, int batch, void *stream);
/* a6/a7: geometry-free transfer operators on arbitrary shapes. */
int gsb_restrict_full_weight(const double *fine_dev, double *coarse_dev, int nz_f, int nr_f,
                             int batch, void *stream);
int gsb_prolong_bilinear(const double *coarse_dev, double *fine_dev, int nz_c, int nr_c, int nz_f,
                         int nr_f, int batch, void *stream);
/* a8: one V-cycle, psi updated in place (multigrid_vcycle, :252-335; wall not re-applied). */
int gsb_vcycle(gsb_ctx *ctx, double *psi_dev, const double *src_dev, int batch, double omega,
               int pre, int post, int min_grid, void *stream);
/* a9: V-cycles until interior Linf residual < tol (multigrid_solve, :352-463).
 * psi_dev holds psi_bc on entry and the solution on exit; per-equilibrium outputs
 * (device): residual, n_cycles, converged. */
int gsb_mg_solve(gsb_ctx *ctx, const double *src_dev, double *psi_dev, int batch, double tol,
                 int max_cycles, double omega, int pre, int post, int min_grid, double *res_dev,
                 int *cycles_dev, int *converged_dev, void *stream);

/* --- Picard pieces (fusion_kernel.py) ------------------------------------- */

/* a10+a11: O-point (first global max, |psi|<1e-6 -> 1e-6) and X-point (first min of
 * hypot(grad psi) over rows with Z < 0.5*z_min, optional 16-candidate saddle filter).
 * out_dev: [batch][8] doubles = iz_ax, ir_ax, psi_ax, iz_x, ir_x, psi_x, found_x, min(psi).
 * found_x==0: no row below 0.5*z_min -> the reference's ((0,0), min psi) fallback. */
int gsb_topology(gsb_ctx *ctx, const double *psi_dev, int batch, double z_min, int saddle,
                 double *out_dev, void *stream);

typedef struct gsb_profile {
  int hmode;         /* 0 = L-mode (1-psi_N), 1 = H-mode mtanh (fusion_kernel.py:359-390) */
  double ped_p[4];   /* ped_top, ped_width, ped_height, core_alpha for p'  */
  double ped_ff[4];  /* same for FF' */
} gsb_profile;

/* a12: J_phi(psi) renormalised to Ip (update_plasma_source_nonlinear, fusion_kernel.py:394-444).
 * axis_bnd_dev: [batch][2] (psi_axis, psi_boundary); ip_dev: [batch];
 * prof_dev: NULL (use `prof` for all) or [batch][8] per-equilibrium pedestal params. */
int gsb_plasma_source(gsb_ctx *ctx, const double *psi_dev, const double *axis_bnd_dev,
                      const double *ip_dev, double mu0, const gsb_profile *prof,
                      const double *prof_dev, double *jphi_dev, int batch, void *stream);

typedef struct gsb_picard_params {
  int max_iterations;          /* solver.max_iterations */
  double tol;                  /* solver.convergence_threshold */
  double alpha;                /* solver.relaxation_factor (default 0.1) */
  double omega;                /* solver.sor_omega (default 1.6) */
  int method;                  /* 0 multigrid (default), 1 sor, 2 jacobi, 3 anderson (SOR sweep + Anderson mixing) */
  int require_gs_residual;     /* solver.require_gs_residual */
  double gs_tol;               /* solver.gs_residual_threshold */
  int saddle;                  /* solver.xpoint_use_saddle_detection */
  double mu0;                  /* physics.vacuum_permeability */
  double z_min, r_min, r_max;  /* dimensions.* (X-point mask, seed centre) */
  int seed;                    /* 1: Gaussian seed + 50 Jacobi (_seed_plasma) */
  int check_every;             /* host polls the active count every this many iterations */
  gsb_profile prof;
  int external_profile;        /* 1: external_profile_mode (fusion_kernel_newton_solver.py:509) - J_phi is NOT updated
                                  from psi inside the loop; every iteration solves with the source left by the seed
                                  (_seed_plasma overwrites J_phi before the loop, also in this mode) */
  int anderson_depth;          /* method 3: solver.anderson_depth (default 5), 0..8; the iterate is mixed on iterations
                                  3, 6, 9, ... over the last min(depth, k+1) relaxed iterates
                                  (fusion_kernel_iterative_solver.py:248-314, fusion_kernel_newton_solver.py:539-550) */
} gsb_picard_params;

/* a13+a14: batched Picard solve (solve_equilibrium, fusion_kernel_newton_solver.py:390-615).
 * psi_dev   [batch][nz][nr] in: initial flux (vacuum field or warm start), out: solution
 * bc_dev    [batch][nz][nr] boundary map (only its wall ring is read)
 * ip_dev    [batch]         plasma current targets
 * prof_dev  NULL or [batch][8] per-equilibrium pedestal parameters
 * jphi_dev  [batch][nz][nr] out: final J_phi
 * summary_dev [batch][16] out: iterations, converged, residual(best diff), gs_residual,
 *            gs_residual_best, status(0 run,1 conv,2 maxiter,3 diverged), psi_axis, psi_bnd,
 *            iz_ax, ir_ax, iz_x, ir_x, diff_last, found_x, Ip/I scale, 0
 * hist_dev / gs_hist_dev  NULL or [batch][max_iterations] histories */
int gsb_picard_solve(gsb_ctx *ctx, const gsb_picard_params *p, double *psi_dev, const double *bc_dev,
                     const double *ip_dev, const double *prof_dev, double *jphi_dev,
                     double *summary_dev, double *hist_dev, double *gs_hist_dev, int batch,
                     void *stream);
/* Picard iterations launched by the last gsb_picard_solve on this ctx (host count). */
int gsb_picard_last_launched_iterations(gsb_ctx *ctx);

typedef struct gsb_free_boundary_params {
  int max_outer_iter;  /* solve_free_boundary(max_outer_iter=20) */
  double tol;          /* solve_free_boundary(tol=1e-4): stop an equilibrium when max|Psi - Psi_old| < tol */
  int warm_j;          /* 1: jphi_dev holds a current density on entry and the plasma wall flux of outer iteration 0
                          is formed from it; 0: outer iteration 0 sees the coil flux alone */
} gsb_free_boundary_params;

/* a17 batched: the free-boundary outer loop of solve_free_boundary (fusion_kernel_free_boundary.py:623-739,
 * optimize_shape=False) for `batch` independent equilibria, entirely on the device.  Per outer iteration and
 * per not-yet-converged equilibrium: wall ring of Psi <- psi_ext ring (:652-655), Psi_old <- Psi (:658), warm-started
 * re-seeded Picard solve with that boundary map (:659-662, gsb_picard_solve semantics), diff = max|Psi - Psi_old|,
 * stop when diff < tol (:708-711).  The host reads one counter per OUTER iteration.
 * psi_dev      [batch][nz][nr] in: starting flux (zeros for a fresh kernel), out: solution
 * psi_ext_dev  [batch][nz][nr] coil flux (compute_external_flux, :83-93; only its wall ring is read)
 * wall_m_dev   NULL (lane A: the wall carries coil flux only, as in the reference's NumPy lane) or the lane-C
 *              response matrix of gsb_wall_matrix: from outer iteration 1 on the wall gets
 *              psi_ext + M @ (J_phi[interior]*dR*dZ) (jax_free_boundary_predictive.py:443-498) with the J_phi of the
 *              previous inner solve, as ONE FP64 tensor-core GEMM over the batch (gsb_wall_flux)
 * summary_dev  [batch][16] gsb_picard_solve summary of the LAST inner solve of each equilibrium
 * fb_summary_dev [batch][4] out: outer_iterations, final_diff, Picard iterations summed over the outer
 *              iterations, converged (final_diff < tol) */
int gsb_free_boundary_solve(gsb_ctx *ctx, const gsb_picard_params *p, const gsb_free_boundary_params *fb,
                            double *psi_dev, const double *psi_ext_dev, const double *wall_m_dev,
                            const double *ip_dev, const double *prof_dev, double *jphi_dev, double *summary_dev,
                            double *fb_summary_dev, int batch, void *stream);

typedef struct gsb_shape_params {
  int n_coils;            /* 1..32 */
  const double *coil_rz;  /* HOST [n_coils][2] coil (R, Z) */
  int n_points;           /* shape-control points P, 1..1024 */
  const double *points;   /* HOST [P][2] (R, Z) of the control points */
  double alpha;           /* Tikhonov weight (tikhonov_alpha), finite and >= 0 */
  int isoflux;            /* 1: target = mean of the bilinear samples of the new Psi at the points (broadcast to P);
                             0: target_dev holds explicit per-equilibrium targets */
  const double *limits;   /* HOST [n_coils] current limits (> 0; bounds are +-limits) or NULL (unbounded) */
} gsb_shape_params;

/* solve_free_boundary(optimize_shape=True) (fusion_kernel_free_boundary.py:623-739) for `batch` independent
 * equilibria on the device.  The outer loop of gsb_free_boundary_solve gains a shape step after each inner Picard
 * solve of every still-active equilibrium: target t (isoflux mean or explicit), then the coil currents x minimising
 * |M^T x - t|^2 + alpha |x|^2 within +-limits (M[c][p] = turns_c G_SI(coil c -> point p)), then the coil flux
 * sum_c x_c turns_c G_c.  The fit is the exact minimiser (bounded-variable least squares on the QR factor of
 * [M^T; sqrt(alpha) I]), not the stopping point of the reference's interior-point lsq_linear(method="trf"); a
 * non-finite target or an iteration cap reached keeps the clipped prior currents (the reference's failure path).
 * A rank-deficient [M^T; sqrt(alpha) I] (alpha = 0 and fewer independent points than coils) fails with GSB_EINVAL
 * before any Picard launch.
 * green_dev    [n_coils][nz][nr] si==1 tables of gsb_green_table for these coils
 * turns_host   HOST [n_coils] integer turns
 * currents_dev [batch][n_coils] in: starting currents, out: final currents
 * target_dev   NULL (isoflux) or [batch][P] explicit targets
 * shape_out_dev [batch][2P+4] out, of each equilibrium's last shape step: target[P], achieved flux M^T x [P],
 *              rmse, max |achieved - target|, active bounds (|x| within 1e-8 of its limit), fallback (1: prior kept)
 * psi_ext_dev  [batch][nz][nr] out: coil flux of the final currents
 * The other arguments are those of gsb_free_boundary_solve. */
int gsb_free_boundary_shape_solve(gsb_ctx *ctx, const gsb_picard_params *p, const gsb_free_boundary_params *fb,
                                  const gsb_shape_params *sp, const double *green_dev, const int *turns_host,
                                  double *currents_dev, const double *target_dev, double *shape_out_dev,
                                  double *psi_dev, double *psi_ext_dev, const double *wall_m_dev,
                                  const double *ip_dev, const double *prof_dev, double *jphi_dev, double *summary_dev,
                                  double *fb_summary_dev, int batch, void *stream);

typedef struct gsb_probe_params {
  int n_coils;             /* 1..32 */
  int n_rows;              /* measurements m (flux loops, then B probes), 1..1024 */
  const double *response;  /* HOST [m][n_coils] probe response R_p (build_magnetic_probe_response_matrix) */
  const double *sigma;     /* HOST [m] measurement sigma (> 0; weights w = 1/sigma) or NULL (w = 1) */
  double alpha;            /* Tikhonov weight (tikhonov_alpha), finite and >= 0 */
  const double *limits;    /* HOST [n_coils] current limits (> 0; bounds are +-limits) or NULL (unbounded) */
  int max_iter;            /* cap on the free-set solves of one fit; 0 = 3 n_coils + 10 */
} gsb_probe_params;

/* reconstruct_coil_currents_from_magnetic_probes (fusion_kernel_free_boundary.py:370-488) for `batch` independent
 * measurement vectors of one diagnostic set.  Context-free: it runs on the current device and `stream`.  Each sample b
 * gets the currents x minimising |diag(w) (R_p x - meas_b)|^2 + alpha |x - prior_b|^2 within +-limits: the exact
 * minimiser (bounded-variable least squares on the QR factor of [diag(w) R_p; sqrt(alpha) I], factored once per
 * call), where the reference stops lsq_linear(method="trf") at its tolerance.  With alpha = 0 the prior is not used.
 * A rank-deficient factor (alpha = 0 and fewer independent rows than coils) fails with GSB_EINVAL before the fit.
 * meas_dev      [batch][m] measurements (flux loops, then B probes)
 * prior_dev     [batch][n_coils] prior currents
 * currents_dev  [batch][n_coils] out: fitted currents (clip(prior, +-limits) where the fit failed)
 * residual_dev  [batch][m] out: R_p x - meas;  wresidual_dev [batch][m] out: residual * w
 * stats_dev     [batch][4] out: residual rms, weighted residual rms, active bounds (np.isclose(x, +-limit)),
 *               failed (1: non-finite right-hand side or max_iter reached)
 * work_dev      device workspace of *work_bytes bytes; with work_dev NULL the call only stores the size it needs in
 *               *work_bytes (n_coils and n_rows must then be set). */
int gsb_probe_reconstruct(const gsb_probe_params *pp, const double *meas_dev, const double *prior_dev,
                          double *currents_dev, double *residual_dev, double *wresidual_dev, double *stats_dev,
                          void *work_dev, long long *work_bytes, int batch, void *stream);

/* Measurement hook (bench.py roofline): while enabled, gsb_free_boundary_solve brackets every inner Picard solve and
 * every wall GEMM with CUDA events on the launching stream and accumulates
 * out4 = {Picard solves: total ms, count; wall GEMMs: total ms, count}.  out4 may be NULL; reset != 0 zeroes the sums. */
int gsb_timing(gsb_ctx *ctx, int enable, double *out4, int reset);

/* compute_b_field (fusion_kernel.py:450-456): np.gradient + 1/max(R,1e-6). */
int gsb_b_field(gsb_ctx *ctx, const double *psi_dev, double *br_dev, double *bz_dev, int batch,
                void *stream);

/* --- Green's functions ---------------------------------------------------- */

/* a15/a16: per-coil unit-current flux tables G[c][nz][nr] on the ctx grid.
 * si==0: calculate_vacuum_field form (fusion_kernel.py:236-249, k2 clip, no self mask), two
 *        planes per coil (see gsb_coil_flux), g_dev [n_coils][2][nz][nr];
 * si==1: _green_function_vectorised (fusion_kernel_free_boundary.py:58-80) incl. mu0_SI and the
 *        self-point mask, g_dev [n_coils][nz][nr].
 * coil_rz: HOST [n_coils][2]. */
int gsb_green_table(gsb_ctx *ctx, const double *coil_rz, int n_coils, int si, double *g_dev,
                    void *stream);
/* psi[b] = sum_c w[b][c] * G[c], accumulated in coil order from 0.0 (w_dev: [batch][n_coils]).
 * si==0: g_dev is [c][2][nz][nr] = (sqrt(R Rc), ((2-k2)K-2E)/k), w = (mu0*I)/(2 pi), each term
 *        evaluated as (w*sqrt)*term exactly like fusion_kernel.py:245-249;
 * si==1: g_dev is [c][nz][nr], w = I*turns (fusion_kernel_free_boundary.py:88-92). */
int gsb_coil_flux(gsb_ctx *ctx, const double *g_dev, const double *w_dev, int n_coils, int si,
                  double *psi_dev, int batch, void *stream);
/* a16: M[coil][point] = turns*G_SI (build_mutual_inductance_matrix, :137-153). HOST inputs. */
int gsb_mutual_matrix(const double *coil_rz, const int *turns, int n_coils, const double *obs_rz,
                      int n_pts, double *m_dev, void *stream);
/* a18: lane-C von Hagenow response matrix M[N_wall][N_int] (build_response_matrix,
 * jax_free_boundary_predictive.py:183-211; greens_psi_si, jax_free_boundary_gs.py:70-86). */
int gsb_wall_matrix(gsb_ctx *ctx, double mu0, double *m_dev, void *stream);
/* a18: wall[b][N_wall] = M @ (J[b][interior]*dA) (:498) as one FP64 tensor-core GEMM over the
 * batch.  jphi_dev is the full (nz,nr) field; interior gather is fused. */
int gsb_wall_flux(gsb_ctx *ctx, const double *m_dev, const double *jphi_dev, double dA,
                  double *wall_dev, int batch, void *stream);
/* Scatter wall[b][N_wall] (+ optional coil wall flux) onto the ring of bc_dev. */
int gsb_wall_scatter(gsb_ctx *ctx, const double *wall_dev, double *bc_dev, int accumulate, int batch,
                     void *stream);

/* --- slab operators: one large grid split into Z-row slabs, one process per GPU ------------- */
/* (the reference's only decomposition code for this path is fusion-core/src/mpi_domain.rs:48-965,
 * an additive-Schwarz scaffold; these keep exact RB-SOR instead, SURVEY.md 8e.)
 * A slab context is gsb_create(rows_loc, nr, r_row_of_the_level, NULL, dr_level, dz_level, 1, dev):
 * the local array [rows_loc][nr] = halo rows + owned rows + halo rows.  Host code exchanges halos. */
/* 1 if `sweeps` fused sweeps of this local array run as a single tile (in-place allowed). */
int gsb_slab_single_tile(gsb_ctx *ctx, int sweeps);
/* sweeps (1..3) RB-SOR sweeps of the local array in one pass; rows 0 and rows_loc-1 are fixed.
 * par_off = global row index of local row 0 (colour parity).  Owned rows are exact when at least
 * 2*sweeps valid halo rows surround them (or the array edge is the true wall). */
int gsb_slab_smooth(gsb_ctx *ctx, const double *in_dev, double *out_dev, const double *src_dev, double omega,
                    int sweeps, int par_off, void *stream);
/* coarse local rows [ci0,ci1) of dc = full weighting of -(L x - src); fine local row of coarse
 * local row I is 2*I + roff; coarse column walls get 0. */
int gsb_slab_residual_restrict(gsb_ctx *fine, const double *x_dev, const double *src_dev, double *dc_dev,
                               int nzc_loc, int nrc, int roff, int ci0, int ci1, void *stream);
/* x[fine local rows fi0..fi1), interior columns] += bilinear prolongation of ec. */
int gsb_slab_prolong_add(gsb_ctx *fine, const double *ec_dev, int nzc_loc, int nrc, double *x_dev, int roff,
                         int fi0, int fi1, void *stream);
/* *out_dev = max(*out_dev, max |L x - src| over local rows [row0,row1), interior columns). */
int gsb_slab_residual_linf(gsb_ctx *ctx, const double *x_dev, const double *src_dev, int row0, int row1,
                           double *out_dev, void *stream);

/* Halo exchange over NVLink peer memory (CUDA IPC; no NCCL launch).  Every rank owns two inboxes
 * and a block of four int64 flags {ready_from_up, ready_from_dn, consumed_by_up, consumed_by_dn} that
 * its neighbours can address.  gsb_halo_push stores `n` doubles of boundary rows straight into the
 * neighbours' inboxes and raises their ready flags; gsb_halo_recv waits for its own ready flags,
 * copies inbox -> halo rows and releases the senders.  `epochs` = four zero-initialised int64 of LOCAL
 * device scratch (exchange counters, kept on the device so a captured CUDA graph can be replayed);
 * both sides must issue the same sequence of exchanges; NULL row pointers = no neighbour on that side. */
int gsb_enable_peer_access(int device, int peer_device);
/* CUDA IPC plumbing for the inboxes/flags: a zero-filled cudaMalloc block + its 64-byte handle; the
 * neighbours map it with gsb_ipc_open. */
int gsb_ipc_alloc(int device, long long bytes, void **ptr_out, unsigned char *handle_out64);
int gsb_ipc_open(int device, const unsigned char *handle64, void **ptr_out);
int gsb_ipc_close(void *ptr);
int gsb_ipc_free(void *ptr);
int gsb_halo_push(const double *rows_up, const double *rows_dn, long long n, double *up_inbox_dn, double *dn_inbox_up,
                  long long *flags_local, long long *flags_up, long long *flags_dn, int *counters, long long *epochs,
                  void *stream);
int gsb_halo_recv(double *halo_up, double *halo_dn, long long n, const double *inbox_up, const double *inbox_dn,
                  long long *flags_local, long long *flags_up, long long *flags_dn, int *counters, long long *epochs,
                  void *stream);

/* Coarse-level gather over NVLink peer memory (replaces the NCCL all-gather inside a slab V-cycle, so that the cycle
 * holds this library's kernels only and replays from a CUDA graph on every rank).  Every rank owns an IPC block
 * {world int64 flags | two halves of buf_doubles doubles}; peer_bufs[p] / peer_flags[p] are rank p's halves / flags as
 * mapped here (own rank included).  gsb_gather_push stores `n` doubles (this rank's owned rows) at offset `off` of the
 * current half of every rank and raises flag[rank] there; gsb_gather_wait waits for all `world` flags, copies the
 * assembled n_total doubles into out_dev and bumps *epoch (device counter of completed gathers, zeroed once;
 * counters: `world` zeroed ints).  host_flag (NULL or mapped pinned host memory) receives the exchange number after
 * out_dev is complete: with out_dev in pinned memory too, the host polls it instead of synchronising the stream
 * (the per-cycle convergence norm of a slab solve travels this way: one value per rank, maximum taken on the host). */
int gsb_gather_push(const double *rows_dev, long long n, long long off, long long buf_doubles, void *const *peer_bufs,
                    void *const *peer_flags, int world, int rank, int *counters, const long long *epoch, void *stream);
int gsb_gather_wait(const double *buf_local, long long buf_doubles, const long long *flags_local, int world,
                    long long n_total, double *out_dev, long long *epoch, long long *host_flag, void *stream);

/* Native driver of the distributed levels of one slab V-cycle: every launch of the descent
 * (gsb_slab_down) and of the ascent (gsb_slab_up) is issued from one call; the host gathers the
 * coarsest distributed right-hand side and runs the replicated coarse V-cycle in between.  Together they
 * are the recursion of multigrid_vcycle (multigrid_solve.py:252-335) on one rank's Z-row slab (the
 * reference's decompose_z partition, mpi_domain.rs:48); halo = NULL on a single rank. */
typedef struct gsb_slab_level_desc {
  gsb_ctx *ctx;              /* slab context of the level (rows_loc x nr) */
  double *x, *f, *alt, *cur; /* solution, right-hand side, ping-pong partner (NULL if single tile), live buffer */
  int rows_loc, nr;
  int own0, own1;            /* owned local rows [own0, own1) */
  int has_up, has_dn;        /* neighbours present */
  int row0;                  /* global row of local row 0 (colour parity) */
  int roff, ci0, ci1;        /* restriction target: fine local row = 2*coarse local row + roff; rows to compute */
  int nzc_loc, nrc;          /* shape of the restriction target (next level's f, or the gathered level's owned rows) */
  int fi0, fi1;              /* fine local rows that receive the prolonged correction */
} gsb_slab_level_desc;
typedef struct gsb_slab_halo_desc {
  double *inbox_up, *inbox_dn;        /* this rank's inboxes */
  double *up_inbox_dn, *dn_inbox_up;  /* the neighbours' inboxes (peer pointers) */
  long long *flags_local, *flags_up, *flags_dn;
  int *counters;
  long long *epochs;
  long long cap;                      /* doubles per inbox */
} gsb_slab_halo_desc;
int gsb_slab_down(gsb_slab_level_desc *lev, int nlev, double *d_last, const gsb_slab_halo_desc *halo, int halo_rows,
                  double omega, int pre, void *stream);
int gsb_slab_up(gsb_slab_level_desc *lev, int nlev, const double *e_last, int nze_last_loc, int roff_last,
                const gsb_slab_halo_desc *halo, int e_rows, double omega, int post, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GSB200_H */

// gsb_core.cu - context, level planning (host), error plumbing.
#include "gsb_internal.cuh"
#include "gsb_resident.cuh"

#include <cstring>
#include <mutex>

namespace gsb {

static thread_local std::string t_err;
static std::string g_err_any;
static std::mutex g_err_mu;
std::atomic<long long> g_launches{0};

void set_error(const std::string &msg) {
  t_err = msg;
  std::lock_guard<std::mutex> lk(g_err_mu);
  g_err_any = msg;
}

// The reference restricts the R meshgrid itself with the 9-point rule
// (multigrid_solve.py:76-91,307).  All rows of the meshgrid are identical, so the
// restricted interior rows are a function of the fine interior row alone:
//   (4*c + 2*(c + c + w + e) + (w + e + w + e)) / 16        (operand order kept)
// Wall columns are injected (:96-97).  Host code is compiled with -ffp-contract=off.
static std::vector<double> restrict_row(const std::vector<double> &f) {
  const int nf = (int)f.size();
  const int nc = (nf + 1) / 2;
  std::vector<double> c(nc, 0.0);
  for (int j = 1; j < nc - 1; ++j) {
    const double cc = f[2 * j], w = f[2 * j - 1], e = f[2 * j + 1];
    volatile double t4 = 4.0 * cc;
    volatile double s1 = cc + cc;
    volatile double s2 = s1 + w;
    volatile double s3 = s2 + e;
    volatile double t2 = 2.0 * s3;
    volatile double q1 = w + e;
    volatile double q2 = q1 + w;
    volatile double q3 = q2 + e;
    volatile double acc = t4 + t2;
    volatile double acc2 = acc + q3;
    c[j] = acc2 / 16.0;
  }
  if (nc >= 1) c[0] = f[0];
  if (nc >= 2) c[nc - 1] = f[nf - 1];
  return c;
}

static void fill_coeffs(HostLevel &L) {
  const int nr = L.nr;
  L.a_e.assign(nr, 0.0);
  L.a_w.assign(nr, 0.0);
  L.r_safe.assign(nr, 1.0);
  L.inv_r_safe.assign(nr, 1.0);
  volatile double dr2 = L.dr * L.dr;
  volatile double dz2 = L.dz * L.dz;
  volatile double inv_dr2 = 1.0 / dr2;
  L.a_ns = 1.0 / dz2;
  volatile double t1 = 2.0 / dr2;
  volatile double t2 = 2.0 / dz2;
  L.a_c = t1 + t2;
  for (int j = 0; j < nr; ++j) {
    volatile double rs = L.r_row[j] > 1e-10 ? L.r_row[j] : 1e-10;  // np.maximum(r, 1e-10)
    volatile double den = (2.0 * rs);
    volatile double den2 = den * L.dr;
    volatile double t = 1.0 / den2;
    L.a_e[j] = inv_dr2 - t;
    L.a_w[j] = inv_dr2 + t;
    L.r_safe[j] = rs;
    L.inv_r_safe[j] = 1.0 / rs;
  }
}

std::vector<HostLevel> plan_levels(int nz, int nr, const double *r_row, double dr, double dz,
                                   int min_grid) {
  std::vector<HostLevel> out;
  HostLevel L;
  L.nz = nz;
  L.nr = nr;
  L.dr = dr;
  L.dz = dz;
  L.r_row.assign(r_row, r_row + nr);
  for (;;) {
    fill_coeffs(L);
    out.push_back(L);
    if (min_grid >= L.nz || min_grid >= L.nr) break;  // base case (multigrid_solve.py:292)
    if (L.nz < 3 || L.nr < 3) break;                  // nothing left to coarsen
    HostLevel C;
    C.nz = (L.nz + 1) / 2;
    C.nr = (L.nr + 1) / 2;
    C.dr = L.dr * 2.0;
    C.dz = L.dz * 2.0;
    C.r_row = restrict_row(L.r_row);
    L = C;
  }
  return out;
}

static void free_levels(gsb_ctx *ctx) {
  for (auto &l : ctx->levels) {
    if (l.tables) cudaFree(l.tables);
    if (l.d) cudaFree(l.d);
    if (l.e) cudaFree(l.e);
    if (l.alt) cudaFree(l.alt);
  }
  ctx->levels.clear();
  ctx->planned_min_grid = -1;
}

int ensure_plan(gsb_ctx *ctx, int min_grid) {
  if (ctx->planned_min_grid == min_grid && !ctx->levels.empty()) return GSB_OK;
  GSB_CUDA(cudaSetDevice(ctx->device));
  free_levels(ctx);
  auto hl = plan_levels(ctx->nz, ctx->nr, ctx->r_row.data(), ctx->dr, ctx->dz, min_grid);
  for (size_t i = 0; i < hl.size(); ++i) {
    const HostLevel &H = hl[i];
    gsb_level_dev D;
    const size_t nr = (size_t)H.nr;
    GSB_CUDA(cudaMalloc(&D.tables, 4 * nr * sizeof(double)));
    std::vector<double> pack(4 * nr);
    memcpy(&pack[0], H.a_e.data(), nr * sizeof(double));
    memcpy(&pack[nr], H.a_w.data(), nr * sizeof(double));
    memcpy(&pack[2 * nr], H.r_safe.data(), nr * sizeof(double));
    memcpy(&pack[3 * nr], H.inv_r_safe.data(), nr * sizeof(double));
    GSB_CUDA(cudaMemcpy(D.tables, pack.data(), pack.size() * sizeof(double), cudaMemcpyHostToDevice));
    LevelGeom &g = D.g;
    g.nz = H.nz;
    g.nr = H.nr;
    g.dr = H.dr;
    g.dz = H.dz;
    volatile double dr2 = H.dr * H.dr, dz2 = H.dz * H.dz, two_dr = 2.0 * H.dr;
    g.dr2 = dr2;
    g.dz2 = dz2;
    g.two_dr = two_dr;
    g.inv_dr2 = 1.0 / dr2;
    g.inv_dz2 = 1.0 / dz2;
    g.inv_two_dr = 1.0 / two_dr;
    g.a_ns = H.a_ns;
    g.a_c = H.a_c;
    g.inv_a_c = 1.0 / H.a_c;
    g.a_e = D.tables;
    g.a_w = D.tables + nr;
    g.r_safe = D.tables + 2 * nr;
    g.inv_r_safe = D.tables + 3 * nr;
    if (i > 0) {
      const size_t bytes = (size_t)ctx->batch_cap * 2 * H.nz * ((H.nr + 1) / 2) * sizeof(double);
      GSB_CUDA(cudaMalloc(&D.d, bytes));
      GSB_CUDA(cudaMalloc(&D.e, bytes));
    }
    ctx->levels.push_back(D);
  }
  ctx->planned_min_grid = min_grid;
  // first level from which the whole V-cycle tail fits one SM's shared memory (none: res_l0 = level count)
  ctx->res_l0 = (int)ctx->levels.size();
  RPlan plan;
  for (int l0 = 0; l0 < (int)ctx->levels.size(); ++l0)
    if (build_rplan(ctx, l0, 0, &plan)) {
      ctx->res_l0 = l0;
      break;
    }
  if (ctx->res_l0 == 0 && !ctx->split_src) {
    const size_t hw = (ctx->nr + 1) / 2;
    GSB_CUDA(cudaMalloc(&ctx->split_src, (size_t)ctx->batch_cap * 2 * ctx->nz * hw * sizeof(double)));
  }
  return GSB_OK;
}

}  // namespace gsb

using namespace gsb;

extern "C" {

int gsb_abi_version(void) { return GSB_ABI_VERSION; }

const char *gsb_last_error(void) {
  if (!t_err.empty()) return t_err.c_str();
  return g_err_any.c_str();
}

int gsb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

long long gsb_launch_count(void) { return g_launches.load(); }

int gsb_plan_levels(int nz, int nr, int min_grid, int *nz_out, int *nr_out, int cap) {
  if (nz < 1 || nr < 1) return GSB_EINVAL;
  std::vector<double> r(nr, 1.0);
  auto hl = plan_levels(nz, nr, r.data(), 1.0, 1.0, min_grid);
  for (size_t i = 0; i < hl.size() && (int)i < cap; ++i) {
    if (nz_out) nz_out[i] = hl[i].nz;
    if (nr_out) nr_out[i] = hl[i].nr;
  }
  return (int)hl.size();
}

int gsb_plan_level_tables(int nz, int nr, const double *r_row, double dr, double dz, int min_grid,
                          int level, double *r_out, double *a_e_out, double *a_w_out,
                          double *scalars_out) {
  if (nz < 1 || nr < 1 || !r_row) return GSB_EINVAL;
  auto hl = plan_levels(nz, nr, r_row, dr, dz, min_grid);
  if (level < 0 || level >= (int)hl.size()) return GSB_EINVAL;
  const HostLevel &H = hl[level];
  for (int j = 0; j < H.nr; ++j) {
    if (r_out) r_out[j] = H.r_row[j];
    if (a_e_out) a_e_out[j] = H.a_e[j];
    if (a_w_out) a_w_out[j] = H.a_w[j];
  }
  if (scalars_out) {
    scalars_out[0] = H.dr;
    scalars_out[1] = H.dz;
    scalars_out[2] = H.a_ns;
    scalars_out[3] = H.a_c;
  }
  return H.nr;
}

int gsb_create(gsb_ctx **out, int nz, int nr, const double *r_row, const double *z_axis, double dr,
               double dz, int batch_cap, int device) {
  GSB_REQUIRE(out != nullptr, "gsb_create: out is NULL");
  *out = nullptr;
  GSB_REQUIRE(nz >= 2 && nr >= 2, "gsb_create: grid must be at least 2x2");
  GSB_REQUIRE(r_row != nullptr, "gsb_create: r_row is NULL");
  GSB_REQUIRE(batch_cap >= 1, "gsb_create: batch_cap must be >= 1");
  GSB_REQUIRE(std::isfinite(dr) && std::isfinite(dz) && dr > 0 && dz > 0,
              "gsb_create: dr, dz must be finite and > 0");
  int ndev = gsb_device_count();
  if (ndev <= 0 || device < 0 || device >= ndev) {
    set_error("gsb_create: no usable CUDA device (libgsb200 has no CPU fallback)");
    return GSB_ENODEV;
  }
  GSB_CUDA(cudaSetDevice(device));
  gsb_ctx *ctx = new gsb_ctx();
  ctx->device = device;
  cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device);
  ctx->nz = nz;
  ctx->nr = nr;
  ctx->n = (size_t)nz * nr;
  ctx->batch_cap = batch_cap;
  ctx->dr = dr;
  ctx->dz = dz;
  ctx->r_row.assign(r_row, r_row + nr);
  if (z_axis) ctx->z_axis.assign(z_axis, z_axis + nz);
  ctx->n_wall = 2 * nr + 2 * (nz - 2);
  ctx->n_int = (nz - 2) * (nr - 2);
  cudaError_t e = cudaSuccess;
  auto A = [&](void **p, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
  };
  A((void **)&ctx->r_dev, nr * sizeof(double));
  A((void **)&ctx->z_dev, nz * sizeof(double));
  // reduction scratch: at least 8192 doubles in total so a single large grid can use thousands of partial blocks
  ctx->red_stride = std::max(kRedStride, (8192 + batch_cap - 1) / batch_cap);
  A((void **)&ctx->red, (size_t)batch_cap * ctx->red_stride * sizeof(double));
  A((void **)&ctx->active, (size_t)batch_cap * sizeof(int));
  A((void **)&ctx->counter, 4 * sizeof(int));
  A((void **)&ctx->mg_bc, (size_t)batch_cap * ring_size(nz, nr) * sizeof(double));
  if (e == cudaSuccess) e = cudaMallocHost((void **)&ctx->h_counter, 4 * sizeof(int));
  if (e == cudaSuccess)
    e = cudaMemcpy(ctx->r_dev, r_row, nr * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && z_axis)
    e = cudaMemcpy(ctx->z_dev, z_axis, nz * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error(std::string("gsb_create: ") + cudaGetErrorString(e));
    gsb_destroy(ctx);
    return e == cudaErrorMemoryAllocation ? GSB_ENOMEM : GSB_ECUDA;
  }
  *out = ctx;
  return GSB_OK;
}

void gsb_picard_ws_free(gsb_ctx *ctx);  // gsb_picard.cu

void gsb_destroy(gsb_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  gsb_picard_ws_free(ctx);
  free_levels(ctx);
  if (ctx->r_dev) cudaFree(ctx->r_dev);
  if (ctx->z_dev) cudaFree(ctx->z_dev);
  if (ctx->red) cudaFree(ctx->red);
  if (ctx->active) cudaFree(ctx->active);
  if (ctx->counter) cudaFree(ctx->counter);
  if (ctx->mg_bc) cudaFree(ctx->mg_bc);
  if (ctx->split_src) cudaFree(ctx->split_src);
  if (ctx->x_alt) cudaFree(ctx->x_alt);
  if (ctx->gstream) cudaStreamDestroy(ctx->gstream);
  if (ctx->gevent) cudaEventDestroy(ctx->gevent);
  if (ctx->gemm_ws) cudaFree(ctx->gemm_ws);
  if (ctx->fb_old) cudaFree(ctx->fb_old);
  if (ctx->fb_part) cudaFree(ctx->fb_part);
  if (ctx->fb_wall) cudaFree(ctx->fb_wall);
  if (ctx->fb_ints) cudaFree(ctx->fb_ints);
  if (ctx->fb_shape) cudaFree(ctx->fb_shape);
  if (ctx->h_counter) cudaFreeHost(ctx->h_counter);
  delete ctx;
}

}  // extern "C"

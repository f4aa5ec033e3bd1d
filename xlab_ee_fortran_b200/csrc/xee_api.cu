// xee_api.cu — C-ABI (include/xee_b200.h): plan entry points and the Fortran-facing drop-ins for
// module elliptic_tools (xtt-lib-fortran/elliptic_tools.f90) and the driver's FD kernels.
#include "xee_plan.cuh"

namespace xee {
thread_local std::string g_last_error;
std::atomic<long long> g_launches{0};
}  // namespace xee

using namespace xee;

struct xee_plan { PlanBase* impl; };

extern "C" {

const char* xee_last_error(void) { return g_last_error.c_str(); }
int xee_device_count(void) { int n = 0; return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0; }
const char* xee_build_info(void) { return "xee_b200 sm_100a " __DATE__ " " __TIME__; }
long long xee_launch_count(int reset) { return reset ? g_launches.exchange(0) : g_launches.load(); }
void xee_release_cached_memory(void) { DevPool::get().trim(0); }
int xee_pool_stats(long long* live_bytes, long long* cached_bytes) { DevPool::get().stats(live_bytes, cached_bytes); return 0; }

int xee_plan_create(const xee_plan_desc* desc, xee_plan** out) {
  std::unique_ptr<PlanBase> p;
  if (make_plan(desc, &p)) return 1;
  *out = new xee_plan{p.release()};
  return 0;
}
// Every plan entry point runs with the plan's device current (and restores the caller's): a process may hold plans on
// several GPUs.
int xee_plan_destroy(xee_plan* p) { if (p) { DeviceGuard g(p->impl->d.device); delete p->impl; delete p; } return 0; }
int xee_plan_set_coe_aos_host(xee_plan* p, const void* c) { DeviceGuard g(p->impl->d.device); return p->impl->set_coe_aos(c, true); }
int xee_plan_set_coe_aos_dev(xee_plan* p, const void* c) { DeviceGuard g(p->impl->d.device); return p->impl->set_coe_aos(c, false); }
int xee_plan_set_abc_dev(xee_plan* p, const void* a, const void* b, const void* c, double dx, double dy) {
  DeviceGuard g(p->impl->d.device);
  return p->impl->set_abc(a, b, c, dx, dy);
}
int xee_plan_solve_dev(xee_plan* p, void* psi, const void* f, const xee_solve_params* prm, int* iters, double* r1o,
                       double* r2o, int* err, void* stream) {
  DeviceGuard g(p->impl->d.device);
  return p->impl->solve(psi, f, prm, iters, r1o, r2o, err, (cudaStream_t)stream, false, nullptr, 0);
}
int xee_plan_solve_host(xee_plan* p, void* psi, const void* f, const xee_solve_params* prm, int* iters, double* r1o,
                        double* r2o, int* err) {
  DeviceGuard g(p->impl->d.device);
  return p->impl->solve(psi, f, prm, iters, r1o, r2o, err, nullptr, true, nullptr, 0);
}
int xee_plan_sweeps_dev(xee_plan* p, void* psi, const void* f, double alpha, int sweeps, double* rms, void* stream) {
  DeviceGuard g(p->impl->d.device);
  return p->impl->sweeps(psi, f, alpha, sweeps, 0, rms, (cudaStream_t)stream);
}
int xee_plan_sweeps_checked_dev(xee_plan* p, void* psi, const void* f, double alpha, int sweeps, int check_step, double* rms,
                                void* stream) {
  DeviceGuard g(p->impl->d.device);
  return p->impl->sweeps(psi, f, alpha, sweeps, check_step, rms, (cudaStream_t)stream);
}
int xee_plan_apply_dev(xee_plan* p, const void* psi, void* out, void* stream) {
  DeviceGuard g(p->impl->d.device);
  return p->impl->apply(psi, out, (cudaStream_t)stream);
}
int xee_sweep_kernel_stats(xee_plan* p, double* ms, long long* launches, int reset) { return p->impl->kernel_stats(ms, launches, reset); }
int xee_plan_cheb_params(xee_plan* p, double* rho, double* gamma) {
  if (rho) *rho = p->impl->cheb_rho_used;
  if (gamma) *gamma = p->impl->cheb_gamma_used;
  return 0;
}
int xee_plan_kernel_info(xee_plan* p, int* variant, int* sweeps_per_pass, long long* kernel_launches) {
  return p->impl->kernel_info(variant, sweeps_per_pass, kernel_launches);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Fortran-facing drop-ins (Part 1 of xee_b200.h).  void functions cannot return a status, so a CUDA
// failure is fatal: print and abort (never a silent CPU fallback).
namespace {
[[noreturn]] void die(const char* where) {
  fprintf(stderr, "xee_b200: %s failed: %s\n", where, xee_last_error());
  abort();
}

template <class T> constexpr int dtype_of() { return sizeof(T) == 4 ? XEE_F32 : XEE_F64; }

// Small device buffer with H2D upload.
template <class T>
struct DevBuf {
  PoolBuf buf; T* p = nullptr; size_t n = 0;
  explicit DevBuf(size_t n_) : n(n_) { if (buf.alloc(&p, sizeof(T) * (n ? n : 1)) != cudaSuccess) { g_last_error = "cudaMalloc"; die("DevBuf"); } }
  // a pageable H2D cudaMemcpy may return before the DMA has landed, and the plans work on non-blocking streams that the
  // legacy default stream does not order: synchronise the device before anyone reads the buffer
  DevBuf(const T* host, size_t n_) : DevBuf(n_) { if (cudaMemcpy(p, host, sizeof(T) * n, cudaMemcpyHostToDevice) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) { g_last_error = "H2D"; die("DevBuf"); } }
  void to_host(T* host) const { if (cudaMemcpy(host, p, sizeof(T) * n, cudaMemcpyDeviceToHost) != cudaSuccess) { g_last_error = "D2H"; die("DevBuf"); } }
};

std::unique_ptr<PlanBase> new_plan_or_die(int dtype, int nx, int ny, int nbatch, int shared) {
  xee_plan_desc d{};
  d.dtype = dtype; d.nx = nx; d.ny = ny; d.nbatch = nbatch; d.shared_coe = shared; d.device = -1;
  const char* ar = getenv("XEE_ARITH");
  d.arith = (ar && !strcmp(ar, "fast")) ? XEE_ARITH_FAST : XEE_ARITH_STRICT;
  const char* me = getenv("XEE_METHOD");
  d.method = !me ? XEE_METHOD_JACOBI : !strcmp(me, "chebyshev") ? XEE_METHOD_CHEBYSHEV : !strcmp(me, "line_jacobi") ? XEE_METHOD_LINE_JACOBI
             : !strcmp(me, "line_chebyshev") ? XEE_METHOD_LINE_CHEBYSHEV : !strcmp(me, "line2_jacobi") ? XEE_METHOD_LINE2_JACOBI
             : !strcmp(me, "line2_chebyshev") ? XEE_METHOD_LINE2_CHEBYSHEV : !strcmp(me, "line_bicgstab") ? XEE_METHOD_LINE_BICGSTAB
             : !strcmp(me, "line2_bicgstab") ? XEE_METHOD_LINE2_BICGSTAB : !strcmp(me, "line2_mixed") ? XEE_METHOD_LINE2_MIXED
             : XEE_METHOD_JACOBI;
  std::unique_ptr<PlanBase> p;
  if (make_plan(&d, &p)) die("plan create");
  return p;
}

template <class T>
void cal_coe_impl(const T* a, const T* b, const T* c, T* coe, const T* dx, const T* dy, const int* nx, const int* ny, int* err) {
  *err = 1;                                                   // elliptic_tools.f90:33
  const int NX = *nx, NY = *ny;
  std::unique_ptr<PlanBase> p = new_plan_or_die(dtype_of<T>(), NX, NY, 1, 1);
  DevBuf<T> da(a, (size_t)(NX - 1) * (NY - 2)), db(b, (size_t)(NX - 1) * (NY - 1)), dc(c, (size_t)(NX - 2) * (NY - 1));
  if (p->set_abc(da.p, db.p, dc.p, (double)*dx, (double)*dy)) die("cal_coe");
  if (p->coe_to_aos_host(coe)) die("cal_coe");
  *err = 0;                                                   // :58
}

template <class T>
void do_elliptic_impl(const T* psi, const T* coe, T* out, const int* nx, const int* ny, int* err) {
  *err = 1;                                                   // :73 (never cleared by the reference)
  const int NX = *nx, NY = *ny;
  const size_t nn = (size_t)NX * NY;
  std::unique_ptr<PlanBase> p = new_plan_or_die(dtype_of<T>(), NX, NY, 1, 1);
  if (p->set_coe_aos(coe, true)) die("do_elliptic");
  DevBuf<T> dpsi(psi, nn), dout(nn);
  if (p->apply(dpsi.p, dout.p, nullptr)) die("do_elliptic");
  if (cudaDeviceSynchronize() != cudaSuccess) die("do_elliptic");
  std::vector<T> h(nn);
  dout.to_host(h.data());
  for (int j = 1; j < NY - 1; ++j)    // interior only; boundary of outdat untouched (:75-76)
    memcpy(out + (size_t)j * NX + 1, h.data() + (size_t)j * NX + 1, sizeof(T) * (NX - 2));
}

template <class T>
void solve_elliptic_impl(int* max_iter, const int* check_step, const int* converge_time, const int* lost_rate,
                         T* r1, T* r2, const T* alpha, T* dat, const T* coe, const T* f, T* workspace, const int* nx,
                         const int* ny, int* err, const int* debug) {
  // :112-129
  const bool check_abs = *r1 > 0, check_rel = *r2 > 0;
  if (!check_abs) *r1 = xee::Rn<T>::huge();
  if (!check_rel) *r2 = xee::Rn<T>::huge();
  if (!check_abs && !check_rel) {
    printf(" ERROR: [check_abs_err] and [check_rel_err] cannot both be non-positive.\n");
    fflush(stdout);
    exit(0);   // Fortran STOP
  }
  const int cs = *check_step > 0 ? *check_step : 100, ct = *converge_time > 0 ? *converge_time : 10;
  if (*debug == 1 || *debug == 2) {                            // :146-158
    printf(" ----- Solve Elliptic Inputs -----\n");
    printf("   max_iter       :  %11d\n", *max_iter);
    printf("   strategy_r1    :  %.8E\n", (double)*r1);
    printf("   strategy_r2    :  %.8E\n", (double)*r2);
    printf("   alpha          :  %.8E\n", (double)*alpha);
    printf("   (nx, ny)       : ( %11d ,  %11d )\n", *nx, *ny);
    printf("   alpha          :  %.8E\n", (double)*alpha);
    printf("   debug          :  %11d\n", *debug);
    printf("   check step     :  %11d\n", cs);
    printf("   converge time :  %11d\n", ct);
    printf(" ---------------------------------\n");
  }
  *err = 0;                                                    // :164
  if (*max_iter <= 0) { memcpy(workspace, dat, sizeof(T) * (size_t)*nx * *ny); return; }  // loop body never runs
  std::unique_ptr<PlanBase> p = new_plan_or_die(dtype_of<T>(), *nx, *ny, 1, 1);
  if (p->set_coe_aos(coe, true)) die("solve_elliptic");
  xee_solve_params prm{};
  prm.max_iter = *max_iter; prm.check_step = *check_step; prm.converge_time = *converge_time; prm.lost_rate = *lost_rate;
  prm.r1 = check_abs ? (double)*r1 : 0.0; prm.r2 = check_rel ? (double)*r2 : 0.0; prm.alpha = (double)*alpha;
  prm.sync_every = 2;
  // XEE_STALL_CHECKS=N (opt-in, for the accelerated methods): the reference's rule needs |ratio| < r2 on converge_time
  // checks, which round-off noise can deny for ever once an accelerated iteration sits on its residual floor.  With N > 0 a
  // solve whose best residual has not improved for N checks stops; if the absolute criterion r1 is met there, that is success.
  prm.stall_checks = env_int("XEE_STALL_CHECKS", 0);
  int iters = 0, e = 0; double r1o = 0, r2o = 0;
  if (p->solve(dat, f, &prm, &iters, &r1o, &r2o, &e, nullptr, true, workspace, *debug)) die("solve_elliptic");
  if ((e & XEE_ERR_STALLED) && check_abs && r1o < (double)*r1) e &= ~XEE_ERR_STALLED;
  *err = e;
  if (*debug == 2) {
    if (e & XEE_ERR_OVER_MAX_ITERATION) printf(" Max iteration reached. Exit iteration.\n");
    printf(" iter :  %11d , err_avg =   %.8E\n", iters, r1o);
  }
  *max_iter = iters; *r1 = (T)r1o; *r2 = (T)r2o;                // :253
  xee_judge_error(err);                                        // :254
}

// Legacy 12-argument solve_elliptic (src/old-diagnose/xtt-lib/elliptic_tools.f90:93-300) on top of the current solver:
//   strategy 1 = r1 only, converge_time 1;   strategy 2 = r2 only, converge_time 10, lost_rate 5;
//   strategies 3 / 4 = the same two rules on err_now = maxval(abs(to_dat)) (:203-204): the largest |residual| of the interior
//   joined with the largest |value| on the rim of the array (to_dat's rim holds the Dirichlet values of dat).
template <class T>
void solve_elliptic_old_impl(const int* max_iter, int* strategy, T* strategy_r, const T* alpha, T* dat, const T* coe,
                             const T* f, T* workspace, const int* nx, const int* ny, int* err, const int* debug) {
  *err = 0;
  if (*strategy < 1 || *strategy > 4) { *err = 1 << 8; fprintf(stderr, "xee_b200: legacy strategy %d does not exist (1..4)\n", *strategy); return; }
  const bool maxnorm = *strategy >= 3, absolute = (*strategy & 1) != 0;
  // The legacy loop `do cnt = 1, max_iter` (:168) runs ALL max_iter sweeps; the stop tests and `cnt == max_iter` are evaluated
  // on check sweeps only (every 100th, :293-305).  A run that never stops on a check and whose max_iter is not a multiple of
  // 100 therefore falls out of the loop with err = 0, strategy / strategy_r untouched and judge_error not called.
  const int mi = *max_iter;
  if (mi <= 0) { memcpy(workspace, dat, sizeof(T) * (size_t)*nx * *ny); return; }
  std::unique_ptr<PlanBase> p = new_plan_or_die(dtype_of<T>(), *nx, *ny, 1, 1);
  if (p->set_coe_aos(coe, true)) die("solve_elliptic(old)");
  if (maxnorm) {
    const int NX = *nx, NY = *ny;
    double m = 0.0;
    auto join = [&](T v) { const double a = std::fabs((double)v); m = (m != m) ? m : (a != a) ? a : std::max(m, a); };
    for (int i = 0; i < NX; ++i) { join(dat[i]); join(dat[(size_t)(NY - 1) * NX + i]); }
    for (int j = 0; j < NY; ++j) { join(dat[(size_t)j * NX]); join(dat[(size_t)j * NX + NX - 1]); }
    p->norm_max = 1; p->norm_floor = m;
  }
  xee_solve_params prm{};
  prm.max_iter = mi; prm.check_step = 100; prm.alpha = (double)*alpha; prm.sync_every = 2;
  prm.detect_explode = 1;   // the legacy isnan tests (:218-240) set err_explode; here: a non-finite residual at a check
  if (absolute) { prm.r1 = (double)*strategy_r; prm.r2 = 0.0; prm.converge_time = 1; prm.lost_rate = 5; if (!(prm.r1 > 0)) prm.r1 = 1e-300; }
  else { prm.r1 = 0.0; prm.r2 = (double)*strategy_r; prm.converge_time = 10; prm.lost_rate = 5; if (!(prm.r2 > 0)) prm.r2 = 1e-300; }
  int iters = 0, e = 0; double r1o = 0, r2o = 0;
  if (p->solve(dat, f, &prm, &iters, &r1o, &r2o, &e, nullptr, true, workspace, *debug == 1 ? 2 : 0)) die("solve_elliptic(old)");
  if ((mi % 100) != 0 && iters == mi && (e & XEE_ERR_OVER_MAX_ITERATION)) {   // fell out of the loop between two checks
    *err = e & ~XEE_ERR_OVER_MAX_ITERATION;
    return;
  }
  *err = e; *strategy = iters; *strategy_r = (T)r1o;
  xee_judge_error(err);
}

template <class T>
struct PhysConst {  // constants.f90:4-5 evaluated in T
  T g0 = T(9.8), theta0 = T(298.0), Rd = T(287.0), Cv, Cp;
  PhysConst() { Cv = T(5.0) / T(2.0) * Rd; Cp = Cv + Rd; }
};

template <class T>
int eta_dev_impl(const void* rchi, void* eta, const void* ra, const void* rc, const void* rho, const void* ex, int nr,
                 int nz, int nb, cudaStream_t s) {
  PhysConst<T> k;
  dim3 g((nr - 1 + 127) / 128, nz, nb);
  xee::eta_kernel<T><<<g, 128, 0, s>>>((const T*)rchi, (T*)eta, (const T*)ra, (const T*)rc, (const T*)rho, (const T*)ex, nr, nz, k.g0, k.Cp, k.theta0);
  XEE_LAUNCH_OK();
  return 0;
}
template <class T>
int uw_dev_impl(const void* rpsi, void* u, void* w, const void* ra, const void* rc, const void* za, const void* rho,
                int nr, int nz, int nb, cudaStream_t s) {
  dim3 g((nr + 127) / 128, nz, nb);
  xee::uw_kernel<T><<<g, 128, 0, s>>>((const T*)rpsi, (T*)u, (T*)w, (const T*)ra, (const T*)rc, (const T*)za, (const T*)rho, nr, nz);
  XEE_LAUNCH_OK();
  return 0;
}

template <class T>
void cal_eta_impl(const T* rchi, T* eta, const T* ra, const T* rc, const T* rho, const T* ex, const int* nr, const int* nz) {
  const int NR = *nr, NZ = *nz;
  DevBuf<T> d_in(rchi, (size_t)NR * NZ), d_out((size_t)(NR - 1) * NZ), dra(ra, NR), drc(rc, NR), drho(rho, NZ), dex(ex, NZ);
  if (eta_dev_impl<T>(d_in.p, d_out.p, dra.p, drc.p, drho.p, dex.p, NR, NZ, 1, nullptr)) die("cal_eta");
  d_out.to_host(eta);
}
template <class T>
void cal_uw_impl(const T* rpsi, T* u, T* w, const T* ra, const T* rc, const T* za, const T* rho, const int* nr, const int* nz) {
  const int NR = *nr, NZ = *nz;
  DevBuf<T> d_in(rpsi, (size_t)NR * NZ), du((size_t)NR * (NZ - 1)), dw((size_t)(NR - 1) * NZ), dra(ra, NR), drc(rc, NR), dza(za, NZ), drho(rho, NZ);
  if (uw_dev_impl<T>(d_in.p, du.p, dw.p, dra.p, drc.p, dza.p, drho.p, NR, NZ, 1, nullptr)) die("cal_uw");
  du.to_host(u); dw.to_host(w);
}
template <class T>
void build_abc_impl(const T* A, const T* B, const T* C, const T* rc, const T* rho, T* a, T* b, T* c, const int* nr, const int* nz) {
  const int NR = *nr, NZ = *nz;
  const size_t nn = (size_t)NR * NZ;
  DevBuf<T> dA(A, nn), dB(B, nn), dC(C, nn), drc(rc, NR), drho(rho, NZ);
  DevBuf<T> da((size_t)(NR - 1) * (NZ - 2)), db((size_t)(NR - 1) * (NZ - 1)), dc((size_t)(NR - 2) * (NZ - 1));
  dim3 blk(64, 4), g((NR + 63) / 64, (NZ + 3) / 4);
  xee::build_abc_kernel<T><<<g, blk>>>(dA.p, dB.p, dC.p, drc.p, drho.p, da.p, db.p, dc.p, NR, NZ);
  g_launches.fetch_add(1);
  if (cudaGetLastError() != cudaSuccess) { g_last_error = "build_abc launch"; die("build_abc"); }
  da.to_host(a); db.to_host(b); dc.to_host(c);
}
}  // namespace

extern "C" {
void xee_cal_coe_f32(const float* a, const float* b, const float* c, float* coe, const float* dx, const float* dy, const int* nx, const int* ny, int* err) { cal_coe_impl<float>(a, b, c, coe, dx, dy, nx, ny, err); }
void xee_cal_coe_f64(const double* a, const double* b, const double* c, double* coe, const double* dx, const double* dy, const int* nx, const int* ny, int* err) { cal_coe_impl<double>(a, b, c, coe, dx, dy, nx, ny, err); }
void xee_do_elliptic_f32(const float* psi, const float* coe, float* out, const int* nx, const int* ny, int* err) { do_elliptic_impl<float>(psi, coe, out, nx, ny, err); }
void xee_do_elliptic_f64(const double* psi, const double* coe, double* out, const int* nx, const int* ny, int* err) { do_elliptic_impl<double>(psi, coe, out, nx, ny, err); }
void xee_solve_elliptic_f32(int* max_iter, const int* check_step, const int* converge_time, const int* lost_rate, float* r1, float* r2, const float* alpha, float* dat, const float* coe, const float* f, float* workspace, const int* nx, const int* ny, int* err, const int* debug) {
  solve_elliptic_impl<float>(max_iter, check_step, converge_time, lost_rate, r1, r2, alpha, dat, coe, f, workspace, nx, ny, err, debug);
}
void xee_solve_elliptic_f64(int* max_iter, const int* check_step, const int* converge_time, const int* lost_rate, double* r1, double* r2, const double* alpha, double* dat, const double* coe, const double* f, double* workspace, const int* nx, const int* ny, int* err, const int* debug) {
  solve_elliptic_impl<double>(max_iter, check_step, converge_time, lost_rate, r1, r2, alpha, dat, coe, f, workspace, nx, ny, err, debug);
}
void xee_solve_elliptic_old_f32(const int* max_iter, int* strategy, float* strategy_r, const float* alpha, float* dat, const float* coe, const float* f, float* workspace, const int* nx, const int* ny, int* err, const int* debug) {
  solve_elliptic_old_impl<float>(max_iter, strategy, strategy_r, alpha, dat, coe, f, workspace, nx, ny, err, debug);
}
void xee_solve_elliptic_old_f64(const int* max_iter, int* strategy, double* strategy_r, const double* alpha, double* dat, const double* coe, const double* f, double* workspace, const int* nx, const int* ny, int* err, const int* debug) {
  solve_elliptic_old_impl<double>(max_iter, strategy, strategy_r, alpha, dat, coe, f, workspace, nx, ny, err, debug);
}
void xee_judge_error(const int* err) {   // elliptic_tools.f90:333-358
  const int e = *err;
  bool known = false;
  if (e == 0) { printf(" Elliptic Tools: Iteration success.\n"); known = true; }
  if (e & XEE_ERR_OVER_MAX_ITERATION) { printf(" Elliptic Tools: [Error] Max iteration reached.\n"); known = true; }
  if (e & XEE_ERR_EXPLODE) { printf(" Elliptic Tools: [Error] Iteration explodes.\n"); known = true; }
  if (!known) printf(" Elliptic Tools: Unknown error code %12d\n", e);
  fflush(stdout);
}
void xee_build_abc_f32(const float* A, const float* B, const float* C, const float* rc, const float* rho, float* a, float* b, float* c, const int* nr, const int* nz) { build_abc_impl<float>(A, B, C, rc, rho, a, b, c, nr, nz); }
void xee_build_abc_f64(const double* A, const double* B, const double* C, const double* rc, const double* rho, double* a, double* b, double* c, const int* nr, const int* nz) { build_abc_impl<double>(A, B, C, rc, rho, a, b, c, nr, nz); }
void xee_cal_eta_f32(const float* rchi, float* eta, const float* ra, const float* rc, const float* rho, const float* ex, const int* nr, const int* nz) { cal_eta_impl<float>(rchi, eta, ra, rc, rho, ex, nr, nz); }
void xee_cal_eta_f64(const double* rchi, double* eta, const double* ra, const double* rc, const double* rho, const double* ex, const int* nr, const int* nz) { cal_eta_impl<double>(rchi, eta, ra, rc, rho, ex, nr, nz); }
void xee_cal_uw_f32(const float* rpsi, float* u, float* w, const float* ra, const float* rc, const float* za, const float* rho, const int* nr, const int* nz) { cal_uw_impl<float>(rpsi, u, w, ra, rc, za, rho, nr, nz); }
void xee_cal_uw_f64(const double* rpsi, double* u, double* w, const double* ra, const double* rc, const double* za, const double* rho, const int* nr, const int* nz) { cal_uw_impl<double>(rpsi, u, w, ra, rc, za, rho, nr, nz); }

int xee_eta_dev(int dtype, const void* rchi, void* eta, const void* ra, const void* rc, const void* rho, const void* ex, int nr, int nz, int nb, void* stream) {
  return dtype == XEE_F32 ? eta_dev_impl<float>(rchi, eta, ra, rc, rho, ex, nr, nz, nb, (cudaStream_t)stream)
                          : eta_dev_impl<double>(rchi, eta, ra, rc, rho, ex, nr, nz, nb, (cudaStream_t)stream);
}
int xee_uw_dev(int dtype, const void* rpsi, void* u, void* w, const void* ra, const void* rc, const void* za, const void* rho, int nr, int nz, int nb, void* stream) {
  return dtype == XEE_F32 ? uw_dev_impl<float>(rpsi, u, w, ra, rc, za, rho, nr, nz, nb, (cudaStream_t)stream)
                          : uw_dev_impl<double>(rpsi, u, w, ra, rc, za, rho, nr, nz, nb, (cudaStream_t)stream);
}
}  // extern "C"

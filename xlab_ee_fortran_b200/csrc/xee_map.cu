// xee_map.cu — the efficiency-map pipeline: one balanced vortex (A,B,C), many heating locations,
// one elliptic solve per location, all on the device.
//
//   geometry (host scalars)     src/diagnose/initialize-variables.f90:45-67
//   K1 build_abc_kernel         initialize-variables.f90:72-95
//   K2 cal_coe_kernel           xtt-lib-fortran/elliptic_tools.f90:35-56
//   background theta            src/old-diagnose/diagnose.f90:329-354, 503-509, 893-912 (testing_dt = 0)
//   K7 heating_rhs_kernel       old-diagnose/diagnose.f90:383-387 (J = Q/(Cp Pi)), :396-406 (g/theta0 dJ/dr -> O)
//   K3/K4 batched solve         elliptic_tools.f90:93-265
//   K6 ke_generation_kernel     old-diagnose/diagnose.f90:915-941 (w), :1117-1127 (w theta), :1094-1113 (integral)
//      sum_q_kernel             :1050-1071      qeta_kernel  :1073-1092 (adjoint check through eta)
//
// The legacy driver's latent bugs are not reproduced; the intended maths is (SURVEY section 7):
// Q is a genuine B-grid (nr-1,nz-1) field, theta is the background state (testing_dt = 0).
#include "xee_map_kernels.cuh"

namespace xee {

struct MapBase {
  xee_map_desc d{};
  int device() const { return d.device; }
  virtual ~MapBase() {}
  virtual int run(const double* heat, bool heat_on_host, const xee_solve_params* prm, double* table, bool table_on_host,
                  cudaStream_t s) = 0;
  virtual PlanBase* plan() = 0;
  virtual int get_field(int which, void* host_out) = 0;
};

template <class T>
struct Map : MapBase, PoolOwner {
  std::unique_ptr<Plan<T>> pl;      // batched solves (shared operator)
  std::unique_ptr<Plan<T>> pl1;     // the single adjoint (chi) solve
  T *A = nullptr, *B = nullptr, *C = nullptr, *ra = nullptr, *za = nullptr, *ex = nullptr, *rho = nullptr,
    *theta = nullptr, *eta = nullptr, *chi = nullptr, *fchi = nullptr, *psi = nullptr, *f = nullptr, *r1v = nullptr;
  Heat* heat_d = nullptr;
  double* integ = nullptr;    // [n][3]
  std::vector<T> h_ra, h_za, h_ex, h_rho;
  T dr = 0, dz = 0;
  size_t nn = 0;
  PhysK<T> k;

  PlanBase* plan() override { return pl.get(); }

  int init(const float* hA, const float* hB, const float* hC) {
    TraceTimer tt("map init (total)");
    const int nr = d.nr, nz = d.nz, nb = d.nheat;
    nn = (size_t)nr * nz;
    // geometry scalars on the host, in T, exactly as initialize-variables.f90:45-57 (std::pow == gfortran's **)
    dr = (T(d.Lr[1]) - T(d.Lr[0])) / T(nr - 1);
    dz = (T(d.Lz[1]) - T(d.Lz[0])) / T(nz - 1);
    h_ra.resize(nr); h_za.resize(nz); h_ex.resize(nz); h_rho.resize(nz);
    for (int i = 1; i <= nr; ++i) h_ra[i - 1] = T(d.Lr[0]) + T(i - 1) * dr;
    for (int j = 1; j <= nz; ++j) {
      h_za[j - 1] = T(d.Lz[0]) + T(j - 1) * dz;
      h_ex[j - 1] = d.density_mode == 0 ? (T(1.0) - h_za[j - 1] / k.h0) : T(1.0);
      h_rho[j - 1] = d.density_mode == 0 ? k.p0 / (k.theta0 * k.Rd) * std::pow(h_ex[j - 1], T(1.0) / k.kappa - T(1.0)) : T(1.0);
    }
    xee_plan_desc pd{};
    pd.dtype = d.dtype; pd.nx = nr; pd.ny = nz; pd.nbatch = nb; pd.shared_coe = 1; pd.arith = d.arith; pd.method = d.method;
    pd.device = d.device;
    pl.reset(new Plan<T>()); pl->d = pd;
    if (pl->init()) return 1;
    cudaStream_t s = pl->own_stream;
    XEE_CHECK(own(&A, sizeof(T) * nn)); XEE_CHECK(own(&B, sizeof(T) * nn)); XEE_CHECK(own(&C, sizeof(T) * nn));
    XEE_CHECK(own(&ra, sizeof(T) * nr)); XEE_CHECK(own(&za, sizeof(T) * nz));
    XEE_CHECK(own(&ex, sizeof(T) * nz)); XEE_CHECK(own(&rho, sizeof(T) * nz));
    XEE_CHECK(own(&theta, sizeof(T) * (nr - 1) * (nz - 1)));
    XEE_CHECK(own(&psi, sizeof(T) * nn * nb)); XEE_CHECK(own(&f, sizeof(T) * nn * nb));
    XEE_CHECK(own(&r1v, sizeof(T) * nb));
    XEE_CHECK(own(&heat_d, sizeof(Heat) * nb)); XEE_CHECK(own(&integ, sizeof(double) * 3 * nb));
    XEE_CHECK(cudaMemcpyAsync(ra, h_ra.data(), sizeof(T) * nr, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(za, h_za.data(), sizeof(T) * nz, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(ex, h_ex.data(), sizeof(T) * nz, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(rho, h_rho.data(), sizeof(T) * nz, cudaMemcpyHostToDevice, s));
    // inputs arrive in the reference's file format: headerless float32, i fastest (field_tools.f90:30-52)
    float* stage = nullptr;
    PoolBuf stage_buf;
    XEE_CHECK(stage_buf.alloc(&stage, sizeof(float) * nn * 3));
    XEE_CHECK(cudaMemcpyAsync(stage, hA, sizeof(float) * nn, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(stage + nn, hB, sizeof(float) * nn, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(stage + 2 * nn, hC, sizeof(float) * nn, cudaMemcpyHostToDevice, s));
    const unsigned gb = (unsigned)((nn + 255) / 256);
    f32_to_T_kernel<T><<<gb, 256, 0, s>>>(stage, A, nn); XEE_LAUNCH_OK();
    f32_to_T_kernel<T><<<gb, 256, 0, s>>>(stage + nn, B, nn); XEE_LAUNCH_OK();
    f32_to_T_kernel<T><<<gb, 256, 0, s>>>(stage + 2 * nn, C, nn); XEE_LAUNCH_OK();
    // K1 + K2 (cylindrical: rcuva = ra)
    T *a = nullptr, *b = nullptr, *c = nullptr;
    PoolBuf a_buf, b_buf, c_buf;
    XEE_CHECK(a_buf.alloc(&a, sizeof(T) * (nr - 1) * (nz - 2))); XEE_CHECK(b_buf.alloc(&b, sizeof(T) * (nr - 1) * (nz - 1)));
    XEE_CHECK(c_buf.alloc(&c, sizeof(T) * (nr - 2) * (nz - 1)));
    dim3 blk(64, 4), g((nr + 63) / 64, (nz + 3) / 4);
    build_abc_kernel<T><<<g, blk, 0, s>>>(A, B, C, ra, rho, a, b, c, nr, nz); XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(s));
    if (pl->set_abc(a, b, c, (double)dr, (double)dz)) return 1;
    background_theta_kernel<T><<<1, 256, 0, s>>>(A, B, theta, ra, za, nr, nz, k.g0, k.theta0); XEE_LAUNCH_OK();
    if (d.adjoint_check) {
      pd.nbatch = 1;
      pl1.reset(new Plan<T>()); pl1->d = pd;
      if (pl1->init()) return 1;
      XEE_CHECK(cudaStreamSynchronize(s));
      if (pl1->set_abc(a, b, c, (double)dr, (double)dz)) return 1;
      XEE_CHECK(own(&eta, sizeof(T) * (nr - 1) * nz)); XEE_CHECK(own(&chi, sizeof(T) * nn));
      XEE_CHECK(own(&fchi, sizeof(T) * nn));
    }
    XEE_CHECK(cudaStreamSynchronize(s));
    return 0;
  }
  ~Map() override {
    TraceTimer tt("map destroy");
    cudaDeviceSynchronize();   // the device is done with the owned blocks before they go back to the pool (see ~Plan)
  }

  // table row: iters, r1, err, sum_Q, ke_gen=(g0/theta0) I[w theta], eff=ke_gen/sum_Q, sum_Qeta, eff_eta=sum_Qeta/sum_Q
  int run(const double* heat, bool heat_on_host, const xee_solve_params* prm_in, double* table, bool table_on_host,
          cudaStream_t s) override {
    TraceTimer tt("map run (total)");
    const int nr = d.nr, nz = d.nz, nb = d.nheat;
    if (!s) s = pl->own_stream;
    XEE_CHECK(cudaMemcpyAsync(heat_d, heat, sizeof(Heat) * nb, heat_on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
    heating_rhs_kernel<T><<<heating_rhs_grid(nr, nz, nb), dim3(kHeatBX, kHeatBY), 0, s>>>(heat_d, f, ra, za, ex, nr, nz, k.g0, k.theta0, k.Cp); XEE_LAUNCH_OK();
    XEE_CHECK(cudaMemsetAsync(psi, 0, sizeof(T) * nn * nb, s));     // rpsi = 0: boundary condition and first guess
    xee_solve_params prm = *prm_in;
    if (d.r1_rel_rms_f > 0) {   // tolerance relative to each location's own forcing: r1_n = r1_rel * rms(f_n)
      rms_interior_kernel<T><<<nb, 256, 0, s>>>(f, nr, nz, (T)d.r1_rel_rms_f, r1v); XEE_LAUNCH_OK();
      prm.r1 = 1.0; prm.r1_per_solve = r1v;
    }
    std::vector<int> iters(nb), err(nb);
    std::vector<double> r1o(nb), r2o(nb);
    {
      TraceTimer t1("  map: batched solve");
      if (pl->solve(psi, f, &prm, iters.data(), r1o.data(), r2o.data(), err.data(), s, false, nullptr, 0)) return 1;
    }
    if (d.adjoint_check) {
      TraceTimer t2("  map: adjoint chi solve + eta");
      dim3 g1((nr + 127) / 128, nz, 1);
      rhs_from_B_kernel<T><<<g1, 128, 0, s>>>(B, fchi, nr, nz); XEE_LAUNCH_OK();
      XEE_CHECK(cudaMemsetAsync(chi, 0, sizeof(T) * nn, s));
      xee_solve_params p1 = *prm_in;
      T* r1c = nullptr;
      PoolBuf r1c_buf;
      if (d.r1_rel_rms_f > 0) {
        XEE_CHECK(r1c_buf.alloc(&r1c, sizeof(T)));
        rms_interior_kernel<T><<<1, 256, 0, s>>>(fchi, nr, nz, (T)d.r1_rel_rms_f, r1c); XEE_LAUNCH_OK();
        p1.r1 = 1.0; p1.r1_per_solve = r1c;
      }
      int it1, e1; double a1, a2;
      if (pl1->solve(chi, fchi, &p1, &it1, &a1, &a2, &e1, s, false, nullptr, 0)) return 1;
      dim3 ge((nr - 1 + 127) / 128, nz, 1);
      eta_kernel<T><<<ge, 128, 0, s>>>(chi, eta, ra, ra, rho, ex, nr, nz, k.g0, k.Cp, k.theta0); XEE_LAUNCH_OK();
    }
    map_integrals_kernel<T><<<nb, 256, 0, s>>>(heat_d, psi, theta, d.adjoint_check ? eta : nullptr, ra, ra, za, rho, nr, nz, integ);
    XEE_LAUNCH_OK();
    std::vector<double> hi(3 * (size_t)nb);
    XEE_CHECK(cudaMemcpyAsync(hi.data(), integ, sizeof(double) * 3 * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    std::vector<double> rows((size_t)nb * XEE_MAP_COLS);
    const double gth = (double)k.g0 / (double)k.theta0;
    for (int n = 0; n < nb; ++n) {
      double* r = &rows[(size_t)n * XEE_MAP_COLS];
      r[0] = iters[n]; r[1] = r1o[n]; r[2] = err[n];
      r[3] = hi[3 * n]; r[4] = hi[3 * n + 1] * gth; r[5] = r[4] / r[3];
      r[6] = hi[3 * n + 2]; r[7] = r[6] / r[3];
    }
    if (table_on_host) memcpy(table, rows.data(), sizeof(double) * rows.size());
    else { XEE_CHECK(cudaMemcpyAsync(table, rows.data(), sizeof(double) * rows.size(), cudaMemcpyHostToDevice, s)); XEE_CHECK(cudaStreamSynchronize(s)); }
    return 0;
  }
  int get_field(int which, void* out) override {
    const int nr = d.nr, nz = d.nz;
    const void* src = nullptr; size_t bytes = 0;
    switch (which) {
      case 0: src = psi; bytes = sizeof(T) * nn * d.nheat; break;
      case 1: src = f; bytes = sizeof(T) * nn * d.nheat; break;
      case 2: src = theta; bytes = sizeof(T) * (nr - 1) * (nz - 1); break;
      case 3: src = eta; bytes = sizeof(T) * (nr - 1) * nz; break;
      case 4: src = chi; bytes = sizeof(T) * nn; break;
      default: return fail("xee_map_get_field: unknown field");
    }
    if (!src) return fail("xee_map_get_field: field not computed (adjoint_check off?)");
    XEE_CHECK(cudaMemcpy(out, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
  }
};

}  // namespace xee

using namespace xee;
struct xee_map { MapBase* impl; };

extern "C" {
int xee_map_create(const xee_map_desc* desc, const float* A, const float* B, const float* C, xee_map** out) {
  int dev = 0;
  if (resolve_device(desc->device, &dev)) return 1;
  DeviceGuard guard(dev);
  if (desc->nr < 4 || desc->nz < 4 || desc->nheat < 1) return fail("xee_map: nr, nz >= 4 and nheat >= 1 required");
  std::unique_ptr<MapBase> m; int rc;
  if (desc->dtype == XEE_F32) { auto* q = new Map<float>(); m.reset(q); q->d = *desc; q->d.device = dev; rc = q->init(A, B, C); }
  else if (desc->dtype == XEE_F64) { auto* q = new Map<double>(); m.reset(q); q->d = *desc; q->d.device = dev; rc = q->init(A, B, C); }
  else return fail("xee_map: dtype must be XEE_F32 or XEE_F64");
  if (rc) return 1;
  *out = new xee_map{m.release()};
  return 0;
}
int xee_map_destroy(xee_map* m) { if (m) { DeviceGuard g(m->impl->device()); delete m->impl; delete m; } return 0; }
int xee_map_run_host(xee_map* m, const double* heat, const xee_solve_params* prm, double* table) {
  DeviceGuard g(m->impl->device());
  return m->impl->run(heat, true, prm, table, true, nullptr);
}
int xee_map_run_dev(xee_map* m, const double* heat_dev, const xee_solve_params* prm, double* table_dev, void* stream) {
  DeviceGuard g(m->impl->device());
  return m->impl->run(heat_dev, false, prm, table_dev, false, (cudaStream_t)stream);
}
int xee_map_get_field(xee_map* m, int which, void* host_out) { DeviceGuard g(m->impl->device()); return m->impl->get_field(which, host_out); }
int xee_map_sweep_kernel_stats(xee_map* m, double* ms, long long* launches, int reset) { return m->impl->plan()->kernel_stats(ms, launches, reset); }
int xee_map_kernel_info(xee_map* m, int* variant, int* sweeps_per_pass, long long* kernel_launches) {
  return m->impl->plan()->kernel_info(variant, sweeps_per_pass, kernel_launches);
}
}  // extern "C"

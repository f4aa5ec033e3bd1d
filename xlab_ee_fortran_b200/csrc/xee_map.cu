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
//   discrete adjoint            xee_adjoint_kernels.cuh: one solve of L^T lambda = g, then the exact efficiency of any
//                               number of heating distributions as weighted sums (adjoint_solve, adjoint_eval)
//
// The legacy driver's latent bugs are not reproduced; the intended maths is (SURVEY section 7):
// Q is a genuine B-grid (nr-1,nz-1) field, theta is the background state (testing_dt = 0).
#include "xee_adjoint_kernels.cuh"

namespace xee {

struct MapBase {
  xee_map_desc d{};
  int device() const { return d.device; }
  virtual ~MapBase() {}
  virtual int run(const double* heat, bool heat_on_host, const xee_solve_params* prm, double* table, bool table_on_host,
                  cudaStream_t s) = 0;
  virtual PlanBase* plan() = 0;
  virtual int get_field(int which, void* host_out) = 0;
  virtual int adjoint_solve(const xee_solve_params* prm, int* iters, double* r1, int* err) = 0;
  virtual int adjoint_eval(const double* heat_host, int n, double* table_host) = 0;
  virtual int adjoint_timings(double* setup_ms, double* probe_ms, double* sweep_ms) = 0;
};

template <class T>
struct Map : MapBase, PoolOwner {
  std::unique_ptr<Plan<T>> pl;      // batched solves (shared operator)
  std::unique_ptr<Plan<T>> pl1;     // the single adjoint (chi) solve
  std::unique_ptr<Plan<T>> pla;     // the discrete adjoint: L^T, made by the first adjoint_solve
  T *adj_g = nullptr, *adj_lam = nullptr, *adj_mu = nullptr, *adj_eta = nullptr, *adj_r1 = nullptr;
  bool adj_ready = false;           // lambda, mu and eta_d hold the result of an adjoint solve
  double adj_setup_ms = 0.0;
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
    relative_theta_kernel<T><<<1, 256, 0, s>>>(BasicState<T>{A, B, nr, nz}, theta, ra, za, nr, nz, k.g0, k.theta0); XEE_LAUNCH_OK();
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
    heating_rhs_kernel<T><<<heating_rhs_grid(nr, nz, nb), dim3(kHeatBX, kHeatBY), 0, s>>>(BlobQ<T>{heat_d}, f, ra, za, ex, nr, nz, k.g0, k.theta0, k.Cp); XEE_LAUNCH_OK();
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
      rhs_from_B_kernel<T><<<g1, 128, 0, s>>>(OGridB<T>{B, nr, nz}, fchi, nr, nz); XEE_LAUNCH_OK();
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
    map_integrals_kernel<T><<<nb, 256, 0, s>>>(BlobQ<T>{heat_d}, psi, theta, d.adjoint_check ? eta : nullptr, ra, ra, za, rho, nr, nz, integ);
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
      case 5: src = adj_ready ? adj_eta : nullptr; bytes = sizeof(T) * (nr - 1) * (nz - 1); break;
      case 6: src = adj_ready ? adj_lam : nullptr; bytes = sizeof(T) * nn; break;
      default: return fail("xee_map_get_field: unknown field");
    }
    if (!src) return fail(which >= 5 ? "xee_map_get_field: field not computed (no xee_map_adjoint_solve yet)"
                                     : "xee_map_get_field: field not computed (adjoint_check off?)");
    XEE_CHECK(cudaMemcpy(out, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
  }

  // Discrete adjoint (xee_adjoint_kernels.cuh).  The first call makes a single-solve plan of the map's dtype, arithmetic and
  // method and writes L^T into it; its line factors, coarse operator and spectral estimate are then those of L^T.
  int adjoint_setup() {
    const double t0 = TraceTimer::now();
    const int nr = d.nr, nz = d.nz;
    xee_plan_desc pd = pl->d;
    pd.nbatch = 1;
    std::unique_ptr<Plan<T>> p(new Plan<T>()); p->d = pd;
    if (p->init()) return 1;
    cudaStream_t s = p->own_stream;
    XEE_CHECK(own(&adj_g, sizeof(T) * nn)); XEE_CHECK(own(&adj_lam, sizeof(T) * nn));
    XEE_CHECK(own(&adj_mu, sizeof(T) * (nr - 1) * (nz - 1))); XEE_CHECK(own(&adj_eta, sizeof(T) * (nr - 1) * (nz - 1)));
    XEE_CHECK(own(&adj_r1, sizeof(T)));
    XEE_CHECK(cudaStreamSynchronize(pl->own_stream));   // L is complete
    transpose_coe_kernel<T><<<dim3((nr + 127) / 128, nz), 128, 0, s>>>(pl->coe, p->coe, nr, nz); XEE_LAUNCH_OK();
    if (p->operator_written()) return 1;
    ke_functional_kernel<T><<<dim3((nr + 127) / 128, nz), 128, 0, s>>>(theta, ra, za, rho, nr, nz, k.g0, k.theta0, adj_g);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(s));
    pla = std::move(p);
    adj_setup_ms = (TraceTimer::now() - t0) * 1e3;
    return 0;
  }
  // L^T lambda = g from lambda = 0, with the tolerance rule of the chi solve; then mu = H^T lambda and eta_d = mu / W.
  int adjoint_solve(const xee_solve_params* prm_in, int* iters, double* r1, int* err) override {
    TraceTimer tt("map adjoint solve");
    const int nr = d.nr, nz = d.nz;
    if (!pla && adjoint_setup()) return 1;
    cudaStream_t s = pla->own_stream;
    adj_ready = false;
    XEE_CHECK(cudaMemsetAsync(adj_lam, 0, sizeof(T) * nn, s));
    xee_solve_params p = *prm_in;
    if (d.r1_rel_rms_f > 0) {
      rms_interior_kernel<T><<<1, 256, 0, s>>>(adj_g, nr, nz, (T)d.r1_rel_rms_f, adj_r1); XEE_LAUNCH_OK();
      p.r1 = 1.0; p.r1_per_solve = adj_r1;
    }
    int it = 0, e = 0; double a1 = 0, a2 = 0;
    if (pla->solve(adj_lam, adj_g, &p, &it, &a1, &a2, &e, s, false, nullptr, 0)) return 1;
    heating_adjoint_kernel<T><<<dim3((nr - 1 + 127) / 128, nz - 1), 128, 0, s>>>(adj_lam, ra, za, ex, rho, nr, nz, k.g0, k.theta0,
                                                                                k.Cp, adj_mu, adj_eta);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(s));
    adj_ready = true;
    if (iters) *iters = it;
    if (r1) *r1 = a1;
    if (err) *err = e;
    return 0;
  }
  // rows [n][XEE_ADJ_COLS]: sum_Q, ke_gen = sum mu Q (g0/theta0 is in mu), efficiency.  XEE_ADJ_FULL_SUM=1 sums over every
  // cell instead of the cells a heating blob can reach (the same bits; the switch exists to show that).
  int adjoint_eval(const double* heat_host, int n, double* table) override {
    if (!adj_ready) return fail("xee_map_adjoint_eval: no adjoint field: call xee_map_adjoint_solve first");
    if (n < 1) return fail("xee_map_adjoint_eval: n >= 1 heating rows required");
    cudaStream_t s = pla->own_stream;
    Heat* hd = nullptr; double* sums = nullptr;
    PoolBuf hd_buf, sums_buf;
    XEE_CHECK(hd_buf.alloc(&hd, sizeof(Heat) * (size_t)n)); XEE_CHECK(sums_buf.alloc(&sums, sizeof(double) * 2 * (size_t)n));
    XEE_CHECK(cudaMemcpyAsync(hd, heat_host, sizeof(Heat) * (size_t)n, cudaMemcpyHostToDevice, s));
    adjoint_eval_kernel<T><<<n, 256, 0, s>>>(hd, adj_mu, ra, za, rho, d.nr, d.nz, env_int("XEE_ADJ_FULL_SUM", 0) ? 0 : 1, sums);
    XEE_LAUNCH_OK();
    std::vector<double> h(2 * (size_t)n);
    XEE_CHECK(cudaMemcpyAsync(h.data(), sums, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    for (size_t q = 0; q < (size_t)n; ++q) {
      double* r = table + q * XEE_ADJ_COLS;
      r[0] = h[2 * q]; r[1] = h[2 * q + 1]; r[2] = r[1] / r[0];
    }
    return 0;
  }
  int adjoint_timings(double* setup_ms, double* probe_ms, double* sweep_ms) override {
    if (!pla) return fail("xee_map_adjoint_timings: no adjoint solve yet");
    if (setup_ms) *setup_ms = adj_setup_ms;
    if (probe_ms) *probe_ms = pla->probe_ms;
    if (sweep_ms) *sweep_ms = pla->sweep_ms;
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
int xee_map_adjoint_solve(xee_map* m, const xee_solve_params* prm, int* iters, double* r1_out, int* err) {
  DeviceGuard g(m->impl->device());
  return m->impl->adjoint_solve(prm, iters, r1_out, err);
}
int xee_map_adjoint_eval_host(xee_map* m, const double* heat_host, int n, double* table_host) {
  DeviceGuard g(m->impl->device());
  return m->impl->adjoint_eval(heat_host, n, table_host);
}
int xee_map_adjoint_timings(xee_map* m, double* setup_ms, double* probe_ms, double* sweep_ms) {
  return m->impl->adjoint_timings(setup_ms, probe_ms, sweep_ms);
}
int xee_map_sweep_kernel_stats(xee_map* m, double* ms, long long* launches, int reset) { return m->impl->plan()->kernel_stats(ms, launches, reset); }
int xee_map_kernel_info(xee_map* m, int* variant, int* sweeps_per_pass, long long* kernel_launches) {
  return m->impl->plan()->kernel_info(variant, sweeps_per_pass, kernel_launches);
}
}  // extern "C"

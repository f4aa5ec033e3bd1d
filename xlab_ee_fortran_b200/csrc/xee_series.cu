// xee_series.cu — time-series diagnosis (BASELINE config 5): many vortex snapshots, ONE OPERATOR PER SOLVE,
// thermal + dynamical source term, Ekman-pumping bottom boundary condition, all built on the device.
//
//   vortex builder      xtt-lib-python/XWindProfile.py:10-23 (piecewise-constant absolute vorticity) x exp(-z/H);
//                       A = N^2, C = r^-3 d(M^2)/dr, B = -r^-3 d(M^2)/dz (thermal wind), values rounded through
//                       float32 exactly as the reference's .bin input files would hold them
//   pumping BC          xtt-lib-python/XPumping.py:40-41, 79-90: r*psi(r, z_bottom)
//   K1/K2 per snapshot  src/diagnose/initialize-variables.f90:72-95, xtt-lib-fortran/elliptic_tools.f90:35-56
//   heating RHS         src/old-diagnose/diagnose.f90:383-387, 396-406
//   dynamical RHS       src/old-diagnose/diagnose.f90:350-354 (rhoC_C), 359-367 (m^2, intended maths), 412-436
//   solve               elliptic_tools.f90:93-265, Chebyshev weights per solve (one spectral radius per operator)
//   u, w, integrals     old-diagnose/diagnose.f90:915-941, 1117-1127, 1029-1113
// The builders above are one producer of the fields A, B, C, Q, F and the rim of psi; run_fields takes the same fields from
// the caller (old-diagnose/diagnose.f90:211-212, 241-242 read them from files).  Both end in the same tail.
// Deviations from the legacy driver's latent bugs are listed in DESIGN.md section 3.
#include "xee_map_kernels.cuh"

namespace xee {

constexpr int kSeriesCols = 21;   // workloads.SERIES_COLS
struct Snap {
  double f0, f_core, f_env, radius, konst1, H, N2, pr0, pr1, pr2, c00, c01, c10, c11, hrc, hzc, hsr, hsz, hq0, fk, fh;
};
static_assert(sizeof(Snap) == kSeriesCols * sizeof(double), "Snap layout");

__device__ __forceinline__ void wind_region(const Snap& s, double r, double& fk, double& kk) {
  if (r < s.radius) { fk = s.f_core; kk = 0.0; } else { fk = s.f_env; kk = s.konst1; }
}
// WindProfile.getWind (XWindProfile.py:16-23): v = sqrt(f_k^2 r^4/4 + K_k)/r - f0 r/2, 0 at r = 0
__device__ __forceinline__ double wind_v(const Snap& s, double r) {
  if (r == 0.0) return 0.0;
  double fk, kk; wind_region(s, r, fk, kk);
  return sqrt(fk * fk * r * r * r * r / 4.0 + kk) / r - 0.5 * s.f0 * r;
}

// A, B, C of snapshot blockIdx.z on the O grid, rounded through float32 (the reference's file format).
template <class T>
__global__ void series_vortex_kernel(const Snap* __restrict__ snaps, T* __restrict__ A, T* __restrict__ B,
                                     T* __restrict__ C, int nr, int nz, double Lr0, double Lr1, double Lz0, double Lz1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr) return;
  const Snap s = snaps[blockIdx.z];
  const double r = Lr0 + i * ((Lr1 - Lr0) / (nr - 1)), z = Lz0 + j * ((Lz1 - Lz0) / (nz - 1));   // numpy.linspace
  double fk, kk; wind_region(s, r, fk, kk);
  const double m2b = fk * fk * (r * r * r * r) / 4.0 + kk, mb = sqrt(m2b);
  const double m = mb - 0.5 * s.f0 * r * r;
  const double dm = (mb > 0.0 ? 0.5 * fk * fk * (r * r * r) / mb : 0.0) - s.f0 * r;
  const double D = exp(-z / s.H), dD = -D / s.H;
  const double M = m * D + 0.5 * s.f0 * r * r, dM_dr = dm * D + s.f0 * r, dM_dz = m * dD;
  const double F = s.f0 + (fk - s.f0) * D;
  double c = r > 0.0 ? 2.0 * M * dM_dr / (r * r * r) : F * F;
  double b = r > 0.0 ? -2.0 * M * dM_dz / (r * r * r) : 0.0;
  c = fmax(c, s.f0 * s.f0);
  const double a = s.N2, lim = sqrt(0.95 * a * c);
  b = fmin(fmax(b, -lim), lim);
  const size_t o = (size_t)blockIdx.z * nr * nz + (size_t)j * nr + i;
  A[o] = (T)(float)a; B[o] = (T)(float)b; C[o] = (T)(float)c;
}

// psi = 0 everywhere except the bottom row: r*psi(r, z_bottom) = Pumping.getRPsi(r).
template <class T>
__global__ void series_bc_kernel(const Snap* __restrict__ snaps, T* __restrict__ psi, const T* __restrict__ ra, int nr, int nz) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr) return;
  T v = T(0);
  if (j == 0) {
    const Snap s = snaps[blockIdx.z];
    const double r = (double)ra[i];
    auto ip = [](double x, double lo, double hi) { return (x * x * x * x) / 4.0 - (lo + hi) / 3.0 * (x * x * x) + lo * hi * (x * x) / 2.0; };
    double p = 0.0;
    if (r <= s.pr0) p = 0.0;
    else if (r <= s.pr1) p = s.c00 * ip(r, s.pr0, s.pr1) + s.c01;
    else if (r <= s.pr2) p = s.c10 * ip(r, s.pr1, s.pr2) + s.c11;
    v = (T)p;
  }
  psi[(size_t)blockIdx.z * nr * nz + (size_t)j * nr + i] = v;
}

// m2 on B by cumulative trapezoid in r of rcuva^3 * rhoC_C (old-diagnose/diagnose.f90:359-367, intended maths),
// rhoC_C(i,j) = (C(i,j)+C(i,j+1))/2 (:350-354).  One thread per (row, snapshot), sequential in i as the reference.
template <class T>
__global__ void series_m2_kernel(const T* __restrict__ C, T* __restrict__ m2, const T* __restrict__ ra,
                                 const T* __restrict__ rc, int nr, int nz, int nsnap) {
  using R = Rn<T>;
  const int j = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
  if (j >= nz - 1) return;
  const T* Cn = C + (size_t)n * nr * nz;
  T* out = m2 + (size_t)n * (nr - 1) * (nz - 1) + (size_t)j * (nr - 1);
  auto rhoC_C = [&](int i) { return R::div(R::add(Cn[(size_t)j * nr + i], Cn[(size_t)(j + 1) * nr + i]), T(2)); };
  const T q = R::div(R::sub(rc[1], rc[0]), T(4));
  T acc = R::div(R::mul(R::mul((T)pow((double)q, 3.0), rhoC_C(0)), R::sub(ra[1], ra[0])), T(2));
  out[0] = acc;
  for (int i = 1; i < nr - 1; ++i) {   // Fortran i = 2..nr-1
    const T t = R::div(R::mul(R::mul((T)pow((double)rc[i], 3.0), rhoC_C(i)), R::sub(ra[i + 1], ra[i - 1])), T(2));
    acc = R::add(acc, t);
    out[i] = acc;
  }
}

// The parametric sources on the B cells of snapshot blockIdx.z: the heating Q = heat_q of the snapshot's blob at the cell
// centre (as heating_rhs_kernel and map_integrals_kernel evaluate it for a map) and the momentum forcing
// F(i,j) = -k v(r_{i+1/2}) exp(-z_{j+1/2}/h), evaluated in double and rounded to T.
template <class T>
__global__ void series_sources_kernel(const Snap* __restrict__ snaps, const Heat* __restrict__ heat, T* __restrict__ Q,
                                      T* __restrict__ F, const T* __restrict__ ra, const T* __restrict__ za, int nr, int nz) {
  const int ib = blockIdx.x * blockDim.x + threadIdx.x, jb = blockIdx.y, n = blockIdx.z;   // 0-based B cell
  if (ib >= nr - 1) return;
  const Snap s = snaps[n];
  const size_t o = (size_t)n * (nr - 1) * (nz - 1) + (size_t)jb * (nr - 1) + ib;
  Q[o] = BlobQ<T>{heat}.at(n)(ib, jb, ra, za);
  const double rm = 0.5 * ((double)ra[ib] + (double)ra[ib + 1]), zm = 0.5 * ((double)za[jb] + (double)za[jb + 1]);
  F[o] = (T)(-s.fk * wind_v(s, rm) * exp(-zm / s.fh));
}

// f += RHS_mom(i,j) = -(wA(i,j)+wA(i-1,j))/rcuva(i)^2, wA = d_dz_B2A(sqrt(m2)*F) on rows 2..nz-2 (0 elsewhere), F on B.
//                                                                        old-diagnose/diagnose.f90:412-436
template <class T>
__global__ void series_mom_rhs_kernel(const T* __restrict__ F, const T* __restrict__ m2, T* __restrict__ f,
                                      const T* __restrict__ rc, const T* __restrict__ za, int nr, int nz) {
  using R = Rn<T>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y, n = blockIdx.z;   // 0-based O point
  if (i < 1 || i >= nr - 1 || j < 1 || j >= nz - 1) return;
  const size_t nB = (size_t)(nr - 1) * (nz - 1);
  const T* m = m2 + (size_t)n * nB;
  const T* Fn = F + (size_t)n * nB;
  auto wB = [&](int ib, int jb) { const size_t o = (size_t)jb * (nr - 1) + ib; return R::mul(R::sqrt(m[o]), Fn[o]); };
  auto wA = [&](int ia) {           // A point (ia, j), Fortran J = j+1 in 2..nz-2  <=>  1 <= j <= nz-3
    if (j < 1 || j > nz - 3) return T(0);
    return R::div(R::sub(wB(ia, j), wB(ia, j - 1)), R::div(R::sub(za[j + 1], za[j - 1]), T(2)));
  };
  const T mom = -R::div(R::add(wA(i), wA(i - 1)), R::mul(rc[i], rc[i]));
  const size_t o = (size_t)n * nr * nz + (size_t)j * nr + i;
  f[o] = R::add(f[o], mom);
}

// Dirichlet data of a caller's psi_bc: keep the rim, zero the interior (the first guess).
template <class T>
__global__ void zero_interior_kernel(T* __restrict__ psi, int nr, int nz) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i < 1 || i >= nr - 1 || j < 1 || j >= nz - 1) return;
  psi[(size_t)blockIdx.z * nr * nz + (size_t)j * nr + i] = T(0);
}

template <class T>
__global__ void __launch_bounds__(256) absmax_kernel(const T* __restrict__ x, long long count, double* __restrict__ out) {
  __shared__ double red[32];
  const T* p = x + (size_t)blockIdx.x * count;
  double m = 0;
  for (long long q = threadIdx.x; q < count; q += 256) { const double v = fabs((double)p[q]); if (v == v && v <= 1e300) m = fmax(m, v); }
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) { for (int w = 1; w < 8; ++w) m = fmax(m, red[w]); out[blockIdx.x] = m; }
}

struct SeriesBase {
  xee_series_desc d{};
  int device() const { return d.device; }
  virtual ~SeriesBase() {}
  virtual int run(const double* params_host, const xee_solve_params* prm, double* table_host) = 0;
  virtual int run_fields(const void* A, const void* B, const void* C, const void* Q, const void* F, const void* psi_bc,
                         bool on_host, const xee_solve_params* prm, double* table_host, cudaStream_t stream) = 0;
  virtual int get_field(int which, void* host_out) = 0;
  virtual PlanBase* plan() = 0;
};

// A run is a producer that fills A, B, C, Q, F and the rim of psi, followed by one shared tail from those fields to the table.
// The parametric producer builds them from XEE_SERIES_PARAMS per snapshot; the field producer copies a caller's arrays.
template <class T>
struct Series : SeriesBase, PoolOwner {
  std::unique_ptr<Plan<T>> pl;
  T *A = nullptr, *B = nullptr, *C = nullptr, *Q = nullptr, *F = nullptr, *a = nullptr, *b = nullptr, *c = nullptr, *m2 = nullptr,
    *theta = nullptr, *psi = nullptr, *f = nullptr, *u = nullptr, *w = nullptr, *r1v = nullptr, *ra = nullptr, *za = nullptr,
    *ex = nullptr, *rho = nullptr;
  Snap* snaps = nullptr; Heat* heat = nullptr; double* integ = nullptr; double* mx = nullptr;
  bool has_F = false;   // F holds the last run's momentum forcing (a field run without F has none)
  size_t nn = 0;
  T dr = 0, dz = 0;
  PhysK<T> k;
  PlanBase* plan() override { return pl.get(); }

  int init() {
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    nn = (size_t)nr * nz;
    dr = (T(d.Lr[1]) - T(d.Lr[0])) / T(nr - 1); dz = (T(d.Lz[1]) - T(d.Lz[0])) / T(nz - 1);
    std::vector<T> h_ra(nr), h_za(nz), h_ex(nz), h_rho(nz);
    for (int i = 1; i <= nr; ++i) h_ra[i - 1] = T(d.Lr[0]) + T(i - 1) * dr;
    for (int j = 1; j <= nz; ++j) {   // initialize-variables.f90:52-57
      h_za[j - 1] = T(d.Lz[0]) + T(j - 1) * dz;
      h_ex[j - 1] = d.density_mode == 0 ? (T(1.0) - h_za[j - 1] / k.h0) : T(1.0);
      h_rho[j - 1] = d.density_mode == 0 ? k.p0 / (k.theta0 * k.Rd) * std::pow(h_ex[j - 1], T(1.0) / k.kappa - T(1.0)) : T(1.0);
    }
    xee_plan_desc pd{};
    pd.dtype = d.dtype; pd.nx = nr; pd.ny = nz; pd.nbatch = nb; pd.shared_coe = 0; pd.arith = d.arith; pd.method = d.method; pd.device = d.device;
    pl.reset(new Plan<T>()); pl->d = pd;
    if (pl->init()) return 1;
    const size_t nB = (size_t)(nr - 1) * (nz - 1);
    XEE_CHECK(own(&A, sizeof(T) * nn * nb)); XEE_CHECK(own(&B, sizeof(T) * nn * nb)); XEE_CHECK(own(&C, sizeof(T) * nn * nb));
    XEE_CHECK(own(&Q, sizeof(T) * nB * nb)); XEE_CHECK(own(&F, sizeof(T) * nB * nb));
    XEE_CHECK(own(&a, sizeof(T) * (nr - 1) * (nz - 2) * nb)); XEE_CHECK(own(&b, sizeof(T) * nB * nb));
    XEE_CHECK(own(&c, sizeof(T) * (nr - 2) * (nz - 1) * nb));
    XEE_CHECK(own(&m2, sizeof(T) * nB * nb)); XEE_CHECK(own(&theta, sizeof(T) * nB * nb));
    XEE_CHECK(own(&psi, sizeof(T) * nn * nb)); XEE_CHECK(own(&f, sizeof(T) * nn * nb));
    XEE_CHECK(own(&u, sizeof(T) * (size_t)nr * (nz - 1) * nb)); XEE_CHECK(own(&w, sizeof(T) * (size_t)(nr - 1) * nz * nb));
    XEE_CHECK(own(&r1v, sizeof(T) * nb));
    XEE_CHECK(own(&ra, sizeof(T) * nr)); XEE_CHECK(own(&za, sizeof(T) * nz));
    XEE_CHECK(own(&ex, sizeof(T) * nz)); XEE_CHECK(own(&rho, sizeof(T) * nz));
    XEE_CHECK(own(&snaps, sizeof(Snap) * nb)); XEE_CHECK(own(&heat, sizeof(Heat) * nb));
    XEE_CHECK(own(&integ, sizeof(double) * 3 * nb)); XEE_CHECK(own(&mx, sizeof(double) * 2 * nb));
    cudaStream_t s = pl->own_stream;
    XEE_CHECK(cudaMemcpyAsync(ra, h_ra.data(), sizeof(T) * nr, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(za, h_za.data(), sizeof(T) * nz, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(ex, h_ex.data(), sizeof(T) * nz, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(rho, h_rho.data(), sizeof(T) * nz, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    return 0;
  }
  ~Series() override {
    cudaDeviceSynchronize();   // the device is done with the owned blocks before they go back to the pool (see ~Plan)
  }

  // Parametric producer: the vortex, the blob heating, the friction and the pumping rim of every snapshot.
  int run(const double* params, const xee_solve_params* prm, double* table) override {
    TraceTimer tt("series run (total)");
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    XEE_CHECK(cudaMemcpyAsync(snaps, params, sizeof(Snap) * nb, cudaMemcpyHostToDevice, s));
    std::vector<Heat> hh(nb);
    for (int n = 0; n < nb; ++n) { const double* p = params + (size_t)n * kSeriesCols; hh[n] = Heat{p[14], p[15], p[16], p[17], p[18]}; }
    XEE_CHECK(cudaMemcpyAsync(heat, hh.data(), sizeof(Heat) * nb, cudaMemcpyHostToDevice, s));
    dim3 gO((nr + 127) / 128, nz, nb), gB((nr - 1 + 127) / 128, nz - 1, nb);
    series_vortex_kernel<T><<<gO, 128, 0, s>>>(snaps, A, B, C, nr, nz, d.Lr[0], d.Lr[1], d.Lz[0], d.Lz[1]); XEE_LAUNCH_OK();
    series_sources_kernel<T><<<gB, 128, 0, s>>>(snaps, heat, Q, F, ra, za, nr, nz); XEE_LAUNCH_OK();
    series_bc_kernel<T><<<gO, 128, 0, s>>>(snaps, psi, ra, nr, nz); XEE_LAUNCH_OK();
    has_F = true;
    // Spectral probes of the accelerated methods: when the snapshots form a smooth series (every vortex parameter changes by
    // less than 5 % from one snapshot to the next) only every 8th operator is probed and the rest interpolated.
    double worst = 0.0;
    for (int n = 1; n < nb; ++n)
      for (int q = 0; q < 14; ++q) {
        const double a0 = params[(size_t)(n - 1) * kSeriesCols + q], a1 = params[(size_t)n * kSeriesCols + q];
        const double sc = std::max(std::fabs(a0), std::fabs(a1));
        if (sc > 0) worst = std::max(worst, std::fabs(a1 - a0) / sc);
      }
    return tail((nb >= 32 && worst < 0.05) ? env_int("XEE_RHO_SUBSAMPLE", 8) : 0, prm, table);
  }

  // Field producer: the caller's arrays of T (host, or device read on `in` after the work queued there).  F == nullptr: no
  // momentum term; psi_bc == nullptr: a zero rim.  Only the rim of psi_bc is read; the first guess is 0 inside.
  int run_fields(const void* A_in, const void* B_in, const void* C_in, const void* Q_in, const void* F_in, const void* bc_in,
                 bool on_host, const xee_solve_params* prm, double* table, cudaStream_t in) override {
    if (!A_in || !B_in || !C_in || !Q_in) return fail("xee_series_run_fields: A, B, C and Q must not be NULL");
    TraceTimer tt("series run_fields (total)");
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    if (on_host) in = s;
    else {   // device arrays must live on the series' device: a copy from another device would depend on peer access
      for (const void* p : {A_in, B_in, C_in, Q_in, F_in, bc_in}) {
        if (!p) continue;
        cudaPointerAttributes pa{};
        if (cudaPointerGetAttributes(&pa, p) != cudaSuccess || (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) ||
            pa.device != d.device) {
          cudaGetLastError();
          return fail("xee_series_run_fields_dev: every array must be device memory on the series' device");
        }
      }
    }
    // a run that failed part-way may have left work on the own stream that still reads these buffers
    XEE_CHECK(cudaStreamSynchronize(s));
    const cudaMemcpyKind kind = on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const size_t bO = sizeof(T) * nn * nb, bB = sizeof(T) * (size_t)(nr - 1) * (nz - 1) * nb;
    XEE_CHECK(cudaMemcpyAsync(A, A_in, bO, kind, in)); XEE_CHECK(cudaMemcpyAsync(B, B_in, bO, kind, in));
    XEE_CHECK(cudaMemcpyAsync(C, C_in, bO, kind, in)); XEE_CHECK(cudaMemcpyAsync(Q, Q_in, bB, kind, in));
    has_F = F_in != nullptr;
    if (has_F) XEE_CHECK(cudaMemcpyAsync(F, F_in, bB, kind, in));
    if (bc_in) XEE_CHECK(cudaMemcpyAsync(psi, bc_in, bO, kind, in));
    else XEE_CHECK(cudaMemsetAsync(psi, 0, bO, in));
    XEE_CHECK(cudaStreamSynchronize(in));   // the caller's arrays are consumed; the rest runs on the series' own stream
    if (bc_in) { zero_interior_kernel<T><<<dim3((nr + 127) / 128, nz, nb), 128, 0, s>>>(psi, nr, nz); XEE_LAUNCH_OK(); }
    // Probe every operator: no smoothness rule for arbitrary fields has been calibrated.
    return tail(0, prm, table);
  }

  // Shared tail: operators, theta, right-hand sides, the batched solve and the table from the fields of the producer.
  // table row: iters, r1, err, sum_Q, ke_gen, efficiency, max|w|, max|u|
  int tail(int rho_subsample, const xee_solve_params* prm_in, double* table) {
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    dim3 gO((nr + 127) / 128, nz, nb);
    dim3 blk(64, 4), g2((nr + 63) / 64, (nz + 3) / 4, nb);
    build_abc_kernel<T><<<g2, blk, 0, s>>>(A, B, C, ra, rho, a, b, c, nr, nz); XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(s));
    if (pl->set_abc(a, b, c, (double)dr, (double)dz)) return 1;
    const FieldQ<T> qsrc{Q, nr, nz};
    background_theta_kernel<T><<<nb, 256, 0, s>>>(A, B, theta, ra, za, nr, nz, k.g0, k.theta0); XEE_LAUNCH_OK();
    heating_rhs_kernel<T><<<heating_rhs_grid(nr, nz, nb), dim3(kHeatBX, kHeatBY), 0, s>>>(qsrc, f, ra, za, ex, nr, nz, k.g0, k.theta0, k.Cp); XEE_LAUNCH_OK();
    dim3 gm((nz - 1 + 63) / 64, nb);
    series_m2_kernel<T><<<gm, 64, 0, s>>>(C, m2, ra, ra, nr, nz, nb); XEE_LAUNCH_OK();
    if (has_F) { series_mom_rhs_kernel<T><<<gO, 128, 0, s>>>(F, m2, f, ra, za, nr, nz); XEE_LAUNCH_OK(); }
    pl->rho_subsample = rho_subsample;
    xee_solve_params prm = *prm_in;
    if (d.r1_rel_rms_f > 0) {
      // tolerance relative to the INITIAL residual L psi0 - f: with the pumping boundary condition the boundary data,
      // not f, set the scale of the problem (the plan's second ping-pong buffer is free scratch before the solve)
      if (pl->apply(psi, pl->x1, s)) return 1;
      rms_diff_interior_kernel<T><<<nb, 256, 0, s>>>(pl->x1, f, nr, nz, (T)d.r1_rel_rms_f, r1v); XEE_LAUNCH_OK();
      prm.r1 = 1.0; prm.r1_per_solve = r1v;
    }
    std::vector<int> iters(nb), err(nb);
    std::vector<double> r1o(nb), r2o(nb);
    if (pl->solve(psi, f, &prm, iters.data(), r1o.data(), r2o.data(), err.data(), s, false, nullptr, 0)) return 1;
    uw_kernel<T><<<gO, 128, 0, s>>>(psi, u, w, ra, ra, za, rho, nr, nz); XEE_LAUNCH_OK();
    map_integrals_kernel<T><<<nb, 256, 0, s>>>(qsrc, psi, theta, nullptr, ra, ra, za, rho, nr, nz, integ, (long long)(nr - 1) * (nz - 1));
    XEE_LAUNCH_OK();
    absmax_kernel<T><<<nb, 256, 0, s>>>(w, (long long)(nr - 1) * nz, mx); XEE_LAUNCH_OK();
    absmax_kernel<T><<<nb, 256, 0, s>>>(u, (long long)nr * (nz - 1), mx + nb); XEE_LAUNCH_OK();
    std::vector<double> hi(3 * (size_t)nb), hm(2 * (size_t)nb);
    XEE_CHECK(cudaMemcpyAsync(hi.data(), integ, sizeof(double) * 3 * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaMemcpyAsync(hm.data(), mx, sizeof(double) * 2 * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    const double gth = (double)k.g0 / (double)k.theta0;
    for (int n = 0; n < nb; ++n) {
      double* r = table + (size_t)n * XEE_MAP_COLS;
      r[0] = iters[n]; r[1] = r1o[n]; r[2] = err[n]; r[3] = hi[3 * n]; r[4] = hi[3 * n + 1] * gth; r[5] = r[4] / r[3];
      r[6] = hm[n]; r[7] = hm[nb + n];
    }
    return 0;
  }
  int get_field(int which, void* out) override {
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    const size_t nB = (size_t)(nr - 1) * (nz - 1);
    const void* src = nullptr; size_t bytes = 0;
    switch (which) {
      case 0: src = psi; bytes = sizeof(T) * nn * nb; break;
      case 1: src = f; bytes = sizeof(T) * nn * nb; break;
      case 2: src = theta; bytes = sizeof(T) * nB * nb; break;
      case 3: src = u; bytes = sizeof(T) * (size_t)nr * (nz - 1) * nb; break;
      case 4: src = w; bytes = sizeof(T) * (size_t)(nr - 1) * nz * nb; break;
      case 5: src = A; bytes = sizeof(T) * nn * nb; break;
      case 6: src = B; bytes = sizeof(T) * nn * nb; break;
      case 7: src = C; bytes = sizeof(T) * nn * nb; break;
      case 8: src = m2; bytes = sizeof(T) * nB * nb; break;
      case 9: src = Q; bytes = sizeof(T) * nB * nb; break;
      case 10:
        if (!has_F) return fail("xee_series_get_field: the last run had no momentum forcing F");
        src = F; bytes = sizeof(T) * nB * nb; break;
      default: return fail("xee_series_get_field: unknown field");
    }
    XEE_CHECK(cudaMemcpy(out, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
  }
};

}  // namespace xee

using namespace xee;
struct xee_series { SeriesBase* impl; };

extern "C" {
int xee_series_create(const xee_series_desc* desc, xee_series** out) {
  int dev = 0;
  if (resolve_device(desc->device, &dev)) return 1;
  DeviceGuard guard(dev);
  if (desc->nr < 4 || desc->nz < 5 || desc->nsnap < 1) return fail("xee_series: nr >= 4, nz >= 5 and nsnap >= 1 required");
  std::unique_ptr<SeriesBase> m; int rc;
  if (desc->dtype == XEE_F32) { auto* q = new Series<float>(); m.reset(q); q->d = *desc; q->d.device = dev; rc = q->init(); }
  else if (desc->dtype == XEE_F64) { auto* q = new Series<double>(); m.reset(q); q->d = *desc; q->d.device = dev; rc = q->init(); }
  else return fail("xee_series: dtype must be XEE_F32 or XEE_F64");
  if (rc) return 1;
  *out = new xee_series{m.release()};
  return 0;
}
int xee_series_destroy(xee_series* m) { if (m) { DeviceGuard g(m->impl->device()); delete m->impl; delete m; } return 0; }
int xee_series_run_host(xee_series* m, const double* params, const xee_solve_params* prm, double* table) { DeviceGuard g(m->impl->device()); return m->impl->run(params, prm, table); }
int xee_series_run_fields_host(xee_series* m, const void* A, const void* B, const void* C, const void* Q, const void* F,
                               const void* psi_bc, const xee_solve_params* prm, double* table) {
  DeviceGuard g(m->impl->device());
  return m->impl->run_fields(A, B, C, Q, F, psi_bc, true, prm, table, nullptr);
}
int xee_series_run_fields_dev(xee_series* m, const void* A, const void* B, const void* C, const void* Q, const void* F,
                              const void* psi_bc, const xee_solve_params* prm, double* table, void* stream) {
  DeviceGuard g(m->impl->device());
  return m->impl->run_fields(A, B, C, Q, F, psi_bc, false, prm, table, (cudaStream_t)stream);
}
int xee_series_get_field(xee_series* m, int which, void* out) { DeviceGuard g(m->impl->device()); return m->impl->get_field(which, out); }
int xee_series_sweep_kernel_stats(xee_series* m, double* ms, long long* launches, int reset) { return m->impl->plan()->kernel_stats(ms, launches, reset); }
int xee_series_probe_stats(xee_series* m, double* ms, int reset) {
  PlanBase* p = m->impl->plan();
  if (ms) *ms = p->probe_ms;
  if (reset) p->probe_ms = 0;
  return 0;
}
int xee_series_kernel_info(xee_series* m, int* variant, int* sweeps_per_pass, long long* kernel_launches) {
  return m->impl->plan()->kernel_info(variant, sweeps_per_pass, kernel_launches);
}
}  // extern "C"

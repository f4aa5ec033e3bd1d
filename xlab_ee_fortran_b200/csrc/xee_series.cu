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
// decompose is a second tail on the field producer's buffers: the legacy efficiency decomposition (old-diagnose/diagnose.f90:
// 447-841, xee_old_diagnose.cpp) of every snapshot, each of its up to nine solves batched over the snapshots.
// Deviations from the legacy driver's latent bugs are listed in DESIGN.md section 3.
#include <limits>

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

// ---- the legacy efficiency decomposition (old-diagnose/diagnose.f90:468-772), one block or one thread per cell per snapshot

// Stage II tendency on the B cells of snapshot blockIdx.x (:488-493) and its integral integrate_weight_B (:496):
//   dtheta_dt = J - theta0/g0 (rhoA_A w)avg_z + theta0/g0 (rhoB_C u)avg_r,  J = Q/(Cp exner),
// rhoA_A = (A(i,j)+A(i+1,j))/2 and rhoB_C = (B(i,j)+B(i,j+1))/2 of the basic state.  out[n] = the weighted sum in double,
// in the fixed order of map_integrals_kernel.
template <class T>
__global__ void __launch_bounds__(256) tendency_kernel(FieldQ<T> src, const T* __restrict__ A, const T* __restrict__ B,
                                                       const T* __restrict__ u, const T* __restrict__ w, T* __restrict__ dth,
                                                       const T* __restrict__ ra, const T* __restrict__ za,
                                                       const T* __restrict__ ex, const T* __restrict__ rho, int nr, int nz,
                                                       T g0, T theta0, T Cp, double* __restrict__ out) {
  using R = Rn<T>;
  __shared__ double red[32];
  const int n = blockIdx.x;
  const auto Qn = src.at(n);
  A += (size_t)n * nr * nz; B += (size_t)n * nr * nz;
  u += (size_t)n * nr * (nz - 1); w += (size_t)n * (nr - 1) * nz; dth += (size_t)n * (nr - 1) * (nz - 1);
  const T k = R::div(theta0, g0);
  const int ncell = (nr - 1) * (nz - 1);
  double s = 0;
  for (int q = threadIdx.x; q < ncell; q += 256) {
    const int i = q % (nr - 1), j = q / (nr - 1);
    const size_t o = (size_t)j * nr + i, oa = (size_t)j * (nr - 1) + i;
    const T J = R::div(Qn(i, j, ra, za), R::mul(Cp, ex[j]));
    const T rA0 = R::div(R::add(A[o], A[o + 1]), T(2)), rA1 = R::div(R::add(A[o + nr], A[o + nr + 1]), T(2));
    const T rC0 = R::div(R::add(B[o], B[o + nr]), T(2)), rC1 = R::div(R::add(B[o + 1], B[o + nr + 1]), T(2));
    const T tw = R::div(R::mul(k, R::add(R::mul(rA0, w[oa]), R::mul(rA1, w[oa + nr - 1]))), T(2));
    const T tu = R::div(R::mul(k, R::add(R::mul(rC0, u[o]), R::mul(rC1, u[o + 1]))), T(2));
    const T v = R::add(R::sub(J, tw), tu);
    dth[oa] = v;
    s += (double)weighted<T>(v, ra, ra, za, rho, i, j);
  }
  const double t = block_sum(s, red, threadIdx.x, 8);
  if (threadIdx.x == 0) out[n] = t;
}

// The anomaly of a tendency step of length dt on B cell (i, j) of snapshot blockIdx.z (:497-500, 513-514):
//   b_anom = -g0/theta0 d_dr_B2B(dtheta_dt dt)                 (one-sided in the first and last column, :975-990)
//   b_op   = b_basic + b_anom / rcuv / rho_                    the b of L(A, B0+dB, C) in set_abc's normalisation
template <class T>
__global__ void anomaly_kernel(const T* __restrict__ dth, const T* __restrict__ b_basic, T* __restrict__ b_anom,
                               T* __restrict__ b_op, const T* __restrict__ ra, const T* __restrict__ rho, int nr, int nz,
                               T dt, T g0, T theta0) {
  using R = Rn<T>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr - 1) return;
  const size_t o = (size_t)blockIdx.z * (nr - 1) * (nz - 1) + (size_t)j * (nr - 1) + i;
  const T* row = dth + (o - i);
  const int m = i == 0 ? 0 : -1, p = i == nr - 2 ? 0 : 1;
  const T d = R::div(R::sub(R::mul(row[i + m], dt), R::mul(row[i + p], dt)), R::sub(ra[i + m], ra[i + p]));
  const T ba = R::mul(R::div(-g0, theta0), d);
  const T sb = R::div(R::div(ba, R::div(R::add(ra[i], ra[i + 1]), T(2))), R::div(R::add(rho[j], rho[j + 1]), T(2)));
  b_anom[o] = ba;
  b_op[o] = R::add(b_basic[o], sb);
}

// The state after the tendency step, for relative_theta_kernel (:497-509): rhoB_B + b_anom, its rhoB_C, and
// rhoA_A + g0/theta0 d_dz_B2A(dtheta_dt dt) (0 on the rows d_dz_B2A does not write, [D3] of xee_old_diagnose.cpp).
template <class T>
struct TendencyState {
  const T* A; const T* B; const T* dth; const T* b_anom; const T* za; T dt, g0, theta0; int nr, nz;
  struct At {
    const T* A; const T* B; const T* dth; const T* b_anom; const T* za; T dt, g0, theta0; int nr, nz;
    __device__ __forceinline__ T rhoB_C(int i) const {
      using R = Rn<T>;
      return R::div(R::add(R::add(rhoB_B_of(B, nr, i - 1, 0), b_anom[i - 1]), R::add(rhoB_B_of(B, nr, i, 0), b_anom[i])), T(2));
    }
    __device__ __forceinline__ T rhoA_A(int i, int j) const {
      using R = Rn<T>;
      const T rA = R::div(R::add(A[(size_t)j * nr + i], A[(size_t)j * nr + i + 1]), T(2));
      T dA = T(0);
      if (j <= nz - 3) {
        const T t1 = R::mul(dth[(size_t)j * (nr - 1) + i], dt), t0 = R::mul(dth[(size_t)(j - 1) * (nr - 1) + i], dt);
        dA = R::div(R::sub(t1, t0), R::div(R::sub(za[j + 1], za[j - 1]), T(2)));
      }
      return R::add(rA, R::mul(R::div(g0, theta0), dA));
    }
  };
  __device__ __forceinline__ At at(int n) const {
    const size_t nO = (size_t)nr * nz, nB = (size_t)(nr - 1) * (nz - 1);
    return At{A + n * nO, B + n * nO, dth + n * nB, b_anom + n * nB, za, dt, g0, theta0, nr, nz};
  }
};

// One boundary term of cal_exchange_conversion (:1152-1166) at mid-point i+1/2: values at columns i, i+1 of the boundary row
// (b), and of the rows hi > lo of the one-sided z difference;  (C/rho) ((psi)avg dchi/dz - (chi)avg dpsi/dz) / r^2.
template <class T>
__device__ __forceinline__ T exchange_term(T C0, T C1, T rho_b, T p0, T p1, T ph0, T ph1, T pl0, T pl1, T c0, T c1, T ch0, T ch1,
                                           T cl0, T cl1, T dz2, T r) {
  using R = Rn<T>;
  const T dchi = R::div(R::sub(R::sub(R::add(ch0, ch1), cl0), cl1), dz2);
  const T dpsi = R::div(R::sub(R::sub(R::add(ph0, ph1), pl0), pl1), dz2);
  const T fac = R::div(R::add(C0, C1), R::mul(T(2), rho_b));
  const T x = R::sub(R::mul(R::div(R::add(p0, p1), T(2)), dchi), R::mul(R::div(R::add(c0, c1), T(2)), dpsi));
  return R::div(R::mul(fac, x), R::mul(r, r));
}

// cal_exchange_conversion (:730-772, :1143-1174, [D5]: real r, dr, dz) of snapshot blockIdx.x, both methods in one pass:
// chi = chi_bc + chi_dB + chi_B0 (method 1) and chi_dB + chi_B0 (method 2), summed in working precision as the legacy
// driver adds the fields;  out[n][m] = -sum_i (bnd_top - bnd_bottom) r dr, in double in a fixed order.
template <class T>
__global__ void __launch_bounds__(256) exchange_conversion_kernel(const T* __restrict__ psi, const T* __restrict__ chi_bc,
                                                                  const T* __restrict__ chi_dB, const T* __restrict__ chi_B0,
                                                                  const T* __restrict__ C, const T* __restrict__ ra,
                                                                  const T* __restrict__ za, const T* __restrict__ rho,
                                                                  int nr, int nz, double* __restrict__ out /*[n][2]*/) {
  using R = Rn<T>;
  __shared__ double red[32];
  const size_t off = (size_t)blockIdx.x * nr * nz;
  psi += off; chi_bc += off; chi_dB += off; chi_B0 += off; C += off;
  const T dz2 = R::mul(T(2), R::sub(za[1], za[0])), ddr = R::sub(ra[1], ra[0]);
  const size_t top = (size_t)(nz - 1) * nr, below = (size_t)(nz - 2) * nr;
  double s[2] = {0, 0};
  for (int i = threadIdx.x; i < nr - 1; i += 256) {
    const T r = R::div(R::add(ra[i], ra[i + 1]), T(2));
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      auto chi = [&](size_t o) { const T c = R::add(chi_dB[o], chi_B0[o]); return m == 0 ? R::add(R::add(chi_bc[o], chi_dB[o]), chi_B0[o]) : c; };
      const size_t b0 = i, b1 = (size_t)nr + i, t1 = top + i, t0 = below + i;
      const T bot = exchange_term(C[b0], C[b0 + 1], rho[0], psi[b0], psi[b0 + 1], psi[b1], psi[b1 + 1], psi[b0], psi[b0 + 1],
                                  chi(b0), chi(b0 + 1), chi(b1), chi(b1 + 1), chi(b0), chi(b0 + 1), dz2, r);
      const T tp = exchange_term(C[t1], C[t1 + 1], rho[nz - 1], psi[t1], psi[t1 + 1], psi[t1], psi[t1 + 1], psi[t0], psi[t0 + 1],
                                 chi(t1), chi(t1 + 1), chi(t1), chi(t1 + 1), chi(t0), chi(t0 + 1), dz2, r);
      s[m] -= (double)R::mul(R::mul(R::sub(tp, bot), r), ddr);
    }
  }
  const double a = block_sum(s[0], red, threadIdx.x, 8);
  const double b = block_sum(s[1], red, threadIdx.x, 8);
  if (threadIdx.x == 0) { out[2 * blockIdx.x] = a; out[2 * blockIdx.x + 1] = b; }
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
  virtual int decompose(const xee_decomp_desc* dd, const void* A, const void* B, const void* C, const void* Q, const void* F,
                        const void* psi_bc, const void* chi_bc, bool on_host, const xee_solve_params* prm_psi,
                        const xee_solve_params* prm_chi, double* table, int* iters, int* err, cudaStream_t stream) = 0;
  virtual int get_decomp_field(int which, void* host_out) = 0;
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
  // The decomposition's buffers, allocated by its first call: dfield[2 + slot] = the field of solve slot (XEE_DECOMP_SOLVES
  // order), dfield[0] = dtheta_dt, dfield[1] = theta_after; dmade[w]: the last decomposition made dfield[w].
  static constexpr int kDecompFields = 2 + XEE_DECOMP_SOLVES;
  T* dfield[kDecompFields] = {};
  bool dmade[kDecompFields] = {};
  T *eta = nullptr, *b_anom = nullptr, *b_op = nullptr, *zero = nullptr, *f_basic = nullptr, *f_anom = nullptr,
    *chi_rim = nullptr, *r0v = nullptr;
  double *dsum = nullptr /*[slot][n][3]*/, *sdt = nullptr /*[n]*/, *exch = nullptr /*[tag][n][2]*/;
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
    TraceTimer tt("series run_fields (total)");
    if (load_fields("xee_series_run_fields", A_in, B_in, C_in, Q_in, F_in, bc_in,
                    nullptr, nullptr, on_host, in))
      return 1;
    // Probe every operator: no smoothness rule for arbitrary fields has been calibrated.
    return tail(0, prm, table);
  }

  // Field producer: copies the caller's A, B, C, Q, F and the rim of psi_bc (and of chi_bc into chi_rim) into the series.
  // `who` names the entry point in messages (its _dev form for device arrays).
  int load_fields(const char* who, const void* A_in, const void* B_in, const void* C_in, const void* Q_in, const void* F_in,
                  const void* bc_in, const void* chi_in, T* chi_rim, bool on_host, cudaStream_t in) {
    if (!A_in || !B_in || !C_in || !Q_in) return fail((std::string(who) + ": A, B, C and Q must not be NULL").c_str());
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    if (on_host) in = s;
    else {   // device arrays must live on the series' device: a copy from another device would depend on peer access
      for (const void* p : {A_in, B_in, C_in, Q_in, F_in, bc_in, chi_in}) {
        if (!p) continue;
        cudaPointerAttributes pa{};
        if (cudaPointerGetAttributes(&pa, p) != cudaSuccess || (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) ||
            pa.device != d.device) {
          cudaGetLastError();
          return fail((std::string(who) + "_dev: every array must be device memory on the series' device").c_str());
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
    if (chi_in) XEE_CHECK(cudaMemcpyAsync(chi_rim, chi_in, bO, kind, in));
    XEE_CHECK(cudaStreamSynchronize(in));   // the caller's arrays are consumed; the rest runs on the series' own stream
    if (bc_in) { zero_interior_kernel<T><<<dim3((nr + 127) / 128, nz, nb), 128, 0, s>>>(psi, nr, nz); XEE_LAUNCH_OK(); }
    if (chi_in) { zero_interior_kernel<T><<<dim3((nr + 127) / 128, nz, nb), 128, 0, s>>>(chi_rim, nr, nz); XEE_LAUNCH_OK(); }
    return 0;
  }

  // Shared tail: operators, theta, right-hand sides, the batched solve and the table from the fields of the producer.
  int tail(int rho_subsample, const xee_solve_params* prm_in, double* table) {
    if (prepare(true)) return 1;
    pl->rho_subsample = rho_subsample;
    return solve_psi(prm_in, table);
  }
  // a, b, c, (with set_op) the operator L(A, B, C) of every snapshot, the background theta, the forcing f and m2
  int prepare(bool set_op) {
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    dim3 gO((nr + 127) / 128, nz, nb);
    dim3 blk(64, 4), g2((nr + 63) / 64, (nz + 3) / 4, nb);
    build_abc_kernel<T><<<g2, blk, 0, s>>>(A, B, C, ra, rho, a, b, c, nr, nz); XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(s));
    if (set_op && pl->set_abc(a, b, c, (double)dr, (double)dz)) return 1;
    const FieldQ<T> qsrc{Q, nr, nz};
    relative_theta_kernel<T><<<nb, 256, 0, s>>>(BasicState<T>{A, B, nr, nz}, theta, ra, za, nr, nz, k.g0, k.theta0); XEE_LAUNCH_OK();
    heating_rhs_kernel<T><<<heating_rhs_grid(nr, nz, nb), dim3(kHeatBX, kHeatBY), 0, s>>>(qsrc, f, ra, za, ex, nr, nz, k.g0, k.theta0, k.Cp); XEE_LAUNCH_OK();
    dim3 gm((nz - 1 + 63) / 64, nb);
    series_m2_kernel<T><<<gm, 64, 0, s>>>(C, m2, ra, ra, nr, nz, nb); XEE_LAUNCH_OK();
    if (has_F) { series_mom_rhs_kernel<T><<<gO, 128, 0, s>>>(F, m2, f, ra, za, nr, nz); XEE_LAUNCH_OK(); }
    return 0;
  }
  // The batched solve L psi = f on the current operator, u, w and the table.
  // table row: iters, r1, err, sum_Q, ke_gen, efficiency, max|w|, max|u|
  int solve_psi(const xee_solve_params* prm_in, double* table) {
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    dim3 gO((nr + 127) / 128, nz, nb);
    const FieldQ<T> qsrc{Q, nr, nz};
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
  // ---- The legacy efficiency decomposition (old-diagnose/diagnose.f90:447-841) on the field producer's snapshots.
  int decomp_alloc() {   // once per series, on the first decomposition
    if (zero) return 0;
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    const size_t bO = sizeof(T) * nn * nb, bB = sizeof(T) * (size_t)(nr - 1) * (nz - 1) * nb;
    XEE_CHECK(own(&dfield[0], bB)); XEE_CHECK(own(&dfield[1], bB));
    for (int w = 2; w < kDecompFields; ++w) XEE_CHECK(own(&dfield[w], bO));
    XEE_CHECK(own(&eta, sizeof(T) * (size_t)(nr - 1) * nz * nb));
    XEE_CHECK(own(&b_anom, bB)); XEE_CHECK(own(&b_op, bB));
    XEE_CHECK(own(&f_basic, bO)); XEE_CHECK(own(&f_anom, bO)); XEE_CHECK(own(&chi_rim, bO));
    XEE_CHECK(own(&r0v, sizeof(T) * nb));
    XEE_CHECK(own(&dsum, sizeof(double) * 3 * nb * XEE_DECOMP_SOLVES)); XEE_CHECK(own(&sdt, sizeof(double) * nb));
    XEE_CHECK(own(&exch, sizeof(double) * 4 * nb));
    T* z = nullptr;
    XEE_CHECK(own(&z, bO));
    XEE_CHECK(cudaMemsetAsync(z, 0, bO, pl->own_stream));
    zero = z;   // set last: a call that failed above allocates again
    return 0;
  }

  // The batched solve of decomposition slot `slot` on the current operator, from the first guess in x (the Dirichlet rim,
  // 0 inside); tolerance as in the tail, r1_rel_rms_f * rms of the initial residual.  A snapshot whose initial residual is
  // exactly 0 (a right-hand side and rim of zeros) keeps its first guess with iters 0 and err 0: its tolerance would be 0,
  // which disables the stop rule.  When no snapshot has a residual nothing is solved.
  int solve_slot(T* x, const T* rhs, const xee_solve_params* prm_in, int slot, std::vector<int>& its, std::vector<int>& errs) {
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    cudaStream_t s = pl->own_stream;
    if (pl->apply(x, pl->x1, s)) return 1;
    rms_diff_interior_kernel<T><<<nb, 256, 0, s>>>(pl->x1, rhs, nr, nz, T(1), r0v); XEE_LAUNCH_OK();
    std::vector<T> h0(nb);
    XEE_CHECK(cudaMemcpyAsync(h0.data(), r0v, sizeof(T) * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    std::vector<int> it(nb, 0), er(nb, 0);
    std::vector<double> r1o(nb), r2o(nb);
    bool any = false;
    for (int n = 0; n < nb; ++n) any |= !(h0[n] == T(0));
    if (any) {
      xee_solve_params prm = *prm_in;
      if (d.r1_rel_rms_f > 0) {
        rms_diff_interior_kernel<T><<<nb, 256, 0, s>>>(pl->x1, rhs, nr, nz, (T)d.r1_rel_rms_f, r1v); XEE_LAUNCH_OK();
        prm.r1 = 1.0; prm.r1_per_solve = r1v;
      }
      if (pl->solve(x, rhs, &prm, it.data(), r1o.data(), r2o.data(), er.data(), s, false, nullptr, 0)) return 1;
      for (int n = 0; n < nb; ++n)
        if (h0[n] == T(0)) {
          zero_interior_kernel<T><<<dim3((nr + 127) / 128, nz, 1), 128, 0, s>>>(x + (size_t)n * nn, nr, nz); XEE_LAUNCH_OK();
          it[n] = 0; er[n] = 0;
        }
    }
    for (int n = 0; n < nb; ++n) { its[(size_t)n * XEE_DECOMP_SOLVES + slot] = it[n]; errs[(size_t)n * XEE_DECOMP_SOLVES + slot] = er[n]; }
    return 0;
  }

  // Stage I (TENDENCY): the tail's solve L(B0) psi = f.  Stage II: the tendency, the anomaly, theta_after, f_anomaly.
  // Then per operator L(A, B=0, C) (tag 0) and L(A, B=B0+dB, C) (tag B0dB): the chi solves, eta and sum(Q eta), the
  // integral-check psi solve and its w theta integral, and with chi_bc the exchange conversion.  Every solve starts from a
  // zero interior; each operator is set (and probed) once.
  int decompose(const xee_decomp_desc* dd, const void* A_in, const void* B_in, const void* C_in, const void* Q_in,
                const void* F_in, const void* bc_in, const void* chi_in, bool on_host, const xee_solve_params* prm_psi,
                const xee_solve_params* prm_chi, double* table, int* iters_out, int* err_out, cudaStream_t in) override {
    if (!dd || !prm_psi || !prm_chi || !table) return fail("xee_series_decompose: desc, prm_psi, prm_chi and table must not be NULL");
    if (dd->baro < 0 || dd->baro > 2) return fail("xee_series_decompose: baro must be 0 (BAROTROPIC), 1 (BAROCLINIC) or 2 (BARO_ALL)");
    const bool tend = dd->tendency != 0;
    if (tend && !std::isfinite(dd->testing_dt)) return fail("xee_series_decompose: testing_dt must be finite in TENDENCY mode");
    TraceTimer tt("series decompose (total)");
    if (decomp_alloc()) return 1;
    for (bool& m : dmade) m = false;
    if (load_fields("xee_series_decompose", A_in, B_in, C_in, Q_in, F_in, bc_in, chi_in, chi_rim, on_host, in)) return 1;
    const int nr = d.nr, nz = d.nz, nb = d.nsnap;
    const size_t nB = (size_t)(nr - 1) * (nz - 1), bO = sizeof(T) * nn * nb, bB = sizeof(T) * nB * nb;
    cudaStream_t s = pl->own_stream;
    const bool bc = chi_in != nullptr, use[2] = {dd->baro != 1, dd->baro != 0};
    const T dt = (T)dd->testing_dt;
    std::vector<int> its((size_t)nb * XEE_DECOMP_SOLVES, -1), errs(its.size(), 0);
    if (prepare(tend)) return 1;
    pl->rho_subsample = 0;   // every operator probed, as in run_fields
    for (int t = 0; t < 2; ++t)   // first guesses of the integral checks: the rim of psi_bc, 0 inside
      if (use[t]) XEE_CHECK(cudaMemcpyAsync(dfield[9 + t], psi, bO, cudaMemcpyDeviceToDevice, s));
    const FieldQ<T> qsrc{Q, nr, nz};
    const dim3 gO((nr + 127) / 128, nz, nb), gB((nr - 1 + 127) / 128, nz - 1, nb);
    if (tend) {
      std::vector<double> t8((size_t)nb * XEE_MAP_COLS);
      {
        TraceTimer t1("  decompose: stage I solve");
        if (solve_psi(prm_psi, t8.data())) return 1;
      }
      TraceTimer t2("  decompose: stage II");
      for (int n = 0; n < nb; ++n) { its[(size_t)n * XEE_DECOMP_SOLVES] = (int)t8[(size_t)n * XEE_MAP_COLS]; errs[(size_t)n * XEE_DECOMP_SOLVES] = (int)t8[(size_t)n * XEE_MAP_COLS + 2]; }
      XEE_CHECK(cudaMemcpyAsync(dfield[2], psi, bO, cudaMemcpyDeviceToDevice, s));
      dmade[2] = true;
      tendency_kernel<T><<<nb, 256, 0, s>>>(qsrc, A, B, u, w, dfield[0], ra, za, ex, rho, nr, nz, k.g0, k.theta0, k.Cp, sdt); XEE_LAUNCH_OK();
      anomaly_kernel<T><<<gB, 128, 0, s>>>(dfield[0], b, b_anom, b_op, ra, rho, nr, nz, dt, k.g0, k.theta0); XEE_LAUNCH_OK();
      relative_theta_kernel<T><<<nb, 256, 0, s>>>(TendencyState<T>{A, B, dfield[0], b_anom, za, dt, k.g0, k.theta0, nr, nz}, dfield[1],
                                                  ra, za, nr, nz, k.g0, k.theta0); XEE_LAUNCH_OK();
      rhs_from_B_kernel<T><<<gO, 128, 0, s>>>(BGridB<T>{b_anom, nr, nz}, f_anom, nr, nz); XEE_LAUNCH_OK();
      dmade[0] = true;
    } else {   // INSTANT ([D4] of xee_old_diagnose.cpp): b_anom = 0, theta_after = the background state
      XEE_CHECK(cudaMemcpyAsync(dfield[1], theta, bB, cudaMemcpyDeviceToDevice, s));
      XEE_CHECK(cudaMemsetAsync(f_anom, 0, bO, s));
    }
    dmade[1] = true;
    rhs_from_B_kernel<T><<<gO, 128, 0, s>>>(OGridB<T>{B, nr, nz}, f_basic, nr, nz); XEE_LAUNCH_OK();
    const T* bop[2] = {zero, tend ? b_op : b};
    const T* chi_rhs[3] = {zero, f_anom, f_basic};
    const dim3 ge((nr - 1 + 127) / 128, nz, nb);
    for (int t = 0; t < 2; ++t) {
      if (!use[t]) continue;
      XEE_CHECK(cudaStreamSynchronize(s));
      {
        TraceTimer t3("  decompose: operator set");
        if (pl->set_abc(a, bop[t], c, (double)dr, (double)dz)) return 1;
      }
      {
        TraceTimer t4("  decompose: chi solves");
        for (int kind = bc ? 0 : 1; kind < 3; ++kind) {   // chi with the chi_bc rim and rhs 0, then -dB, then -B0
          const int slot = 1 + 2 * kind + t;
          T* x = dfield[2 + slot];
          if (kind == 0) XEE_CHECK(cudaMemcpyAsync(x, chi_rim, bO, cudaMemcpyDeviceToDevice, s));
          else XEE_CHECK(cudaMemsetAsync(x, 0, bO, s));
          if (solve_slot(x, chi_rhs[kind], prm_chi, slot, its, errs)) return 1;
          eta_kernel<T><<<ge, 128, 0, s>>>(x, eta, ra, ra, rho, ex, nr, nz, k.g0, k.Cp, k.theta0); XEE_LAUNCH_OK();
          map_integrals_kernel<T><<<nb, 256, 0, s>>>(qsrc, x, dfield[1], eta, ra, ra, za, rho, nr, nz, dsum + (size_t)3 * nb * slot,
                                                     (long long)nB, (long long)(nr - 1) * nz);
          XEE_LAUNCH_OK();
          dmade[2 + slot] = true;
        }
      }
      TraceTimer t5("  decompose: check solve");
      const int slot = 7 + t;   // the integral check L psi = f with theta_after
      T* x = dfield[2 + slot];
      if (solve_slot(x, f, prm_psi, slot, its, errs)) return 1;
      map_integrals_kernel<T><<<nb, 256, 0, s>>>(qsrc, x, dfield[1], nullptr, ra, ra, za, rho, nr, nz, dsum + (size_t)3 * nb * slot, (long long)nB);
      XEE_LAUNCH_OK();
      dmade[2 + slot] = true;
      if (bc) {
        exchange_conversion_kernel<T><<<nb, 256, 0, s>>>(x, dfield[3 + t], dfield[5 + t], dfield[7 + t], C, ra, za, rho, nr, nz, exch + (size_t)2 * nb * t);
        XEE_LAUNCH_OK();
      }
    }
    std::vector<double> hs((size_t)3 * nb * XEE_DECOMP_SOLVES), ht(nb), hx((size_t)4 * nb);
    XEE_CHECK(cudaMemcpyAsync(hs.data(), dsum, sizeof(double) * hs.size(), cudaMemcpyDeviceToHost, s));
    if (tend) XEE_CHECK(cudaMemcpyAsync(ht.data(), sdt, sizeof(double) * nb, cudaMemcpyDeviceToHost, s));
    if (bc) XEE_CHECK(cudaMemcpyAsync(hx.data(), exch, sizeof(double) * hx.size(), cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    const double gth = (double)k.g0 / (double)k.theta0, nan = std::numeric_limits<double>::quiet_NaN();
    auto sums = [&](int slot, int n) { return &hs[((size_t)slot * nb + n) * 3]; };
    for (int n = 0; n < nb; ++n) {
      double* r = table + (size_t)n * XEE_DECOMP_COLS;
      r[0] = sums(use[0] ? 7 : 8, n)[0];
      r[1] = tend ? ht[n] : nan;
      r[2] = r[1] / r[0];
      for (int t = 0; t < 2; ++t) {
        double* q = r + 3 + 7 * t;
        if (!use[t]) { for (int m = 0; m < 7; ++m) q[m] = nan; continue; }
        q[0] = bc ? sums(1 + t, n)[2] : nan;
        q[1] = sums(3 + t, n)[2];
        q[2] = sums(5 + t, n)[2];
        q[3] = bc ? hx[((size_t)t * nb + n) * 2] : nan;
        q[4] = bc ? hx[((size_t)t * nb + n) * 2 + 1] : nan;
        q[5] = ((bc ? q[0] : 0.0) + q[1]) + q[2];   // the decomposition sum, in the legacy driver's order
        if (bc) q[5] += q[3];
        q[6] = sums(7 + t, n)[1] * gth;
      }
    }
    if (iters_out) std::copy(its.begin(), its.end(), iters_out);
    if (err_out) std::copy(errs.begin(), errs.end(), err_out);
    return 0;
  }
  int get_decomp_field(int which, void* out) override {
    if (which < 0 || which >= kDecompFields) return fail("xee_series_get_decomp_field: unknown field");
    if (!dmade[which]) return fail("xee_series_get_decomp_field: the last decomposition did not make this field");
    const size_t bytes = sizeof(T) * (which < 2 ? (size_t)(d.nr - 1) * (d.nz - 1) : nn) * d.nsnap;
    XEE_CHECK(cudaMemcpy(out, dfield[which], bytes, cudaMemcpyDeviceToHost));
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
int xee_series_decompose_host(xee_series* m, const xee_decomp_desc* dd, const void* A, const void* B, const void* C, const void* Q,
                              const void* F, const void* psi_bc, const void* chi_bc, const xee_solve_params* prm_psi,
                              const xee_solve_params* prm_chi, double* table, int* iters, int* err) {
  DeviceGuard g(m->impl->device());
  return m->impl->decompose(dd, A, B, C, Q, F, psi_bc, chi_bc, true, prm_psi, prm_chi, table, iters, err, nullptr);
}
int xee_series_decompose_dev(xee_series* m, const xee_decomp_desc* dd, const void* A, const void* B, const void* C, const void* Q,
                             const void* F, const void* psi_bc, const void* chi_bc, const xee_solve_params* prm_psi,
                             const xee_solve_params* prm_chi, double* table, int* iters, int* err, void* stream) {
  DeviceGuard g(m->impl->device());
  return m->impl->decompose(dd, A, B, C, Q, F, psi_bc, chi_bc, false, prm_psi, prm_chi, table, iters, err, (cudaStream_t)stream);
}
int xee_series_get_decomp_field(xee_series* m, int which, void* out) { DeviceGuard g(m->impl->device()); return m->impl->get_decomp_field(which, out); }
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

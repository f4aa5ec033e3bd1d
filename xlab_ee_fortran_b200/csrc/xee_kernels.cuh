// xee_kernels.cuh — CUDA kernels of the elliptic-solve hot path (sm_100a).
//
//   K1  build_abc_kernel      src/diagnose/initialize-variables.f90:72-95
//   K2  cal_coe_kernel        xtt-lib-fortran/elliptic_tools.f90:35-56  (planar output + 1/(-coe5))
//   K3  sweep_direct_kernel   elliptic_tools.f90:189-190, 236-240 fused into one pass
//   K4  residual partials fused into K3 on check sweeps + finalize_check_kernel = the
//       stop-rule state machine of elliptic_tools.f90:193-233 run per solve on the device
//   K5  eta_kernel / uw_kernel   src/diagnose/quick-tools1.f90, quick-tools2.f90
//
// Device layout: a Fortran field f(nx,ny) is [ny][nx] (i contiguous); a batch is
// [n][ny][nx]; the operator is PLANAR: coe[set][10][ny][nx], planes 0..8 = coe1..coe9 and
// plane 9 = 1/(-coe5) (boundary entries 0).  The reference's AoS coe(9,nx,ny) exists only at
// the host boundary.
#pragma once
#include "xee_common.cuh"

namespace xee {

constexpr int kPlanes = 10;  // 9 coefficients + reciprocal of -coe5

// ------------------------------------------------------------------------------------ K1
template <class T>
__global__ void build_abc_kernel(const T* __restrict__ A, const T* __restrict__ B, const T* __restrict__ C,
                                 const T* __restrict__ rc, const T* __restrict__ rho, T* __restrict__ a,
                                 T* __restrict__ b, T* __restrict__ c, int nr, int nz) {
  using R = Rn<T>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // 0-based i-1
  const int j = blockIdx.y * blockDim.y + threadIdx.y;  // 0-based j-1
  if (i >= nr || j >= nz) return;
  {  // blockIdx.z = field set (time series: one vortex per snapshot)
    const size_t z = blockIdx.z;
    A += z * (size_t)nr * nz; B += z * (size_t)nr * nz; C += z * (size_t)nr * nz;
    a += z * (size_t)(nr - 1) * (nz - 2); b += z * (size_t)(nr - 1) * (nz - 1); c += z * (size_t)(nr - 2) * (nz - 1);
  }
  const size_t o = (size_t)j * nr + i;
  if (i < nr - 1 && j < nz - 2) {  // a(i,j) = (A(i,j+1)+A(i+1,j+1))/(rc(i)+rc(i+1))/rho(j+1)
    T v = R::add(A[o + nr], A[o + nr + 1]);
    a[(size_t)j * (nr - 1) + i] = R::div(R::div(v, R::add(rc[i], rc[i + 1])), rho[j + 1]);
  }
  if (i < nr - 1 && j < nz - 1) {  // b(i,j) = (B(i,j)+B(i+1,j)+B(i,j+1)+B(i+1,j+1))/(rc+rc)/(rho+rho)
    T v = R::add(R::add(R::add(B[o], B[o + 1]), B[o + nr]), B[o + nr + 1]);
    b[(size_t)j * (nr - 1) + i] = R::div(R::div(v, R::add(rc[i], rc[i + 1])), R::add(rho[j], rho[j + 1]));
  }
  if (i < nr - 2 && j < nz - 1) {  // c(i,j) = (C(i+1,j)+C(i+1,j+1))/rc(i+1)/(rho(j)+rho(j+1))
    T v = R::add(C[o + 1], C[o + nr + 1]);
    c[(size_t)j * (nr - 2) + i] = R::div(R::div(v, rc[i + 1]), R::add(rho[j], rho[j + 1]));
  }
}

// ------------------------------------------------------------------------------------ K2
// One thread per interior point.  a(nx-1,ny-2), b(nx-1,ny-1), c(nx-2,ny-1) as in the reference.
template <class T>
__global__ void cal_coe_kernel(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ c,
                               T* __restrict__ coe, T dx, T dy, int nx, int ny, long long abc_stride_a,
                               long long abc_stride_b, long long abc_stride_c, long long coe_set_stride) {
  using R = Rn<T>;
  const int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;  // 0-based
  const int j = 1 + blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= nx - 1 || j >= ny - 1) return;
  const int set = blockIdx.z;
  a += (size_t)set * abc_stride_a; b += (size_t)set * abc_stride_b; c += (size_t)set * abc_stride_c;
  coe += (size_t)set * coe_set_stride;
  const T PP = R::mul(dx, dx), QQ = R::mul(dy, dy), PQ4 = R::mul(R::mul(T(4), dx), dy);
  const T two_pq4 = R::mul(T(2), PQ4);
  // Fortran (I,J) = (i+1, j+1);  a(I,J-1) -> a[(j-1)*(nx-1) + i] etc.
  const size_t na = nx - 1, nb = nx - 1, nc = nx - 2;
  const T Ap = R::div(a[(size_t)(j - 1) * na + i], PP);
  const T Am = R::div(a[(size_t)(j - 1) * na + i - 1], PP);
  const T Cp = R::div(c[(size_t)j * nc + i - 1], QQ);
  const T Cm = R::div(c[(size_t)(j - 1) * nc + i - 1], QQ);
  const T b_ij = b[(size_t)j * nb + i], b_ijm = b[(size_t)(j - 1) * nb + i];
  const T b_imj = b[(size_t)j * nb + i - 1], b_imjm = b[(size_t)(j - 1) * nb + i - 1];
  const T BXp = R::div(R::add(b_ij, b_ijm), two_pq4);
  const T BXm = R::div(R::add(b_imj, b_imjm), two_pq4);
  const T BYp = R::div(R::add(b_imj, b_ij), two_pq4);
  const T BYm = R::div(R::add(b_imjm, b_ijm), two_pq4);
  const size_t nn = (size_t)nx * ny, o = (size_t)j * nx + i;
  const T c5 = -R::add(R::add(R::add(Am, Ap), Cm), Cp);
  coe[0 * nn + o] = -R::add(BXm, BYp);
  coe[1 * nn + o] = R::add(Cp, R::sub(BXp, BXm));
  coe[2 * nn + o] = R::add(BXp, BYp);
  coe[3 * nn + o] = R::sub(Am, R::sub(BYp, BYm));
  coe[4 * nn + o] = c5;
  coe[5 * nn + o] = R::add(Ap, R::sub(BYp, BYm));
  coe[6 * nn + o] = R::add(BXm, BYm);
  coe[7 * nn + o] = R::sub(Cm, R::sub(BXp, BXm));
  coe[8 * nn + o] = -R::add(BXp, BYm);
  coe[9 * nn + o] = R::rcp(-c5);
}

// AoS coe(9,nx,ny) [+ set] -> planar (+ reciprocal plane).  Boundary entries -> 0.
template <class T>
__global__ void aos_to_planar_kernel(const T* __restrict__ aos, T* __restrict__ coe, int nx, int ny) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= nx) return;
  const size_t nn = (size_t)nx * ny, o = (size_t)j * nx + i;
  const T* s = aos + ((size_t)blockIdx.z * nn + o) * 9;
  T* d = coe + (size_t)blockIdx.z * kPlanes * nn;
  const bool interior = i > 0 && i < nx - 1 && j > 0 && j < ny - 1;
  T c5 = 0;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    T v = interior ? s[k] : T(0);
    if (k == 4) c5 = v;
    d[k * nn + o] = v;
  }
  d[9 * nn + o] = interior ? Rn<T>::rcp(-c5) : T(0);
}
// planar -> AoS, interior only (the reference never writes coe's boundary entries).
template <class T>
__global__ void planar_to_aos_kernel(const T* __restrict__ coe, T* __restrict__ aos, int nx, int ny) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= nx) return;
  const size_t nn = (size_t)nx * ny, o = (size_t)j * nx + i;
  const bool interior = i > 0 && i < nx - 1 && j > 0 && j < ny - 1;
#pragma unroll
  for (int k = 0; k < 9; ++k) aos[o * 9 + k] = interior ? coe[k * nn + o] : T(0);
}

// ------------------------------------------------------------------------------------ K3/K4
template <class T>
struct SweepArgs {
  const T* src;    // psi_k       [n][ny][nx]
  T* dst;          // psi_{k+1}   (Chebyshev: holds psi_{k-1} on entry)
  const T* f;      // RHS
  const T* coe;    // planar operator
  long long coe_set_stride;  // elements between operator sets; 0 = shared
  long long field_stride;    // nx*ny
  int nx, ny, nbatch, spb;   // spb = solves handled by one block (operator kept in registers)
  T alpha;         // Jacobi weight
  T omega;         // Chebyshev weight of this sweep (1 on the first sweep); used when rho_ps == NULL
  const T* rho_ps; // per-solve Jacobi spectral radius (one operator per solve): omega computed in-kernel
  int cheb_k;      // index of this sweep in the Chebyshev sequence (1, 2, ...)
  const int* done; // per-solve stop flags (NULL = none)
  double* partial; // [n][ntiles] sum of r^2 per tile (check sweeps only)
  int ntiles;
  T* apply_out;    // APPLY mode: out = L psi
  int two_slot;    // two-level methods: which coarse-correction slot (0/1) belongs to `src` (the other one to `dst`)
};

enum { MODE_JACOBI = 0, MODE_CHEBYSHEV = 1, MODE_APPLY = 2 };

// Chebyshev weight of sweep k for Jacobi spectral radius rho:  omega_1 = 1,
// omega_k = 2 T_{k-1}(1/rho) / (rho T_k(1/rho)), in the stable ratio form with q = 1/rho - sqrt(1/rho^2 - 1).
__host__ __device__ inline double cheb_omega(int k, double rho) {
  if (k <= 1) return 1.0;
  const double sg = 1.0 / rho, q = sg - sqrt(sg * sg - 1.0);
  const double q2k = pow(q, 2.0 * (k - 1));
  return (2.0 / rho) * q * (1.0 + q2k) / (1.0 + q2k * q * q);
}

// The sequence omega_k converges to 2/(1+sqrt(1-rho^2)); beyond kChebClamp sweeps it is constant to double precision
// for any rho <= 1 - 1e-7.  Every kernel variant uses omega_{min(k, kChebClamp)} so that they stay bit-identical.
constexpr int kChebClamp = 8192;
inline double cheb_omega_host(int k, double rho) { return cheb_omega(k < kChebClamp ? k : kChebClamp, rho); }

constexpr int kDirBX = 64, kDirBY = 4;

// v1 "direct" sweep: one thread per grid point, the block walks `spb` solves with the nine
// coefficients (shared operator) held in registers; psi neighbours come through L1 (ld.global.nc).
// One pass = apply + subtract f (+ residual partial) + update: passes 1,2,(3),4 of the reference.
template <class T, int ARITH, int MODE, bool CHECK>
__global__ void __launch_bounds__(kDirBX* kDirBY) sweep_direct_kernel(const SweepArgs<T> a) {
  using R = Rn<T>;
  __shared__ double red[32];
  const int tid = threadIdx.y * kDirBX + threadIdx.x;
  const int i = 1 + blockIdx.x * kDirBX + threadIdx.x;
  const int j = 1 + blockIdx.y * kDirBY + threadIdx.y;
  const bool inside = (i < a.nx - 1) && (j < a.ny - 1);
  const size_t o = inside ? (size_t)j * a.nx + i : (size_t)a.nx + 1;
  const size_t nn = (size_t)a.field_stride;
  const int n0 = blockIdx.z * a.spb;
  const int n1 = min(n0 + a.spb, a.nbatch);
  const int nx = a.nx;
  T c[9], rcp = 0;
  const bool shared_op = (a.coe_set_stride == 0);
  if (shared_op) {
#pragma unroll
    for (int k = 0; k < 9; ++k) c[k] = __ldg(a.coe + k * nn + o);
    rcp = __ldg(a.coe + 9 * nn + o);
  }
  for (int n = n0; n < n1; ++n) {
    if (a.done != nullptr && a.done[n]) continue;  // block-uniform
    if (!shared_op) {
      const T* cc = a.coe + (size_t)n * a.coe_set_stride;
#pragma unroll
      for (int k = 0; k < 9; ++k) c[k] = __ldg(cc + k * nn + o);
      rcp = __ldg(cc + 9 * nn + o);
    }
    const T* s = a.src + (size_t)n * nn + o;
    T p[9];
    p[0] = __ldg(s + nx - 1); p[1] = __ldg(s + nx); p[2] = __ldg(s + nx + 1);
    p[3] = __ldg(s - 1);      p[4] = __ldg(s);      p[5] = __ldg(s + 1);
    p[6] = __ldg(s - nx - 1); p[7] = __ldg(s - nx); p[8] = __ldg(s - nx + 1);
    T r = apply9<T, ARITH>(c, p);
    if (MODE == MODE_APPLY) {
      if (inside) a.apply_out[(size_t)n * nn + o] = r;
      continue;
    }
    const T fv = __ldg(a.f + (size_t)n * nn + o);
    r = (ARITH == XEE_ARITH_STRICT) ? R::sub(r, fv) : r - fv;
    if (inside) {
      T* d = a.dst + (size_t)n * nn + o;
      if (MODE == MODE_JACOBI) {
        *d = jacobi_update<T, ARITH>(p[4], r, a.alpha, c[4], rcp);
      } else {  // Chebyshev-accelerated Jacobi: x+ = omega*(xJ - x-) + x-
        const T om = a.rho_ps ? (T)cheb_omega(a.cheb_k, (double)a.rho_ps[n]) : a.omega;
        const T xj = jacobi_update<T, ARITH>(p[4], r, T(1), c[4], rcp);
        const T xm = *d;
        *d = R::fma(om, xj - xm, xm);
      }
    }
    if (CHECK) {
      const double rr = inside ? (double)r * (double)r : 0.0;
      const double tot = block_sum(rr, red, tid, (kDirBX * kDirBY) / 32);
      if (tid == 0) a.partial[(size_t)n * a.ntiles + blockIdx.y * gridDim.x + blockIdx.x] = tot;
    }
  }
}

// Start vectors of the spectral probes (estimate_rho), for every operator set at once (grid.y = sets): kind 0 = the lowest sine
// mode sin(pi i/(nx-1)) sin(pi j/(ny-1)); kind 1 = the same, alternating in z and modulated (rough: for the largest eigenvalue
// of the two-level operator).  Zero on the boundary.  (Generated on the host and uploaded set by set until round 2: 4 ms of
// libm and pageable copies per probe.)
template <class T>
__global__ void probe_start_kernel(T* __restrict__ e, int nx, int ny, long long nn, int kind) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nx * ny) return;
  const int j = q / nx, i = q - j * nx;
  double v = 0.0;
  if (i >= 1 && i < nx - 1 && j >= 1 && j < ny - 1) {
    v = sin(M_PI * i / (nx - 1)) * sin(M_PI * j / (ny - 1));
    if (kind == 1) v = (double)(T)v * (double)((T)((j & 1) ? -1.0 : 1.0) * (T)(1.0 + 0.25 * sin(0.7 * i + 1.3 * j)));
  }
  e[(size_t)blockIdx.y * nn + q] = (T)v;
}
// set 0 of a probe vector copied to the sets 1 .. gridDim.y
template <class T>
__global__ void probe_replicate_kernel(T* __restrict__ e, long long nn) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < nn) e[(size_t)(blockIdx.y + 1) * nn + q] = e[q];
}

// D-weighted norm per solve, sum |coe5| x^2, for the spectral-radius probes: kWnormParts blocks per solve write partial sums
// (a single block per solve took 150 us for one 512x256 field: pure latency); the host adds them in a fixed order.
constexpr int kWnormParts = 32;
template <class T>
__global__ void __launch_bounds__(256) wnorm_kernel(const T* __restrict__ x, const T* __restrict__ coe,
                                                    long long coe_set_stride, long long nn, double* __restrict__ out) {
  __shared__ double red[32];
  const int n = blockIdx.y, part = blockIdx.x;
  const T* xp = x + (size_t)n * nn;
  const T* w = coe + (size_t)n * coe_set_stride + 4 * nn;
  double s = 0;
  for (long long q = (long long)part * 256 + threadIdx.x; q < nn; q += 256LL * kWnormParts) s += fabs((double)w[q]) * (double)xp[q] * (double)xp[q];
  const double t = block_sum(s, red, threadIdx.x, 8);
  if (threadIdx.x == 0) out[(size_t)n * kWnormParts + part] = t;
}

// Per-solve control state of solve_elliptic (elliptic_tools.f90:160-164, 201-233).
template <class T>
struct SolveState {
  int* done; int* iters; int* ccnt; int* lcnt; int* errb;
  T* err_before; T* err_now; T* ratio; T* r1; T* r2;
  T* best_err; int* stall;   // stagnation detector (opt-in, not in the reference)
  int* active;          // solves still iterating
  T* trace_err; T* trace_ratio; int trace_cap;   // solve 0 only (debug prints)
};

template <class T>
__global__ void init_state_kernel(SolveState<T> st, int nbatch, T r1, T r2, const T* r1_per_solve) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nbatch) return;
  T a1 = r1_per_solve ? r1_per_solve[n] : r1;
  // elliptic_tools.f90:112-124: a non-positive criterion is disabled by setting it to HUGE
  st.r1[n] = (a1 > T(0)) ? a1 : Rn<T>::huge();
  st.r2[n] = (r2 > T(0)) ? r2 : Rn<T>::huge();
  st.done[n] = 0; st.iters[n] = 0; st.ccnt[n] = 0; st.lcnt[n] = 0; st.errb[n] = 0;
  st.err_before[n] = Rn<T>::huge();   // :163
  st.err_now[n] = T(0); st.ratio[n] = T(0);
  st.best_err[n] = Rn<T>::huge(); st.stall[n] = 0;
  if (n == 0) *st.active = nbatch;
}

// max that lets a NaN through (the legacy isnan tests, old-diagnose/xtt-lib/elliptic_tools.f90:218-240, must still see it)
__device__ __forceinline__ double nanmax(double a, double b) { return (a != a) ? a : (b != b) ? b : (a > b ? a : b); }

constexpr int kResmaxBlocks = 64;
// Legacy strategies 3/4 (old-diagnose/xtt-lib/elliptic_tools.f90:203-204): err_now = maxval(abs(to_dat)) with to_dat = L psi - f
// on the interior.  One pass over psi on check sweeps only: partial[n][block] = max |L psi - f| over the block's points, in the
// same arithmetic as the sweep kernels (the maximum itself is exact in any order).
template <class T, int ARITH>
__global__ void __launch_bounds__(256) resmax_kernel(const T* __restrict__ src, const T* __restrict__ f, const T* __restrict__ coe,
                                                     long long coe_set_stride, long long field_stride, int nx, int ny,
                                                     const int* __restrict__ done, double* __restrict__ partial) {
  using R = Rn<T>;
  __shared__ double red[8];
  const int n = blockIdx.y;
  if (done != nullptr && done[n]) return;
  const size_t nn = (size_t)field_stride;
  const T* cc = coe + (size_t)n * coe_set_stride;
  const T* s0 = src + (size_t)n * nn;
  const T* f0 = f + (size_t)n * nn;
  const int wi = nx - 2, npts = wi * (ny - 2);
  double m = 0.0;
  for (int q = blockIdx.x * 256 + threadIdx.x; q < npts; q += gridDim.x * 256) {
    const int j = 1 + q / wi, i = 1 + q - (j - 1) * wi;
    const size_t o = (size_t)j * nx + i;
    T c[9], p[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) c[k] = __ldg(cc + k * nn + o);
    const T* s = s0 + o;
    p[0] = __ldg(s + nx - 1); p[1] = __ldg(s + nx); p[2] = __ldg(s + nx + 1);
    p[3] = __ldg(s - 1);      p[4] = __ldg(s);      p[5] = __ldg(s + 1);
    p[6] = __ldg(s - nx - 1); p[7] = __ldg(s - nx); p[8] = __ldg(s - nx + 1);
    T r = apply9<T, ARITH>(c, p);
    const T fv = __ldg(f0 + o);
    r = (ARITH == XEE_ARITH_STRICT) ? R::sub(r, fv) : r - fv;
    m = nanmax(m, fabs((double)r));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = nanmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = nanmax(m, red[w]);
    partial[(size_t)n * gridDim.x + blockIdx.x] = m;
  }
}

// The stop rule of one solve at one check (elliptic_tools.f90:201-233) and its two extensions: the explode rules
// (detect_explode) and the stall detector (stall_checks > 0).  The one copy of the rule: the per-launch sweep loop
// (finalize_check_kernel) and the resident solver call it.  Returns whether the solve stops here; `ratio` receives the
// signed relative change (err_before - err_now) / err_before of :201.
template <class T>
struct StopRule {
  T err_before, best;          // residual of the previous check (HUGE before the first one) and the best one seen
  int ccnt, lcnt, errb, stall;
};

template <class T>
__device__ __forceinline__ bool stop_rule_check(StopRule<T>& s, T err_now, T r1, T r2, int converge_time, int lost_rate,
                                                int detect_explode, int stall_checks, T& ratio) {
  using R = Rn<T>;
  ratio = R::div(R::sub(s.err_before, err_now), s.err_before);                   // :201
  const T aratio = R::abs(ratio);                                                 // :205
  bool stop = false;
  if (s.err_before == T(0)) {                                                     // :206
    stop = true;
  } else if ((err_now < r1) && (aratio < r2)) {                                   // :211
    s.ccnt += 1; s.lcnt = 0;
    if (s.ccnt >= converge_time) stop = true;
  } else if (s.ccnt > 0) {                                                        // :221
    s.lcnt += 1;
    if (s.lcnt >= lost_rate) { s.ccnt -= 1; s.lcnt = 0; }
  }
  if (detect_explode && !(err_now == err_now && R::abs(err_now) <= R::huge())) { stop = true; s.errb |= XEE_ERR_EXPLODE; }
  // (accelerated methods pass detect_explode = 1) a residual 10^6 above the best one seen is a divergent iteration too
  if (detect_explode && stall_checks > 0 && err_now > s.best * T(1e6)) { stop = true; s.errb |= XEE_ERR_EXPLODE; }
  if (stall_checks > 0 && !stop) {   // opt-in: the residual sits on its round-off floor above r1
    if (err_now < s.best * T(0.999)) { s.best = err_now; s.stall = 0; }
    else if (++s.stall >= stall_checks) { stop = true; s.errb |= XEE_ERR_STALLED; }
  }
  s.err_before = err_now;                                                         // :233
  return stop;
}

// One block per solve: deterministic sum of the tile partials, then the stop-rule state machine.
// norm_max != 0 (legacy strategies 3/4): the partials are maxima of |r| and err_now = max(they, floor_max), floor_max = the
// largest |boundary value| (the legacy maxval runs over the whole array, whose rim holds the Dirichlet values).
template <class T>
__global__ void __launch_bounds__(128) finalize_check_kernel(SolveState<T> st, const double* __restrict__ partial,
                                                             int ntiles, int ninterior, int cnt, int check_idx,
                                                             int converge_time, int lost_rate, int max_iter,
                                                             int detect_explode, int stall_checks, int norm_max = 0,
                                                             double floor_max = 0.0) {
  using R = Rn<T>;
  __shared__ double red[32];
  const int n = blockIdx.x;
  if (st.done[n]) return;
  double v = 0.0, tot;
  if (norm_max) {
    for (int t = threadIdx.x; t < ntiles; t += 128) v = nanmax(v, partial[(size_t)n * ntiles + t]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = nanmax(v, __shfl_down_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0)
      for (int w = 1; w < 4; ++w) v = nanmax(v, red[w]);
    tot = v;
  } else {
    for (int t = threadIdx.x; t < ntiles; t += 128) v += partial[(size_t)n * ntiles + t];
    tot = block_sum(v, red, threadIdx.x, 4);
  }
  if (threadIdx.x != 0) return;
  const T err_now = norm_max ? (T)nanmax(tot, floor_max) : R::sqrt(R::div((T)tot, (T)ninterior));   // :199 / legacy :204
  StopRule<T> r{st.err_before[n], st.best_err[n], st.ccnt[n], st.lcnt[n], st.errb[n], st.stall[n]};
  T ratio;
  bool stop = stop_rule_check(r, err_now, st.r1[n], st.r2[n], converge_time, lost_rate, detect_explode, stall_checks, ratio);
  if (n == 0 && check_idx < st.trace_cap) { st.trace_err[check_idx] = err_now; st.trace_ratio[check_idx] = ratio; }
  st.err_before[n] = r.err_before; st.best_err[n] = r.best; st.stall[n] = r.stall;
  st.err_now[n] = err_now; st.ratio[n] = R::abs(ratio);
  int errb = r.errb;
  if (cnt == max_iter) { stop = true; errb |= XEE_ERR_OVER_MAX_ITERATION; }       // :242-244
  st.ccnt[n] = r.ccnt; st.lcnt[n] = r.lcnt; st.errb[n] = errb;
  if (stop) { st.done[n] = 1; st.iters[n] = cnt; atomicSub(st.active, 1); }
}

// max_iter reached on a non-check sweep (elliptic_tools.f90:242-248).
template <class T>
__global__ void finalize_maxiter_kernel(SolveState<T> st, int nbatch, int max_iter) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nbatch || st.done[n]) return;
  st.done[n] = 1; st.iters[n] = max_iter; st.errb[n] |= XEE_ERR_OVER_MAX_ITERATION;
  atomicSub(st.active, 1);
}

// Final gather: solve n's result is in buffer (iters[n] & 1); copy it into x0 when it sits in x1.
// With `mirror_other` the other buffer gets what the reference leaves in `workspace`.
template <class T>
__global__ void select_result_kernel(T* __restrict__ x0, T* __restrict__ x1, const int* __restrict__ iters,
                                     long long nn, int mirror_other) {
  const int n = blockIdx.y;
  const bool in_x1 = iters[n] & 1;
  if (!in_x1) return;   // result already in x0; x1 holds the penultimate iterate (== reference workspace)
  T* a = x0 + (size_t)n * nn; const T* b = x1 + (size_t)n * nn;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nn; q += (long long)gridDim.x * blockDim.x) a[q] = b[q];
}

// Final gather of the temporally blocked solver (v4).  Pass p reads the iterate pair p&1 and writes the other one
// (pair 0 = (x0, x1), pair 1 = (x2, x3), each (latest, previous)); a solve that stopped after `iters` sweeps has been
// through npass = (iters / check_step) * ceil(check_step / tb) + ceil((iters % check_step) / tb) passes.  Leaves the
// result in x0 and in x1 what the reference leaves in `workspace` (elliptic_tools.f90:259-264: the penultimate iterate
// when the sweep count is even, a copy of the result when it is odd).
template <class T>
__global__ void select_result_tb_kernel(T* __restrict__ x0, T* __restrict__ x1, const T* __restrict__ x2,
                                        const T* __restrict__ x3, const int* __restrict__ iters, long long nn,
                                        int check_step, int tb) {
  const int n = blockIdx.y;
  const int it = iters[n];
  const int npass = (it / check_step) * ((check_step + tb - 1) / tb) + ((it % check_step) + tb - 1) / tb;
  const bool pair1 = npass & 1, odd = it & 1;
  if (!pair1 && !odd) return;
  T* a = x0 + (size_t)n * nn; T* b = x1 + (size_t)n * nn;
  const T* sn = pair1 ? x2 + (size_t)n * nn : a;
  const T* sp = pair1 ? x3 + (size_t)n * nn : b;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nn; q += (long long)gridDim.x * blockDim.x) {
    const T vn = sn[q], vp = sp[q];
    a[q] = vn;
    b[q] = odd ? vn : vp;
  }
}

// ------------------------------------------------------------------------------------ K5
// eta = d_rcuvdr_O2A(rchi) * g0 / (rho*Cp*exner*theta0)      quick-tools1.f90:1-13, quick-tools2.f90:59-85
template <class T>
__global__ void eta_kernel(const T* __restrict__ rchi, T* __restrict__ eta, const T* __restrict__ ra,
                           const T* __restrict__ rc, const T* __restrict__ rho, const T* __restrict__ ex, int nr,
                           int nz, T g0, T Cp, T theta0) {
  using R = Rn<T>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr - 1) return;
  const T* s = rchi + (size_t)blockIdx.z * nr * nz + (size_t)j * nr + i;
  T v = R::div(R::sub(s[1], s[0]), R::sub(ra[i + 1], ra[i]));
  v = R::div(v, R::div(R::add(rc[i], rc[i + 1]), T(2)));
  const T den = R::mul(R::mul(R::mul(rho[j], Cp), ex[j]), theta0);
  eta[(size_t)blockIdx.z * (nr - 1) * nz + (size_t)j * (nr - 1) + i] = R::div(R::mul(v, g0), den);
}
// w = d_rcuvdr_O2A(rpsi)/rho(j) on A; u = -d_dz_O2C(rpsi)/(rcuva(i)*(rho(j)+rho(j+1))/2) on C, 0 where ra(i)==0
template <class T>
__global__ void uw_kernel(const T* __restrict__ rpsi, T* __restrict__ u, T* __restrict__ w,
                          const T* __restrict__ ra, const T* __restrict__ rc, const T* __restrict__ za,
                          const T* __restrict__ rho, int nr, int nz) {
  using R = Rn<T>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr) return;
  const T* s = rpsi + (size_t)blockIdx.z * nr * nz + (size_t)j * nr + i;
  if (i < nr - 1) {
    T v = R::div(R::sub(s[1], s[0]), R::sub(ra[i + 1], ra[i]));
    v = R::div(v, R::div(R::add(rc[i], rc[i + 1]), T(2)));
    w[(size_t)blockIdx.z * (nr - 1) * nz + (size_t)j * (nr - 1) + i] = R::div(v, rho[j]);
  }
  if (j < nz - 1) {
    T v = -R::div(R::sub(s[nr], s[0]), R::sub(za[j + 1], za[j]));
    T out = T(0);
    if (ra[i] != T(0)) out = R::div(v, R::div(R::mul(rc[i], R::add(rho[j], rho[j + 1])), T(2)));
    u[(size_t)blockIdx.z * nr * (nz - 1) + (size_t)j * nr + i] = out;
  }
}

}  // namespace xee

// xee_map_kernels.cuh — kernels of the efficiency-map / time-series pipelines (see xee_map.cu, xee_series.cu).
#pragma once
#include "xee_plan.cuh"

namespace xee {

template <class T>
struct PhysK {  // xtt-lib-fortran/constants.f90:4-5 evaluated in T
  T g0 = T(9.8), theta0 = T(298.0), Rd = T(287.0), Cv, Cp, kappa, h0, p0 = T(101300.0);
  PhysK() { Cv = T(5.0) / T(2.0) * Rd; Cp = Cv + Rd; kappa = Rd / Cp; h0 = Cp * theta0 / g0; }
};

// Heating blob n: Q(r,z) = Q0 exp(-((r-rc)/sr)^2 - ((z-zc)/sz)^2) sampled at B-cell centres.
struct Heat { double rc, zc, sr, sz, q0; };

template <class T>
__device__ __forceinline__ T heat_q(const Heat& h, T r, T z) {
  const double dr = ((double)r - h.rc) / h.sr, dz = ((double)z - h.zc) / h.sz;
  return (T)(h.q0 * exp(-dr * dr - dz * dz));
}

// Where the kernels below take the heating Q on B cell (ci, cj) of solve n from.  at(n) gives the solve's evaluator once;
// calling it gives Q of one cell.
// BlobQ: the Gaussian blob heat[n] at the cell centre ((ra(ci)+ra(ci+1))/2, (za(cj)+za(cj+1))/2), evaluated in T.
template <class T>
struct BlobQ {
  const Heat* heat;
  struct At {
    Heat h;
    __device__ __forceinline__ T operator()(int ci, int cj, const T* ra, const T* za) const {
      using R = Rn<T>;
      const T rm = R::div(R::add(ra[ci], ra[ci + 1]), T(2)), zm = R::div(R::add(za[cj], za[cj + 1]), T(2));
      return heat_q<T>(h, rm, zm);
    }
  };
  __device__ __forceinline__ At at(int n) const {
    const Heat* h = heat + n;
    return At{Heat{__ldg(&h->rc), __ldg(&h->zc), __ldg(&h->sr), __ldg(&h->sz), __ldg(&h->q0)}};
  }
};
// FieldQ: a caller's field, [n][nz-1][nr-1] with i fastest.
template <class T>
struct FieldQ {
  const T* Q;
  int nr, nz;
  struct At {
    const T* q; int ld;
    __device__ __forceinline__ T operator()(int ci, int cj, const T*, const T*) const { return __ldg(q + (size_t)cj * ld + ci); }
  };
  __device__ __forceinline__ At at(int n) const { return At{Q + (size_t)n * (nr - 1) * (nz - 1), nr - 1}; }
};

// K7: f(i,j) = g0/theta0 * ( dJ(i,j) + dJ(i,j-1) )/2 on the O interior, 0 on the boundary,
//     dJ(i,j) = (J(i,j)-J(i-1,j)) / ((ra(i+1)-ra(i-1))/2),  J(i,j) = Q(i,j)/(Cp*exner(j))   [B grid]
// A block of kHeatBX x kHeatBY points first forms J on the (kHeatBX+1) x (kHeatBY+1) B cells it touches (an exp and a division
// each; every cell is shared by four points: a thread that evaluates its own four cells spends 4 exps and 12 divisions per
// point and the kernel is fp64-pipe bound, 2.1 ms per 512-solve map), then every point combines its four cells with exactly
// the operations, in the order, of the reference: the values are bit for bit the same.
constexpr int kHeatBX = 64, kHeatBY = 4;
inline dim3 heating_rhs_grid(int nr, int nz, int nb) { return dim3((nr + kHeatBX - 1) / kHeatBX, (nz + kHeatBY - 1) / kHeatBY, nb); }
template <class T, class QSrc>
__global__ void __launch_bounds__(kHeatBX* kHeatBY) heating_rhs_kernel(QSrc src, T* __restrict__ f,
                                                                      const T* __restrict__ ra, const T* __restrict__ za,
                                                                      const T* __restrict__ ex, int nr, int nz, T g0, T theta0, T Cp) {
  using R = Rn<T>;
  __shared__ T Jc[kHeatBY + 1][kHeatBX + 1];     // cell (ci, cj) = (i0 - 1 + x, j0 - 1 + y)
  const int i0 = blockIdx.x * kHeatBX, j0 = blockIdx.y * kHeatBY, n = blockIdx.z;
  const int tid = threadIdx.y * kHeatBX + threadIdx.x;
  const auto Qn = src.at(n);
  for (int q = tid; q < (kHeatBX + 1) * (kHeatBY + 1); q += kHeatBX * kHeatBY) {
    const int x = q % (kHeatBX + 1), y = q / (kHeatBX + 1);
    const int ci = i0 - 1 + x, cj = j0 - 1 + y;
    T v = T(0);
    if (ci >= 0 && ci <= nr - 2 && cj >= 0 && cj <= nz - 2) {
      // Fortran (I,J) = (ci+1,cj+1); J(.,J) uses exner(J)
      v = R::div(Qn(ci, cj, ra, za), R::mul(Cp, ex[cj]));
    }
    Jc[y][x] = v;
  }
  __syncthreads();
  const int i = i0 + threadIdx.x, j = j0 + threadIdx.y;  // 0-based O index
  if (i >= nr || j >= nz) return;
  T out = T(0);
  if (i > 0 && i < nr - 1 && j > 0 && j < nz - 1) {
    const int x = threadIdx.x + 1, y = threadIdx.y + 1;  // cell (i, j); (i-1, .) and (., j-1) sit one to the left / below
    const T dist = R::div(R::sub(ra[i + 1], ra[i - 1]), T(2));
    const T dJU = R::div(R::sub(Jc[y][x], Jc[y][x - 1]), dist);
    const T dJD = R::div(R::sub(Jc[y - 1][x], Jc[y - 1][x - 1]), dist);
    out = R::div(R::mul(R::div(R::add(dJU, dJD), T(2)), g0), theta0);
  }
  f[(size_t)n * nr * nz + (size_t)j * nr + i] = out;
}

// Cell weight rho_ * rcuv * dr * dz of integrate_weight_B (old-diagnose/diagnose.f90:1038-1044), applied
// left to right to `v` exactly as the reference multiplies.
template <class T>
__device__ __forceinline__ T weighted(T v, const T* ra, const T* rc, const T* za, const T* rho, int i, int j) {
  using R = Rn<T>;
  const T rcuv = R::div(R::add(rc[i], rc[i + 1]), T(2));
  const T dr = R::sub(ra[i + 1], ra[i]);
  const T dz = R::sub(za[j + 1], za[j]);
  const T rho_ = R::div(R::add(rho[j + 1], rho[j]), T(2));
  return R::mul(R::mul(R::mul(R::mul(v, rho_), rcuv), dr), dz);
}

// One block per heating location: sum_Q, (g0/theta0) * I[w theta], optional I[Q (eta(i,j)+eta(i,j+1))/2].
// Deterministic tree reduction in double (the reference sums sequentially in real(4)).
template <class T, class QSrc>
__global__ void __launch_bounds__(256) map_integrals_kernel(QSrc src, const T* __restrict__ psi,
                                                            const T* __restrict__ theta, const T* __restrict__ eta,
                                                            const T* __restrict__ ra, const T* __restrict__ rc,
                                                            const T* __restrict__ za, const T* __restrict__ rho,
                                                            int nr, int nz, double* __restrict__ out /*[n][3]*/,
                                                            long long theta_stride = 0, long long eta_stride = 0) {
  using R = Rn<T>;
  __shared__ double red[32];
  const int n = blockIdx.x;
  const auto Qn = src.at(n);
  const T* p = psi + (size_t)n * nr * nz;
  theta += (size_t)n * theta_stride;
  if (eta != nullptr) eta += (size_t)n * eta_stride;
  const int ncell = (nr - 1) * (nz - 1);
  double sq = 0, swt = 0, sqe = 0;
  for (int q = threadIdx.x; q < ncell; q += 256) {
    const int i = q % (nr - 1), j = q / (nr - 1);
    const T Q = Qn(i, j, ra, za);
    sq += (double)weighted<T>(Q, ra, rc, za, rho, i, j);
    // w(i,j) = d_rcuvdr_O2A(rpsi)/rho(j)  (rpsiToUW, old-diagnose/diagnose.f90:921-927)
    const T den_r = R::sub(ra[i + 1], ra[i]), rcm = R::div(R::add(rc[i], rc[i + 1]), T(2));
    const T w0 = R::div(R::div(R::div(R::sub(p[(size_t)j * nr + i + 1], p[(size_t)j * nr + i]), den_r), rcm), rho[j]);
    const T w1 = R::div(R::div(R::div(R::sub(p[(size_t)(j + 1) * nr + i + 1], p[(size_t)(j + 1) * nr + i]), den_r), rcm), rho[j + 1]);
    const T wth = R::mul(R::div(R::add(w0, w1), T(2)), theta[(size_t)j * (nr - 1) + i]);        // cal_wtheta :1124
    swt += (double)weighted<T>(wth, ra, rc, za, rho, i, j);
    if (eta != nullptr) {
      const T e = R::div(R::add(eta[(size_t)j * (nr - 1) + i], eta[(size_t)(j + 1) * (nr - 1) + i]), T(2));
      sqe += (double)weighted<T>(R::mul(e, Q), ra, rc, za, rho, i, j);                         // cal_sum_Qeta :1088
    }
  }
  const double a = block_sum(sq, red, threadIdx.x, 8);
  const double b = block_sum(swt, red, threadIdx.x, 8);
  const double c = block_sum(sqe, red, threadIdx.x, 8);
  if (threadIdx.x == 0) { out[3 * n + 0] = a; out[3 * n + 1] = b; out[3 * n + 2] = c; }
}

// rhoB_B(i,j) = 4-point average of an O-grid B on B cell (i, j), 0-based   old-diagnose/diagnose.f90:335-336
template <class T>
__device__ __forceinline__ T rhoB_B_of(const T* B, int nr, int i, int j) {
  using R = Rn<T>;
  const size_t o = (size_t)j * nr + i;
  return R::div(R::add(R::add(R::add(B[o], B[o + 1]), B[o + nr]), B[o + nr + 1]), T(4));
}

// The state relative_theta_kernel integrates, per field set n: at(n) gives rhoB_C(i) on the bottom row (0-based C index
// i = 1..nr-2) and rhoA_A(i, j) (0-based A index, j = 1..nz-2).
// BasicState: the basic state of A and B, rhoA_A = (A(i,j)+A(i+1,j))/2, rhoB_C(i,j) = (rhoB_B(i-1,j)+rhoB_B(i,j))/2
// (old-diagnose/diagnose.f90:329-354, 503-509); the state after a tendency step is another (xee_series.cu).
template <class T>
struct BasicState {
  const T* A; const T* B; int nr, nz;
  struct At {
    const T* A; const T* B; int nr;
    __device__ __forceinline__ T rhoB_C(int i) const {
      using R = Rn<T>;
      return R::div(R::add(rhoB_B_of(B, nr, i - 1, 0), rhoB_B_of(B, nr, i, 0)), T(2));
    }
    __device__ __forceinline__ T rhoA_A(int i, int j) const {
      using R = Rn<T>;
      return R::div(R::add(A[(size_t)j * nr + i], A[(size_t)j * nr + i + 1]), T(2));
    }
  };
  __device__ __forceinline__ At at(int n) const { return At{A + (size_t)n * nr * nz, B + (size_t)n * nr * nz, nr}; }
};

// Potential temperature on B of a state S (blockIdx.x = field set):
//   theta = relativeTheta(theta, rhoA_A*theta0/g0, rhoB_C*(-theta0/g0))          old-diagnose/diagnose.f90:893-912
// One block; thread 0 integrates the bottom row in r, then one thread per column integrates in z.
template <class T, class S>
__global__ void relative_theta_kernel(S st, T* __restrict__ theta, const T* __restrict__ ra, const T* __restrict__ za,
                                      int nr, int nz, T g0, T theta0) {
  using R = Rn<T>;
  const auto sn = st.at(blockIdx.x);
  theta += (size_t)blockIdx.x * (nr - 1) * (nz - 1);
  const T k = R::div(theta0, g0);
  if (threadIdx.x == 0) {
    theta[0] = theta0;
    for (int i = 1; i < nr - 1; ++i) {   // Fortran i = 2..nr-1
      const T dist = R::div(R::sub(ra[i + 1], ra[i - 1]), T(2));
      theta[i] = R::add(theta[i - 1], R::mul(dist, R::mul(sn.rhoB_C(i), -k)));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nr - 1; i += blockDim.x) {
    for (int j = 1; j < nz - 1; ++j) {   // Fortran j = 2..nz-1
      const T dist = R::div(R::sub(za[j + 1], za[j - 1]), T(2));
      theta[(size_t)j * (nr - 1) + i] = R::add(theta[(size_t)(j - 1) * (nr - 1) + i], R::mul(dist, R::mul(sn.rhoA_A(i, j), k)));
    }
  }
}

// Where rhs_from_B_kernel takes the B-cell field b of set n from.  OGridB: rhoB_B of an O-grid B [n][nz][nr] (f_basic);
// BGridB: a B-cell field [n][nz-1][nr-1] (f_anomaly of the time series' decomposition).
template <class T>
struct OGridB {
  const T* B; int nr, nz;
  struct At {
    const T* B; int nr;
    __device__ __forceinline__ T operator()(int i, int j) const { return rhoB_B_of(B, nr, i, j); }
  };
  __device__ __forceinline__ At at(int n) const { return At{B + (size_t)n * nr * nz, nr}; }
};
template <class T>
struct BGridB {
  const T* b; int nr, nz;
  struct At {
    const T* b; int ld;
    __device__ __forceinline__ T operator()(int i, int j) const { return b[(size_t)j * ld + i]; }
  };
  __device__ __forceinline__ At at(int n) const { return At{b + (size_t)n * (nr - 1) * (nz - 1), nr - 1}; }
};

// f = -(4-point average of b) on the O interior, 0 on the rim; blockIdx.z = field set   old-diagnose/diagnose.f90:524-530
template <class T, class BSrc>
__global__ void rhs_from_B_kernel(BSrc src, T* __restrict__ f, int nr, int nz) {
  using R = Rn<T>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr) return;
  const auto bb = src.at(blockIdx.z);
  T out = T(0);
  if (i > 0 && i < nr - 1 && j > 0 && j < nz - 1)
    out = -R::div(R::add(R::add(R::add(bb(i - 1, j - 1), bb(i - 1, j)), bb(i, j)), bb(i, j - 1)), T(4));
  f[(size_t)blockIdx.z * nr * nz + (size_t)j * nr + i] = out;
}

template <class T>
__global__ void f32_to_T_kernel(const float* __restrict__ in, T* __restrict__ out, size_t n) {
  const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < n) out[q] = (T)in[q];
}
// out[n] = scale * rms over the interior of (x - y): the initial residual L psi0 - f of a solve.
template <class T>
__global__ void rms_diff_interior_kernel(const T* __restrict__ x, const T* __restrict__ y, int nr, int nz, T scale,
                                         T* __restrict__ out) {
  __shared__ double red[32];
  const T* p = x + (size_t)blockIdx.x * nr * nz;
  const T* q = y + (size_t)blockIdx.x * nr * nz;
  double s = 0;
  for (int k = threadIdx.x; k < nr * nz; k += 256) {
    const int i = k % nr, j = k / nr;
    if (i > 0 && i < nr - 1 && j > 0 && j < nz - 1) { const double dv = (double)p[k] - (double)q[k]; s += dv * dv; }
  }
  const double t = block_sum(s, red, threadIdx.x, 8);
  if (threadIdx.x == 0) out[blockIdx.x] = (T)(sqrt(t / ((double)(nr - 2) * (nz - 2))) * (double)scale);
}
template <class T>
__global__ void rms_interior_kernel(const T* __restrict__ f, int nr, int nz, T scale, T* __restrict__ out) {
  __shared__ double red[32];
  const T* p = f + (size_t)blockIdx.x * nr * nz;
  double s = 0;
  for (int q = threadIdx.x; q < nr * nz; q += 256) {
    const int i = q % nr, j = q / nr;
    if (i > 0 && i < nr - 1 && j > 0 && j < nz - 1) s += (double)p[q] * (double)p[q];
  }
  const double t = block_sum(s, red, threadIdx.x, 8);
  if (threadIdx.x == 0) out[blockIdx.x] = (T)(sqrt(t / ((double)(nr - 2) * (nz - 2))) * (double)scale);
}

}  // namespace xee

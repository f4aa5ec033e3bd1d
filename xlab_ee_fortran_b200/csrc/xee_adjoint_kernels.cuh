// xee_adjoint_kernels.cuh — the discrete adjoint of the efficiency map (see xee_map.cu, DESIGN.md "Discrete-adjoint
// efficiency maps").
//
// ke_gen of one heating location is linear in its field psi, psi = L^-1 f, and f = H Q is linear in its heating Q:
//     ke_gen = <g, L^-1 H Q> = <H^T L^-T g, Q> = sum over the B cells of mu_c Q_c
// with g the gradient of ke_gen in psi (ke_functional_kernel), lambda the solution of L^T lambda = g (one solve, operator
// from transpose_coe_kernel) and mu = H^T lambda (heating_adjoint_kernel).  Every transpose below is the exact transpose of
// the map kernel it names, so the efficiencies agree with the direct solves' to solver tolerance.
#pragma once
#include "xee_map_kernels.cuh"

namespace xee {

// L^T in the plan's planar layout, from L (set 0 of `coe`).  Slot k sits at offset o_k = ((k % 3) - 1, 1 - k / 3) (apply9);
// slot k of L^T at interior point p is slot 8 - k of L at p + o_k (the pairs 1-9, 2-8, 3-7, 4-6, 5-5 of the reference's
// numbering), 0 where p + o_k is on the rim: rim points are Dirichlet data and carry no row.  Plane 9 = 1/(-coe5), as
// aos_to_planar_kernel forms it; the diagonal is its own transpose.  Rim entries 0.
template <class T>
__global__ void transpose_coe_kernel(const T* __restrict__ coe, T* __restrict__ coe_t, int nx, int ny) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nx) return;
  const size_t nn = (size_t)nx * ny, o = (size_t)j * nx + i;
  const bool interior = i > 0 && i < nx - 1 && j > 0 && j < ny - 1;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int qi = i + (k % 3) - 1, qj = j + 1 - k / 3;
    const bool q_in = qi > 0 && qi < nx - 1 && qj > 0 && qj < ny - 1;
    coe_t[k * nn + o] = interior && q_in ? coe[(size_t)(8 - k) * nn + (size_t)qj * nx + qi] : T(0);
  }
  coe_t[9 * nn + o] = interior ? Rn<T>::rcp(-coe[4 * nn + o]) : T(0);
}

// g = d ke_gen / d psi on the O grid, ke_gen = (g0/theta0) * swt of map_integrals_kernel:
//   swt = sum_c W_c theta_c (w0_c + w1_c) / 2,  w0 = (psi(i+1,j) - psi(i,j)) / (dr_i rbar_i rho_j),  w1 the same on row j+1
// so psi(I,J) enters the cells (I-1, cj) with + and (I, cj) with -, cj in {J-1, J}, each through 1/rho_J:
//   g(I,J) = (g0/theta0) / (2 rho_J) * sum_cj [ W theta / (dr rbar) (I-1, cj) - W theta / (dr rbar) (I, cj) ]
// Interior points only (the map's psi is 0 on the rim); all four cells of an interior point exist.
template <class T>
__global__ void ke_functional_kernel(const T* __restrict__ theta, const T* __restrict__ ra, const T* __restrict__ za,
                                     const T* __restrict__ rho, int nr, int nz, T g0, T theta0, T* __restrict__ g) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= nr) return;
  T out = T(0);
  if (i > 0 && i < nr - 1 && j > 0 && j < nz - 1) {
    auto cell = [&](int ci, int cj) {   // W theta / (dr rbar) of B cell (ci, cj)
      const T wt = weighted<T>(theta[(size_t)cj * (nr - 1) + ci], ra, ra, za, rho, ci, cj);
      return wt / ((ra[ci + 1] - ra[ci]) * ((ra[ci] + ra[ci + 1]) / T(2)));
    };
    const T s = (cell(i - 1, j - 1) - cell(i, j - 1)) + (cell(i - 1, j) - cell(i, j));
    out = g0 / theta0 * s / (T(2) * rho[j]);
  }
  g[(size_t)j * nr + i] = out;
}

// mu = H^T lambda on the (nr-1) x (nz-1) B cells, H = heating_rhs_kernel's map Q -> f:
//   f(i,j) = (g0/theta0)/2 * sum_{cj in {j-1, j}} (J(i,cj) - J(i-1,cj)) / d_i,  J = Q / (Cp exner_cj),  d_i = (r_{i+1} - r_{i-1})/2
//   mu(ci,cj) = (g0/theta0) / (2 Cp exner_cj) * [ (lambda(ci,cj) + lambda(ci,cj+1)) / d_ci - (lambda(ci+1,cj) + lambda(ci+1,cj+1)) / d_ci+1 ]
// lambda is 0 on the rim: a term whose column ci or ci+1 is a rim column drops out.  eta_d = mu / W_c is the efficiency of
// heating concentrated in cell c.
template <class T>
__global__ void heating_adjoint_kernel(const T* __restrict__ lam, const T* __restrict__ ra, const T* __restrict__ za,
                                       const T* __restrict__ ex, const T* __restrict__ rho, int nr, int nz, T g0, T theta0,
                                       T Cp, T* __restrict__ mu, T* __restrict__ eta_d) {
  const int ci = blockIdx.x * blockDim.x + threadIdx.x, cj = blockIdx.y;
  if (ci >= nr - 1) return;
  T s = T(0);
  if (ci >= 1) s += (lam[(size_t)cj * nr + ci] + lam[(size_t)(cj + 1) * nr + ci]) / ((ra[ci + 1] - ra[ci - 1]) / T(2));
  if (ci + 1 <= nr - 2) s -= (lam[(size_t)cj * nr + ci + 1] + lam[(size_t)(cj + 1) * nr + ci + 1]) / ((ra[ci + 2] - ra[ci]) / T(2));
  const T m = g0 / theta0 * s / (T(2) * Cp * ex[cj]);
  const size_t o = (size_t)cj * (nr - 1) + ci;
  mu[o] = m;
  eta_d[o] = m / weighted<T>(T(1), ra, ra, za, rho, ci, cj);
}

// Cells whose heating exponent -(dr^2 + dz^2) lies below -kExpZero have Q = q0 exp(...) = 0 exactly: exp underflows to 0
// below about -745.1 in fp64, and 800 leaves a margin no rounding of the exponent can cross.
constexpr double kExpZero = 800.0;

// One block per heating location: out[n] = {sum_c W_c Q_c, sum_c mu_c Q_c}, Q = heat_q exactly as in the direct path.
// Thread t takes the cells q = t (mod 256) of the row-major cell order in increasing q and the block sums its partials in a
// fixed tree, as map_integrals_kernel does: a row depends on its own heating only, not on how many rows share the call, and
// sum_Q is bit for bit column 3 of the map table.  window = 1 visits only the rows and columns of cells whose exponent can
// be above -kExpZero; the cells it skips add exact zeros, so the partial sums and the results are the same bits as window = 0.
template <class T>
__global__ void __launch_bounds__(256) adjoint_eval_kernel(const Heat* __restrict__ heat, const T* __restrict__ mu,
                                                           const T* __restrict__ ra, const T* __restrict__ za,
                                                           const T* __restrict__ rho, int nr, int nz, int window,
                                                           double* __restrict__ out /*[n][2]*/) {
  using R = Rn<T>;
  __shared__ double red[32];
  __shared__ int win[4];   // first and last cell column, first and last cell row
  const int n = blockIdx.x, ncr = nr - 1, ncz = nz - 1;
  const Heat h = heat[n];
  int i0 = 0, i1 = ncr - 1, j0 = 0, j1 = ncz - 1;
  if (window) {
    if (threadIdx.x == 0) { win[0] = ncr; win[1] = -1; win[2] = ncz; win[3] = -1; }
    __syncthreads();
    for (int i = threadIdx.x; i < ncr; i += 256) {
      const T rm = R::div(R::add(ra[i], ra[i + 1]), T(2));
      const double x = ((double)rm - h.rc) / h.sr;
      if (!(x * x > kExpZero)) { atomicMin(&win[0], i); atomicMax(&win[1], i); }
    }
    for (int j = threadIdx.x; j < ncz; j += 256) {
      const T zm = R::div(R::add(za[j], za[j + 1]), T(2));
      const double y = ((double)zm - h.zc) / h.sz;
      if (!(y * y > kExpZero)) { atomicMin(&win[2], j); atomicMax(&win[3], j); }
    }
    __syncthreads();
    i0 = win[0]; i1 = win[1]; j0 = win[2]; j1 = win[3];
  }
  double sq = 0, smq = 0;
  for (int j = j0; j <= j1; ++j) {
    const long long row = (long long)j * ncr;
    const int lead = (int)(((long long)threadIdx.x - (row + i0)) % 256 + 256) % 256;   // first i >= i0 with q = t (mod 256)
    for (int i = i0 + lead; i <= i1; i += 256) {
      const T rm = R::div(R::add(ra[i], ra[i + 1]), T(2)), zm = R::div(R::add(za[j], za[j + 1]), T(2));
      const T Q = heat_q<T>(h, rm, zm);
      sq += (double)weighted<T>(Q, ra, ra, za, rho, i, j);
      smq += (double)mu[row + i] * (double)Q;
    }
  }
  const double a = block_sum(sq, red, threadIdx.x, 8);
  const double b = block_sum(smq, red, threadIdx.x, 8);
  if (threadIdx.x == 0) { out[2 * (size_t)n] = a; out[2 * (size_t)n + 1] = b; }
}

}  // namespace xee

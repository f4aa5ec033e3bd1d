// xee_mixed.cuh — fp64 iterative refinement around fp32 two-level block-line Chebyshev sweeps (XEE_METHOD_LINE2_MIXED),
// sm_100a.
//
// Same discrete problem, same residual (do_elliptic's nine-term sum, xtt-lib-fortran/elliptic_tools.f90:77-85, in fp64 on
// the fp64 operator) and the same stop rule (:193-233, stop_rule_check) as every other method; fp64 fields in and out.
// Only the CORRECTION is computed in fp32:
//
//   start    r = f - L psi                                      (mixed_residual_kernel, twice: the scale needs the norm)
//   step     e = 0;  check_step fp32 two-level Chebyshev sweeps on  L32 e = r32,  r32 = r / s  (sweep_line_kernel<float,
//            .., TWO> + the fp64 coarse solve of xee_twolevel.cuh; the coarse vectors c stay fp64)
//            psi += s (e + P c)                                 (mixed_fold_kernel, fp64; also zeroes e for the next step)
//            r = f - L psi, r32 = r / s', Sum r^2 per tile     (mixed_residual_kernel -> the unchanged finalize_check_kernel)
//
// L32 is the fp64 operator rounded to fp32, with its block-line factors and pack built from it in fp32 (line_factor_kernel
// <float>, line_pack_kernel<float>); the Galerkin inverse and the Chebyshev parameters (estimate_rho on the fp64 operator)
// are the fp64 ones: both only shape the approximate inverse, which the fp64 residual of every step corrects.
//
// Semantics:
//   * iters, max_iter and check_step count fp32 sweeps; a refinement step is check_step sweeps and ends with one check.
//     The Chebyshev sequence restarts with every step (weight index 1 .. check_step).
//   * s is a power of two per solve: the one just above the RMS of the previous check's residual (of the first guess for
//     the first step), so r32 = r / s and s (e + P c) are exact scalings.  With a step's contraction of 1e-6 .. 1e-7, r32 then
//     has an RMS around that contraction, never near fp32's range limits, whatever the scale of f; fp32 arithmetic is
//     invariant under power-of-two scaling, so the correction does not depend on which power of two was picked.
//   * A solve that reaches max_iter inside a step applies the partial correction and ends; sweeps(n) does the same, so a
//     solve that stops at iters = n returns the bits of sweeps(n) with the same check_step.
//   * The fp32 pair (e, previous e) of the Chebyshev recurrence lives in the plan's fp64 scratch field x1 (two fp32 fields
//     per solve); r32 is one more fp32 field per solve.
//   * The update is two passes, not one: an in-place stencil pass would read neighbours of psi that another block has
//     already overwritten.  The point-wise fold also clears e, which the next step needs anyway.
#pragma once
#include "xee_krylov.cuh"
#include "xee_twolevel.cuh"

namespace xee {
namespace mx {

constexpr int BX = kDirBX, BY = kDirBY;   // residual pass: one thread per interior point, partials per 64 x 4 tile

static __global__ void to_f32_kernel(const double* __restrict__ src, float* __restrict__ dst, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = (float)src[i];
}

// psi += s (e + P c) on the interior points, e = the fp32 iterate of the last sweep (buffer `e_last`), c its coarse vector,
// s = scale[n]; then both fp32 buffers of the solve are zeroed.  Thread = one 8-point radial segment of one row, the
// prolongation as in tl::prolong_add_kernel.
static __global__ void __launch_bounds__(256) mixed_fold_kernel(double* __restrict__ psi, const float* __restrict__ e_last,
                                                                float* __restrict__ e_pair, const double* __restrict__ Cv,
                                                                const double* __restrict__ scale, const int* __restrict__ done,
                                                                int nx, int ny, int nb, int px, int pzpx) {
  using namespace tl;
  const int n = blockIdx.z;
  if (done && done[n]) return;
  const int nseg = (nx + 7) / 8;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = idx / nseg, sgm = idx % nseg;
  if (j >= ny) return;
  const size_t nn = (size_t)nx * ny, o = (size_t)n * nn + (size_t)j * nx + 8 * sgm;
  if (j >= 1 && j <= ny - 2) {
    const double* cv = Cv + (size_t)n * pzpx + COL0;
    const int q0 = j / HZ, p0 = sgm / 2; const double tz = (double)(j % HZ) * (1.0 / HZ);
    const double c00 = cv[q0 * px + p0], c01 = cv[q0 * px + p0 + 1], c10 = cv[(q0 + 1) * px + p0], c11 = cv[(q0 + 1) * px + p0 + 1];
    const double vl = fma(tz, c10 - c00, c00), vr = fma(tz, c11 - c01, c01);
    const double sl = (vr - vl) * (1.0 / HR), base = fma(sl, (double)(8 * (sgm & 1)), vl);
    const double sc = scale[n];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int i = 8 * sgm + e;
      if (i >= 1 && i <= nx - 2) psi[o + e] = fma(sc, (double)e_last[o + e] + fma(sl, (double)e, base), psi[o + e]);
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e)
    if (8 * sgm + e < nx) { e_pair[o + e] = 0.f; e_pair[(size_t)nb * nn + o + e] = 0.f; }
}

// r = f - L psi on the interior (fp64, the nine-term sum in the reference's order on the fp64 operator), Sum r^2 per
// (solve, tile) into `partial`; with r32 != NULL also r32 = r / div[n] (div a power of two: exact up to the fp32 rounding).
static __global__ void __launch_bounds__(BX* BY) mixed_residual_kernel(const double* __restrict__ psi, const double* __restrict__ f,
                                                                       const double* __restrict__ coe, long long coe_set_stride,
                                                                       int nx, int ny, const double* __restrict__ div,
                                                                       float* __restrict__ r32, double* __restrict__ partial,
                                                                       const int* __restrict__ done) {
  __shared__ double red[32];
  const kr::Point q = kr::point(nx, ny);
  if (done && done[q.n]) return;
  const long long nn = (long long)nx * ny;
  double rr = 0.0;
  if (q.inside) {
    const size_t oc = q.o - (size_t)q.n * nn;
    const double r = __ldg(f + q.o) - kr::apply_d(coe + (size_t)q.n * coe_set_stride, psi, oc, q.o, nx, nn);
    if (r32) r32[q.o] = (float)(r / div[q.n]);
    rr = r * r;
  }
  const double tot = block_sum(rr, red, q.tid, BX * BY / 32);
  if (q.tid == 0) partial[(size_t)q.n * gridDim.x * gridDim.y + q.tile] = tot;
}

// The scale of the next residual pass from the one just measured, per solve (fixed summation order):
// shift = 1: scale[n] = scale[nb + n] (the divisor of the r32 now in memory, the multiplier of the next fold) first; then
// scale[nb + n] = the power of two at or above the RMS (1 for a zero or non-finite RMS).
static __global__ void __launch_bounds__(128) mixed_scale_kernel(const double* __restrict__ partial, int ntiles, int ninterior,
                                                                 double* __restrict__ scale, int nb, int shift, const int* __restrict__ done) {
  __shared__ double red[32];
  const int n = blockIdx.x;
  if (done && done[n]) return;
  double v = 0.0;
  for (int t = threadIdx.x; t < ntiles; t += 128) v += partial[(size_t)n * ntiles + t];
  const double tot = block_sum(v, red, threadIdx.x, 4);
  if (threadIdx.x != 0) return;
  const double rms = sqrt(tot / (double)ninterior);
  int ex = 0;
  frexp(rms, &ex);                                   // rms = m 2^ex, m in [0.5, 1)
  if (shift) scale[n] = scale[nb + n];
  scale[nb + n] = (rms > 0.0 && isfinite(rms)) ? ldexp(1.0, ex) : 1.0;
}

}  // namespace mx
}  // namespace xee

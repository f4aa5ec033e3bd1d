// xee_krylov.cuh — BiCGStab on the block-line and two-level preconditioners (XEE_METHOD_LINE_BICGSTAB,
// XEE_METHOD_LINE2_BICGSTAB), sm_100a.
//
// Same discrete problem, same residual L psi - f (do_elliptic's nine-term sum, xtt-lib-fortran/elliptic_tools.f90:77-85)
// and the same stop rule (:193-233, stop_rule_check) as every other method, but no spectral estimate: right-preconditioned
// BiCGStab (van der Vorst 1992) on A = L with
//     line_bicgstab:   K^-1 = M^-1                   (the 32-point radial block solve of xee_sweep_line.cuh)
//     line2_bicgstab:  K^-1 = M^-1 + P Ac^-1 P^T     (plus the Galerkin coarse correction of xee_twolevel.cuh)
// It does not assume a real spectrum, which the Chebyshev methods do (DESIGN.md section 7).  Internally r = f - L x.
//
//   start    r = f - L x, r0 = r, p = r, rho = r.r
//   iterate  ph = K^-1 p,  v = L ph,  alpha = rho / (r0.v),  s = r - alpha v,  x += alpha ph
//            sh = K^-1 s,  t = L sh,  omega = (t.s) / (t.t),  x += omega sh,    r = s - omega t
//            [check]  r = f - L x: its RMS goes to finalize_check_kernel, and it replaces the recurrence residual
//            rho' = r0.r,  beta = (rho' / rho)(alpha / omega),  p = r + beta (p - omega v)
//
// Semantics:
//   * iters, max_iter and check_step count BiCGStab iterations; one iteration applies K^-1 twice and L twice.
//   * On a check iteration (iters % check_step == 0) the true residual of the current iterate is computed; its RMS over the
//     interior goes through the unchanged finalize_check_kernel, so r1, r2, converge_time, lost_rate, stall_checks,
//     r1_per_solve and the err bits mean what they mean for every method.  The true residual then replaces the
//     recurrence residual (residual replacement): without it the recurrence drifts from L x - f and 1e-12 rms(f) is out of
//     reach.  detect_explode is always on: a non-finite residual at a check sets XEE_ERR_EXPLODE and stops that solve.
//   * Breakdown (|rho'| <= 1e-30 |r0| |r|, omega = 0, or a non-finite alpha, omega or beta) restarts the solve from its
//     current iterate: r0 = r, p = r.  A bad alpha (omega) is replaced by 0 for the rest of the iteration, which leaves a
//     minimal-residual step on s (a plain step along ph), so no iteration is lost and no NaN reaches x.
//   * alpha and rho_jacobi of the solve parameters are ignored; cheb_params() reports (0, 1) and no probe runs.
//   * sweeps(psi, f, alpha, k, check_step) runs exactly k iterations with the residual replacements of a solve with that
//     check_step and no stop rule; a solve that stops at iters = n returns the same bits as sweeps(n).
//   * Every reduction is per solve in a fixed order: partial sums per (solve, 64 x 4 tile) in fp64, summed by one block per
//     solve with a fixed tree.  A solve's bits do not depend on the other solves, the batch order or sync_every.
//
// K^-1 v is the existing v5 sweep in Jacobi mode with alpha 1 from a zero field and f = v: psi' = 0 - M^-1 (L 0 - v) = M^-1 v,
// and for the two-level methods the coarse solve after it leaves c = Ac^-1 P^T v in coarse slot 1, which prolong_add_kernel
// adds to the field.  Vectors are stored in the plan's dtype (zero on the rim); every scalar, dot product and update is
// computed in fp64.
#pragma once
#include "xee_kernels.cuh"

namespace xee {
namespace kr {

constexpr int BX = kDirBX, BY = kDirBY;   // one thread per interior point, 64 x 4 points per block (= per partial-sum tile)
constexpr int NP = 2;                     // dot products per (solve, tile)

template <class T>
struct Vecs { T *r, *r0, *p, *ph, *s, *v, *t; };   // ph holds K^-1 p, then K^-1 s (sh)
struct Scal { double *rho, *alpha, *omega, *beta, *r0n; int* restart; };   // [nbatch] each; r0n = r0.r0

template <class T>
struct Args {
  const T* coe; long long coe_set_stride, nn;
  int nx, ny;
  const int* done;     // per-solve stop flags (NULL = none)
  double* part;        // [n][tile][NP] dot-product partials
  double* partial;     // [n][tile] sum of r^2 for finalize_check_kernel (residual kernel only)
  Vecs<T> v;
};

struct Point {
  int n, tile, tid; bool inside; size_t o;
};
__device__ __forceinline__ Point point(int nx, int ny) {
  Point q;
  q.n = blockIdx.z; q.tile = blockIdx.y * gridDim.x + blockIdx.x; q.tid = threadIdx.y * BX + threadIdx.x;
  const int i = 1 + blockIdx.x * BX + threadIdx.x, j = 1 + blockIdx.y * BY + threadIdx.y;
  q.inside = i < nx - 1 && j < ny - 1;
  q.o = (size_t)blockIdx.z * nx * ny + (q.inside ? (size_t)j * nx + i : (size_t)nx + 1);
  return q;
}
// (L x)(o) in fp64, slots 1..9 in the reference's order (rows j+1, j, j-1; i-1, i, i+1)
template <class T>
__device__ __forceinline__ double apply_d(const T* __restrict__ c, const T* __restrict__ x, size_t oc, size_t o, int nx, long long nn) {
  const long long off[9] = {nx - 1, nx, nx + 1, -1, 0, 1, -nx - 1, -nx, -nx + 1};
  double acc = (double)__ldg(c + oc) * (double)__ldg(x + o + off[0]);
#pragma unroll
  for (int k = 1; k < 9; ++k) acc = fma((double)__ldg(c + k * nn + oc), (double)__ldg(x + o + off[k]), acc);
  return acc;
}
template <class T>
__device__ __forceinline__ double apply_at(const Args<T>& a, const T* x, const Point& q) {
  const size_t oc = q.o - (size_t)q.n * a.nn;
  return apply_d(a.coe + (size_t)q.n * a.coe_set_stride, x, oc, q.o, a.nx, a.nn);
}
// block sums of the NP partials of this (solve, tile), fixed order; returns the second one (in thread 0)
template <class T>
__device__ __forceinline__ double store_part(const Args<T>& a, const Point& q, double d0, double d1, double* red) {
  const double s0 = block_sum(d0, red, q.tid, BX * BY / 32);
  const double s1 = block_sum(d1, red, q.tid, BX * BY / 32);
  if (q.tid == 0) {
    const int ntiles = gridDim.x * gridDim.y;
    double* out = a.part + ((size_t)q.n * ntiles + q.tile) * NP;
    out[0] = s0; out[1] = s1;
  }
  return s1;
}

// r = f - L x on the interior; partials r0.r, r.r (and r.r into `partial` for the stop rule)
template <class T>
__global__ void __launch_bounds__(BX* BY) residual_kernel(const Args<T> a, const T* __restrict__ x, const T* __restrict__ f) {
  __shared__ double red[32];
  const Point q = point(a.nx, a.ny);
  if (a.done && a.done[q.n]) return;
  double d0 = 0.0, d1 = 0.0;
  if (q.inside) {
    const T r = (T)((double)__ldg(f + q.o) - apply_at(a, x, q));
    a.v.r[q.o] = r;
    d0 = (double)a.v.r0[q.o] * (double)r; d1 = (double)r * (double)r;
  }
  const double rr = store_part(a, q, d0, d1, red);
  if (q.tid == 0) a.partial[(size_t)q.n * gridDim.x * gridDim.y + q.tile] = rr;
}
// v = L ph; partial r0.v
template <class T>
__global__ void __launch_bounds__(BX* BY) apply_dot_kernel(const Args<T> a) {
  __shared__ double red[32];
  const Point q = point(a.nx, a.ny);
  if (a.done && a.done[q.n]) return;
  double d0 = 0.0;
  if (q.inside) {
    const T v = (T)apply_at(a, a.v.ph, q);
    a.v.v[q.o] = v;
    d0 = (double)a.v.r0[q.o] * (double)v;
  }
  store_part(a, q, d0, 0.0, red);
}
// s = r - alpha v, x += alpha ph
template <class T>
__global__ void __launch_bounds__(BX* BY) s_kernel(const Args<T> a, const Scal sc, T* __restrict__ x) {
  const Point q = point(a.nx, a.ny);
  if ((a.done && a.done[q.n]) || !q.inside) return;
  const double al = sc.alpha[q.n];
  a.v.s[q.o] = (T)fma(-al, (double)a.v.v[q.o], (double)a.v.r[q.o]);
  x[q.o] = (T)fma(al, (double)a.v.ph[q.o], (double)x[q.o]);
}
// t = L sh; partials t.s, t.t
template <class T>
__global__ void __launch_bounds__(BX* BY) t_kernel(const Args<T> a) {
  __shared__ double red[32];
  const Point q = point(a.nx, a.ny);
  if (a.done && a.done[q.n]) return;
  double d0 = 0.0, d1 = 0.0;
  if (q.inside) {
    const T t = (T)apply_at(a, a.v.ph, q);
    a.v.t[q.o] = t;
    d0 = (double)t * (double)a.v.s[q.o]; d1 = (double)t * (double)t;
  }
  store_part(a, q, d0, d1, red);
}
// x += omega sh, r = s - omega t; partials r0.r, r.r
template <class T>
__global__ void __launch_bounds__(BX* BY) update_kernel(const Args<T> a, const Scal sc, T* __restrict__ x) {
  __shared__ double red[32];
  const Point q = point(a.nx, a.ny);
  if (a.done && a.done[q.n]) return;
  double d0 = 0.0, d1 = 0.0;
  if (q.inside) {
    const double om = sc.omega[q.n];
    x[q.o] = (T)fma(om, (double)a.v.ph[q.o], (double)x[q.o]);
    const T r = (T)fma(-om, (double)a.v.t[q.o], (double)a.v.s[q.o]);
    a.v.r[q.o] = r;
    d0 = (double)a.v.r0[q.o] * (double)r; d1 = (double)r * (double)r;
  }
  store_part(a, q, d0, d1, red);
}
// p = r + beta (p - omega v), or r0 = p = r on a restart
template <class T>
__global__ void __launch_bounds__(BX* BY) p_kernel(const Args<T> a, const Scal sc) {
  const Point q = point(a.nx, a.ny);
  if ((a.done && a.done[q.n]) || !q.inside) return;
  const T r = a.v.r[q.o];
  if (sc.restart[q.n]) { a.v.r0[q.o] = r; a.v.p[q.o] = r; return; }
  a.v.p[q.o] = (T)fma(sc.beta[q.n], fma(-sc.omega[q.n], (double)a.v.v[q.o], (double)a.v.p[q.o]), (double)r);
}

// The recurrence scalars of one solve from its tile partials (one block per solve, fixed summation order).
enum { STAGE_ALPHA = 0, STAGE_OMEGA = 1, STAGE_RHO = 2, STAGE_START = 3 };
static __global__ void __launch_bounds__(128) finish_kernel(Scal sc, const double* __restrict__ part, int ntiles, const int* __restrict__ done, int stage) {
  __shared__ double red[32];
  const int n = blockIdx.x;
  if (done && done[n]) return;
  double a = 0.0, b = 0.0;
  for (int t = threadIdx.x; t < ntiles; t += 128) {
    a += part[((size_t)n * ntiles + t) * NP];
    b += part[((size_t)n * ntiles + t) * NP + 1];
  }
  a = block_sum(a, red, threadIdx.x, 4);
  b = block_sum(b, red, threadIdx.x, 4);
  if (threadIdx.x != 0) return;
  if (stage == STAGE_ALPHA) {                 // a = r0.v
    const double al = sc.rho[n] / a;
    const bool bad = !isfinite(al);
    sc.alpha[n] = bad ? 0.0 : al; sc.restart[n] = bad;
  } else if (stage == STAGE_OMEGA) {          // a = t.s, b = t.t
    const double om = a / b;
    const bool bad = !isfinite(om) || om == 0.0;
    sc.omega[n] = bad ? 0.0 : om;
    if (bad) sc.restart[n] = 1;
  } else {                                    // a = r0.r, b = r.r
    bool bad = stage == STAGE_START || sc.restart[n] || !isfinite(a) || !(fabs(a) > 1e-30 * sqrt(sc.r0n[n]) * sqrt(b));
    double beta = 0.0;
    if (!bad) { beta = (a / sc.rho[n]) * (sc.alpha[n] / sc.omega[n]); bad = !isfinite(beta); }
    if (bad) { sc.rho[n] = b; sc.r0n[n] = b; sc.beta[n] = 0.0; sc.restart[n] = 1; }
    else { sc.rho[n] = a; sc.beta[n] = beta; }
  }
}

}  // namespace kr
}  // namespace xee

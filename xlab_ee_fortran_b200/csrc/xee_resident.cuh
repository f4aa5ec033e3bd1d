// xee_resident.cuh — v3 "resident" solver for single (or a few) solves: the WHOLE solve_elliptic loop
// (xtt-lib-fortran/elliptic_tools.f90:177-257) runs inside ONE cooperative kernel launch.
//
// A single 512x256 solve is 12 MiB and lives in L2; launched sweep by sweep it is bound by launch latency
// (~6 us per sweep for ~0.3 us of work).  Here the grid is decomposed into horizontal strips, one CTA per strip:
//   * the 9 coefficients, 1/(-coe5), f and the thread's own psi values stay in REGISTERS for the whole solve;
//     the strip (+ one halo row above and below) lives in shared memory;
//   * after every sweep a CTA publishes its first and last row to a double-buffered global exchange area and
//     signals its two neighbours with a release store on a per-CTA sweep counter; it waits (acquire loads) only
//     for those two neighbours - there is no grid-wide barrier on the sweep path;
//   * on check sweeps every CTA adds its sum of r^2 to a per-check slot; all CTAs then read all G partials in a
//     fixed order and run the stop-rule state machine REDUNDANTLY (bit-identical decisions, no broadcast);
//   * arithmetic is the same Rn<T>/apply9/jacobi_update code as the other sweep kernels: STRICT iterates are
//     bit-identical to the reference order.
// All CTAs must be co-resident (they wait on one another): the launch goes through
// cudaLaunchCooperativeKernel, which refuses grids that do not fit.  Every spin loop has a watchdog.
#pragma once
#include "xee_kernels.cuh"

namespace xee {
namespace res {

constexpr int NT_MAX = 1024;          // threads per CTA: 1024 x 1 point, or 512 x 2..3 points per thread
constexpr int FLAG_PAD = 32;          // ints per flag: one 128-byte line per CTA, so pollers never share a line with a writer
constexpr long long SPIN_LIMIT = 1LL << 22;   // watchdog: ~1-2 s of spinning on one flag, then the solve aborts

__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_relaxed(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acq_rel() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void st_release(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <class T>
struct ResArgs {
  const T* psi0;        // [nb][ny][nx] boundary + first guess
  const T* f;           // [nb][ny][nx]
  const T* coe;         // planar operator
  long long coe_set_stride, field_stride;
  T* out_final;         // [nb][ny][nx] last iterate
  T* out_prev;          // [nb][ny][nx] penultimate iterate (what the reference leaves in the other buffer)
  T* halo;              // [nb][2][G][2][nx] exchange rows
  int* flags;           // [nb][G][FLAG_PAD] sweeps completed by each CTA (word 0 of its own 128-byte line)
  double* partial;      // [nb][2][G] sum of r^2 per CTA, double-buffered by check parity
  int* check_cnt;       // [nb][64] monotonic arrival counter for checks (padded)
  int* abort_flag;      // [1] watchdog tripped
  int nx, ny, G;
  int max_iter, check_step, converge_time, lost_rate;
  T alpha; double rho;  // rho: Jacobi spectral radius (Chebyshev)
  const T* omega_tab;   // [kChebClamp] host-computed Chebyshev weights
  const T* r1; const T* r2;   // [nb] thresholds (HUGE when disabled)
  int detect_explode, stall_checks;
  // results
  int* iters; int* errb; T* err_now; T* ratio;
  T* trace_err; T* trace_ratio; int trace_cap;
};

// rows [r0, r1) (0-based global row indices of the interior, i.e. 1..ny-2) owned by CTA g
__host__ __device__ inline void strip_rows(int g, int G, int ny, int& r0, int& r1) {
  const int rows = ny - 2, base = rows / G, rem = rows % G;
  r0 = 1 + g * base + (g < rem ? g : rem);
  r1 = r0 + base + (g < rem ? 1 : 0);
}

template <class T, int ARITH, int MODE, int P, int NT>
__global__ void __launch_bounds__(NT, 1) solve_resident_kernel(const ResArgs<T> a) {
  using R = Rn<T>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);          // [(rows+2)][nx]: row 0 = halo below (global row r0-1)
  __shared__ double red[NT / 32];
  __shared__ double sh_tot;
  __shared__ T sh_omega;
  __shared__ int sh_abort;
  if (threadIdx.x == 0) sh_abort = 0;

  const int g = blockIdx.x, n = blockIdx.y, G = a.G, tid = threadIdx.x;
  const int nx = a.nx, ny = a.ny, w = nx - 2;
  int r0, r1;
  strip_rows(g, G, ny, r0, r1);
  const int rows = r1 - r0, npts = rows * w;
  const size_t nn = (size_t)a.field_stride;
  const T* psi0 = a.psi0 + (size_t)n * nn;
  const T* fn = a.f + (size_t)n * nn;
  const T* cn = a.coe + (size_t)n * a.coe_set_stride;
  T* halo = a.halo + (size_t)n * 2 * G * 2 * nx;
  int* flags = a.flags + (size_t)n * G * FLAG_PAD;
  double* partial = a.partial + (size_t)n * 2 * G;

  // ---- load the strip (+ halo rows, + boundary columns) and the per-point operator
  for (int q = tid; q < (rows + 2) * nx; q += NT) sp[q] = psi0[(size_t)(r0 - 1) * nx + q];
  T c[P][9], rcp[P], fv[P], x[P], xprev[P];
  int lr[P], lc[P];                               // local row (1..rows) and column (1..w) in sp
  bool act[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const int q = tid + p * NT;
    act[p] = q < npts;
    const int qq = act[p] ? q : 0;
    lr[p] = 1 + qq / w; lc[p] = 1 + qq % w;
    const size_t o = (size_t)(r0 - 1 + lr[p]) * nx + lc[p];
#pragma unroll
    for (int k = 0; k < 9; ++k) c[p][k] = cn[k * nn + o];
    rcp[p] = cn[9 * nn + o];
    fv[p] = fn[o];
    x[p] = psi0[o]; xprev[p] = x[p];
  }
  __syncthreads();

  // ---- replicated control state (elliptic_tools.f90:160-164)
  StopRule<T> rule{R::huge(), R::huge(), 0, 0, 0, 0};
  int used = 0, check_idx = 0;
  T err_now = T(0), ratio = T(0);
  const T r1v = a.r1[n], r2v = a.r2[n];
  bool stop = false, aborted = false;

  for (int cnt = 1; cnt <= a.max_iter && !stop && !aborted; ++cnt) {
    const bool check = (cnt % a.check_step) == 0;
    if (MODE == MODE_CHEBYSHEV) {
      if (tid == 0) sh_omega = a.omega_tab[(cnt < kChebClamp ? cnt : kChebClamp) - 1];
    }
    // PASS 1+2(+3)+4 fused: new value of every owned point from the OLD strip in shared memory
    T xn[P];
    double rr = 0.0;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const T* s0 = sp + (size_t)lr[p] * nx + lc[p];
      const T pp[9] = {s0[nx - 1], s0[nx], s0[nx + 1], s0[-1], s0[0], s0[1], s0[-nx - 1], s0[-nx], s0[-nx + 1]};
      T res = apply9<T, ARITH>(c[p], pp);
      res = (ARITH == XEE_ARITH_STRICT) ? R::sub(res, fv[p]) : res - fv[p];
      if (check && act[p]) rr += (double)res * (double)res;
      if (MODE == MODE_JACOBI) xn[p] = jacobi_update<T, ARITH>(pp[4], res, a.alpha, c[p][4], rcp[p]);
      else xn[p] = jacobi_update<T, ARITH>(pp[4], res, T(1), c[p][4], rcp[p]);   // x_J; combined below
    }
    __syncthreads();                                // every read of the old strip is done (and sh_omega is visible)
    if (MODE == MODE_CHEBYSHEV) {
      const T om = sh_omega;
#pragma unroll
      for (int p = 0; p < P; ++p) xn[p] = R::fma(om, xn[p] - xprev[p], xprev[p]);
    }
    const int par = cnt & 1;
    T* my_halo = halo + ((size_t)par * G + g) * 2 * nx;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      if (act[p]) {
        xprev[p] = x[p]; x[p] = xn[p];
        sp[(size_t)lr[p] * nx + lc[p]] = xn[p];
        if (lr[p] == 1) __stcg(my_halo + lc[p], xn[p]);                 // first owned row -> CTA g-1's upper halo
        if (lr[p] == rows) __stcg(my_halo + nx + lc[p], xn[p]);        // last owned row  -> CTA g+1's lower halo
      }
    }
    if (check) {   // block partial of sum r^2 (deterministic tree), published for all CTAs
      const double tot = block_sum(rr, red, tid, NT / 32);
      if (tid == 0) { __stcg(&partial[(size_t)(check_idx & 1) * G + g], tot); }
    }
    __syncthreads();                                // strip updated; exchange rows and partial issued by the CTA
    if (tid == 0) {
      // release (cumulative over the CTA's writes ordered before it by the barrier): publish sweep `cnt`
      st_release(&flags[(size_t)g * FLAG_PAD], cnt);
      if (check) atomicAdd(&a.check_cnt[(size_t)n * 64], 1);
    }
    // ---- wait for the two neighbours to have finished sweep cnt, then pull their rows into the halo rows.
    // Only the two polling threads ever touch the flags; the shared abort word is read only while spinning long.
    if (tid < 2) {
      const int nb = (tid == 0) ? g - 1 : g + 1;
      if (nb >= 0 && nb < G) {
        long long spins = 0;
        while (ld_acquire(&flags[(size_t)nb * FLAG_PAD]) < cnt) {
          if ((++spins & 0xfff) == 0 && (spins > SPIN_LIMIT || ld_acquire(a.abort_flag))) { atomicExch(a.abort_flag, 1); sh_abort = 1; break; }
        }
      }
    }
    __syncthreads();
    if (sh_abort) { aborted = true; break; }
    {   // both neighbour rows: issue every load before the first shared-memory store
      const T* lo = halo + ((size_t)par * G + (g > 0 ? g - 1 : 0)) * 2 * nx + nx;       // last row of CTA g-1
      const T* hi = halo + ((size_t)par * G + (g < G - 1 ? g + 1 : g)) * 2 * nx;        // first row of CTA g+1
      for (int i = 1 + tid; i <= w; i += NT) {
        const T vlo = (g > 0) ? __ldcg(lo + i) : sp[i];
        const T vhi = (g < G - 1) ? __ldcg(hi + i) : sp[(size_t)(rows + 1) * nx + i];
        sp[i] = vlo; sp[(size_t)(rows + 1) * nx + i] = vhi;
      }
    }
    // ---- stop rule (elliptic_tools.f90:192-234), evaluated redundantly by every CTA on identical data
    if (check) {
      if (tid == 0) {
        long long spins = 0;
        const int want = (check_idx + 1) * G;
        while (ld_acquire(&a.check_cnt[(size_t)n * 64]) < want) {
          if ((++spins & 0xfff) == 0 && (spins > SPIN_LIMIT || ld_acquire(a.abort_flag))) { atomicExch(a.abort_flag, 1); sh_abort = 1; break; }
        }
        double t = 0.0;
        for (int q = 0; q < G; ++q) t += __ldcg(&partial[(size_t)(check_idx & 1) * G + q]);
        sh_tot = t;
      }
      __syncthreads();
      if (sh_abort) { aborted = true; break; }
      const double tot = sh_tot;
      err_now = R::sqrt(R::div((T)tot, (T)((nx - 2) * (ny - 2))));                 // :199
      stop = stop_rule_check(rule, err_now, r1v, r2v, a.converge_time, a.lost_rate, a.detect_explode, a.stall_checks, ratio);
      if (g == 0 && tid == 0 && check_idx < a.trace_cap && n == 0) { a.trace_err[check_idx] = err_now; a.trace_ratio[check_idx] = ratio; }
      ratio = R::abs(ratio);
      ++check_idx;
    }
    if (cnt == a.max_iter) { stop = true; rule.errb |= XEE_ERR_OVER_MAX_ITERATION; }    // :242-244
    used = cnt;
    __syncthreads();                                // halo rows in place before the next sweep reads them
  }

  // ---- results
  T* of = a.out_final + (size_t)n * nn;
  T* op = a.out_prev + (size_t)n * nn;
#pragma unroll
  for (int p = 0; p < P; ++p)
    if (act[p]) {
      const size_t o = (size_t)(r0 - 1 + lr[p]) * nx + lc[p];
      of[o] = x[p]; op[o] = xprev[p];
    }
  if (g == 0 && tid == 0) {
    a.iters[n] = used; a.errb[n] = rule.errb | (aborted ? 0x100 : 0); a.err_now[n] = err_now; a.ratio[n] = ratio;
  }
}

}  // namespace res
}  // namespace xee

// xee_sweep_line.cuh — v5 sweep kernel for sm_100a: BLOCK-LINE relaxation along the radius.
//
// Same discrete problem, same residual r = L psi - f (do_elliptic's nine-term sum, xtt-lib-fortran/
// elliptic_tools.f90:77-85) and the same stop rule (:193-233) as solve_elliptic, but the correction is not the
// reference's point-wise r / (-coe5) (:238): the radial line is cut into blocks of 32 points (global index aligned)
// and every block's tridiagonal system  coe4 z(i-1) + coe5 z(i) + coe6 z(i+1) = r(i)  is solved exactly,
// psi' = psi - alpha z.  On the secondary-circulation operator the radial coupling carries ~97 % of the diagonal
// (dr >> dz after the 1/(rho r) scaling), so this block-Jacobi splitting has a ~18x larger spectral gap than point
// Jacobi and its Chebyshev acceleration needs ~4x fewer sweeps for the same residual tolerance.
// XEE_METHOD_LINE_JACOBI / XEE_METHOD_LINE_CHEBYSHEV; FAST arithmetic.  Shared operator (map: constants reloaded once
// per chunk of solves) or one operator per solve (time series: every work unit is one (tile, solve) and reloads them).
//
// The block solve is split over 4 threads of a warp (partitioned / SPIKE form, everything operator-dependent
// precomputed once per operator by line_factor_kernel):
//   * thread = 8 consecutive radial points of one row.  It solves its own 8-point segment with the Thomas algorithm
//     in registers (z0 = M_t^-1 r), exchanges the two end values of z0 with the 3 other threads of the block by
//     two butterfly shuffles, forms the true values of its neighbours' end points from 2 x 8 precomputed reduced-
//     system coefficients, and subtracts the two precomputed spike vectors:  z = z0 - v b(t-1) - w a(t+1);
//   * the 9 coefficients of its points (144 registers) stay in registers for the whole chunk of solves, the 4 x 8 factors
//     (m, u, v, w) and the 16 reduced coefficients in thread-private shared-memory cells.  The coupling data (v, w
//     and the reduced coefficients) are stored in FLOAT: the local Thomas solve is exact in working precision, the
//     coupling correction carries a 6e-8 relative perturbation.  That only perturbs the (fixed, linear) approximate
//     inverse that multiplies the residual — the fixed point L psi = f and the residual-based stop rule are untouched —
//     and it halves the shared-memory traffic and the registers of the coupling step.
//
// Data movement (one sweep per pass, HBM-bound like the v2 kernel):
//   * warp = 32 columns x 8 rows (lane = segment-in-block * 8 + row).  TMA boxes are 70 (psi, with halo) and 66
//     (f, psi_{k-1}) elements wide, i.e. an ODD number of 16-byte chunks per shared-memory row, so the 128-bit loads of
//     8 lanes with the same columns and consecutive rows hit distinct banks without any swizzle;
//   * TWO persistent CTAs of 128 threads per SM (255 registers per thread: the register file is full), tiles of
//     64 x 16 points, a 2-stage TMA ring per CTA (80 KB of shared memory each), one named barrier per (tile, solve) to
//     hand the stage back; while one CTA reloads the operator of its next work unit or waits at its barrier the other
//     one computes.  Results are staged in shared memory (128-bit stores) and leave with one 4-D TMA store per
//     (tile, solve) (tensor map = column in tile, tile column, row, solve: the pad columns of the last tile are dropped by
//     the bounds check); a.tstore == 0 keeps the 128-bit global stores of round 1 (shapes the map cannot describe);
//   * the operator and the factors are repacked once per operator in tile/thread order (line_pack_kernel), so the
//     per-unit reload of a thread's constants is fully coalesced 128-bit loads (2-3 us per unit instead of 10).
// TWO = true is the two-level variant (xee_twolevel.cuh): the iterate is stored as (field y, coarse vector c) with
// psi = y + P c; the 3 x 8 coarse patch of a tile arrives with its stage, the correction is added to the values as they are
// read, and the restriction moments of the new residual leave as 32 doubles per (tile, solve).  The same reducer warp that
// forms them also sums r^2 over the tile on check sweeps, so a check sweep adds no reduction before the CTA barrier.
// Measured on B200 (512 solves, 512x256, fp64, Chebyshev, ncu, profiles/r02_*): one level 355 us per sweep = 6.05 TB/s
// algorithmic (97 % of the measured copy peak) with a shared operator; two-level 585 us (instruction/latency bound).
#pragma once
#include <cuda.h>

#include "xee_sweep_tma.cuh"

namespace xee {

enum { MODE_LINE_JACOBI = 3, MODE_LINE_CHEBYSHEV = 4 };

namespace ln {
constexpr int SEG = 8;             // points per thread
constexpr int BLK = 4;             // threads per block of the line relaxation: blocks of SEG * BLK = 32 radial points
#ifndef XEE_LINE_TH
#define XEE_LINE_TH 16
#endif
constexpr int TW = 64, TH = XEE_LINE_TH;    // tile (grid points); TH = 16 runs two CTAs of 128 threads per SM
constexpr int CTAS_PER_SM = 32 / TH;
constexpr int NSEG = TW / SEG;     // 8 warps
constexpr int NT = NSEG * TH;      // 256 threads
#ifndef XEE_LINE_NSTAGE
#define XEE_LINE_NSTAGE 2
#endif
constexpr int NSTAGE = XEE_LINE_NSTAGE;
template <class T> struct Cfg {
  static constexpr int ES = (int)sizeof(T);
  static constexpr int V = 16 / ES;                 // elements per 16-byte chunk
  static constexpr int NV = SEG / V;                // chunks per segment
  static constexpr int XW = TW + 3 * V;             // psi box: columns i0-V .. i0+TW+2V-1, odd number of chunks
  static constexpr int FW = TW + V;                 // f / psi_{k-1} box: columns i0 .. i0+TW+V-1, odd number of chunks
  static constexpr int XP = XW * ES, FP = FW * ES;  // shared-memory row pitches (bytes)
  static constexpr int X_RAW = XP * (TH + 2), F_RAW = FP * TH;
  static constexpr int X_BYTES = (X_RAW + 127) / 128 * 128, F_BYTES = (F_RAW + 127) / 128 * 128;
  static constexpr int STAGE_BYTES = X_BYTES + 2 * F_BYTES;
  // thread-private cells of the current tile's factor planes: m, u in working precision (pitch FP), then four float planes
  // (8 floats = 2 chunks per thread, pitch AP = 17 chunks): the spikes v, w and the reduced-system rows cB, cA
  static constexpr int AP = (TW + 4) * 4, A_BYTES = AP * TH;
  static constexpr int FAC_BYTES = 2 * F_BYTES + 4 * A_BYTES;
  // result staging for the TMA store (two buffers, same [TH][FW] layout as the f box: odd chunk pitch, conflict-free STS.128)
  static constexpr int OUT_BYTES = F_BYTES, NOUT = 2;
  // two-level method: per-thread restriction moments (S0, S1) of the residual, [TH rows][NSEG segments] double2, then the
  // thread's sum of r^2 (CHECK), [NT threads] double; two buffers
  static constexpr int RES_BYTES = TH * NSEG * 16 + NT * 8;
  static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + FAC_BYTES + NOUT * OUT_BYTES;
  // two-level method: every stage also carries two 3 x 8 patches of coarse-correction values (current / previous iterate)
  static constexpr int CP_RAW = 3 * 8 * 8, CP_BYTES = 2 * 256;
  static constexpr int SMEM_BYTES_TWO = SMEM_BYTES + NSTAGE * CP_BYTES + 2 * RES_BYTES;
  static_assert((XW / V) % 2 == 1 && (FW / V) % 2 == 1, "row pitches must be an odd number of 16-byte chunks");
};
// TMA store of one [1][TH][1][FW] box (4-D map: column-in-tile, tile column, row, solve) from shared memory; bulk async-group
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];" ::"l"(map), "r"(c0), "r"(c1),
               "r"(c2), "r"(c3), "r"(smem_src)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void cta_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); }

// 16-byte shared-memory load into V consecutive elements.
__device__ __forceinline__ void lds16(uint32_t addr, double* v) {
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr));
}
__device__ __forceinline__ void lds16(uint32_t addr, float* v) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}
__device__ __forceinline__ void ldg16(const double* p, double* v) {
  const double2 t = __ldg(reinterpret_cast<const double2*>(p)); v[0] = t.x; v[1] = t.y;
}
__device__ __forceinline__ void ldg16(const float* p, float* v) {
  const float4 t = __ldg(reinterpret_cast<const float4*>(p)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void sts16(uint32_t addr, const double* v) { asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(v[0]), "d"(v[1])); }
__device__ __forceinline__ void sts16(uint32_t addr, const float* v) { asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3])); }
__device__ __forceinline__ void stg16(double* p, const double* v) { *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]); }
__device__ __forceinline__ void stg16(float* p, const float* v) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }

// SEG + 2 consecutive elements of one shared-memory row: [0] = left neighbour of the segment, [1..SEG] the segment,
// [SEG+1] = right neighbour.  `seg_addr` = address of the segment's first element (16-byte aligned).
template <class T> __device__ __forceinline__ void load_row(uint32_t seg_addr, T (&w)[SEG + 2]) {
  constexpr int V = Cfg<T>::V, NV = Cfg<T>::NV;
  T t[V];
  lds16(seg_addr - 16u, t); w[0] = t[V - 1];
#pragma unroll
  for (int q = 0; q < NV; ++q) {
    lds16(seg_addr + 16u * q, t);
#pragma unroll
    for (int e = 0; e < V; ++e) w[1 + q * V + e] = t[e];
  }
  lds16(seg_addr + 16u * NV, t); w[SEG + 1] = t[0];
}
template <class T> __device__ __forceinline__ void load_seg(uint32_t seg_addr, T (&w)[SEG]) {
  constexpr int V = Cfg<T>::V, NV = Cfg<T>::NV;
#pragma unroll
  for (int q = 0; q < NV; ++q) lds16(seg_addr + 16u * q, &w[q * V]);
}
// thread -> (segment column, row) of the tile: warp = (32-column half, 8-row group), lane = segment-in-block * 8 + row,
// so the 4 threads of a block sit in one warp (lanes l, l^8, l^16, l^24) and 8 consecutive lanes read consecutive rows.
__device__ __forceinline__ int seg_of(int tid) { return ((tid >> 5) & 1) * BLK + ((tid >> 3) & 3); }
__device__ __forceinline__ int row_of(int tid) { return (tid >> 6) * 8 + (tid & 7); }
__device__ __forceinline__ double shfl_xor(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ float shfl_xor(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
}  // namespace ln

constexpr int kLineFacPlanes = 6;
// Everything the block solve needs from an operator, once per operator: fac[set][6][ny][nx] =
//   0: m(i) = 1 / (coe5(i) - lo(i) u(i-1))   1: u(i) = up(i) m(i)      Thomas factors of the 8-point segments
//      (lo = coe4 except at a segment start, up = coe6 except at a segment end; 0 on boundary points, which therefore
//      get a zero correction),
//   2: v = M_t^-1 (coe4(first) e_first)      3: w = M_t^-1 (coe6(last) e_last)      spike vectors of segment t,
//   (planes 2..5 hold float-representable values: the sweep kernel keeps them in float)
//   4: cB[k]   5: cA[k]   (8 values per segment)  rows of the inverse of the 8 x 8 reduced system that give b(t-1), the
//      true last value of the segment to the left, and a(t+1), the true first value of the segment to the right, from
//      the end values of the four local solutions in the order a thread holds them after the two butterfly exchanges:
//      [own first, own last, those of t^1, of t^2, of t^3].
// One thread per (block of 32 points, row, operator set).
template <class T>
__global__ void line_factor_kernel(const T* __restrict__ coe, T* __restrict__ fac, int nx, int ny) {
  constexpr int S = ln::SEG, B = ln::BLK, NB = S * B;
  const int blk = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  const int ib = blk * NB;
  if (ib >= nx) return;
  const size_t nn = (size_t)nx * ny;
  coe += (size_t)blockIdx.z * kPlanes * nn;            // operator set (one per solve for a time series)
  fac += (size_t)blockIdx.z * kLineFacPlanes * nn;
  T m[NB], u[NB], v[NB], w[NB];
  for (int t = 0; t < B; ++t) {
    T c4f = T(0), c6l = T(0);
    T u_prev = T(0);
    for (int e = 0; e < S; ++e) {
      const int q = t * S + e, i = ib + q;
      const bool interior = i > 0 && i < nx - 1 && j > 0 && j < ny - 1;
      m[q] = T(0); u[q] = T(0);
      if (interior) {
        const size_t o = (size_t)j * nx + i;
        const T lo = e == 0 ? T(0) : coe[3 * nn + o];
        const T up = e == S - 1 ? T(0) : coe[5 * nn + o];
        m[q] = T(1) / (coe[4 * nn + o] - lo * u_prev);
        u[q] = up * m[q];
        if (e == 0 && t > 0) c4f = coe[3 * nn + o];
        if (e == S - 1 && t < B - 1) c6l = coe[5 * nn + o];
      }
      u_prev = u[q];
    }
    // spikes: the same forward / backward recurrences as the sweep kernel, right-hand sides c4f e_0 and c6l e_{S-1}
    T y = T(0);
    for (int e = 0; e < S; ++e) {
      const int q = t * S + e, i = ib + q;
      const T c4 = (e > 0 && i < nx && m[q] != T(0)) ? coe[3 * nn + (size_t)j * nx + i] : T(0);
      y = ((e == 0 ? c4f : T(0)) - c4 * y) * m[q];
      v[q] = y;
    }
    for (int e = S - 2; e >= 0; --e) v[t * S + e] -= u[t * S + e] * v[t * S + e + 1];
    for (int e = 0; e < S; ++e) w[t * S + e] = T(0);
    w[t * S + S - 1] = c6l * m[t * S + S - 1];
    for (int e = S - 2; e >= 0; --e) w[t * S + e] = -u[t * S + e] * w[t * S + e + 1];
  }
  // reduced system R (a_0, b_0, a_1, b_1, ...) = (first, last of the local solutions), then its inverse (Gauss-Jordan;
  // R = I + off-diagonal entries of magnitude < 1 for a diagonally dominant operator)
  constexpr int NR = 2 * B;
  double R[NR][NR], Ri[NR][NR];
  for (int p = 0; p < NR; ++p)
    for (int q = 0; q < NR; ++q) { R[p][q] = p == q ? 1.0 : 0.0; Ri[p][q] = p == q ? 1.0 : 0.0; }
  for (int t = 0; t < B; ++t) {
    if (t > 0) { R[2 * t][2 * (t - 1) + 1] = (double)v[t * S]; R[2 * t + 1][2 * (t - 1) + 1] = (double)v[t * S + S - 1]; }
    if (t < B - 1) { R[2 * t][2 * (t + 1)] = (double)w[t * S]; R[2 * t + 1][2 * (t + 1)] = (double)w[t * S + S - 1]; }
  }
  for (int p = 0; p < NR; ++p) {
    const double piv = 1.0 / R[p][p];
    for (int q = 0; q < NR; ++q) { R[p][q] *= piv; Ri[p][q] *= piv; }
    for (int o = 0; o < NR; ++o) {
      if (o == p) continue;
      const double fct = R[o][p];
      if (fct == 0.0) continue;
      for (int q = 0; q < NR; ++q) { R[o][q] -= fct * R[p][q]; Ri[o][q] -= fct * Ri[p][q]; }
    }
  }
  for (int t = 0; t < B; ++t) {
    for (int e = 0; e < S; ++e) {
      const int q = t * S + e, i = ib + q;
      if (i >= nx) continue;
      const size_t o = (size_t)j * nx + i;
      fac[o] = m[q]; fac[nn + o] = u[q]; fac[2 * nn + o] = (T)(float)v[q]; fac[3 * nn + o] = (T)(float)w[q];
      const int src = t ^ (e >> 1), col = 2 * src + (e & 1);        // gathered order: own, t^1, t^2, t^3
      fac[4 * nn + o] = t > 0 ? (T)(float)Ri[2 * (t - 1) + 1][col] : T(0);
      fac[5 * nn + o] = t < B - 1 ? (T)(float)Ri[2 * (t + 1)][col] : T(0);
    }
  }
}

// Operator + factors repacked per tile in the order the sweep kernel's threads read them: 11 planes in working precision
// pack[tile][plane 0..10][chunk q][thread][V] (coe1..coe9, m, u), then 4 float planes [plane][chunk 0..1][thread][4]
// (v, w, cB, cA); zeros outside the field.  A warp's 128-bit load of (plane, chunk) is one contiguous 512-byte run
// instead of 32 rows 4 KB apart.
template <class T> __host__ __device__ constexpr size_t line_pack_tile_bytes() {
  return (size_t)(11 * ln::Cfg<T>::NV + 4 * 2) * ln::NT * 16;
}
template <class T>
__global__ void __launch_bounds__(ln::NT) line_pack_kernel(const T* __restrict__ coe, const T* __restrict__ fac,
                                                           unsigned char* __restrict__ pack, int nx, int ny, int tiles_x) {
  using C = ln::Cfg<T>;
  const int tile = blockIdx.x, tid = threadIdx.x;
  const int sg = ln::seg_of(tid), r = ln::row_of(tid);
  const int gi = (tile % tiles_x) * ln::TW + ln::SEG * sg, gj = (tile / tiles_x) * ln::TH + r;
  const size_t nn = (size_t)nx * ny;
  coe += (size_t)blockIdx.y * kPlanes * nn;
  fac += (size_t)blockIdx.y * kLineFacPlanes * nn;
  unsigned char* base = pack + ((size_t)blockIdx.y * gridDim.x + tile) * line_pack_tile_bytes<T>();
  T* out = reinterpret_cast<T*>(base);
  float* aux = reinterpret_cast<float*>(base + (size_t)11 * C::NV * ln::NT * 16);
  for (int k = 0; k < 15; ++k) {
    const T* src = k < 9 ? coe + k * nn : fac + (k - 9) * nn;
    for (int e = 0; e < ln::SEG; ++e) {
      const bool in = gj < ny && gi + e < nx;
      const T val = in ? src[(size_t)gj * nx + gi + e] : T(0);
      if (k < 11) out[((size_t)(k * C::NV + e / C::V) * ln::NT + tid) * C::V + e % C::V] = val;
      else aux[((size_t)((k - 11) * 2 + e / 4) * ln::NT + tid) * 4 + e % 4] = (float)val;
    }
  }
}

template <class T>
struct LineArgs {
  const unsigned char* pack;   // operator + factors in tile/thread order (line_pack_kernel)
  long long pack_set_stride;   // bytes between the packs of consecutive solves; 0 = one shared operator
  T* dst;                  // psi_{k+1} (holds psi_{k-1} on entry: read through map_xm at the own cells only)
  long long field_stride;  // nx*ny
  int nx, ny, nbatch;
  T alpha, omega;
  const T* rho_ps;         // per-solve spectral radius (probe): omega computed in-kernel from cheb_k
  int cheb_k;
  const int* done;
  double* partial;         // [n][ntiles] sum of r^2 (CHECK)
  int tiles_x, tiles_y, nchunks, chunk;
  int tstore;              // 1: results leave through shared memory + TMA stores (needs nx % TW == 0); 0: 128-bit global stores
  T gamma;                 // Chebyshev: psi+ = omega ((psi - gamma z) - psi-) + psi-   (1 for the one-level methods)
  double* cpart;           // TWO: [n][ntiles][32] restriction of the residual to the coarse grid, per tile (see xee_twolevel.cuh)
  int cv_cur_z, cv_prev_z; // TWO: first index (slot * nbatch) of the coarse corrections of the iterate read / of the previous one in map_cv
};

// TWO = two-level method (xee_twolevel.cuh).  The iterates live in global memory WITHOUT their latest coarse-grid correction:
// the field y_k is stored, the iterate is psi_k = y_k + P c_k with c_k a small coarse vector per solve (written by the coarse
// solve that follows every sweep).  The kernel adds P c_k on the fly to everything it reads (psi tile with halo: bilinear,
// linear along the thread's 8 points; likewise P c_{k-1} to psi_{k-1}) - a 3 x 8 patch of coarse values per iterate travels
// with the TMA stage - so the coarse correction costs no pass over the fields.  The kernel also restricts the residual r = L psi - f of its tile to the coarse
// grid (bilinear weights, nodes every 16 points in r and z; tiles are TH = 16 rows = one coarse cell high).  Every thread
// forms the two moments S0 = sum r(e), S1 = sum e r(e) of its 8-point segment; one warp per (tile, solve), rotating, reduces
// them over the 16 rows with the weights (1 - j/16) and j/16 and writes 32 doubles: [4 kinds][8 segments].
template <class T, bool CHEB, bool CHECK, bool TWO = false>
__global__ void __launch_bounds__(ln::NT, ln::CTAS_PER_SM)
    sweep_line_kernel(const __grid_constant__ LineArgs<T> a, const __grid_constant__ CUtensorMap map_x,
                      const __grid_constant__ CUtensorMap map_xm, const __grid_constant__ CUtensorMap map_f,
                      const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_cv) {
  using namespace ln;
  using tma::mbar_init; using tma::mbar_expect_tx; using tma::mbar_wait; using tma::tma_load_3d;
  using C = Cfg<T>;
  constexpr int V = C::V, NV = C::NV;
  constexpr int SB = C::STAGE_BYTES + (TWO ? C::CP_BYTES : 0);     // stage stride
  constexpr int AFTER = NSTAGE * SB;                                // factor cells, result staging, restriction moments follow
  constexpr int RES_OFS = AFTER + C::FAC_BYTES + C::NOUT * C::OUT_BYTES;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t full_bar[NSTAGE];
  __shared__ double red[2][NT / 32];          // per-warp sums of r^2 (CHECK without TWO), double-buffered by iteration parity
  __shared__ uint32_t sdone[kDoneWords];   // stop flags of the batch as a bit mask: no global load per (tile, solve)

  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) mbar_init(&full_bar[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const bool done_in_smem = stage_done_flags(a.done, a.nbatch, sdone, tid, NT);
  __syncthreads();
  auto is_done = [&](int n) -> bool {
    if (a.done == nullptr) return false;
    return done_in_smem ? ((sdone[n >> 5] >> (n & 31)) & 1u) != 0u : a.done[n] != 0;
  };

  const int ntiles = a.tiles_x * a.tiles_y;
  const int nunits = ntiles * a.nchunks;
  const size_t nn = (size_t)a.field_stride;

  // ---- prefetch cursor (thread 0): the same (unit, solve) sequence as the consumers, NSTAGE items ahead
  // (the unit -> (chunk, tile row, tile column) divisions happen once per unit: thread 0's warp is the one the others wait for)
  int pu = (int)blockIdx.x - (int)gridDim.x, pn = 0, pn1 = 0, ptx = 0, pty = 0;
  uint32_t issued = 0;
  auto issue_next = [&]() {
    for (;;) {
      if (pn >= pn1) {                         // next unit of this CTA
        if (pu < nunits) pu += gridDim.x;
        if (pu >= nunits) return false;
        const int ch = pu / ntiles, tile = pu - ch * ntiles;
        pn = ch * a.chunk; pn1 = min(pn + a.chunk, a.nbatch);
        pty = tile / a.tiles_x; ptx = tile - pty * a.tiles_x;
        continue;
      }
      const int n = pn++;
      if (is_done(n)) continue;
      const int i0 = ptx * TW, j0 = pty * TH;
      const int s = issued % NSTAGE;
      unsigned char* st = smem_raw + (size_t)s * SB;
      mbar_expect_tx(&full_bar[s], (uint32_t)(C::X_RAW + (CHEB ? 2 : 1) * C::F_RAW + (TWO ? (CHEB ? 2 : 1) * C::CP_RAW : 0)));
      if (TWO) {   // coarse patches: nodes 4 tx - 1 .. 4 tx + 6 (node p sits in column p + 1), coarse rows ty - 1 .. ty + 1
        tma_load_3d(st + C::STAGE_BYTES, &map_cv, 4 * ptx, pty - 1, a.cv_cur_z + n, &full_bar[s]);
        if (CHEB) tma_load_3d(st + C::STAGE_BYTES + 256, &map_cv, 4 * ptx, pty - 1, a.cv_prev_z + n, &full_bar[s]);
      }
      tma_load_3d(st, &map_x, i0 - V, j0 - 1, n, &full_bar[s]);
      tma_load_3d(st + C::X_BYTES, &map_f, i0, j0, n, &full_bar[s]);
      if (CHEB) tma_load_3d(st + C::X_BYTES + C::F_BYTES, &map_xm, i0, j0, n, &full_bar[s]);
      ++issued;
      return true;
    }
  };
  if (tid == 0)
    for (int q = 0; q < NSTAGE; ++q)
      if (!issue_next()) break;

  const int sg = seg_of(tid);       // segment column of the tile (0..7)
  const int r = row_of(tid);        // row of the tile (0..31)
  const uint32_t sm0 = tma::smem_u32(smem_raw);
  const uint32_t xofs = (uint32_t)((r + 1) * C::XP + (V + SEG * sg) * C::ES);   // own segment in the psi box
  const uint32_t fofs = (uint32_t)(C::X_BYTES + r * C::FP + SEG * sg * C::ES);  // ... in the f box
  const uint32_t faca = sm0 + (uint32_t)(AFTER + r * C::FP + SEG * sg * C::ES);   // own cells of the factor planes m, u
  const uint32_t auxa = sm0 + (uint32_t)(AFTER + 2 * C::F_BYTES + r * C::AP + SEG * sg * 4);   // ... v, w (float)
  const uint32_t outa = sm0 + (uint32_t)(AFTER + C::FAC_BYTES + r * C::FP + SEG * sg * C::ES);  // own cells of result buffer 0
  const bool tstore = a.tstore != 0;
  const uint32_t resa = sm0 + (uint32_t)RES_OFS;            // TWO: restriction moments (two buffers)
  uint32_t it = 0;

  for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
    const int tile = u % ntiles, ch = u / ntiles;
    const int i0 = (tile % a.tiles_x) * TW, j0 = (tile / a.tiles_x) * TH;
    const int n0 = ch * a.chunk, n1 = min(n0 + a.chunk, a.nbatch);
    const int gi = i0 + SEG * sg, gj = j0 + r;
    const bool row_in = gj < a.ny;
    const bool seg_full = row_in && gi + SEG <= a.nx;      // whole segment inside the field: vector accesses
    const long long gofs = (long long)gj * a.nx + gi;
    unsigned inb = 0;   // bit e: point (gi+e, gj) is a domain-interior point (residual norm)
#pragma unroll
    for (int e = 0; e < SEG; ++e)
      if (gi + e >= 1 && gi + e < a.nx - 1 && gj >= 1 && gj < a.ny - 1) inb |= 1u << e;
    // TWO: where the coarse correction applies.  It vanishes by itself on the bottom row and the first column (zero rim of
    // the coarse values); on the top row (j = ny-1) and the last column (i = nx-1) it must be switched off: Dirichlet values.
    // cmask bit k: column gi - 1 + k (k = 0..9: left neighbour, the 8 points, right neighbour) is not the last column.
    unsigned cmask = 0x3ffu;
    double fu = 1.0, fm = 1.0;      // row factors of the stencil rows j+1 and j
    if (TWO) {
#pragma unroll
      for (int k = 0; k < SEG + 2; ++k)
        if (gi - 1 + k >= a.nx - 1) cmask &= ~(1u << k);
      if (gj + 1 >= a.ny - 1) fu = 0.0;
      if (gj >= a.ny - 1) fm = 0.0;
    }
    // stop flags of this unit's solves (chunk <= 32) as one register mask: no shared-memory load per (tile, solve)
    uint32_t umask = 0;
    if (a.done != nullptr) {
      if (done_in_smem) {
        const int w0 = n0 >> 5;
        umask = __funnelshift_r(sdone[w0], w0 + 1 < kDoneWords ? sdone[w0 + 1] : 0u, n0 & 31);
      } else {
        for (int n = n0; n < n1; ++n) umask |= (a.done[n] != 0 ? 1u : 0u) << (n - n0);
      }
    }
    {
      const uint32_t full = n1 - n0 >= 32 ? 0xffffffffu : (1u << (n1 - n0)) - 1u;
      if ((umask & full) == full) continue;   // every solve of the unit has stopped: skip it before reloading the operator
    }
    // the 9 coefficients of the thread's points stay in registers for the whole chunk; the factors m, u, v, w and the
    // reduced-system rows cB, cA go to thread-private cells of shared memory (read back by the same thread only).  cB and cA
    // in registers made ptxas keep them as 16 doubles, 10 of which it spilled to local memory in the two-level variants.
    T cf[9][SEG];
    {
      // one operator per solve: the host makes every unit one solve (chunk = 1), so n0 names the operator set
      const unsigned char* pb = a.pack + (size_t)n0 * a.pack_set_stride + (size_t)tile * line_pack_tile_bytes<T>();
      const T* pk = reinterpret_cast<const T*>(pb) + (size_t)tid * V;
      const float* pa = reinterpret_cast<const float*>(pb + (size_t)11 * NV * NT * 16) + (size_t)tid * 4;
#pragma unroll
      for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int q = 0; q < NV; ++q) ldg16(pk + (size_t)(k * NV + q) * NT * V, &cf[k][q * V]);
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int q = 0; q < NV; ++q) {
          T t[V];
          ldg16(pk + (size_t)((9 + k) * NV + q) * NT * V, t); sts16(faca + k * C::F_BYTES + 16u * q, t);
        }
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float t[4];
          ldg16(pa + (size_t)(k * 2 + q) * NT * 4, t); sts16(auxa + k * C::A_BYTES + 16u * q, t);
        }
    }
    for (int n = n0; n < n1; ++n) {
      if ((umask >> (n - n0)) & 1u) continue;
      const uint32_t s = it % NSTAGE;
      mbar_wait(&full_bar[s], (it / NSTAGE) & 1);
      const uint32_t sb = sm0 + s * SB;
      const uint32_t xa = sb + xofs;
      // ---- residual: the nine-term sum in the reference's order (rows j+1, j, j-1; i-1, i, i+1), minus f
      T acc[SEG];
      // TWO: coarse values of this thread's cell: patch columns cl, cl+1, cl+2 = nodes p-1, p, p+1 (p = left node of the cell
      // of the segment), patch rows 0..2 = coarse rows ty-1, ty, ty+1.  Along z the correction is linear in the local row
      // offset zo in [0, 16]; the halo row zo = -1 lies in the cell below.
      const double* pc = reinterpret_cast<const double*>(smem_raw + (size_t)s * SB + C::STAGE_BYTES) + (sg >> 1);
      auto add_corr = [&](T (&w)[SEG + 2], const double* pq, int zo, double rowf) {
        // node values of the row: V_m = c1_m + slope_m zo, slope towards the upper coarse row (zo >= 0) or the lower one (zo = -1)
        double vv[3];
#pragma unroll
        for (int m = 0; m < 3; ++m) {
          const double c1 = pq[8 + m];
          const double sl = zo >= 0 ? (pq[16 + m] - c1) : (c1 - pq[m]);
          vv[m] = fma(sl, (double)zo * (1.0 / 16.0), c1) * rowf;
        }
        const double S = (vv[2] - vv[1]) * (1.0 / 16.0);
        const double b0 = fma(S, (double)(SEG * (sg & 1)), vv[1]);              // value at the segment's first point
        const double left = (sg & 1) ? b0 - S : fma(vv[1] - vv[0], 15.0 / 16.0, vv[0]);   // point before it: same cell / the cell to the left
        if (cmask == 0x3ffu) {
          w[0] += (T)left;
#pragma unroll
          for (int k = 1; k < SEG + 2; ++k) w[k] += (T)fma(S, (double)(k - 1), b0);
        } else {
          if (cmask & 1u) w[0] += (T)left;
#pragma unroll
          for (int k = 1; k < SEG + 2; ++k)
            if ((cmask >> k) & 1u) w[k] += (T)fma(S, (double)(k - 1), b0);
        }
      };
      {
        T w[SEG + 2];
        load_row<T>(xa + C::XP, w);
        if (TWO) add_corr(w, pc, r + 1, fu);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = cf[0][e] * w[e];
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[1][e], w[e + 1], acc[e]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[2][e], w[e + 2], acc[e]);
        load_row<T>(xa, w);
        if (TWO) add_corr(w, pc, r, fm);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[3][e], w[e], acc[e]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[4][e], w[e + 1], acc[e]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[5][e], w[e + 2], acc[e]);
        load_row<T>(xa - C::XP, w);
        if (TWO) add_corr(w, pc, r - 1, 1.0);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[6][e], w[e], acc[e]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[7][e], w[e + 1], acc[e]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(cf[8][e], w[e + 2], acc[e]);
      }
      {
        T fv[SEG];
        load_seg<T>(sb + fofs, fv);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = acc[e] - fv[e];
      }
      double rr = 0.0;
      if (CHECK) {
#pragma unroll
        for (int e = 0; e < SEG; ++e)
          if ((inb >> e) & 1u) rr += (double)acc[e] * (double)acc[e];
      }
      if (TWO) {   // restriction moments of the residual over the thread's interior points
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int e = 0; e < SEG; ++e)
          if ((inb >> e) & 1u) { s0 += (double)acc[e]; s1 = fma((double)e, (double)acc[e], s1); }
        const double mom[2] = {s0, s1};
        sts16(resa + (it & 1u) * C::RES_BYTES + (uint32_t)((r * NSEG + sg) * 16), mom);
        if (CHECK)   // the tile's sum of r^2 is formed by the reducer warp too: no reduction before the barrier
          asm volatile("st.shared.f64 [%0], %1;" ::"r"(resa + (it & 1u) * C::RES_BYTES + (uint32_t)(TH * NSEG * 16 + tid * 8)), "d"(rr));
      }
      // ---- Thomas solve of the segment: forward  y(i) = (r(i) - coe4(i) y(i-1)) m(i),  back  z(i) = y(i) - u(i) z(i+1)
      {
        T mf[SEG];
        load_seg<T>(faca, mf);
        acc[0] = acc[0] * mf[0];
#pragma unroll
        for (int e = 1; e < SEG; ++e) acc[e] = Rn<T>::fma(-cf[3][e], acc[e - 1], acc[e]) * mf[e];
      }
      {
        T uf[SEG];
        load_seg<T>(faca + C::F_BYTES, uf);
#pragma unroll
        for (int e = SEG - 2; e >= 0; --e) acc[e] = Rn<T>::fma(-uf[e], acc[e + 1], acc[e]);
      }
      // ---- couple the 4 segments of the 32-point block: end values of the local solutions around the block (two
      // butterfly exchanges), true neighbour end values from the reduced system, minus the spikes
      {
        T g[2 * BLK];
        g[0] = acc[0]; g[1] = acc[SEG - 1];
        g[2] = shfl_xor(g[0], 8); g[3] = shfl_xor(g[1], 8);
#pragma unroll
        for (int k = 0; k < 4; ++k) g[4 + k] = shfl_xor(g[k], 16);
        float cB[SEG], cA[SEG];
        lds16(auxa + 2 * C::A_BYTES, &cB[0]); lds16(auxa + 2 * C::A_BYTES + 16u, &cB[4]);
        lds16(auxa + 3 * C::A_BYTES, &cA[0]); lds16(auxa + 3 * C::A_BYTES + 16u, &cA[4]);
        T bl = (T)cB[0] * g[0], ar = (T)cA[0] * g[0];
#pragma unroll
        for (int k = 1; k < 2 * BLK; ++k) { bl = Rn<T>::fma((T)cB[k], g[k], bl); ar = Rn<T>::fma((T)cA[k], g[k], ar); }
        float vf[SEG];
        lds16(auxa, &vf[0]); lds16(auxa + 16u, &vf[4]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(-(T)vf[e], bl, acc[e]);
        lds16(auxa + C::A_BYTES, &vf[0]); lds16(auxa + C::A_BYTES + 16u, &vf[4]);
#pragma unroll
        for (int e = 0; e < SEG; ++e) acc[e] = Rn<T>::fma(-(T)vf[e], ar, acc[e]);
      }
      // ---- update
      T out[SEG];
      {
        // TWO: the coarse correction at the thread's own points (interior points only), for the current and the previous iterate
        auto own_corr = [&](T (&v)[SEG], const double* pq) {
          const double tz = (double)r * (1.0 / 16.0);
          const double vl = fma(pq[17] - pq[9], tz, pq[9]), vr = fma(pq[18] - pq[10], tz, pq[10]);
          const double S = (vr - vl) * (1.0 / 16.0), b0 = fma(S, (double)(SEG * (sg & 1)), vl);
#pragma unroll
          for (int e = 0; e < SEG; ++e)
            if ((inb >> e) & 1u) v[e] += (T)fma(S, (double)e, b0);
        };
        T x[SEG];
        load_seg<T>(xa, x);
        if (TWO) own_corr(x, pc);
        if (!CHEB) {
#pragma unroll
          for (int e = 0; e < SEG; ++e) out[e] = Rn<T>::fma(-a.alpha, acc[e], x[e]);
        } else {
          T xm[SEG];
          load_seg<T>(sb + fofs + C::F_BYTES, xm);
          if (TWO) own_corr(xm, pc + 32);
          const T om = a.rho_ps ? (T)cheb_omega(a.cheb_k, (double)a.rho_ps[n]) : a.omega;
#pragma unroll
          for (int e = 0; e < SEG; ++e) out[e] = Rn<T>::fma(om, Rn<T>::fma(-a.gamma, acc[e], x[e]) - xm[e], xm[e]);
        }
      }
      if (tstore) {
        // results -> this iteration's staging buffer; made visible to the async proxy before the barrier.  Thread 0 first
        // makes sure the previous TMA store has finished READING its buffer, which the next iteration overwrites.
        const uint32_t ob = outa + (it & 1u) * C::OUT_BYTES;
#pragma unroll
        for (int q = 0; q < NV; ++q) sts16(ob + 16u * q, &out[q * V]);
        fence_proxy_async_smem();
        if (tid == 0) tma_store_wait_read0();
      }
      if (CHECK && !TWO) {   // per-warp sum of r^2 into this iteration's buffer BEFORE the barrier: no barrier of its own
#pragma unroll
        for (int q = 16; q > 0; q >>= 1) rr += __shfl_down_sync(0xffffffffu, rr, q);
        if ((tid & 31) == 0) red[it & 1u][tid >> 5] = rr;
      }
      cta_bar_sync();                           // every thread is done with the stage (and has staged its results)
      if (tid == 0) {
        issue_next();                           // ... refill it, NSTAGE items ahead
        if (tstore) {
          // box [TH][FW] at (column 0 of tile column tile % tiles_x, row j0, solve n): columns >= TW and rows >= ny are out
          // of bounds of the 4-D map and are not written
          tma_store_4d(&map_out, sm0 + (uint32_t)(AFTER + C::FAC_BYTES) + (it & 1u) * C::OUT_BYTES, 0,
                       tile % a.tiles_x, j0, n);
          tma_store_commit();
        }
      }
      if (TWO && (uint32_t)(tid >> 5) == (it & 3u)) {
        // this iteration's reducer warp: lane = kind * 8 + segment; kinds 0/1 = sum_j (1 - j/16) S0/S1 (coarse row of the
        // tile's first row), kinds 2/3 = sum_j (j/16) S0/S1 (the next coarse row)
        const int lane = tid & 31, kind = lane >> 3;
        const double* red = reinterpret_cast<const double*>(smem_raw + RES_OFS + (it & 1u) * C::RES_BYTES) + (lane & 7) * 2 + (kind & 1);
        double t4[4] = {0.0, 0.0, 0.0, 0.0};       // four short chains instead of one of 16
#pragma unroll
        for (int j = 0; j < TH; ++j) {
          const double wz = kind < 2 ? 1.0 - (double)j / TH : (double)j / TH;
          t4[j & 3] = fma(wz, red[j * NSEG * 2], t4[j & 3]);
        }
        const double t = (t4[0] + t4[1]) + (t4[2] + t4[3]);
        a.cpart[((size_t)n * ntiles + tile) * 32 + lane] = t;
        if (CHECK) {
          // sum of r^2 over the tile in the order of the per-warp reduction below (a shuffle-down tree over the 32 lanes of
          // warp w, then w = 0..3 in turn), so the check partials keep their bits: lane 8 w + p starts from the tree's first
          // two levels for lane p of warp w, (v_p + v_p+16) + (v_p+8 + v_p+24), and finishes it with three shuffles
          const double* rv = reinterpret_cast<const double*>(smem_raw + RES_OFS + (it & 1u) * C::RES_BYTES + TH * NSEG * 16) +
                             32 * (lane >> 3) + (lane & 7);
          double b = (rv[0] + rv[16]) + (rv[8] + rv[24]);
#pragma unroll
          for (int q = 4; q > 0; q >>= 1) b += __shfl_down_sync(0xffffffffu, b, q);
          double w4[NT / 32];
#pragma unroll
          for (int q = 0; q < NT / 32; ++q) w4[q] = __shfl_sync(0xffffffffu, b, 8 * q);
          if (lane == 0) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < NT / 32; ++q) s += w4[q];
            a.partial[(size_t)n * ntiles + tile] = s;
          }
        }
      }
      if (!tstore) {
        T* const o = a.dst + ((size_t)n * nn + gofs);
        if (seg_full) {
#pragma unroll
          for (int q = 0; q < NV; ++q) stg16(o + q * V, &out[q * V]);
        } else if (row_in) {
#pragma unroll
          for (int e = 0; e < SEG; ++e)
            if (gi + e < a.nx) o[e] = out[e];
        }
      }
      if (CHECK && !TWO && tid == 0) {   // fixed order: deterministic.  (The buffer is rewritten two iterations on, after a barrier this thread has passed.)
        double t = 0.0;
        for (int q = 0; q < NT / 32; ++q) t += red[it & 1u][q];
        a.partial[(size_t)n * ntiles + tile] = t;
      }
      ++it;
    }
  }
  if (tstore && tid == 0) tma_store_wait_all();   // the staging buffers must outlive the last stores
}

}  // namespace xee

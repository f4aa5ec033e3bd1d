// xee_plan.cuh — solve plans: device state, launch logic and the host control loop of
// solve_elliptic (xtt-lib-fortran/elliptic_tools.f90:93-265).
// No CPU compute path exists here: without a usable CUDA device every entry point fails loudly.
#pragma once
#include <algorithm>
#include <atomic>
#include <cmath>
#include <ctime>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "xee_kernels.cuh"
#include "xee_sweep_tma.cuh"
#include "xee_sweep_tb.cuh"
#include "xee_sweep_line.cuh"
#include "xee_twolevel.cuh"
#include "xee_resident.cuh"
#include "xee_krylov.cuh"
#include "xee_mixed.cuh"

namespace xee {

extern thread_local std::string g_last_error;
extern std::atomic<long long> g_launches;

#define XEE_CHECK(expr)                                                                          \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      char _b[512];                                                                              \
      snprintf(_b, sizeof _b, "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      g_last_error = _b;                                                                         \
      return 1;                                                                                  \
    }                                                                                            \
  } while (0)

#define XEE_LAUNCH_OK()                                   \
  do {                                                    \
    g_launches.fetch_add(1, std::memory_order_relaxed);   \
    XEE_CHECK(cudaGetLastError());                        \
  } while (0)

inline int fail(const char* msg) { g_last_error = msg; return 1; }

// The dynamic-shared-memory opt-in is a per-DEVICE function attribute: set it once per (kernel instantiation, device).
template <class K>
inline int opt_in_smem(K kernel, int bytes, std::atomic<unsigned long long>& done_mask) {
  int dev = 0;
  XEE_CHECK(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if (done_mask.load(std::memory_order_acquire) & bit) return 0;
  if (bytes < 0) {   // everything the SM has left beside the kernel's static shared memory
    cudaFuncAttributes fa{};
    XEE_CHECK(cudaFuncGetAttributes(&fa, kernel));
    bytes = 227 * 1024 - (int)fa.sharedSizeBytes;
  }
  XEE_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done_mask.fetch_or(bit, std::memory_order_release);
  return 0;
}

// Makes the plan's device current for the duration of an entry point and restores the caller's device afterwards.
struct DeviceGuard {
  int prev = -1; bool switched = false;
  explicit DeviceGuard(int dev) {
    if (dev < 0) return;
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

inline int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

// Runtime flags to compile-time ones: calls f(std::bool_constant<b0>{}, std::bool_constant<b1>{}, ...), so that a launch
// site spells its kernel's template arguments once and instantiates one kernel per combination of the flags it passes.
template <class F> int dispatch(F&& f) { return f(); }
template <class F, class... B> int dispatch(F&& f, bool b, B... rest) {
  if (b) return dispatch([&](auto... c) { return f(std::true_type{}, c...); }, rest...);
  return dispatch([&](auto... c) { return f(std::false_type{}, c...); }, rest...);
}
constexpr int arith_of(bool strict) { return strict ? XEE_ARITH_STRICT : XEE_ARITH_FAST; }
constexpr int mode_of(bool cheb) { return cheb ? MODE_CHEBYSHEV : MODE_JACOBI; }

// The device of a new plan, map or series: `want`, or the current device when want < 0, resolved so that later entry
// points can return to it.
inline int resolve_device(int want, int* dev) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("xee: no CUDA device available - this library has no CPU fallback");
  *dev = want;
  if (*dev < 0) XEE_CHECK(cudaGetDevice(dev));
  if (*dev >= ndev) return fail("xee: device index out of range");
  return 0;
}

// Caching device allocator for the large field buffers: cudaFree of GiB-sized blocks costs tens of ms
// (unmap + implicit sync), which a driver that creates a plan per solve_elliptic call would pay every time.
// cudaMalloc/cudaFree are also erratic (an occasional cudaFree was measured at 0.2-1.6 s on a busy box), so EVERY
// device allocation of the library goes through this pool.  Freed blocks are kept (exact-size match) up to
// XEE_CACHE_MB (default 16384) and reused; xee_release_cached_memory() returns them to the driver.
struct DevPool {
  std::mutex mu;
  typedef std::pair<int, size_t> Key;            // (device, bytes): blocks never migrate between devices
  std::multimap<Key, void*> free_blocks;
  std::map<void*, Key> live;
  size_t cached = 0, live_bytes = 0;
  static DevPool& get() { static DevPool p; return p; }
  cudaError_t alloc(void** out, size_t bytes) {
    int dev = 0;
    cudaGetDevice(&dev);
    const Key key(dev, bytes);
    {
      std::lock_guard<std::mutex> g(mu);
      auto it = free_blocks.find(key);
      if (it != free_blocks.end()) {
        *out = it->second; cached -= bytes; free_blocks.erase(it); live[*out] = key; live_bytes += bytes;
        return cudaSuccess;
      }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();   // clear the sticky-free allocation error: the retry below may succeed and the next launch check must not see it
      trim(0); e = cudaMalloc(out, bytes);
    }
    if (e == cudaSuccess) { std::lock_guard<std::mutex> g(mu); live[*out] = key; live_bytes += bytes; }
    return e;
  }
  void release(void* p) {
    if (!p) return;
    {
      std::lock_guard<std::mutex> g(mu);
      auto it = live.find(p);
      if (it == live.end()) { cudaFree(p); return; }
      const Key key = it->second; live.erase(it); live_bytes -= key.second;
      const size_t cap = (size_t)env_int("XEE_CACHE_MB", 16384) << 20;
      if (cached + key.second <= cap) { free_blocks.emplace(key, p); cached += key.second; return; }
    }
    cudaFree(p);
  }
  void trim(size_t keep) {
    std::lock_guard<std::mutex> g(mu);
    while (cached > keep && !free_blocks.empty()) {
      auto it = std::prev(free_blocks.end());
      cudaFree(it->second); cached -= it->first.second; free_blocks.erase(it);
    }
  }
  void stats(long long* live_out, long long* cached_out) {
    std::lock_guard<std::mutex> g(mu);
    if (live_out) *live_out = (long long)live_bytes;
    if (cached_out) *cached_out = (long long)cached;
  }
};
inline void pool_free(void* p) { DevPool::get().release(p); }

// The one owner of a pool block: the block goes back to the pool when the handle is destroyed.  The pool does not track
// streams, so whoever destroys a handle makes sure the device has finished with its block.
class PoolBuf {
  void* p_ = nullptr;
 public:
  PoolBuf() = default;
  PoolBuf(PoolBuf&& o) noexcept : p_(o.p_) { o.p_ = nullptr; }
  ~PoolBuf() { pool_free(p_); }
  // allocates the block of an empty handle and points *view at it (nullptr on failure)
  template <class P> cudaError_t alloc(P** view, size_t bytes) {
    const cudaError_t e = DevPool::get().alloc(&p_, bytes);
    if (e != cudaSuccess) p_ = nullptr;
    *view = (P*)p_;
    return e;
  }
};

// The device memory of a plan, map or series: own() allocates a block, keeps its handle and sets the raw view the kernels
// take.  The blocks go back to the pool when the owner is destroyed, after the body of its destructor.
struct PoolOwner {
  std::vector<PoolBuf> owned;
  template <class P> cudaError_t own(P** view, size_t bytes) {
    owned.emplace_back();
    return owned.back().alloc(view, bytes);
  }
};

// XEE_TRACE=1: wall-clock phase timings on stderr (host side, after a device sync).
struct TraceTimer {
  const char* what; double t0; bool on;
  static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }
  explicit TraceTimer(const char* w) : what(w), t0(0), on(env_int("XEE_TRACE", 0) != 0) { if (on) { cudaDeviceSynchronize(); t0 = now(); } }
  ~TraceTimer() { if (on) { cudaDeviceSynchronize(); fprintf(stderr, "xee trace: %-28s %9.3f ms\n", what, (now() - t0) * 1e3); } }
};

struct PlanBase {
  xee_plan_desc d{};
  virtual ~PlanBase() {}
  virtual int set_coe_aos(const void* coe, bool on_host) = 0;
  virtual int set_abc(const void* a, const void* b, const void* c, double dx, double dy) = 0;
  virtual int solve(void* psi, const void* f, const xee_solve_params* prm, int* iters, double* r1o, double* r2o,
                    int* err, cudaStream_t s, bool host_io, void* workspace_host, int debug) = 0;
  // check_step: the BiCGStab methods replace the recurrence residual every check_step iterations, as a solve does (the
  // other methods ignore it)
  virtual int sweeps(void* psi, const void* f, double alpha, int sweeps, int check_step, double* rms, cudaStream_t s) = 0;
  virtual int apply(const void* psi, void* out, cudaStream_t s) = 0;
  virtual int coe_to_aos_host(void* coe_host) = 0;
  double sweep_ms = 0.0;
  double probe_ms = 0.0;             // host wall time spent in the spectral-radius probes (estimate_rho)
  long long sweep_launches = 0;      // sweeps performed (v4 does up to tb_depth of them per kernel launch)
  long long kernel_launches = 0;     // launches of the sweep kernel
  int variant_used = 0, depth_used = 1;   // sweep-kernel variant of the last solve/sweeps call (1..5) and its sweeps per pass
  double cheb_rho_used = 0.0, cheb_gamma_used = 1.0;   // Chebyshev parameters of the last accelerated call
  // residual norm of the stop rule: 0 = RMS over the interior (elliptic_tools.f90:190-199); 1 = max |r|, joined with norm_floor
  // (legacy strategies 3/4, old-diagnose/xtt-lib/elliptic_tools.f90:203-204; point methods only)
  int norm_max = 0;
  double norm_floor = 0.0;
  int rho_subsample = 0;   // > 1 (one operator per solve): probe every rho_subsample-th operator set only and interpolate the
                           // spectral data in between - for series whose operators vary smoothly with the index (set by the caller)
  // the *_sweep_kernel_stats and *_kernel_info entry points of plans, maps and series
  int kernel_stats(double* ms, long long* launches, int reset) {
    if (ms) *ms = sweep_ms;
    if (launches) *launches = sweep_launches;
    if (reset) { sweep_ms = 0; sweep_launches = 0; kernel_launches = 0; }
    return 0;
  }
  int kernel_info(int* variant, int* sweeps_per_pass, long long* launches) const {
    if (variant) *variant = variant_used;
    if (sweeps_per_pass) *sweeps_per_pass = depth_used;
    if (launches) *launches = kernel_launches;
    return 0;
  }
};

template <class T>
struct Plan : PlanBase, PoolOwner {
  size_t nn = 0;
  int nsets = 1;
  T* coe = nullptr;       // [nsets][10][ny][nx]
  T* x1 = nullptr;        // second ping-pong buffer [nbatch][ny][nx]
  T* io_psi = nullptr;    // device staging for the host-pointer entry points
  T* io_f = nullptr;
  SolveState<T> st{};
  double* partial = nullptr;
  double* partial_max = nullptr;   // [nbatch][kResmaxBlocks] (norm_max only)
  int ntiles = 0, gx = 0, gy = 0, gz = 0, spb = 1;
  int* h_active = nullptr;  // pinned
  cudaStream_t own_stream = nullptr;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  cudaEvent_t poll_ev[4]{};
  double cheb_rho = 0.0;             // shared operator: one spectral radius
  std::vector<double> rho_ps;        // one operator per solve: per-solve spectral radii (host copy)
  std::vector<double> est_rho_ps;    // the spectral estimate of the current operator (rho_ps of the calls that estimate)
  T* rho_dev = nullptr;              //   ... and on the device
  // v2 (TMA) sweep kernel: launch geometry + tensor maps of the buffers of the current call
  bool use_tma = false;
  int tma_tiles_x = 0, tma_tiles_y = 0, tma_chunk = 1, tma_nchunks = 1, tma_grid = 1, tma_nstage = 6, num_sms = 148;
  CUtensorMap map_halo[2]{}, map_plain[2]{}, map_f{}, map_coe{};
  bool map_coe_ready = false;
  const void* map_ptrs[3] = {nullptr, nullptr, nullptr};
  // v5 (segment-line relaxation, XEE_METHOD_LINE_*): Thomas factors, tiling, tensor-map cache
  bool use_line = false;
  T* linefac = nullptr;              // [nsets][6][ny][nx]: m, u, v, w, cB, cA (line_factor_kernel)
  unsigned char* linepack = nullptr; // operator + factors in tile/thread order
  bool linefac_ready = false;
  int ln_tiles_x = 0, ln_tiles_y = 0, ln_chunk = 1, ln_nchunks = 1;
  struct LineMap { const void* ptr; int nb; int kind; int es; CUtensorMap map; };
  std::vector<LineMap> line_maps;    // kind 0: psi box (with halo), 1: f / psi_{k-1} box, 2: 4-D store view of the result
  bool ln_tstore = false;            // results leave through TMA stores (nx a multiple of the tile width)
  bool method_is_cheb() const { return d.method == XEE_METHOD_CHEBYSHEV || d.method == XEE_METHOD_LINE_CHEBYSHEV || d.method == XEE_METHOD_LINE2_CHEBYSHEV || d.method == XEE_METHOD_LINE2_MIXED; }
  // two-level block-line methods (XEE_METHOD_LINE2_*, xee_twolevel.cuh): coarse-grid data of the operator and of a batch
  bool use_two = false;
  tl::Dims tld{};
  double *tl_ainv = nullptr, *tl_tmp = nullptr;   // [ncp][ncp]: Ac^-1, and Ac for the band factorisation
  double *tl_part = nullptr;                      // [nbatch][ntiles][32] per-tile restriction of the residual
  double *tl_band = nullptr;                      // [nsets][2][nc][ncx + 2] band LU factors of the coarse operators
  double *tl_scale = nullptr;                     // [nbatch] per-solve factor of the coarse correction (one operator per solve)
  double *tl_ck = nullptr;                        // [GSPLIT][nbatch][ncp] partial products of the coarse solve
  double *tl_rc = nullptr, *tl_cv = nullptr;      // [nbatch][ncp] restricted residual, [2 slots][nbatch][pz][px] coarse corrections
  CUtensorMap map_cv{};                           //   ... and the TMA view of them ({px, pz, 2 nbatch}, boxes of 8 x 3)
  double tl_gamma = 1.0, tl_lmax = 0.0, tl_lmin = 0.0;
  bool tl_ready = false;
  // v4 (temporal blocking) sweep kernel: two more iterate buffers (passes cannot update in place), tiling, maps
  bool use_tb = false;
  int tb_depth = 4, tb_tiles_x = 0, tb_tiles_y = 0, tb_chunk = 1, tb_nchunks = 1, tb_grid = 1;
  T *x2 = nullptr, *x3 = nullptr;
  CUtensorMap map_tb[4]{}, map_tb_f{};
  const void* map_tb_ptrs[3] = {nullptr, nullptr, nullptr};
  // BiCGStab (XEE_METHOD_LINE*_BICGSTAB, xee_krylov.cuh): the Krylov vectors, per-(solve, tile) dot-product partials and
  // the per-solve recurrence scalars; x1 serves as the zero field the preconditioner sweeps start from
  bool use_krylov = false;
  kr::Vecs<T> kv{};
  kr::Scal ksc{};
  double* kpart = nullptr;
  int kcheck = 100;                  // iterations between residual replacements in the current call (its check_step)
  // line2_mixed (xee_mixed.cuh): the fp32 operator pack, r32 [nbatch][ny][nx], the per-solve scales [2][nbatch] and a float
  // copy of the per-solve Chebyshev radii; the fp32 pair of the Chebyshev recurrence lives in x1
  bool use_mixed = false;
  unsigned char* linepack32 = nullptr;
  float *mx_r32 = nullptr, *mx_rho = nullptr;
  double* mx_scale = nullptr;
  std::vector<float> mx_rho_h;

  int init() {
    TraceTimer tt("plan init");
    nn = (size_t)d.nx * d.ny;
    nsets = d.shared_coe ? 1 : d.nbatch;
    XEE_CHECK(cudaStreamCreateWithFlags(&own_stream, cudaStreamNonBlocking));
    XEE_CHECK(own(&coe, sizeof(T) * kPlanes * nn * nsets));
    // on the plan's own (non-blocking) stream: a cudaMemset on the legacy default stream is asynchronous and NOT ordered with
    // it, and could land after the operator assembly (seen under multi-process timing: a zeroed operator, NaN factors)
    XEE_CHECK(cudaMemsetAsync(coe, 0, sizeof(T) * kPlanes * nn * nsets, own_stream));
    XEE_CHECK(own(&x1, sizeof(T) * nn * d.nbatch));
    const int nb = d.nbatch;
    XEE_CHECK(own(&st.done, sizeof(int) * nb)); XEE_CHECK(own(&st.iters, sizeof(int) * nb));
    XEE_CHECK(own(&st.ccnt, sizeof(int) * nb)); XEE_CHECK(own(&st.lcnt, sizeof(int) * nb));
    XEE_CHECK(own(&st.errb, sizeof(int) * nb));
    XEE_CHECK(own(&st.err_before, sizeof(T) * nb)); XEE_CHECK(own(&st.err_now, sizeof(T) * nb));
    XEE_CHECK(own(&st.ratio, sizeof(T) * nb)); XEE_CHECK(own(&st.r1, sizeof(T) * nb));
    XEE_CHECK(own(&st.r2, sizeof(T) * nb)); XEE_CHECK(own(&st.active, sizeof(int)));
    XEE_CHECK(own(&st.best_err, sizeof(T) * nb)); XEE_CHECK(own(&st.stall, sizeof(int) * nb));
    st.trace_cap = 4096;
    XEE_CHECK(own(&st.trace_err, sizeof(T) * st.trace_cap));
    XEE_CHECK(own(&st.trace_ratio, sizeof(T) * st.trace_cap));
    XEE_CHECK(cudaMallocHost(&h_active, sizeof(int) * 4));
    for (auto& e : poll_ev) XEE_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    // launch geometry of the direct kernel
    gx = (d.nx - 2 + kDirBX - 1) / kDirBX;
    gy = (d.ny - 2 + kDirBY - 1) / kDirBY;
    ntiles = gx * gy;
    // Keep the operator in registers across `spb` solves, but leave >= ~4 waves of blocks on 148 SMs.
    spb = 1;
    if (d.shared_coe) {
      spb = 8;
      while (spb > 1 && (long long)ntiles * ((d.nbatch + spb - 1) / spb) < 148LL * 8 * 4) spb /= 2;
    }
    gz = (d.nbatch + spb - 1) / spb;
    int dev = 0;
    XEE_CHECK(cudaGetDevice(&dev));
    XEE_CHECK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    // Kernel variant: 1 = v1 direct, 2 = v2 TMA pipeline.  auto: TMA for shared-operator batches whose rows are
    // 16-byte multiples (TMA global-stride rule); everything else takes the direct kernel.
    int want = d.kernel > 0 ? d.kernel : env_int("XEE_KERNEL", 0);
    const bool tma_ok = ((size_t)d.nx * sizeof(T)) % 16 == 0 && d.nx >= 8 && d.ny >= 4;
    if (want == 2 && !tma_ok) return fail("xee: kernel=2 (TMA) needs nx*sizeof(real) % 16 == 0");
    use_tma = (want == 2) || (want == 0 && tma_ok && (long long)d.nbatch * d.nx * d.ny >= (1 << 16));
    if (use_tma) {
      tma_tiles_x = (d.nx - 2 + tma::TW - 1) / tma::TW;
      tma_tiles_y = (d.ny - 2 + tma::TH - 1) / tma::TH;
      const int nt = tma_tiles_x * tma_tiles_y;
      // operator registers reused across the solves of a unit; +2: operator reload per unit
      tma_chunk = pick_chunk(nt, std::min(4, d.nbatch), std::min(32, d.nbatch), [](long long rounds, int ch) { return rounds * ch + 2; });
      tma_nchunks = (d.nbatch + tma_chunk - 1) / tma_chunk;
      tma_grid = (int)std::min<long long>(num_sms, (long long)nt * tma_nchunks);
      static_assert(tma::NSTAGE_MAX >= 6, "six pipeline stages for a shared operator");
      tma_nstage = d.shared_coe ? 6 : 2;   // one operator per solve: its tiles travel with every stage, 2 x ~110 KB (fp64)
    }
    // v5: segment-line relaxation is a METHOD, not a variant of the reference iteration: explicit request only.
    use_krylov = d.method == XEE_METHOD_LINE_BICGSTAB || d.method == XEE_METHOD_LINE2_BICGSTAB;
    use_mixed = d.method == XEE_METHOD_LINE2_MIXED;
    use_two = d.method == XEE_METHOD_LINE2_JACOBI || d.method == XEE_METHOD_LINE2_CHEBYSHEV || d.method == XEE_METHOD_LINE2_BICGSTAB || use_mixed;
    use_line = use_two || use_krylov || d.method == XEE_METHOD_LINE_JACOBI || d.method == XEE_METHOD_LINE_CHEBYSHEV;
    if (d.method < 0 || d.method > XEE_METHOD_LINE2_MIXED) return fail("xee: unknown method");
    if (use_mixed && sizeof(T) != 8) return fail("xee: line2_mixed returns fp64 answers from fp32 sweeps: it needs an fp64 plan");
    if (use_line) {
      if (d.arith != XEE_ARITH_FAST || !tma_ok)
        return fail("xee: the line-relaxation methods need FAST arithmetic and nx*sizeof(real) % 16 == 0");
      if (want != 0 && want != 5) return fail("xee: the line-relaxation methods run on sweep kernel 5 only");
      use_tma = false;
      ln_tiles_x = (d.nx + ln::TW - 1) / ln::TW; ln_tiles_y = (d.ny + ln::TH - 1) / ln::TH;
      const int nt = ln_tiles_x * ln_tiles_y;
      const int chmax = d.shared_coe ? std::min(32, d.nbatch) : 1;
      ln_chunk = pick_chunk(nt, std::min(4, chmax), chmax, [](long long rounds, int ch) { return rounds * (ch + 1); });
      ln_nchunks = (d.nbatch + ln_chunk - 1) / ln_chunk;
      ln_tstore = d.nx % ln::TW == 0;
      XEE_CHECK(own(&linefac, sizeof(T) * kLineFacPlanes * nn * nsets));
      XEE_CHECK(own(&linepack, (size_t)nt * line_pack_tile_bytes<T>() * nsets));
      want = 5;
      if (use_two) {
        static_assert(ln::TH == tl::HZ && 2 * ln::SEG == tl::HR, "the two-level restriction assumes 16-row tiles and two 8-point segments per coarse cell");
        if (sizeof(T) != 8) return fail("xee: the two-level methods need fp64 fields");
        tld = tl::dims(d.nx, d.ny);
        if (tld.ncx < 1 || tld.ncz < 1) return fail("xee: the two-level methods need at least 18 x 18 grid points (one coarse node)");
        const size_t ab = sizeof(double) * (size_t)tld.ncp * tld.ncp * nsets;     // one coarse operator per operator set
        XEE_CHECK(own(&tl_ainv, ab)); XEE_CHECK(own(&tl_tmp, ab));
        XEE_CHECK(own(&tl_scale, sizeof(double) * nb));
        XEE_CHECK(own(&tl_band, sizeof(double) * 2 * (size_t)tld.nc * (tld.ncx + 2) * nsets));
        XEE_CHECK(own(&tl_part, sizeof(double) * (size_t)nb * nt * 32));
        XEE_CHECK(own(&tl_rc, sizeof(double) * (size_t)nb * tld.ncp));
        XEE_CHECK(own(&tl_ck, sizeof(double) * tl::GSPLIT * (size_t)nb * tld.ncp));
        XEE_CHECK(own(&tl_cv, sizeof(double) * 2 * (size_t)nb * tld.pz * tld.px));
        XEE_CHECK(cudaMemsetAsync(tl_rc, 0, sizeof(double) * (size_t)nb * tld.ncp, own_stream));                 // padding stays 0
        XEE_CHECK(cudaMemsetAsync(tl_cv, 0, sizeof(double) * 2 * (size_t)nb * tld.pz * tld.px, own_stream));     // rim stays 0
        if (encode_map(&map_cv, tl_cv, tld.px, tld.pz, 2 * nb, 8, 3)) return 1;
      }
      if (use_mixed) {
        if (((size_t)d.nx * sizeof(float)) % 16) return fail("xee: line2_mixed needs nx % 4 == 0 (rows of its fp32 fields are 16-byte multiples)");
        XEE_CHECK(own(&linepack32, (size_t)nt * line_pack_tile_bytes<float>() * nsets));
        XEE_CHECK(own(&mx_r32, sizeof(float) * nn * nb));
        XEE_CHECK(cudaMemsetAsync(mx_r32, 0, sizeof(float) * nn * nb, own_stream));   // the rim stays 0
        XEE_CHECK(own(&mx_scale, sizeof(double) * 2 * nb));
        XEE_CHECK(own(&mx_rho, sizeof(float) * nsets));
      }
      if (use_krylov) {
        T** vecs[7] = {&kv.r, &kv.r0, &kv.p, &kv.ph, &kv.s, &kv.v, &kv.t};
        for (T** v : vecs) XEE_CHECK(own(v, sizeof(T) * nn * nb));
        XEE_CHECK(own(&kpart, sizeof(double) * kr::NP * (size_t)ntiles * nb));
        double** sc[5] = {&ksc.rho, &ksc.alpha, &ksc.omega, &ksc.beta, &ksc.r0n};
        for (double** v : sc) XEE_CHECK(own(v, sizeof(double) * nb));
        XEE_CHECK(own(&ksc.restart, sizeof(int) * nb));
      }
    } else if (want == 5) return fail("xee: kernel=5 is the line-relaxation kernel: select it with method = XEE_METHOD_LINE_*");
    // v4: temporal blocking.  auto: large shared-operator batches in FAST arithmetic (STRICT is bound by its true
    // divisions, where the redundant halo work of overlapping tiles costs more than the saved traffic).
    tb_depth = std::max(1, std::min(env_int("XEE_TB", 4), std::min(tb::TBMAX, tb::H / 2 - 1)));
    if (sizeof(T) == 4 && (tb_depth & 1)) tb_depth += 1;    // tile origins must stay 16-byte aligned (4 floats)
    const bool tb_ok = tma_ok && d.shared_coe && !use_line;
    if (want == 4 && !tb_ok) return fail("xee: kernel=4 (temporal blocking) needs a shared operator and nx*sizeof(real) % 16 == 0");
    use_tb = (want == 4) || (want == 0 && tb_ok && d.arith == XEE_ARITH_FAST && d.nbatch >= 32 &&
                             (long long)d.nbatch * d.nx * d.ny >= (1 << 22));
    if (use_tb) {
      const int sx = tb::W - 2 * tb_depth, sy = tb::H - 2 * tb_depth;
      tb_tiles_x = d.nx <= tb::W ? 1 : (d.nx - tb::W + sx - 1) / sx + 1;
      tb_tiles_y = d.ny <= tb::H ? 1 : (d.ny - tb::H + sy - 1) / sy + 1;
      const int nt = tb_tiles_x * tb_tiles_y;
      // the operator registers are reloaded (from L2) once per unit, worth ~2 solves
      const int chmax = std::min(64, d.nbatch);
      tb_chunk = pick_chunk(nt, std::min(8, chmax), chmax, [](long long rounds, int ch) { return rounds * (ch + 2); });
      tb_nchunks = (d.nbatch + tb_chunk - 1) / tb_chunk;
      tb_grid = (int)std::min<long long>(num_sms, (long long)nt * tb_nchunks);
      XEE_CHECK(own(&x2, sizeof(T) * nn * d.nbatch));
      XEE_CHECK(own(&x3, sizeof(T) * nn * d.nbatch));
    }
    // the residual partials are per (solve, tile): room for the tiling with the most tiles
    const int ptiles = std::max({ntiles, use_tma ? tma_tiles_x * tma_tiles_y : 0, use_line ? ln_tiles_x * ln_tiles_y : 0, use_tb ? tb_ntiles() : 0});
    XEE_CHECK(own(&partial, sizeof(double) * (size_t)ptiles * nb));
    return 0;
  }
  int sweep_ntiles() const { return use_line ? ln_tiles_x * ln_tiles_y : use_tma ? tma_tiles_x * tma_tiles_y : ntiles; }
  int tb_ntiles() const { return tb_tiles_x * tb_tiles_y; }
  int check_ntiles() const { return use_krylov || use_mixed ? ntiles : use_tb ? tb_ntiles() : sweep_ntiles(); }   // residual partials per solve

  // Solves per work unit of a persistent kernel: the chunk in [chmin, chmax] that minimises the makespan
  // cost(rounds, chunk) of the static round-robin of the units over at most num_sms CTAs (ties: the largest chunk).
  template <class Cost>
  int pick_chunk(int nt, int chmin, int chmax, Cost cost) const {
    long long best = -1; int chunk = 1;
    for (int ch = chmax; ch >= chmin; --ch) {
      const long long units = (long long)nt * ((d.nbatch + ch - 1) / ch);
      const long long g = std::min<long long>(num_sms, units);
      const long long makespan = cost((units + g - 1) / g, ch);
      if (best < 0 || makespan < best) { best = makespan; chunk = ch; }
    }
    return chunk;
  }

  // cuTensorMapEncodeTiled through the runtime (no link-time dependency on libcuda): elements of type E (the plan's T, or
  // float for the fp32 fields of line2_mixed), no interleave, no swizzle, 128-byte L2 promotion, no out-of-bounds fill.
  // dims and box have `rank` entries, byte_strides rank - 1.
  template <class E = T>
  static int encode_tiled(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* byte_strides,
                          const cuuint32_t* box) {
    typedef CUresult (*Fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                           const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                           CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static Fn fn = nullptr;
    if (!fn) {
      void* p = nullptr; cudaDriverEntryPointQueryResult q;
      XEE_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
      if (!p) return fail("xee: cuTensorMapEncodeTiled not available from the driver");
      fn = (Fn)p;
    }
    const cuuint32_t es[4] = {1, 1, 1, 1};
    const CUresult r = fn(m, sizeof(E) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank,
                          const_cast<void*>(base), dims, byte_strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { char b[128]; snprintf(b, sizeof b, "xee: cuTensorMapEncodeTiled (rank %d) failed (%d)", rank, (int)r); return fail(b); }
    return 0;
  }
  // a batch of nb fields [nb][ny][nx] in boxes of box_w x box_h
  template <class E = T>
  static int encode_map(CUtensorMap* m, const void* base, int nx, int ny, int nb, int box_w, int box_h) {
    const cuuint64_t dims[3] = {(cuuint64_t)nx, (cuuint64_t)ny, (cuuint64_t)nb};
    const cuuint64_t strides[2] = {(cuuint64_t)nx * sizeof(E), (cuuint64_t)nx * ny * sizeof(E)};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    return encode_tiled<E>(m, base, 3, dims, strides, box);
  }
  // (Re)build the tensor maps when the buffers of this call differ from the cached ones.
  int prepare_maps(const T* x0, const T* x1buf, const T* f, int nb) {
    if (!use_tma) return 0;
    if (map_ptrs[0] == x0 && map_ptrs[1] == x1buf && map_ptrs[2] == f) return 0;
    if (((uintptr_t)x0 | (uintptr_t)x1buf | (uintptr_t)f) & 15) return fail("xee: TMA path needs 16-byte aligned field buffers");
    const int hw = tma::Cfg<T>::HALO_W;
    if (encode_map(&map_halo[0], x0, d.nx, d.ny, nb, hw, tma::TH + 2) || encode_map(&map_halo[1], x1buf, d.nx, d.ny, nb, hw, tma::TH + 2) ||
        encode_map(&map_plain[0], x0, d.nx, d.ny, nb, hw, tma::TH) || encode_map(&map_plain[1], x1buf, d.nx, d.ny, nb, hw, tma::TH) ||
        encode_map(&map_f, f, d.nx, d.ny, nb, hw, tma::TH))
      return 1;
    map_ptrs[0] = x0; map_ptrs[1] = x1buf; map_ptrs[2] = f;
    if (!d.shared_coe && !map_coe_ready) {   // the operator planes of every set, kPlanes of them per box
      const cuuint64_t dims[4] = {(cuuint64_t)d.nx, (cuuint64_t)d.ny, (cuuint64_t)kPlanes, (cuuint64_t)nsets};
      const cuuint64_t strides[3] = {(cuuint64_t)d.nx * sizeof(T), (cuuint64_t)nn * sizeof(T), (cuuint64_t)nn * kPlanes * sizeof(T)};
      const cuuint32_t box[4] = {(cuuint32_t)hw, (cuuint32_t)tma::TH, (cuuint32_t)kPlanes, 1};
      if (encode_tiled(&map_coe, coe, 4, dims, strides, box)) return 1;
      map_coe_ready = true;
    }
    return 0;
  }
  ~Plan() override {
    // The pool recycles blocks without stream tracking: before the owned blocks go back on the free list (after this body),
    // no kernel of this plan, nor of a caller's stream that used its buffers (apply / eta / uw return without
    // synchronising), may still touch them.  ~Map and ~Series keep the same rule for their own blocks.
    cudaDeviceSynchronize();
    if (h_active) cudaFreeHost(h_active);
    for (auto& e : poll_ev) if (e) cudaEventDestroy(e);
    for (auto& e : ev_pool) cudaEventDestroy(e);
    if (own_stream) cudaStreamDestroy(own_stream);
  }

  int set_coe_aos(const void* src, bool on_host) override {
    const size_t bytes = sizeof(T) * 9 * nn * nsets;
    const T* dev = (const T*)src;
    PoolBuf stage;
    if (on_host) {
      T* tmp = nullptr;
      XEE_CHECK(stage.alloc(&tmp, bytes));
      XEE_CHECK(cudaMemcpyAsync(tmp, src, bytes, cudaMemcpyHostToDevice, own_stream));
      dev = tmp;
    }
    dim3 g((d.nx + 127) / 128, d.ny, nsets);
    aos_to_planar_kernel<T><<<g, 128, 0, own_stream>>>(dev, coe, d.nx, d.ny);
    XEE_LAUNCH_OK();
    return operator_written();
  }
  int set_abc(const void* a, const void* b, const void* c, double dx, double dy) override {
    dim3 blk(64, 4), g((d.nx - 2 + 63) / 64, (d.ny - 2 + 3) / 4, nsets);
    const long long sa = nsets > 1 ? (long long)(d.nx - 1) * (d.ny - 2) : 0;
    const long long sb = nsets > 1 ? (long long)(d.nx - 1) * (d.ny - 1) : 0;
    const long long sc = nsets > 1 ? (long long)(d.nx - 2) * (d.ny - 1) : 0;
    cal_coe_kernel<T><<<g, blk, 0, own_stream>>>((const T*)a, (const T*)b, (const T*)c, coe, (T)dx, (T)dy, d.nx,
                                                 d.ny, sa, sb, sc, (long long)kPlanes * nn);
    XEE_LAUNCH_OK();
    return operator_written();
  }
  // A new planar operator has been written into `coe` on own_stream (set_coe_aos, set_abc, or a kernel of the caller's, as
  // the transposed operator of a map's adjoint): forget the spectral data of the old one, rebuild what derives from it.
  int operator_written() {
    XEE_CHECK(cudaStreamSynchronize(own_stream));
    cheb_rho = 0.0; rho_ps.clear(); est_rho_ps.clear();
    return line_factors();
  }
  int line_factors() {   // Thomas factors of the radial segments (v5), once per operator
    if (!use_line) return 0;
    const int nblk = (d.nx + ln::SEG * ln::BLK - 1) / (ln::SEG * ln::BLK);
    dim3 g((nblk + 31) / 32, d.ny, nsets);
    line_factor_kernel<T><<<g, 32, 0, own_stream>>>(coe, linefac, d.nx, d.ny);
    XEE_LAUNCH_OK();
    line_pack_kernel<T><<<dim3(ln_tiles_x * ln_tiles_y, nsets), ln::NT, 0, own_stream>>>(coe, linefac, linepack, d.nx, d.ny, ln_tiles_x);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(own_stream));
    linefac_ready = true;
    if (use_mixed && mixed_factors()) return 1;
    return use_two ? two_setup() : 0;
  }
  // line2_mixed, once per operator: the operator rounded to fp32, its block-line factors computed from it in fp32, packed
  int mixed_factors() {
    float *c32 = nullptr, *f32 = nullptr;
    PoolBuf c32_buf, f32_buf;
    XEE_CHECK(c32_buf.alloc(&c32, sizeof(float) * kPlanes * nn * nsets));
    XEE_CHECK(f32_buf.alloc(&f32, sizeof(float) * kLineFacPlanes * nn * nsets));
    mx::to_f32_kernel<<<1024, 256, 0, own_stream>>>(reinterpret_cast<const double*>(coe), c32, kPlanes * nn * nsets);
    XEE_LAUNCH_OK();
    const int nblk = (d.nx + ln::SEG * ln::BLK - 1) / (ln::SEG * ln::BLK);
    line_factor_kernel<float><<<dim3((nblk + 31) / 32, d.ny, nsets), 32, 0, own_stream>>>(c32, f32, d.nx, d.ny);
    XEE_LAUNCH_OK();
    line_pack_kernel<float><<<dim3(ln_tiles_x * ln_tiles_y, nsets), ln::NT, 0, own_stream>>>(c32, f32, linepack32, d.nx, d.ny, ln_tiles_x);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(own_stream));
    return 0;
  }
  // Two-level methods, once per operator: Galerkin coarse operator Ac = P^T L P and its inverse (band LU on the device).
  int two_setup() {
    TraceTimer tt("two-level setup");
    const int nc = tld.nc, ncp = tld.ncp;
    const size_t ab = sizeof(double) * (size_t)ncp * ncp * nsets;
    XEE_CHECK(cudaMemsetAsync(tl_ainv, 0, ab, own_stream));
    tl::galerkin_kernel<T><<<dim3(nc, nsets), 256, 0, own_stream>>>(coe, tl_ainv, d.nx, d.ny, tld.ncx, tld.ncz, ncp);
    XEE_LAUNCH_OK();
    if (ncp > nc) { tl::pad_identity_kernel<<<dim3((ncp - nc + 63) / 64, nsets), 64, 0, own_stream>>>(tl_ainv, nc, ncp); XEE_LAUNCH_OK(); }
    // band LU of every Ac (half-bandwidth ncx + 1), then the dense inverse column by column (tl_tmp holds Ac, tl_ainv the inverse)
    const int bw = tld.ncx + 1;
    XEE_CHECK(cudaMemcpyAsync(tl_tmp, tl_ainv, ab, cudaMemcpyDeviceToDevice, own_stream));
    {
      static std::atomic<unsigned long long> attr_done{0};
      const int smem = (bw + 1) * (2 * bw + 1) * (int)sizeof(double);
      if (smem > 200 * 1024) return fail("xee: two-level: coarse grid too wide for the band factorisation");
      if (opt_in_smem(tl::band_lu_kernel, std::max(smem, 48 * 1024), attr_done)) return 1;
      tl::band_lu_kernel<<<nsets, 1024, smem, own_stream>>>(tl_tmp, tl_band, nc, ncp, bw);
      XEE_LAUNCH_OK();
    }
    XEE_CHECK(cudaMemsetAsync(tl_ainv, 0, ab, own_stream));
    if (ncp > nc) { tl::pad_identity_kernel<<<dim3((ncp - nc + 63) / 64, nsets), 64, 0, own_stream>>>(tl_ainv, nc, ncp); XEE_LAUNCH_OK(); }
    tl::band_inverse_kernel<<<dim3((nc + 127) / 128, nsets), 128, 0, own_stream>>>(tl_band, tl_ainv, nc, ncp, bw);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaStreamSynchronize(own_stream));
    tl_ready = true; tl_lmax = tl_lmin = 0.0; tl_gamma = 1.0;
    return 0;
  }
  // Coarse half of one two-level sweep, after the sweep kernel has left P^T r per tile: gather, dense coarse solve for the
  // batch, scaled by `scale` = -omega gamma, written as the coarse correction c of the NEW iterate (slot `slot`).  The fields
  // are not touched: psi = y + P c is formed by whoever reads them (the next sweep; two_flush at the end).
  double* two_cv(int slot, int nb) const { return tl_cv + (size_t)slot * nb * tld.pz * tld.px; }
  template <class E>
  int two_coarse(int slot, int nb, double scale, const E* rho_ps_dev, int cheb_k, const int* done, cudaStream_t s) {
    const int nt = ln_tiles_x * ln_tiles_y;
    if (d.shared_coe && nb <= 4 && !rho_ps_dev && tld.nc <= tl::kMaxNcSmem) {   // single solves, probes: one launch instead of two
      tl::coarse_gather_matvec_kernel<<<dim3((tld.nc + 7) / 8, nb), 256, 0, s>>>(tl_ainv, tl_part, two_cv(slot, d.nbatch), done, scale, nt, ln_tiles_x,
                                                                              ln_tiles_y, tld.nc, tld.ncp, tld.ncx, tld.px, tld.pz * tld.px);
      XEE_LAUNCH_OK();
      return 0;
    }
    tl::coarse_gather_kernel<<<nb, 256, 0, s>>>(tl_part, tl_rc, done, nt, ln_tiles_x, ln_tiles_y, tld.ncx, tld.ncz, tld.ncp);
    XEE_LAUNCH_OK();
    if (!d.shared_coe || nb <= 4) {
      // one coarse operator per solve (time series), or a handful of solves (spectral probes): a matrix-vector product per solve
      const double* sps = nullptr;
      if (rho_ps_dev) {
        tl::coarse_scale_kernel<E><<<(nb + 127) / 128, 128, 0, s>>>(rho_ps_dev, cheb_k, tl_gamma, tl_scale, nb);
        XEE_LAUNCH_OK();
        sps = tl_scale;
      }
      tl::coarse_matvec_kernel<<<dim3((tld.nc + 7) / 8, nb), 256, 0, s>>>(tl_ainv, d.shared_coe ? 0 : (long long)tld.ncp * tld.ncp, tl_rc,
                                                                       two_cv(slot, d.nbatch), done, scale, sps, nb, tld.nc, tld.ncp, tld.ncx,
                                                                       tld.px, tld.pz * tld.px);
    } else {
      tl::coarse_gemm_kernel<<<dim3(tld.ncp / tl::GM, (nb + tl::GN - 1) / tl::GN, tl::GSPLIT), 128, 0, s>>>(tl_ainv, tl_rc, tl_ck, nb, tld.ncp);
      XEE_LAUNCH_OK();
      tl::coarse_finish_kernel<<<dim3((tld.nc + 127) / 128, nb), 128, 0, s>>>(tl_ck, two_cv(slot, d.nbatch), done, scale, nb, tld.nc, tld.ncp, tld.ncx,
                                                                           tld.px, tld.pz * tld.px);
    }
    XEE_LAUNCH_OK();
    return 0;
  }
  // c = 0 for both iterates: the stored fields ARE the iterates (start of a solve / of a probe)
  int two_reset(cudaStream_t s) {
    XEE_CHECK(cudaMemsetAsync(tl_cv, 0, sizeof(double) * 2 * (size_t)d.nbatch * tld.pz * tld.px, s));
    return 0;
  }
  // psi = y + P c made explicit in both buffers (b0 owns slot 0, b1 slot 1), then c = 0: the same state, stored plainly
  int two_flush(T* b0, T* b1, int nb, cudaStream_t s) {
    const dim3 g((((d.nx + 7) / 8) * d.ny + 255) / 256, 1, nb);
    tl::prolong_add_kernel<T><<<g, 256, 0, s>>>(b0, two_cv(0, nb), nullptr, d.nx, d.ny, tld.px, tld.pz * tld.px);
    XEE_LAUNCH_OK();
    tl::prolong_add_kernel<T><<<g, 256, 0, s>>>(b1, two_cv(1, nb), nullptr, d.nx, d.ny, tld.px, tld.pz * tld.px);
    XEE_LAUNCH_OK();
    return two_reset(s);
  }
  int coe_to_aos_host(void* coe_host) override {  // set 0 only (Fortran-facing cal_coe)
    T* tmp = nullptr;
    const size_t bytes = sizeof(T) * 9 * nn;
    PoolBuf tmp_buf;
    XEE_CHECK(tmp_buf.alloc(&tmp, bytes));
    dim3 g((d.nx + 127) / 128, d.ny, 1);
    planar_to_aos_kernel<T><<<g, 128, 0, own_stream>>>(coe, tmp, d.nx, d.ny);
    XEE_LAUNCH_OK();
    std::vector<T> stage(9 * nn);
    XEE_CHECK(cudaMemcpyAsync(stage.data(), tmp, bytes, cudaMemcpyDeviceToHost, own_stream));
    XEE_CHECK(cudaStreamSynchronize(own_stream));
    // interior only: the reference never writes coe's boundary entries (elliptic_tools.f90:35-36)
    T* out = (T*)coe_host;
    for (int j = 1; j < d.ny - 1; ++j)
      memcpy(out + ((size_t)j * d.nx + 1) * 9, stage.data() + ((size_t)j * d.nx + 1) * 9, sizeof(T) * 9 * (d.nx - 2));
    return 0;
  }

  SweepArgs<T> args(const T* src, T* dst, const T* f, T alpha, T omega, const int* done) const {
    SweepArgs<T> a{};
    a.src = src; a.dst = dst; a.f = f; a.coe = coe;
    a.coe_set_stride = d.shared_coe ? 0 : (long long)kPlanes * nn;
    a.field_stride = (long long)nn;
    a.nx = d.nx; a.ny = d.ny; a.nbatch = d.nbatch; a.spb = spb;
    a.alpha = alpha; a.omega = omega; a.done = done; a.partial = partial; a.ntiles = sweep_ntiles();
    a.rho_ps = nullptr; a.cheb_k = 1;
    return a;
  }

  template <int ARITH, int MODE, bool CHECK, bool PERSOLVE>
  int launch_tma_inst(const TmaSweepArgs<T>& P, const CUtensorMap& ms, const CUtensorMap& mp, cudaStream_t s) {
    constexpr int coe_off = tma::Cfg<T>::PSI_BYTES + tma::Cfg<T>::FLD_BYTES + (MODE == MODE_CHEBYSHEV ? tma::Cfg<T>::FLD_BYTES : 0);
    constexpr int stage = coe_off + (PERSOLVE ? (kPlanes * tma::Cfg<T>::FLD_RAW + 127) / 128 * 128 : 0);
    const size_t smem = (size_t)stage * P.nstage;
    static std::atomic<unsigned long long> attr_done{0};
    if (opt_in_smem(sweep_tma_kernel<T, ARITH, MODE, CHECK, PERSOLVE>, -1, attr_done)) return 1;
    sweep_tma_kernel<T, ARITH, MODE, CHECK, PERSOLVE><<<tma_grid, tma::NTHREADS, smem, s>>>(P, ms, mp, map_f, map_coe);
    return 0;
  }
  int launch_sweep_tma(const SweepArgs<T>& a, int mode, bool check, cudaStream_t s) {
    TmaSweepArgs<T> P{};
    P.a = a; P.tiles_x = tma_tiles_x; P.tiles_y = tma_tiles_y; P.nchunks = tma_nchunks; P.chunk = tma_chunk; P.nstage = tma_nstage;
    const int si = (a.src == (const T*)map_ptrs[0]) ? 0 : 1;      // which ping-pong buffer is the source
    const CUtensorMap& ms = map_halo[si];
    const CUtensorMap& mp = map_plain[si ^ 1];
    const int rc = dispatch([&](auto strict, auto cheb, auto chk, auto persolve) {
      return launch_tma_inst<arith_of(strict), mode_of(cheb), chk, persolve>(P, ms, mp, s);
    }, d.arith == XEE_ARITH_STRICT, mode == MODE_CHEBYSHEV, check, !d.shared_coe);
    if (rc) return rc;
    XEE_LAUNCH_OK();
    return 0;
  }
  // ---- v5: segment-line relaxation.  E: element type of the fields (the plan's T; float for the fp32 sweeps of line2_mixed)
  template <class E = T>
  int line_map(const void* ptr, int nb, int kind, CUtensorMap* out) {
    for (auto& m : line_maps) if (m.ptr == ptr && m.nb == nb && m.kind == kind && m.es == (int)sizeof(E)) { *out = m.map; return 0; }
    if ((uintptr_t)ptr & 15) return fail("xee: TMA path needs 16-byte aligned field buffers");
    if (line_maps.size() >= 24) line_maps.erase(line_maps.begin());
    LineMap lm{ptr, nb, kind, (int)sizeof(E), {}};
    if (kind < 2) {
      if (encode_map<E>(&lm.map, ptr, d.nx, d.ny, nb, kind == 0 ? ln::Cfg<E>::XW : ln::Cfg<E>::FW, kind == 0 ? ln::TH + 2 : ln::TH)) return 1;
    } else {   // (column within a TW-wide tile column, tile column, row, solve): a [TH][FW] staging box stored at column 0
               // loses its FW - TW pad columns as out-of-bounds elements
      const cuuint64_t dims[4] = {(cuuint64_t)ln::TW, (cuuint64_t)(d.nx / ln::TW), (cuuint64_t)d.ny, (cuuint64_t)nb};
      const cuuint64_t strides[3] = {(cuuint64_t)ln::TW * sizeof(E), (cuuint64_t)d.nx * sizeof(E), (cuuint64_t)d.nx * d.ny * sizeof(E)};
      const cuuint32_t box[4] = {(cuuint32_t)ln::Cfg<E>::FW, 1, (cuuint32_t)ln::TH, 1};
      if (encode_tiled<E>(&lm.map, ptr, 4, dims, strides, box)) return 1;
    }
    line_maps.push_back(lm);
    *out = lm.map;
    return 0;
  }
  template <class E, bool CHEB, bool CHECK, bool TWO>
  int launch_line_inst(const LineArgs<E>& A, int grid, const CUtensorMap& mx, const CUtensorMap& mxm, const CUtensorMap& mf, const CUtensorMap& mo, cudaStream_t s) {
    constexpr int smem = TWO ? ln::Cfg<E>::SMEM_BYTES_TWO : ln::Cfg<E>::SMEM_BYTES;
    static std::atomic<unsigned long long> attr_done{0};
    if (opt_in_smem(sweep_line_kernel<E, CHEB, CHECK, TWO>, smem, attr_done)) return 1;
    sweep_line_kernel<E, CHEB, CHECK, TWO><<<grid, ln::NT, smem, s>>>(A, mx, mxm, mf, mo, TWO ? map_cv : mf);
    return 0;
  }
  // Kernel arguments and tensor maps of one sweep from src to dst (dst holds the previous iterate) with right-hand side f,
  // the operator and factors from `pack`.  The caller fills in the per-sweep weights.
  struct LineLaunch { CUtensorMap cx, cxm, cf, co; int grid; };
  template <class E>
  int line_setup(const E* src, E* dst, const E* f, int nbatch, int two_slot, const int* done, const unsigned char* pack, LineArgs<E>& A, LineLaunch& L) {
    if (!linefac_ready) return fail("xee: line relaxation: the operator has not been set");
    if (line_map<E>(src, nbatch, 0, &L.cx) || line_map<E>(f, nbatch, 1, &L.cf) || line_map<E>(dst, nbatch, 1, &L.cxm)) return 1;
    if (ln_tstore) { if (line_map<E>(dst, nbatch, 2, &L.co)) return 1; } else L.co = L.cxm;
    A = LineArgs<E>{};
    A.pack = pack; A.pack_set_stride = d.shared_coe ? 0 : (long long)(ln_tiles_x * ln_tiles_y) * (long long)line_pack_tile_bytes<E>();
    A.dst = dst; A.field_stride = (long long)nn; A.nx = d.nx; A.ny = d.ny; A.nbatch = nbatch;
    A.done = done; A.partial = partial;
    A.tiles_x = ln_tiles_x; A.tiles_y = ln_tiles_y;
    A.chunk = std::min(ln_chunk, nbatch); A.nchunks = (nbatch + A.chunk - 1) / A.chunk;
    A.tstore = ln_tstore ? 1 : 0;
    A.gamma = (E)(use_two ? tl_gamma : 1.0); A.cpart = tl_part;
    // the coarse correction of `src` sits in slot two_slot, the one of the previous iterate (held by `dst`) in the other
    // slot, which the coarse solve after this sweep overwrites with the correction of the NEW iterate; the batch index of a
    // launch over a sub-batch (spectral probes) still strides by the plan's nbatch
    A.cv_cur_z = two_slot * d.nbatch; A.cv_prev_z = (1 - two_slot) * d.nbatch;
    if (use_two && !tl_ready) return fail("xee: two-level method: the operator has not been set");
    L.grid = (int)std::min<long long>((long long)num_sms * ln::CTAS_PER_SM, (long long)ln_tiles_x * ln_tiles_y * A.nchunks);
    return 0;
  }
  int launch_sweep_line(const SweepArgs<T>& a, int mode, bool check, cudaStream_t s) {
    LineArgs<T> A; LineLaunch L;
    if (line_setup<T>(a.src, a.dst, a.f, a.nbatch, a.two_slot, a.done, linepack, A, L)) return 1;
    A.alpha = a.alpha; A.omega = a.omega; A.rho_ps = a.rho_ps; A.cheb_k = a.cheb_k;
    const int rc = dispatch([&](auto cheb, auto chk, auto two) { return launch_line_inst<T, cheb, chk, two>(A, L.grid, L.cx, L.cxm, L.cf, L.co, s); },
                            mode == MODE_CHEBYSHEV, check, use_two);
    if (rc) return rc;
    XEE_LAUNCH_OK();
    if (use_two) {   // psi' = psi - alpha (z + P E) (Jacobi) / y - omega gamma P E (Chebyshev; omega from the per-launch value)
      const double scale = mode == MODE_CHEBYSHEV ? -(double)a.omega * tl_gamma : -(double)a.alpha;
      return two_coarse(1 - a.two_slot, a.nbatch, scale, mode == MODE_CHEBYSHEV ? a.rho_ps : nullptr, a.cheb_k, a.done, s);
    }
    return 0;
  }
  int launch_sweep(const SweepArgs<T>& a, int mode, bool check, cudaStream_t s) {
    if (use_line && mode != MODE_APPLY) return launch_sweep_line(a, mode, check, s);
    if (use_tma && mode != MODE_APPLY && a.nbatch == d.nbatch && (a.src == map_ptrs[0] || a.src == map_ptrs[1]))
      return launch_sweep_tma(a, mode, check, s);
    const dim3 blk(kDirBX, kDirBY), g(gx, gy, gz);
    dispatch([&](auto strict, auto cheb, auto apply, auto chk) {
      sweep_direct_kernel<T, arith_of(strict), apply ? MODE_APPLY : mode_of(cheb), chk><<<g, blk, 0, s>>>(a);
      return 0;
    }, d.arith == XEE_ARITH_STRICT, mode == MODE_CHEBYSHEV, mode == MODE_APPLY, check);
    XEE_LAUNCH_OK();
    return 0;
  }

  // ---- v4: temporal blocking.  Iterates live in two buffer pairs (new, prev): pair 0 = (x0, x1), pair 1 = (x2, x3);
  // pass p reads pair p&1 and writes the other one.
  int prepare_tb_maps(const T* x0, const T* f, int nb) {
    if (map_tb_ptrs[0] == x0 && map_tb_ptrs[1] == f && map_tb_ptrs[2] == x1) return 0;
    if (((uintptr_t)x0 | (uintptr_t)f | (uintptr_t)x1 | (uintptr_t)x2 | (uintptr_t)x3) & 15) return fail("xee: TMA path needs 16-byte aligned field buffers");
    const T* bufs[4] = {x0, x1, x2, x3};
    for (int q = 0; q < 4; ++q)
      if (encode_map(&map_tb[q], bufs[q], d.nx, d.ny, nb, tb::W, tb::H)) return 1;
    if (encode_map(&map_tb_f, f, d.nx, d.ny, nb, tb::W, tb::H)) return 1;
    map_tb_ptrs[0] = x0; map_tb_ptrs[1] = f; map_tb_ptrs[2] = x1;
    return 0;
  }
  template <int ARITH, int MODE, bool CHECK>
  int launch_tb_inst(const TbArgs<T>& A, const CUtensorMap& mx, const CUtensorMap& mxm, cudaStream_t s) {
    static std::atomic<unsigned long long> attr_done{0};
    if (opt_in_smem(sweep_tb_kernel<T, ARITH, MODE, CHECK>, tb::Cfg<T>::SMEM_BYTES, attr_done)) return 1;
    sweep_tb_kernel<T, ARITH, MODE, CHECK><<<tb_grid, tb::NT, tb::Cfg<T>::SMEM_BYTES, s>>>(A, mx, mxm, map_tb_f);
    return 0;
  }
  // One pass: sweeps first_cnt .. first_cnt+t-1 (1-based sweep numbers) of every solve that is not done.
  int launch_tb_pass(T* x0, int pass_idx, int first_cnt, int t, bool check, T alpha, int mode, const int* done, cudaStream_t s) {
    T* bufs[4] = {x0, x1, x2, x3};
    const int pin = pass_idx & 1, pout = pin ^ 1;
    TbArgs<T> A{};
    A.coe = coe; A.out_new = bufs[2 * pout]; A.out_prev = bufs[2 * pout + 1];
    A.field_stride = (long long)nn; A.nx = d.nx; A.ny = d.ny; A.nbatch = d.nbatch;
    A.nsweeps = t; A.tbh = tb_depth; A.alpha = alpha;
    for (int q = 0; q < t; ++q) A.omega[q] = mode == MODE_CHEBYSHEV ? (T)cheb_omega_host(first_cnt + q, cheb_rho) : T(1);
    A.done = done; A.partial = partial;
    A.tiles_x = tb_tiles_x; A.tiles_y = tb_tiles_y; A.nchunks = tb_nchunks; A.chunk = tb_chunk;
    const CUtensorMap& mx = map_tb[2 * pin];
    const CUtensorMap& mxm = map_tb[2 * pin + 1];
    const int rc = dispatch([&](auto strict, auto cheb, auto chk) { return launch_tb_inst<arith_of(strict), mode_of(cheb), chk>(A, mx, mxm, s); },
                            d.arith == XEE_ARITH_STRICT, mode == MODE_CHEBYSHEV, check);
    if (rc) return rc;
    XEE_LAUNCH_OK();
    ++kernel_launches;
    return 0;
  }
  // Boundary values and the first guess in every iterate buffer (elliptic_tools.f90:166-171: workspace = dat), and the tensor
  // maps of this call's buffers.
  int seed_buffers(T* x0, const T* f, cudaStream_t s) {
    const size_t fbytes = sizeof(T) * nn * d.nbatch;
    XEE_CHECK(cudaMemcpyAsync(x1, x0, fbytes, cudaMemcpyDeviceToDevice, s));
    if (!use_tb) return prepare_maps(x0, x1, f, d.nbatch);
    XEE_CHECK(cudaMemcpyAsync(x2, x0, fbytes, cudaMemcpyDeviceToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(x3, x0, fbytes, cudaMemcpyDeviceToDevice, s));
    return prepare_tb_maps(x0, f, d.nbatch);
  }
  // Sweeps cnt+1 .. cnt+k (1-based sweep numbers) of every solve that is not done, with the residual partials of the last
  // one when `check`.  v4 runs them in passes of up to tb_depth sweeps (tb_pass counts the passes of the call); the other
  // kernels ping-pong: sweep c reads x0 when c is odd, x1 when it is even.
  int run_sweeps(T* x0, const T* f, T alpha, int mode, int cnt, int k, bool check, const int* done, int& tb_pass, cudaStream_t s) {
    const int end = cnt + k;
    if (use_mixed) {    // fp32 sweeps; a refinement step ends with the fold and the residual pass (the check partials)
      while (cnt < end)
        if (mixed_sweep((cnt++ % kcheck) + 1, done, s) || (cnt % kcheck == 0 && mixed_check(x0, f, done, s))) return 1;
      kernel_launches += k; sweep_launches += k;
      return 0;
    }
    if (use_krylov) {   // iterations, two preconditioner sweeps each; the residual replacements leave the check partials
      while (cnt < end)
        if (krylov_iteration(x0, f, ++cnt % kcheck == 0, done, s)) return 1;
      kernel_launches += 2LL * k; sweep_launches += 2LL * k;
      return 0;
    }
    if (use_tb) {
      for (; cnt < end; ++tb_pass) {
        const int t = std::min(tb_depth, end - cnt);
        if (launch_tb_pass(x0, tb_pass, cnt + 1, t, check && cnt + t == end, alpha, mode, done, s)) return 1;
        cnt += t;
      }
    } else {
      while (cnt < end) {
        ++cnt;
        const T* src = (cnt & 1) ? x0 : x1;
        T* dst = (cnt & 1) ? x1 : x0;
        const double om = mode == MODE_CHEBYSHEV ? cheb_omega_host(cnt, cheb_rho) : 1.0;
        SweepArgs<T> a = args(src, dst, f, alpha, (T)om, done);
        a.two_slot = (cnt & 1) ? 0 : 1;      // x0 owns coarse slot 0, x1 slot 1
        if (mode == MODE_CHEBYSHEV && !d.shared_coe) { a.rho_ps = rho_dev; a.cheb_k = cnt; }
        if (launch_sweep(a, mode, check && cnt == end, s)) return 1;
      }
      kernel_launches += k;
    }
    sweep_launches += k;
    return 0;
  }

  // ---- line2_mixed (xee_mixed.cuh)
  float* mixed_e(int buf) const { return reinterpret_cast<float*>(x1) + (size_t)buf * nn * d.nbatch; }
  // fp32 sweep number k (1 .. kcheck) of the current refinement step: buffer e(b) owns coarse slot b, sweep k reads e(k & 1)
  int mixed_sweep(int k, const int* done, cudaStream_t s) {
    LineArgs<float> A; LineLaunch L;
    const int slot = k & 1;
    if (line_setup<float>(mixed_e(slot), mixed_e(slot ^ 1), mx_r32, d.nbatch, slot, done, linepack32, A, L)) return 1;
    A.alpha = 1.f; A.omega = (float)cheb_omega_host(k, cheb_rho); A.cheb_k = k;
    A.rho_ps = d.shared_coe ? nullptr : mx_rho;
    if (launch_line_inst<float, true, false, true>(A, L.grid, L.cx, L.cxm, L.cf, L.co, s)) return 1;
    XEE_LAUNCH_OK();
    return two_coarse(slot ^ 1, d.nbatch, -(double)A.omega * tl_gamma, A.rho_ps, k, done, s);
  }
  // psi += s (e + P c) with the iterate of the step's last sweep (k sweeps into the step: buffer and slot (k + 1) & 1), then
  // e = c = 0 for the next step
  int mixed_fold(T* x0, int k, const int* done, cudaStream_t s) {
    const dim3 g((((d.nx + 7) / 8) * d.ny + 255) / 256, 1, d.nbatch);
    const int last = (k + 1) & 1;
    mx::mixed_fold_kernel<<<g, 256, 0, s>>>(reinterpret_cast<double*>(x0), mixed_e(last), mixed_e(0), two_cv(last, d.nbatch), mx_scale,
                                            done, d.nx, d.ny, d.nbatch, tld.px, tld.pz * tld.px);
    XEE_LAUNCH_OK();
    return two_reset(s);
  }
  // r = f - L psi: Sum r^2 per tile into `partial`; write_r32: also r32 = r / s' and the scales move on
  int mixed_residual(const T* x0, const T* f, bool write_r32, const int* done, cudaStream_t s) {
    mx::mixed_residual_kernel<<<dim3(gx, gy, d.nbatch), dim3(mx::BX, mx::BY), 0, s>>>(
        reinterpret_cast<const double*>(x0), reinterpret_cast<const double*>(f), reinterpret_cast<const double*>(coe),
        d.shared_coe ? 0 : (long long)kPlanes * nn, d.nx, d.ny, mx_scale + d.nbatch, write_r32 ? mx_r32 : nullptr, partial, done);
    XEE_LAUNCH_OK();
    if (!write_r32) return 0;
    mx::mixed_scale_kernel<<<d.nbatch, 128, 0, s>>>(partial, ntiles, (d.nx - 2) * (d.ny - 2), mx_scale, d.nbatch, 1, done);
    XEE_LAUNCH_OK();
    return 0;
  }
  // end of a refinement step: fold, then the residual of the new iterate (the check partials) and the next step's r32
  int mixed_check(T* x0, const T* f, const int* done, cudaStream_t s) {
    return mixed_fold(x0, kcheck, done, s) || mixed_residual(x0, f, true, done, s);
  }
  // Start of a solve or of sweeps(): e = c = 0, the scale from the first guess's residual, then the first r32.
  int mixed_begin(const T* x0, const T* f, const int* done, cudaStream_t s) {
    XEE_CHECK(cudaMemsetAsync(x1, 0, sizeof(T) * nn * d.nbatch, s));
    if (two_reset(s) || mixed_residual(x0, f, false, done, s)) return 1;
    mx::mixed_scale_kernel<<<d.nbatch, 128, 0, s>>>(partial, ntiles, (d.nx - 2) * (d.ny - 2), mx_scale, d.nbatch, 0, done);
    XEE_LAUNCH_OK();
    if (!d.shared_coe) {   // the per-solve Chebyshev radii as the fp32 sweeps and their coarse scaling read them
      mx_rho_h.resize(nsets);
      for (int n = 0; n < nsets; ++n) mx_rho_h[n] = (float)rho_ps[n];
      XEE_CHECK(cudaMemcpyAsync(mx_rho, mx_rho_h.data(), sizeof(float) * nsets, cudaMemcpyHostToDevice, s));
    }
    return mixed_residual(x0, f, true, done, s);
  }

  // ---- BiCGStab (xee_krylov.cuh)
  kr::Args<T> krylov_args(const int* done) const {
    kr::Args<T> a{};
    a.coe = coe; a.coe_set_stride = d.shared_coe ? 0 : (long long)kPlanes * nn; a.nn = (long long)nn;
    a.nx = d.nx; a.ny = d.ny; a.done = done; a.part = kpart; a.partial = partial; a.v = kv;
    return a;
  }
  // ph = K^-1 v: one Jacobi-mode v5 sweep with alpha 1 from the zero field x1 (its coarse slot 0 stays zero), f = v, plus
  // the coarse correction it leaves in slot 1
  int krylov_precond(const T* v, const int* done, cudaStream_t s) {
    SweepArgs<T> a = args(x1, kv.ph, v, T(1), T(1), done);
    a.two_slot = 0;
    if (launch_sweep_line(a, MODE_JACOBI, false, s)) return 1;
    if (use_two) {
      const dim3 g((((d.nx + 7) / 8) * d.ny + 255) / 256, 1, d.nbatch);
      tl::prolong_add_kernel<T><<<g, 256, 0, s>>>(kv.ph, two_cv(1, d.nbatch), done, d.nx, d.ny, tld.px, tld.pz * tld.px);
      XEE_LAUNCH_OK();
    }
    return 0;
  }
  int krylov_finish(int stage, const int* done, cudaStream_t s) {
    kr::finish_kernel<<<d.nbatch, 128, 0, s>>>(ksc, kpart, ntiles, done, stage);
    XEE_LAUNCH_OK();
    return 0;
  }
  // r = f - L x; the start of a solve also sets r0 = p = r
  int krylov_residual(const T* x, const T* f, const int* done, bool start, cudaStream_t s) {
    kr::residual_kernel<T><<<dim3(gx, gy, d.nbatch), dim3(kr::BX, kr::BY), 0, s>>>(krylov_args(done), x, f);
    XEE_LAUNCH_OK();
    if (!start) return 0;
    if (krylov_finish(kr::STAGE_START, done, s)) return 1;
    kr::p_kernel<T><<<dim3(gx, gy, d.nbatch), dim3(kr::BX, kr::BY), 0, s>>>(krylov_args(done), ksc);
    XEE_LAUNCH_OK();
    return 0;
  }
  // Start of a solve or of sweeps(): the vectors' rims and the zero field the preconditioner starts from, then r0 = p = r.
  int krylov_begin(const T* x, const T* f, const int* done, cudaStream_t s) {
    T* const bufs[8] = {x1, kv.r, kv.r0, kv.p, kv.ph, kv.s, kv.v, kv.t};
    for (T* v : bufs) XEE_CHECK(cudaMemsetAsync(v, 0, sizeof(T) * nn * d.nbatch, s));
    if (use_two && two_reset(s)) return 1;
    return krylov_residual(x, f, done, true, s);
  }
  // One iteration of every solve that is not done; `replace`: a check iteration (true residual, check partials)
  int krylov_iteration(T* x, const T* f, bool replace, const int* done, cudaStream_t s) {
    const dim3 g(gx, gy, d.nbatch), b(kr::BX, kr::BY);
    const kr::Args<T> A = krylov_args(done);
    if (krylov_precond(kv.p, done, s)) return 1;
    kr::apply_dot_kernel<T><<<g, b, 0, s>>>(A);
    XEE_LAUNCH_OK();
    if (krylov_finish(kr::STAGE_ALPHA, done, s)) return 1;
    kr::s_kernel<T><<<g, b, 0, s>>>(A, ksc, x);
    XEE_LAUNCH_OK();
    if (krylov_precond(kv.s, done, s)) return 1;
    kr::t_kernel<T><<<g, b, 0, s>>>(A);
    XEE_LAUNCH_OK();
    if (krylov_finish(kr::STAGE_OMEGA, done, s)) return 1;
    kr::update_kernel<T><<<g, b, 0, s>>>(A, ksc, x);
    XEE_LAUNCH_OK();
    if (replace && krylov_residual(x, f, done, false, s)) return 1;
    if (krylov_finish(kr::STAGE_RHO, done, s)) return 1;
    kr::p_kernel<T><<<g, b, 0, s>>>(A, ksc);
    XEE_LAUNCH_OK();
    return 0;
  }

  cudaEvent_t next_event() {
    if (ev_used == ev_pool.size()) {
      cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e);
    }
    return ev_pool[ev_used++];
  }
  void harvest_events() {  // pairs (begin,end) around runs of sweep launches
    for (size_t k = 0; k + 1 < ev_used; k += 2) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ev_pool[k], ev_pool[k + 1]) == cudaSuccess) sweep_ms += ms;
    }
    ev_used = 0;
  }

  int apply(const void* psi, void* out, cudaStream_t s) override {
    SweepArgs<T> a = args((const T*)psi, nullptr, nullptr, T(1), T(1), nullptr);
    a.apply_out = (T*)out;
    XEE_CHECK(cudaMemsetAsync(out, 0, sizeof(T) * nn * d.nbatch, s));
    return launch_sweep(a, MODE_APPLY, false, s);
  }

  // v3 resident solver (one cooperative launch per solve_elliptic call); see xee_resident.cuh
  int res_G = 0, res_P = 0;          // strips per solve, points per thread (0 = does not fit)
  T *res_final = nullptr, *res_prev = nullptr, *res_halo = nullptr;
  int* res_ints = nullptr;           // flags[nb*G] | check_cnt[nb] | abort[1]
  T* res_omega = nullptr;            // Chebyshev weights omega_1..omega_kChebClamp
  double* res_partial = nullptr;
  bool resident_fits() {
    if (res_G) return res_P > 0;
    const int rows = d.ny - 2, w = d.nx - 2;
    int G = std::min(num_sms / std::max(1, d.nbatch), rows);
    if (G < 1) { res_G = 1; res_P = 0; return false; }
    const int rows_max = (rows + G - 1) / G;
    const long long pts = (long long)rows_max * w;
    res_G = G;
    res_P = pts <= 512 ? 1 : pts <= 2 * 512 ? 2 : pts <= 3 * 512 ? 3 : 0;       // 512 threads x P points (1024 x 1 measured slower)
    if ((size_t)(rows_max + 2) * d.nx * sizeof(T) > 200 * 1024) res_P = 0;
    return res_P > 0;
  }
  template <int ARITH, int MODE, int P, int NT>
  int launch_resident(res::ResArgs<T>& ra, cudaStream_t s) {
    auto kern = res::solve_resident_kernel<T, ARITH, MODE, P, NT>;
    const int rows_max = (d.ny - 2 + res_G - 1) / res_G;
    const size_t smem = (size_t)(rows_max + 2) * d.nx * sizeof(T);
    XEE_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    XEE_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NT, smem));
    if ((long long)per_sm * num_sms < (long long)res_G * d.nbatch) return fail("xee: resident solver does not fit on the device (co-residency)");
    void* params[] = {(void*)&ra};
    XEE_CHECK(cudaLaunchCooperativeKernel((void*)kern, dim3(res_G, d.nbatch), dim3(NT), params, smem, s));
    XEE_LAUNCH_OK();
    return 0;
  }
  int solve_resident(T* x0, const T* fd, const xee_solve_params* prm, int check_step, int converge_time, int lost_rate, int mode,
                     int detect_explode, cudaStream_t s);
  int estimate_rho(cudaStream_t s);
  int estimate_rho_subsampled(cudaStream_t s);
  std::vector<double> lmin_ps;       // two-level: per-set smallest eigenvalue of M^-1 L (host copy, for the subsampled estimate)
  std::vector<double> radius_ps;     // per-set spectral radius rho (rho_ps holds the focal distance the weights are computed from)
  // Per-set Chebyshev parameters to rho_dev; h receives them in T, the values the device computes with.
  int upload_rho(const std::vector<double>& v, std::vector<T>& h, cudaStream_t s) {
    if (!rho_dev) XEE_CHECK(own(&rho_dev, sizeof(T) * nsets));
    h.resize(nsets);
    for (int n = 0; n < nsets; ++n) h[n] = (T)v[n];
    XEE_CHECK(cudaMemcpyAsync(rho_dev, h.data(), sizeof(T) * nsets, cudaMemcpyHostToDevice, s));
    return 0;
  }
  // Two-level step length from the smallest eigenvalues lmin[n] of M^-1 L and the common largest one tl_lmax: one step from
  // the mean lmin, with which the spectrum of solve n lies in [1 - gamma lmax, 1 - gamma lmin_n]; rho[n] its radius.
  void two_step(const std::vector<double>& lmin, std::vector<double>& rho) {
    double mean = 0.0;
    for (int n = 0; n < nsets; ++n) mean += lmin[n] / nsets;
    lmin_ps = lmin;
    tl_lmin = mean;
    tl_gamma = 2.0 / (tl_lmax + tl_lmin);
    for (int n = 0; n < nsets; ++n) rho[n] = std::max(tl_gamma * tl_lmax - 1.0, 1.0 - tl_gamma * lmin[n]);
  }
  // Make the Chebyshev parameters of this call available: an explicit value for this call only, else the estimate of the
  // current operator, computed once and uploaded again when an earlier call replaced it with an explicit value.
  int prepare_cheb(double rho_given, cudaStream_t s) {
    if (rho_given > 0 && !use_two) {   // (the two-level methods also need the step length: they always estimate)
      rho_ps.assign(nsets, rho_given);
    } else if (!est_rho_ps.empty()) {
      if (rho_ps == est_rho_ps) return 0;
      rho_ps = est_rho_ps;
    } else {
      XEE_CHECK(cudaStreamSynchronize(s));
      const double t0 = TraceTimer::now();
      const bool sub = !d.shared_coe && rho_subsample > 1 && nsets >= 4 * rho_subsample;
      const int rc = sub ? estimate_rho_subsampled(s) : estimate_rho(s);      // synchronises the stream before it returns
      probe_ms += (TraceTimer::now() - t0) * 1e3;
      if (rc == 0) est_rho_ps = rho_ps;
      return rc;
    }
    cheb_rho = rho_ps[0];
    std::vector<T> h;
    if (upload_rho(rho_ps, h, s)) return 1;
    XEE_CHECK(cudaStreamSynchronize(s));
    return 0;
  }

  int sweeps(void* psi, const void* f, double alpha, int nsw, int check_step, double* rms, cudaStream_t s) override {
    T* x0 = (T*)psi;
    kcheck = check_step > 0 ? check_step : 100;
    const int mode = method_is_cheb() ? MODE_CHEBYSHEV : MODE_JACOBI;
    if (mode == MODE_CHEBYSHEV && prepare_cheb(0.0, s)) return 1;   // before the start event: the spectral probe is not sweep time
    if (!use_mixed && seed_buffers(x0, (const T*)f, s)) return 1;
    cheb_rho_used = cheb_rho; cheb_gamma_used = use_two ? tl_gamma : 1.0;
    cudaEvent_t e0 = next_event(), e1 = next_event();
    XEE_CHECK(cudaEventRecord(e0, s));
    if (use_two && two_reset(s)) return 1;
    if (use_krylov && krylov_begin(x0, (const T*)f, nullptr, s)) return 1;
    if (use_mixed && mixed_begin(x0, (const T*)f, nullptr, s)) return 1;
    int tb_pass = 0;
    if (run_sweeps(x0, (const T*)f, (T)alpha, mode, 0, nsw, rms != nullptr, nullptr, tb_pass, s)) return 1;
    variant_used = use_line ? 5 : use_tb ? 4 : use_tma ? 2 : 1; depth_used = use_tb ? tb_depth : 1;
    if (use_mixed) {    // a partial last step is applied as a solve that reaches max_iter inside a step applies it
      if (nsw % kcheck && (mixed_fold(x0, nsw % kcheck, nullptr, s) || (rms && mixed_residual(x0, (const T*)f, false, nullptr, s)))) return 1;
      XEE_CHECK(cudaEventRecord(e1, s));
    } else if (use_krylov) {   // the iterate is x0 itself; rms: the true residual after the last iteration
      if (rms && krylov_residual(x0, (const T*)f, nullptr, false, s)) return 1;
      XEE_CHECK(cudaEventRecord(e1, s));
    } else {
      if (use_two && two_flush(x0, x1, d.nbatch, s)) return 1;
      XEE_CHECK(cudaEventRecord(e1, s));
      // the last iterate: v4 leaves it in the pair (x2, x3) after an odd number of passes, the others in x1 after an odd sweep count
      if (use_tb ? (tb_pass & 1) : (nsw & 1)) XEE_CHECK(cudaMemcpyAsync(x0, use_tb ? x2 : x1, sizeof(T) * nn * d.nbatch, cudaMemcpyDeviceToDevice, s));
    }
    XEE_CHECK(cudaStreamSynchronize(s));
    harvest_events();
    if (rms && nsw > 0) {
      const int nt = check_ntiles();
      std::vector<double> h((size_t)nt * d.nbatch);
      XEE_CHECK(cudaMemcpy(h.data(), partial, sizeof(double) * h.size(), cudaMemcpyDeviceToHost));
      const double N = (double)(d.nx - 2) * (d.ny - 2);
      for (int n = 0; n < d.nbatch; ++n) {
        double t = 0;
        for (int q = 0; q < nt; ++q) t += h[(size_t)n * nt + q];
        rms[n] = std::sqrt(t / N);
      }
    }
    return 0;
  }

  int solve(void* psi, const void* f, const xee_solve_params* prm, int* iters, double* r1o, double* r2o, int* err,
            cudaStream_t s, bool host_io, void* workspace_host, int debug) override;
};

template <class T>
int Plan<T>::estimate_rho(cudaStream_t s) {
  TraceTimer tt("estimate_rho");
  // Spectral radius rho of the Jacobi iteration matrix G = I - D^-1 L of every operator set (1 for a shared
  // operator, nbatch for one operator per solve), on homogeneous probe problems (f = 0, zero boundary):
  //   stage A  power iteration from the lowest sine mode: rho_A = ||G^k e|| / ||G^(k-1) e||.  Norms are taken in
  //            the D-weighted inner product (D = -coe5 > 0): G is similar to a symmetric matrix through D^(1/2)
  //            (exactly so for B = 0 or constant B), so the quotient is a monotone UNDER-estimate of rho;
  //   stage B  Chebyshev probe (Hageman & Young's adaptive idea): iterate the homogeneous problem with the
  //            Chebyshev weights of the current estimate rho_E.  Modes inside [-rho_E, rho_E] are damped at the
  //            optimal rate, the dominant mode rho_1 > rho_E more slowly, so it soon dominates and the measured
  //            decay B between sweeps p and 2p gives rho_1 from  T_2p(x1)/T_p(x1) = B T_2p(xE)/T_p(xE),
  //            x1 = rho_1/rho_E, xE = 1/rho_E.  Repeated until the correction is below 2 % of 1 - rho.
  const int ns = nsets;
  T *e0 = nullptr, *e1 = nullptr, *zf = nullptr; double* nrm_d = nullptr;
  PoolBuf e0_buf, e1_buf, zf_buf, nrm_buf;
  // the probe changes the launch geometry (nbatch, gz, spb): restored on every exit path
  struct Restore {
    Plan<T>* p; int nb, gz, spb;
    ~Restore() { p->d.nbatch = nb; p->gz = gz; p->spb = spb; }
  } restore{this, d.nbatch, gz, spb};
  XEE_CHECK(e0_buf.alloc(&e0, sizeof(T) * nn * ns)); XEE_CHECK(e1_buf.alloc(&e1, sizeof(T) * nn * ns));
  XEE_CHECK(zf_buf.alloc(&zf, sizeof(T) * nn * ns)); XEE_CHECK(nrm_buf.alloc(&nrm_d, sizeof(double) * ns * kWnormParts));
  if (!rho_dev) XEE_CHECK(own(&rho_dev, sizeof(T) * ns));
  XEE_CHECK(cudaMemsetAsync(zf, 0, sizeof(T) * nn * ns, s));
  auto start_vector = [&](int kind) -> int {     // e0 = e1 = start vector of `kind` (probe_start_kernel) in every set
    probe_start_kernel<T><<<dim3((unsigned)((nn + 255) / 256), ns), 256, 0, s>>>(e0, d.nx, d.ny, (long long)nn, kind);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaMemcpyAsync(e1, e0, sizeof(T) * nn * ns, cudaMemcpyDeviceToDevice, s));
    return 0;
  };
  if (start_vector(0)) return 1;
  // probe launch geometry: `ns` solves through the direct kernel
  d.nbatch = ns; spb = 1; gz = ns;
  std::vector<double> nA(ns), nB(ns), rho(ns, 0.0);
  std::vector<T> rho_h(ns);
  std::vector<double> nrm_h((size_t)ns * kWnormParts);
  auto norms = [&](const T* x, std::vector<double>& out) -> int {
    wnorm_kernel<T><<<dim3(kWnormParts, ns), 256, 0, s>>>(x, coe, d.shared_coe ? 0 : (long long)kPlanes * nn, (long long)nn, nrm_d);
    XEE_LAUNCH_OK();
    XEE_CHECK(cudaMemcpyAsync(nrm_h.data(), nrm_d, sizeof(double) * ns * kWnormParts, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    for (int n = 0; n < ns; ++n) {
      double t = 0.0;
      for (int q = 0; q < kWnormParts; ++q) t += nrm_h[(size_t)n * kWnormParts + q];
      out[n] = std::sqrt(t);
    }
    return 0;
  };
  int rc = 0, parity = 0;   // current iterate lives in (parity ? e1 : e0)
  auto sweep = [&](int mode, int k) -> int {
    const T* src = parity ? e1 : e0; T* dst = parity ? e0 : e1;
    SweepArgs<T> a = args(src, dst, zf, (T)(use_two ? tl_gamma : 1.0), T(1), nullptr);
    a.nbatch = ns; a.rho_ps = rho_dev; a.cheb_k = k;
    if (use_two) {
      a.two_slot = parity;                  // e0 owns coarse slot 0, e1 slot 1
      if (d.shared_coe) {   // one shared operator: the host-computed weight goes to the sweep kernel AND scales the coarse correction
        a.rho_ps = nullptr;
        a.omega = mode == MODE_CHEBYSHEV ? (T)cheb_omega_host(k, (double)rho_h[0]) : T(1);
      }                     // (one operator per solve: both take the weight of solve n from rho_dev[n])
    }
    parity ^= 1;
    return launch_sweep(a, mode, false, s);
  };
  // two-level: the probe vectors are (stored field, coarse vector) pairs; norms and differences need them made explicit
  auto flush = [&]() -> int { return use_two ? two_flush(e0, e1, ns, s) : 0; };
  // one probe round: 2p Chebyshev sweeps from the current iterate, norms after p (nA) and after 2p (nB)
  auto cheb_round = [&](int p) -> int {
    int r = 0;
    for (int k = 1; k <= 2 * p && !r; ++k) {
      r = sweep(MODE_CHEBYSHEV, k);
      if (k == p || k == 2 * p) r = r || flush();
      if (k == p) r = r || norms(parity ? e1 : e0, nA);
      if (k == 2 * p) r = r || norms(parity ? e1 : e0, nB);
    }
    return r;
  };
  if (use_two && two_reset(s)) return 1;
  if (use_two) {
    // ---- two-level: the spectrum of M^-1 L (M^-1 = block lines + coarse space) is [lmin, lmax] with lmax around 2, possibly
    // above it, so the step length gamma is part of the method:  G = I - gamma M^-1 L,  gamma = 2 / (lmax + lmin),
    // rho = (lmax - lmin) / (lmax + lmin).
    // lmax: the block-line part alone is bounded by 2 (L and its block-diagonal part are diagonally dominant with the same
    // sign), but the modes just below 2 (oscillating in z) form a dense cluster in which a power iteration creeps (measured:
    // 1.90 after 40 and 1.98 after 160 iterations for a true 1.9986), and UNDER-estimating lmax makes the Chebyshev iteration
    // diverge.  So: lmax = 1.02 max(2, power-iteration estimate): the iteration is only there to catch a coarse space that
    // pushes an isolated eigenvalue above 2 (such a mode separates quickly).  Over-estimating lmax by 2 % costs 1 % in sweeps.
    // lmin: the estimator below on G with the provisional step gamma0 = 1 / lmax, whose spectrum [0, 1 - lmin/lmax] is
    // non-negative, so its dominant mode is the smooth one the probes look for.
    TraceTimer t1("  probe: largest eigenvalue");
    if (start_vector(1)) return 1;
    tl_gamma = 1.0;
    const int itL = ns > 1 ? 24 : 60;
    for (int k = 1; k <= itL && !rc; ++k) {
      const T* cur = parity ? e1 : e0;
      if (k == itL) rc = rc || norms(cur, nA);
      rc = rc || sweep(MODE_JACOBI, 1);                         // other = cur - M^-1 L cur   (parity now names `other`)
      rc = rc || flush();
      T* oth = parity ? e1 : e0; const T* was = parity ? e0 : e1;
      tl::diff_kernel<T><<<1024, 256, 0, s>>>(oth, was, nn * ns);     // other = other - cur = -M^-1 L cur
      XEE_LAUNCH_OK();
      if (k == itL) rc = rc || norms(oth, nB);
    }
    if (rc) return 1;
    double grow = 0.0;
    for (int n = 0; n < ns; ++n) grow = std::max(grow, nA[n] > 0 ? nB[n] / nA[n] : 0.0);
    tl_lmax = 1.02 * std::max(2.0, 1.01 * grow);      // one bound for every operator set: the step length gamma is common
    if (!(tl_lmax > 0.5 && tl_lmax < 8.0)) {
      char msg[200]; snprintf(msg, sizeof msg, "xee: two-level: largest eigenvalue estimate of M^-1 L out of range (%.6e)", tl_lmax);
      return fail(msg);
    }
    tl_gamma = 1.0 / tl_lmax;
    // restore the smooth start vector of stage A
    if (start_vector(0)) return 1;
    parity = 0;
  }
  // ---- stage A
  // probe lengths: the block-line splitting has a ~20x larger spectral gap than point Jacobi, so its modes separate in
  // proportionally fewer sweeps (64/64 measured: same sweep counts to tolerance as 200/200; 32/32 costs 2-3 % more sweeps)
  const int itA = use_two ? 32 : use_line ? 64 : 200;
  { TraceTimer t2("  probe: stage A");
  for (int k = 1; k <= itA && !rc; ++k) {
    rc = sweep(MODE_JACOBI, 1);
    if (k >= itA - 1) rc = rc || flush();
    if (k == itA - 1) rc = rc || norms(parity ? e1 : e0, nA);
    if (k == itA) rc = rc || norms(parity ? e1 : e0, nB);
  }
  }
  for (int n = 0; n < ns && !rc; ++n) {
    rho[n] = nA[n] > 0 ? nB[n] / nA[n] : 0.0;
    if (!(rho[n] > 0.0 && rho[n] < 1.0)) {
      char msg[320];
      snprintf(msg, sizeof msg, "xee: Jacobi spectral-radius estimate outside (0,1); operator not diagonally dominant? "
               "[set %d of %d: |G^%d e| = %.6e, |G^%d e| = %.6e, ratio %.9f, line=%d]", n, ns, itA - 1, nA[n], itA, nB[n], rho[n], (int)use_line);
      rc = fail(msg);
    }
  }
  // ---- stage B
  const int rounds = 4, p = itA;
  std::vector<char> settled(ns, 0);
  auto lncosh = [](double x) { return x + std::log1p(std::exp(-2.0 * x)) - M_LN2; };
  for (int r = 0; r < rounds && !rc; ++r) {
    TraceTimer t3("  probe: stage B round");
    if (upload_rho(rho, rho_h, s)) return 1;
    // restart the Chebyshev sequence from the current iterate: x_{-1} := x_0
    XEE_CHECK(cudaMemcpyAsync(parity ? e0 : e1, parity ? e1 : e0, sizeof(T) * nn * ns, cudaMemcpyDeviceToDevice, s));
    rc = cheb_round(p);
    if (rc) break;
    bool all_settled = true;
    for (int n = 0; n < ns; ++n) {
      if (settled[n]) continue;
      if (!(nA[n] > 1e-280) || !(nB[n] > 1e-280)) { settled[n] = 1; continue; }
      const double rE = (double)rho_h[n];          // the value the device actually used
      const double o = std::acosh(1.0 / rE);
      const double target = std::log(nB[n] / nA[n]) + lncosh(2.0 * p * o) - lncosh((double)p * o);
      auto g = [&](double a) { return lncosh(2.0 * p * a) - lncosh((double)p * a) - target; };
      if (g(0.0) >= 0.0) { settled[n] = 1; continue; }   // decays at the optimal rate: rho_E already covers rho_1
      double lo = 0.0, hi = o;
      if (g(hi) < 0.0) hi = 4.0 * o;
      for (int itb = 0; itb < 80; ++itb) { const double mid = 0.5 * (lo + hi); (g(mid) < 0.0 ? lo : hi) = mid; }
      const double rho_new = std::min(rE * std::cosh(0.5 * (lo + hi)), 1.0 - 1e-10);
      const double rel = std::fabs(rho_new - rE) / (1.0 - rE);
      rho[n] = rho_new;
      if (rel < 0.02) settled[n] = 1; else all_settled = false;
    }
    if (env_int("XEE_TRACE", 0)) {
      double worst = 0.0;
      for (int n = 0; n < ns; ++n) worst = std::max(worst, std::fabs(rho[n] - (double)rho_h[n]) / (1.0 - (double)rho_h[n]));
      fprintf(stderr, "xee: stage B round %d: 1 - rho[0] = %.4e, largest relative change of the gap %.3f\n", r, 1.0 - rho[0], worst);
    }
    if (all_settled) break;
  }
  if (rc) return 1;
  if (use_two) {   // rho[n] is the spectral radius of I - gamma0 M^-1 L_n: lmin_n = (1 - rho_n) / gamma0, then the final step and radii
    std::vector<double> lmin(ns);
    for (int n = 0; n < ns; ++n) lmin[n] = (1.0 - rho[n]) / tl_gamma;
    two_step(lmin, rho);
    if (env_int("XEE_TRACE", 0)) fprintf(stderr, "xee: two-level spectrum of M^-1 L: [%.4e, %.4f], gamma %.4f\n", tl_lmin, tl_lmax, tl_gamma);
  }
  // ---- stage C (line methods): complex eigenvalues.  With a strongly varying B the operator is not symmetric and the
  // iteration matrix of a LINE splitting can have a complex pair mu = +- i b (measured on the later snapshots of the time
  // series: b = 0.09 at |rho| = 0.9995; the point splitting keeps a real spectrum).  Chebyshev weights for the real interval
  // [-rho, rho] amplify such a mode by e^(asinh(b) - acosh(1/rho)) per sweep: divergence once b > sqrt(2 (1 - rho)).  The
  // spectrum then lies in the ellipse with semi-axes (rho, b), for which the same recurrence with the FOCAL distance
  // c = sqrt(rho^2 - b^2) in place of rho is the optimal choice (Manteuffel), convergence factor (rho + b) / (1 + sqrt(1 - c^2)).
  // b is measured like rho in stage B: homogeneous problem, rough start vector, decay between sweeps p and 2p against the
  // decay 1/T_k(1/c) that every mode inside the ellipse shows; repeated with the new c until the excess is gone.
  std::vector<double> foci(rho);
  radius_ps = rho;
  if (use_line) {
    const int pc = 64, roundsC = 3;
    uint32_t lcg = 12345u;
    std::vector<T> h(nn, T(0));
    for (int j = 1; j < d.ny - 1; ++j)
      for (int i = 1; i < d.nx - 1; ++i) { lcg = lcg * 1664525u + 1013904223u; h[(size_t)j * d.nx + i] = (T)((double)(lcg >> 8) / 8388608.0 - 1.0); }
    std::vector<char> doneC(ns, 0);
    for (int r = 0; r < roundsC && !rc; ++r) {
      TraceTimer t4("  probe: stage C round");
      if (upload_rho(foci, rho_h, s)) return 1;
      XEE_CHECK(cudaMemcpyAsync(e0, h.data(), sizeof(T) * nn, cudaMemcpyHostToDevice, s));      // one upload, replicated on the device
      if (ns > 1) { probe_replicate_kernel<T><<<dim3((unsigned)((nn + 255) / 256), ns - 1), 256, 0, s>>>(e0, (long long)nn); XEE_LAUNCH_OK(); }
      XEE_CHECK(cudaMemcpyAsync(e1, e0, sizeof(T) * nn * ns, cudaMemcpyDeviceToDevice, s));
      if (use_two && two_reset(s)) return 1;
      parity = 0;
      rc = cheb_round(pc);
      if (rc) break;
      bool all = true;
      for (int n = 0; n < ns; ++n) {
        if (doneC[n]) continue;
        if (!(nA[n] > 1e-280) || !(nB[n] > 1e-280) || !std::isfinite(nB[n])) { doneC[n] = 1; continue; }
        const double c = (double)rho_h[n], o = std::acosh(1.0 / c);
        const double excess = std::log(nB[n] / nA[n]) - (lncosh((double)pc * o) - lncosh(2.0 * pc * o));   // vs the decay of the modes inside
        if (excess < 0.7) { doneC[n] = 1; continue; }                 // within the scatter of a sum over many modes
        // the dominant outside mode multiplies its amplitude by e^(asinh(y)) per sweep, y = distance from the focal segment in
        // units of c along the imaginary axis; the ellipse through it keeps the real semi-axis rho
        const double y = std::sinh(excess / pc);
        const double bsq = (c * y) * (c * y) + (rho[n] * rho[n] - c * c);   // imaginary semi-axis of the new ellipse (squared)
        const double c2 = rho[n] * rho[n] - 1.21 * bsq;                       // 10 % margin on b
        foci[n] = std::sqrt(std::max(c2, 1e-4));
        all = false;
      }
      if (all) break;
    }
    if (rc) return 1;
    if (env_int("XEE_TRACE", 0)) {
      double worst = 0.0;
      for (int n = 0; n < ns; ++n) worst = std::max(worst, std::sqrt(std::max(rho[n] * rho[n] - foci[n] * foci[n], 0.0)));
      fprintf(stderr, "xee: largest imaginary semi-axis of the iteration spectrum: %.4f\n", worst);
    }
  }
  rho_ps = foci;   // what the Chebyshev weights are computed from
  if (upload_rho(foci, rho_h, s)) return 1;
  XEE_CHECK(cudaStreamSynchronize(s));
  cheb_rho = foci[0];
  if (env_int("XEE_TRACE", 0)) fprintf(stderr, "xee: Jacobi spectral radius estimate rho[0] = 1 - %.4e (%d operator set%s)\n", 1.0 - rho[0], ns, ns > 1 ? "s" : "");
  return 0;
}

// One operator per solve, operators varying smoothly with the solve index (a time series): the spectral probes run on every
// rho_subsample-th operator set only (a small plan of its own holding copies of those operators), and the quantity that
// drives the Chebyshev weights - the gap 1 - rho of the one-level methods, the smallest eigenvalue of M^-1 L of the two-level
// ones - is interpolated (log-linearly in the index) for the sets in between.  A wrong value costs sweeps, not correctness:
// the residual and the stop rule are those of every other method.
template <class T>
int Plan<T>::estimate_rho_subsampled(cudaStream_t s) {
  TraceTimer tt("estimate_rho (subsampled)");
  std::vector<int> idx;
  for (int n = 0; n < nsets; n += rho_subsample) idx.push_back(n);
  if (idx.back() != nsets - 1) idx.push_back(nsets - 1);
  const int nq = (int)idx.size();
  Plan<T> sub;
  sub.d = d; sub.d.nbatch = nq; sub.d.shared_coe = 0; sub.d.kernel = 0;
  if (sub.init()) return 1;
  XEE_CHECK(cudaStreamSynchronize(s));
  for (int q = 0; q < nq; ++q)
    XEE_CHECK(cudaMemcpyAsync(sub.coe + (size_t)q * kPlanes * nn, coe + (size_t)idx[q] * kPlanes * nn, sizeof(T) * kPlanes * nn, cudaMemcpyDeviceToDevice, sub.own_stream));
  XEE_CHECK(cudaStreamSynchronize(sub.own_stream));
  if (sub.line_factors()) return 1;
  if (sub.estimate_rho(sub.own_stream)) return 1;
  // the interpolated quantity at the sampled sets
  std::vector<double> v(nq);
  std::vector<double> bq(nq);       // imaginary semi-axis of the iteration spectrum at the sampled sets (stage C)
  for (int q = 0; q < nq; ++q) {
    v[q] = use_two ? sub.lmin_ps[q] : 1.0 - sub.radius_ps[q];
    bq[q] = std::sqrt(std::max(sub.radius_ps[q] * sub.radius_ps[q] - sub.rho_ps[q] * sub.rho_ps[q], 0.0));
  }
  for (int q = 0; q < nq; ++q)
    if (!(v[q] > 0.0)) return fail("xee: subsampled spectral estimate: non-positive gap");
  std::vector<double> rho(nsets), lmin(nsets), bim(nsets);
  for (int n = 0, q = 0; n < nsets; ++n) {
    while (q + 1 < nq - 1 && idx[q + 1] <= n) ++q;
    const double t = idx[q + 1] > idx[q] ? (double)(n - idx[q]) / (idx[q + 1] - idx[q]) : 0.0;
    lmin[n] = std::exp((1.0 - t) * std::log(v[q]) + t * std::log(v[q + 1]));
    bim[n] = std::max(bq[q], bq[q + 1]);        // the larger neighbour: an over-estimate costs sweeps, an under-estimate convergence
  }
  if (use_two) {
    tl_lmax = sub.tl_lmax;
    two_step(lmin, rho);
  } else {
    for (int n = 0; n < nsets; ++n) rho[n] = 1.0 - lmin[n];
  }
  radius_ps = rho;
  for (int n = 0; n < nsets; ++n) rho[n] = std::sqrt(std::max(rho[n] * rho[n] - bim[n] * bim[n], 1e-4));   // focal distances
  std::vector<T> rho_h;
  if (upload_rho(rho, rho_h, s)) return 1;
  XEE_CHECK(cudaStreamSynchronize(s));
  rho_ps = rho; cheb_rho = rho[0];
  if (env_int("XEE_TRACE", 0)) fprintf(stderr, "xee: subsampled spectral estimate: %d of %d operator sets probed, gap[0] = %.4e, gap[last] = %.4e\n", nq, nsets, lmin[0], lmin[nsets - 1]);
  return 0;
}

template <class T>
int Plan<T>::solve_resident(T* x0, const T* fd, const xee_solve_params* prm, int check_step, int converge_time,
                            int lost_rate, int mode, int detect_explode, cudaStream_t s) {
  const int nb = d.nbatch, G = res_G;
  const size_t fbytes = sizeof(T) * nn * nb;
  if (!res_final) {
    XEE_CHECK(own(&res_final, fbytes)); XEE_CHECK(own(&res_prev, fbytes));
    XEE_CHECK(own(&res_halo, sizeof(T) * (size_t)nb * 2 * G * 2 * d.nx));
    XEE_CHECK(own(&res_ints, sizeof(int) * ((size_t)nb * G * res::FLAG_PAD + 64 * nb + 64)));
    XEE_CHECK(own(&res_partial, sizeof(double) * (size_t)nb * 2 * G));
  }
  XEE_CHECK(cudaMemsetAsync(res_ints, 0, sizeof(int) * ((size_t)nb * G * res::FLAG_PAD + 64 * nb + 64), s));
  XEE_CHECK(cudaMemcpyAsync(res_final, x0, fbytes, cudaMemcpyDeviceToDevice, s));   // boundary values in both outputs
  XEE_CHECK(cudaMemcpyAsync(res_prev, x0, fbytes, cudaMemcpyDeviceToDevice, s));
  res::ResArgs<T> ra{};
  ra.psi0 = x0; ra.f = fd; ra.coe = coe;
  ra.coe_set_stride = d.shared_coe ? 0 : (long long)kPlanes * nn; ra.field_stride = (long long)nn;
  ra.out_final = res_final; ra.out_prev = res_prev; ra.halo = res_halo;
  ra.flags = res_ints; ra.check_cnt = res_ints + (size_t)nb * G * res::FLAG_PAD; ra.abort_flag = ra.check_cnt + 64 * nb;
  ra.partial = res_partial;
  ra.nx = d.nx; ra.ny = d.ny; ra.G = G;
  ra.max_iter = prm->max_iter; ra.check_step = check_step; ra.converge_time = converge_time; ra.lost_rate = lost_rate;
  ra.alpha = (T)prm->alpha; ra.rho = cheb_rho;
  if (mode == MODE_CHEBYSHEV) {   // host-computed weights, the same values the per-launch kernels receive
    if (!res_omega) XEE_CHECK(own(&res_omega, sizeof(T) * kChebClamp));
    std::vector<T> tab(kChebClamp);
    for (int k = 1; k <= kChebClamp; ++k) tab[k - 1] = (T)cheb_omega_host(k, cheb_rho);
    XEE_CHECK(cudaMemcpyAsync(res_omega, tab.data(), sizeof(T) * kChebClamp, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaStreamSynchronize(s));
  }
  ra.omega_tab = res_omega;
  ra.r1 = st.r1; ra.r2 = st.r2; ra.detect_explode = detect_explode; ra.stall_checks = prm->stall_checks;
  ra.iters = st.iters; ra.errb = st.errb; ra.err_now = st.err_now; ra.ratio = st.ratio;
  ra.trace_err = st.trace_err; ra.trace_ratio = st.trace_ratio; ra.trace_cap = st.trace_cap;
  const int rc = dispatch([&](auto strict, auto cheb) {
    constexpr int A = arith_of(strict), M = mode_of(cheb);
    return res_P == 1 ? launch_resident<A, M, 1, 512>(ra, s) : res_P == 2 ? launch_resident<A, M, 2, 512>(ra, s) : launch_resident<A, M, 3, 512>(ra, s);
  }, d.arith == XEE_ARITH_STRICT, mode == MODE_CHEBYSHEV);
  if (rc) return rc;
  // dat <- last iterate; the other buffer as the reference leaves `workspace` (penultimate iterate when the
  // sweep count is even, a copy of the result when it is odd: elliptic_tools.f90:259-264)
  XEE_CHECK(cudaMemcpyAsync(x0, res_final, fbytes, cudaMemcpyDeviceToDevice, s));
  std::vector<int> hi(nb);
  XEE_CHECK(cudaMemcpyAsync(hi.data(), st.iters, sizeof(int) * nb, cudaMemcpyDeviceToHost, s));
  XEE_CHECK(cudaStreamSynchronize(s));
  for (int n = 0; n < nb; ++n)
    XEE_CHECK(cudaMemcpyAsync(x1 + (size_t)n * nn, ((hi[n] & 1) ? res_final : res_prev) + (size_t)n * nn, sizeof(T) * nn, cudaMemcpyDeviceToDevice, s));
  return 0;
}

template <class T>
int Plan<T>::solve(void* psi, const void* f, const xee_solve_params* prm, int* iters, double* r1o, double* r2o,
                   int* err, cudaStream_t s, bool host_io, void* workspace_host, int debug) {
  const int nb = d.nbatch;
  const size_t fbytes = sizeof(T) * nn * nb;
  T* x0 = (T*)psi;
  const T* fd = (const T*)f;
  if (host_io) {
    if (!io_psi) { XEE_CHECK(own(&io_psi, fbytes)); XEE_CHECK(own(&io_f, fbytes)); }
    XEE_CHECK(cudaMemcpyAsync(io_psi, psi, fbytes, cudaMemcpyHostToDevice, s));
    XEE_CHECK(cudaMemcpyAsync(io_f, f, fbytes, cudaMemcpyHostToDevice, s));
    x0 = io_psi; fd = io_f;
  }
  const int check_step = prm->check_step > 0 ? prm->check_step : 100;          // :131-134
  const int converge_time = prm->converge_time > 0 ? prm->converge_time : 10;  // :136-139
  const int lost_rate = prm->lost_rate > 0 ? prm->lost_rate : 5;               // :141-144
  const int max_iter = prm->max_iter;
  const int mode = method_is_cheb() ? MODE_CHEBYSHEV : MODE_JACOBI;
  // an accelerated iteration with a wrong spectral estimate diverges: the explode rules always apply to it (err bit 1)
  const int detect_explode = prm->detect_explode || mode == MODE_CHEBYSHEV || use_krylov;
  if (mode == MODE_CHEBYSHEV) {
    if (prepare_cheb(prm->rho_jacobi, s)) return 1;
    cheb_rho_used = cheb_rho; cheb_gamma_used = use_two ? tl_gamma : 1.0;
  }
  init_state_kernel<T><<<(nb + 127) / 128, 128, 0, s>>>(st, nb, (T)prm->r1, (T)prm->r2, (const T*)prm->r1_per_solve);
  XEE_LAUNCH_OK();
  // v3: the whole loop in one cooperative launch (single / few solves that fit on the chip)
  int want_kernel = d.kernel > 0 ? d.kernel : env_int("XEE_KERNEL", 0);
  if (norm_max && (use_line || use_tb)) return fail("xee: the max-abs residual norm (legacy strategies 3/4) is provided for the point methods only");
  if (norm_max && !partial_max) XEE_CHECK(own(&partial_max, sizeof(double) * nb * kResmaxBlocks));
  const bool resident_ok = !norm_max && !use_line && (d.shared_coe || nb == 1) && max_iter >= 1 && resident_fits();
  if (want_kernel == 3 && !resident_ok) return fail("xee: kernel=3 (resident) needs a problem that fits: nbatch*strips <= SMs, <= 1536 points per strip");
  // the results: fields back to the host (host entry points), iters, err, r1 and r2 of every solve
  auto finish = [&](bool resident) -> int {
    if (host_io) {
      XEE_CHECK(cudaMemcpyAsync(psi, x0, fbytes, cudaMemcpyDeviceToHost, s));
      if (workspace_host) XEE_CHECK(cudaMemcpyAsync(workspace_host, x1, fbytes, cudaMemcpyDeviceToHost, s));
    }
    std::vector<int> hi(nb), he(nb);
    std::vector<T> h1(nb), h2(nb);
    XEE_CHECK(cudaMemcpyAsync(hi.data(), st.iters, sizeof(int) * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaMemcpyAsync(he.data(), st.errb, sizeof(int) * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaMemcpyAsync(h1.data(), st.err_now, sizeof(T) * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaMemcpyAsync(h2.data(), st.ratio, sizeof(T) * nb, cudaMemcpyDeviceToHost, s));
    XEE_CHECK(cudaStreamSynchronize(s));
    harvest_events();
    for (int n = 0; n < nb; ++n) {
      if (resident) {   // one launch ran every sweep of the solve
        if (he[n] & 0x100) return fail("xee: resident solver watchdog tripped (a CTA waited too long for its neighbour)");
        sweep_launches += hi[n];
      }
      if (iters) iters[n] = hi[n];
      if (err) err[n] = he[n];
      if (r1o) r1o[n] = (double)h1[n];
      if (r2o) r2o[n] = (double)h2[n];
    }
    if (resident && debug == 2) {   // the per-check lines of solve 0 (the loop below prints them as it goes)
      const int nchk = std::min(hi[0] / check_step, st.trace_cap);
      std::vector<T> te(nchk), tr(nchk);
      if (nchk > 0) {
        XEE_CHECK(cudaMemcpy(te.data(), st.trace_err, sizeof(T) * nchk, cudaMemcpyDeviceToHost));
        XEE_CHECK(cudaMemcpy(tr.data(), st.trace_ratio, sizeof(T) * nchk, cudaMemcpyDeviceToHost));
      }
      for (int q = 0; q < nchk; ++q) printf("Iter: %8d, err_now: %12.3E, ratio: %12.3E\n", (q + 1) * check_step, (double)te[q], (double)tr[q]);
    }
    return 0;
  };
  if (want_kernel == 3 || (want_kernel == 0 && resident_ok && nb <= 2)) {
    cudaEvent_t e0 = next_event(), e1 = next_event();
    XEE_CHECK(cudaEventRecord(e0, s));
    if (solve_resident(x0, fd, prm, check_step, converge_time, lost_rate, mode, detect_explode, s)) return 1;
    ++kernel_launches; variant_used = 3; depth_used = 1;
    XEE_CHECK(cudaEventRecord(e1, s));
    return finish(true);
  }
  if (!use_mixed && seed_buffers(x0, fd, s)) return 1;
  if (use_two && two_reset(s)) return 1;
  kcheck = check_step;
  if (use_krylov && krylov_begin(x0, fd, st.done, s)) return 1;
  if (use_mixed && mixed_begin(x0, fd, st.done, s)) return 1;
  int tb_pass = 0;
  variant_used = use_line ? 5 : use_tb ? 4 : use_tma ? 2 : 1; depth_used = use_tb ? tb_depth : 1;
  const int ninterior = (d.nx - 2) * (d.ny - 2);
  const int lookahead = prm->sync_every > 0 ? prm->sync_every : 1;
  int cnt = 0, check_idx = 0, printed = 0;
  int pending = 0;  // checks issued whose active-count has not been read yet
  bool all_done = false;
  std::vector<T> tr_e, tr_r;
  while (cnt < max_iter && !all_done) {
    const int to_check = check_step - (cnt % check_step);
    const int chunk = std::min(to_check, max_iter - cnt);
    cudaEvent_t e0 = next_event(), e1 = next_event();
    XEE_CHECK(cudaEventRecord(e0, s));
    const bool check = ((cnt + chunk) % check_step) == 0;                        // :179-183
    if (run_sweeps(x0, fd, (T)prm->alpha, mode, cnt, chunk, check, st.done, tb_pass, s)) return 1;
    cnt += chunk;
    XEE_CHECK(cudaEventRecord(e1, s));
    if (check) {
      if (norm_max) {   // the residual of the iterate this check sweep read (it is still in its buffer), in the max norm
        const T* src = (cnt & 1) ? x0 : x1;
        dispatch([&](auto strict) {
          resmax_kernel<T, arith_of(strict)><<<dim3(kResmaxBlocks, nb), 256, 0, s>>>(src, fd, coe, d.shared_coe ? 0 : (long long)kPlanes * nn,
                                                                                    (long long)nn, d.nx, d.ny, st.done, partial_max);
          return 0;
        }, d.arith == XEE_ARITH_STRICT);
        XEE_LAUNCH_OK();
      }
      finalize_check_kernel<T><<<nb, 128, 0, s>>>(st, norm_max ? partial_max : partial, norm_max ? kResmaxBlocks : check_ntiles(),
                                                  ninterior, cnt, check_idx, converge_time, lost_rate, max_iter,
                                                  detect_explode, prm->stall_checks, norm_max, norm_floor);
      XEE_LAUNCH_OK();
      const int slot = check_idx & 3;
      XEE_CHECK(cudaMemcpyAsync(&h_active[slot], st.active, sizeof(int), cudaMemcpyDeviceToHost, s));
      XEE_CHECK(cudaEventRecord(poll_ev[slot], s));
      ++check_idx; ++pending;
      // Keep at most `lookahead` (<= 3) checks in flight; read the oldest outstanding one.
      const int depth = std::min(lookahead, 3);
      while (pending >= depth && !all_done) {
        const int rs = (check_idx - pending) & 3;
        XEE_CHECK(cudaEventSynchronize(poll_ev[rs]));
        if (h_active[rs] <= 0) all_done = true;
        --pending;
      }
      if (debug == 2) {  // per-check line of elliptic_tools.f90:202-204 for solve 0
        XEE_CHECK(cudaStreamSynchronize(s));
        const int upto = std::min(check_idx, st.trace_cap);
        tr_e.resize(upto); tr_r.resize(upto);
        XEE_CHECK(cudaMemcpy(tr_e.data(), st.trace_err, sizeof(T) * upto, cudaMemcpyDeviceToHost));
        XEE_CHECK(cudaMemcpy(tr_r.data(), st.trace_ratio, sizeof(T) * upto, cudaMemcpyDeviceToHost));
        for (; printed < upto; ++printed)
          printf("Iter: %8d, err_now: %12.3E, ratio: %12.3E\n", (printed + 1) * check_step, (double)tr_e[printed], (double)tr_r[printed]);
      }
    }
    if (ev_used > 4096) { XEE_CHECK(cudaStreamSynchronize(s)); harvest_events(); }
  }
  if (!all_done) {  // max_iter exhausted (possibly on a non-check sweep)
    if (use_mixed && cnt % check_step && mixed_fold(x0, cnt % check_step, st.done, s)) return 1;   // the partial last step
    finalize_maxiter_kernel<T><<<(nb + 127) / 128, 128, 0, s>>>(st, nb, max_iter);
    XEE_LAUNCH_OK();
  }
  if (use_krylov || use_mixed) {   // the result is x0 itself; `workspace` receives a copy of it
    XEE_CHECK(cudaMemcpyAsync(x1, x0, fbytes, cudaMemcpyDeviceToDevice, s));
    return finish(false);
  }
  if (use_two && two_flush(x0, x1, nb, s)) return 1;    // psi = y + P c in both buffers (final and penultimate iterate of every solve)
  dim3 g((unsigned)std::min<size_t>((nn + 255) / 256, 64), nb);
  if (use_tb) select_result_tb_kernel<T><<<g, 256, 0, s>>>(x0, x1, x2, x3, st.iters, (long long)nn, check_step, tb_depth);
  else select_result_kernel<T><<<g, 256, 0, s>>>(x0, x1, st.iters, (long long)nn, 1);
  XEE_LAUNCH_OK();
  return finish(false);
}

inline int make_plan(const xee_plan_desc* desc, std::unique_ptr<PlanBase>* out) {
  int dev = 0;
  if (resolve_device(desc->device, &dev)) return 1;
  if (desc->nx < 3 || desc->ny < 3 || desc->nbatch < 1) return fail("xee: nx, ny >= 3 and nbatch >= 1 required");
  DeviceGuard guard(dev);
  std::unique_ptr<PlanBase> p;
  int rc;
  if (desc->dtype == XEE_F32) { auto* q = new Plan<float>(); p.reset(q); q->d = *desc; q->d.device = dev; rc = q->init(); }
  else if (desc->dtype == XEE_F64) { auto* q = new Plan<double>(); p.reset(q); q->d = *desc; q->d.device = dev; rc = q->init(); }
  else return fail("xee: dtype must be XEE_F32 or XEE_F64");
  if (rc) return 1;
  *out = std::move(p);
  return 0;
}

}  // namespace xee


/* xee_b200.h — C-ABI of the B200-native elliptic-solve hot path of XLab-EE-fortran.
 *
 * The reference (meteorologytoday/XLab-EE-fortran) has NO C ABI of its own: the hot
 * path is the Fortran module `elliptic_tools` (xtt-lib-fortran/elliptic_tools.f90),
 * called from src/diagnose/diagnose.f90:7,15,34,42.  This header is what a
 * `bind(C)` interface block in a replacement `module elliptic_tools` binds to
 * (fortran/elliptic_tools.f90 in this repo; INTEGRATION.md shows the stub).
 *
 * Part 1 mirrors the module procedures one to one (Fortran conventions: every
 * argument by reference, default INTEGER = 32 bit, arrays column-major and
 * contiguous, HOST pointers, synchronous).  Part 2 is the batched device API the
 * efficiency-map / time-series callers use (plain pointers and sizes only).
 *
 * All compute runs in hand-written CUDA for sm_100a.  There is no CPU fallback:
 * every entry point fails loudly (message on stderr + non-zero status / abort for
 * the Fortran-style void entry points) when no CUDA device is usable.
 */
#ifndef XEE_B200_H
#define XEE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* elliptic_tools.f90:3-4 — public error bits of the `err` bitmask */
#define XEE_ERR_OVER_MAX_ITERATION 1
#define XEE_ERR_EXPLODE 2
/* Not in the reference (batched API only, opt-in through xee_solve_params.stall_checks): the residual stopped
 * improving before r1 was reached - the solve sits on its round-off floor. */
#define XEE_ERR_STALLED 4

/* =====================================================================================
 * Part 1 — drop-in for `module elliptic_tools` (+ the driver's FD post-processing)
 * ===================================================================================== */

/* cal_coe(a,b,c,workspace,dx,dy,nx,ny,err)            elliptic_tools.f90:8-60
 * a(nx-1,ny-2) b(nx-1,ny-1) c(nx-2,ny-1) -> coe(9,nx,ny).  Only interior entries
 * (2..nx-1, 2..ny-1) of coe are written, as in the reference.  err: 0 on return. */
void xee_cal_coe_f32(const float* a, const float* b, const float* c, float* coe, const float* dx,
                     const float* dy, const int* nx, const int* ny, int* err);
void xee_cal_coe_f64(const double* a, const double* b, const double* c, double* coe, const double* dx,
                     const double* dy, const int* nx, const int* ny, int* err);

/* do_elliptic(psi,coe,outdat,nx,ny,err)               elliptic_tools.f90:64-90
 * outdat interior = 9-point apply; boundary of outdat untouched; err = 1 on
 * return (the reference sets it to 1 at :73 and never clears it). */
void xee_do_elliptic_f32(const float* psi, const float* coe, float* outdat, const int* nx, const int* ny, int* err);
void xee_do_elliptic_f64(const double* psi, const double* coe, double* outdat, const int* nx, const int* ny, int* err);

/* solve_elliptic(max_iter,check_step,converge_time,lost_rate,strategy_r1,strategy_r2,
 *                alpha,dat,coe,f,workspace,nx,ny,err,debug)   elliptic_tools.f90:93-265
 * Weighted-Jacobi relaxation with the reference's stop-rule state machine.
 * In/out: max_iter (sweeps used), strategy_r1 (last RMS residual), strategy_r2 (last
 * |ratio|), dat (boundary + first guess in, solution out).  workspace: scratch, left as
 * the reference leaves it (the other ping-pong buffer).  err: bitmask (bit 0 = max_iter
 * hit).  Both criteria non-positive: prints the reference's message and stops the
 * process like Fortran STOP (exit status 0), elliptic_tools.f90:126-129.
 * Environment: XEE_ARITH=strict|fast (default strict: no FMA contraction, true division,
 * iterates bit-identical to the reference's operation order); XEE_METHOD=jacobi|chebyshev|line_jacobi|line_chebyshev|
 * line2_jacobi|line2_chebyshev|line_bicgstab|line2_bicgstab|line2_mixed (default jacobi, the reference's iteration). */
void xee_solve_elliptic_f32(int* max_iter, const int* check_step, const int* converge_time, const int* lost_rate,
                            float* strategy_r1, float* strategy_r2, const float* alpha, float* dat,
                            const float* coe, const float* f, float* workspace, const int* nx, const int* ny,
                            int* err, const int* debug);
void xee_solve_elliptic_f64(int* max_iter, const int* check_step, const int* converge_time, const int* lost_rate,
                            double* strategy_r1, double* strategy_r2, const double* alpha, double* dat,
                            const double* coe, const double* f, double* workspace, const int* nx, const int* ny,
                            int* err, const int* debug);

/* LEGACY signature: solve_elliptic(max_iter, strategy, strategy_r, alpha, dat, coe, f, workspace, nx, ny, err, debug)
 * src/old-diagnose/xtt-lib/elliptic_tools.f90:93-300, called nine times by src/old-diagnose/diagnose.f90:449-714.
 * strategy 1: stop when the RMS residual < strategy_r at a check (every 100 sweeps); strategy 2: stop when the relative
 * change of the residual stays < strategy_r for 10 checks (hysteresis 5).  On return strategy = sweeps used,
 * strategy_r = last residual.  Strategies 3 / 4: the same two rules with the residual measured as maxval(abs(to_dat)) (:203-204) -
 * the largest |L psi - f| of the interior joined with the largest |boundary value| of dat; point methods only.
 * As in the legacy code, max_iter is only honoured on check sweeps (multiples of 100). */
void xee_solve_elliptic_old_f32(const int* max_iter, int* strategy, float* strategy_r, const float* alpha, float* dat,
                                const float* coe, const float* f, float* workspace, const int* nx, const int* ny,
                                int* err, const int* debug);
void xee_solve_elliptic_old_f64(const int* max_iter, int* strategy, double* strategy_r, const double* alpha, double* dat,
                                const double* coe, const double* f, double* workspace, const int* nx, const int* ny,
                                int* err, const int* debug);

/* judge_error(err)                                     elliptic_tools.f90:333-358 */
void xee_judge_error(const int* err);

/* a/b/c normalisation                                  src/diagnose/initialize-variables.f90:72-95
 * A,B,C on O(nr,nz); rcuva(nr), rho(nz) -> a sA(nr-1,nz-2), b B(nr-1,nz-1), c sC(nr-2,nz-1) */
void xee_build_abc_f32(const float* A, const float* B, const float* C, const float* rcuva, const float* rho,
                       float* a, float* b, float* c, const int* nr, const int* nz);
void xee_build_abc_f64(const double* A, const double* B, const double* C, const double* rcuva, const double* rho,
                       double* a, double* b, double* c, const int* nr, const int* nz);

/* cal_eta(rchi,eta)                                    src/diagnose/quick-tools1.f90:1-13
 * host-associated driver variables (ra, rcuva, rho, exner) become explicit arguments. */
void xee_cal_eta_f32(const float* rchi, float* eta, const float* ra, const float* rcuva, const float* rho,
                     const float* exner, const int* nr, const int* nz);
void xee_cal_eta_f64(const double* rchi, double* eta, const double* ra, const double* rcuva, const double* rho,
                     const double* exner, const int* nr, const int* nz);

/* cal_uw(from_rpsi,to_u,to_w)                          src/diagnose/quick-tools1.f90:15-41 */
void xee_cal_uw_f32(const float* rpsi, float* u, float* w, const float* ra, const float* rcuva, const float* za,
                    const float* rho, const int* nr, const int* nz);
void xee_cal_uw_f64(const double* rpsi, double* u, double* w, const double* ra, const double* rcuva,
                    const double* za, const double* rho, const int* nr, const int* nz);

/* =====================================================================================
 * Part 2 — batched device API (new; not in the reference).  Status codes: 0 = ok.
 * ===================================================================================== */
#define XEE_F32 0
#define XEE_F64 1
#define XEE_ARITH_STRICT 0 /* reference operation order, no FMA, true division          */
#define XEE_ARITH_FAST 1   /* FMA + precomputed reciprocal (same fixed point, 1e-13 rel) */
#define XEE_METHOD_JACOBI 0    /* the reference's weighted Jacobi                        */
#define XEE_METHOD_CHEBYSHEV 1 /* Chebyshev-accelerated Jacobi (same residual definition)*/
/* Block-line relaxation along the radius (not in the reference): same discrete problem, residual and stop rule, but
 * the correction solves coe4 z(i-1) + coe5 z(i) + coe6 z(i+1) = r(i) exactly on aligned BLOCKS OF 32 radial points
 * (four 8-point thread segments coupled through a precomputed reduced system) instead of dividing r by coe5.
 * Shared operator or one operator per solve; FAST arithmetic only; sweep kernel 5. */
#define XEE_METHOD_LINE_JACOBI 2
#define XEE_METHOD_LINE_CHEBYSHEV 3
/* Two-level block-line relaxation (not in the reference): the block-line correction PLUS a coarse-grid correction
 * P Ac^-1 P^T r (bilinear coarse space, nodes every 16 grid points, Galerkin Ac = P^T L P inverted once per operator);
 * same discrete problem, residual and stop rule.  Shared operator, FAST arithmetic, grids of at least 34 x 34 points. */
#define XEE_METHOD_LINE2_JACOBI 4
#define XEE_METHOD_LINE2_CHEBYSHEV 5
/* Right-preconditioned BiCGStab on L (not in the reference) with the block-line (LINE_) or the two-level (LINE2_)
 * preconditioner: no spectral estimate, no assumption of a real spectrum.  iters, max_iter and check_step count iterations
 * (two preconditioner sweeps and two operator applications each); a check computes the true residual L psi - f, feeds the
 * unchanged stop rule and replaces the recurrence residual; a breakdown restarts the solve from its current iterate.
 * alpha and rho_jacobi are ignored, detect_explode is always on.  Configurations as the Chebyshev counterparts: shared
 * operator or one per solve, FAST arithmetic, sweep kernel 5; LINE2_BICGSTAB needs fp64 fields. */
#define XEE_METHOD_LINE_BICGSTAB 6
#define XEE_METHOD_LINE2_BICGSTAB 7
/* Mixed-precision two-level method (not in the reference): fp64 iterative refinement around fp32 two-level block-line
 * Chebyshev sweeps.  psi, f, the residual L psi - f and the stop rule stay fp64; each refinement step solves
 * L e = r / s approximately with check_step fp32 sweeps (the operator rounded to fp32, fp64 coarse solve, fp64 spectral
 * estimate, s a power of two per solve) and applies psi += s e in fp64.  iters and max_iter count fp32 sweeps, and
 * check_step is the number of sweeps per refinement step: every step ends with one check of the fp64 residual.  A solve
 * that reaches max_iter inside a step applies the partial correction.  fp64 plans only (an fp32 plan is refused), shared
 * operator or one per solve, FAST arithmetic, sweep kernel 5, the grids of LINE2_CHEBYSHEV with nx % 4 == 0. */
#define XEE_METHOD_LINE2_MIXED 8

typedef struct xee_plan xee_plan;

typedef struct xee_plan_desc {
  int dtype;      /* XEE_F32 | XEE_F64                                                   */
  int nx, ny;     /* grid (nr, nz); fields are [ny][nx] with i (radius) contiguous       */
  int nbatch;     /* independent solves per call                                         */
  int shared_coe; /* 1: one operator for the whole batch (map); 0: one per solve         */
  int arith;      /* XEE_ARITH_*                                                         */
  int method;     /* XEE_METHOD_*                                                        */
  int device;     /* CUDA device ordinal, -1 = current                                   */
  int kernel;     /* 0 = auto; >0 forces a sweep-kernel variant (see DESIGN.md)          */
} xee_plan_desc;

typedef struct xee_solve_params {
  int max_iter, check_step, converge_time, lost_rate; /* as solve_elliptic's arguments  */
  double r1, r2, alpha;                               /* r1/r2 <= 0 disables a criterion */
  const void* r1_per_solve; /* optional DEVICE array [nbatch] of the plan's dtype         */
  double rho_jacobi;        /* Chebyshev only: spectral-radius estimate, <=0 = estimate   */
  int detect_explode;       /* 1: non-finite residual sets XEE_ERR_EXPLODE and stops      */
  int sync_every;           /* host polls the active-solve count every N checks (>=1)     */
  int stall_checks;         /* >0: stop (XEE_ERR_STALLED) when the best residual has not improved by 0.1 %
                               for this many consecutive checks; 0 = reference semantics (off)             */
} xee_solve_params;

const char* xee_last_error(void);
int xee_device_count(void);
const char* xee_build_info(void);

int xee_plan_create(const xee_plan_desc* desc, xee_plan** out);
int xee_plan_destroy(xee_plan* p);
/* Operator upload.  AoS = the reference's coe(9,nx,ny)[,nbatch] layout. */
int xee_plan_set_coe_aos_host(xee_plan* p, const void* coe_host);
int xee_plan_set_coe_aos_dev(xee_plan* p, const void* coe_dev);
/* K1+K2 on device: a,b,c (device, reference shapes) -> planar operator.  Per-solve when shared_coe==0. */
int xee_plan_set_abc_dev(xee_plan* p, const void* a_dev, const void* b_dev, const void* c_dev, double dx, double dy);
/* Solve: psi_dev [nbatch][ny][nx] in/out (boundary + first guess in), f_dev same shape.
 * Per-solve outputs are HOST arrays (may be NULL): iters[nbatch], r1_out/r2_out[nbatch] (double), err[nbatch]. */
int xee_plan_solve_dev(xee_plan* p, void* psi_dev, const void* f_dev, const xee_solve_params* prm, int* iters,
                       double* r1_out, double* r2_out, int* err, void* stream);
/* Same with HOST psi/f (pageable or pinned): the end-to-end entry the bench's e2e leg times. */
int xee_plan_solve_host(xee_plan* p, void* psi_host, const void* f_host, const xee_solve_params* prm, int* iters,
                        double* r1_out, double* r2_out, int* err);
/* Exactly `sweeps` sweeps, no stop rule (bench / fixed-sweep parity).  rms_out: HOST [nbatch] RMS residual of
 * the last sweep, or NULL.  Result left in psi_dev. */
int xee_plan_sweeps_dev(xee_plan* p, void* psi_dev, const void* f_dev, double alpha, int sweeps, double* rms_out,
                        void* stream);
/* Same; the BiCGStab methods run `sweeps` iterations with the residual replacements of a solve with this check_step
 * (xee_plan_sweeps_dev: check_step 100), so that a solve stopping at iters = n returns the field of sweeps = n.  rms_out:
 * the true residual after them.  The other methods ignore check_step. */
int xee_plan_sweeps_checked_dev(xee_plan* p, void* psi_dev, const void* f_dev, double alpha, int sweeps, int check_step,
                                double* rms_out, void* stream);
/* out = L psi (interior; boundary 0) for the whole batch. */
int xee_plan_apply_dev(xee_plan* p, const void* psi_dev, void* out_dev, void* stream);
/* The library keeps freed device buffers of every size for reuse (cap: XEE_CACHE_MB, default 16 GiB); this returns them
 * to the driver. */
void xee_release_cached_memory(void);
/* Bytes of the library's device-memory pool, over all devices: held by live plans, maps and series (live_bytes), and freed
 * but kept for reuse (cached_bytes).  Either pointer may be NULL. */
int xee_pool_stats(long long* live_bytes, long long* cached_bytes);
/* Kernel-launch counter (bench.py's gpu_launches): launches issued by this library since reset. */
long long xee_launch_count(int reset);
/* Time (ms, CUDA events on the plan's stream) spent in the dominant sweep kernel and SWEEPS it performed since reset. */
int xee_sweep_kernel_stats(xee_plan* p, double* ms_total, long long* sweeps, int reset);
/* Sweep-kernel variant of the last solve (1 direct, 2 TMA pipeline, 3 resident, 4 temporal blocking, 5 block-line), the
 * sweeps one launch of it performs (>1 only for variant 4) and its launches since the last stats reset. */
int xee_plan_kernel_info(xee_plan* p, int* variant, int* sweeps_per_pass, long long* kernel_launches);
/* Chebyshev parameters in use (after a solve / sweeps call of an accelerated method): spectral radius rho of the iteration
 * matrix I - gamma M^-1 L and the step length gamma (1 for the one-level methods). */
int xee_plan_cheb_params(xee_plan* p, double* rho, double* gamma);

/* Post-processing on device fields (K5/K6), batch-wide.  geometry arrays are DEVICE pointers of the plan dtype. */
int xee_eta_dev(int dtype, const void* rchi, void* eta, const void* ra, const void* rcuva, const void* rho,
                const void* exner, int nr, int nz, int nbatch, void* stream);
int xee_uw_dev(int dtype, const void* rpsi, void* u, void* w, const void* ra, const void* rcuva, const void* za,
               const void* rho, int nr, int nz, int nbatch, void* stream);

/* =====================================================================================
 * Part 3 - efficiency map: one vortex (A,B,C), one elliptic solve per heating location.
 * Restates the heating -> secondary circulation -> kinetic-energy generation -> efficiency
 * chain of src/old-diagnose/diagnose.f90 (:383-406 source term, :449-461 solve, :915-941 w,
 * :1117-1127 w*theta, :1029-1113 integrals, :780-839 ratios) and, as the adjoint check,
 * src/diagnose's eta field (diagnose.f90:31-48, quick-tools1.f90:1-13).  Cylindrical geometry.
 * ===================================================================================== */
#define XEE_MAP_COLS 8 /* iters, r1, err, sum_Q, ke_gen, efficiency, sum_Qeta, efficiency_eta */

typedef struct xee_map xee_map;
typedef struct xee_map_desc {
  int dtype;         /* XEE_F32 | XEE_F64 (working precision; inputs are float32 files)   */
  int nr, nz;        /* grid points                                                       */
  int nheat;         /* heating locations = independent solves per run                    */
  int density_mode;  /* 0 DENSITY_NORMAL, 1 DENSITY_BOUSSINESQ (read-input.f90:33-40)      */
  int arith, method; /* XEE_ARITH_*, XEE_METHOD_*                                         */
  int device;        /* CUDA ordinal, -1 = current                                        */
  int adjoint_check; /* 1: also solve L chi = -B once and report sum(Q eta)/sum(Q)        */
  double Lr[2], Lz[2];  /* domain (read-input.f90:56)                                     */
  double r1_rel_rms_f;  /* >0: per-location tolerance r1_n = r1_rel * rms(f_n)            */
} xee_map_desc;

/* A,B,C: HOST float32 nr x nz fields in the reference's .bin layout (field_tools.f90:30-52). */
int xee_map_create(const xee_map_desc* desc, const float* A, const float* B, const float* C, xee_map** out);
int xee_map_destroy(xee_map* m);
/* heat: [nheat][5] doubles {r_c, z_c, sigma_r, sigma_z, Q0}; table: [nheat][XEE_MAP_COLS] doubles. */
int xee_map_run_host(xee_map* m, const double* heat_host, const xee_solve_params* prm, double* table_host);
int xee_map_run_dev(xee_map* m, const double* heat_dev, const xee_solve_params* prm, double* table_dev, void* stream);
/* which: 0 psi [nheat][nz][nr], 1 f, 2 theta_B [(nz-1)][(nr-1)], 3 eta [nz][nr-1], 4 chi,
 * 5 eta_d [(nz-1)][(nr-1)] and 6 lambda [nz][nr] of the last xee_map_adjoint_solve.  Plan dtype, HOST out. */
int xee_map_get_field(xee_map* m, int which, void* host_out);
/* Discrete adjoint.  ke_gen of a heating Q is <g, L^-1 H Q> = <mu, Q> with mu = H^T lambda and L^T lambda = g, g the
 * gradient of ke_gen in psi and H the map Q -> f: one solve gives the exact discrete efficiency sum(mu Q) / sum(W Q) of any
 * heating, equal to column 5 of the table to solver tolerance (efficiency_eta, column 7, is the continuous adjoint's, first
 * order in the grid spacing).  eta_d = mu / W is the efficiency of heating concentrated in one B cell.
 * adjoint_solve: L^T lambda = g from lambda = 0 with the map's dtype, arithmetic and method; r1 = r1_rel_rms_f * rms(g) when
 * r1_rel_rms_f > 0, else prm->r1.  Leaves lambda, mu and eta_d on the device.
 * adjoint_eval_host: heat [n][5] as for run, any n >= 1; table [n][XEE_ADJ_COLS] doubles.  Fails before an adjoint solve.
 * adjoint_timings: host wall time of the first call's setup (plan, L^T, line factors, coarse operator), of the spectral
 * probes and of the sweep kernels of the adjoint plan, in ms, summed over its calls. */
#define XEE_ADJ_COLS 3 /* sum_Q, ke_gen (scaled by g0/theta0 like table column 4), efficiency */
int xee_map_adjoint_solve(xee_map* m, const xee_solve_params* prm, int* iters, double* r1_out, int* err);
int xee_map_adjoint_eval_host(xee_map* m, const double* heat_host, int n, double* table_host);
int xee_map_adjoint_timings(xee_map* m, double* setup_ms, double* probe_ms, double* sweep_ms);
int xee_map_sweep_kernel_stats(xee_map* m, double* ms_total, long long* sweeps, int reset);
int xee_map_kernel_info(xee_map* m, int* variant, int* sweeps_per_pass, long long* kernel_launches);

/* =====================================================================================
 * Part 4 - time-series diagnosis (BASELINE config 5): one vortex snapshot = one operator per
 * solve; thermal + dynamical source term (src/old-diagnose/diagnose.f90:383-436), Ekman-pumping
 * bottom boundary condition (xtt-lib-python/XPumping.py:79-90), vortex fields built on the device
 * from wind-profile parameters (xtt-lib-python/XWindProfile.py:10-23).  Cylindrical geometry.
 * ===================================================================================== */
#define XEE_SERIES_PARAMS 21 /* doubles per snapshot: f0, f_core, f_env, radius, konst1, H, N2, pump r0 r1 r2,
                                pump c00 c01 c10 c11, heat r_c z_c sigma_r sigma_z Q0, friction k, friction h */
typedef struct xee_series xee_series;
typedef struct xee_series_desc {
  int dtype, nr, nz, nsnap, density_mode, arith, method, device;
  double Lr[2], Lz[2];
  double r1_rel_rms_f; /* >0: per-snapshot tolerance r1_n = r1_rel * rms(L psi0_n - f_n), the initial residual */
} xee_series_desc;
int xee_series_create(const xee_series_desc* desc, xee_series** out);
int xee_series_destroy(xee_series* s);
/* params: HOST [nsnap][XEE_SERIES_PARAMS]; table: HOST [nsnap][XEE_MAP_COLS] =
 * iters, r1, err, sum_Q, ke_gen, efficiency, max|w|, max|u| */
int xee_series_run_host(xee_series* s, const double* params_host, const xee_solve_params* prm, double* table_host);
/* The same series on caller-supplied snapshots (e.g. the reference's A.bin, B.bin, C.bin, Q and F files), arrays of the
 * plan dtype with i (r) fastest:
 *   A, B, C  [nsnap][nz][nr] on the O grid; required.
 *   Q        [nsnap][nz-1][nr-1] heating on the B cells; required.  sum_Q = 0 gives a non-finite efficiency.
 *   F        [nsnap][nz-1][nr-1] momentum forcing on the B cells; NULL: no momentum term (the bits of F = 0).
 *   psi_bc   [nsnap][nz][nr]; only its rim is read, as Dirichlet values of r*psi; NULL: 0.  The first guess is 0 inside,
 *            so r1_rel_rms_f keeps its meaning (relative to the initial residual).
 * Every operator gets its own spectral probe (the parametric run may subsample a smooth series).  table as for run_host.
 * _host: host pointers.  _dev: device pointers, read after the work already queued on `stream` (a cudaStream_t, NULL =
 * the legacy default stream); the call returns after the table is on the host. */
int xee_series_run_fields_host(xee_series* s, const void* A, const void* B, const void* C, const void* Q, const void* F,
                               const void* psi_bc, const xee_solve_params* prm, double* table_host);
int xee_series_run_fields_dev(xee_series* s, const void* A, const void* B, const void* C, const void* Q, const void* F,
                              const void* psi_bc, const xee_solve_params* prm, double* table_host, void* stream);
/* which: 0 psi, 1 f, 2 theta_B, 3 u (C grid), 4 w (A grid), 5 A, 6 B, 7 C, 8 m2 (B grid), 9 Q (B grid), 10 F (B grid; fails
 * after a field run without F); all [nsnap][...], plan dtype */
int xee_series_get_field(xee_series* s, int which, void* host_out);
/* The legacy efficiency decomposition (src/old-diagnose/diagnose.f90, the chain behind efficiency.txt) of every snapshot, on
 * the inputs of xee_series_run_fields_* plus chi_bc [nsnap][nz][nr] (only its rim is read, as Dirichlet values of r*chi;
 * NULL: no boundary-condition chi solves and no exchange conversion).  CYLINDRICAL geometry, the series' density mode.
 *   tendency 1 (TENDENCY): stage I solves L(B0) psi = f, stage II forms dtheta/dt, the anomaly over testing_dt (finite),
 *            theta_after and the operator B0 + dB.  tendency 0 (INSTANT): no stage I, dB = 0, theta_after = the background.
 *   baro     0 BAROTROPIC (operator tag 0: B = 0), 1 BAROCLINIC (tag B0dB: B = B0 + dB), 2 BARO_ALL (both).
 * Per tag: the chi solves L chi = 0 (chi_bc rim), = f_anomaly, = f_basic; sum(Q eta) of each; the integral-check solve
 * L psi = f and its w theta integral with theta_after; with chi_bc the exchange conversion, methods 1 and 2 ([D5] of the
 * re-host: real r, dr, dz, from the working-precision fields).  prm_psi governs the psi solves, prm_chi the chi solves,
 * tolerances as for run_fields.  Deviations from the legacy driver: every solve starts from its rim with a zero interior
 * (the legacy driver carries chi from one chi solve into the next and starts psi from the whole psi_bc); the solves use this
 * library's stop rule, not legacy strategies 1-4; converged answers agree to the tolerance.  A solve whose initial residual
 * is exactly 0 (zero right-hand side and rim: f_anomaly in INSTANT mode) is not run: its field is its first guess, iters 0.
 * table [nsnap][XEE_DECOMP_COLS], raw sums (an efficiency.txt line is "value , value / sum_Q"); NaN = not computed (a tag
 * baro excludes, the chi_bc terms without chi_bc, the tendency terms in INSTANT mode):
 *   0 sum_Q, 1 sum_dtheta_dt, 2 local heat response sum_dtheta_dt / sum_Q,
 *   3..9 tag 0 and 10..16 tag B0dB: eta_bc, eta_dB, eta_B0, bndconv, bndconv2, etaQ (decomposition sum), wtheta.
 * iters, err: HOST [nsnap][XEE_DECOMP_SOLVES] or NULL, in the order psi_before, chi 0_0, chi B0dB_0, chi 0_dB, chi B0dB_dB,
 * chi 0_B0, chi B0dB_B0, psi_after 0, psi_after B0dB; iters -1 for a solve not run.  _host / _dev as for run_fields. */
typedef struct xee_decomp_desc { int tendency; double testing_dt; int baro; } xee_decomp_desc;
#define XEE_DECOMP_COLS 17
#define XEE_DECOMP_SOLVES 9
int xee_series_decompose_host(xee_series* s, const xee_decomp_desc* desc, const void* A, const void* B, const void* C,
                              const void* Q, const void* F, const void* psi_bc, const void* chi_bc,
                              const xee_solve_params* prm_psi, const xee_solve_params* prm_chi, double* table, int* iters,
                              int* err);
int xee_series_decompose_dev(xee_series* s, const xee_decomp_desc* desc, const void* A, const void* B, const void* C,
                             const void* Q, const void* F, const void* psi_bc, const void* chi_bc,
                             const xee_solve_params* prm_psi, const xee_solve_params* prm_chi, double* table, int* iters,
                             int* err, void* stream);
/* which: 0 dtheta_dt, 1 theta_after (B grid [nsnap][nz-1][nr-1]); 2 + k: the field of solve k in the iters order (O grid
 * [nsnap][nz][nr]).  Fails for a field the last decomposition did not make.  Plan dtype, HOST out. */
int xee_series_get_decomp_field(xee_series* s, int which, void* host_out);
int xee_series_sweep_kernel_stats(xee_series* s, double* ms_total, long long* sweeps, int reset);
int xee_series_kernel_info(xee_series* s, int* variant, int* sweeps_per_pass, long long* kernel_launches);
/* Host wall time (ms) the spectral-radius probes of the accelerated methods have taken since the last reset (with one
 * operator per solve they run once per run(): bench.py reports their share of a step). */
int xee_series_probe_stats(xee_series* s, double* ms_total, int reset);

#ifdef __cplusplus
}
#endif
#endif /* XEE_B200_H */

/*
 * f16_b200.h -- C ABI of libf16_b200.so, the B200 (sm_100a) batched F-16 plant.
 *
 * Drop-in boundary.  The reference project (johnviljoen/f16_mpc_oop_py) loads `C/nlplant_xcg25.so` or
 * `C/nlplant_xcg35.so` with ctypes.CDLL (parameters.py:108-114) and calls exactly two symbols:
 *     Nlplant(xu*, xdot*, int)   env.py:100, env.py:187      (C/nlplant.c:14,23)
 *     atmos(alt, vt, coeff*)     utils.py:291                (C/nlplant.c:8,467)
 * Both are exported here with the reference's signatures; the batched entry points below are new and take
 * struct-of-arrays buffers.  Plain pointers and sizes only; the caller owns every buffer; nothing is retained.
 *
 * There is no CPU implementation behind any of these calls: every one of them runs the CUDA kernels of this
 * library and returns F16_ERR_CUDA (or writes NaN for the two void legacy symbols) if no B200 is usable.
 *
 * Conventions
 *   state  x[18] = {npos,epos,h,phi,theta,psi,V,alpha,beta,p,q,r,T,dh,da,dr,lf2,lf1}   (parameters.py:116)
 *   input  u[4]  = {T,dh,da,dr}                                                          (parameters.py:117)
 *   xu[17]       = x[0:17] as Nlplant reads it (C/nlplant.c:76-114; xu[16] = lef)
 *   SoA layout   plane i of an [M][N] array starts at base + i*ld (ld = N for the host entry points)
 *   fidelity     1 = hifi (Nguyen tables), 0 = lofi (Stevens-Lewis)                      (C/nlplant.c:183,245)
 *   xcg          centre of gravity as a fraction of cbar; the reference compiles 0.25 or 0.35 in (C/nlplant.c:34)
 */
#ifndef F16_B200_H
#define F16_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes ------------------------------------------------------------------------------ */
#define F16_OK 0
#define F16_ERR_CUDA (-1)    /* CUDA runtime error or no usable device; see f16_last_error() */
#define F16_ERR_TABLES (-2)  /* aero tables not found or corrupt */
#define F16_ERR_ARG (-3)     /* bad argument */
#define F16_ERR_NOINIT (-4)  /* internal: initialisation failed earlier */
#define F16_ERR_HOST (-5)    /* host memory or thread creation failed inside the library */

/* ---- per-aircraft status word (int32, sticky within one call) ------------------------------------
 * The reference's behaviour in these cases is exit() (env.py:117-124) or undefined (mexndinterp.c:121-123);
 * here the aircraft is flagged, Nlplant_batch writes NaN derivatives and step_batch freezes the state at
 * the first violating step. */
#define F16_ST_BOUND(i) (1 << (i)) /* bits 0..17: state i outside parameters.py:122-123 (compared raw, as there) */
#define F16_ST_ALPHA (1 << 18)     /* alpha outside the tables: hifi [-20,45] deg */
#define F16_ST_BETA (1 << 19)      /* beta outside [-30,30] deg */
#define F16_ST_DELE (1 << 20)      /* elevator outside [-25,25] deg (hifi) */
#define F16_ST_NAN (1 << 21)       /* NaN in a state or input */
#define F16_ST_FIDELITY (1 << 22)  /* fidelity flag neither 0 nor 1 */

/* ---- arithmetic mode ---------------------------------------------------------------------------- */
#define F16_MATH_STRICT 0 /* reference operation order, no FMA contraction: the parity build */
#define F16_MATH_FAST 1   /* throughput build.  step_batch / trim_batch run the RE-ASSOCIATED arithmetic of csrc/f16_fast.cuh
                           * ((f, d) table image with node deltas, polynomial sin/cos and tfac^4.14, one shared reciprocal,
                           * wind-axis equations with vt cancelled); Nlplant_batch / calc_xdot_batch run the strict
                           * expressions with FMA contraction and reciprocal multiplies.  Both stay within the parity bars
                           * (<= 1e-12 scaled per derivative, <= 1e-9 after 10 s; tests/test_gpu_parity.py);
                           * linearise_batch runs f16_fast.cuh too (two aircraft per warp, csrc/f16_linearise_fast.cu): the quotient
                           * multiplies last-bit differences of f by 1/eps, so its entries agree with the reference's to
                           * 1e-8 + 4 ulp(f_i) / h (up to 3.4e-8 on the 900 ft/s navigation rows; the reference's own source built
                           * with -O3 -march=native moves as much, profiles/r02_jacobian_noise_floor.md).
                           * f16_set_linearise_variant(2) keeps the strict kernel in fast mode. */

/* ---- CLr table quirk ---------------------------------------------------------------------------
 * The reference never loads CL1320_ALPHA1_606.dat (hifi_F16_AeroData.c:965-972: the fscanf loop is the
 * body of `if(fp==NULL)`), so its binaries compute with CLr = 0.  Default: as built. */
#define F16_CLR_AS_BUILT 0
#define F16_CLR_FROM_FILE 1

/* ---- finite-difference schemes of linearise_batch ------------------------------------------------ */
#define F16_FD_FORWARD 0 /* (f(x+eps e_i) - f(x))/eps, env.py:319-340 */
#define F16_FD_CENTRAL 1 /* (f(x+eps e_i) - f(x-eps e_i))/(2 eps) */

/* ---- closed-loop law fused into step_batch -------------------------------------------------------
 * For every input row r with bit r of row_mask set:
 *     u[r] = u0[r] - sum_{j<n_sel} K[r][j] * (x[sel[j]] - x_ref[j])        (accumulated in j order)
 * other rows keep the open-loop input.  With sel = parameters.py mpc_states indices [3,4,7,8,9,10,11,17,16],
 * rows {1,2,3} and K from env.py:344-358 this is test_env.py:294 (u = u0 - K(x - x_ref)); env.py:360-371
 * (x_ref = x except p,q,r) is the same law with only the p,q,r columns of K non-zero. */
typedef struct f16_lqr_t {
  int n_sel;
  int row_mask;
  int sel[18];
  double K[4][18];
  double x_ref[18];
  double u0[4];
} f16_lqr_t;

/* ---- legacy symbols: the reference ABI ------------------------------------------------------------ */
/* Replaces C/nlplant.c:23-457.  Reads xu[0..16], writes xdot[0..17] ([12..14] = nx,ny,nz, [15..17] = mach,
 * qbar,ps).  xcg comes from f16_set_default_xcg (the C/nlplant_xcg25.so / xcg35.so shims fix it).  Outside
 * the table envelope the reference is undefined; this writes NaN and sets f16_last_status(). */
void Nlplant(double *xu, double *xdot, int fidelity);
/* Replaces C/nlplant.c:467-490.  coeff[0..2] = mach, qbar, ps. */
void atmos(double alt, double vt, double *coeff);
/* Same as Nlplant with an explicit xcg, and atmos under a second name: what the two drop-in shim libraries
 * (C/nlplant_xcg25.so, C/nlplant_xcg35.so, csrc/f16_shim.c) forward to. */
void f16_nlplant_xcg(const double *xu, double *xdot, int fidelity, double xcg);
void f16_atmos(double alt, double vt, double *coeff);

/* ---- library state --------------------------------------------------------------------------------- */
/* Idempotent.  table_path: the packed blob (f16_aero_v1.bin), or a directory holding the reference's C/<table>.dat
 * files, or NULL to search $F16_TABLE_PATH, <lib dir>/../data/f16_aero_v1.bin, ./C/.  device: CUDA ordinal,
 * or -1 for $F16_DEVICE / $LOCAL_RANK / 0.  Called implicitly (NULL, -1) by every other entry point. */
int f16_init(const char *table_path, int device);
/* Several GPUs of one box behind the same entry points (SURVEY 8b/8e).  One context -- stream, table images, scratch -- per entry
 * of devices[0..ndev) (CUDA ordinals; NULL or ndev <= 0: every visible device; an ordinal may be listed more than once, which
 * gives independent streams on that GPU).  From then on every HOST-buffer batch call (Nlplant_batch, calc_xdot_batch, step_batch,
 * step_batch_traj, step_batch_stats, linearise_batch, trim_batch, state_summary_batch) cuts its N aircraft into contiguous
 * slices, one per context (boundaries on multiples of 32 aircraft), and runs the slices concurrently, each from its own host
 * thread with its own H2D / kernel / D2H pipeline: aircraft never interact, so nothing is exchanged between devices and the
 * results are bit-identical to a single-device call.  Batches too small to feed every device use fewer of them.  The *_dev
 * entry points, the memory helpers, the timers and the legacy symbols work on ONE context: the first, or the one selected by
 * f16_use_device.  Must be the first call into the library (or follow f16_shutdown); f16_init is f16_init_devices with one entry. */
int f16_init_devices(const char *table_path, const int *devices, int ndev);
int f16_device_count(void);      /* number of contexts; 0 before init */
int f16_use_device(int index);   /* context (index into the f16_init_devices list) of the *_dev entry points, the memory helpers
                                    and the timers; returns the previous index or an F16_ERR_* code */
/* The host logic behind the two calls above, without a GPU (used by the CPU tests): the slices a batch of N aircraft is cut into
 * over `contexts` device contexts (lo_n [2 * contexts] = first aircraft and count of each; returns the number of slices), and the
 * pipeline chunks of one slice (returns their number; *chunk = aircraft per chunk, *slots = device slots in use). */
int f16_plan_slices(long long N, long long min_per_device, int contexts, long long *lo_n);
int f16_plan_chunks(long long n, long long min_chunk, int max_chunks, long long *chunk, int *slots);
int f16_set_host_pipeline(int on); /* 1 (default): the host-buffer batch calls run as a chunk pipeline on each device (H2D of chunk
                                      c + 1 and D2H of chunk c - 1 under the kernels of chunk c); 0: one chunk.  Same bits. */
void f16_shutdown(void);
const char *f16_last_error(void);
int f16_last_status(void);            /* status word of the last legacy Nlplant call */
int f16_device(void);                 /* CUDA ordinal of the current context, -1 before init */
int f16_sm_count(void);
int f16_set_math_mode(int mode);      /* F16_MATH_*; returns the previous mode */
int f16_set_clr_mode(int mode);       /* F16_CLR_*; rebuilds the device tables; returns previous mode */
void f16_set_default_xcg(double xcg); /* for the legacy Nlplant symbol; default 0.25 or $F16_XCG */
int f16_set_table_staging(int mode);  /* 1 (default): tables staged in shared memory by TMA bulk copy;
                                         0: read through L1/L2 with ld.global.nc (for A/B measurements) */
int f16_set_step_threads(int threads); /* CTA size of the fused step kernel: 256, 384 (default), 512, 640, 768 or 1024 */
int f16_set_step_chunking(int on);     /* 1 (default): long runs of the fast hifi step are scheduled in time chunks (work item = 32 aircraft x
                                          K/16 steps) so the persistent grid has no tail; 0: one warp-task = all K steps.  Same bits. */
int f16_set_step_compaction(int on);    /* 1: a long uniform-fidelity run (K >= 4096 steps, >= 65536 aircraft) is cut into chunks of K / 8 steps
                                          (doubling while no aircraft is lost); once more than 1/16 of the active lanes belong to aircraft
                                          that have left the envelope, the survivors are repacked into full warps (csrc/f16_partition.cu)
                                          and the stopped aircraft retired to the caller's arrays.  Same bits as one launch.  Measured at 2^20
                                          aircraft x 10^4 steps: xcg 0.35 open loop (57 % of the batch lost) 369 -> 291 ms; a run that loses
                                          nobody pays for the extra launches (+0.5 %).  0 (default): one launch.  $F16_STEP_COMPACTION. */
int f16_set_trim_fixed_point_exit(int on); /* 1 (default): trim_batch leaves a Nelder-Mead search whose shrink step moves no vertex any more (the
                                             simplex has collapsed onto neighbouring floating-point numbers without meeting xatol /
                                             fatol: a kink of the cost at a clipped control).  Every further iteration would repeat
                                             the last one bit for bit, so the result at maxiter is known: same point, info = maxiter
                                             iterations and the evaluations they would have made.  Results identical to 0 (spin to
                                             maxiter like scipy, env.py:273); the cfg-4 grid at xcg 0.25 takes 36 ms instead of 537. */
int f16_set_linearise_variant(int variant); /* linearise_batch kernel.  0 (default): in F16_MATH_STRICT the staged strict kernel (CTA per
                                               32 aircraft, columns over warps), in F16_MATH_FAST the two-aircraft-per-warp kernel on
                                               the fast arithmetic; 1 = strict, warp per aircraft, column per lane; 2 = strict, CTA
                                               per 32 aircraft, in either math mode.  1 and 2 give the same bits. */
/* sha256 (hex, 64 chars + NUL) of the canonical table payload in use */
int f16_tables_sha256(char *out65);

/* ---- batched entry points, HOST buffers (H2D/D2H inside the call) ------------------------------------ */
/* xu_soa [17][N] -> xdot_soa [18][N].  fi / xcg: per-aircraft arrays or NULL to use the defaults. */
int Nlplant_batch(const double *xu_soa, double *xdot_soa, const unsigned char *fi, int fi_default, const double *xcg,
                  double xcg_default, long long N, int *status);
/* env.py::_calc_xdot (env.py:65-103) for N aircraft: x_soa [18][N], u_soa [4][N] -> xdot_soa [18][N]. */
int calc_xdot_batch(const double *x_soa, const double *u_soa, double *xdot_soa, const unsigned char *fi, int fi_default,
                    const double *xcg, double xcg_default, long long N, int *status);
/* K fused explicit-Euler steps of env.py::step (env.py:105-130): x_soa [18][N] in/out, u_soa [4][N].
 * lqr: NULL = open loop.  status [N] (may be NULL), steps_done [N] (may be NULL) = steps taken before freeze. */
int step_batch(double *x_soa, const double *u_soa, long long N, int K, double dt, const f16_lqr_t *lqr,
               const unsigned char *fi, int fi_default, const double *xcg, double xcg_default, int *status,
               int *steps_done);
/* step_batch with the whole state recorded every snap_every steps: traj [K / snap_every][18][N] (what the reference's
 * drivers collect in x_storage, test_env.py:452-462).  Bit-identical to one step_batch call of K steps. */
int step_batch_traj(double *x_soa, const double *u_soa, long long N, int K, int snap_every, double dt, const f16_lqr_t *lqr,
                    const unsigned char *fi, int fi_default, const double *xcg, double xcg_default, double *traj, int *status);
/* Finite-difference Jacobians of _calc_xdot (env.py:294-342): A [N][18][18], B [N][18][4], row-major.
 * Always computed by the strict (no FMA contraction) build: the quotient amplifies rounding noise by 1/eps.
 * eps must lie in [1e-12, 1e3] (the reference uses 1e-5). */
int linearise_batch(const double *x_soa, const double *u_soa, long long N, double eps, int scheme, double *A, double *B,
                    const unsigned char *fi, int fi_default, const double *xcg, double xcg_default, int *status);

/* env.py::trim (env.py:198-292) for N flight conditions: h [N] ft, V [N] ft/s -> x_trim_soa [18][N], the state
 * env.py:288 builds from the optimiser's output.  Nelder-Mead exactly as scipy runs it for the reference (env.py:273:
 * tol -> xatol = fatol, maxiter, default coefficients, default initial simplex) from ux0 = {P3, dh, da, dr, alpha}
 * (NULL = the reference's guess {5000, -0.09, 8.49, -0.01, 0.01}, env.py:264-271).  info_soa [4][N] (may be NULL) =
 * cost, iterations, objective evaluations, converged.  status [N]: envelope status of the returned point. */
int trim_batch(const double *h, const double *V, long long N, double tol, int maxiter, const double *ux0, double *x_trim_soa,
               double *info_soa, const unsigned char *fi, int fi_default, const double *xcg, double xcg_default, int *status);

/* ---- between linearise and the control law (f16_linalg.cu) ---------------------------------------------------
 * reduce_jacobian_batch: A [N][18][18] (forward linearise) -> the reference's 9-state / 3-input model (env.py:49,152-193):
 *   A_na [N][9][9] over mpc_states {phi,theta,alpha,beta,p,q,r,lf1,lf2}, B_na [N][9][3] over {dh,da,dr}.  An exact gather:
 *   _calc_xdot_na perturbs the same full-model evaluation (rows 3,4,7,8,9,10,11,16,17; the LEF derivatives swap, :184,189).
 * discretise_batch: scipy.signal.cont2discrete(method='zoh') of env.py:46,50 for N systems, A [N][n][n], B [N][n][m];
 *   a non-finite dt is F16_ERR_ARG.
 * dlqr_batch: utils.py:219-245, K [N][m][n] = (B'PB + R)^-1 B'PA with P [N][n][n] (may be NULL) from the discrete Riccati
 *   equation; Q [n][n], R [m][m] shared by all systems; info [N][2] (may be NULL) = {status, doublings done}, status:
 *      0  converged, P solves the equation (residual test), A - BK stable (its powers shrink below 1/2 in norm)
 *      1  tolerance not met in 64 doublings     -4  R + B'PB singular
 *     -1  R singular                            -5  converged to a P for which A - BK is not stable ((A, Q) not detectable)
 *     -2  I + GH singular in a doubling         -6  converged to an H that fails the residual test (the doubling broke
 *     -3  NaN or Inf in the data or an iterate      down numerically)
 *   K of a system with a negative status is NaN; P is still written.
 * lqr_gain_batch: F16._calc_LQR_gain (env.py:344-358) for N operating points, device end to end: K [N][3][9] = -dlqr(...).
 * n <= 18, n + m <= 22. */
int reduce_jacobian_batch(const double *A, long long N, double *A_na, double *B_na);
int discretise_batch(const double *A, const double *B, int n, int m, long long N, double dt, double *Ad, double *Bd);
int dlqr_batch(const double *Ad, const double *Bd, const double *Q, const double *R, int n, int m, long long N, double *K,
               double *P, int *info);
int lqr_gain_batch(const double *x_soa, const double *u_soa, long long N, double dt, double *K, const unsigned char *fi,
                   int fi_default, const double *xcg, double xcg_default, int *status);

/* ---- end-of-run statistics, reduced on the device (f16_stats.cu; SURVEY 8e: the row a rank contributes to the one
 * collective of a run; the reference's drivers keep the whole x_storage on the host instead, test_env.py:452-462) ----
 * Over the aircraft with status[n] == 0 (all of them if status == NULL):
 *   row [74] = { N, alive, min[18], max[18], mean[18], M2[18] },  M2 = sum (x - mean)^2  (two passes, no cancellation).
 * An empty selection gives min = +inf, max = -inf, mean = M2 = 0.  Bit-reproducible for a given device and N. */
int state_summary_batch(const double *x_soa /* [18][N] */, long long N, const int *status, double *row);
/* A Monte-Carlo rollout that keeps statistics instead of trajectories (BASELINE cfg 5: 64 Mi aircraft -- x_storage of
 * test_env.py:452-462 would be 9 GB per snapshot): K steps as step_batch, and after every snap_every steps the summary row of
 * the whole batch -> rows [K / snap_every][74].  States and status words end bit-identical to one step_batch call of K steps. */
int step_batch_stats(double *x_soa, const double *u_soa, long long N, int K, int snap_every, double dt, const f16_lqr_t *lqr,
                     const unsigned char *fi, int fi_default, const double *xcg, double xcg_default, double *rows, int *status);

/* ---- batched entry points, DEVICE buffers (asynchronous on f16_stream(); ld = plane stride) ---------
 * step_batch_dev with a per-aircraft fi array (N >= 4096, K >= 8) orders the batch by fidelity on the device first
 * (csrc/f16_partition.cu) and synchronises the stream once to read the class sizes. */
int Nlplant_batch_dev(const double *xu_soa, long long ld_in, double *xdot_soa, long long ld_out, const unsigned char *fi,
                      int fi_default, const double *xcg, double xcg_default, long long N, int *status);
int calc_xdot_batch_dev(const double *x_soa, long long ld_x, const double *u_soa, long long ld_u, double *xdot_soa,
                        long long ld_out, const unsigned char *fi, int fi_default, const double *xcg, double xcg_default,
                        long long N, int *status);
int step_batch_dev(double *x_soa, long long ld_x, const double *u_soa, long long ld_u, long long N, int K, double dt,
                   const f16_lqr_t *lqr /* host pointer */, const unsigned char *fi, int fi_default, const double *xcg,
                   double xcg_default, int *status, int *steps_done);
int linearise_batch_dev(const double *x_soa, long long ld_x, const double *u_soa, long long ld_u, long long N, double eps,
                        int scheme, double *A, double *B, const unsigned char *fi, int fi_default, const double *xcg,
                        double xcg_default, int *status);

int trim_batch_dev(const double *h, const double *V, long long N, double tol, int maxiter, const double *ux0 /* host */,
                   double *x_trim_soa, long long ld_x, double *info_soa, long long ld_info, const unsigned char *fi,
                   int fi_default, const double *xcg, double xcg_default, int *status);

int state_summary_batch_dev(const double *x_soa, long long ld_x, long long N, const int *status /* device or NULL */,
                            double *row /* host, 74 doubles */);
int step_batch_stats_dev(double *x_soa, long long ld_x, const double *u_soa, long long ld_u, long long N, int K, int snap_every,
                         double dt, const f16_lqr_t *lqr /* host */, const unsigned char *fi, int fi_default, const double *xcg,
                         double xcg_default, double *rows /* host, [K / snap_every][74] */, int *status /* device, required */);

int reduce_jacobian_batch_dev(const double *A, long long N, double *A_na, double *B_na);
int discretise_batch_dev(const double *A, const double *B, int n, int m, long long N, double dt, double *Ad, double *Bd);
int dlqr_batch_dev(const double *Ad, const double *Bd, const double *Q, const double *R, int n, int m, long long N, double *K,
                   double *P, int *info);

/* ---- parity probes (used by the tests; device work, host buffers) ------------------------------------ */
/* For N query points (alpha_deg, beta_deg, el): coef [44][N] in the order of the reference aggregators
 * hifi_C, hifi_damping, hifi_C_lef, hifi_damping_lef, hifi_rudder, hifi_ailerons, hifi_other_coeffs
 * (hifi_F16_AeroData.c:1871-1934) and cells [8][N] = (lo,hi) of ALPHA, BETA1, DH1, DH2 in getHyperCube's
 * convention (mexndinterp.c:126-137: exact hit -> lo == hi). */
int f16_hifi_probe(const double *alpha_deg, const double *beta_deg, const double *el, long long N, double *coef,
                   int *cells, int *status);
/* The same 44 outputs from the F16_MATH_FAST table image with the step kernel's own cell search (csrc/f16_fast.cuh:
 * locate_hifi, (f, d) gathers): cells [4][N] = cell index k of ALPHA, BETA1, DH1, DH2 (the cell spans breakpoints k, k+1),
 * lam [4][N] = weight inside the cell.  getHyperCube's (lo, hi) maps to k = lo when lo != hi; on an exact hit lo == hi the
 * search returns (lo, lam = 0) or (lo - 1, lam = 1), the same node value.  Slots 24 (delta_CZq_lef, unused by
 * nlplant.c:339) and 43 (delta_Cm_ds = 0) are returned as 0. */
int f16_fast_probe(const double *alpha_deg, const double *beta_deg, const double *el, long long N, double *coef,
                   int *cells, double *lam, int *status);
/* lofi coefficients: out [19][N] = damping[9], dmomdcon[4], clcn[2], cxcm[2], cz, Cy(-.02b+.021da+.086dr) */
int f16_lofi_probe(const double *alpha_deg, const double *beta_deg, const double *el, const double *dail,
                   const double *drud, long long N, double *out);
int atmos_batch(const double *alt, const double *vt, long long N, double *coeff_soa /* [3][N] */);
/* the strict build's two division helpers against the device's IEEE division: out [3][N] = { branch-free division sequence,
 * reciprocal + residual correction with RN(1/b), a / b } (csrc/f16_model.cuh: F16_DIV, div_by) */
int f16_div_probe(const double *a, const double *b, long long N, double *out);

/* ---- device memory / timing helpers so that callers need no CUDA binding of their own ---------------- */
void *f16_dev_alloc(unsigned long long bytes);
void f16_dev_free(void *p);
void *f16_host_alloc_pinned(unsigned long long bytes);
void f16_host_free_pinned(void *p);
int f16_memcpy_h2d(void *dst_dev, const void *src_host, unsigned long long bytes);
int f16_memcpy_d2h(void *dst_host, const void *src_dev, unsigned long long bytes);
int f16_memcpy_d2d(void *dst_dev, const void *src_dev, unsigned long long bytes); /* asynchronous on f16_stream() */
int f16_memset_dev(void *dst_dev, int value, unsigned long long bytes);
int f16_sync(void);
void *f16_stream(void);            /* cudaStream_t the kernels run on */
int f16_timer_start(void);         /* cudaEventRecord on f16_stream() */
int f16_timer_stop(float *ms);     /* records, synchronises, returns elapsed ms */
unsigned long long f16_launch_count(void); /* kernels of this library launched since init (all contexts) */
/* Sustained FP64 FMA rate of this GPU (TFLOP/s, 2 flop per DFMA) from a register-only DFMA kernel run for
 * about `ms` milliseconds: the measured denominator of the FP64 roofline. */
int f16_measure_fp64_peak(double ms, double *tflops);
/* write a buffer larger than L2 so that the next timed launch starts cold */
int f16_flush_l2(void);

#ifdef __cplusplus
}
#endif
#endif /* F16_B200_H */

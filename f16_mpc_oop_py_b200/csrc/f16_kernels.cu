// f16_kernels.cu -- sm_100a kernels of the batched F-16 plant in the reference operation order, compiled with -fmad=false
// (no FMA contraction): the parity build, namespace f16::strict.  F16_MATH_FAST runs the kernels of f16_step_fast.cu and
// f16_linearise_fast.cu where they apply and these everywhere else.
//
// Execution model: one thread per aircraft (or per aircraft x perturbation column in linearise), the 18-element
// state lives in registers across the K fused Euler steps of step_kernel.  The aero tables (105 KB hifi image,
// 6 KB lofi image, f16_tables.h) are staged into shared memory once per CTA by TMA bulk copies
// (cp.async.bulk + mbarrier) and the CTAs are persistent (grid = resident CTAs, grid-stride over aircraft).
// FP64 pipe and shared-memory gathers bound these kernels; HBM traffic is 320 B per aircraft per launch.
#include <stdint.h>

#include "f16_kernels.cuh"
#include "f16_kernels_common.cuh"

#define F16_THREADS 384  // derivative-only kernels: one CTA per SM, 12 warps, <= 168 registers per thread
// step_kernel: 384 threads per CTA with the tables staged (168 registers per thread, one CTA per SM because of the 105 KB
// table image), 256 with the tables read through L2.
#define F16_LIN_WARPS 8    // linearise: 8 warps x 32 aircraft per CTA, <= 255 registers per thread (the staged evaluation holds 60 doubles of reusable stages)
#define F16_LIN_TILE_LD 397  // doubles per aircraft in the output tile (396 + 1: conflict-free for both phases)

namespace f16 {
namespace strict {

template <int FI>
struct Img {
  static constexpr int DOUBLES = FI ? F16_IMG_HIFI_DOUBLES : F16_IMG_LOFI_DOUBLES;
  static constexpr int BYTES = DOUBLES * 8;
  static constexpr int SMEM_BYTES = BYTES + 16;  // + the mbarrier
};

template <int FI, bool SMEM>
__device__ __forceinline__ const double* acquire_tables(const DevTables& t) {
  const double* g = FI ? t.hifi : t.lofi;
  if (!SMEM) return g;
  stage_tables_tma<Img<FI>::BYTES>(f16_smem, g, reinterpret_cast<unsigned long long*>(f16_smem + Img<FI>::BYTES));
  return reinterpret_cast<const double*>(f16_smem);
}

// ------------------------------------------------------------------------------------------------------
// Input pipeline of the one-shot kernels (Nlplant_batch, calc_xdot_batch).  One evaluation per aircraft makes them
// HBM-bound (280-324 B per aircraft); with plain loads a warp's memory phase and its ~1500-instruction compute phase
// alternate and the bytes in flight per SM cover only half of the bandwidth-latency product.  Here every warp owns
// NP x 32 doubles of shared memory and copies the input planes of the aircraft it takes NEXT with cp.async (8 bytes per
// lane and plane: one 256-byte transaction per warp and plane) before it starts computing the current one, so the loads
// of iteration i + 1 are in flight during the arithmetic of iteration i.  A lane reads back only what it copied itself:
// no barrier, the warps stay independent.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async8(double* dst_smem, const double* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}

template <int NA, int NB>
__device__ __forceinline__ void pipe_issue(double* buf, int lane, const double* __restrict__ a, long long lda,
                                           const double* __restrict__ b, long long ldb, long long n, bool valid) {
  if (valid) {
#pragma unroll
    for (int i = 0; i < NA; i++) cp_async8(buf + i * 32 + lane, a + i * lda + n);
#pragma unroll
    for (int i = 0; i < NB; i++) cp_async8(buf + (NA + i) * 32 + lane, b + i * ldb + n);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int NP>
__device__ __forceinline__ void pipe_take(const double* buf, int lane, double (&v)[NP]) {
  asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
  for (int i = 0; i < NP; i++) v[i] = buf[i * 32 + lane];
  asm volatile("" ::: "memory");  // the reads stay above the next cp.async into the same slots
}

template <int FI, bool SMEM, int NP>
struct PipeSmem {
  static constexpr int OFF = SMEM ? (Img<FI>::SMEM_BYTES + 127) / 128 * 128 : 0;
  static constexpr int TOTAL = OFF + (F16_THREADS / 32) * NP * 32 * 8;
};

// ------------------------------------------------------------------------------------------------------
// Nlplant_batch: xu [17][N] -> xdot [18][N]
// ------------------------------------------------------------------------------------------------------
template <int FI, bool SMEM>
__global__ void __launch_bounds__(F16_THREADS, 1)
nlplant_kernel(DevTables tabs, BatchSel sel, const double* __restrict__ xu_g, long long ld_in, double* __restrict__ xd_g,
               long long ld_out, long long N, int* __restrict__ status) {
  const double* img = acquire_tables<FI, SMEM>(tabs);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* buf = reinterpret_cast<double*>(f16_smem + PipeSmem<FI, SMEM, 17>::OFF) + warp * (17 * 32);
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // an aircraft of the other fidelity is neither copied nor evaluated here (mixed batches: the other launch takes it)
  pipe_issue<17, 0>(buf, lane, xu_g, ld_in, nullptr, 0, n, n < N && owns<FI>(sel, n) != 0);
  for (; n < N; n += stride) {
    double xu[17], xd[18];
    pipe_take<17>(buf, lane, xu);
    const long long nn = n + stride;
    pipe_issue<17, 0>(buf, lane, xu_g, ld_in, nullptr, 0, nn, nn < N && owns<FI>(sel, nn) != 0);
    const int own = owns<FI>(sel, n);
    if (own == 0) continue;
    unsigned st = ST_FIDELITY;
    if (own == 1) st = nlplant_eval<FI>(img, xu, sel.xcg ? sel.xcg[n] : sel.xcg_default, xd);
    if (st) {
#pragma unroll
      for (int i = 0; i < 18; i++) xd[i] = qnan();
    }
#pragma unroll
    for (int i = 0; i < 18; i++) xd_g[i * ld_out + n] = xd[i];
    if (status) status[n] = (int)st;
  }
}

// ------------------------------------------------------------------------------------------------------
// calc_xdot_batch: env.py::_calc_xdot for N aircraft
// ------------------------------------------------------------------------------------------------------
template <int FI, bool SMEM>
__global__ void __launch_bounds__(F16_THREADS, 1)
calc_xdot_kernel(DevTables tabs, BatchSel sel, const double* __restrict__ x_g, long long ld_x,
                 const double* __restrict__ u_g, long long ld_u, double* __restrict__ xd_g, long long ld_out,
                 long long N, int* __restrict__ status) {
  const double* img = acquire_tables<FI, SMEM>(tabs);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* buf = reinterpret_cast<double*>(f16_smem + PipeSmem<FI, SMEM, 22>::OFF) + warp * (22 * 32);
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  pipe_issue<18, 4>(buf, lane, x_g, ld_x, u_g, ld_u, n, n < N && owns<FI>(sel, n) != 0);
  for (; n < N; n += stride) {
    double xin[22], x[18], u[4], xd[18];
    pipe_take<22>(buf, lane, xin);
    const long long nn = n + stride;
    pipe_issue<18, 4>(buf, lane, x_g, ld_x, u_g, ld_u, nn, nn < N && owns<FI>(sel, nn) != 0);
#pragma unroll
    for (int i = 0; i < 18; i++) x[i] = xin[i];
#pragma unroll
    for (int i = 0; i < 4; i++) u[i] = xin[18 + i];
    const int own = owns<FI>(sel, n);
    if (own == 0) continue;
    unsigned st = ST_FIDELITY;
    if (own == 1) st = calc_xdot<FI>(img, x, u, sel.xcg ? sel.xcg[n] : sel.xcg_default, xd);
    if (st) {
#pragma unroll
      for (int i = 0; i < 18; i++) xd[i] = qnan();
    }
#pragma unroll
    for (int i = 0; i < 18; i++) xd_g[i * ld_out + n] = xd[i];
    if (status) status[n] = (int)st;
  }
}

// ------------------------------------------------------------------------------------------------------
// step_batch: K fused explicit-Euler steps of env.py::step, state in registers, optional fused LQR law
// ------------------------------------------------------------------------------------------------------
// The law travels as a kernel parameter (constant bank, like a __constant__ symbol, but owned by the launch: nothing to upload,
// nothing shared between launches, streams or devices).
template <int FI, bool SMEM, bool LQR, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
step_kernel(DevTables tabs, BatchSel sel, double* __restrict__ x_g, long long ld_x, const double* __restrict__ u_g,
            long long ld_u, long long N, int K, double dt, int* __restrict__ status, int* __restrict__ steps_done,
            const __grid_constant__ LqrLaw c_lqr) {
  const double* img = acquire_tables<FI, SMEM>(tabs);
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const int own = owns<FI>(sel, n);
    if (own == 0) continue;
    if (own < 0) {
      if (status) status[n] = (int)ST_FIDELITY;
      if (steps_done) steps_done[n] = 0;
      continue;
    }
    double x[18], u_in[4];
#pragma unroll
    for (int i = 0; i < 18; i++) x[i] = x_g[i * ld_x + n];
#pragma unroll
    for (int i = 0; i < 4; i++) u_in[i] = u_g[i * ld_u + n];
    const double xcg = sel.xcg ? sel.xcg[n] : sel.xcg_default;
    // env.py:117 -- the reference exit()s on a state outside its bounds; we freeze this aircraft.  The check is an integer
    // screen (bounds_screen) with step_bounds() behind it for a state the screen is not sure about, and it is asked about the
    // NEW state at the bottom of the loop body, where its integer instructions issue in the shadow of the step's FP64 tail
    // (same scheme as fastmath::run_steps; same bits as checking every state with step_bounds at the top).
    unsigned st = 0;
    int k = 0;
    bool go = false;
    if (K > 0) {
      go = !(either_nan(u_in[0], u_in[1]) || either_nan(u_in[2], u_in[3])) && bounds_screen(x);
      if (!go) {
        st = step_bounds(x, u_in);
        go = st == 0;
      }
    }
#pragma unroll 1
    while (go) {
      double u[4], xd[18];
      if (LQR) {
        lqr_action(c_lqr, x, u_in, u);
      } else {
#pragma unroll
        for (int i = 0; i < 4; i++) u[i] = u_in[i];
      }
      st = calc_xdot<FI>(img, x, u, xcg, xd);
      if (st) break;
#pragma unroll
      for (int i = 0; i < 18; i++) x[i] = x[i] + xd[i] * dt;  // env.py:126
      k++;
      go = bounds_screen(x);
      if (!go & (k < K)) {
        st = step_bounds(x, u_in);
        go = st == 0;
      }
      go &= k < K;
    }
#pragma unroll
    for (int i = 0; i < 18; i++) x_g[i * ld_x + n] = x[i];
    if (status) status[n] = (int)st;
    if (steps_done) steps_done[n] = k;
  }
}

// ------------------------------------------------------------------------------------------------------
// linearise_batch: finite-difference A [18x18], B [18x4] of _calc_xdot (env.py:294-342).
// CTA = 32 aircraft x F16_LIN_WARPS warps, lane = aircraft, so every warp is column-uniform.
//   phase A  the stages of f at the unperturbed point go to shared memory: one sin/cos pair per warp (five warps), the
//            atmosphere, the alpha-beta tables and the other tables (one warp each);
//   phase B  warp w evaluates perturbation columns w, w+W, ... of columns 2..16: calc_xdot_col recomputes only the stages
//            the perturbed component feeds (f16_model.cuh) -- bit-identical to a full evaluation.  npos / epos (columns
//            0, 1) feed nothing: those columns of A are exactly zero, as in the reference; lf1 and the four inputs
//            (columns 17..21) feed only the actuator rows 12..17, so they skip Nlplant altogether;
//   phase C  the padded shared tile is written out as contiguous [aircraft][18][18] / [aircraft][18][4] runs.
// The kernel is latency-bound (8 warps per SM: 255 registers, 105 KB tables + 101 KB tile): measured, 12- and 16-warp
// variants that keep the stages in shared memory, barrier-free warp-autonomous variants and a cost-balanced column deal all
// lose to this one through spills into a 28 KB L1 and instruction-cache misses; what paid was fewer passes (actuator-only
// columns), fewer instructions (div_by) and less code (one evaluation site, calls on the rare paths).
// ------------------------------------------------------------------------------------------------------
template <int FI>
struct LinSmem {
  static constexpr int TILE_OFF = (Img<FI>::SMEM_BYTES + 127) / 128 * 128;
  static constexpr int TILE_BYTES = 32 * F16_LIN_TILE_LD * 8;
  static constexpr int BASE_OFF = TILE_OFF + TILE_BYTES;  // f(x,u) per aircraft: [32][19]
  static constexpr int BASE_BYTES = 32 * 19 * 8;
  static constexpr int STAGE_OFF = BASE_OFF + BASE_BYTES;  // XdotBase as [61][32]
  static constexpr int STAGE_BYTES = XDOT_BASE_DOUBLES * 32 * 8;
  static constexpr int STAT_OFF = STAGE_OFF + STAGE_BYTES;
  static constexpr int TOTAL = STAT_OFF + 2 * 32 * 4;  // per-aircraft status, base-point envelope status
};

// XdotBase in shared memory as [field][lane]: fields 0..9 and 60 Trig, 10..15 the two Atmos, 16..59 Coef.  Explicit field lists
// (no pointer casts) keep the struct in registers.  XB_COEF_AB = what hifi_coefs_ab writes, XB_COEF_REST = the others.
#define XB_TRIG(X) X(0, tr.sa) X(1, tr.ca) X(2, tr.sb) X(3, tr.cb) X(4, tr.st) X(5, tr.ct) X(6, tr.sphi) X(7, tr.cphi) X(8, tr.spsi) X(9, tr.cpsi) X(60, tr.tt)
#define XB_ATMOS(X) X(10, al.mach) X(11, al.qbar) X(12, al.ps) X(13, an.mach) X(14, an.qbar) X(15, an.ps)
#define XB_COEF_AB(X) X(19, c.Cy) X(31, c.dCx_lef) X(32, c.dCz_lef) X(33, c.dCm_lef) X(34, c.dCy_lef) X(35, c.dCn_lef) X(36, c.dCl_lef) X(46, c.dCy_r30) X(47, c.dCn_r30) X(48, c.dCl_r30) X(49, c.dCy_a20) X(50, c.dCy_a20_lef) X(51, c.dCn_a20) X(52, c.dCn_a20_lef) X(53, c.dCl_a20) X(54, c.dCl_a20_lef)
#define XB_COEF_REST(X) X(16, c.Cx) X(17, c.Cz) X(18, c.Cm) X(20, c.Cn) X(21, c.Cl) X(22, c.Cxq) X(23, c.Cyr) X(24, c.Cyp) X(25, c.Czq) X(26, c.Clr) X(27, c.Clp) X(28, c.Cmq) X(29, c.Cnr) X(30, c.Cnp) X(37, c.dCxq_lef) X(38, c.dCyr_lef) X(39, c.dCyp_lef) X(40, c.dCzq_lef) X(41, c.dClr_lef) X(42, c.dClp_lef) X(43, c.dCmq_lef) X(44, c.dCnr_lef) X(45, c.dCnp_lef) X(55, c.dCnbeta) X(56, c.dClbeta) X(57, c.dCm) X(58, c.eta_el) X(59, c.dCm_ds)
#define XB_ST(k, f) stage[(k) * 32 + lane] = b.f;
#define XB_LD(k, f) b.f = stage[(k) * 32 + lane];

// The quotient of the finite difference, (f(x + eps e_c) - f(x)) / eps (env.py:330,339) or (f+ - f-) / (2 eps): the IEEE
// quotient through div_by (f16_model.cuh) -- most entries of a Jacobian are exactly 0, which the compiler's division
// sequence sends down its slow path.  The entry points accept steps in [1e-12, 1e3] only; the kernel still carries the
// plain division for a step outside [1e-15, 1e15] (never taken; with it ptxas lays the write-out loop out 8 % faster).
static __device__ __noinline__ double div_plain(double a, double y) { return a / y; }
struct FdQuot {
  double den, rden;
  bool inv_ok;
  __device__ __forceinline__ FdQuot(double eps, int scheme) {
    den = scheme == 0 ? eps : 2 * eps;
    rden = 1.0 / den;
    inv_ok = den >= 1e-15 && den <= 1e15;
  }
  __device__ __forceinline__ double operator()(double num) const { return inv_ok ? div_by(num, den, rden) : div_plain(num, den); }
  __device__ __forceinline__ double q(double num) const { return div_by(num, den, rden); }  // branch-free (write-out loop)
};

// evaluation order, dealt round-robin to the warps (warp w takes entries w and w + 8): the three columns that recompute the
// table look-ups are paired with plain columns, the sin/cos columns with each other; the base point last

__constant__ signed char c_lin_order[16] = {7, 8, 13, 2, 6, 14, 15, 3, 9, 10, 11, 12, 16, 4, 5, 22};

template <int FI>
__global__ void __launch_bounds__(F16_LIN_WARPS * 32, 1)
linearise_kernel(DevTables tabs, BatchSel sel, const double* __restrict__ x_g, long long ld_x,
                 const double* __restrict__ u_g, long long ld_u, long long N, double eps, int scheme,
                 double* __restrict__ A_g, double* __restrict__ B_g, int* __restrict__ status) {
  const double* img = acquire_tables<FI, true>(tabs);
  double* tile = reinterpret_cast<double*>(f16_smem + LinSmem<FI>::TILE_OFF);
  double* base = reinterpret_cast<double*>(f16_smem + LinSmem<FI>::BASE_OFF);
  double* stage = reinterpret_cast<double*>(f16_smem + LinSmem<FI>::STAGE_OFF);
  int* stat = reinterpret_cast<int*>(f16_smem + LinSmem<FI>::STAT_OFF);
  int* stat0 = stat + 32;  // envelope status of the unperturbed point
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const FdQuot fd(eps, scheme);
  const long long n_groups = (N + 31) / 32;
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const long long n = grp * 32 + lane;
    const bool live = n < N;
    const int own = live ? owns<FI>(sel, n) : 0;
    double x0[18], u0[4];
#pragma unroll
    for (int i = 0; i < 18; i++) x0[i] = live ? x_g[i * ld_x + n] : 0.0;
#pragma unroll
    for (int i = 0; i < 4; i++) u0[i] = live ? u_g[i * ld_u + n] : 0.0;
    const double xcg = (live && sel.xcg) ? sel.xcg[n] : sel.xcg_default;
    double xu0[17];
#pragma unroll
    for (int i = 0; i < 17; i++) xu0[i] = x0[i];
    const unsigned st_base = envelope_of<FI>(xu0);
    if (threadIdx.x < 32) {
      stat[lane] = (own < 0) ? (int)ST_FIDELITY : 0;
      stat0[lane] = (int)st_base;
    }
    // ---- phase A: the stages of f at the unperturbed point ----
    if (own == 1 && (warp == 0 || warp >= 4)) {  // one sin/cos pair per warp: alpha | beta, theta (+ tan), phi, psi
      const int k = warp == 0 ? 0 : warp - 3;
      const double ang = k == 0 ? xu0[7] : k == 1 ? xu0[8] : k == 2 ? xu0[4] : k == 3 ? xu0[3] : xu0[5];
      double sn, cs;
#if defined(__CUDA_ARCH__)
      // the five angles decide together, exactly as trig_eval does, so that the staged sines carry a full evaluation's bits
      const bool nb = trig_small(xu0[7]) & trig_small(xu0[8]) & trig_small(xu0[4]) & trig_small(xu0[3]) & trig_small(xu0[5]);
      if (nb) sincos_nb(ang, sn, cs);
      else
#endif
      sincos_pair(ang, sn, cs);
      stage[(2 * k) * 32 + lane] = sn;  // the field order of XB_TRIG
      stage[(2 * k + 1) * 32 + lane] = cs;
#if defined(__CUDA_ARCH__)
      if (k == 2) stage[60 * 32 + lane] = nb ? F16_DIV(sn, cs) : tan(xu0[4]);
#else
      if (k == 2) stage[60 * 32 + lane] = tan(xu0[4]);
#endif
    } else if (own == 1) {
      XdotBase b;
      if (warp == 1) {
        atmos_pair(x0, b.al, b.an);
        XB_ATMOS(XB_ST)
      } else if (!st_base) {
        const double r2d = 180.0 / 3.141592653589793;
        const double alpha = xu0[7] * r2d, beta = xu0[8] * r2d;
        if (FI == 1) {
          const HifiLoc L = hifi_locate(img, alpha, beta, xu0[13]);
          if (warp == 2) {
            hifi_coefs_ab(img, L, b.c);
            XB_COEF_AB(XB_ST)
          } else {
            hifi_coefs_rest(img, L, b.c);
            XB_COEF_REST(XB_ST)
          }
        } else if (warp == 2) {
          coef_eval<0>(img, alpha, beta, xu0[13], F16_DIVC(xu0[14], 21.5), F16_DIVC(xu0[15], 30.0), b.c);
          XB_COEF_AB(XB_ST) XB_COEF_REST(XB_ST)
        }
      }
    }
    __syncthreads();
    // ---- phase B: perturbation columns ----
    const int n_items = scheme == 0 ? 16 : 15;  // columns 2..16; forward also needs the unperturbed point (last item)
    for (int it = warp; it < n_items; it += F16_LIN_WARPS) {
      if (own != 1) continue;
      const int c = c_lin_order[it];
      const int col = c == 22 ? -1 : c;
      const bool reuse_coef = !col_feeds_coef<FI>(col);
      double* out = c == 22 ? base + lane * 19 : tile + lane * F16_LIN_TILE_LD + (c < 18 ? c : 324 + (c - 18));
      const int ld = c == 22 ? 1 : (c < 18 ? 18 : 4);
      unsigned st = 0;
#pragma unroll 1
      for (int pass = 0; pass < (scheme != 0 ? 2 : 1) && !st; pass++) {  // one evaluation site: half the code of two
        const double d = pass ? -eps : eps;
        double x[18], u[4], f[18];
        XdotBase b;
#pragma unroll
        for (int i = 0; i < 18; i++) x[i] = x0[i] + (i == c ? d : 0.0);
#pragma unroll
        for (int i = 0; i < 4; i++) u[i] = u0[i] + (i + 18 == c ? d : 0.0);
        XB_TRIG(XB_LD) XB_ATMOS(XB_LD)
        if (reuse_coef) { XB_COEF_AB(XB_LD) XB_COEF_REST(XB_LD) }
        st = calc_xdot_col<FI>(img, x, u, xcg, b, col, f);
        if (!st) {
#pragma unroll
          for (int r = 0; r < 18; r++) out[r * ld] = pass ? fd(out[r * ld] - f[r]) : f[r];  // central: f+ waits in the tile for f-
        }
      }
      if (st) {
        atomicOr(&stat[lane], (int)st);
#pragma unroll
        for (int r = 0; r < 18; r++) out[r * ld] = qnan();
      }
    }
    // columns 17 (lf1) and 18..21 (the inputs) reach f through actuator_xdot only: rows 0..11 are exact zeros (identical
    // bits on both sides of the difference) and rows 12..17 need no Nlplant evaluation -- a quarter of the passes saved
    if (own == 1 && warp >= 3) {
      const int c = 17 + (warp - 3);
      double* out = tile + lane * F16_LIN_TILE_LD + (c < 18 ? c : 324 + (c - 18));
      const int ld = c < 18 ? 18 : 4;
      if (st_base) {
        atomicOr(&stat[lane], (int)st_base);
#pragma unroll
        for (int r = 0; r < 18; r++) out[r * ld] = qnan();
      } else {
        Atmos al;
        al.mach = stage[10 * 32 + lane];
        al.qbar = stage[11 * 32 + lane];
        al.ps = stage[12 * 32 + lane];
        double x[18], u[4], f[18], g[18];
#pragma unroll
        for (int i = 0; i < 18; i++) x[i] = x0[i] + (i == c ? eps : 0.0);
#pragma unroll
        for (int i = 0; i < 4; i++) u[i] = u0[i] + (i + 18 == c ? eps : 0.0);
        actuator_xdot(x, u, al, f);
        if (scheme == 0) {
#pragma unroll
          for (int r = 12; r < 18; r++) out[r * ld] = f[r];  // rows 0..11: the write-out knows they are zero
        } else {
#pragma unroll
          for (int i = 0; i < 18; i++) x[i] = x0[i] - (i == c ? eps : 0.0);
#pragma unroll
          for (int i = 0; i < 4; i++) u[i] = u0[i] - (i + 18 == c ? eps : 0.0);
          actuator_xdot(x, u, al, g);
#pragma unroll
          for (int r = 0; r < 12; r++) out[r * ld] = 0.0;
#pragma unroll
          for (int r = 12; r < 18; r++) out[r * ld] = fd(f[r] - g[r]);
        }
      }
    }
    __syncthreads();
    // ---- phase C: write-out, 32 aircraft x 324 (A) and x 72 (B) contiguous doubles ----
    const long long n0 = grp * 32;
    const int n_here = (int)((N - n0) < 32 ? (N - n0) : 32);
    // one warp per aircraft, lanes along the 396 contiguous output doubles (A then B): no per-element divisions
    for (int a = warp; a < n_here; a += F16_LIN_WARPS) {
      if (owns<FI>(sel, n0 + a) == 0) continue;
      const bool void_all = (stat[a] & (int)ST_FIDELITY) != 0;
      const double zero_col = stat0[a] ? qnan() : 0.0;  // d f / d npos, d f / d epos: f does not read them
      const double* t = tile + a * F16_LIN_TILE_LD;
      const double* f0 = base + a * 19;
      double* Ao = A_g + (n0 + a) * 324;
      double* Bo = B_g + (n0 + a) * 72;
#pragma unroll
      for (int j = 0; j < 11; j++) {  // 324 = 10 * 32 + 4
        const int k = j * 32 + lane;
        if (k < 324) {
          const int r = k / 18, col = k - r * 18;
          double v = t[k];
          if (scheme == 0) {  // env.py:330; the quotient is formed for every element and selected afterwards: a branch
            const double qv = fd.q(v - f0[r]);  // around it would stop the 11 independent chains from interleaving
            v = (col == 17 && r < 12) ? zero_col : qv;
          }
          if (col < 2) v = zero_col;
          if (void_all) v = qnan();
          Ao[k] = v;
        }
      }
#pragma unroll
      for (int j = 0; j < 3; j++) {  // 72 = 2 * 32 + 8
        const int k = j * 32 + lane;
        if (k < 72) {
          double v = t[324 + k];
          if (scheme == 0) {  // env.py:339; rows 0..11 of B are zero
            const double qv = fd.q(v - f0[k >> 2]);
            v = k < 48 ? zero_col : qv;
          }
          if (void_all) v = qnan();
          Bo[k] = v;
        }
      }
    }
    if (status && threadIdx.x < n_here && owns<FI>(sel, n0 + threadIdx.x) != 0)
      status[n0 + threadIdx.x] = stat[threadIdx.x] | ((stat[threadIdx.x] & (int)ST_FIDELITY) ? 0 : stat0[threadIdx.x]);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------------
// trim_batch: env.py::trim (Nelder-Mead, ~2000 objective evaluations) for N flight conditions, one thread each.
// The simplex lives in registers (f16_model.cuh::nelder_mead_trim); lanes differ only in how many iterations they need.
// ------------------------------------------------------------------------------------------------------
#define F16_TRIM_THREADS 256

template <int FI, bool SMEM>
__global__ void __launch_bounds__(F16_TRIM_THREADS, 1)
trim_kernel(DevTables tabs, BatchSel sel, const double* __restrict__ h_g, const double* __restrict__ v_g, long long N, double tol,
            int maxiter, TrimGuess guess, double* __restrict__ x_g, long long ld_x, double* __restrict__ info_g, long long ld_info,
            int* __restrict__ status) {
  const double* img = acquire_tables<FI, SMEM>(tabs);
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const int own = owns<FI>(sel, n);
    if (own == 0) continue;
    double x[18];
    TrimResult r;
    if (own == 1) {
      double ux[5];
#pragma unroll
      for (int k = 0; k < 5; k++) ux[k] = guess.ux[k];
      const TrimPoint t = trim_point(h_g[n], v_g[n]);
      r = nelder_mead_trim<FI>(img, t, sel.xcg ? sel.xcg[n] : sel.xcg_default, tol, maxiter, ux, guess.fixed_point_exit != 0);
      trim_state(t, ux, x);  // env.py:275-288: the optimiser's (unclipped) point
    } else {
      r.cost = qnan(); r.iterations = 0; r.fcalls = 0; r.converged = 0; r.status = ST_FIDELITY;
#pragma unroll
      for (int i = 0; i < 18; i++) x[i] = qnan();
    }
#pragma unroll
    for (int i = 0; i < 18; i++) x_g[i * ld_x + n] = x[i];
    if (info_g) {
      info_g[n] = r.cost;
      info_g[ld_info + n] = (double)r.iterations;
      info_g[2 * ld_info + n] = (double)r.fcalls;
      info_g[3 * ld_info + n] = (double)r.converged;
    }
    if (status) status[n] = (int)r.status;
  }
}

// ------------------------------------------------------------------------------------------------------
// parity probes
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
hifi_probe_kernel(DevTables tabs, const double* __restrict__ alpha, const double* __restrict__ beta,
                  const double* __restrict__ el, long long N, double* __restrict__ coef, int* __restrict__ cells,
                  int* __restrict__ status) {
  const double* img = tabs.hifi;
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const double a = alpha[n], b = beta[n], e = el[n];
    const unsigned st = hifi_envelope(a, b, e);
    double o[44];
    int cl[8];
    if (st) {
#pragma unroll
      for (int i = 0; i < 44; i++) o[i] = qnan();
#pragma unroll
      for (int i = 0; i < 8; i++) cl[i] = -1;
    } else {
      const HifiLoc L = hifi_locate(img, a, b, e);
      Coef c;
      hifi_coefs(img, L, c);
      o[0] = c.Cx; o[1] = c.Cz; o[2] = c.Cm; o[3] = c.Cy; o[4] = c.Cn; o[5] = c.Cl;
      o[6] = c.Cxq; o[7] = c.Cyr; o[8] = c.Cyp; o[9] = c.Czq; o[10] = c.Clr; o[11] = c.Clp; o[12] = c.Cmq;
      o[13] = c.Cnr; o[14] = c.Cnp;
      o[15] = c.dCx_lef; o[16] = c.dCz_lef; o[17] = c.dCm_lef; o[18] = c.dCy_lef; o[19] = c.dCn_lef; o[20] = c.dCl_lef;
      o[21] = c.dCxq_lef; o[22] = c.dCyr_lef; o[23] = c.dCyp_lef; o[24] = c.dCzq_lef; o[25] = c.dClr_lef;
      o[26] = c.dClp_lef; o[27] = c.dCmq_lef; o[28] = c.dCnr_lef; o[29] = c.dCnp_lef;
      o[30] = c.dCy_r30; o[31] = c.dCn_r30; o[32] = c.dCl_r30;
      o[33] = c.dCy_a20; o[34] = c.dCy_a20_lef; o[35] = c.dCn_a20; o[36] = c.dCn_a20_lef; o[37] = c.dCl_a20;
      o[38] = c.dCl_a20_lef;
      o[39] = c.dCnbeta; o[40] = c.dClbeta; o[41] = c.dCm; o[42] = c.eta_el; o[43] = c.dCm_ds;
      ref_cell(img + F16_IMG_A, L.a, a, cl[0], cl[1]);
      ref_cell(img + F16_IMG_B, L.b, b, cl[2], cl[3]);
      ref_cell(img + F16_IMG_D1, L.d1, e, cl[4], cl[5]);
      ref_cell(img + F16_IMG_D2, L.d2, e, cl[6], cl[7]);
    }
#pragma unroll
    for (int i = 0; i < 44; i++) coef[i * N + n] = o[i];
#pragma unroll
    for (int i = 0; i < 8; i++) cells[i * N + n] = cl[i];
    if (status) status[n] = (int)st;
  }
}

__global__ void __launch_bounds__(256)
lofi_probe_kernel(DevTables tabs, const double* __restrict__ alpha, const double* __restrict__ beta,
                  const double* __restrict__ el, const double* __restrict__ dail, const double* __restrict__ drud,
                  long long N, double* __restrict__ out) {
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    Coef c;
    lofi_coefs(tabs.lofi, alpha[n], beta[n], el[n], dail[n], drud[n], c);
    const double o[19] = {c.Cxq, c.Cyr, c.Cyp, c.Czq, c.Clr, c.Clp, c.Cmq, c.Cnr, c.Cnp, c.dCl_a20,
                          c.dCl_r30, c.dCn_a20, c.dCn_r30, c.Cl, c.Cn, c.Cx, c.Cm, c.Cz, c.Cy};
#pragma unroll
    for (int i = 0; i < 19; i++) out[i * N + n] = o[i];
  }
}

__global__ void __launch_bounds__(256)
atmos_kernel(const double* __restrict__ alt, const double* __restrict__ vt, long long N, double* __restrict__ coeff) {
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const Atmos a = atmos_eval(alt[n], vt[n]);
    coeff[n] = a.mach;
    coeff[N + n] = a.qbar;
    coeff[2 * N + n] = a.ps;
  }
}

// ------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------
template <int FI>
static int table_smem(bool smem_tables) { return smem_tables ? Img<FI>::SMEM_BYTES : 0; }

cudaError_t launch_nlplant(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* xu,
                           long long ld_in, double* xdot, long long ld_out, long long N, int* status) {
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  const bool s = cfg.smem_tables;
  if (wants(sel, 1))
    e = launch_persistent(cfg, s ? nlplant_kernel<1, true> : nlplant_kernel<1, false>, F16_THREADS,
                          s ? PipeSmem<1, true, 17>::TOTAL : PipeSmem<1, false, 17>::TOTAL, N, F16_THREADS, tabs, sel, xu, ld_in,
                          xdot, ld_out, N, status);
  if (e == cudaSuccess && wants(sel, 0))
    e = launch_persistent(cfg, s ? nlplant_kernel<0, true> : nlplant_kernel<0, false>, F16_THREADS,
                          s ? PipeSmem<0, true, 17>::TOTAL : PipeSmem<0, false, 17>::TOTAL, N, F16_THREADS, tabs, sel, xu, ld_in,
                          xdot, ld_out, N, status);
  return e;
}

cudaError_t launch_calc_xdot(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* x,
                             long long ld_x, const double* u, long long ld_u, double* xdot, long long ld_out,
                             long long N, int* status) {
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  const bool s = cfg.smem_tables;
  if (wants(sel, 1))
    e = launch_persistent(cfg, s ? calc_xdot_kernel<1, true> : calc_xdot_kernel<1, false>, F16_THREADS,
                          s ? PipeSmem<1, true, 22>::TOTAL : PipeSmem<1, false, 22>::TOTAL, N, F16_THREADS, tabs, sel, x, ld_x, u,
                          ld_u, xdot, ld_out, N, status);
  if (e == cudaSuccess && wants(sel, 0))
    e = launch_persistent(cfg, s ? calc_xdot_kernel<0, true> : calc_xdot_kernel<0, false>, F16_THREADS,
                          s ? PipeSmem<0, true, 22>::TOTAL : PipeSmem<0, false, 22>::TOTAL, N, F16_THREADS, tabs, sel, x, ld_x, u,
                          ld_u, xdot, ld_out, N, status);
  return e;
}

using StepKern = void (*)(DevTables, BatchSel, double*, long long, const double*, long long, long long, int, double, int*,
                          int*, const LqrLaw);

// 384 threads with the tables staged, 256 with the tables read through L2 (the other CTA sizes measured slower: DESIGN.md)
template <int FI, bool LQR>
static StepKern step_kern(bool smem_tables) {
  return smem_tables ? step_kernel<FI, true, LQR, 384> : step_kernel<FI, false, LQR, 256>;
}

cudaError_t launch_step(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, double* x, long long ld_x,
                        const double* u, long long ld_u, long long N, int K, double dt, const LqrLaw* lqr_host,
                        int* status, int* steps_done) {
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  const int threads = cfg.smem_tables ? 384 : 256;
  for (int FI = 1; FI >= 0 && e == cudaSuccess; FI--) {
    if (!wants(sel, FI)) continue;
    StepKern k = FI ? (lqr_host ? step_kern<1, true>(cfg.smem_tables) : step_kern<1, false>(cfg.smem_tables))
                    : (lqr_host ? step_kern<0, true>(cfg.smem_tables) : step_kern<0, false>(cfg.smem_tables));
    const int smem = FI ? table_smem<1>(cfg.smem_tables) : table_smem<0>(cfg.smem_tables);
    e = launch_persistent(cfg, k, threads, smem, N, threads, tabs, sel, x, ld_x, u, ld_u, N, K, dt, status, steps_done,
                          lqr_host ? *lqr_host : LqrLaw());
  }
  return e;
}

cudaError_t launch_linearise(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* x,
                             long long ld_x, const double* u, long long ld_u, long long N, double eps, int scheme,
                             double* A, double* B, int* status) {
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  const long long groups = (N + 31) / 32;
  const int threads = F16_LIN_WARPS * 32;
  if (wants(sel, 1))
    e = launch_persistent(cfg, linearise_kernel<1>, threads, LinSmem<1>::TOTAL, groups, 1, tabs, sel, x, ld_x, u, ld_u,
                          N, eps, scheme, A, B, status);
  if (e == cudaSuccess && wants(sel, 0))
    e = launch_persistent(cfg, linearise_kernel<0>, threads, LinSmem<0>::TOTAL, groups, 1, tabs, sel, x, ld_x, u, ld_u,
                          N, eps, scheme, A, B, status);
  return e;
}

cudaError_t launch_trim(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* h, const double* v,
                        long long N, double tol, int maxiter, const double* ux0, double* x_trim, long long ld_x, double* info,
                        long long ld_info, int* status) {
  if (N <= 0) return cudaSuccess;
  TrimGuess g;
  for (int k = 0; k < 5; k++) g.ux[k] = ux0[k];
  g.fixed_point_exit = cfg.trim_fixed_point_exit ? 1 : 0;
  cudaError_t e = cudaSuccess;
  const bool s = cfg.smem_tables;
  if (wants(sel, 1))
    e = launch_persistent(cfg, s ? trim_kernel<1, true> : trim_kernel<1, false>, F16_TRIM_THREADS, table_smem<1>(s), N,
                          F16_TRIM_THREADS, tabs, sel, h, v, N, tol, maxiter, g, x_trim, ld_x, info, ld_info, status);
  if (e == cudaSuccess && wants(sel, 0))
    e = launch_persistent(cfg, s ? trim_kernel<0, true> : trim_kernel<0, false>, F16_TRIM_THREADS, table_smem<0>(s), N,
                          F16_TRIM_THREADS, tabs, sel, h, v, N, tol, maxiter, g, x_trim, ld_x, info, ld_info, status);
  return e;
}

// parity probe of the two exact-division helpers: out[0][n] = F16_DIV(a, b), out[1][n] = div_by(a, b, RN(1 / b)), out[2][n] = a / b
__global__ void __launch_bounds__(256)
div_probe_kernel(const double* __restrict__ a, const double* __restrict__ b, long long N, double* __restrict__ out) {
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const double x = a[n], y = b[n];
    out[n] = F16_DIV(x, y);
    out[N + n] = div_by(x, y, 1.0 / y);
    out[2 * N + n] = x / y;
  }
}

cudaError_t launch_div_probe(const LaunchCfg& cfg, const double* a, const double* b, long long N, double* out) {
  if (N <= 0) return cudaSuccess;
  div_probe_kernel<<<grid_for(N, 256, cfg.sm_count * 8), 256, 0, cfg.stream>>>(a, b, N, out);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

cudaError_t launch_hifi_probe(const LaunchCfg& cfg, const DevTables& tabs, const double* alpha, const double* beta,
                              const double* el, long long N, double* coef, int* cells, int* status) {
  if (N <= 0) return cudaSuccess;
  hifi_probe_kernel<<<grid_for(N, 256, cfg.sm_count * 8), 256, 0, cfg.stream>>>(tabs, alpha, beta, el, N, coef, cells,
                                                                                status);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

cudaError_t launch_lofi_probe(const LaunchCfg& cfg, const DevTables& tabs, const double* alpha, const double* beta,
                              const double* el, const double* dail, const double* drud, long long N, double* out) {
  if (N <= 0) return cudaSuccess;
  lofi_probe_kernel<<<grid_for(N, 256, cfg.sm_count * 8), 256, 0, cfg.stream>>>(tabs, alpha, beta, el, dail, drud, N,
                                                                                out);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

cudaError_t launch_atmos(const LaunchCfg& cfg, const double* alt, const double* vt, long long N, double* coeff) {
  if (N <= 0) return cudaSuccess;
  atmos_kernel<<<grid_for(N, 256, cfg.sm_count * 8), 256, 0, cfg.stream>>>(alt, vt, N, coeff);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

}  // namespace strict
}  // namespace f16

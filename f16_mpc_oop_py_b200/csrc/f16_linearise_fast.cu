// f16_linearise_fast.cu -- linearise_batch in F16_MATH_FAST: finite-difference A [18x18], B [18x4] of _calc_xdot
// (env.py:294-342: forward differences, eps on every state / input; and the central scheme) on the arithmetic of
// f16_fast.cuh.  Compiled like f16_step_fast.cu (-fmad=false, explicit fma()).
//
// The strict kernel (f16_kernels.cu: CTA = 32 aircraft x 8 warps, stages of f shared between columns through shared
// memory, three barriers and a 101 KB transposing tile per group) is bound by latency: 252 registers -> 8 warps per SM, FP64
// pipe 31 % busy.  A full evaluation on the fast arithmetic is ~640 instructions, which makes a barrier-free mapping
// affordable:
//
//   * a warp-task is TWO aircraft; the 16 lanes of a half-warp are the 15 perturbation columns that need Nlplant (states
//     2..16: h, phi, theta, psi, V, alpha, beta, p, q, r, T, dh, da, dr, lf2) plus the unperturbed point.  Every lane runs the
//     same code on its own perturbed copy of the state -- no divergence, and the 16 lanes of an aircraft gather from the same
//     table cells (broadcast);
//   * columns 0, 1 (npos, epos) feed nothing: exact zeros, as in the reference.  Columns 17 (lf1) and the four inputs reach
//     f through rows 12..17 only (fastmath::actuator_rows): lanes 0..4 re-evaluate those six rows with the flap-schedule
//     terms of the unperturbed point, rows 0..11 are exact zeros (identical bits on both sides of the difference);
//   * central scheme: f(x + eps e_c) waits in a per-thread shared-memory slot (18 doubles) while f(x - eps e_c) is computed
//     at the same evaluation site;
//   * the quotient is the IEEE quotient (div_by), formed in registers; row r of A is then 16 consecutive doubles (columns
//     2..17) held by the 16 lanes: one 128-byte store per row straight from registers, no transposing tile.  A block of A
//     (2592 B) and of B (576 B) is written completely by one half-warp within a few hundred cycles, so L2 sees whole sectors;
//   * an aircraft with any evaluation outside the preconditions of the fast arithmetic or outside the tables is marked and
//     redone after the main loop on the reference-order arithmetic (f16_model.cuh, tables in global memory), which also
//     produces the status word and the NaN columns of the strict kernel.
#include <stdlib.h>

#include "f16_kernels_common.cuh"
#include "f16_fast.cuh"

namespace f16 {
namespace fast {

// CTA size and scheme.  The kernel is instantiated per scheme: with the scheme a compile-time constant the forward kernel has no
// second pass, no stash and no stash memory (L1 keeps 90 KB instead of 8), the central kernel no base-point shuffles.  Measured at
// 2^20 points, A,B pairs per second:
//   one kernel for both schemes (scheme a run-time argument), 256 threads / 255 registers: central 6.07e8, forward 9.1e8
//       (384 threads / 168 registers: 5.6e8 / 7.9e8 -- two spills, reloaded from L2 with 220 KB of shared memory in use;
//        320 / 288 / 224 / 192 threads: all slower)
//   per-scheme kernels, 256 threads both: central 6.27e8, forward 1.08e9
//   forward kernel at 384 threads / 168 registers (12 warps per SM; its 24 bytes of spills stay in L1): 1.11e9  <- forward
//   forward kernel at 320 threads: 1.00e9 (uneven warps per scheduler)
//   central kernel: 256 threads / 255 registers, no spills (the 55 KB stash of a 384-thread CTA leaves no L1)  <- central
constexpr int LF_THREADS_CENTRAL = 256, LF_THREADS_FORWARD = 384;
constexpr int LF_IN_LD = 24;  // 18 states + 4 inputs (+ 2 pad) per staged aircraft

template <int FI, int THREADS, bool CENTRAL>
struct LfSmem {
  static constexpr int IMG_BYTES = FI ? F16_FI_BYTES : F16_LOFI_STEP_IMG_DOUBLES * 8;
  static constexpr int BAR_OFF = (IMG_BYTES + 15) / 16 * 16;
  static constexpr int STASH_OFF = (BAR_OFF + 16 + 127) / 128 * 128;
  // stash: f(x + eps e_c) of the central scheme, [18][thread]; the forward instantiation has none
  static constexpr int IN_OFF = STASH_OFF + (CENTRAL ? 18 * THREADS * 8 : 0);
  static constexpr int TOTAL = IN_OFF + (THREADS / 32) * 2 * 2 * LF_IN_LD * 8;  // per warp: 2 stages x 2 aircraft x 24 doubles
};

// (f+ - f-) / den (the reference divides, env.py:330,339).  The reference-order pass forms the IEEE quotient (div_by); the fast
// pass multiplies by the rounded reciprocal: one ulp of the quotient, against a numerator that carries 1e5 ulp of f.
struct LinQuot {
  double den, rden;
  __device__ __forceinline__ LinQuot(double eps, int scheme) {
    den = scheme == 0 ? eps : 2 * eps;
    rden = 1.0 / den;
  }
  __device__ __forceinline__ double operator()(double num) const { return div_by(num, den, rden); }
  __device__ __forceinline__ double fast(double num) const { return num * rden; }
};

__device__ __forceinline__ void cp_async8(double* dst_smem, const double* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ double shfl_half(double v, int src_in_half) { return __shfl_sync(0xffffffffu, v, src_in_half, 16); }

// x0 with component `col` moved by d (col outside 0..17: unchanged).  A select per element, not an addition of zero: -0.0
// stays -0.0.
__device__ __forceinline__ void perturbed(const double (&x0)[18], int col, double d, double (&x)[18]) {
#pragma unroll
  for (int i = 0; i < 18; i++) x[i] = (i == col) ? x0[i] + d : x0[i];
}

// What one half-warp writes for its aircraft.  q[r]: rows of this lane's column (lane j < 15: state column 2 + j);
// actq[i]: rows 12 + i of column 17 + j (lanes j < 5); c17[i]: lane 0's actq[i]; zero_col: 0, or NaN when the unperturbed point
// has no value.  No shuffles in here: the two halves of a warp may take different branches around the call.
__device__ __forceinline__ void lin_store(double* __restrict__ A_g, double* __restrict__ B_g, int* __restrict__ status, long long n,
                                          int j, const double (&q)[18], const double (&actq)[6], const double (&c17)[6],
                                          double zero_col, bool void_all, int st) {
  double* Ao = A_g + n * 324;
  double* Bo = B_g + n * 72;
  const double nanv = qnan();
#pragma unroll
  for (int r = 0; r < 18; r++) {
    double v = q[r];
    // column 17 (lf1) is stored by lane 15: rows 12..17 are lane 0's actuator rows (c17, shuffled by the caller), rows 0..11 zero
    if (j == 15) v = r < 12 ? zero_col : c17[r < 12 ? 0 : r - 12];
    if (void_all) v = nanv;
    Ao[r * 18 + 2 + j] = v;                                      // columns 2..17: 16 consecutive doubles
    if (j < 2) Ao[r * 18 + j] = void_all ? nanv : zero_col;      // columns 0, 1: f reads neither npos nor epos
  }
#pragma unroll
  for (int k = 0; k < 3; k++) Bo[16 * k + j] = void_all ? nanv : zero_col;  // rows 0..11 of B
  if (j >= 1 && j <= 4) {
#pragma unroll
    for (int i = 0; i < 6; i++) Bo[(12 + i) * 4 + (j - 1)] = void_all ? nanv : actq[i];
  }
  if (status && j == 0) status[n] = st;
}

// ------------------------------------------------------------------------------------------------------
// rare path: one marked aircraft per half-warp on the reference-order arithmetic, full evaluations for every column
// ------------------------------------------------------------------------------------------------------
template <int FI>
static __device__ __noinline__ void lin_redo_pass(DevTables tabs, BatchSel sel, const double* __restrict__ x_g, long long ld_x,
                                                  const double* __restrict__ u_g, long long ld_u, long long N, double eps, int scheme,
                                                  double* __restrict__ A_g, double* __restrict__ B_g, int* __restrict__ status,
                                                  const unsigned* redo, long long t, long long stride, long long n_tasks, int lane) {
  const double* img = FI ? tabs.hifi : tabs.lofi;
  const int half = lane >> 4, j = lane & 15;
  const LinQuot fd(eps, scheme);
#pragma unroll 1
  for (; t < n_tasks; t += stride) {
    const unsigned word = redo[t];
    if (!word) continue;  // warp-uniform
    const long long n = 2 * t + half;
    const bool mine = ((word >> half) & 1u) != 0 && n < N;
    double x0[18], u0[4];
#pragma unroll
    for (int i = 0; i < 18; i++) x0[i] = mine ? x_g[i * ld_x + n] : 0.0;
#pragma unroll
    for (int i = 0; i < 4; i++) u0[i] = mine ? u_g[i * ld_u + n] : 0.0;
    const double xcg = (mine && sel.xcg) ? sel.xcg[n] : sel.xcg_default;
    double xu0[17];
#pragma unroll
    for (int i = 0; i < 17; i++) xu0[i] = x0[i];
    const unsigned st_base = envelope_of<FI>(xu0);
    unsigned stat = 0;
    double q[18], actq[6], fp[18];
    // columns 2..16 and the unperturbed point (lane 15)
    {
      const int col = j < 15 ? 2 + j : -1;
      unsigned st = 0;
#pragma unroll 1
      for (int pass = 0; pass < (scheme != 0 ? 2 : 1); pass++) {
        double x[18], f[18];
        perturbed(x0, col, pass ? -eps : eps, x);
        unsigned s1 = (mine && !(scheme != 0 && j == 15)) ? calc_xdot<FI>(img, x, u0, xcg, f) : 0u;
        st |= s1;
#pragma unroll
        for (int r = 0; r < 18; r++) {
          const double v = s1 ? qnan() : f[r];
          if (pass == 0) fp[r] = v;
          else q[r] = fd(fp[r] - v);
        }
      }
      if (scheme == 0) {
#pragma unroll
        for (int r = 0; r < 18; r++) q[r] = fd(fp[r] - shfl_half(fp[r], 15));  // a NaN base makes every quotient NaN
      }
      if (st) {
#pragma unroll
        for (int r = 0; r < 18; r++) q[r] = qnan();
      }
      stat |= st;
    }
    // columns 17..21 on lanes 0..4: rows 12..17 (rows 0..11 are exact zeros)
    {
      const int c = 17 + j;  // lanes >= 5 compute nothing that is stored
      double fa[18], fb[18];
      double x[18], u[4];
      perturbed(x0, c, eps, x);
#pragma unroll
      for (int i = 0; i < 4; i++) u[i] = (18 + i == c) ? u0[i] + eps : u0[i];
      const bool act = mine && j < 5 && !st_base;
      if (act) calc_xdot<FI>(img, x, u, xcg, fa);
      if (scheme != 0) {
        perturbed(x0, c, -eps, x);
#pragma unroll
        for (int i = 0; i < 4; i++) u[i] = (18 + i == c) ? u0[i] - eps : u0[i];
        if (act) calc_xdot<FI>(img, x, u, xcg, fb);
      }
#pragma unroll
      for (int i = 0; i < 6; i++) {
        const double base_row = shfl_half(fp[12 + i], 15);
        const double num = scheme != 0 ? fa[12 + i] - fb[12 + i] : fa[12 + i] - base_row;
        actq[i] = act ? fd(num) : qnan();
      }
      if (st_base) stat |= st_base;
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) stat |= __shfl_xor_sync(0xffffffffu, stat, o, 16);
    double c17[6];
#pragma unroll
    for (int i = 0; i < 6; i++) c17[i] = shfl_half(actq[i], 0);
    if (mine) lin_store(A_g, B_g, status, n, j, q, actq, c17, st_base ? qnan() : 0.0, false, (int)(stat | st_base));
  }
}

// One instantiation per scheme (the scheme is a compile-time constant inside: the forward kernel carries no second pass, no stash
// and no stash memory) and CTA size (LF_THREADS_FORWARD / LF_THREADS_CENTRAL above).
template <int FI, int LF_THREADS, bool CENTRAL>
__global__ void __launch_bounds__(LF_THREADS, 1)
linearise_fast_kernel(DevTables tabs, BatchSel sel, const double* __restrict__ x_g, long long ld_x, const double* __restrict__ u_g,
                      long long ld_u, long long N, double eps, double* __restrict__ A_g, double* __restrict__ B_g,
                      int* __restrict__ status, unsigned* __restrict__ redo) {
  using S = LfSmem<FI, LF_THREADS, CENTRAL>;
  constexpr int scheme = CENTRAL ? 1 : 0;
  const double* img = reinterpret_cast<const double*>(f16_smem);
  if (FI) {
    stage_tables_tma<F16_FI_BYTES>(f16_smem, tabs.hifi_fast, reinterpret_cast<unsigned long long*>(f16_smem + S::BAR_OFF));
  } else {
    double* li = reinterpret_cast<double*>(f16_smem);
    for (int i = threadIdx.x; i < F16_LOFI_STEP_IMG_DOUBLES; i += LF_THREADS)
      li[i] = i < F16_IMG_LOFI_DOUBLES ? tabs.lofi[i] : tabs.hifi_fast[F16_FI_POW + (i - F16_IMG_LOFI_DOUBLES)];
    __syncthreads();
  }
  double* stash = reinterpret_cast<double*>(f16_smem + S::STASH_OFF) + threadIdx.x;  // element r at stash[r * LF_THREADS]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, half = lane >> 4, j = lane & 15;
  // input staging: the 22 doubles of each of a task's two aircraft, two stages per warp, filled by cp.async one task ahead
  double* inbuf = reinterpret_cast<double*>(f16_smem + S::IN_OFF) + warp * (2 * 2 * LF_IN_LD);
  const LinQuot fd(eps, scheme);
  const long long n_tasks = (N + 1) >> 1;
  const long long stride = (long long)(LF_THREADS / 32) * gridDim.x;
  const long long t0 = (long long)warp * gridDim.x + blockIdx.x;  // warp-major slots: a partial last round covers all SMs
  const double* src = lane < 18 ? x_g + lane * ld_x : u_g + (lane < 22 ? lane - 18 : 0) * ld_u;  // the plane this lane fetches
  auto prefetch = [&](long long task, int stage) {
    if (task < n_tasks && lane < 22) {
      const long long na = 2 * task;
      double* dst = inbuf + stage * (2 * LF_IN_LD) + lane;
      cp_async8(dst, src + na);
      if (na + 1 < N) cp_async8(dst + LF_IN_LD, src + na + 1);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  prefetch(t0, 0);
  unsigned any_redo = 0;
  int stage = 0;
  const int col = j < 15 ? 2 + j : -1;
  for (long long t = t0; t < n_tasks; t += stride, stage ^= 1) {
    const long long n = 2 * t + half;
    const int own = n < N ? owns<FI>(sel, n) : 0;
    const bool mine = own == 1;
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    double x0[18], u0[4];
    {
      const double* row = inbuf + stage * (2 * LF_IN_LD) + half * LF_IN_LD;
#pragma unroll
      for (int i = 0; i < 18; i++) x0[i] = row[i];   // a half without an aircraft of this launch computes on whatever the slot
#pragma unroll
      for (int i = 0; i < 4; i++) u0[i] = row[18 + i];  // holds: nothing of it is stored, and `ok` ignores it
    }
    prefetch(t + stride, stage ^ 1);
    const double xcg = (mine && sel.xcg) ? sel.xcg[n] : sel.xcg_default;
    double uc[4];
    fastmath::clip_commands(u0, uc);
    bool ok = true;
    double q[18], aux[2] = {0.0, 0.0};
    {
      double f[18];
#pragma unroll 1
      for (int pass = 0; pass < (scheme != 0 ? 2 : 1); pass++) {  // one evaluation site
        const double d = pass ? -eps : eps;
        double x[18];
        x[0] = x0[0]; x[1] = x0[1]; x[17] = x0[17];
#pragma unroll
        for (int i = 2; i < 17; i++) x[i] = (i == col) ? x0[i] + d : x0[i];  // a select, not "+ 0": -0.0 stays -0.0
        double a2[2];
        bool k = fastmath::fast_ok<FI>(x);
        if (k) k = FI ? fastmath::calc_xdot_hifi<false, false, true>(img, x, uc, xcg, f, a2)
                      : fastmath::calc_xdot_lofi<false, false, true>(img, x, uc, xcg, f, a2);
        ok &= k | !mine | (pass == 1 && j == 15);
        if (pass == 0) {
          aux[0] = a2[0];
          aux[1] = a2[1];
          if (scheme != 0) {
#pragma unroll
            for (int r = 0; r < 18; r++) stash[r * LF_THREADS] = f[r];
          }
        }
      }
      if (scheme != 0) {
#pragma unroll
        for (int r = 0; r < 18; r++) q[r] = fd.fast(stash[r * LF_THREADS] - f[r]);
      } else {
#pragma unroll
        for (int r = 0; r < 18; r++) q[r] = fd.fast(f[r] - shfl_half(f[r], 15));
      }
      // rows 12..17 of the unperturbed point for the forward quotients of the actuator-only columns
#pragma unroll
      for (int i = 0; i < 6; i++) f[i] = shfl_half(f[12 + i], 15);
      // ---- columns 17 (lf1) and 18..21 (inputs) on lanes 0..4: rows 12..17 only ----
      const double a_out = shfl_half(aux[0], 15), a_deg = shfl_half(aux[1], 15);
      double actq[6];
      {
        // only x[12..17] and the commands enter actuator_rows: lane 0 moves lf1, lanes 1..4 one command each
        double xa[18], ua[4], uca[4], rp[18], rm[18];
#pragma unroll
        for (int i = 0; i < 17; i++) xa[i] = x0[i];
        xa[17] = j == 0 ? x0[17] + eps : x0[17];
#pragma unroll
        for (int i = 0; i < 4; i++) ua[i] = (1 + i == j) ? u0[i] + eps : u0[i];
        fastmath::clip_commands(ua, uca);
        fastmath::actuator_rows(xa, uca, a_out, a_deg, rp);
        if (scheme != 0) {
          xa[17] = j == 0 ? x0[17] - eps : x0[17];
#pragma unroll
          for (int i = 0; i < 4; i++) ua[i] = (1 + i == j) ? u0[i] - eps : u0[i];
          fastmath::clip_commands(ua, uca);
          fastmath::actuator_rows(xa, uca, a_out, a_deg, rm);
        }
#pragma unroll
        for (int i = 0; i < 6; i++) actq[i] = fd.fast(scheme != 0 ? rp[12 + i] - rm[12 + i] : rp[12 + i] - f[i]);
        // a NaN command or lf1 is not a precondition of fast_ok: the reference-order pass decides what it means
        ok &= !mine | !(either_nan(u0[0], u0[1]) | either_nan(u0[2], u0[3]) | either_nan(x0[17], x0[17]));
      }
      const unsigned bad = __ballot_sync(0xffffffffu, !ok);
      const bool redo_me = (bad & (half ? 0xffff0000u : 0x0000ffffu)) != 0;
      if (lane == 0) redo[t] = ((bad & 0x0000ffffu) ? 1u : 0u) | ((bad & 0xffff0000u) ? 2u : 0u);
      any_redo |= bad;
      double c17[6];
#pragma unroll
      for (int i = 0; i < 6; i++) c17[i] = shfl_half(actq[i], 0);
      if (mine && !redo_me) {
        // lane 15 holds the unperturbed point: its own quotients are exact zeros (identical bits on both sides), which is what
        // rows 0..11 of column 17 are; rows 12..17 of that column are lane 0's actuator rows
#pragma unroll
        for (int i = 0; i < 6; i++) q[12 + i] = j == 15 ? c17[i] : q[12 + i];
        double* Ao = A_g + n * 324;
        double* Bo = B_g + n * 72;
#pragma unroll
        for (int r = 0; r < 18; r++) {
          Ao[r * 18 + 2 + j] = q[r];          // columns 2..17: 16 consecutive doubles
          if (j < 2) Ao[r * 18 + j] = 0.0;    // columns 0, 1: f reads neither npos nor epos
        }
#pragma unroll
        for (int k = 0; k < 3; k++) Bo[16 * k + j] = 0.0;  // rows 0..11 of B
        if (j >= 1 && j <= 4) {
#pragma unroll
          for (int i = 0; i < 6; i++) Bo[(12 + i) * 4 + (j - 1)] = actq[i];
        }
        if (status && j == 0) status[n] = 0;
      } else if (own < 0) {
        lin_store(A_g, B_g, status, n, j, q, actq, c17, 0.0, true, (int)ST_FIDELITY);
      }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if (!any_redo) return;
  __syncwarp();
  lin_redo_pass<FI>(tabs, sel, x_g, ld_x, u_g, ld_u, N, eps, scheme, A_g, B_g, status, redo, t0, stride, n_tasks, lane);
}

cudaError_t launch_linearise_fast(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* x, long long ld_x,
                                  const double* u, long long ld_u, long long N, double eps, int scheme, double* A, double* B,
                                  int* status, unsigned* redo) {
  if (N <= 0) return cudaSuccess;
  const long long n_tasks = (N + 1) / 2;
  cudaError_t e = cudaSuccess;
  const bool want1 = sel.fi != nullptr || sel.fi_default != 0, want0 = sel.fi != nullptr || sel.fi_default == 0;
  auto go = [&](auto kern, int threads, int smem) {
    return launch_persistent(cfg, kern, threads, smem, n_tasks, threads / 32, tabs, sel, x, ld_x, u, ld_u, N, eps, A, B, status, redo);
  };
  constexpr int TC = LF_THREADS_CENTRAL, TF = LF_THREADS_FORWARD;
  if (want1)
    e = scheme != 0 ? go(linearise_fast_kernel<1, TC, true>, TC, LfSmem<1, TC, true>::TOTAL)
                    : go(linearise_fast_kernel<1, TF, false>, TF, LfSmem<1, TF, false>::TOTAL);
  if (e == cudaSuccess && want0)
    e = scheme != 0 ? go(linearise_fast_kernel<0, TC, true>, TC, LfSmem<0, TC, true>::TOTAL)
                    : go(linearise_fast_kernel<0, TF, false>, TF, LfSmem<0, TF, false>::TOTAL);
  return e;
}

}  // namespace fast
}  // namespace f16

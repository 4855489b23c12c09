// f16_step_fast.cu -- the hifi fused Euler step of F16_MATH_FAST (f16_fast.cuh).
// Compiled with -fmad=false: every fused multiply-add in this kernel is an explicit fma() in the source, so the
// result does not depend on which mul/add pairs ptxas would have chosen to contract in a given instantiation
// (CTA size, table staging) -- all variants of the kernel, and the host emulation of the tests, agree bit for bit.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "f16_kernels_common.cuh"
#include "f16_fast.cuh"

namespace f16 {
namespace fast {

// The closed-loop law (make_dense_law) travels as a kernel parameter of the launch: constant bank like a __constant__ symbol,
// but nothing is uploaded, nothing is shared between launches, streams or devices, and no launch waits for an earlier one.

// ------------------------------------------------------------------------------------------------------
// step_batch, hifi, F16_MATH_FAST: the same K fused Euler steps on the re-associated arithmetic of f16_fast.cuh
// (fast table image: 157 KB in shared memory, one CTA per SM).  The per-step checks are the cheap "all inside"
// form; the exact status word is rebuilt from the frozen state when an aircraft stops.
// ------------------------------------------------------------------------------------------------------
constexpr int FAST_SMEM_BYTES = F16_FI_BYTES + 16;

static bool sel_wants(const BatchSel& s, int FI) { return s.fi != nullptr || s.fi_default == FI || (FI == 1 && s.fi_default != 0); }

template <bool SMEM, bool LQR, int THREADS, int COLMASK = 0>
__global__ void __launch_bounds__(THREADS, 1)
step_hifi_fast_kernel(DevTables tabs, BatchSel sel, double* __restrict__ x_g, long long ld_x,
                      const double* __restrict__ u_g, long long ld_u, long long N, int K, double dt,
                      int* __restrict__ status, int* __restrict__ steps_done, const __grid_constant__ fastmath::LqrDense c_lqr_fast) {
  const double* img = tabs.hifi_fast;
  if (SMEM) {
    stage_tables_tma<F16_FI_BYTES>(f16_smem, img, reinterpret_cast<unsigned long long*>(f16_smem + F16_FI_BYTES));
    img = reinterpret_cast<const double*>(f16_smem);
  }
#if defined(F16_FAST_LDS64)
  img += tabs.zero;  // always 0; keeps the table gathers 8-byte loads (see fastmath::fd)
#endif
  // The warps of a CTA leave the table staging together and run the same instruction stream: the three warps that share a
  // scheduler (warp, warp + 4, warp + 8) would sit in the FP64-dense and in the integer / gather parts of a step at the same
  // time.  Starting them a third of a microsecond apart keeps them out of phase: +2 % on a batch without a grid tail (2^20
  // aircraft less 2.4 %: 336.3 -> 329.9 ms; the time-chunked kernel gets the same effect from the jitter of its item
  // boundaries, which is why it was the faster one per aircraft-step even without counting the tail).
  if (threadIdx.x >> 7) __nanosleep((threadIdx.x >> 7) * 300);
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const int own = owns<1>(sel, n);
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
    int k;
    const unsigned st = fastmath::step_aircraft<LQR, 1, COLMASK>(img, x, u_in, LQR ? &c_lqr_fast : nullptr, xcg, dt, K, k);
#pragma unroll
    for (int i = 0; i < 18; i++) x_g[i * ld_x + n] = x[i];
    if (status) status[n] = (int)st;
    if (steps_done) steps_done[n] = k;
  }
}

// ------------------------------------------------------------------------------------------------------
// The same step, scheduled in TIME CHUNKS so that the grid has no tail.  With one warp-task = 32 aircraft x all K steps, 2^20
// aircraft are 18.45 rounds of the 148 x 12 warp slots: the 19th round runs 45 % full and 3 % of the launch is idle SMs
// (VERDICT r01 weak #7).  Here a work item is (chunk c of the K steps, group g of 32 aircraft), item c G + g goes to warp slot
// (c G + g) mod S, slots numbered warp-major over the grid: every slot gets the same number of items to within one, and an
// item is 1/C of a round, so what is left over at the end is 1/C of a round spread over all SMs.  The state of a group goes
// through global memory between its chunks (L2: see the item order in the kernel) -- 320 B per aircraft per chunk --
// and progress[g] counts the chunks of group g that are complete: the warp that takes (c, g) waits for progress[g] == c
// (release / acquire at gpu scope; in practice the predecessor finished a whole round of chunks earlier).  All CTAs of the
// persistent grid are resident (one per SM), items are taken in increasing order and depend only on smaller items: no wait
// can cycle.  step_batch is restartable bit for bit at any step boundary, so the result equals the unchunked kernel's.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

struct ChunkPlan {  // the blocks of groups of the item order (below), computed by the launcher
  long long blk_lo, blk_rem, big_items;
};
// item i -> (chunk c, group g), packed as c << 40 | g.  A function of its own (called once per item = every few hundred steps):
// the 64-bit divisions and their temporaries stay out of the register allocation of the step loop.
static __device__ __noinline__ long long chunk_item(long long i, long long blk_lo, long long blk_rem, long long big_items, int C) {
  long long b, r, bs, g0;
  if (i < big_items) {
    bs = blk_lo + 1;
    b = i / (bs * C);
    r = i - b * bs * C;
    g0 = b * bs;
  } else {
    bs = blk_lo;
    const long long i2 = i - big_items;
    b = i2 / (bs * C);
    r = i2 - b * bs * C;
    g0 = blk_rem * (blk_lo + 1) + b * bs;
  }
  const long long c = r / bs;
  return (c << 40) | (g0 + (r - c * bs));
}
template <bool LQR, int COLMASK>
__global__ void __launch_bounds__(384, 1)
step_hifi_fast_chunked_kernel(DevTables tabs, BatchSel sel, double* x_g, long long ld_x, const double* __restrict__ u_g, long long ld_u,
                              long long N, int K, int chunk, double dt, int* status, int* steps_done, int* progress,
                              const __grid_constant__ ChunkPlan plan, const __grid_constant__ fastmath::LqrDense c_lqr_fast) {
  stage_tables_tma<F16_FI_BYTES>(f16_smem, tabs.hifi_fast, reinterpret_cast<unsigned long long*>(f16_smem + F16_FI_BYTES));
  const double* img = reinterpret_cast<const double*>(f16_smem);
#if defined(F16_FAST_LDS64)
  img += tabs.zero;
#endif
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long G = (N + 31) >> 5;
  const int C = (K + chunk - 1) / chunk;
  const long long items = G * C, S = (long long)(blockDim.x >> 5) * gridDim.x;
  // Item order: the groups are cut into blocks of ~2 S groups (36 MB of state: it stays in L2), and inside a block the order is
  // chunk-major -- (block b, chunk c, group g of b).  The successor chunk of a group is then one block-row = two rounds of the
  // grid later, its state still in L2 (with ONE block = all groups, as the first version had it, the 340 MB of a 2^20-aircraft
  // batch went to DRAM and back for every chunk: 5.4 GB per launch, ncu).  Blocks are equal to within one group and never smaller
  // than 2 S (a single block when there are fewer groups than that), so a predecessor item is always >= two rounds older.
  // (the block sizes come from the host as kernel parameters -- constant bank --, so that nothing but i is live across the steps)
  for (long long i = (long long)warp * gridDim.x + blockIdx.x; i < items; i += S) {
    const long long cg = chunk_item(i, plan.blk_lo, plan.blk_rem, plan.big_items, C);
    const int c = (int)(cg >> 40);
    const long long g = cg & ((1LL << 40) - 1);
    const long long n = (g << 5) + lane;
    const int k0 = c * chunk, kc = (K - k0) < chunk ? (K - k0) : chunk;
    if (c > 0) {
      if (lane == 0)
        while (ld_acquire_gpu(progress + g) < c) __nanosleep(100);
      __syncwarp();
    }
    if (n < N) {
      // chunk c > 0 continues only an aircraft whose earlier chunks ran to their end (status 0); L1 is not coherent: .cg loads
      const int st_prev = c > 0 ? __ldcg(status + n) : 0;
      if (st_prev == 0) {
        double x[18], u_in[4];
#pragma unroll
        for (int j = 0; j < 18; j++) x[j] = __ldcg(x_g + j * ld_x + n);
#pragma unroll
        for (int j = 0; j < 4; j++) u_in[j] = u_g[j * ld_u + n];
        const double xcg = sel.xcg ? sel.xcg[n] : sel.xcg_default;
        int k;
        const unsigned st = fastmath::step_aircraft<LQR, 1, COLMASK>(img, x, u_in, LQR ? &c_lqr_fast : nullptr, xcg, dt, kc, k);
#pragma unroll
        for (int j = 0; j < 18; j++) x_g[j * ld_x + n] = x[j];
        status[n] = (int)st;
        if (steps_done) steps_done[n] = k0 + k;
      }
    }
    __threadfence();  // this lane's stores are visible at gpu scope before the flag moves
    __syncwarp();
    if (lane == 0) st_release_gpu(progress + g, c + 1);
  }
}

// ------------------------------------------------------------------------------------------------------
// step_batch, lofi, F16_MATH_FAST: the Stevens-Lewis model on the same arithmetic (fastmath::calc_xdot_lofi).  Its step
// image is 7 KB (lofi tables + the centre table of half_rho), copied into shared memory by the CTA itself.
// ------------------------------------------------------------------------------------------------------
template <bool LQR, int THREADS, int COLMASK = 0>
__global__ void __launch_bounds__(THREADS, 1)
step_lofi_fast_kernel(DevTables tabs, BatchSel sel, double* __restrict__ x_g, long long ld_x,
                      const double* __restrict__ u_g, long long ld_u, long long N, int K, double dt,
                      int* __restrict__ status, int* __restrict__ steps_done, const __grid_constant__ fastmath::LqrDense c_lqr_fast) {
  double* img = reinterpret_cast<double*>(f16_smem);
  for (int i = threadIdx.x; i < F16_LOFI_STEP_IMG_DOUBLES; i += THREADS)
    img[i] = i < F16_IMG_LOFI_DOUBLES ? tabs.lofi[i] : tabs.hifi_fast[F16_FI_POW + (i - F16_IMG_LOFI_DOUBLES)];
  __syncthreads();
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    if (owns<0>(sel, n) == 0) continue;  // fidelity flags other than 0 / 1 are reported by the hifi kernel
    double x[18], u_in[4];
#pragma unroll
    for (int i = 0; i < 18; i++) x[i] = x_g[i * ld_x + n];
#pragma unroll
    for (int i = 0; i < 4; i++) u_in[i] = u_g[i * ld_u + n];
    const double xcg = sel.xcg ? sel.xcg[n] : sel.xcg_default;
    int k;
    const unsigned st = fastmath::step_aircraft<LQR, 0, COLMASK>(img, x, u_in, LQR ? &c_lqr_fast : nullptr, xcg, dt, K, k);
#pragma unroll
    for (int i = 0; i < 18; i++) x_g[i * ld_x + n] = x[i];
    if (status) status[n] = (int)st;
    if (steps_done) steps_done[n] = k;
  }
}

// ------------------------------------------------------------------------------------------------------
// trim_batch, F16_MATH_FAST: the same Nelder-Mead search (f16_model.cuh::nelder_mead_trim_with) with the objective on the
// step kernel's arithmetic -- a third of the instructions per evaluation, and the search is ~2000 dependent evaluations
// per thread.  obj_func clips thrust, the three surfaces and alpha into their ranges (env.py:240-250) and leaves the
// flap state unclipped, so the precondition here is what calc_xdot_hifi / _lofi actually need (altitude inside the
// density table, no NaN), not the step bounds; a trial point outside it takes the reference-order objective on the
// standard image in global memory.
// ------------------------------------------------------------------------------------------------------
template <int FI>
static __device__ __noinline__ double trim_cost_reference_order(const double* img_std, double h, double V, double lef_q, double u0,
                                                                double u1, double u2, double u3, double u4, double xcg,
                                                                unsigned* st) {
  TrimPoint t;
  t.h = h;
  t.V = V;
  t.lef_q = lef_q;
  const double ux[5] = {u0, u1, u2, u3, u4};
  unsigned s = 0;
  const double c = trim_cost<FI>(img_std, t, ux, xcg, s);
  *st = s;
  return c;
}

template <int FI>
struct TrimCostFast {
  const double* img;      // the step image of this fidelity, in shared memory
  const double* img_std;  // the standard image, in global memory (rare path)
  __device__ __forceinline__ double operator()(const TrimPoint& t, const double (&ux)[5], double xcg, unsigned& st) const {
    double x[18], u[4], xd[18];
    trim_cost_inputs(t, ux, x, u);
    // trim_state: phi = psi = beta = p = q = r = 0, theta = alpha; what can be out of range is the caller's h and V
    const bool ok = (x[2] >= 0.0) & (x[2] <= 100000.0) & !either_nan(x[6], x[7]) & !either_nan(x[12], x[13]) &
                    !either_nan(x[14], x[15]) & !either_nan(x[16], x[17]);
    if (!ok) {
      unsigned s = 0;
      const double c = trim_cost_reference_order<FI>(img_std, t.h, t.V, t.lef_q, ux[0], ux[1], ux[2], ux[3], ux[4], xcg, &s);
      st = s;
      return c;
    }
    double uc[4];
    fastmath::clip_commands(u, uc);
    const bool inside = FI ? fastmath::calc_xdot_hifi<false>(img, x, uc, xcg, xd) : fastmath::calc_xdot_lofi<false>(img, x, uc, xcg, xd);
    if (!inside) {
      const double a = x[7] * (180.0 / 3.141592653589793), b = x[8] * (180.0 / 3.141592653589793);
      st = FI ? hifi_envelope(a, b, x[13]) : lofi_envelope(a, b, x[13]);
      return __builtin_huge_val();
    }
    st = 0;
    return trim_cost_sum(xd);
  }
};

struct TrimGuessFast {
  double ux[5];
  int fixed_point_exit;
};

template <int FI>
__global__ void __launch_bounds__(256, 1)
trim_fast_kernel(DevTables tabs, BatchSel sel, const double* __restrict__ h_g, const double* __restrict__ v_g, long long N,
                 double tol, int maxiter, TrimGuessFast guess, double* __restrict__ x_g, long long ld_x,
                 double* __restrict__ info_g, long long ld_info, int* __restrict__ status) {
  const double* img;
  if (FI) {
    stage_tables_tma<F16_FI_BYTES>(f16_smem, tabs.hifi_fast, reinterpret_cast<unsigned long long*>(f16_smem + F16_FI_BYTES));
    img = reinterpret_cast<const double*>(f16_smem);
#if defined(F16_FAST_LDS64)
    img += tabs.zero;
#endif
  } else {
    double* li = reinterpret_cast<double*>(f16_smem);
    for (int i = threadIdx.x; i < F16_LOFI_STEP_IMG_DOUBLES; i += blockDim.x)
      li[i] = i < F16_IMG_LOFI_DOUBLES ? tabs.lofi[i] : tabs.hifi_fast[F16_FI_POW + (i - F16_IMG_LOFI_DOUBLES)];
    __syncthreads();
    img = li;
  }
  const TrimCostFast<FI> cost{img, FI ? tabs.hifi : tabs.lofi};
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
      r = nelder_mead_trim_with(cost, t, sel.xcg ? sel.xcg[n] : sel.xcg_default, tol, maxiter, ux, guess.fixed_point_exit != 0);
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

cudaError_t launch_trim(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* h, const double* v, long long N,
                        double tol, int maxiter, const double* ux0, double* x_trim, long long ld_x, double* info, long long ld_info,
                        int* status) {
  if (N <= 0) return cudaSuccess;
  TrimGuessFast g;
  for (int k = 0; k < 5; k++) g.ux[k] = ux0[k];
  g.fixed_point_exit = cfg.trim_fixed_point_exit ? 1 : 0;
  cudaError_t e = cudaSuccess;
  if (sel_wants(sel, 1))
    e = launch_persistent(cfg, trim_fast_kernel<1>, 256, FAST_SMEM_BYTES, N, 256, tabs, sel, h, v, N, tol, maxiter, g, x_trim, ld_x,
                          info, ld_info, status);
  if (e == cudaSuccess && sel_wants(sel, 0))
    e = launch_persistent(cfg, trim_fast_kernel<0>, 256, F16_LOFI_STEP_IMG_DOUBLES * 8, N, 256, tabs, sel, h, v, N, tol, maxiter, g,
                          x_trim, ld_x, info, ld_info, status);
  return e;
}

// ------------------------------------------------------------------------------------------------------
// Nlplant_batch / calc_xdot_batch, F16_MATH_FAST: one evaluation per aircraft on the arithmetic of f16_fast.cuh.
//
// These launches move 284 / 324 B per aircraft for ~480 FP64 instructions: HBM-bound.  Layout of the work:
//   * a warp-task is 32 consecutive aircraft (one 256-byte run of every SoA plane); task t goes to warp slot
//     t mod (12 warps x grid), slots numbered warp-major (slot = warp * grid + cta), so a partial last round is spread
//     over all SMs instead of filling some CTAs and leaving the others idle;
//   * input: the SoA arrays are described to the TMA unit as 2-D tensors (planes x aircraft, CUtensorMap), and the 18 + 4
//     (17) plane runs of a task arrive as ONE box each (cp.async.bulk.tensor.2d, issued by one lane: 22 separate 256-byte
//     bulk copies cost 340 instructions per task in address arithmetic and uniform-register moves, a third of the kernel)
//     in the warp's own 5.5 KB shared buffer, completing on the warp's own mbarrier; a box that sticks out of the batch is
//     zero-filled by the hardware, so the ragged last task needs no special case.  The boxes of the warp's NEXT task are
//     requested as soon as the current values are in registers, so they fly during the arithmetic and the stores of the
//     current one; the first task's boxes are requested before the CTA waits for its table image;
//   * tables: the (f, d) image in shared memory (157 KB hifi / 7 KB lofi), one CTA of 384 threads per SM;
//   * output: 18 coalesced 8-byte stores per lane straight from registers (a shared output tile does not fit beside the
//     image).
// An aircraft outside the preconditions of the fast arithmetic (a NaN anywhere, altitude outside the density table, an angle
// beyond 2^30 rad, alpha / beta / elevator outside the tables) takes the reference-order evaluation on the standard image in
// global memory, which also produces the exact status word.  Pointers that are not 16-byte aligned or an odd plane stride
// (a tensor map needs 16-byte strides) fall back to plain loads.
// ------------------------------------------------------------------------------------------------------

#ifndef XF_TABLE_CHUNK
#define XF_TABLE_CHUNK 8192
#endif
template <int FI, bool NLP, int THREADS>
struct XfSmem {
  static constexpr int XF_WARPS = THREADS / 32;
  static constexpr int NPL = NLP ? 17 : 22;
  static constexpr int IMG_BYTES = FI ? F16_FI_BYTES : F16_LOFI_STEP_IMG_DOUBLES * 8;
  static constexpr int IMG_PAD = (IMG_BYTES + 127) / 128 * 128;
  static constexpr int BUF_DOUBLES = NPL * 32;
  static constexpr int BARS = IMG_PAD + XF_WARPS * BUF_DOUBLES * 8;
  static constexpr int TOTAL = BARS + (1 + XF_WARPS) * 8;
};

__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, int bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, int bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}

__device__ __forceinline__ void tma_box_g2s(uint32_t dst, const CUtensorMap* map, int col, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(map), "r"(col), "r"(0), "r"(bar)
               : "memory");
}

// rare path: the reference-order evaluation (f16_model.cuh) on the standard image in global memory
template <int FI, bool NLP>
static __device__ __noinline__ unsigned xdot_reference_order(const double* img_std, const double* x_, const double* u_, double xcg,
                                                             double* xd_) {
  double xd[18];
  unsigned st;
  if (NLP) {
    double xu[17];
#pragma unroll
    for (int i = 0; i < 17; i++) xu[i] = x_[i];
    st = nlplant_eval<FI>(img_std, xu, xcg, xd);
  } else {
    double x[18], u[4];
#pragma unroll
    for (int i = 0; i < 18; i++) x[i] = x_[i];
#pragma unroll
    for (int i = 0; i < 4; i++) u[i] = u_[i];
    st = calc_xdot<FI>(img_std, x, u, xcg, xd);
  }
#pragma unroll
  for (int i = 0; i < 18; i++) xd_[i] = xd[i];
  return st;
}

// The marked aircraft of a warp's tasks: reference-order evaluation on the standard image in global memory (also the exact
// status word).  A function of its own, called once after the main loop, so that its registers, its call and its local
// arrays do not take part in the register allocation of that loop.
template <int FI, bool NLP>
static __device__ __noinline__ void xdot_redo_pass(DevTables tabs, BatchSel sel, const double* __restrict__ x_g, long long ld_x,
                                                   const double* __restrict__ u_g, long long ld_u, double* __restrict__ xd_g,
                                                   long long ld_out, int* __restrict__ status, const unsigned* redo, long long t,
                                                   long long stride, long long tiles, int lane) {
  constexpr int NX = NLP ? 17 : 18;
#pragma unroll 1
  for (; t < tiles; t += stride) {
    const unsigned later = redo[t];
    if (!((later >> lane) & 1u)) continue;
    const long long n = (t << 5) + lane;
    double xs[18], us[4], xo[18];
#pragma unroll
    for (int i = 0; i < NX; i++) xs[i] = x_g[i * ld_x + n];
    if (NLP) xs[17] = 0.0;
#pragma unroll
    for (int i = 0; i < 4; i++) us[i] = NLP ? 0.0 : u_g[i * ld_u + n];
    const unsigned st = xdot_reference_order<FI, NLP>(FI ? tabs.hifi : tabs.lofi, xs, us, sel.xcg ? sel.xcg[n] : sel.xcg_default, xo);
#pragma unroll
    for (int i = 0; i < 18; i++) xd_g[i * ld_out + n] = st ? qnan() : xo[i];
    if (status) status[n] = (int)st;
  }
}

template <int FI, bool NLP, int THREADS>
__global__ void __maxnreg__(65536 / THREADS / 8 * 8 > 255 ? 255 : 65536 / THREADS / 8 * 8)
xdot_fast_kernel(DevTables tabs, BatchSel sel, const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_u,
                 const double* __restrict__ x_g, long long ld_x, const double* __restrict__ u_g, long long ld_u,
                 double* __restrict__ xd_g, long long ld_out, long long N, int* __restrict__ status, int bulk_ok,
                 unsigned* __restrict__ redo) {
  using S = XfSmem<FI, NLP, THREADS>;
  constexpr int NX = NLP ? 17 : 18, NU = NLP ? 0 : 4, XF_WARPS = THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double* img = reinterpret_cast<const double*>(f16_smem);
  double* buf = reinterpret_cast<double*>(f16_smem + S::IMG_PAD) + warp * S::BUF_DOUBLES;
  const uint32_t bar_tab = smem_u32(f16_smem + S::BARS), bar_w = bar_tab + 8 * (1 + warp), buf_a = smem_u32(buf);
  if (threadIdx.x == 0) {
    for (int i = 0; i <= XF_WARPS; i++) mbar_init(bar_tab + 8 * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // table image: global -> shared, completes on bar_tab
    mbar_expect_tx(bar_tab, S::IMG_BYTES);
    if (FI) {
      // every CTA of the grid reads the same 157 KB at the same moment: each starts at a different chunk, so that at any time
      // the requests of the 148 SMs are spread over the L2 slices instead of queueing at the few that hold "the current" chunk
      constexpr int CHUNK = XF_TABLE_CHUNK, NCHUNK = (S::IMG_BYTES + CHUNK - 1) / CHUNK;
      int c = (int)(blockIdx.x % NCHUNK);
#pragma unroll 1
      for (int k = 0; k < NCHUNK; k++) {
        const int off = c * CHUNK;
        bulk_g2s(smem_u32(f16_smem + off), reinterpret_cast<const char*>(tabs.hifi_fast) + off,
                 (S::IMG_BYTES - off) < CHUNK ? (S::IMG_BYTES - off) : CHUNK, bar_tab);
        c = c + 1 == NCHUNK ? 0 : c + 1;
      }
    } else {  // lofi step image = the lofi tables + the centre table of half_rho
      bulk_g2s(smem_u32(f16_smem), tabs.lofi, F16_IMG_LOFI_BYTES, bar_tab);
      bulk_g2s(smem_u32(f16_smem + F16_IMG_LOFI_BYTES), tabs.hifi_fast + F16_FI_POW, 2 * F16_FI_NPOW * 8, bar_tab);
    }
  }
  const long long tiles = (N + 31) >> 5;
  const long long stride = (long long)XF_WARPS * gridDim.x;
  long long t = (long long)warp * gridDim.x + blockIdx.x;

  auto issue = [&](long long tile) {  // the whole warp, converged
    if (!bulk_ok || tile >= tiles) return;
    if (lane == 0) {
      const int col = (int)(tile << 5);  // tensor coordinates are 32-bit: launch_xdot_fast keeps N below 2^31 on this path
      mbar_expect_tx(bar_w, S::NPL * 256);
      tma_box_g2s(buf_a, &map_x, col, bar_w);
      if (NU) tma_box_g2s(buf_a + NX * 256, &map_u, col, bar_w);
    }
  };
  issue(t);
  mbar_wait(bar_tab, 0);
  uint32_t phase = 0;
  unsigned any_later = 0;
  for (; t < tiles; t += stride) {
    const long long n = (t << 5) + lane;
    const bool staged = bulk_ok != 0;
    double x[18], u[4];
    if (staged) {
      mbar_wait(bar_w, phase);
      phase ^= 1;
#pragma unroll
      for (int i = 0; i < NX; i++) x[i] = buf[i * 32 + lane];
#pragma unroll
      for (int i = 0; i < NU; i++) u[i] = buf[(NX + i) * 32 + lane];
      __syncwarp();
      // the reads above (generic proxy) are ordered before the next task's bulk copies (async proxy) into the same buffer
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    } else {
      const long long m = n < N ? n : N - 1;
#pragma unroll
      for (int i = 0; i < NX; i++) x[i] = x_g[i * ld_x + m];
#pragma unroll
      for (int i = 0; i < NU; i++) u[i] = u_g[i * ld_u + m];
    }
    if (NLP) x[17] = 0.0;
    issue(t + stride);
    // A lane that cannot take the fast arithmetic is only MARKED here (one 4-byte word per task) and evaluated after the loop:
    // the reference-order function is a call, and a call inside this loop makes every value that is live across it a spill
    // (measured: 17 local loads per task; 255 registers instead of 168 to get rid of them).
    const int own = n < N ? owns<FI>(sel, n) : 0;
    bool ok = false;
    if (own == 1) {
      const double xcg = sel.xcg ? sel.xcg[n] : sel.xcg_default;
      ok = fastmath::fast_ok<FI>(x);
      double uc[4] = {0.0, 0.0, 0.0, 0.0};
      if (!NLP) {
        ok &= !either_nan(u[0], u[1]) & !either_nan(u[2], u[3]) & !either_nan(x[17], x[17]);
        fastmath::clip_commands(u, uc);
      }
      if (ok) {
        double xd[18];
        ok = FI ? fastmath::calc_xdot_hifi<false, NLP>(img, x, uc, xcg, xd) : fastmath::calc_xdot_lofi<false, NLP>(img, x, uc, xcg, xd);
        if (ok) {
#pragma unroll
          for (int i = 0; i < 18; i++) xd_g[i * ld_out + n] = xd[i];
          if (status) status[n] = 0;
        }
      }
    } else if (own < 0) {  // a fidelity flag that is neither 0 nor 1: reported by the hifi launch
#pragma unroll
      for (int i = 0; i < 18; i++) xd_g[i * ld_out + n] = qnan();
      if (status) status[n] = (int)ST_FIDELITY;
    }
    const unsigned later = __ballot_sync(0xffffffffu, own == 1 && !ok);
    if (lane == 0) redo[t] = later;  // always (4 bytes per task): the pass below reads only words of this launch
    any_later |= later;
  }
  if (!any_later) return;  // warp-uniform, and the common case
  __syncwarp();            // lane 0's redo[] stores are visible to the other lanes of its warp
  xdot_redo_pass<FI, NLP>(tabs, sel, x_g, ld_x, u_g, ld_u, xd_g, ld_out, status, redo, (long long)warp * gridDim.x + blockIdx.x, stride,
                          tiles, lane);
}

// ------------------------------------------------------------------------------------------------------
// step_batch with FEW steps per call (K < 8: the reference's own driving pattern, one env.step per controller update).  Such a
// launch is HBM-bound like the one-shot kernels -- 324 B per aircraft and call against K x 690 instructions --, so it gets
// their memory side: warp-tasks of 32 aircraft in warp-major order, the 18 + 4 input plane runs of a task as two TMA tensor
// boxes, the boxes of the warp's next task in flight during the arithmetic and the stores of the current one.  The arithmetic
// is step_aircraft() itself (bounds, envelope, exact status word, libm fall-back for huge Euler angles), so the results are
// the bits of step_hifi_fast_kernel.  Measured at 2^20 aircraft, K = 1: 77 -> 66 us.
// ------------------------------------------------------------------------------------------------------
template <int FI, bool LQR, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
step_tiled_fast_kernel(DevTables tabs, BatchSel sel, const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_u,
                       double* __restrict__ x_g, long long ld_x, long long N, int K, double dt, int* __restrict__ status,
                       int* __restrict__ steps_done, const __grid_constant__ fastmath::LqrDense c_lqr_fast) {
  using S = XfSmem<FI, false, THREADS>;
  constexpr int XF_WARPS = THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double* img = reinterpret_cast<const double*>(f16_smem);
  double* buf = reinterpret_cast<double*>(f16_smem + S::IMG_PAD) + warp * S::BUF_DOUBLES;
  const uint32_t bar_tab = smem_u32(f16_smem + S::BARS), bar_w = bar_tab + 8 * (1 + warp), buf_a = smem_u32(buf);
  if (threadIdx.x == 0) {
    for (int i = 0; i <= XF_WARPS; i++) mbar_init(bar_tab + 8 * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // table image: global -> shared, completes on bar_tab (chunks in a per-CTA rotation, as in xdot_fast_kernel)
    mbar_expect_tx(bar_tab, S::IMG_BYTES);
    if (FI) {
      constexpr int CHUNK = XF_TABLE_CHUNK, NCHUNK = (S::IMG_BYTES + CHUNK - 1) / CHUNK;
      int c = (int)(blockIdx.x % NCHUNK);
#pragma unroll 1
      for (int k = 0; k < NCHUNK; k++) {
        const int off = c * CHUNK;
        bulk_g2s(smem_u32(f16_smem + off), reinterpret_cast<const char*>(tabs.hifi_fast) + off,
                 (S::IMG_BYTES - off) < CHUNK ? (S::IMG_BYTES - off) : CHUNK, bar_tab);
        c = c + 1 == NCHUNK ? 0 : c + 1;
      }
    } else {
      bulk_g2s(smem_u32(f16_smem), tabs.lofi, F16_IMG_LOFI_BYTES, bar_tab);
      bulk_g2s(smem_u32(f16_smem + F16_IMG_LOFI_BYTES), tabs.hifi_fast + F16_FI_POW, 2 * F16_FI_NPOW * 8, bar_tab);
    }
  }
  const long long tiles = (N + 31) >> 5;
  const long long stride = (long long)XF_WARPS * gridDim.x;
  long long t = (long long)warp * gridDim.x + blockIdx.x;
  auto issue = [&](long long tile) {  // the whole warp, converged
    if (tile >= tiles) return;
    if (lane == 0) {
      const int col = (int)(tile << 5);
      mbar_expect_tx(bar_w, 22 * 256);
      tma_box_g2s(buf_a, &map_x, col, bar_w);
      tma_box_g2s(buf_a + 18 * 256, &map_u, col, bar_w);
    }
  };
  issue(t);
  mbar_wait(bar_tab, 0);
  uint32_t phase = 0;
  for (; t < tiles; t += stride) {
    const long long n = (t << 5) + lane;
    double x[18], u_in[4];
    mbar_wait(bar_w, phase);
    phase ^= 1;
#pragma unroll
    for (int i = 0; i < 18; i++) x[i] = buf[i * 32 + lane];
#pragma unroll
    for (int i = 0; i < 4; i++) u_in[i] = buf[(18 + i) * 32 + lane];
    __syncwarp();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the reads above before the next task's bulk copies
    issue(t + stride);
    const int own = n < N ? owns<FI>(sel, n) : 0;
    if (own == 1) {
      const double xcg = sel.xcg ? sel.xcg[n] : sel.xcg_default;
      int k;
      const unsigned st = fastmath::step_aircraft<LQR, FI, 0>(img, x, u_in, LQR ? &c_lqr_fast : nullptr, xcg, dt, K, k);
#pragma unroll
      for (int i = 0; i < 18; i++) x_g[i * ld_x + n] = x[i];
      if (status) status[n] = (int)st;
      if (steps_done) steps_done[n] = k;
    } else if (own < 0) {  // a fidelity flag that is neither 0 nor 1: reported by the hifi launch
      if (status) status[n] = (int)ST_FIDELITY;
      if (steps_done) steps_done[n] = 0;
    }
  }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point query (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static const EncodeTiledFn fn = [] {  // initialised once, thread-safe (the multi-device entry points launch from several threads)
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<EncodeTiledFn>(p);
    cudaGetLastError();
    return (EncodeTiledFn) nullptr;
  }();
  return fn;
}

// SoA array [planes][ld] of doubles, N valid columns, as a 2-D tensor with boxes of `planes` x 32 aircraft
static bool soa_tensor_map(CUtensorMap* m, const double* base, long long ld, long long N, int planes) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || (reinterpret_cast<uintptr_t>(base) & 15) || (ld & 1) || N >= (1LL << 31) || N < 1) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)planes};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
  const cuuint32_t box[2] = {32, (cuuint32_t)planes};
  const cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int FI, bool NLP>
static cudaError_t launch_xdot_fast_one(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* x,
                                        long long ld_x, const double* u, long long ld_u, double* xd, long long ld_out, long long N,
                                        int* status, unsigned* redo) {
  CUtensorMap mx, mu;
  memset(&mx, 0, sizeof mx);
  memset(&mu, 0, sizeof mu);
  bool tma = soa_tensor_map(&mx, x, ld_x, N, NLP ? 17 : 18);
  if (tma && !NLP) tma = soa_tensor_map(&mu, u, ld_u, N, 4);
  // CTA size: what keeps the main loop free of spills (measured at 2^20 aircraft, hifi): Nlplant 384 threads / 168 registers
  // 61 us, calc_xdot (22 input values instead of 17) 256 threads / 255 registers 68 us against 76 us at 384.  F16_XF_THREADS
  // overrides for experiments.
  static const int forced = getenv("F16_XF_THREADS") ? atoi(getenv("F16_XF_THREADS")) : 0;
  const int threads = forced ? forced : (NLP ? 384 : 256);
  if (threads == 256)
    return launch_persistent(cfg, xdot_fast_kernel<FI, NLP, 256>, 256, XfSmem<FI, NLP, 256>::TOTAL, N, 256, tabs, sel, mx, mu, x, ld_x, u,
                             ld_u, xd, ld_out, N, status, tma ? 1 : 0, redo);
  return launch_persistent(cfg, xdot_fast_kernel<FI, NLP, 384>, 384, XfSmem<FI, NLP, 384>::TOTAL, N, 384, tabs, sel, mx, mu, x, ld_x, u,
                           ld_u, xd, ld_out, N, status, tma ? 1 : 0, redo);
}

// u == nullptr: Nlplant_batch (x is xu [17][N]); else calc_xdot_batch
// redo: device scratch of one unsigned per 32 aircraft (which lanes of a task take the reference-order path)
cudaError_t launch_xdot_fast(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, const double* x, long long ld_x,
                             const double* u, long long ld_u, double* xd, long long ld_out, long long N, int* status, unsigned* redo) {
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaSuccess;
  if (sel_wants(sel, 1))
    e = u ? launch_xdot_fast_one<1, false>(cfg, tabs, sel, x, ld_x, u, ld_u, xd, ld_out, N, status, redo)
          : launch_xdot_fast_one<1, true>(cfg, tabs, sel, x, ld_x, nullptr, 0, xd, ld_out, N, status, redo);
  if (e == cudaSuccess && sel_wants(sel, 0))
    e = u ? launch_xdot_fast_one<0, false>(cfg, tabs, sel, x, ld_x, u, ld_u, xd, ld_out, N, status, redo)
          : launch_xdot_fast_one<0, true>(cfg, tabs, sel, x, ld_x, nullptr, 0, xd, ld_out, N, status, redo);
  return e;
}

// ------------------------------------------------------------------------------------------------------
// f16_fast_probe: the fast image and its cell search as the step kernel uses them (fastmath::probe_hifi), one query per
// thread, image read from global memory.  coef [44][N], cells [4][N], lam [4][N]; a query outside the hifi tables gets
// NaN / -1 and the status word of hifi_envelope().
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
fast_probe_kernel(DevTables tabs, const double* __restrict__ alpha, const double* __restrict__ beta,
                  const double* __restrict__ el, long long N, double* __restrict__ coef, int* __restrict__ cells,
                  double* __restrict__ lam, int* __restrict__ status) {
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    const double a = alpha[n], b = beta[n], e = el[n];
    const unsigned st = hifi_envelope(a, b, e);
    double o[44], l[4];
    int c[4];
    if (st) {
      for (int i = 0; i < 44; i++) o[i] = qnan();
      for (int i = 0; i < 4; i++) { c[i] = -1; l[i] = qnan(); }
    } else {
      fastmath::probe_hifi(tabs.hifi_fast, a, b, e, o, c, l);
    }
    for (int i = 0; i < 44; i++) coef[i * N + n] = o[i];
    for (int i = 0; i < 4; i++) { cells[i * N + n] = c[i]; lam[i * N + n] = l[i]; }
    if (status) status[n] = (int)st;
  }
}

cudaError_t launch_fast_probe(const LaunchCfg& cfg, const DevTables& tabs, const double* alpha, const double* beta,
                              const double* el, long long N, double* coef, int* cells, double* lam, int* status) {
  if (N <= 0) return cudaSuccess;
  long long g = (N + 255) / 256;
  if (g > cfg.sm_count * 8) g = cfg.sm_count * 8;
  fast_probe_kernel<<<(unsigned)g, 256, 0, cfg.stream>>>(tabs, alpha, beta, el, N, coef, cells, lam, status);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

// the short-step launch: true when it was taken (K < 8, a batch worth staging tables for, arrays a tensor map can describe)
template <int FI>
static bool launch_step_tiled(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, double* x, long long ld_x, const double* u,
                              long long ld_u, long long N, int K, double dt, const LqrLaw* lqr_host, const fastmath::LqrDense& dense,
                              int* status, int* steps_done, cudaError_t* err) {
  static const bool off = getenv("F16_STEP_TILED") && atoi(getenv("F16_STEP_TILED")) == 0;
  if (off || !cfg.smem_tables || K < 1 || K >= 8 || N < 4096) return false;
  CUtensorMap mx, mu;
  memset(&mx, 0, sizeof mx);
  memset(&mu, 0, sizeof mu);
  if (!soa_tensor_map(&mx, x, ld_x, N, 18) || !soa_tensor_map(&mu, u, ld_u, N, 4)) return false;
  constexpr int T = 256;
  *err = lqr_host ? launch_persistent(cfg, step_tiled_fast_kernel<FI, true, T>, T, XfSmem<FI, false, T>::TOTAL, N, T, tabs, sel, mx, mu, x,
                                      ld_x, N, K, dt, status, steps_done, dense)
                  : launch_persistent(cfg, step_tiled_fast_kernel<FI, false, T>, T, XfSmem<FI, false, T>::TOTAL, N, T, tabs, sel, mx, mu, x,
                                      ld_x, N, K, dt, status, steps_done, dense);
  return true;
}

using StepKern = void (*)(DevTables, BatchSel, double*, long long, const double*, long long, long long, int, double, int*,
                          int*, const fastmath::LqrDense);

template <bool LQR>
static StepKern pick_step_hifi_fast(bool smem_tables, int& threads) {
  if (!smem_tables) { threads = 256; return step_hifi_fast_kernel<false, LQR, 256>; }
  if (threads <= 256) { threads = 256; return step_hifi_fast_kernel<true, LQR, 256>; }
  if (threads <= 384) { threads = 384; return step_hifi_fast_kernel<true, LQR, 384>; }
  if (threads <= 512) { threads = 512; return step_hifi_fast_kernel<true, LQR, 512>; }
  if (threads <= 640) { threads = 640; return step_hifi_fast_kernel<true, LQR, 640>; }
  threads = 768;
  return step_hifi_fast_kernel<true, LQR, 768>;
}

static cudaError_t launch_step_hifi_fast(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, double* x, long long ld_x,
                                         const double* u, long long ld_u, long long N, int K, double dt, const LqrLaw* lqr_host,
                                         int* status, int* steps_done) {
  if (N <= 0) return cudaSuccess;
  fastmath::LqrDense dense = fastmath::LqrDense();
  if (lqr_host) fastmath::make_dense_law(*lqr_host, dense);
  const bool mpc_cols = lqr_host && dense.colmask == F16_LQR_MPC_COLMASK && dense.row_mask == 0xE;  // the reference's own law: compile-time shape
  cudaError_t te = cudaSuccess;
  if (launch_step_tiled<1>(cfg, tabs, sel, x, ld_x, u, ld_u, N, K, dt, lqr_host, dense, status, steps_done, &te)) return te;
  int threads = cfg.step_threads;
  // time-chunked scheduling (no grid tail): the default CTA size, a uniform hifi batch, enough steps to cut into chunks and
  // more than one round of warp-tasks; needs the status words (they carry "stopped" between chunks) and the progress flags
  // ... and a tail worth removing: with R = groups / (12 warps x SMs) rounds of warp-tasks the plain kernel idles
  // (ceil(R) - R) / ceil(R) of the launch (2.9 % at 2^20 aircraft, 0.3 % at 2^23, where the plain kernel is the faster one:
  // measured 2.68e10 against 2.60e10 aircraft-steps/s closed loop)
  const long long groups = (N + 31) / 32, slots = 12LL * cfg.sm_count, full = (groups + slots - 1) / slots;
  const bool tail = (full * slots - groups) * 100 > full * slots;  // more than 1 % idle
  if (cfg.step_chunking && cfg.smem_tables && threads > 256 && threads <= 384 && sel.fi == nullptr && K >= 512 && status &&
      cfg.step_progress && groups <= cfg.step_progress_cap && groups > slots && tail) {
    const int chunk = (K + 15) / 16 < 64 ? 64 : (K + 15) / 16;
    cudaError_t e = cudaMemsetAsync(cfg.step_progress, 0, (size_t)groups * 4, cfg.stream);
    if (e != cudaSuccess) return e;
    using ChunkKern = void (*)(DevTables, BatchSel, double*, long long, const double*, long long, long long, int, int, double, int*, int*,
                               int*, const ChunkPlan, const fastmath::LqrDense);
    // item order of the kernel: blocks of >= 2 x (12 warps x grid) groups, equal to within one group.  The grid is the persistent
    // one (one CTA per SM: the launch below asks for exactly that)
    const int C = (K + chunk - 1) / chunk;
    const long long S = slots, n_blk = groups / (2 * S) > 0 ? groups / (2 * S) : 1;
    ChunkPlan plan;
    plan.blk_lo = groups / n_blk;
    plan.blk_rem = groups - plan.blk_lo * n_blk;
    plan.big_items = (plan.blk_lo + 1) * C * plan.blk_rem;
    ChunkKern ck = !lqr_host ? step_hifi_fast_chunked_kernel<false, 0>
                   : mpc_cols ? step_hifi_fast_chunked_kernel<true, F16_LQR_MPC_SHAPE>
                              : step_hifi_fast_chunked_kernel<true, 0>;
    return launch_persistent(cfg, ck, 384, FAST_SMEM_BYTES, N, 384, tabs, sel, x, ld_x, u, ld_u, N, K, chunk, dt, status, steps_done,
                             cfg.step_progress, plan, dense);
  }
  StepKern k = lqr_host ? pick_step_hifi_fast<true>(cfg.smem_tables, threads) : pick_step_hifi_fast<false>(cfg.smem_tables, threads);
  if (mpc_cols && cfg.smem_tables && threads == 384) k = step_hifi_fast_kernel<true, true, 384, F16_LQR_MPC_SHAPE>;
  const int smem = cfg.smem_tables ? FAST_SMEM_BYTES : 0;
  return launch_persistent(cfg, k, threads, smem, N, threads, tabs, sel, x, ld_x, u, ld_u, N, K, dt, status, steps_done, dense);
}

static cudaError_t launch_step_lofi_fast(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, double* x, long long ld_x,
                                         const double* u, long long ld_u, long long N, int K, double dt, const LqrLaw* lqr_host,
                                         int* status, int* steps_done) {
  if (N <= 0) return cudaSuccess;
  fastmath::LqrDense dense = fastmath::LqrDense();
  if (lqr_host) fastmath::make_dense_law(*lqr_host, dense);
  cudaError_t te = cudaSuccess;
  if (launch_step_tiled<0>(cfg, tabs, sel, x, ld_x, u, ld_u, N, K, dt, lqr_host, dense, status, steps_done, &te)) return te;
  const int smem = F16_LOFI_STEP_IMG_DOUBLES * 8;
  StepKern k = !lqr_host ? step_lofi_fast_kernel<false, 384>
               : (dense.colmask == F16_LQR_MPC_COLMASK && dense.row_mask == 0xE) ? step_lofi_fast_kernel<true, 384, F16_LQR_MPC_SHAPE>
                                                      : step_lofi_fast_kernel<true, 384>;
  return launch_persistent(cfg, k, 384, smem, N, 384, tabs, sel, x, ld_x, u, ld_u, N, K, dt, status, steps_done, dense);
}

cudaError_t launch_step(const LaunchCfg& cfg, const DevTables& tabs, const BatchSel& sel, double* x, long long ld_x, const double* u,
                        long long ld_u, long long N, int K, double dt, const LqrLaw* lqr_host, int* status, int* steps_done) {
  cudaError_t e = cudaSuccess;
  if (sel_wants(sel, 1)) e = launch_step_hifi_fast(cfg, tabs, sel, x, ld_x, u, ld_u, N, K, dt, lqr_host, status, steps_done);
  if (e == cudaSuccess && sel_wants(sel, 0))
    e = launch_step_lofi_fast(cfg, tabs, sel, x, ld_x, u, ld_u, N, K, dt, lqr_host, status, steps_done);
  return e;
}

}  // namespace fast
}  // namespace f16

// f16_stats.cu -- the summary a Monte-Carlo run ends with, reduced on the device (SURVEY.md 8e / 8f rank 4): over the
// aircraft whose status word is 0 ("alive": the reference would not have exit()ed, env.py:117-124), per state
// min, max, mean and M2 = sum (x - mean)^2, plus the two counts.  One row of 74 doubles
//     [n, alive, min[18], max[18], mean[18], M2[18]]
// is what a rank contributes to the only collective of a run (an all-gather of these rows, shard.py::merge_summaries).
//
// HBM-bound, ONE pass: every plane of the SoA state is read once and the status words three times (once per group of six
// states), 152 B per aircraft, fully coalesced (thread n reads x[i][n]).  Mean and M2 come out of the same pass by the
// textbook shifted-data form: with a shift c_i taken from INSIDE the data -- state i of the first surviving aircraft of the
// batch (aircraft 0 when there is no status array) -- the kernel accumulates S1 = sum (v - c) and S2 = sum (v - c)^2, which
// add up exactly like plain sums over threads, warps and CTAs, and the finishing CTA forms mean = c + S1 / n,
// M2 = S2 - S1^2 / n.  The subtraction v - c is exact for values within a factor of two of c, and the final difference loses
// (|mean - c| / sigma)^2 ulps: nothing for a shift inside the cloud, 1e-10 relative only when the first survivor sits a
// thousand standard deviations out.  The shift must be a survivor: a dead aircraft's state is frozen wherever it left the
// envelope (a crash below h = 0, a NaN), arbitrarily far from the survivors, and a shift of 0 against h = 1e4 +- 1e-3 ft
// costs 6e-3 of M2.  So when a status array is given, first_alive_kernel finds that aircraft first (a 64-bit atomicMin;
// warps stop scanning above a survivor already found, so a batch whose first survivor is aircraft j reads about
// j + 128 x (warps in the grid) status words).  (Combining per-thread MEANS by Chan's update is first-order in the rounding
// of those means and misses 1e-10 on a plane like h = 10000 +- 0.001 ft; two passes -- sums, then squared deviations about
// the mean, the round-1 kernel -- cost twice the bytes: 0.119 ms at 2^20 aircraft.)  Reductions are a fixed tree (per
// thread -> warp shuffles -> shared memory -> one partial per CTA -> one finishing CTA, lane-strided), so the result is
// bit-reproducible for a given device and batch size; the one atomic picks a minimum, which does not depend on the order.
#include <math.h>
#include <stdint.h>

#include "f16_kernels.cuh"

namespace f16 {
namespace stats {

constexpr int THREADS = 256;
constexpr int NS = 18;
constexpr int PARTIAL_STRIDE = 80;  // doubles of scratch per CTA column of the reduction (73 used)

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// partial[b] of CTA column b (stride PARTIAL_STRIDE): S1[18] | S2[18] | min[18] | max[18] | alive count
// blockIdx.y picks NS / NG of the eighteen states (six: 24 accumulators + 6 shifts per thread); the loads in flight, not the
// arithmetic, set the pace.

// the shift aircraft: the first survivor (*first, from first_alive_kernel), aircraft 0 without a status array, -1 when no
// aircraft survives
__device__ __forceinline__ long long shift_aircraft(const int* status, long long N, const unsigned long long* first) {
  if (N <= 0) return -1;  // launch_summary neither clears nor searches for an empty batch: *first is not read
  if (!status) return 0;
  const unsigned long long f = *first;
  return f < (unsigned long long)N ? (long long)f : -1;
}

// *first = the lowest n with status[n] == 0 (left at its initial ULLONG_MAX when there is none).  Warp w scans status words
// [128 w, 128 w + 128), then the same span one grid of warps further on, and stops at a span that starts above a survivor
// some warp has already found.
constexpr int SPAN = 128;
__global__ void __launch_bounds__(THREADS)
first_alive_kernel(const int* __restrict__ status, long long N, unsigned long long* first) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (THREADS / 32);
  for (long long base = ((long long)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5)) * SPAN; base < N; base += warps * SPAN) {
    unsigned long long known = lane == 0 ? *(volatile const unsigned long long*)first : 0;
    known = __shfl_sync(0xffffffffu, known, 0);
    if ((unsigned long long)base >= known) return;
    int st[SPAN / 32];
#pragma unroll
    for (int k = 0; k < SPAN / 32; k++) {
      const long long n = base + k * 32 + lane;
      st[k] = n < N ? status[n] : 1;
    }
#pragma unroll
    for (int k = 0; k < SPAN / 32; k++) {
      const unsigned m = __ballot_sync(0xffffffffu, st[k] == 0);
      if (m) {
        if (lane == 0) atomicMin(first, (unsigned long long)(base + k * 32 + __ffs(m) - 1));
        return;
      }
    }
  }
}

template <int NG, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
partial_kernel(const double* __restrict__ x, long long ld, long long N, const int* __restrict__ status,
               const unsigned long long* __restrict__ first, double* __restrict__ partial) {
  constexpr int NH = NS / NG;
  __shared__ double red[THREADS / 32][4 * NH + 1];
  const int s0 = blockIdx.y * NH;  // first state of this group
  x += (long long)s0 * ld;
  const long long j0 = shift_aircraft(status, N, first);
  double c[NH], s1[NH], s2[NH], mn[NH], mx[NH];
  double cnt = 0.0;
#pragma unroll
  for (int i = 0; i < NH; i++) {
    const double v0 = j0 >= 0 ? x[i * ld + j0] : 0.0;
    c[i] = fabs(v0) < INFINITY ? v0 : 0.0;  // a NaN or an infinity is no shift
    s1[i] = 0.0;
    s2[i] = 0.0;
    mn[i] = INFINITY;
    mx[i] = -INFINITY;
  }
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
    if (status && status[n] != 0) continue;
    cnt += 1.0;
#pragma unroll
    for (int i = 0; i < NH; i++) {
      const double v = x[i * ld + n];
      const double d = v - c[i];
      s1[i] += d;
      s2[i] = fma(d, d, s2[i]);
      mn[i] = v < mn[i] ? v : mn[i];  // a NaN never wins a comparison: skipped, as fmin / fmax would
      mx[i] = v > mx[i] ? v : mx[i];
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  cnt = warp_sum(cnt);
  if (lane == 0) red[warp][4 * NH] = cnt;
#pragma unroll
  for (int i = 0; i < NH; i++) {
    const double a = warp_sum(s1[i]), q = warp_sum(s2[i]), lo = warp_min(mn[i]), hi = warp_max(mx[i]);
    if (lane == 0) {
      red[warp][i] = a;
      red[warp][NH + i] = q;
      red[warp][2 * NH + i] = lo;
      red[warp][3 * NH + i] = hi;
    }
  }
  __syncthreads();
  if (threadIdx.x < 4 * NH + 1) {
    const int f = threadIdx.x, kind = f / NH;  // 0 S1, 1 S2, 2 min, 3 max, 4 count
    double a = red[0][f];
    for (int w = 1; w < THREADS / 32; w++) {
      const double b = red[w][f];
      a = kind == 2 ? fmin(a, b) : kind == 3 ? fmax(a, b) : a + b;
    }
    const int dst = kind == 4 ? 4 * NS : kind * NS + s0 + (f - kind * NH);
    if (kind != 4 || blockIdx.y == 0) partial[(long long)blockIdx.x * PARTIAL_STRIDE + dst] = a;
  }
}

// one CTA of 32 warps: warp w folds fields w, w + 32, w + 64 of the per-CTA partials (lanes stride over the partials, then the
// same shuffle tree); then 18 threads form the 74-double row from the totals and the shift
__global__ void __launch_bounds__(1024)
finish_kernel(const double* __restrict__ partial, int n_part, const double* __restrict__ x, long long ld, long long N,
              const int* __restrict__ status, const unsigned long long* __restrict__ first, double* __restrict__ row) {
  __shared__ double tot[4 * NS + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int f = warp; f < 4 * NS + 1; f += 32) {
    const bool is_min = f >= 2 * NS && f < 3 * NS, is_max = f >= 3 * NS && f < 4 * NS;
    double a = is_min ? INFINITY : is_max ? -INFINITY : 0.0;
    for (int b = lane; b < n_part; b += 32) {
      const double v = partial[(long long)b * PARTIAL_STRIDE + f];
      a = is_min ? fmin(a, v) : is_max ? fmax(a, v) : a + v;
    }
    a = is_min ? warp_min(a) : is_max ? warp_max(a) : warp_sum(a);
    if (lane == 0) tot[f] = a;
  }
  __syncthreads();
  const int f = threadIdx.x;
  if (f == 0) {
    row[0] = (double)N;
    row[1] = tot[4 * NS];
  }
  if (f < NS) {
    const double n = tot[4 * NS];
    const long long j0 = shift_aircraft(status, N, first);
    const double v0 = j0 >= 0 ? x[f * ld + j0] : 0.0;
    const double c = fabs(v0) < INFINITY ? v0 : 0.0;
    const double s1 = tot[f], s2 = tot[NS + f];
    const double inv = n > 0.0 ? 1.0 / n : 0.0;
    double m2 = fma(-s1, s1 * inv, s2);
    m2 = m2 > 0.0 ? m2 : (m2 == m2 ? 0.0 : m2);  // rounding may leave a negative ulp; a NaN stays a NaN
    row[2 + f] = tot[2 * NS + f];
    row[20 + f] = tot[3 * NS + f];
    row[38 + f] = n > 0.0 ? c + s1 * inv : 0.0;
    row[56 + f] = n > 0.0 ? m2 : 0.0;
  }
}

size_t summary_scratch(int grid) { return (size_t)grid * PARTIAL_STRIDE + 1; }

// row: 74 doubles on the device; scratch: summary_scratch(grid) doubles on the device, the per-CTA partials and then the
// first survivor's index
cudaError_t launch_summary(const LaunchCfg& cfg, const double* x, long long ld, long long N, const int* status, double* row,
                           double* scratch, int grid) {
  unsigned long long* first = reinterpret_cast<unsigned long long*>(scratch + (size_t)grid * PARTIAL_STRIDE);
  if (status && N > 0) {
    const cudaError_t e = cudaMemsetAsync(first, 0xff, sizeof *first, cfg.stream);
    if (e != cudaSuccess) return e;
    first_alive_kernel<<<grid, THREADS, 0, cfg.stream>>>(status, N, first);
    if (cfg.launch_counter) ++*cfg.launch_counter;
  }
  // six states per CTA, two CTAs (512 threads, 116 registers, no spills) per SM: measured best of {2, 3, 6} groups x {2, 3, 4}
  // CTAs per SM; the three-CTA build spills its accumulators.  tools/bench_entry_points.py --only summary on a B200 (1000 W),
  // L2 flushed, best of 20, 2^20 / 2^23 aircraft: no status array 0.096 / 0.263 ms (4.8 TB/s at 2^23); status words, all
  // alive 0.121 / 0.489 ms (0.117 / 0.484 ms with the search limited to the first 32 aircraft); only the last aircraft alive,
  // the search reading every status word, 0.078 / 0.166 ms (0.074 / 0.172 ms).
  partial_kernel<3, 2><<<dim3(grid, 3), THREADS, 0, cfg.stream>>>(x, ld, N, status, first, scratch);
  finish_kernel<<<1, 1024, 0, cfg.stream>>>(scratch, grid, x, ld, N, status, first, row);
  if (cfg.launch_counter) *cfg.launch_counter += 2;
  return cudaGetLastError();
}

int summary_grid(const LaunchCfg& cfg, long long N) {
  // grid.x x 3 (state groups) CTAs of 256 threads, two resident per SM, six independent loads per thread and iteration in
  // flight; never more CTAs than there is work for
  long long want = (N + THREADS - 1) / THREADS;
  const long long cap = (long long)cfg.sm_count * 3;
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  return (int)want;
}

}  // namespace stats
}  // namespace f16

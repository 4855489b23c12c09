// f16_linalg.cu -- the small dense algebra between linearise_batch and the fused LQR law, one thread per aircraft:
//
//   reduce_jacobian   env.py:49,152-193,350  the 9-state / 3-input model the reference feeds to LQR and MPC.  Its forward
//                     differences perturb the same full-model evaluation as F16.linearise does, so A_na / B_na are an
//                     exact gather of rows {3,4,7,8,9,10,11,16,17} and columns mpc_x_idx / {13,14,15} of the 18x18 A
//                     (the two LEF derivatives swap places, env.py:184,189).
//   zoh               env.py:46,50  scipy.signal.cont2discrete(method='zoh'): expm([[A, B], [0, 0]] dt) -> Ad, Bd,
//                     by scaling and squaring with a degree-14 Taylor polynomial (||M|| <= 1/2 after scaling).
//   dlqr              utils.py:219-245  K = (B'PB + R)^-1 B'PA with P from the discrete algebraic Riccati equation,
//                     solved by the structured doubling algorithm (quadratically convergent; ~21 doublings at dt = 1 ms);
//                     a solution that does not stabilise A - BK is flagged (info -5), as are non-finite iterates (-3).
//
// These are tolerance-parity kernels (scipy uses Pade / QZ for the same quantities); FP64 throughout, no tensor cores:
// the matrices are 9x9 .. 22x22 and there are a few thousand of them.
#include <math.h>

#include "f16_kernels.cuh"
#include "f16_linalg.cuh"

namespace f16 {
namespace linalg {

// the per-system bodies (zoh_one, dlqr_one, reduce_one) live in f16_linalg.cuh, shared with the host build of the tests

__global__ void __launch_bounds__(64)
zoh_kernel(const double* __restrict__ A, const double* __restrict__ B, int n, int m, long long N, double dt,
           double* __restrict__ Ad, double* __restrict__ Bd) {
  double M[MAXD * MAXD], T1[MAXD * MAXD], T2[MAXD * MAXD];
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += (long long)gridDim.x * blockDim.x)
    zoh_one(A, B, n, m, p, dt, Ad, Bd, M, T1, T2);
}

__global__ void __launch_bounds__(64)
dlqr_kernel(const double* __restrict__ Ad, const double* __restrict__ Bd, const double* __restrict__ Q, const double* __restrict__ R,
            int n, int m, long long N, int max_doublings, double tol, double* __restrict__ K, double* __restrict__ P_out,
            int* __restrict__ info) {
  double Ak[MAXD * MAXD], G[MAXD * MAXD], H[MAXD * MAXD], W[MAXD * MAXD], T1[MAXD * MAXD], T2[MAXD * MAXD], T3[MAXD * MAXD];
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += (long long)gridDim.x * blockDim.x)
    dlqr_one(Ad, Bd, Q, R, n, m, p, max_doublings, tol, K, P_out, info, Ak, G, H, W, T1, T2, T3);
}

__global__ void __launch_bounds__(256)
reduce_jacobian_kernel(const double* __restrict__ A, long long N, double* __restrict__ A_na, double* __restrict__ B_na) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < N * 108; e += (long long)gridDim.x * blockDim.x) {
    const long long p = e / 108;
    reduce_one(A, p, (int)(e - p * 108), A_na, B_na);
  }
}

static int blocks_for(long long items, int per_block, int sm_count) {
  long long b = (items + per_block - 1) / per_block;
  const long long cap = (long long)sm_count * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

cudaError_t launch_zoh(const LaunchCfg& cfg, const double* A, const double* B, int n, int m, long long N, double dt, double* Ad,
                       double* Bd) {
  if (N <= 0) return cudaSuccess;
  zoh_kernel<<<blocks_for(N, 64, cfg.sm_count), 64, 0, cfg.stream>>>(A, B, n, m, N, dt, Ad, Bd);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

cudaError_t launch_dlqr(const LaunchCfg& cfg, const double* Ad, const double* Bd, const double* Q, const double* R, int n, int m,
                        long long N, int max_doublings, double tol, double* K, double* P, int* info) {
  if (N <= 0) return cudaSuccess;
  dlqr_kernel<<<blocks_for(N, 64, cfg.sm_count), 64, 0, cfg.stream>>>(Ad, Bd, Q, R, n, m, N, max_doublings, tol, K, P, info);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

cudaError_t launch_reduce_jacobian(const LaunchCfg& cfg, const double* A, long long N, double* A_na, double* B_na) {
  if (N <= 0) return cudaSuccess;
  reduce_jacobian_kernel<<<blocks_for(N * 108, 256, cfg.sm_count), 256, 0, cfg.stream>>>(A, N, A_na, B_na);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

}  // namespace linalg
}  // namespace f16

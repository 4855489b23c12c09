// f16_kernels.cuh -- launch interface between the C ABI (f16_api.cu) and the kernel translation units.  f16::strict is
// f16_kernels.cu, the parity build (reference operation order, -fmad=false); f16::fast is f16_step_fast.cu and
// f16_linearise_fast.cu, the arithmetic of f16_fast.cuh that F16_MATH_FAST runs.
#pragma once
#include <cuda_runtime.h>

#include "f16_model.cuh"

namespace f16 {

struct DevTables {
  const double* hifi;  // F16_IMG_HIFI_DOUBLES, 16-byte aligned
  const double* lofi;  // F16_IMG_LOFI_DOUBLES
  const double* hifi_fast;  // F16_FI_DOUBLES: the (f, d) image of f16_fast.cuh, used by the F16_MATH_FAST step kernel
  // Read by no kernel, but part of the parameter block of every kernel that takes DevTables: without it the later parameters
  // move up by 8 bytes and ptxas allocates registers differently in the step kernels (166 <-> 168 / 252 <-> 254 registers),
  // which has not been measured on the GPU.
  int zero;
};

struct BatchSel {           // which aircraft run which model
  const unsigned char* fi;  // per-aircraft fidelity (device) or nullptr
  int fi_default;
  const double* xcg;  // per-aircraft xcg (device) or nullptr
  double xcg_default;
};

struct LaunchCfg {
  cudaStream_t stream;
  int sm_count;
  bool smem_tables;  // stage tables in shared memory with TMA bulk copies (default) or read them through L1/L2
  unsigned long long* launch_counter;
  // time-chunked scheduling of the fast hifi step (f16_step_fast.cu): on/off, and the device scratch of one int per 32 aircraft
  bool step_chunking = false;
  int* step_progress = nullptr;
  long long step_progress_cap = 0;
  bool trim_fixed_point_exit = true;  // Nelder-Mead: leave a search that has reached a bitwise fixed point (f16_model.cuh)
};

namespace strict {
cudaError_t launch_nlplant(const LaunchCfg&, const DevTables&, const BatchSel&, const double* xu, long long ld_in, double* xdot,
                           long long ld_out, long long N, int* status);
cudaError_t launch_calc_xdot(const LaunchCfg&, const DevTables&, const BatchSel&, const double* x, long long ld_x, const double* u,
                             long long ld_u, double* xdot, long long ld_out, long long N, int* status);
cudaError_t launch_step(const LaunchCfg&, const DevTables&, const BatchSel&, double* x, long long ld_x, const double* u, long long ld_u,
                        long long N, int K, double dt, const LqrLaw* lqr_host, int* status, int* steps_done);
cudaError_t launch_linearise(const LaunchCfg&, const DevTables&, const BatchSel&, const double* x, long long ld_x, const double* u,
                             long long ld_u, long long N, double eps, int scheme, double* A, double* B, int* status);
cudaError_t launch_hifi_probe(const LaunchCfg&, const DevTables&, const double* alpha, const double* beta, const double* el,
                              long long N, double* coef, int* cells, int* status);
cudaError_t launch_lofi_probe(const LaunchCfg&, const DevTables&, const double* alpha, const double* beta, const double* el,
                              const double* dail, const double* drud, long long N, double* out);
cudaError_t launch_atmos(const LaunchCfg&, const double* alt, const double* vt, long long N, double* coeff);
cudaError_t launch_div_probe(const LaunchCfg&, const double* a, const double* b, long long N, double* out);
cudaError_t launch_trim(const LaunchCfg&, const DevTables&, const BatchSel&, const double* h, const double* v, long long N, double tol,
                        int maxiter, const double* ux0, double* x_trim, long long ld_x, double* info, long long ld_info, int* status);
}  // namespace strict

namespace fast {
// f16_step_fast.cu: step_batch, both fidelities
cudaError_t launch_step(const LaunchCfg&, const DevTables&, const BatchSel&, double* x, long long ld_x, const double* u, long long ld_u,
                        long long N, int K, double dt, const LqrLaw* lqr_host, int* status, int* steps_done);
// trim_batch with the objective on the step kernel's arithmetic; always stages the tables in shared memory
cudaError_t launch_trim(const LaunchCfg&, const DevTables&, const BatchSel&, const double* h, const double* v, long long N, double tol,
                        int maxiter, const double* ux0, double* x_trim, long long ld_x, double* info, long long ld_info, int* status);
// Nlplant_batch (u == nullptr, x = xu [17][N]) / calc_xdot_batch on the arithmetic of f16_fast.cuh, TMA-staged input tiles
cudaError_t launch_xdot_fast(const LaunchCfg&, const DevTables&, const BatchSel&, const double* x, long long ld_x, const double* u,
                             long long ld_u, double* xdot, long long ld_out, long long N, int* status, unsigned* redo);
// f16_linearise_fast.cu: linearise_batch on the arithmetic of f16_fast.cuh (two aircraft per warp, no tile, no barriers)
cudaError_t launch_linearise_fast(const LaunchCfg&, const DevTables&, const BatchSel&, const double* x, long long ld_x, const double* u,
                                  long long ld_u, long long N, double eps, int scheme, double* A, double* B, int* status, unsigned* redo);
cudaError_t launch_fast_probe(const LaunchCfg&, const DevTables&, const double* alpha, const double* beta, const double* el,
                              long long N, double* coef, int* cells, double* lam, int* status);
}  // namespace fast

// f16_linalg.cu: reduced-model gather, zero-order-hold discretisation, discrete LQR gain (one thread per aircraft)
namespace linalg {
cudaError_t launch_reduce_jacobian(const LaunchCfg&, const double* A, long long N, double* A_na, double* B_na);
cudaError_t launch_zoh(const LaunchCfg&, const double* A, const double* B, int n, int m, long long N, double dt, double* Ad,
                       double* Bd);
cudaError_t launch_dlqr(const LaunchCfg&, const double* Ad, const double* Bd, const double* Q, const double* R, int n, int m,
                        long long N, int max_doublings, double tol, double* K, double* P, int* info);
}  // namespace linalg

// f16_stats.cu: per-state summary of a batch (count, alive, min, max, mean, M2), reduced on the device
namespace stats {
size_t summary_scratch(int grid);  // doubles of device scratch launch_summary needs at this grid
cudaError_t launch_summary(const LaunchCfg&, const double* x, long long ld, long long N, const int* status, double* row,
                           double* scratch, int grid);
int summary_grid(const LaunchCfg&, long long N);
}  // namespace stats

// f16_partition.cu: a mixed batch ordered by fidelity for the fused step (stable three-way partition, gather, scatter)
namespace partition {
cudaError_t launch_build(const LaunchCfg&, const unsigned char* fi, long long N, unsigned* perm, long long* totals_dev,
                         unsigned* scratch);
cudaError_t launch_gather_f64(const LaunchCfg&, const double* src, long long ld_src, double* dst, long long ld_dst, int planes,
                              const unsigned* perm, long long N);
cudaError_t launch_scatter_f64(const LaunchCfg&, const double* src, long long ld_src, double* dst, long long ld_dst, int planes,
                               const unsigned* perm, long long N);
cudaError_t launch_scatter_i32(const LaunchCfg&, const int* src, int* dst, const unsigned* perm, long long N);
cudaError_t launch_fill_i32(const LaunchCfg&, int* dst, int value, long long N);
cudaError_t launch_gather_i32(const LaunchCfg&, const int* src, int* dst, const unsigned* perm, long long N);
cudaError_t launch_mark_survivors(const LaunchCfg&, const int* status, const int* k_launch, int* k_total, int base, long long N,
                                  unsigned char* flag);
cudaError_t launch_close_steps(const LaunchCfg&, int* k_total, int K, long long N);
int n_cta(long long N);
}  // namespace partition

// FP64 FMA micro-benchmark (f16_peak.cu): returns flops executed
cudaError_t launch_dfma_peak(cudaStream_t stream, int sm_count, long long iters, double* sink, double* flops);

}  // namespace f16

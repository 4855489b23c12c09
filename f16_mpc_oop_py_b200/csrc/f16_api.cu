// f16_api.cu -- the C ABI of libf16_b200.so (include/f16_b200.h): library state, table upload, host<->device
// plumbing and dispatch into the strict / fast kernel builds.  No arithmetic of the plant happens on the host.
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <cmath>
#include <memory>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/f16_b200.h"
#include "f16_kernels.cuh"
#include "f16_tables_host.h"

static_assert(sizeof(f16_lqr_t) == sizeof(f16::LqrLaw), "f16_lqr_t and the device-side law must have one layout");

namespace {

struct DevBuf {  // grow-only device scratch; a reserve that grows it moves it
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
};

constexpr int kMaxArrays = 16;    // per-aircraft arrays of one host-buffer call (lqr_gain_batch: 13)
constexpr int kMaxContexts = 64;  // device contexts of f16_init_devices

// Everything that belongs to ONE device: streams, events, the three table images, scratch.  The library keeps one context per
// device handed to f16_init_devices (exactly one after f16_init); aircraft never interact, so contexts share nothing.
struct Dev {
  int ordinal = -1;
  int sm_count = 0;
  cudaStream_t stream = nullptr;                 // kernels, and the copies of the *_dev-side helpers (f16_memcpy_*)
  cudaStream_t s_in = nullptr, s_out = nullptr;  // H2D / D2H of the host-buffer entry points
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;      // f16_timer_*
  cudaEvent_t e_in[3] = {}, e_work[3] = {}, e_out[3] = {};  // the three slots of the chunk pipeline
  cudaEvent_t e_snap[2] = {}, e_snap_out[2] = {};         // step_batch_traj: snapshot slot filled (stream) / copied out (s_out)
  double* d_hifi = nullptr;
  double* d_lofi = nullptr;
  double* d_hifi_fast = nullptr;
  unsigned long long launches = 0;
  // legacy single-aircraft path: mapped pinned host memory, the kernel reads and writes it directly
  double* pin = nullptr;      // [17 in | 18 out | 3 atmos in/out ...]
  double* pin_dev = nullptr;
  // Scratch.  A reserve may move a buffer, so two stages that are live at the same time never share one.
  // slot[i]: array i of the running host-buffer call, all its chunk slots (run_pipeline).  What runs inside that call's work
  // has its own buffers:
  //   step_on_device -> step_partitioned: b_perm, b_pscr, b_px, b_pu, b_pxcg, b_pst, b_pk
  //                  -> step_compacting:  b_perm, b_pscr, b_pk, b_c*  (the two are alternatives, neither runs inside the other)
  //   the step kernels: b_prog;  run_xdot / run_linearise: b_redo;  the summary rows: b_sum;  step_batch_traj's two
  //   snapshots: b_snap;  the Q / R of dlqr_batch and lqr_gain_batch: b_qr
  // b_flush: f16_flush_l2, and the sink of f16_measure_fp64_peak; neither runs inside another call.
  DevBuf slot[kMaxArrays];
  DevBuf b_perm, b_pscr, b_px, b_pu, b_pxcg, b_pst, b_pk;
  DevBuf b_cx[2], b_cu[2], b_cxcg[2], b_cst[2], b_ck[2], b_co[2], b_cflag, b_ckl;  // survivor compaction (step_compacting)
  DevBuf b_prog, b_redo, b_sum, b_snap, b_qr, b_flush;
  ~Dev() {  // tolerant of a half-built context (a failed init releases what it had created); the buffers go after this body
    if (ordinal < 0 || cudaSetDevice(ordinal) != cudaSuccess) { cudaGetLastError(); return; }
    if (stream) cudaStreamSynchronize(stream);
    if (s_in) cudaStreamSynchronize(s_in);
    if (s_out) cudaStreamSynchronize(s_out);
    if (d_hifi) cudaFree(d_hifi);
    if (d_lofi) cudaFree(d_lofi);
    if (d_hifi_fast) cudaFree(d_hifi_fast);
    if (pin) cudaFreeHost(pin);
    for (cudaEvent_t e : {ev0, ev1, e_in[0], e_in[1], e_in[2], e_work[0], e_work[1], e_work[2], e_out[0], e_out[1], e_out[2],
                          e_snap[0], e_snap[1], e_snap_out[0], e_snap_out[1]})
      if (e) cudaEventDestroy(e);
    for (cudaStream_t st : {stream, s_in, s_out})
      if (st) cudaStreamDestroy(st);
    cudaGetLastError();
  }
};

struct State {
  bool ready = false;
  int init_rc = F16_ERR_NOINIT;
  std::vector<std::unique_ptr<Dev>> devs;  // index = position in the list given to f16_init_devices
  int cur = 0;                             // the context the *_dev entry points and the memory helpers work on
  std::vector<double> payload;
  std::string table_source;
  int math_mode = F16_MATH_STRICT;
  int clr_mode = F16_CLR_AS_BUILT;
  bool smem_tables = true;
  int lin_variant = 0;         // f16_set_linearise_variant: 0 = the default kernel of the math mode, 1 / 2 = reference order
  bool step_chunking = true;
  bool host_pipeline = true;   // chunked H2D / kernel / D2H overlap in the host-buffer entry points
  bool trim_fp_exit = true;    // trim_batch: fixed-point exit of the Nelder-Mead search (same results, see f16_model.cuh)
  bool compaction = false;     // long runs: survivors repacked between chunks of steps (step_compacting); opt-in
  std::atomic<double> default_xcg{0.25};
  std::atomic<int> last_status{0};
};

State G;
std::mutex G_mu;
thread_local Dev* D = nullptr;  // the context the calling thread works on (worker threads of a multi-device call: their own)
thread_local std::string t_err;

void set_err(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  t_err = buf;
}

int cuda_fail(cudaError_t e, const char* what) {
  set_err("%s: %s", what, cudaGetErrorString(e));
  return F16_ERR_CUDA;
}
#define CK(call)                                          \
  do {                                                    \
    cudaError_t e__ = (call);                             \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

std::string lib_dir() {
  Dl_info info;
  if (dladdr((void*)&f16_init, &info) && info.dli_fname) {
    std::string p = info.dli_fname;
    size_t s = p.rfind('/');
    return s == std::string::npos ? std::string(".") : p.substr(0, s);
  }
  return std::string();
}

// the three table images of the context D (current device = D->ordinal)
int upload_tables() {
  std::vector<double> img;
  f16::build_hifi_image(G.payload, G.clr_mode == F16_CLR_FROM_FILE, img);
  if (!D->d_hifi) CK(cudaMalloc(&D->d_hifi, F16_IMG_HIFI_BYTES));
  CK(cudaMemcpy(D->d_hifi, img.data(), F16_IMG_HIFI_BYTES, cudaMemcpyHostToDevice));
  f16::build_hifi_fast_image(G.payload, G.clr_mode == F16_CLR_FROM_FILE, img);
  if (!D->d_hifi_fast) CK(cudaMalloc(&D->d_hifi_fast, F16_FI_BYTES));
  CK(cudaMemcpy(D->d_hifi_fast, img.data(), F16_FI_BYTES, cudaMemcpyHostToDevice));
  f16::build_lofi_image(img);
  if (!D->d_lofi) CK(cudaMalloc(&D->d_lofi, F16_IMG_LOFI_BYTES));
  CK(cudaMemcpy(D->d_lofi, img.data(), F16_IMG_LOFI_BYTES, cudaMemcpyHostToDevice));
  return F16_OK;
}

// one device context: streams, events, pinned scratch of the legacy symbols, table images
int create_context(Dev* d, int ordinal) {
  D = d;
  CK(cudaSetDevice(ordinal));
  d->ordinal = ordinal;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, ordinal));
  if (prop.major != 10) {
    set_err("device %d is sm_%d%d; libf16_b200 is built for sm_100a only", ordinal, prop.major, prop.minor);
    return F16_ERR_CUDA;
  }
  d->sm_count = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&d->s_in, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&d->s_out, cudaStreamNonBlocking));
  CK(cudaEventCreate(&d->ev0));
  CK(cudaEventCreate(&d->ev1));
  for (int i = 0; i < 3; i++) {
    CK(cudaEventCreateWithFlags(&d->e_in[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&d->e_work[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&d->e_out[i], cudaEventDisableTiming));
  }
  for (int i = 0; i < 2; i++) {
    CK(cudaEventCreateWithFlags(&d->e_snap[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&d->e_snap_out[i], cudaEventDisableTiming));
  }
  CK(cudaHostAlloc((void**)&d->pin, 64 * sizeof(double), cudaHostAllocMapped));
  CK(cudaHostGetDevicePointer((void**)&d->pin_dev, d->pin, 0));
  return upload_tables();
}

// devices == nullptr: one context on `device` (-1: $F16_DEVICE / $LOCAL_RANK / 0); else one context per entry of devices[0..ndev)
// (ndev <= 0: every visible device).  Every failure path releases what it had created and leaves its code in G.init_rc.
int init_locked(const char* table_path, int device, const int* devices, int ndev) {
  if (G.ready) return F16_OK;
  int present = 0;
  cudaError_t e = cudaGetDeviceCount(&present);
  if (e != cudaSuccess || present == 0) {
    set_err("no CUDA device: %s (libf16_b200 has no CPU path)", e != cudaSuccess ? cudaGetErrorString(e) : "count = 0");
    return G.init_rc = F16_ERR_CUDA;
  }
  std::vector<int> want;
  if (devices && ndev > 0) {
    want.assign(devices, devices + ndev);
  } else if (devices || ndev != 0) {  // f16_init_devices(NULL / anything, <= 0): all of them
    for (int i = 0; i < present; i++) want.push_back(i);
  } else {
    if (device < 0) {
      const char* v = getenv("F16_DEVICE");
      if (!v || !*v) v = getenv("LOCAL_RANK");
      device = (v && *v) ? atoi(v) % present : 0;
    }
    want.push_back(device);
  }
  for (int o : want)
    if (o < 0 || o >= present) { set_err("device %d out of range (%d present)", o, present); return G.init_rc = F16_ERR_ARG; }
  if ((int)want.size() > kMaxContexts) { set_err("more than %d device contexts", kMaxContexts); return G.init_rc = F16_ERR_ARG; }

  std::string err;
  if (!f16::load_canonical(table_path, lib_dir(), G.payload, G.table_source, err)) {
    set_err("%s", err.c_str());
    return G.init_rc = F16_ERR_TABLES;
  }
  if (!f16::check_grids(G.payload, err)) { set_err("%s", err.c_str()); return G.init_rc = F16_ERR_TABLES; }

  if (const char* v = getenv("F16_XCG")) G.default_xcg = atof(v);
  if (const char* v = getenv("F16_MATH")) G.math_mode = (!strcmp(v, "fast") || !strcmp(v, "1")) ? F16_MATH_FAST : F16_MATH_STRICT;
  if (const char* v = getenv("F16_CLR")) G.clr_mode = (!strcmp(v, "file") || !strcmp(v, "1")) ? F16_CLR_FROM_FILE : F16_CLR_AS_BUILT;
  if (const char* v = getenv("F16_TABLE_STAGING")) G.smem_tables = atoi(v) != 0;
  if (const char* v = getenv("F16_STEP_CHUNKING")) G.step_chunking = atoi(v) != 0;
  if (const char* v = getenv("F16_HOST_PIPELINE")) G.host_pipeline = atoi(v) != 0;
  if (const char* v = getenv("F16_STEP_COMPACTION")) G.compaction = atoi(v) != 0;
  if (const char* v = getenv("F16_LIN_VARIANT")) G.lin_variant = (atoi(v) == 1 || atoi(v) == 2) ? atoi(v) : 0;

  for (int o : want) {
    G.devs.emplace_back(new Dev());
    const int rc = create_context(G.devs.back().get(), o);
    if (rc != F16_OK) {
      const std::string keep = t_err;
      G.devs.clear();
      D = nullptr;
      t_err = keep;
      return G.init_rc = rc;
    }
  }
  G.cur = 0;
  D = G.devs[0].get();
  if (cudaSetDevice(D->ordinal) != cudaSuccess) return G.init_rc = F16_ERR_CUDA;
  G.ready = true;
  return G.init_rc = F16_OK;
}

// every entry point (library mutex held): the calling thread works on the current context
int ensure() {
  if (!G.ready) {
    const int rc = init_locked(nullptr, -1, nullptr, 0);
    if (rc != F16_OK) return rc;
  }
  D = G.devs[(size_t)G.cur].get();
  if (cudaSetDevice(D->ordinal) != cudaSuccess) { set_err("cudaSetDevice(%d) failed", D->ordinal); return F16_ERR_CUDA; }
  return F16_OK;
}

f16::LaunchCfg cfg(bool smem_tables) {
  f16::LaunchCfg c;
  c.stream = D->stream;
  c.sm_count = D->sm_count;
  c.smem_tables = smem_tables;
  c.launch_counter = &D->launches;
  c.step_chunking = G.step_chunking;
  c.step_progress = (int*)D->b_prog.p;
  c.step_progress_cap = (long long)(D->b_prog.cap / 4);
  c.trim_fixed_point_exit = G.trim_fp_exit;
  return c;
}
f16::DevTables tabs() { return f16::DevTables{D->d_hifi, D->d_lofi, D->d_hifi_fast, 0}; }
f16::BatchSel sel_of(const unsigned char* fi, int fi_default, const double* xcg, double xcg_default) {
  return f16::BatchSel{fi, fi_default, xcg, xcg_default};
}

// F16_MATH_FAST runs the kernels of f16_step_fast.cu and f16_linearise_fast.cu (the arithmetic of f16_fast.cuh) where the entry
// point below takes them, and the parity build (f16::strict) everywhere else
bool fast_mode() { return G.math_mode == F16_MATH_FAST; }

// Nlplant_batch (u == NULL: x is xu [17][ld_x]) and calc_xdot_batch.  A batch worth staging tables for runs the TMA-tiled kernels
// of f16_step_fast.cu in F16_MATH_FAST; a handful of aircraft (the legacy Nlplant symbol among them) read the tables through L2
cudaError_t run_xdot(const f16::BatchSel& sel, const double* x, long long ld_x, const double* u, long long ld_u, double* xdot,
                     long long ld_out, long long N, int* status) {
  const bool staged = G.smem_tables && N >= 4096;
  if (fast_mode() && staged) {
    cudaError_t e = D->b_redo.reserve((size_t)((N + 31) / 32) * 4);
    if (e != cudaSuccess) return e;
    return f16::fast::launch_xdot_fast(cfg(true), tabs(), sel, x, ld_x, u, ld_u, xdot, ld_out, N, status, (unsigned*)D->b_redo.p);
  }
  if (!u) return f16::strict::launch_nlplant(cfg(staged), tabs(), sel, x, ld_x, xdot, ld_out, N, status);
  return f16::strict::launch_calc_xdot(cfg(staged), tabs(), sel, x, ld_x, u, ld_u, xdot, ld_out, N, status);
}
// linearise_batch.  F16_MATH_STRICT: the staged reference-order kernel (CTA per 32 aircraft).  F16_MATH_FAST, variant 0: the
// two-aircraft-per-warp kernel on the arithmetic of f16_fast.cuh (f16_linearise_fast.cu); variants 1 and 2 keep the
// reference-order kernel in fast mode as well.
cudaError_t run_linearise(const f16::BatchSel& sel, const double* x, long long ld_x, const double* u, long long ld_u, long long N,
                          double eps, int scheme, double* A, double* B, int* status) {
  if (fast_mode() && G.lin_variant == 0 && N < (1LL << 31)) {
    cudaError_t e = D->b_redo.reserve((size_t)((N + 1) / 2) * 4);
    if (e != cudaSuccess) return e;
    return f16::fast::launch_linearise_fast(cfg(true), tabs(), sel, x, ld_x, u, ld_u, N, eps, scheme, A, B, status,
                                            (unsigned*)D->b_redo.p);
  }
  return f16::strict::launch_linearise(cfg(true), tabs(), sel, x, ld_x, u, ld_u, N, eps, scheme, A, B, status);
}
// every launch of the fused step: in F16_MATH_FAST both fidelities run the step kernels of f16_step_fast.cu
cudaError_t run_step(const f16::LaunchCfg& c, const f16::BatchSel& sel, double* x, long long ld_x, const double* u, long long ld_u,
                     long long N, int K, double dt, const f16::LqrLaw* law, int* status, int* steps_done) {
  return (fast_mode() ? f16::fast::launch_step : f16::strict::launch_step)(c, tabs(), sel, x, ld_x, u, ld_u, N, K, dt, law, status,
                                                                           steps_done);
}
// trim_batch: in F16_MATH_FAST with table staging on, the objective of f16_step_fast.cu at every batch size -- measured on a B200
// (1000 W), 1 / 512 points take 2.5 / 11.9 ms there and 5.1 / 25.4 ms on the parity build; that stages its tables from 1024 points
cudaError_t run_trim(const f16::BatchSel& sel, const double* h, const double* V, long long N, double tol, int maxiter, const double* ux0,
                     double* x_trim, long long ld_x, double* info, long long ld_info, int* status) {
  if (fast_mode() && G.smem_tables)
    return f16::fast::launch_trim(cfg(true), tabs(), sel, h, V, N, tol, maxiter, ux0, x_trim, ld_x, info, ld_info, status);
  return f16::strict::launch_trim(cfg(G.smem_tables && N >= 1024), tabs(), sel, h, V, N, tol, maxiter, ux0, x_trim, ld_x, info,
                                  ld_info, status);
}

int bad_arg(const char* entry) {
  set_err("%s: bad argument", entry);
  return F16_ERR_ARG;
}

// ---- the argument checks, one per operation: the host-buffer form of an operation is its *_dev form with every ld = N ----
bool lqr_ok(const f16_lqr_t* lqr) {
  if (!lqr) return true;
  if (lqr->n_sel < 0 || lqr->n_sel > 18) return false;
  for (int j = 0; j < lqr->n_sel; j++)
    if (lqr->sel[j] < 0 || lqr->sel[j] > 17) return false;
  return true;
}
bool nlplant_ok(const double* xu, long long ld_in, const double* xdot, long long ld_out, long long N) {
  return N >= 0 && (N == 0 || (xu && xdot)) && ld_in >= N && ld_out >= N;
}
bool calc_xdot_ok(const double* x, long long ld_x, const double* u, long long ld_u, const double* xdot, long long ld_out, long long N) {
  return nlplant_ok(x, ld_x, xdot, ld_out, N) && (N == 0 || u) && ld_u >= N;
}
bool step_ok(const double* x, long long ld_x, const double* u, long long ld_u, long long N, int K, const f16_lqr_t* lqr) {
  return N >= 0 && K >= 0 && (N == 0 || (x && u)) && ld_x >= N && ld_u >= N && lqr_ok(lqr);
}
bool stats_ok(const double* x, long long ld_x, const double* u, long long ld_u, long long N, int K, int snap_every,
              const f16_lqr_t* lqr, const double* rows) {
  return step_ok(x, ld_x, u, ld_u, N, K, lqr) && snap_every >= 1 && (rows || K < snap_every);
}
bool linearise_ok(const double* x, long long ld_x, const double* u, long long ld_u, long long N, double eps, int scheme,
                  const double* A, const double* B) {
  return N >= 0 && (N == 0 || (x && u && A && B)) && ld_x >= N && ld_u >= N && (scheme == 0 || scheme == 1) &&
         eps >= 1e-12 && eps <= 1e3;
}
bool trim_ok(const double* h, const double* V, long long N, double tol, int maxiter, const double* x_trim, long long ld_x,
             const double* info, long long ld_info) {
  return N >= 0 && (N == 0 || (h && V && x_trim)) && ld_x >= N && (!info || ld_info >= N) && tol >= 0 && maxiter >= 1;
}
bool summary_ok(const double* x, long long ld_x, long long N, const double* row) {
  return N >= 0 && row && (N == 0 || x) && ld_x >= N;
}
bool dims_ok(int n, int m) { return n >= 1 && m >= 1 && n <= 18 && n + m <= 22; }
bool reduce_ok(const double* A, long long N, const double* A_na, const double* B_na) {
  return N >= 0 && (N == 0 || (A && A_na && B_na));
}
bool zoh_ok(const double* A, const double* B, int n, int m, long long N, double dt, const double* Ad, const double* Bd) {
  return N >= 0 && dims_ok(n, m) && std::isfinite(dt) && (N == 0 || (A && B && Ad && Bd));
}
bool dlqr_ok(const double* Ad, const double* Bd, const double* Q, const double* R, int n, int m, long long N, const double* K) {
  return N >= 0 && dims_ok(n, m) && (N == 0 || (Ad && Bd && Q && R && K));
}

// ---- host arrays <-> device slots of the host-buffer entry points -----------------------------------------------------
// One per-aircraft array of a host-buffer call.  In the caller's array aircraft i has `planes` elements `ld` apart starting at
// element i (SoA) or the `row` elements from i * row on (AoS); on the device a chunk of m aircraft is packed: planes m apart, or
// m rows.  A NULL array gets no slot and the kernels see NULL, unless it is `scratch`: then the kernels get a slot and nothing
// is copied (status words the caller does not want, the intermediates of lqr_gain_batch).
enum Dir { IN = 1, OUT = 2, INOUT = 3 };
struct Arr {
  void* host;
  int dir;
  int esize;   // bytes per element
  int planes;  // SoA: planes per aircraft (AoS: 1)
  int row;     // AoS: elements per aircraft (SoA: 1)
  bool scratch;
};
Arr soa(const void* host, int dir, int esize, int planes = 1, bool scratch = false) {
  return Arr{const_cast<void*>(host), dir, esize, planes, 1, scratch};
}
Arr aos(const void* host, int dir, int esize, int row, bool scratch = false) {
  return Arr{const_cast<void*>(host), dir, esize, 1, row, scratch};
}

// aircraft [first, first + m) of `a` (plane stride ld) <-> its packed device slot
cudaError_t copy_chunk(const Arr& a, void* slot, long long ld, long long first, long long m, cudaMemcpyKind kind, cudaStream_t st) {
  char* host = (char*)a.host + (size_t)first * a.row * a.esize;
  const size_t w = (size_t)m * a.row * a.esize;  // bytes of one plane of the chunk
  const bool in = kind == cudaMemcpyHostToDevice;
  void* dst = in ? slot : host;
  const void* src = in ? (const void*)host : slot;
  if (a.planes == 1 || ld == m) return cudaMemcpyAsync(dst, src, (size_t)a.planes * w, kind, st);
  const size_t hp = (size_t)ld * a.esize;
  return cudaMemcpy2DAsync(dst, in ? w : hp, src, in ? hp : w, w, (size_t)a.planes, kind, st);
}

struct Slots {  // the device slots of one chunk, by array position (NULL: the array was not passed)
  void* p[kMaxArrays];
  double* f64(int i) const { return (double*)p[i]; }
  int* i32(int i) const { return (int*)p[i]; }
  const unsigned char* u8(int i) const { return (const unsigned char*)p[i]; }
};

// A host-buffer call on one device is a pipeline of chunks: while the kernels of chunk c run on D->stream, chunk c + 1 arrives on
// D->s_in and the result of chunk c - 1 leaves on D->s_out (PCIe is full duplex: a copy-bound call -- one derivative, one step --
// takes max(in, out) instead of in + kernel + out).  Chunk c lives in slot c mod 3 of each array's buffer; chunks are multiples
// of 32 aircraft, so that slots stay 256-byte aligned and a warp-task never straddles two chunks.  Results do not depend on the
// cut: every aircraft is computed by the same arithmetic wherever it lands.
struct Chunks {
  long long chunk = 0;
  int count = 0, slots = 0;
};
Chunks plan_chunks(long long n, long long min_chunk, int max_chunks) {
  Chunks c;
  long long k = G.host_pipeline ? n / min_chunk : 1;
  if (k < 1) k = 1;
  if (k > max_chunks) k = max_chunks;
  c.chunk = (((n + k - 1) / k) + 31) / 32 * 32;
  c.count = (int)((n + c.chunk - 1) / c.chunk);
  c.slots = c.count < 3 ? c.count : 3;
  return c;
}
// a call whose kernels must see all n aircraft at once (n >= 1): a trim launch lasts as long as its slowest point, a summary
// row reduces the whole slice
Chunks one_chunk(long long n) { return plan_chunks(n, n, 1); }

// Aircraft [lo, lo + n) of the arrays `arr` (plane stride ld) in the chunks `ch`: the pipeline copies in the IN arrays of each
// chunk, calls work(slots, m) to enqueue its kernels on D->stream, and copies out the OUT arrays.  Returns after everything has
// landed.  Issue order on the host: normally in(c), work(c), out(c - 1) -- work() only enqueues, and a pageable in(c + 1), which
// blocks the host while the driver stages it, then runs under the kernels of chunk c.  With work_blocks (work() waits on the
// device: the survivor counts of step_compacting) the copies either side of a chunk are enqueued BEFORE its work: in(c + 1),
// out(c - 1), work(c).
template <size_t NA, class Work>
int run_pipeline(const Arr (&arr)[NA], long long ld, long long lo, long long n, const Chunks& ch, bool work_blocks, Work work) {
  static_assert(NA <= kMaxArrays, "one slot buffer per array");
  size_t bytes[NA];  // per aircraft
  for (size_t i = 0; i < NA; i++) {
    bytes[i] = (size_t)arr[i].planes * arr[i].row * arr[i].esize;
    if (arr[i].host || arr[i].scratch) CK(D->slot[i].reserve((size_t)ch.slots * ch.chunk * bytes[i]));
  }
  auto slot = [&](size_t i, int c) -> void* {
    if (!arr[i].host && !arr[i].scratch) return nullptr;
    return (char*)D->slot[i].p + (size_t)(c % 3) * ch.chunk * bytes[i];
  };
  auto span = [&](int c, long long* first, long long* m) {
    *first = (long long)c * ch.chunk;
    *m = (n - *first) < ch.chunk ? (n - *first) : ch.chunk;
    *first += lo;
  };
  auto copies = [&](int c, int dir, cudaStream_t st) -> int {
    long long first, m;
    span(c, &first, &m);
    for (size_t i = 0; i < NA; i++)
      if (arr[i].host && (arr[i].dir & dir))
        CK(copy_chunk(arr[i], slot(i, c), ld, first, m, dir == IN ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, st));
    return F16_OK;
  };
  auto fetch = [&](int c) -> int {
    if (c >= 3) CK(cudaStreamWaitEvent(D->s_in, D->e_out[c % 3], 0));  // the slot is free once its previous result has left
    const int rc = copies(c, IN, D->s_in);
    if (rc != F16_OK) return rc;
    CK(cudaEventRecord(D->e_in[c % 3], D->s_in));
    return F16_OK;
  };
  auto run = [&](int c) -> int {
    long long first, m;
    span(c, &first, &m);
    Slots p;
    for (size_t i = 0; i < NA; i++) p.p[i] = slot(i, c);
    CK(cudaStreamWaitEvent(D->stream, D->e_in[c % 3], 0));
    const int rc = work(p, m);
    if (rc != F16_OK) return rc;
    CK(cudaEventRecord(D->e_work[c % 3], D->stream));
    return F16_OK;
  };
  auto flush = [&](int c) -> int {
    CK(cudaStreamWaitEvent(D->s_out, D->e_work[c % 3], 0));
    const int rc = copies(c, OUT, D->s_out);
    if (rc != F16_OK) return rc;
    CK(cudaEventRecord(D->e_out[c % 3], D->s_out));
    return F16_OK;
  };
  int rc = F16_OK;
  if (work_blocks) {
    rc = fetch(0);
    for (int c = 0; c < ch.count && rc == F16_OK; c++) {
      if (c + 1 < ch.count) rc = fetch(c + 1);  // slot (c + 1) mod 3 held chunk c - 2, flushed one iteration ago
      if (rc == F16_OK && c >= 1) rc = flush(c - 1);
      if (rc == F16_OK) rc = run(c);
    }
  } else {
    for (int c = 0; c < ch.count && rc == F16_OK; c++) {
      rc = fetch(c);
      if (rc == F16_OK) rc = run(c);
      if (rc == F16_OK && c >= 1) rc = flush(c - 1);
    }
  }
  if (rc == F16_OK) rc = flush(ch.count - 1);
  // drain all three streams whatever happened: the caller's buffers must not be touched after the call returns
  const cudaError_t e0 = cudaStreamSynchronize(D->s_in), e1 = cudaStreamSynchronize(D->stream), e2 = cudaStreamSynchronize(D->s_out);
  if (rc != F16_OK) return rc;
  CK(e0);
  CK(e1);
  CK(e2);
  return F16_OK;
}

// ---- one call over several devices ------------------------------------------------------------------------------------
// Aircraft are independent: the batch is cut into contiguous slices, one per device context (boundaries on multiples of 32
// aircraft), and every slice runs the single-device path on its own context from its own host thread -- copies and kernels of
// the slices overlap, nothing is exchanged between devices (SURVEY 8e: no collective on the data path).  A batch too small to
// feed more than one device stays on the current context.
struct Span {
  long long lo, n;
};
struct Spans {
  int count = 0;
  Span at[kMaxContexts];
};
Spans device_spans(long long N, long long min_per_device, long long contexts) {
  long long parts = contexts;
  if (min_per_device > 0 && N / min_per_device < parts) parts = N / min_per_device;
  if (parts < 1) parts = 1;
  Spans v;
  const long long groups = (N + 31) / 32;
  long long g0 = 0;
  for (long long i = 0; i < parts; i++) {
    const long long g1 = groups * (i + 1) / parts;
    const long long lo = g0 * 32, hi = g1 * 32 < N ? g1 * 32 : N;
    if (hi > lo) v.at[v.count++] = Span{lo, hi - lo};
    g0 = g1;
  }
  return v;
}
// the slices of a call over the library's contexts (N >= 1)
Spans slices(long long N, long long min_per_device) { return device_spans(N, min_per_device, (long long)G.devs.size()); }

// f(i, lo, n) for every slice i, with D set to context i (one slice: the current context, on the calling thread)
template <class F>
int on_devices(const Spans& spans, F f) {
  if (spans.count <= 1) return f(0, spans.at[0].lo, spans.at[0].n);
  try {
    std::vector<int> rcs(spans.count, F16_OK);
    std::vector<std::string> errs(spans.count);
    std::vector<std::thread> workers;
    auto body = [&](int i) {
      D = G.devs[i].get();
      if (cudaSetDevice(D->ordinal) != cudaSuccess) {
        set_err("cudaSetDevice(%d) failed", D->ordinal);
        rcs[i] = F16_ERR_CUDA;
      } else {
        rcs[i] = f(i, spans.at[i].lo, spans.at[i].n);
      }
      errs[i] = t_err;
    };
    Dev* mine = D;
    int started = 1;
    try {
      for (; started < spans.count; started++) workers.emplace_back(body, started);
    } catch (...) {  // no more threads: the calling thread takes the remaining slices one after the other
    }
    body(0);
    for (int i = started; i < spans.count; i++) body(i);
    for (std::thread& w : workers) w.join();
    D = mine;
    cudaSetDevice(D->ordinal);
    for (int i = 0; i < spans.count; i++)
      if (rcs[i] != F16_OK) {
        set_err("device context %d (cuda:%d): %s", i, G.devs[i]->ordinal, errs[i].c_str());
        return rcs[i];
      }
    return F16_OK;
  } catch (const std::exception& e) {
    set_err("host resources: %s", e.what());
    return F16_ERR_HOST;
  }
}

// Chan et al. update of two summary rows [N, alive, min[18], max[18], mean[18], M2[18]] (f16_stats.cu): a += b
void merge_summary_row(double* a, const double* b) {
  const double na = a[1], nb = b[1], nt = na + nb;
  a[0] += b[0];
  a[1] = nt;
  for (int i = 0; i < 18; i++) {
    a[2 + i] = b[2 + i] < a[2 + i] ? b[2 + i] : a[2 + i];
    a[20 + i] = b[20 + i] > a[20 + i] ? b[20 + i] : a[20 + i];
    if (nb > 0) {
      const double d = b[38 + i] - a[38 + i];
      a[38 + i] = a[38 + i] + d * (nb / nt);
      a[56 + i] = a[56 + i] + b[56 + i] + d * d * (na * nb / nt);
    }
  }
}

// K steps in launches of snap_every back to back on D->stream (step_batch is restartable bit for bit at any step boundary),
// snap(j) after the j-th full launch
template <class Snap>
int snapshot_steps(double* d_x, long long ld_x, const double* d_u, long long ld_u, long long N, int K, int snap_every,
                          double dt, const f16_lqr_t* lqr, const f16::BatchSel& sel, int* d_status, Snap snap) {
  const bool smem = G.smem_tables && (N * (long long)snap_every >= 4096);
  for (int done = 0, j = 0; done < K;) {
    const int k = (K - done) < snap_every ? (K - done) : snap_every;
    CK(run_step(cfg(smem), sel, d_x, ld_x, d_u, ld_u, N, k, dt, reinterpret_cast<const f16::LqrLaw*>(lqr), d_status, nullptr));
    done += k;
    if (k == snap_every) {
      const int rc = snap(j++);
      if (rc != F16_OK) return rc;
    }
  }
  return F16_OK;
}

// Statistics of a batch sliced over the device contexts: f(lo, n, rows) writes the n_rows summary rows of aircraft [lo, lo + n)
// on its context; the rows of the slices are combined on the host (Chan's update, slice order).  N >= 1.
template <class F>
int merged_rows(long long N, long long min_per_device, int n_rows, double* rows, F f) {
  try {
    const Spans spans = slices(N, min_per_device);
    const size_t per = (size_t)n_rows * 74;
    std::vector<double> part(spans.count * per);
    const int rc = on_devices(spans, [&](int i, long long lo, long long n) { return f(lo, n, part.data() + i * per); });
    if (rc != F16_OK) return rc;
    for (int r = 0; r < n_rows; r++) {
      double* dst = rows + (size_t)r * 74;
      memcpy(dst, part.data() + (size_t)r * 74, 74 * 8);
      for (int i = 1; i < spans.count; i++) merge_summary_row(dst, part.data() + i * per + (size_t)r * 74);
    }
    return F16_OK;
  } catch (const std::exception& e) {
    set_err("host resources: %s", e.what());
    return F16_ERR_HOST;
  }
}

}  // namespace

extern "C" {
#pragma GCC visibility push(default)

int f16_init(const char* table_path, int device) {
  std::lock_guard<std::mutex> lk(G_mu);
  return init_locked(table_path, device, nullptr, 0);
}

int f16_init_devices(const char* table_path, const int* devices, int ndev) {
  std::lock_guard<std::mutex> lk(G_mu);
  if (G.ready) {  // idempotent for the same list; a different list needs f16_shutdown first
    std::vector<int> want;
    int present = 0;
    if (devices && ndev > 0) want.assign(devices, devices + ndev);
    else if (cudaGetDeviceCount(&present) == cudaSuccess)
      for (int i = 0; i < present; i++) want.push_back(i);
    bool same = want.size() == G.devs.size();
    for (size_t i = 0; same && i < want.size(); i++) same = want[i] == G.devs[i]->ordinal;
    if (same) return F16_OK;
    set_err("f16_init_devices: the library is already initialised on another device list (f16_shutdown first)");
    return F16_ERR_ARG;
  }
  return init_locked(table_path, -1, devices, devices && ndev > 0 ? ndev : -1);
}

void f16_shutdown(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  G.devs.clear();
  D = nullptr;
  G.ready = false;
  G.init_rc = F16_ERR_NOINIT;
  G.cur = 0;
  G.payload.clear();
  G.table_source.clear();
}

// host logic only (no CUDA call): how a host-buffer batch call would cut N aircraft over `contexts` device contexts and, on one
// context, into pipeline chunks.  lo_n [2 * contexts] = (first aircraft, count) per slice; returns the number of slices used.
int f16_plan_slices(long long N, long long min_per_device, int contexts, long long* lo_n) {
  if (N < 0 || contexts < 1 || contexts > kMaxContexts || !lo_n) return F16_ERR_ARG;
  if (N == 0) return 0;
  const Spans v = device_spans(N, min_per_device, contexts);
  for (int i = 0; i < v.count; i++) {
    lo_n[2 * i] = v.at[i].lo;
    lo_n[2 * i + 1] = v.at[i].n;
  }
  return v.count;
}
int f16_plan_chunks(long long n, long long min_chunk, int max_chunks, long long* chunk, int* slots) {
  if (n < 1 || min_chunk < 1 || max_chunks < 1 || !chunk || !slots) return F16_ERR_ARG;
  const Chunks c = plan_chunks(n, min_chunk, max_chunks);
  *chunk = c.chunk;
  *slots = c.slots;
  return c.count;
}

int f16_device_count(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  return G.ready ? (int)G.devs.size() : 0;
}

int f16_use_device(int index) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (index < 0 || index >= (int)G.devs.size()) { set_err("f16_use_device: index %d out of range (%d contexts)", index, (int)G.devs.size()); return F16_ERR_ARG; }
  const int prev = G.cur;
  G.cur = index;
  return ensure() == F16_OK ? prev : F16_ERR_CUDA;
}

const char* f16_last_error(void) { return t_err.c_str(); }
int f16_last_status(void) { return G.last_status.load(); }
int f16_device(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  return G.ready ? G.devs[(size_t)G.cur]->ordinal : -1;
}
int f16_sm_count(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  return G.ready ? G.devs[(size_t)G.cur]->sm_count : 0;
}
unsigned long long f16_launch_count(void) {  // kernels launched since init, all contexts
  std::lock_guard<std::mutex> lk(G_mu);
  unsigned long long n = 0;
  for (auto& d : G.devs) n += d->launches;
  return n;
}
void* f16_stream(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  return G.ready ? (void*)G.devs[(size_t)G.cur]->stream : nullptr;
}

int f16_set_math_mode(int mode) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.math_mode;
  G.math_mode = mode == F16_MATH_FAST ? F16_MATH_FAST : F16_MATH_STRICT;
  return prev;
}

int f16_set_clr_mode(int mode) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  int prev = G.clr_mode;
  G.clr_mode = mode == F16_CLR_FROM_FILE ? F16_CLR_FROM_FILE : F16_CLR_AS_BUILT;
  if (G.clr_mode != prev) {
    for (auto& d : G.devs) {  // the table images of every context
      D = d.get();
      CK(cudaSetDevice(D->ordinal));
      CK(cudaStreamSynchronize(D->stream));
      if ((rc = upload_tables()) != F16_OK) break;
    }
    const int back = ensure();
    if (rc != F16_OK) return rc;
    if (back != F16_OK) return back;
  }
  return prev;
}

void f16_set_default_xcg(double xcg) { G.default_xcg.store(xcg); }

int f16_set_table_staging(int mode) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.smem_tables ? 1 : 0;
  G.smem_tables = mode != 0;
  return prev;
}

int f16_set_step_chunking(int on) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.step_chunking ? 1 : 0;
  G.step_chunking = on != 0;
  return prev;
}

int f16_set_trim_fixed_point_exit(int on) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.trim_fp_exit ? 1 : 0;
  G.trim_fp_exit = on != 0;
  return prev;
}

int f16_set_step_compaction(int on) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.compaction ? 1 : 0;
  G.compaction = on != 0;
  return prev;
}

int f16_set_host_pipeline(int on) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.host_pipeline ? 1 : 0;
  G.host_pipeline = on != 0;
  return prev;
}

int f16_set_linearise_variant(int variant) {
  std::lock_guard<std::mutex> lk(G_mu);
  int prev = G.lin_variant;
  G.lin_variant = (variant == 1 || variant == 2) ? variant : 0;
  return prev;
}

int f16_tables_sha256(char* out65) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  f16::payload_sha256_hex(G.payload, out65);
  return F16_OK;
}

// ---- legacy reference ABI -------------------------------------------------------------------------------
void f16_nlplant_xcg(const double* xu, double* xdot, int fidelity, double xcg) {
  std::lock_guard<std::mutex> lk(G_mu);
  const double nan = __builtin_nan("");
  if (ensure() != F16_OK) {
    for (int i = 0; i < 18; i++) xdot[i] = nan;
    G.last_status = F16_ST_NAN;
    fprintf(stderr, "libf16_b200: Nlplant: %s\n", t_err.c_str());
    return;
  }
  memcpy(D->pin, xu, 17 * sizeof(double));
  int* st_host = reinterpret_cast<int*>(D->pin + 40);
  int* st_dev = reinterpret_cast<int*>(D->pin_dev + 40);
  // one aircraft: tables read through L2 (no 105 KB staging), inputs and outputs in mapped pinned memory
  cudaError_t e = f16::strict::launch_nlplant(cfg(false), tabs(), sel_of(nullptr, fidelity, nullptr, xcg), D->pin_dev, 1,
                                              D->pin_dev + 17, 1, 1, st_dev);
  if (e == cudaSuccess) e = cudaStreamSynchronize(D->stream);
  if (e != cudaSuccess) {
    cuda_fail(e, "Nlplant");
    fprintf(stderr, "libf16_b200: Nlplant: %s\n", t_err.c_str());
    for (int i = 0; i < 18; i++) xdot[i] = nan;
    G.last_status = F16_ST_NAN;
    return;
  }
  memcpy(xdot, D->pin + 17, 18 * sizeof(double));
  G.last_status = *st_host;
}

void Nlplant(double* xu, double* xdot, int fidelity) { f16_nlplant_xcg(xu, xdot, fidelity, G.default_xcg.load()); }

void atmos(double alt, double vt, double* coeff) { f16_atmos(alt, vt, coeff); }

void f16_atmos(double alt, double vt, double* coeff) {
  std::lock_guard<std::mutex> lk(G_mu);
  const double nan = __builtin_nan("");
  coeff[0] = coeff[1] = coeff[2] = nan;
  if (ensure() != F16_OK) {
    fprintf(stderr, "libf16_b200: atmos: %s\n", t_err.c_str());
    return;
  }
  D->pin[48] = alt;
  D->pin[49] = vt;
  cudaError_t e = f16::strict::launch_atmos(cfg(false), D->pin_dev + 48, D->pin_dev + 49, 1, D->pin_dev + 50);
  if (e == cudaSuccess) e = cudaStreamSynchronize(D->stream);
  if (e != cudaSuccess) {
    cuda_fail(e, "atmos");
    fprintf(stderr, "libf16_b200: atmos: %s\n", t_err.c_str());
    return;
  }
  coeff[0] = D->pin[50];
  coeff[1] = D->pin[51];
  coeff[2] = D->pin[52];
}

// ---- device-pointer entry points ---------------------------------------------------------------------------
int Nlplant_batch_dev(const double* xu_soa, long long ld_in, double* xdot_soa, long long ld_out, const unsigned char* fi,
                      int fi_default, const double* xcg, double xcg_default, long long N, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!nlplant_ok(xu_soa, ld_in, xdot_soa, ld_out, N)) return bad_arg("Nlplant_batch_dev");
  CK(run_xdot(sel_of(fi, fi_default, xcg, xcg_default), xu_soa, ld_in, nullptr, 0, xdot_soa, ld_out, N, status));
  return F16_OK;
}

int calc_xdot_batch_dev(const double* x_soa, long long ld_x, const double* u_soa, long long ld_u, double* xdot_soa,
                        long long ld_out, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default,
                        long long N, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!calc_xdot_ok(x_soa, ld_x, u_soa, ld_u, xdot_soa, ld_out, N)) return bad_arg("calc_xdot_batch_dev");
  CK(run_xdot(sel_of(fi, fi_default, xcg, xcg_default), x_soa, ld_x, u_soa, ld_u, xdot_soa, ld_out, N, status));
  return F16_OK;
}

// scratch of the time-chunked step schedule (one int per 32 aircraft); without it the launch falls back to the plain kernel
static void reserve_step_progress(long long N) {
  if (G.step_chunking && N > 0 && D->b_prog.reserve((size_t)((N + 31) / 32) * 4) != cudaSuccess) cudaGetLastError();
}

// A mixed batch (per-aircraft fidelity flags) for the fused step: ordered by fidelity first, so that each of the two launches
// runs on a contiguous range with every lane busy (f16_partition.cu; SURVEY 8e).  Applies when the reorder is amortised
// (N >= 4096 aircraft, K >= 8 steps); *handled = false leaves the call to the caller's direct launch -- with *uniform = the one
// fidelity every flag names when the "mixed" batch turns out not to be mixed (no gather, no scatter, no second copy).
static int step_partitioned(double* d_x, long long ld_x, const double* d_u, long long ld_u, long long N, int K, double dt,
                            const f16_lqr_t* lqr, const unsigned char* d_fi, const double* d_xcg, double xcg_default,
                            int* d_status, int* d_steps, bool* handled, int* uniform) {
  *handled = false;
  *uniform = -1;
  if (!d_fi || N < 4096 || K < 8 || N >= (1LL << 31)) return F16_OK;
  const size_t n = (size_t)N;
  const int n_cta = f16::partition::n_cta(N);
  if (D->b_perm.reserve(n * 4) != cudaSuccess || D->b_pscr.reserve((size_t)n_cta * 6 * 4 + 64) != cudaSuccess) {
    cudaGetLastError();
    return F16_OK;
  }
  const f16::LaunchCfg c = cfg(G.smem_tables);
  unsigned* perm = (unsigned*)D->b_perm.p;
  unsigned* scr = (unsigned*)D->b_pscr.p;
  long long* totals_dev = (long long*)(scr + (size_t)n_cta * 6 + 2);  // 8-byte aligned: n_cta * 24 + 8 bytes in
  CK(f16::partition::launch_build(c, d_fi, N, perm, totals_dev, scr));
  long long* tot = reinterpret_cast<long long*>(D->pin + 56);  // pinned: the copy is asynchronous, the wait below is the only one
  CK(cudaMemcpyAsync(tot, totals_dev, 3 * sizeof(long long), cudaMemcpyDeviceToHost, D->stream));
  CK(cudaStreamSynchronize(D->stream));
  const long long n1 = tot[0], n0 = tot[1], nbad = tot[2];
  if (n1 == N || n0 == N) {
    *uniform = n1 == N ? 1 : 0;
    return F16_OK;
  }
  // scratch for the reordered copy is optional: when the device cannot hold it the masked path does the job
  if (D->b_px.reserve(18 * n * 8) != cudaSuccess || D->b_pu.reserve(4 * n * 8) != cudaSuccess ||
      D->b_pst.reserve(n * 4) != cudaSuccess || D->b_pk.reserve(n * 4) != cudaSuccess ||
      (d_xcg && D->b_pxcg.reserve(n * 8) != cudaSuccess)) {
    cudaGetLastError();
    return F16_OK;
  }
  double* px = (double*)D->b_px.p;
  double* pu = (double*)D->b_pu.p;
  double* pxcg = d_xcg ? (double*)D->b_pxcg.p : nullptr;
  int* pst = (int*)D->b_pst.p;
  int* pk = (int*)D->b_pk.p;
  CK(f16::partition::launch_gather_f64(c, d_x, ld_x, px, N, 18, perm, N));
  CK(f16::partition::launch_gather_f64(c, d_u, ld_u, pu, N, 4, perm, N));
  if (d_xcg) CK(f16::partition::launch_gather_f64(c, d_xcg, N, pxcg, N, 1, perm, N));
  const f16::LqrLaw* law = reinterpret_cast<const f16::LqrLaw*>(lqr);
  if (n1 > 0)
    CK(run_step(c, sel_of(nullptr, 1, pxcg, xcg_default), px, N, pu, N, n1, K, dt, law, pst, pk));
  if (n0 > 0)
    CK(run_step(c, sel_of(nullptr, 0, pxcg ? pxcg + n1 : nullptr, xcg_default), px + n1, N, pu + n1, N, n0, K, dt, law, pst + n1,
                pk + n1));
  if (nbad > 0) {  // neither model: the state stays as it is, status = F16_ST_FIDELITY, no step taken
    CK(f16::partition::launch_fill_i32(c, pst + n1 + n0, (int)F16_ST_FIDELITY, nbad));
    CK(cudaMemsetAsync(pk + n1 + n0, 0, (size_t)nbad * 4, D->stream));
  }
  CK(f16::partition::launch_scatter_f64(c, px, N, d_x, ld_x, 18, perm, N));
  if (d_status) CK(f16::partition::launch_scatter_i32(c, pst, d_status, perm, N));
  if (d_steps) CK(f16::partition::launch_scatter_i32(c, pk, d_steps, perm, N));
  *handled = true;
  return F16_OK;
}

static int step_on_device(double* d_x, long long ld_x, const double* d_u, long long ld_u, long long n, int K, double dt,
                          const f16_lqr_t* lqr, const unsigned char* d_fi, int fi_default, const double* d_xcg, double xcg_default,
                          int* d_st, int* d_k);

int step_batch_dev(double* x_soa, long long ld_x, const double* u_soa, long long ld_u, long long N, int K, double dt,
                   const f16_lqr_t* lqr, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default,
                   int* status, int* steps_done) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!step_ok(x_soa, ld_x, u_soa, ld_u, N, K, lqr)) return bad_arg("step_batch_dev");
  reserve_step_progress(N);
  return step_on_device(x_soa, ld_x, u_soa, ld_u, N, K, dt, lqr, fi, fi_default, xcg, xcg_default, status, steps_done);
}

int linearise_batch_dev(const double* x_soa, long long ld_x, const double* u_soa, long long ld_u, long long N, double eps,
                        int scheme, double* A, double* B, const unsigned char* fi, int fi_default, const double* xcg,
                        double xcg_default, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!linearise_ok(x_soa, ld_x, u_soa, ld_u, N, eps, scheme, A, B)) return bad_arg("linearise_batch_dev");
  CK(run_linearise(sel_of(fi, fi_default, xcg, xcg_default), x_soa, ld_x, u_soa, ld_u, N, eps, scheme, A, B, status));
  return F16_OK;
}

// ---- host-pointer entry points: slices over the device contexts, a chunk pipeline on each -------------------------------
// The arrays of a call are listed in a fixed order; its work() finds the device slot of array i at p.*(i).

// Nlplant_batch (u == NULL: x is xu [17][ld]) / calc_xdot_batch for aircraft [lo, lo + n) of the caller's arrays on the context D
static int xdot_host(const double* x, const double* u, double* xdot, long long ld, long long lo, long long n, const unsigned char* fi,
                     int fi_default, const double* xcg, double xcg_default, int* status) {
  return run_pipeline({soa(x, IN, 8, u ? 18 : 17), soa(u, IN, 8, 4), soa(fi, IN, 1), soa(xcg, IN, 8), soa(xdot, OUT, 8, 18),
                       soa(status, OUT, 4, 1, true)},
                      ld, lo, n, plan_chunks(n, 1 << 16, 8), false, [&](const Slots& p, long long m) -> int {
                        CK(run_xdot(sel_of(p.u8(2), fi_default, p.f64(3), xcg_default), p.f64(0), m, p.f64(1), u ? m : 0, p.f64(4),
                                    m, m, p.i32(5)));
                        return F16_OK;
                      });
}

int Nlplant_batch(const double* xu_soa, double* xdot_soa, const unsigned char* fi, int fi_default, const double* xcg,
                  double xcg_default, long long N, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!nlplant_ok(xu_soa, N, xdot_soa, N, N)) return bad_arg("Nlplant_batch");
  if (N == 0) return F16_OK;
  return on_devices(slices(N, 16384), [&](int, long long lo, long long n) {
    return xdot_host(xu_soa, nullptr, xdot_soa, N, lo, n, fi, fi_default, xcg, xcg_default, status);
  });
}

int calc_xdot_batch(const double* x_soa, const double* u_soa, double* xdot_soa, const unsigned char* fi, int fi_default,
                    const double* xcg, double xcg_default, long long N, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!calc_xdot_ok(x_soa, N, u_soa, N, xdot_soa, N, N)) return bad_arg("calc_xdot_batch");
  if (N == 0) return F16_OK;
  return on_devices(slices(N, 16384), [&](int, long long lo, long long n) {
    return xdot_host(x_soa, u_soa, xdot_soa, N, lo, n, fi, fi_default, xcg, xcg_default, status);
  });
}

// A Monte-Carlo run with casualties (BASELINE cfg 5 without the regulator; xcg 0.35 open loop loses half of a +-5 % batch within
// 10 s).  An aircraft that leaves the envelope is frozen and keeps its lane; deaths are scattered, so nearly every warp keeps a
// survivor and runs all K steps: the launch lasts as long as if nobody had died.  Here a long run is cut into eight chunks of
// steps (step_batch is restartable bit for bit at any step boundary); after a chunk the survivors are counted, and once more
// than 1/16 of the active lanes idle, the active set is reordered -- survivors first (stable partition of f16_partition.cu on
// the status words, gather of the 23 planes), the newly stopped aircraft scattered to their final place in the caller's arrays
// -- and the next chunk runs on the survivors only, in full warps.  Per-aircraft results are the same bits as one launch of K
// steps.  Without casualties the cost is the chunking (the launches drain and refill the GPU): chunks double while nobody is
// lost, three extra launches for a clean 10^4-step run.  Opt-in: f16_set_step_compaction(1).
static int step_compacting(double* d_x, long long ld_x, const double* d_u, long long ld_u, long long N, int K, double dt,
                           const f16_lqr_t* lqr, int fi, const double* d_xcg, double xcg_default, int* d_st, int* d_k, bool smem) {
  const size_t n = (size_t)N;
  const int n_cta = f16::partition::n_cta(N);
  CK(D->b_ckl.reserve(n * 4));
  CK(D->b_cflag.reserve(n));
  CK(D->b_perm.reserve(n * 4));
  CK(D->b_pscr.reserve((size_t)n_cta * 6 * 4 + 64));
  if (!d_k) CK(D->b_pk.reserve(n * 4));  // the step counts are kept even when the caller does not ask for them
  int* kl = (int*)D->b_ckl.p;
  unsigned char* flag = (unsigned char*)D->b_cflag.p;
  unsigned* perm = (unsigned*)D->b_perm.p;
  unsigned* scr = (unsigned*)D->b_pscr.p;
  long long* totals_dev = (long long*)(scr + (size_t)n_cta * 6 + 2);
  long long* tot = reinterpret_cast<long long*>(D->pin + 56);
  const f16::LqrLaw* law = reinterpret_cast<const f16::LqrLaw*>(lqr);
  const f16::LaunchCfg c = cfg(smem);

  // the working view: the caller's arrays until the first reorder, then one of the two scratch sets
  double* x = d_x;
  const double* u = d_u;
  const double* xcg = d_xcg;
  long long ldx = ld_x, ldu = ld_u;
  int* st = d_st;
  int* ktot = d_k ? d_k : (int*)D->b_pk.p;
  const unsigned* orig = nullptr;  // working slot -> aircraft index (identity while on the caller's arrays)
  int set = -1;
  long long n_act = N;
  CK(cudaMemsetAsync(ktot, 0xff, n * 4, D->stream));  // -1: still flying
  // chunks of K / 8 steps while aircraft are being lost; every chunk that loses nobody doubles the next one
  const int chunk0 = (K + 7) / 8;
  int chunk = chunk0, base = 0;
  long long idle_before = 0;  // stopped aircraft still inside the active set
  while (base < K) {
    const int kc = (K - base) < chunk ? (K - base) : chunk;
    CK(run_step(c, sel_of(nullptr, fi, xcg, xcg_default), x, ldx, u, ldu, n_act, kc, dt, law, st, kl));
    CK(f16::partition::launch_mark_survivors(c, st, kl, ktot, base, n_act, flag));
    base += kc;
    if (base >= K) break;
    CK(f16::partition::launch_build(c, flag, n_act, perm, totals_dev, scr));
    CK(cudaMemcpyAsync(tot, totals_dev, 3 * sizeof(long long), cudaMemcpyDeviceToHost, D->stream));
    CK(cudaStreamSynchronize(D->stream));
    const long long n_alive = tot[0], n_dead = n_act - n_alive;
    if (n_alive == 0) break;
    chunk = n_dead == idle_before ? (chunk < K ? 2 * chunk : chunk) : chunk0;
    idle_before = n_dead;
    if (n_dead * 16 < n_act) continue;  // fewer than 1/16 of the active lanes idle: not worth a reorder yet
    idle_before = 0;
    const int nx = set < 0 ? 0 : 1 - set;
    const size_t m = (size_t)n_act;
    CK(D->b_cx[nx].reserve(18 * m * 8));
    CK(D->b_cu[nx].reserve(4 * m * 8));
    CK(D->b_cst[nx].reserve(m * 4));
    CK(D->b_co[nx].reserve(m * 4));
    if (d_xcg) CK(D->b_cxcg[nx].reserve(m * 8));
    CK(D->b_ck[nx].reserve(m * 4));
    double* xn = (double*)D->b_cx[nx].p;
    double* un = (double*)D->b_cu[nx].p;
    int* stn = (int*)D->b_cst[nx].p;
    int* kn = (int*)D->b_ck[nx].p;
    unsigned* on = (unsigned*)D->b_co[nx].p;
    CK(f16::partition::launch_gather_f64(c, x, ldx, xn, n_act, 18, perm, n_act));
    CK(f16::partition::launch_gather_f64(c, u, ldu, un, n_act, 4, perm, n_act));
    if (d_xcg) CK(f16::partition::launch_gather_f64(c, xcg, n_act, (double*)D->b_cxcg[nx].p, n_act, 1, perm, n_act));
    CK(f16::partition::launch_gather_i32(c, st, stn, perm, n_act));
    CK(f16::partition::launch_gather_i32(c, ktot, kn, perm, n_act));
    if (orig) CK(f16::partition::launch_gather_i32(c, (const int*)orig, (int*)on, perm, n_act));
    else CK(cudaMemcpyAsync(on, perm, m * 4, cudaMemcpyDeviceToDevice, D->stream));
    // the aircraft that stopped since the last reorder sit in [n_alive, n_act): they go to their final place now
    CK(f16::partition::launch_scatter_f64(c, xn + n_alive, n_act, d_x, ld_x, 18, on + n_alive, n_dead));
    CK(f16::partition::launch_scatter_i32(c, stn + n_alive, d_st, on + n_alive, n_dead));
    if (d_k) CK(f16::partition::launch_scatter_i32(c, kn + n_alive, d_k, on + n_alive, n_dead));
    x = xn; ldx = n_act;
    u = un; ldu = n_act;
    xcg = d_xcg ? (const double*)D->b_cxcg[nx].p : nullptr;
    st = stn;
    ktot = kn;
    orig = on;
    set = nx;
    n_act = n_alive;
  }
  // the end: whoever never stopped has taken all K steps; a reordered working set goes back to the caller's arrays
  CK(f16::partition::launch_close_steps(c, ktot, K, n_act));
  if (set >= 0) {
    CK(f16::partition::launch_scatter_f64(c, x, ldx, d_x, ld_x, 18, orig, n_act));
    CK(f16::partition::launch_scatter_i32(c, st, d_st, orig, n_act));
    if (d_k) CK(f16::partition::launch_scatter_i32(c, ktot, d_k, orig, n_act));
  }
  return F16_OK;
}

// the fused step on device arrays of the context D: mixed batches through the fidelity partition, the rest directly; tables go
// to shared memory whenever the launch does real work, a handful of aircraft-steps read them via L2
static int step_on_device(double* d_x, long long ld_x, const double* d_u, long long ld_u, long long n, int K, double dt,
                          const f16_lqr_t* lqr, const unsigned char* d_fi, int fi_default, const double* d_xcg, double xcg_default,
                          int* d_st, int* d_k) {
  int uniform = -1;
  bool handled = false;
  int rc = step_partitioned(d_x, ld_x, d_u, ld_u, n, K, dt, lqr, d_fi, d_xcg, xcg_default, d_st, d_k, &handled, &uniform);
  if (rc != F16_OK || handled) return rc;
  if (uniform >= 0) { d_fi = nullptr; fi_default = uniform; }  // every flag says the same: no partition, no per-lane masking
  const bool smem = G.smem_tables && (n * (long long)(K > 0 ? K : 1) >= 4096);
  if (G.compaction && !d_fi && d_st && K >= 4096 && n >= 65536 && n < (1LL << 31) && (fi_default == 0 || fi_default == 1))
    return step_compacting(d_x, ld_x, d_u, ld_u, n, K, dt, lqr, fi_default, d_xcg, xcg_default, d_st, d_k, smem);
  CK(run_step(cfg(smem), sel_of(d_fi, fi_default, d_xcg, xcg_default), d_x, ld_x, d_u, ld_u, n, K, dt,
              reinterpret_cast<const f16::LqrLaw*>(lqr), d_st, d_k));
  return F16_OK;
}

// step_batch for aircraft [lo, lo + n) of the caller's arrays on the context D.  A long run (K >= 512) is cut into at most four
// chunks of >= 2^18 aircraft (the time-chunked schedule of the step kernel wants many rounds of warp-tasks per launch); a short
// one, which is copy-bound, into up to eight of >= 2^16.  The kernels always get status and step-count slots: step_compacting
// needs the status words.
static int step_host(double* x, const double* u, long long ld, long long lo, long long n, int K, double dt, const f16_lqr_t* lqr,
                     const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, int* status, int* steps_done) {
  const Chunks ch = K >= 512 ? plan_chunks(n, 1 << 18, 4) : plan_chunks(n, 1 << 16, 8);
  reserve_step_progress(ch.chunk);
  return run_pipeline({soa(x, INOUT, 8, 18), soa(u, IN, 8, 4), soa(fi, IN, 1), soa(xcg, IN, 8), soa(status, OUT, 4, 1, true),
                       soa(steps_done, OUT, 4, 1, true)},
                      ld, lo, n, ch, G.compaction && K >= 4096, [&](const Slots& p, long long m) {
                        return step_on_device(p.f64(0), m, p.f64(1), m, m, K, dt, lqr, p.u8(2), fi_default, p.f64(3), xcg_default,
                                              p.i32(4), p.i32(5));
                      });
}

int step_batch(double* x_soa, const double* u_soa, long long N, int K, double dt, const f16_lqr_t* lqr,
               const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, int* status,
               int* steps_done) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!step_ok(x_soa, N, u_soa, N, N, K, lqr)) return bad_arg("step_batch");
  if (N == 0) return F16_OK;
  return on_devices(slices(N, 16384), [&](int, long long lo, long long n) {
    return step_host(x_soa, u_soa, N, lo, n, K, dt, lqr, fi, fi_default, xcg, xcg_default, status, steps_done);
  });
}

// K Euler steps with a snapshot of the whole state every `snap_every` steps: traj [K / snap_every][18][N], each snapshot copied
// out of one of two device slots while the next launch runs.  Aircraft [lo, lo + n) of the caller's arrays on the context D.
static int traj_host(double* x, const double* u, long long ld, long long lo, long long n, int K, int snap_every, double dt,
                     const f16_lqr_t* lqr, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default,
                     double* traj, int* status) {
  CK(D->b_snap.reserve(2 * 18 * (size_t)n * 8));
  reserve_step_progress(n);
  return run_pipeline(
      {soa(x, INOUT, 8, 18), soa(u, IN, 8, 4), soa(fi, IN, 1), soa(xcg, IN, 8), soa(status, OUT, 4, 1, true)}, ld, lo, n,
      one_chunk(n), false, [&](const Slots& p, long long m) {
        const f16::BatchSel sel = sel_of(p.u8(2), fi_default, p.f64(3), xcg_default);
        return snapshot_steps(p.f64(0), m, p.f64(1), m, m, K, snap_every, dt, lqr, sel, p.i32(4), [&](int j) -> int {
          double* snap = (double*)D->b_snap.p + (size_t)(j & 1) * 18 * m;
          // the slot's previous copy-out (two snapshots ago, on s_out) has completed before this copy overwrites it
          if (j >= 2) CK(cudaStreamWaitEvent(D->stream, D->e_snap_out[j & 1], 0));
          CK(cudaMemcpyAsync(snap, p.f64(0), 18 * (size_t)m * 8, cudaMemcpyDeviceToDevice, D->stream));
          CK(cudaEventRecord(D->e_snap[j & 1], D->stream));
          CK(cudaStreamWaitEvent(D->s_out, D->e_snap[j & 1], 0));
          CK(copy_chunk(soa(traj + (size_t)j * 18 * ld, OUT, 8, 18), snap, ld, lo, m, cudaMemcpyDeviceToHost, D->s_out));
          CK(cudaEventRecord(D->e_snap_out[j & 1], D->s_out));
          return F16_OK;
        });
      });
}

int step_batch_traj(double* x_soa, const double* u_soa, long long N, int K, int snap_every, double dt, const f16_lqr_t* lqr,
                    const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, double* traj, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!step_ok(x_soa, N, u_soa, N, N, K, lqr) || snap_every < 1 || (N > 0 && !traj && K >= snap_every)) return bad_arg("step_batch_traj");
  if (N == 0) return F16_OK;
  return on_devices(slices(N, 16384), [&](int, long long lo, long long n) {
    return traj_host(x_soa, u_soa, N, lo, n, K, snap_every, dt, lqr, fi, fi_default, xcg, xcg_default, traj, status);
  });
}

// linearise_batch for aircraft [lo, lo + n): 176 B in, 3168 B out per aircraft -- the D2H of A and B is what the call costs, and
// the pipeline keeps it running from the first chunk to the last
static int linearise_host(const double* x, const double* u, long long ld, long long lo, long long n, double eps, int scheme, double* A,
                          double* B, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, int* status) {
  return run_pipeline({soa(x, IN, 8, 18), soa(u, IN, 8, 4), soa(fi, IN, 1), soa(xcg, IN, 8), aos(A, OUT, 8, 324), aos(B, OUT, 8, 72),
                       soa(status, OUT, 4, 1, true)},
                      ld, lo, n, plan_chunks(n, 1 << 14, 8), false, [&](const Slots& p, long long m) -> int {
                        CK(run_linearise(sel_of(p.u8(2), fi_default, p.f64(3), xcg_default), p.f64(0), m, p.f64(1), m, m, eps, scheme,
                                         p.f64(4), p.f64(5), p.i32(6)));
                        return F16_OK;
                      });
}

int linearise_batch(const double* x_soa, const double* u_soa, long long N, double eps, int scheme, double* A, double* B,
                    const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!linearise_ok(x_soa, N, u_soa, N, N, eps, scheme, A, B)) return bad_arg("linearise_batch");
  if (N == 0) return F16_OK;
  return on_devices(slices(N, 4096), [&](int, long long lo, long long n) {
    return linearise_host(x_soa, u_soa, N, lo, n, eps, scheme, A, B, fi, fi_default, xcg, xcg_default, status);
  });
}

// ---- trim_batch: env.py::trim for N flight conditions ------------------------------------------------------------
static const double kTrimGuess[5] = {5000, -0.09, 8.49, -0.01, 0.01};  // env.py:264-271 (unpacked as P3, dh, da, dr, alpha)

int trim_batch_dev(const double* h, const double* V, long long N, double tol, int maxiter, const double* ux0, double* x_trim_soa,
                   long long ld_x, double* info_soa, long long ld_info, const unsigned char* fi, int fi_default, const double* xcg,
                   double xcg_default, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!trim_ok(h, V, N, tol, maxiter, x_trim_soa, ld_x, info_soa, ld_info)) return bad_arg("trim_batch_dev");
  CK(run_trim(sel_of(fi, fi_default, xcg, xcg_default), h, V, N, tol, maxiter, ux0 ? ux0 : kTrimGuess, x_trim_soa, ld_x, info_soa,
              ld_info, status));
  return F16_OK;
}

// flight conditions [lo, lo + n) of the caller's arrays on the context D (a search is ~2000 dependent evaluations per point:
// nothing to pipeline, the copies are 16 + 180 B per point)
static int trim_host(const double* h, const double* V, long long ld, long long lo, long long n, double tol, int maxiter, const double* ux0,
                     double* x_trim, double* info, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default,
                     int* status) {
  return run_pipeline({soa(h, IN, 8), soa(V, IN, 8), soa(fi, IN, 1), soa(xcg, IN, 8), soa(x_trim, OUT, 8, 18),
                       soa(info, OUT, 8, 4, true), soa(status, OUT, 4, 1, true)},
                      ld, lo, n, one_chunk(n), false, [&](const Slots& p, long long m) -> int {
                        CK(run_trim(sel_of(p.u8(2), fi_default, p.f64(3), xcg_default), p.f64(0), p.f64(1), m, tol, maxiter,
                                    ux0 ? ux0 : kTrimGuess, p.f64(4), m, p.f64(5), m, p.i32(6)));
                        return F16_OK;
                      });
}

int trim_batch(const double* h, const double* V, long long N, double tol, int maxiter, const double* ux0, double* x_trim_soa,
               double* info_soa, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!trim_ok(h, V, N, tol, maxiter, x_trim_soa, N, info_soa, N)) return bad_arg("trim_batch");
  if (N == 0) return F16_OK;
  return on_devices(slices(N, 2048), [&](int, long long lo, long long n) {
    return trim_host(h, V, N, lo, n, tol, maxiter, ux0, x_trim_soa, info_soa, fi, fi_default, xcg, xcg_default, status);
  });
}

// ---- end-of-run statistics, reduced on the device (f16_stats.cu) ------------------------------------------------------
// enqueue the summary row of aircraft [0, N) and its copy to row_host (74 doubles) on D->stream
static int summary_row(const double* d_x, long long ld, long long N, const int* d_status, double* row_host) {
  const int grid = f16::stats::summary_grid(cfg(false), N);
  const size_t scratch_n = f16::stats::summary_scratch(grid);
  CK(D->b_sum.reserve((scratch_n + 74) * 8));
  double* scratch = (double*)D->b_sum.p;
  double* row = scratch + scratch_n;  // must not alias the scratch
  CK(f16::stats::launch_summary(cfg(false), d_x, ld, N, d_status, row, scratch, grid));
  CK(cudaMemcpyAsync(row_host, row, 74 * 8, cudaMemcpyDeviceToHost, D->stream));
  return F16_OK;
}

// K steps in chunks of snap_every, one summary row per chunk; x / u / status on the device.  rows_host [K / snap_every][74].
static int step_stats_core(double* d_x, long long ld_x, const double* d_u, long long ld_u, long long N, int K, int snap_every,
                           double dt, const f16_lqr_t* lqr, const f16::BatchSel& sel, int* d_status, double* rows_host) {
  const int n_rows = K / snap_every;
  const int grid = f16::stats::summary_grid(cfg(false), N);
  const size_t scratch_n = f16::stats::summary_scratch(grid);
  CK(D->b_sum.reserve((scratch_n + (size_t)(n_rows > 0 ? n_rows : 1) * 74) * 8));
  double* scratch = (double*)D->b_sum.p;
  double* rows_dev = scratch + scratch_n;
  const int rc = snapshot_steps(d_x, ld_x, d_u, ld_u, N, K, snap_every, dt, lqr, sel, d_status, [&](int j) -> int {
    CK(f16::stats::launch_summary(cfg(false), d_x, ld_x, N, d_status, rows_dev + (size_t)j * 74, scratch, grid));
    return F16_OK;
  });
  if (rc != F16_OK) return rc;
  if (n_rows > 0) CK(cudaMemcpyAsync(rows_host, rows_dev, (size_t)n_rows * 74 * 8, cudaMemcpyDeviceToHost, D->stream));
  return F16_OK;
}

int step_batch_stats_dev(double* x_soa, long long ld_x, const double* u_soa, long long ld_u, long long N, int K, int snap_every,
                         double dt, const f16_lqr_t* lqr, const unsigned char* fi, int fi_default, const double* xcg,
                         double xcg_default, double* rows, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!stats_ok(x_soa, ld_x, u_soa, ld_u, N, K, snap_every, lqr, rows) || (N > 0 && !status)) return bad_arg("step_batch_stats_dev");
  rc = step_stats_core(x_soa, ld_x, u_soa, ld_u, N, K, snap_every, dt, lqr, sel_of(fi, fi_default, xcg, xcg_default), status, rows);
  if (rc != F16_OK) return rc;
  CK(cudaStreamSynchronize(D->stream));
  return F16_OK;
}

// aircraft [lo, lo + n) of the caller's arrays on the context D; rows_out [K / snap_every][74] of this slice.  The status slot
// starts at 0: with K = 0 no step writes it.
static int stats_host(double* x, const double* u, long long ld, long long lo, long long n, int K, int snap_every, double dt,
                      const f16_lqr_t* lqr, const unsigned char* fi, int fi_default, const double* xcg, double xcg_default,
                      double* rows_out, int* status) {
  reserve_step_progress(n);
  return run_pipeline(
      {soa(x, INOUT, 8, 18), soa(u, IN, 8, 4), soa(fi, IN, 1), soa(xcg, IN, 8), soa(status, OUT, 4, 1, true)}, ld, lo, n,
      one_chunk(n), false, [&](const Slots& p, long long m) {
        CK(cudaMemsetAsync(p.i32(4), 0, (size_t)m * 4, D->stream));
        return step_stats_core(p.f64(0), m, p.f64(1), m, m, K, snap_every, dt, lqr, sel_of(p.u8(2), fi_default, p.f64(3), xcg_default),
                               p.i32(4), rows_out);
      });
}

int step_batch_stats(double* x_soa, const double* u_soa, long long N, int K, int snap_every, double dt, const f16_lqr_t* lqr,
                     const unsigned char* fi, int fi_default, const double* xcg, double xcg_default, double* rows, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!stats_ok(x_soa, N, u_soa, N, N, K, snap_every, lqr, rows)) return bad_arg("step_batch_stats");
  if (N == 0) {  // an empty batch still has rows: count 0, min = +inf, max = -inf
    rc = step_stats_core(nullptr, 0, nullptr, 0, 0, K, snap_every, dt, lqr, sel_of(nullptr, fi_default, nullptr, xcg_default), nullptr,
                         rows);
    if (rc != F16_OK) return rc;
    CK(cudaStreamSynchronize(D->stream));
    return F16_OK;
  }
  return merged_rows(N, 16384, K / snap_every, rows, [&](long long lo, long long n, double* part) {
    return stats_host(x_soa, u_soa, N, lo, n, K, snap_every, dt, lqr, fi, fi_default, xcg, xcg_default, part, status);
  });
}

int state_summary_batch_dev(const double* x_soa, long long ld_x, long long N, const int* status, double* row) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!summary_ok(x_soa, ld_x, N, row)) return bad_arg("state_summary_batch_dev");
  rc = summary_row(x_soa, ld_x, N, status, row);
  if (rc != F16_OK) return rc;
  CK(cudaStreamSynchronize(D->stream));
  return F16_OK;
}

int state_summary_batch(const double* x_soa, long long N, const int* status, double* row) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!summary_ok(x_soa, N, N, row)) return bad_arg("state_summary_batch");
  if (N == 0) {  // the empty row
    rc = summary_row(nullptr, 0, 0, nullptr, row);
    if (rc != F16_OK) return rc;
    CK(cudaStreamSynchronize(D->stream));
    return F16_OK;
  }
  return merged_rows(N, 65536, 1, row, [&](long long lo, long long n, double* part) {
    return run_pipeline({soa(x_soa, IN, 8, 18), soa(status, IN, 4)}, N, lo, n, one_chunk(n), false,
                        [&](const Slots& p, long long m) { return summary_row(p.f64(0), m, m, p.i32(1), part); });
  });
}

// ---- between linearise and the LQR law: reduced model, zero-order hold, discrete LQR gain --------------------------------
int reduce_jacobian_batch_dev(const double* A, long long N, double* A_na, double* B_na) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!reduce_ok(A, N, A_na, B_na)) return bad_arg("reduce_jacobian_batch_dev");
  CK(f16::linalg::launch_reduce_jacobian(cfg(false), A, N, A_na, B_na));
  return F16_OK;
}

int discretise_batch_dev(const double* A, const double* B, int n, int m, long long N, double dt, double* Ad, double* Bd) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!zoh_ok(A, B, n, m, N, dt, Ad, Bd)) return bad_arg("discretise_batch_dev");
  CK(f16::linalg::launch_zoh(cfg(false), A, B, n, m, N, dt, Ad, Bd));
  return F16_OK;
}

int dlqr_batch_dev(const double* Ad, const double* Bd, const double* Q /* device, n x n */, const double* R /* device, m x m */,
                   int n, int m, long long N, double* K, double* P, int* info) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!dlqr_ok(Ad, Bd, Q, R, n, m, N, K)) return bad_arg("dlqr_batch_dev");
  CK(f16::linalg::launch_dlqr(cfg(false), Ad, Bd, Q, R, n, m, N, 64, 1e-15, K, P, info));
  return F16_OK;
}

int reduce_jacobian_batch(const double* A, long long N, double* A_na, double* B_na) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!reduce_ok(A, N, A_na, B_na)) return bad_arg("reduce_jacobian_batch");
  if (N == 0) return F16_OK;
  return run_pipeline({aos(A, IN, 8, 324), aos(A_na, OUT, 8, 81), aos(B_na, OUT, 8, 27)}, N, 0, N, one_chunk(N), false,
                      [&](const Slots& p, long long len) -> int {
                        CK(f16::linalg::launch_reduce_jacobian(cfg(false), p.f64(0), len, p.f64(1), p.f64(2)));
                        return F16_OK;
                      });
}

int discretise_batch(const double* A, const double* B, int n, int m, long long N, double dt, double* Ad, double* Bd) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!zoh_ok(A, B, n, m, N, dt, Ad, Bd)) return bad_arg("discretise_batch");
  if (N == 0) return F16_OK;
  return run_pipeline({aos(A, IN, 8, n * n), aos(B, IN, 8, n * m), aos(Ad, OUT, 8, n * n), aos(Bd, OUT, 8, n * m)}, N, 0, N,
                      one_chunk(N), false, [&](const Slots& p, long long len) -> int {
                        CK(f16::linalg::launch_zoh(cfg(false), p.f64(0), p.f64(1), n, m, len, dt, p.f64(2), p.f64(3)));
                        return F16_OK;
                      });
}

// dlqr_batch and lqr_gain_batch: Q [n][n], R [m][m], shared by all systems, copied to b_qr on D->stream
static int stage_qr(const double* Q, const double* R, int n, int m) {
  CK(D->b_qr.reserve((size_t)(n * n + m * m) * 8));
  CK(cudaMemcpyAsync(D->b_qr.p, Q, (size_t)n * n * 8, cudaMemcpyHostToDevice, D->stream));
  CK(cudaMemcpyAsync((double*)D->b_qr.p + n * n, R, (size_t)m * m * 8, cudaMemcpyHostToDevice, D->stream));
  return F16_OK;
}

int dlqr_batch(const double* Ad, const double* Bd, const double* Q, const double* R, int n, int m, long long N, double* K, double* P,
               int* info) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (!dlqr_ok(Ad, Bd, Q, R, n, m, N, K)) return bad_arg("dlqr_batch");
  if (N == 0) return F16_OK;
  return run_pipeline({aos(Ad, IN, 8, n * n), aos(Bd, IN, 8, n * m), aos(K, OUT, 8, m * n), aos(P, OUT, 8, n * n), aos(info, OUT, 4, 2)},
                      N, 0, N, one_chunk(N), false, [&](const Slots& p, long long len) -> int {
                        const int st = stage_qr(Q, R, n, m);
                        if (st != F16_OK) return st;
                        const double* q = (const double*)D->b_qr.p;
                        CK(f16::linalg::launch_dlqr(cfg(false), p.f64(0), p.f64(1), q, q + n * n, n, m, len, 64, 1e-15, p.f64(2),
                                                    p.f64(3), p.i32(4)));
                        return F16_OK;
                      });
}

// F16._calc_LQR_gain (env.py:344-358) for N operating points, every stage on the device:
// forward linearise -> reduced 9-state / 3-input model -> cont2discrete(dt) -> K = -dlqr(Ad, Bd, C'C = I, R = I)
int lqr_gain_batch(const double* x_soa, const double* u_soa, long long N, double dt, double* K /* [N][3][9] */, const unsigned char* fi,
                   int fi_default, const double* xcg, double xcg_default, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (N < 0 || (N > 0 && (!x_soa || !u_soa || !K)) || !(dt > 0)) return bad_arg("lqr_gain_batch");
  if (N == 0) return F16_OK;
  static const double kI9[81] = {1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0,
                                 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0,
                                 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1};
  static const double kI3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  const size_t n = (size_t)N;
  try {  // the host copy of the dlqr info must not throw through the C ABI
    std::vector<int> info(status ? 2 * n : 0);
    rc = run_pipeline(
        {soa(x_soa, IN, 8, 18), soa(u_soa, IN, 8, 4), soa(fi, IN, 1), soa(xcg, IN, 8), aos(K, OUT, 8, 27),
         soa(status, OUT, 4, 1, true), aos(status ? info.data() : nullptr, OUT, 4, 2, true), aos(nullptr, OUT, 8, 324, true),
         aos(nullptr, OUT, 8, 72, true), aos(nullptr, OUT, 8, 81, true), aos(nullptr, OUT, 8, 27, true),
         aos(nullptr, OUT, 8, 81, true), aos(nullptr, OUT, 8, 27, true)},
        N, 0, N, one_chunk(N), false, [&](const Slots& p, long long len) -> int {
          // the reduced model evaluates at X with the actuator states replaced by the inputs (env.py:175-177)
          CK(cudaMemcpyAsync(p.f64(0) + 13 * len, p.f64(1) + len, 3 * (size_t)len * 8, cudaMemcpyDeviceToDevice, D->stream));
          const int st = stage_qr(kI9, kI3, 9, 3);
          if (st != F16_OK) return st;
          const double* q = (const double*)D->b_qr.p;
          CK(f16::strict::launch_linearise(cfg(true), tabs(), sel_of(p.u8(2), fi_default, p.f64(3), xcg_default), p.f64(0), len,
                                           p.f64(1), len, len, 1e-5, F16_FD_FORWARD, p.f64(7), p.f64(8), p.i32(5)));
          CK(f16::linalg::launch_reduce_jacobian(cfg(false), p.f64(7), len, p.f64(9), p.f64(10)));
          CK(f16::linalg::launch_zoh(cfg(false), p.f64(9), p.f64(10), 9, 3, len, dt, p.f64(11), p.f64(12)));
          CK(f16::linalg::launch_dlqr(cfg(false), p.f64(11), p.f64(12), q, q + 81, 9, 3, len, 64, 1e-15, p.f64(4), nullptr, p.i32(6)));
          return F16_OK;
        });
    if (rc != F16_OK) return rc;
    for (size_t i = 0; i < 27 * n; i++) K[i] = -K[i];  // env.py:356: K = - dlqr(A, B, Q, R)
    if (status)
      for (size_t i = 0; i < n; i++) status[i] = status[i] ? status[i] : (info[2 * i] < 0 ? (int)F16_ST_NAN : 0);
    return F16_OK;
  } catch (const std::exception& e) {
    set_err("lqr_gain_batch: host resources: %s", e.what());
    return F16_ERR_HOST;
  }
}

// ---- parity probes: one chunk on the current context ----------------------------------------------------------------
int f16_hifi_probe(const double* alpha_deg, const double* beta_deg, const double* el, long long N, double* coef, int* cells,
                   int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (N <= 0 || !alpha_deg || !beta_deg || !el || !coef || !cells) return bad_arg("f16_hifi_probe");
  return run_pipeline({soa(alpha_deg, IN, 8), soa(beta_deg, IN, 8), soa(el, IN, 8), soa(coef, OUT, 8, 44), soa(cells, OUT, 4, 8),
                       soa(status, OUT, 4, 1, true)},
                      N, 0, N, one_chunk(N), false, [&](const Slots& p, long long m) -> int {
                        CK(f16::strict::launch_hifi_probe(cfg(false), tabs(), p.f64(0), p.f64(1), p.f64(2), m, p.f64(3), p.i32(4),
                                                          p.i32(5)));
                        return F16_OK;
                      });
}

int f16_fast_probe(const double* alpha_deg, const double* beta_deg, const double* el, long long N, double* coef, int* cells,
                   double* lam, int* status) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (N <= 0 || !alpha_deg || !beta_deg || !el || !coef || !cells || !lam) return bad_arg("f16_fast_probe");
  return run_pipeline({soa(alpha_deg, IN, 8), soa(beta_deg, IN, 8), soa(el, IN, 8), soa(coef, OUT, 8, 44), soa(cells, OUT, 4, 4),
                       soa(lam, OUT, 8, 4), soa(status, OUT, 4, 1, true)},
                      N, 0, N, one_chunk(N), false, [&](const Slots& p, long long m) -> int {
                        CK(f16::fast::launch_fast_probe(cfg(false), tabs(), p.f64(0), p.f64(1), p.f64(2), m, p.f64(3), p.i32(4),
                                                        p.f64(5), p.i32(6)));
                        return F16_OK;
                      });
}

int f16_lofi_probe(const double* alpha_deg, const double* beta_deg, const double* el, const double* dail,
                   const double* drud, long long N, double* out) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (N <= 0 || !alpha_deg || !beta_deg || !el || !dail || !drud || !out) return bad_arg("f16_lofi_probe");
  return run_pipeline({soa(alpha_deg, IN, 8), soa(beta_deg, IN, 8), soa(el, IN, 8), soa(dail, IN, 8), soa(drud, IN, 8),
                       soa(out, OUT, 8, 19)},
                      N, 0, N, one_chunk(N), false, [&](const Slots& p, long long m) -> int {
                        CK(f16::strict::launch_lofi_probe(cfg(false), tabs(), p.f64(0), p.f64(1), p.f64(2), p.f64(3), p.f64(4), m,
                                                          p.f64(5)));
                        return F16_OK;
                      });
}

int f16_div_probe(const double* a, const double* b, long long N, double* out) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (N <= 0 || !a || !b || !out) return bad_arg("f16_div_probe");
  return run_pipeline({soa(a, IN, 8), soa(b, IN, 8), soa(out, OUT, 8, 3)}, N, 0, N, one_chunk(N), false,
                      [&](const Slots& p, long long m) -> int {
                        CK(f16::strict::launch_div_probe(cfg(false), p.f64(0), p.f64(1), m, p.f64(2)));
                        return F16_OK;
                      });
}

int atmos_batch(const double* alt, const double* vt, long long N, double* coeff_soa) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  if (N <= 0 || !alt || !vt || !coeff_soa) return bad_arg("atmos_batch");
  return run_pipeline({soa(alt, IN, 8), soa(vt, IN, 8), soa(coeff_soa, OUT, 8, 3)}, N, 0, N, one_chunk(N), false,
                      [&](const Slots& p, long long m) -> int {
                        CK(f16::strict::launch_atmos(cfg(false), p.f64(0), p.f64(1), m, p.f64(2)));
                        return F16_OK;
                      });
}

// ---- memory / timing helpers ------------------------------------------------------------------------------------------
void* f16_dev_alloc(unsigned long long bytes) {
  std::lock_guard<std::mutex> lk(G_mu);
  if (ensure() != F16_OK) return nullptr;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) { cuda_fail(e, "cudaMalloc"); return nullptr; }
  return p;
}
void f16_dev_free(void* p) {
  if (p) cudaFree(p);
}
void* f16_host_alloc_pinned(unsigned long long bytes) {
  std::lock_guard<std::mutex> lk(G_mu);
  if (ensure() != F16_OK) return nullptr;
  void* p = nullptr;
  cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
  if (e != cudaSuccess) { cuda_fail(e, "cudaHostAlloc"); return nullptr; }
  return p;
}
void f16_host_free_pinned(void* p) {
  if (p) cudaFreeHost(p);
}
int f16_memcpy_h2d(void* dst_dev, const void* src_host, unsigned long long bytes) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, D->stream));
  CK(cudaStreamSynchronize(D->stream));
  return F16_OK;
}
int f16_memcpy_d2h(void* dst_host, const void* src_dev, unsigned long long bytes) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, D->stream));
  CK(cudaStreamSynchronize(D->stream));
  return F16_OK;
}
int f16_memcpy_d2d(void* dst_dev, const void* src_dev, unsigned long long bytes) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaMemcpyAsync(dst_dev, src_dev, bytes, cudaMemcpyDeviceToDevice, D->stream));
  return F16_OK;
}
int f16_memset_dev(void* dst_dev, int value, unsigned long long bytes) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaMemsetAsync(dst_dev, value, bytes, D->stream));
  return F16_OK;
}
int f16_sync(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaStreamSynchronize(D->stream));
  return F16_OK;
}
int f16_timer_start(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaEventRecord(D->ev0, D->stream));
  return F16_OK;
}
int f16_timer_stop(float* ms) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(cudaEventRecord(D->ev1, D->stream));
  CK(cudaEventSynchronize(D->ev1));
  CK(cudaEventElapsedTime(ms, D->ev0, D->ev1));
  return F16_OK;
}

int f16_measure_fp64_peak(double ms, double* tflops) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  CK(D->b_flush.reserve(64));
  double flops = 0;
  float t = 0;
  long long iters = 2000;
  // calibrate, then run for about `ms`
  for (int pass = 0; pass < 2; pass++) {
    CK(cudaEventRecord(D->ev0, D->stream));
    CK(f16::launch_dfma_peak(D->stream, D->sm_count, iters, (double*)D->b_flush.p, &flops));
    ++D->launches;
    CK(cudaEventRecord(D->ev1, D->stream));
    CK(cudaEventSynchronize(D->ev1));
    CK(cudaEventElapsedTime(&t, D->ev0, D->ev1));
    if (pass == 0) {
      double want = ms > 1 ? ms : 1;
      iters = (long long)(iters * want / (t > 1e-3f ? t : 1e-3f));
      if (iters < 100) iters = 100;
    }
  }
  *tflops = flops / (t * 1e-3) / 1e12;
  return F16_OK;
}

int f16_flush_l2(void) {
  std::lock_guard<std::mutex> lk(G_mu);
  int rc = ensure();
  if (rc != F16_OK) return rc;
  const size_t bytes = 256u << 20;  // > 126 MB L2
  CK(D->b_flush.reserve(bytes));
  CK(cudaMemsetAsync(D->b_flush.p, 0, bytes, D->stream));
  return F16_OK;
}

#pragma GCC visibility pop
}  // extern "C"

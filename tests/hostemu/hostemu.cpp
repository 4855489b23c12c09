// hostemu.cpp -- DEVELOPMENT AID, TESTS ONLY.  Compiles the device arithmetic headers (csrc/f16_model.cuh, f16_fast.cuh,
// f16_linalg.cuh) for the host so that the kernels' logic (cell search, node-interleaved gathers, operation order, the
// linalg bodies) can be checked against the oracle and high-precision references on a machine without a GPU.  It is never part of libf16_b200.so and nothing in the package loads it;
// the product has no CPU path.
#include <string>
#include <vector>

#include "../../f16_mpc_oop_py_b200/csrc/f16_model.cuh"
#include "../../f16_mpc_oop_py_b200/csrc/f16_fast.cuh"
#include "../../f16_mpc_oop_py_b200/csrc/f16_linalg.cuh"
#include "../../f16_mpc_oop_py_b200/csrc/f16_tables_host.h"

static std::vector<double> g_hifi, g_lofi, g_fast;

extern "C" {
__attribute__((visibility("default"))) int emu_init(const char* path, int clr_from_file) {
  std::vector<double> payload;
  std::string src, err;
  if (!f16::load_canonical(path, "", payload, src, err)) return -1;
  if (!f16::check_grids(payload, err)) return -2;
  f16::build_hifi_image(payload, clr_from_file != 0, g_hifi);
  f16::build_lofi_image(g_lofi);
  f16::build_hifi_fast_image(payload, clr_from_file != 0, g_fast);
  return 0;
}

__attribute__((visibility("default"))) unsigned emu_nlplant(const double* xu_, double* xd_, int fi, double xcg) {
  double xu[17], xd[18];
  for (int i = 0; i < 17; i++) xu[i] = xu_[i];
  unsigned st = fi ? f16::nlplant_eval<1>(g_hifi.data(), xu, xcg, xd) : f16::nlplant_eval<0>(g_lofi.data(), xu, xcg, xd);
  for (int i = 0; i < 18; i++) xd_[i] = st ? __builtin_nan("") : xd[i];
  return st;
}

__attribute__((visibility("default"))) unsigned emu_calc_xdot(const double* x_, const double* u_, double* xd_, int fi, double xcg) {
  double x[18], u[4], xd[18];
  for (int i = 0; i < 18; i++) x[i] = x_[i];
  for (int i = 0; i < 4; i++) u[i] = u_[i];
  unsigned st = fi ? f16::calc_xdot<1>(g_hifi.data(), x, u, xcg, xd) : f16::calc_xdot<0>(g_lofi.data(), x, u, xcg, xd);
  for (int i = 0; i < 18; i++) xd_[i] = st ? __builtin_nan("") : xd[i];
  return st;
}

__attribute__((visibility("default"))) unsigned emu_step(double* x_, const double* u_, int K, double dt, int fi, double xcg,
                                                         const f16::LqrLaw* lqr, int* steps_done) {
  double x[18], u_in[4];
  for (int i = 0; i < 18; i++) x[i] = x_[i];
  for (int i = 0; i < 4; i++) u_in[i] = u_[i];
  unsigned st = 0;
  int k = 0;
  for (; k < K; k++) {
    st = f16::step_bounds(x, u_in);
    if (st) break;
    double u[4], xd[18];
    if (lqr) f16::lqr_action(*lqr, x, u_in, u);
    else for (int i = 0; i < 4; i++) u[i] = u_in[i];
    st = fi ? f16::calc_xdot<1>(g_hifi.data(), x, u, xcg, xd) : f16::calc_xdot<0>(g_lofi.data(), x, u, xcg, xd);
    if (st) break;
    for (int i = 0; i < 18; i++) x[i] = x[i] + xd[i] * dt;
  }
  for (int i = 0; i < 18; i++) x_[i] = x[i];
  if (steps_done) *steps_done = k;
  return st;
}

__attribute__((visibility("default"))) unsigned emu_hifi_probe(double a, double b, double e, double* o, int* cl) {
  unsigned st = f16::hifi_envelope(a, b, e);
  if (st) return st;
  const double* img = g_hifi.data();
  f16::HifiLoc L = f16::hifi_locate(img, a, b, e);
  f16::Coef c;
  f16::hifi_coefs(img, L, c);
  const double v[44] = {c.Cx, c.Cz, c.Cm, c.Cy, c.Cn, c.Cl, c.Cxq, c.Cyr, c.Cyp, c.Czq, c.Clr, c.Clp, c.Cmq, c.Cnr, c.Cnp,
                        c.dCx_lef, c.dCz_lef, c.dCm_lef, c.dCy_lef, c.dCn_lef, c.dCl_lef,
                        c.dCxq_lef, c.dCyr_lef, c.dCyp_lef, c.dCzq_lef, c.dClr_lef, c.dClp_lef, c.dCmq_lef, c.dCnr_lef, c.dCnp_lef,
                        c.dCy_r30, c.dCn_r30, c.dCl_r30, c.dCy_a20, c.dCy_a20_lef, c.dCn_a20, c.dCn_a20_lef, c.dCl_a20, c.dCl_a20_lef,
                        c.dCnbeta, c.dClbeta, c.dCm, c.eta_el, c.dCm_ds};
  for (int i = 0; i < 44; i++) o[i] = v[i];
  f16::ref_cell(img + F16_IMG_A, L.a, a, cl[0], cl[1]);
  f16::ref_cell(img + F16_IMG_B, L.b, b, cl[2], cl[3]);
  f16::ref_cell(img + F16_IMG_D1, L.d1, e, cl[4], cl[5]);
  f16::ref_cell(img + F16_IMG_D2, L.d2, e, cl[6], cl[7]);
  return 0;
}
// the fast image + cell search as f16_fast_probe runs them (fastmath::probe_hifi)
__attribute__((visibility("default"))) unsigned emu_fast_probe(double a, double b, double e, double* o, int* cl, double* lam) {
  unsigned st = f16::hifi_envelope(a, b, e);
  if (st) return st;
  double oo[44], ll[4];
  int cc[4];
  f16::fastmath::probe_hifi(g_fast.data(), a, b, e, oo, cc, ll);
  for (int i = 0; i < 44; i++) o[i] = oo[i];
  for (int i = 0; i < 4; i++) { cl[i] = cc[i]; lam[i] = ll[i]; }
  return 0;
}
// the F16_MATH_FAST arithmetic of f16_fast.cuh (hifi step), same control flow as step_hifi_fast_kernel
__attribute__((visibility("default"))) unsigned emu_calc_xdot_fast(const double* x_, const double* u_, double* xd_, double xcg) {
  double x[18], u[4], xd[18];
  for (int i = 0; i < 18; i++) x[i] = x_[i];
  for (int i = 0; i < 4; i++) u[i] = u_[i];
  double uc[4];
  f16::fastmath::clip_commands(u, uc);
  const bool ok = f16::fastmath::calc_xdot_hifi<false>(g_fast.data(), x, uc, xcg, xd);
  for (int i = 0; i < 18; i++) xd_[i] = ok ? xd[i] : __builtin_nan("");
  return ok ? 0u : f16::hifi_envelope(x[7] * (180.0 / 3.141592653589793), x[8] * (180.0 / 3.141592653589793), x[13]);
}

__attribute__((visibility("default"))) unsigned emu_step_fast(double* x_, const double* u_, int K, double dt, double xcg,
                                                              const f16::LqrLaw* lqr, int* steps_done) {
  double x[18], u_in[4];
  for (int i = 0; i < 18; i++) x[i] = x_[i];
  for (int i = 0; i < 4; i++) u_in[i] = u_[i];
  int k = 0;
  f16::fastmath::LqrDense dense;
  if (lqr) f16::fastmath::make_dense_law(*lqr, dense);
  const unsigned st = lqr ? f16::fastmath::step_aircraft<true>(g_fast.data(), x, u_in, &dense, xcg, dt, K, k)
                          : f16::fastmath::step_aircraft<false>(g_fast.data(), x, u_in, nullptr, xcg, dt, K, k);
  for (int i = 0; i < 18; i++) x_[i] = x[i];
  if (steps_done) *steps_done = k;
  return st;
}

// the lofi step on the same arithmetic (step_lofi_fast_kernel): its image is the lofi tables + the centre table of half_rho
__attribute__((visibility("default"))) unsigned emu_step_fast_lofi(double* x_, const double* u_, int K, double dt, double xcg,
                                                                   const f16::LqrLaw* lqr, int* steps_done) {
  static std::vector<double> img;
  if (img.empty()) {
    img = g_lofi;
    img.insert(img.end(), g_fast.begin() + F16_FI_POW, g_fast.begin() + F16_FI_POW + 2 * F16_FI_NPOW);
  }
  double x[18], u_in[4];
  for (int i = 0; i < 18; i++) x[i] = x_[i];
  for (int i = 0; i < 4; i++) u_in[i] = u_[i];
  int k = 0;
  f16::fastmath::LqrDense dense;
  if (lqr) f16::fastmath::make_dense_law(*lqr, dense);
  const unsigned st = lqr ? f16::fastmath::step_aircraft<true, 0>(img.data(), x, u_in, &dense, xcg, dt, K, k)
                          : f16::fastmath::step_aircraft<false, 0>(img.data(), x, u_in, nullptr, xcg, dt, K, k);
  for (int i = 0; i < 18; i++) x_[i] = x[i];
  if (steps_done) *steps_done = k;
  return st;
}

// accuracy probes of the fast elementary functions: out = {sin, cos (sincos_any), sin, cos (sincos_quarter), half_rho}
__attribute__((visibility("default"))) void emu_fastmath_probe(double x, double tfac, double* out) {
  f16::fastmath::sincos_any(x, out[0], out[1]);
  f16::fastmath::sincos_quarter(x, out[2], out[3]);
  out[4] = f16::fastmath::half_rho(g_fast.data(), tfac);
}
// linearise_kernel's staged evaluation: base stages at (x0,u0), then f at the point perturbed in component `col`
__attribute__((visibility("default"))) unsigned emu_calc_xdot_col(const double* x0_, const double* u0_, int col, double delta,
                                                                  double* xd_, int fi, double xcg) {
  double x[18], u[4], xd[18], xu0[17];
  for (int i = 0; i < 18; i++) x[i] = x0_[i];
  for (int i = 0; i < 4; i++) u[i] = u0_[i];
  for (int i = 0; i < 17; i++) xu0[i] = x[i];
  const double* img = fi ? g_hifi.data() : g_lofi.data();
  f16::XdotBase b;
  b.tr = f16::trig_eval(xu0);
  f16::atmos_pair(x, b.al, b.an);
  const double r2d = 180.0 / 3.141592653589793;
  const unsigned st0 = fi ? f16::envelope_of<1>(xu0) : f16::envelope_of<0>(xu0);
  if (!st0) {
    if (fi) f16::coef_eval<1>(img, xu0[7] * r2d, xu0[8] * r2d, xu0[13], xu0[14] / 21.5, xu0[15] / 30.0, b.c);
    else f16::coef_eval<0>(img, xu0[7] * r2d, xu0[8] * r2d, xu0[13], xu0[14] / 21.5, xu0[15] / 30.0, b.c);
  }
  if (col >= 0 && col < 18) x[col] = x[col] + delta;
  if (col >= 18) u[col - 18] = u[col - 18] + delta;
  const unsigned st = fi ? f16::calc_xdot_col<1>(img, x, u, xcg, b, col, xd) : f16::calc_xdot_col<0>(img, x, u, xcg, b, col, xd);
  for (int i = 0; i < 18; i++) xd_[i] = st ? __builtin_nan("") : xd[i];
  return st;
}
// trim (Nelder-Mead on the device arithmetic): x_trim[18], info = {cost, iterations, fcalls, converged}
// fixed_point_exit: leave a search that has reached a bitwise fixed point (1, the library's default) or spin to maxiter (0)
__attribute__((visibility("default"))) unsigned emu_trim_fp(double h, double V, int fi, double xcg, double tol, int maxiter,
                                                            int fixed_point_exit, double* x_trim, double* info) {
  double ux[5] = {5000, -0.09, 8.49, -0.01, 0.01};
  const f16::TrimPoint t = f16::trim_point(h, V);
  const f16::TrimResult r = fi ? f16::nelder_mead_trim<1>(g_hifi.data(), t, xcg, tol, maxiter, ux, fixed_point_exit != 0)
                               : f16::nelder_mead_trim<0>(g_lofi.data(), t, xcg, tol, maxiter, ux, fixed_point_exit != 0);
  double x[18];
  f16::trim_state(t, ux, x);
  for (int i = 0; i < 18; i++) x_trim[i] = x[i];
  info[0] = r.cost; info[1] = r.iterations; info[2] = r.fcalls; info[3] = r.converged;
  return r.status;
}
__attribute__((visibility("default"))) unsigned emu_trim(double h, double V, int fi, double xcg, double tol, int maxiter,
                                                         double* x_trim, double* info) {
  return emu_trim_fp(h, V, fi, xcg, tol, maxiter, 1, x_trim, info);
}
// div_by (exact division through a rounded reciprocal) on n numerators: out[i] = the device arithmetic's a[i] / y
__attribute__((visibility("default"))) void emu_div_by(const double* a, long long n, double y, double* out) {
  const double r = 1.0 / y;
  for (long long i = 0; i < n; i++) out[i] = f16::div_by(a[i], y, r);
}
// the linalg bodies of f16_linalg.cu, one system after the other (the kernels run one system per thread).  Without FMA
// contraction, unlike linalg.o: the results agree with the device's to rounding, not bit for bit.
__attribute__((visibility("default"))) void emu_zoh(const double* A, const double* B, int n, int m, long long N, double dt,
                                                    double* Ad, double* Bd) {
  const int sz = f16::linalg::MAXD * f16::linalg::MAXD;
  std::vector<double> s(3 * sz);
  for (long long p = 0; p < N; p++) f16::linalg::zoh_one(A, B, n, m, p, dt, Ad, Bd, &s[0], &s[sz], &s[2 * sz]);
}
// the library's settings are max_doublings = 64, tol = 1e-15 (f16_api.cu)
__attribute__((visibility("default"))) void emu_dlqr(const double* A, const double* B, const double* Q, const double* R, int n, int m,
                                                     long long N, int max_doublings, double tol, double* K, double* P, int* info) {
  const int sz = f16::linalg::MAXD * f16::linalg::MAXD;
  std::vector<double> s(7 * sz);
  for (long long p = 0; p < N; p++)
    f16::linalg::dlqr_one(A, B, Q, R, n, m, p, max_doublings, tol, K, P, info, &s[0], &s[sz], &s[2 * sz], &s[3 * sz], &s[4 * sz],
                          &s[5 * sz], &s[6 * sz]);
}
__attribute__((visibility("default"))) void emu_reduce_jacobian(const double* A, long long N, double* A_na, double* B_na) {
  for (long long p = 0; p < N; p++)
    for (int k = 0; k < 108; k++) f16::linalg::reduce_one(A, p, k, A_na, B_na);
}
}

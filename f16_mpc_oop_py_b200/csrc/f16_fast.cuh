// f16_fast.cuh -- the throughput arithmetic of the fused hifi Euler step (F16_MATH_FAST).
//
// Same model as f16_model.cuh (which keeps the reference's operation order and is the parity build), re-associated
// for the B200 FP64 pipe.  Every substitution below moves a derivative by a few ulp of its natural scale; the
// budget (tests/test_gpu_parity.py, tests/test_model_host.py) is 1e-12 scaled per derivative and 1e-9 after 10 s.
//
//   * tables: the "fast image" stores, per alpha CELL, the value at the lower node and the difference to the upper
//     node, so an alpha interpolation is ONE fma(lambda, d, f) instead of lambda*f2 + (1-lambda)*f1
//     (mexndinterp.c:196-197), and one LDS.128 fetches (f, d);
//   * the rudder / aileron / lef tables of one force or moment are combined with their weights at each beta node
//     before the beta interpolation (hifi_F16_AeroData.c:1892-1926 + nlplant.c:333-377 are linear in the tables);
//   * sin/cos: alpha and beta are inside [-pi/4, pi/4] whenever the hifi envelope check passed, so they need no
//     argument reduction; phi, theta, psi use a two-constant Cody-Waite reduction; coefficients live in the
//     constant bank (no UMOV pairs in the instruction stream);
//   * rho = rho0 * tfac^4.14 (nlplant.c:478): tfac in [0.297, 1] on the bounded altitude range, evaluated as
//     c^4.14 * (1+s)^4.14 with c from a 48-entry table and a degree-7 binomial series in |s| <= 0.027;
//   * Vt/alpha/beta dots use U = vt ca cb, V = vt sb, W = vt sa cb to cancel vt analytically; qbar/ps of the LEF
//     schedule (utils.py:296) cancels rho.
//
// Reference lines are cited next to each block; names follow C/nlplant.c.
#pragma once
#include "f16_model.cuh"

#if defined(__CUDACC__)
#define F16_FD __device__ __forceinline__
#define F16_KCONST __constant__
#else
#define F16_FD static inline __attribute__((always_inline))
#define F16_KCONST static const
#endif

namespace f16 {
namespace fastmath {

// Constant-bank operands (one LDCU.64 each instead of two UMOV immediates).  sin/cos kernels on [-pi/4, pi/4]:
// the classic fdlibm minimax coefficients.
struct K_t {
  double S[6], C[6];
  double two_over_pi, pio2_hi, pio2_mid;
  double PW[9];  // binomial coefficients C(4.14, k), k = 1..9
  double r2d, inv15, c5_3, c7_3, tlapse, inv21_5, inv30, ninv25, half_cbar, g, S_m, inv_m, lef_q, inv_pi,
      c1_38, c1_45, c20_2, inv0_136, ixx_qr, ixx_pq, ixx_l, ixx_n, iyy_pr, iyy_p2, inv_Jy, izz_n, izz_l, izz_pq, izz_qr,
      xcg_arm;
  double c0_2, c0_04, c0_01, c0_35;  // literals whose low word is not zero: an FP64 instruction cannot carry them as immediates
};
// inertia terms of nlplant.c:413-436 pre-divided by (Jx Jz - Jxz^2) resp. Jy
#define F16_JX 9496.0
#define F16_JY 55814.0
#define F16_JZ 63100.0
#define F16_JXZ 982.0
#define F16_JD (F16_JX * F16_JZ - F16_JXZ * F16_JXZ)
F16_KCONST K_t K = {
    {-1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04, 2.75573137070700676789e-06,
     -2.50507602534068634195e-08, 1.58969099521155010221e-10},
    {4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05, -2.75573143513906633035e-07,
     2.08757232129817482790e-09, -1.13596475577881948265e-11},
    0.6366197723675814, 1.5707963267948966, 6.123233995736766e-17,
    {4.14, 6.499799999999999, 4.636523999999999, 1.321409339999999, 0.036999461519999895, -0.005303256151199987,
     0.0014091509201759967, -0.0005037714539629189, 0.00021606197914409635},
    180.0 / 3.141592653589793, 1.0 / 15.0, 5.0 / 3.0, 7.0 / 3.0, -.703e-5, 1.0 / 21.5, 1.0 / 30.0,
    -1.0 / 25.0, 0.5 * 11.32, 32.17, 300.0 / 636.94, 1.0 / 636.94, 0.5 * 9.05 / 1715.0, 1.0 / 3.141592653589793,
    1.38, 1.45, 20.2, 1 / 0.136,
    -(F16_JZ * (F16_JZ - F16_JY) + F16_JXZ * F16_JXZ) / F16_JD, F16_JXZ * (F16_JX - F16_JY + F16_JZ) / F16_JD,
    F16_JZ / F16_JD, F16_JXZ / F16_JD,
    (F16_JZ - F16_JX) / F16_JY, -F16_JXZ / F16_JY, 1.0 / F16_JY,
    F16_JX / F16_JD, F16_JXZ / F16_JD, (F16_JX * (F16_JX - F16_JY) + F16_JXZ * F16_JXZ) / F16_JD,
    -F16_JXZ * (F16_JX - F16_JY + F16_JZ) / F16_JD,
    11.32 / 30.0,
    0.2, 0.04, 0.01, 0.35};

F16_FD int lo32(double v) {
#if defined(__CUDA_ARCH__)
  return __double2loint(v);
#else
  long long b;
  __builtin_memcpy(&b, &v, 8);
  return (int)(b & 0xffffffffLL);
#endif
}
F16_FD int hi32(double v) {
#if defined(__CUDA_ARCH__)
  return __double2hiint(v);
#else
  long long b;
  __builtin_memcpy(&b, &v, 8);
  return (int)(b >> 32);
#endif
}
F16_FD double flip_sign(double v, int mask_hi) {  // mask_hi = 0 or 0x80000000
#if defined(__CUDA_ARCH__)
  return __hiloint2double(__double2hiint(v) ^ mask_hi, __double2loint(v));
#else
  unsigned long long b;
  __builtin_memcpy(&b, &v, 8);
  b ^= ((unsigned long long)(unsigned)mask_hi) << 32;
  __builtin_memcpy(&v, &b, 8);
  return v;
#endif
}

// sin and cos for |x| <= pi/4 (16 FP64 instructions)
F16_FD void sincos_quarter(double x, double& s, double& c) {
  const double z = x * x;
  double ps = fma(z, K.S[5], K.S[4]);
  double pc = fma(z, K.C[5], K.C[4]);
  ps = fma(z, ps, K.S[3]);
  pc = fma(z, pc, K.C[3]);
  ps = fma(z, ps, K.S[2]);
  pc = fma(z, pc, K.C[2]);
  ps = fma(z, ps, K.S[1]);
  pc = fma(z, pc, K.C[1]);
  ps = fma(z, ps, K.S[0]);
  pc = fma(z, pc, K.C[0]);
  s = fma(x * z, ps, x);
  c = fma(z, fma(z, pc, -0.5), 1.0);
}

// sin and cos for |x| < 2^30: j = rint(x 2/pi), r = x - j pi/2 in two FMAs (|j (pi/2 - hi - mid)| < 1e-23); the quadrant
// q = j mod 4 swaps / negates the two kernels.  Larger arguments never reach this function (step_ok()).
F16_FD int reduce_pio2(double x, double& r) {
  const double magic = 6755399441055744.0;  // 1.5 * 2^52
  const double t = fma(x, K.two_over_pi, magic);
  const double j = t - magic;
  r = fma(-j, K.pio2_hi, x);
  r = fma(-j, K.pio2_mid, r);
  return lo32(t);
}
F16_FD void quadrant_fix(int q, double& s, double& c) {
  const bool sw = (q & 1) != 0;
  const double s0 = sw ? c : s, c0 = sw ? s : c;
  s = flip_sign(s0, (q & 2) << 30);
  c = flip_sign(c0, ((q + 1) & 2) << 30);
}
F16_FD void sincos_any(double x, double& s, double& c) {
  double r;
  const int q = reduce_pio2(x, r);
  sincos_quarter(r, s, c);
  quadrant_fix(q, s, c);
}

#if defined(__CUDACC__)
static __device__ __noinline__ void sincos_libm(double x, double* s, double* c) { sincos(x, s, c); }
#else
static void sincos_libm(double x, double* s, double* c) { *s = sin(x); *c = cos(x); }
#endif

// 0.5 * rho0 * tfac^4.14 for tfac in [0.28125, 1.03125): table of centres + binomial series (13 FP64 instructions)
F16_FD double half_rho(const double* img, double tfac) {
  const double magic = 6755399441055744.0;
  const double u = fma(tfac, 64.0, -18.5);
  const double tm = u + magic;
  int i = lo32(tm);
  const double d = u - (tm - magic);  // |d| <= 0.5, exact
  i = i < 0 ? 0 : (i > F16_FI_NPOW - 1 ? F16_FI_NPOW - 1 : i);
  const d2 e = ld2(img + F16_FI_POW + 2 * i);
  const double s = d * e.x;  // (tfac - c_i) / c_i
  double p = fma(s, K.PW[6], K.PW[5]);  // degree 7: the terms left out are C(4.14, 8) s^8 <= 1.4e-16 and C(4.14, 9) s^9 <= 2e-18
  p = fma(s, p, K.PW[4]);
  p = fma(s, p, K.PW[3]);
  p = fma(s, p, K.PW[2]);
  p = fma(s, p, K.PW[1]);
  p = fma(s, p, K.PW[0]);
  p = fma(s, p, 1.0);
  return p * e.y;
}

// 1/v for a well-scaled positive or negative v: hardware seed + two Newton steps, no special-case path
F16_FD double rcp_nr(double v) {
#if defined(__CUDA_ARCH__)
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(v));
  double e = fma(-v, y, 1.0);
  y = fma(y, e, y);
  e = fma(-v, y, 1.0);
  y = fma(y, e, y);
  return y;
#else
  return 1.0 / v;
#endif
}

// Cell and weight of a query on the four hifi axes (ALPHA -20:5:45; BETA1 -30:5:-10:2:10:5:30; DH1 -25,-10,0,10,25; DH2 -25,0,25
// -- check_grids() verifies the grids are these).  Every breakpoint is a whole number of degrees, so the cell of a query follows
// from the integer t = floor(query - axis start), and that integer is exact: it is the low word of ONE addition rounded towards
// minus infinity, query + (1.5 * 2^52 - axis start) (no product, no conversion instruction, no comparison on the FP64 pipe).
// alpha: cell = t / 5 (a multiply and a shift); beta: a 61-byte table in the image; elevator: three integer compares.  The weight
// is one fma, lam = fma(query, 1 / cell width, -lower breakpoint / cell width), both constants from the image (F16_FI_AX).
// What this gives (mexndinterp.c:97-143):
//   * the cell is the reference's (j, j+1) for every query strictly inside a cell, with its lambda to an ulp or two;
//   * a query ON breakpoint j is in cell j with lam = 0 up to the rounding of 1 / width (|lam| <= 5e-16), which evaluates to the
//     node value f_j like the reference's exact hit (j, j); at the top of an axis the cell is the last one and lam = 1;
//   * there is no margin anywhere: a query a relative 1e-16 above a breakpoint is in the upper cell, one below it in the lower.
// (Round 1 found the cell by rounding a scaled query shrunk by 2^-30, which put a 2^-30-wide band above every breakpoint into the
// LOWER cell with lam = 1 + delta, an extrapolation with error delta * (slope change): 9e-9 scaled at alpha = 30 deg + 1.5e-8.
// Until this version the position in cell units was formed first and rounded, five FP64 instructions per axis plus the
// comparisons that pick the piece of a piecewise-uniform axis; now two.)
F16_FD int floor_plus(double v, int shift) {  // floor(v) + shift for |v| < 2^31 - shift
#if defined(__CUDA_ARCH__)
  return __double2loint(__dadd_rd(v, 6755399441055744.0 + shift));  // 1.5 * 2^52 + shift: an ulp is 1 up there
#else
  return (int)floor(v) + shift;
#endif
}
F16_FD int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ia, i1, i2: cells on ALPHA, DH1, DH2; ib: cell on BETA1.  The clamps only matter for a query outside an axis (the callers
// exclude it): they keep the table reads inside the image.
F16_FD void locate_hifi(const double* img, double alpha, double beta, double el, int& ia, int& ib, int& i1, int& i2, double& la,
                        double& lb, double& l1, double& l2) {
  const double* ax = img + F16_FI_AX;
  ia = clampi((floor_plus(alpha, 20) * 13108) >> 16, 0, F16_FI_NAC - 1);  // t / 5 for 0 <= t <= 65; alpha = 45 is in the last cell
  la = fma(alpha, K.c0_2, ax[F16_AX_A + ia]);
  const int tb = clampi(floor_plus(beta, 30), 0, 60);
  ib = reinterpret_cast<const unsigned char*>(ax + F16_AX_LUTB)[tb];
  const d2 wb = ld2(ax + F16_AX_TB + 2 * tb);
  lb = fma(beta, wb.x, wb.y);
  const int te = floor_plus(el, 25);
  i1 = clampi((te >= 15) + (te >= 25) + (te >= 35), 0, 3);
  i2 = te >= 25;
  const d2 w1 = ld2(ax + F16_AX_D1 + 2 * i1);
  l1 = fma(el, w1.x, w1.y);
  l2 = fma(el, K.c0_04, i2 ? 0.0 : 1.0);
}

// value of table `slot` of an (f, d) node at alpha weight la
// On B200 a warp-wide LDS.128 occupies the shared-memory pipe for 2 cycles (uniform address) to 4 cycles (>= 4 distinct
// addresses per quarter-warp), an LDS.64 for 0.57 to 1.0 (tools/microbench/mb_lds.cu).  ptxas fuses the two 8-byte loads of
// a node into one 16-byte load wherever it can prove 16-byte alignment; forcing two 8-byte loads measured slower (DESIGN.md).
F16_FD double fd(const double* node, int slot, double la) { return fma(la, node[2 * slot + 1], node[2 * slot]); }
F16_FD double mix(double lam, double lo, double hi) { return fma(lam, hi - lo, lo); }

// |v| < 2^30 and not NaN, on the integer pipe
F16_FD bool small_angle(double v) { return (hi32(v) & 0x7fffffff) < 0x41d00000; }

// "all inside" form of env.py:117 + the NaN rule of step_bounds(): true when every bounded state is inside its
// closed interval (a NaN fails the comparison), no unbounded state is NaN, and (LIBM_TRIG == false) the three
// Euler angles are small enough for sincos_any().
template <bool LIBM_TRIG>
F16_FD bool step_ok(const double (&x)[18]) {
  bool ok = (x[2] >= 0.0) & (x[2] <= 100000.0);
  ok &= (x[6] >= 0.0) & (x[6] <= 900.0);
  ok &= (x[7] >= -20.0) & (x[7] <= 90.0);
  ok &= (fabs(x[8]) <= 30.0) & (fabs(x[9]) <= 300.0) & (fabs(x[10]) <= 100.0) & (fabs(x[11]) <= 50.0);
  ok &= (x[12] >= 1000.0) & (x[12] <= 19000.0);
  ok &= (fabs(x[13]) <= 25.0) & (fabs(x[14]) <= 21.5) & (fabs(x[15]) <= 30.0);
  ok &= (x[16] >= 0.0) & (x[16] <= 25.0);
  ok &= !either_nan(x[0], x[1]) & !either_nan(x[17], x[17]);
  if (LIBM_TRIG) ok &= !either_nan(x[3], x[4]) & !either_nan(x[5], x[5]);
  else ok &= small_angle(x[3]) & small_angle(x[4]) & small_angle(x[5]);
  return ok;
}

// The same question asked on the integer pipe (an FP64 compare occupies the FP64 pipe like a multiply-add and yields no flop):
// a screen on the HIGH WORDS that says "certainly inside" or "look again".  For a bound B whose low word is zero (every bound of
// parameters.py:122-123 is such a number) |v| < B <=> hi(|v|) < hi(B), and lo <= v < hi for 0 <= lo <=> hi(v) - hi(lo) < hi(hi) -
// hi(lo) as unsigned numbers.  A state ON a bound (or in its last 2^-20 relative), -0.0, an infinity and a NaN all fail the
// screen; the caller then asks step_ok(), which is exact.  true implies step_ok() for the bounded states; the three unbounded
// ones keep their NaN test and the Euler angles their small_angle().
F16_FD bool below_abs(double v, unsigned hi_bound) { return (unsigned)(hi32(v) & 0x7fffffff) < hi_bound; }
F16_FD bool in_range_pos(double v, unsigned hi_lo, unsigned hi_hi) { return (unsigned)hi32(v) - hi_lo < hi_hi - hi_lo; }
// Two more comparisons of calc_xdot_* moved off the FP64 pipe; both are exact for every value that is not a NaN (the callers'
// preconditions exclude a NaN altitude or airspeed): doubles order like their bit patterns read as signed integers as long as one
// side is positive, and 35000.0 has a zero low word.
F16_FD bool at_or_above_35000(double alt) { return hi32(alt) >= 0x40E11700; }  // nlplant.c:475
F16_FD bool at_most_0_01(double v) {                                           // nlplant.c:104
#if defined(__CUDA_ARCH__)
  return __double_as_longlong(v) <= 0x3F847AE147AE147BLL;
#else
  long long b;
  __builtin_memcpy(&b, &v, 8);
  return b <= 0x3F847AE147AE147BLL;
#endif
}
template <bool LIBM_TRIG>
F16_FD bool step_screen(const double (&x)[18]) {
  bool ok = in_range_pos(x[2], 0u, 0x40F86A00u);                                  // 0 .. 100000
  ok &= in_range_pos(x[6], 0u, 0x408C2000u);                                      // 0 .. 900
  ok &= below_abs(x[7], 0x40340000u);                                             // inside -20 .. 90: |alpha| < 20
  ok &= below_abs(x[8], 0x403E0000u) & below_abs(x[9], 0x4072C000u) & below_abs(x[10], 0x40590000u) & below_abs(x[11], 0x40490000u);
  ok &= in_range_pos(x[12], 0x408F4000u, 0x40D28E00u);                            // 1000 .. 19000
  ok &= below_abs(x[13], 0x40390000u) & below_abs(x[14], 0x40358000u) & below_abs(x[15], 0x403E0000u);
  ok &= in_range_pos(x[16], 0u, 0x40390000u);                                     // 0 .. 25
  ok &= !either_nan(x[0], x[1]) & !either_nan(x[17], x[17]);
  if (LIBM_TRIG) ok &= !either_nan(x[3], x[4]) & !either_nan(x[5], x[5]);
  else ok &= small_angle(x[3]) & small_angle(x[4]) & small_angle(x[5]);
  return ok;
}

// Preconditions of calc_xdot_hifi / calc_xdot_lofi on a state that did NOT pass the step bounds (one-shot kernels, linearise):
// no NaN in x[0..16], altitude inside the density table of half_rho (tfac in [0.28, 1.03)), Euler angles (lofi: alpha too)
// below 2^30 rad for reduce_pio2, and for hifi the elevator inside its table (calc_xdot_hifi itself checks alpha and beta).
template <int FI>
F16_FD bool fast_ok(const double (&x)[18]) {
  bool ok = (x[2] >= -4000.0) & (x[2] <= 102000.0) & small_angle(x[3]) & small_angle(x[4]) & small_angle(x[5]);
  ok &= !either_nan(x[0], x[1]) & !either_nan(x[6], x[9]) & !either_nan(x[10], x[11]) & !either_nan(x[12], x[14]) &
        !either_nan(x[15], x[16]);
  if (FI) ok &= (fabs(x[13]) <= 25.0);
  else ok &= small_angle(x[7]) & !either_nan(x[13], x[13]);
  return ok;
}

// The closed-loop law of f16_lqr_t scattered to state order by the host (make_dense_law): every selected state is a
// compile-time register here, columns that carry no gain are skipped by warp-uniform branches on `colmask`.
//     u[r] = u0[r] - extra[r] - sum_i Kf[i][r] (x[i] - xr[i])        for rows in row_mask
struct LqrDense {
  int colmask, row_mask;
  double Kf[18][4];
  double xr[18];
  double u0[4];     // u0[r] - extra[r]; extra collects the constant left by states selected more than once
};

#if defined(__CUDACC__)
__host__
#endif
static inline void make_dense_law(const LqrLaw& l, LqrDense& d) {
  d = LqrDense();
  d.row_mask = l.row_mask;
  for (int r = 0; r < 4; r++) d.u0[r] = l.u0[r];
  for (int j = 0; j < l.n_sel; j++) {
    const int i = l.sel[j];
    if (!((d.colmask >> i) & 1)) {
      d.colmask |= 1 << i;
      d.xr[i] = l.x_ref[j];
      for (int r = 0; r < 4; r++) d.Kf[i][r] = l.K[r][j];
    } else {  // K2 (x - r2) = K2 (x - r1) + K2 (r1 - r2)
      for (int r = 0; r < 4; r++) {
        d.Kf[i][r] += l.K[r][j];
        d.u0[r] -= l.K[r][j] * (d.xr[i] - l.x_ref[j]);
      }
    }
  }
}

// COLMASK != 0: the shape of the law is known at compile time (the reference's own law: gains on its nine MPC states,
// parameters.py:135, driving elevator, aileron and rudder; the thrust command stays the caller's) -- bits 0..17 the set of gain
// columns, bits 20..23 the set of driven rows.  No branch per column, so the column updates interleave, and no multiply-add (nor
// gain load) for a row that is not driven.  0: both sets are read from the law.
#define F16_LQR_MPC_COLMASK 0x30F98                              // states 3, 4, 7, 8, 9, 10, 11, 16, 17
#define F16_LQR_MPC_SHAPE (F16_LQR_MPC_COLMASK | (0xE << 20))    // ... driving rows 1, 2, 3
template <int COLMASK = 0>
F16_FD void lqr_action_dense(const LqrDense& l, const double (&x)[18], const double (&u_in)[4], double (&u)[4]) {
  constexpr int COLS = COLMASK & 0x3FFFF, ROWS = (COLMASK >> 20) & 0xF;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < 18; i++) {
    if (COLS ? ((COLS >> i) & 1) : ((l.colmask >> i) & 1)) {
      const double e = x[i] - l.xr[i];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
      for (int r = 0; r < 4; r++)
        if (!ROWS || ((ROWS >> r) & 1)) acc[r] = fma(l.Kf[i][r], e, acc[r]);
    }
  }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int r = 0; r < 4; r++) u[r] = ((ROWS ? ROWS : l.row_mask) >> r) & 1 ? (l.u0[r] - acc[r]) : u_in[r];
}

// utils.py:308-330 command saturation (loop-invariant in open loop)
F16_FD void clip_commands(const double (&u)[4], double (&uc)[4]) {
  uc[0] = clipd(u[0], 1000, 19000);
  uc[1] = clipd(u[1], -25, 25);
  uc[2] = clipd(u[2], -21.5, 21.5);
  uc[3] = clipd(u[3], -30, 30);
}

// rows 12..17 of _calc_xdot: actuator lags and the leading-edge-flap schedule, utils.py:289-330.  atmos_out = 9.05 qbar / ps of
// atmos(alt, x[6]) and alpha_deg come from the caller (calc_xdot_hifi / _lofi compute them from their shared reciprocal).
F16_FD void actuator_rows(const double (&x)[18], const double (&uc)[4], double atmos_out, double alpha_deg, double (&xd)[18]) {
  const double lf_in = fma(2.0, alpha_deg, x[17]);
  // flap command saturation (utils.py:297): active in ordinary flight (the trim flap angle is 0.4 deg), so a select
  const double lef_cmd = clipd(fma(lf_in, K.c1_38, K.c1_45) - atmos_out, 0, 25);
  const double r12 = uc[0] - x[12], r13 = K.c20_2 * (uc[1] - x[13]), r14 = K.c20_2 * (uc[2] - x[14]),
               r15 = K.c20_2 * (uc[3] - x[15]), r16 = K.inv0_136 * (lef_cmd - x[16]);
  xd[12] = r12;
  xd[13] = r13;
  xd[14] = r14;
  xd[15] = r15;
  xd[16] = r16;
  // rate limits (utils.py:299-330) only cost selects when one of them is active (or a value is NaN)
  // asked on the integer pipe like step_screen(): |r| < B <=> hi(|r|) < hi(B) for a bound whose low word is zero; a rate ON its
  // limit, beyond it or NaN takes the exact clips
  if (!(below_abs(r12, 0x40C38800u) & below_abs(r13, 0x404E0000u) & below_abs(r14, 0x40540000u) & below_abs(r15, 0x405E0000u) &
        below_abs(r16, 0x40390000u))) {
    xd[12] = clipd(r12, -10000, 10000);
    xd[13] = clipd(r13, -60, 60);
    xd[14] = clipd(r14, -80, 80);
    xd[15] = clipd(r15, -120, 120);
    xd[16] = clipd(r16, -25, 25);
  }
  xd[17] = (alpha_deg - lf_in) * 7.25;
}

// rows 12..17 of Nlplant's output (nlplant.c:445-450): accels (:512-552, grav = 32.174 and the unclamped velocity v6), then
// mach = vt / sqrt(1.4 * 1716.3 * temp), qbar, ps = 1715 rho temp (:479-485) from the clamped vt.  xd[6..8] are read.
F16_FD void nlplant_extra_rows(double v6, double vt, double sa, double ca, double sb, double cb, double st, double ct,
                               double sphi, double cphi, double P, double Q, double R, double qbar, double hrho, double temp,
                               double inv_temp, double (&xd)[18]) {
  const double inv_grav = 1.0 / 32.174;
  const double vcb = v6 * cb;
  const double vel_u = vcb * ca, vel_v = v6 * sb, vel_w = vcb * sa;
  const double u_dot = fma(cb * ca, xd[6], -fma(vel_v * ca, xd[8], vel_w * xd[7]));
  const double v_dot = fma(sb, xd[6], vcb * xd[8]);
  const double w_dot = fma(cb * sa, xd[6], fma(vel_u, xd[7], -(vel_v * sa) * xd[8]));
  xd[12] = fma(inv_grav, fma(Q, vel_w, fma(-R, vel_v, u_dot)), st);
  xd[13] = fma(inv_grav, fma(R, vel_u, fma(-P, vel_w, v_dot)), -(ct * sphi));
  xd[14] = fma(-inv_grav, fma(P, vel_v, fma(-Q, vel_u, w_dot)), ct * cphi);
  xd[15] = vt * sqrt(inv_temp * (1.0 / (1.4 * 1716.3)));
  xd[16] = qbar;
  const double ps = (3430.0 * hrho) * temp;  // hrho = 0.5 rho
  xd[17] = ps == 0.0 ? 1715.0 : ps;
}

// ------------------------------------------------------------------------------------------------------
// env.py::_calc_xdot (env.py:65-103) for the hifi model, all 18 derivatives.  `img` is the fast image, `uc` the
// saturated commands.  Precondition (checked by the caller through step_ok): states inside parameters.py bounds,
// no NaN.  Returns false when alpha / beta leave the hifi tables (the caller then reports the exact status word).
// ------------------------------------------------------------------------------------------------------
// NLP = true turns the function into Nlplant itself (nlplant.c:23-457): x[0..16] is xu (x[16] the flap angle, x[17] unused),
// `uc` is not read, and rows 12..17 are nx, ny, nz (accels, nlplant.c:512-552), mach, qbar, ps instead of the actuator rows.
// AUX = true also returns aux = {qbar/ps term of the flap schedule, alpha in degrees}: what actuator_rows() needs to re-evaluate
// rows 12..17 alone (linearise: the columns lf1 and the four inputs reach f through those rows only).
template <bool LIBM_TRIG, bool NLP = false, bool AUX = false>
F16_FD bool calc_xdot_hifi(const double* img, const double (&x)[18], const double (&uc)[4], double xcg, double (&xd)[18],
                           double* aux = nullptr) {
  const double B = 30.0, S = 300.0, cbar = 11.32, xcgr = K.c0_35;

  const double alpha = x[7] * K.r2d, beta = x[8] * K.r2d, el = x[13];
  // hifi_envelope(): the elevator range is already guaranteed by the |x[13]| <= 25 bound
  if (!((alpha >= -20.0) & (alpha <= 45.0) & (fabs(beta) <= 30.0))) return false;

  double la, lb, l1, l2;
  int ia, ib, i1, i2;
  locate_hifi(img, alpha, beta, el, ia, ib, i1, i2, la, lb, l1, l2);

  double sa, ca, sb, cb, st, ct, sphi, cphi, spsi, cpsi;
  sincos_quarter(x[7], sa, ca);
  sincos_quarter(x[8], sb, cb);
  if (LIBM_TRIG) {
    sincos_libm(x[4], &st, &ct);
    sincos_libm(x[3], &sphi, &cphi);
    sincos_libm(x[5], &spsi, &cpsi);
  } else {
    double r4, r3, r5;
    const int q4 = reduce_pio2(x[4], r4), q3 = reduce_pio2(x[3], r3), q5 = reduce_pio2(x[5], r5);
    sincos_quarter(r4, st, ct);
    sincos_quarter(r3, sphi, cphi);
    sincos_quarter(r5, spsi, cpsi);
    if (((q4 | q3 | q5) & 3) != 0) {  // some angle outside [-pi/4, pi/4]: swap / negate per quadrant
      quadrant_fix(q4, st, ct);
      quadrant_fix(q3, sphi, cphi);
      quadrant_fix(q5, spsi, cpsi);
    }
  }

  double vt = x[6];
  if (at_most_0_01(vt)) vt = K.c0_01;  // nlplant.c:104
  const double P = x[9], Q = x[10], R = x[11], T = x[12];

  // atmos, nlplant.c:467-490: only qbar (Nlplant) and qbar/ps (upd_lef, utils.py:291-296) are consumed here
  const double tfac = fma(K.tlapse, x[2], 1.0);
  const double temp = at_or_above_35000(x[2]) ? 390.0 : 519.0 * tfac;
  const double hrho = half_rho(img, tfac);
  const double qbar = hrho * (vt * vt);
  // one reciprocal for 1/(vt cb), 1/vt, 1/ct and 1/temp
  const double vc = vt * cb, tc = ct * temp;
  const double rr = rcp_nr(vc * tc);
  const double inv_vc = rr * tc, inv_tc = rr * vc;
  const double inv_vt = inv_vc * cb, inv_ct = inv_tc * temp, inv_temp = inv_tc * ct;

  const double dail = x[14] * K.inv21_5, drud = x[15] * K.inv30;  // nlplant.c:123-124
  const double dlef = fma(x[16], K.ninv25, 1.0);                    // nlplant.c:125

  // navigation + kinematics, nlplant.c:148-176
  const double U = vc * ca, V = vt * sb, W = vc * sa;
  {
    const double sphi_cpsi = sphi * cpsi, cphi_spsi = cphi * spsi, sphi_spsi = sphi * spsi, cphi_cpsi = cphi * cpsi,
                 cphi_st = cphi * st;
    xd[0] = fma(U, ct * cpsi, fma(V, fma(sphi_cpsi, st, -cphi_spsi), W * fma(cphi_st, cpsi, sphi_spsi)));
    xd[1] = fma(U, ct * spsi, fma(V, fma(sphi_spsi, st, cphi_cpsi), W * fma(cphi_st, spsi, -sphi_cpsi)));
    xd[2] = fma(U, st, -fma(V, sphi * ct, W * (cphi * ct)));
  }
  const double qr = fma(Q, sphi, R * cphi);
  xd[3] = fma(st * inv_ct, qr, P);
  xd[4] = fma(Q, cphi, -(R * sphi));
  xd[5] = qr * inv_ct;

  // weights of the damping terms, nlplant.c:333-377
  const double qQ = K.half_cbar * inv_vt * Q, bR = (0.5 * B) * inv_vt * R, bP = (0.5 * B) * inv_vt * P;

  double Cx_tot, Cz_tot, Cm_tot, Cy_tot, Cn_tot, Cl_tot;
  double dCz_lef;

  // ---- alpha x beta group: the delta coefficients of hifi_C_lef, hifi_rudder, hifi_ailerons (hifi:1892-1926),
  //      tabulated at the nodes, weighted per nlplant.c:333-377 before the beta interpolation ----
  {
    const double w_al = dail * dlef;  // weight of delta_C*_a20_lef
    const double* n0 = img + F16_FI_G2 + (ib * F16_FI_NAC + ia) * F16_FI_G2_STRIDE;
    const double* n1 = n0 + F16_FI_NAC * F16_FI_G2_STRIDE;
    double dx[2], dz[2], dm[2], y[2], n[2], l[2];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 2; k++) {
      const double* p = k ? n1 : n0;
      dx[k] = fd(p, FG2_dCx_lef, la);
      dz[k] = fd(p, FG2_dCz_lef, la);
      dm[k] = fd(p, FG2_dCm_lef, la);
      double a = fma(fd(p, FG2_dCy_lef, la), dlef, fd(p, FG2_Cy, la));
      a = fma(fd(p, FG2_dCy_a20, la), dail, a);
      a = fma(fd(p, FG2_dCy_a20_lef, la), w_al, a);
      y[k] = fma(fd(p, FG2_dCy_r30, la), drud, a);
      a = fd(p, FG2_dCn_lef, la) * dlef;
      a = fma(fd(p, FG2_dCn_a20, la), dail, a);
      a = fma(fd(p, FG2_dCn_a20_lef, la), w_al, a);
      n[k] = fma(fd(p, FG2_dCn_r30, la), drud, a);
      a = fd(p, FG2_dCl_lef, la) * dlef;
      a = fma(fd(p, FG2_dCl_a20, la), dail, a);
      a = fma(fd(p, FG2_dCl_a20_lef, la), w_al, a);
      l[k] = fma(fd(p, FG2_dCl_r30, la), drud, a);
    }
    dCz_lef = mix(lb, dz[0], dz[1]);
    Cx_tot = mix(lb, dx[0], dx[1]) * dlef;
    Cm_tot = mix(lb, dm[0], dm[1]) * dlef;
    Cy_tot = mix(lb, y[0], y[1]);
    Cn_tot = mix(lb, n[0], n[1]);
    Cl_tot = mix(lb, l[0], l[1]);
  }
  // ---- alpha x beta x DH2: Cn, Cl (hifi:1876-1877) ----
  {
    const double* p = img + F16_FI_G3B + ((i2 * F16_N_B + ib) * F16_FI_NAC + ia) * F16_FI_G3B_STRIDE;
    const int sb_ = F16_FI_NAC * F16_FI_G3B_STRIDE, sd = F16_N_B * F16_FI_NAC * F16_FI_G3B_STRIDE;
    const double n_lo = mix(lb, fd(p, 0, la), fd(p + sb_, 0, la)), n_hi = mix(lb, fd(p + sd, 0, la), fd(p + sd + sb_, 0, la));
    const double l_lo = mix(lb, fd(p, 1, la), fd(p + sb_, 1, la)), l_hi = mix(lb, fd(p + sd, 1, la), fd(p + sd + sb_, 1, la));
    Cn_tot += mix(l2, n_lo, n_hi);
    Cl_tot += mix(l2, l_lo, l_hi);
  }
  // ---- alpha x beta x DH1: Cx, Cz, Cm (hifi:1872-1874) and eta_el (hifi:1932) ----
  double Cm3;
  {
    const double* p = img + F16_FI_G3A + ((i1 * F16_N_B + ib) * F16_FI_NAC + ia) * F16_FI_G3A_STRIDE;
    const int sb_ = F16_FI_NAC * F16_FI_G3A_STRIDE, sd = F16_N_B * F16_FI_NAC * F16_FI_G3A_STRIDE;
    const double x_lo = mix(lb, fd(p, 0, la), fd(p + sb_, 0, la)), x_hi = mix(lb, fd(p + sd, 0, la), fd(p + sd + sb_, 0, la));
    const double z_lo = mix(lb, fd(p, 1, la), fd(p + sb_, 1, la)), z_hi = mix(lb, fd(p + sd, 1, la), fd(p + sd + sb_, 1, la));
    const double m_lo = mix(lb, fd(p, 2, la), fd(p + sb_, 2, la)), m_hi = mix(lb, fd(p + sd, 2, la), fd(p + sd + sb_, 2, la));
    Cx_tot += mix(l1, x_lo, x_hi);
    Cz_tot = fma(dCz_lef, dlef, mix(l1, z_lo, z_hi));
    Cm3 = mix(l1, m_lo, m_hi);
    const d2 e = ld2(img + F16_FI_ETA + 2 * i1);
    Cm3 *= fma(l1, e.y, e.x);
  }
  // ---- alpha-only group: damping, lef damping, other (hifi:1880-1890,1901-1911,1928-1934) ----
  {
    const double* p = img + F16_FI_G1 + ia * F16_FI_G1_STRIDE;
    Cx_tot = fma(qQ, fma(fd(p, FG1_dCxq_lef, la), dlef, fd(p, FG1_Cxq, la)), Cx_tot);
    // nlplant.c:339 uses delta_Cz_lef where delta_Czq_lef was meant -- reproduced
    Cz_tot = fma(qQ, fma(dCz_lef, dlef, fd(p, FG1_Czq, la)), Cz_tot);
    Cm_tot += Cm3 + fd(p, FG1_dCm, la);
    Cm_tot = fma(qQ, fma(fd(p, FG1_dCmq_lef, la), dlef, fd(p, FG1_Cmq, la)), Cm_tot);
    Cm_tot = fma(Cz_tot, xcgr - xcg, Cm_tot);
    Cy_tot = fma(bR, fma(fd(p, FG1_dCyr_lef, la), dlef, fd(p, FG1_Cyr, la)), Cy_tot);
    Cy_tot = fma(bP, fma(fd(p, FG1_dCyp_lef, la), dlef, fd(p, FG1_Cyp, la)), Cy_tot);
    Cn_tot = fma(bR, fma(fd(p, FG1_dCnr_lef, la), dlef, fd(p, FG1_Cnr, la)), Cn_tot);
    Cn_tot = fma(bP, fma(fd(p, FG1_dCnp_lef, la), dlef, fd(p, FG1_Cnp, la)), Cn_tot);
    Cn_tot = fma(fd(p, FG1_dCnbeta, la), beta, Cn_tot);
    Cn_tot = fma(Cy_tot, (xcg - xcgr) * K.xcg_arm, Cn_tot);
    Cl_tot = fma(bR, fma(fd(p, FG1_dClr_lef, la), dlef, fd(p, FG1_Clr, la)), Cl_tot);
    Cl_tot = fma(bP, fma(fd(p, FG1_dClp_lef, la), dlef, fd(p, FG1_Clp, la)), Cl_tot);
    Cl_tot = fma(fd(p, FG1_dClbeta, la), beta, Cl_tot);
  }

  // body-axis accelerations, nlplant.c:383-387
  const double qS_m = qbar * K.S_m;
  const double gct = K.g * ct;
  const double Udot = fma(T, K.inv_m, fma(qS_m, Cx_tot, fma(-K.g, st, fma(R, V, -(Q * W)))));
  const double Vdot = fma(qS_m, Cy_tot, fma(gct, sphi, fma(P, W, -(R * U))));
  const double Wdot = fma(qS_m, Cz_tot, fma(gct, cphi, fma(Q, U, -(P * V))));
  // nlplant.c:393-405 with U = vt ca cb, V = vt sb, W = vt sa cb substituted (vt cancels)
  const double vtd = fma(ca * cb, Udot, fma(sb, Vdot, (sa * cb) * Wdot));
  xd[6] = vtd;
  xd[7] = fma(ca, Wdot, -(sa * Udot)) * inv_vc;
  xd[8] = fma(-sb, vtd, Vdot) * inv_vc;

  // moments, nlplant.c:413-436 (Heng = 0), inertia ratios folded into constants
  const double qSb = qbar * (S * B);
  const double L_tot = Cl_tot * qSb, N_tot = Cn_tot * qSb, M_tot = Cm_tot * (qbar * (S * cbar));
  const double PQ = P * Q, QR = Q * R;
  xd[9] = fma(K.ixx_l, L_tot, fma(K.ixx_n, N_tot, fma(K.ixx_qr, QR, K.ixx_pq * PQ)));
  xd[10] = fma(K.inv_Jy, M_tot, fma(K.iyy_pr, P * R, K.iyy_p2 * fma(P, P, -(R * R))));
  xd[11] = fma(K.izz_n, N_tot, fma(K.izz_l, L_tot, fma(K.izz_pq, PQ, K.izz_qr * QR)));

  if (NLP) {  // accels (grav = 32.174, the UNCLAMPED x[6]) and the three atmosphere outputs, nlplant.c:445-450,467-490,512-552
    nlplant_extra_rows(x[6], vt, sa, ca, sb, cb, st, ct, sphi, cphi, P, Q, R, qbar, hrho, temp, inv_temp, xd);
    return true;
  }
  // actuators and leading-edge flap, utils.py:289-330.  qbar/ps of atmos(alt, x[6]) = 0.5 x6^2 / (1715 temp)
  const double atmos_out = (x[6] * x[6]) * inv_temp * K.lef_q;
  // utils.py:292 forms x[7] * 180 / pi; x[7] * (180 / pi) is the same angle to two ulp, but a forward difference of the flap rate
  // over eps = 1e-5 turns two ulp of a 20-degree alpha into 1.4e-8 of dA[16][7] (measured on the cfg-4 grid): keep the first product
  const double alpha_deg = (x[7] * 180.0) * K.inv_pi;
  actuator_rows(x, uc, atmos_out, alpha_deg, xd);
  if (AUX) { aux[0] = atmos_out; aux[1] = alpha_deg; }
  return true;
}

// ------------------------------------------------------------------------------------------------------
// Parity probe of the fast image and cell search (f16_fast_probe; never on the step path): the 44 coefficient outputs of
// the reference's aggregators (hifi:1871-1934) in the order of f16_hifi_probe, evaluated the way calc_xdot_hifi evaluates
// them -- locate_hifi, (f, d) gathers, alpha then beta then elevator -- but one table at a time, so that every table of the
// image and every cell decision can be compared with the reference accessors and getHyperCube.  Slot 24 (delta_CZq_lef)
// is not in the fast image (nlplant.c:339 never uses it) and slot 43 (delta_Cm_ds) is the constant 0: both return 0.
// cells = {ia, ib, i1, i2}, lam = {la, lb, l1, l2}.
// ------------------------------------------------------------------------------------------------------
F16_FD void probe_hifi(const double* img, double alpha, double beta, double el, double (&o)[44], int (&cells)[4],
                       double (&lam)[4]) {
  double la, lb, l1, l2;
  int ia, ib, i1, i2;
  locate_hifi(img, alpha, beta, el, ia, ib, i1, i2, la, lb, l1, l2);
  cells[0] = ia; cells[1] = ib; cells[2] = i1; cells[3] = i2;
  lam[0] = la; lam[1] = lb; lam[2] = l1; lam[3] = l2;
  for (int i = 0; i < 44; i++) o[i] = 0.0;
  {
    const double* p = img + F16_FI_G3A + ((i1 * F16_N_B + ib) * F16_FI_NAC + ia) * F16_FI_G3A_STRIDE;
    const int sb_ = F16_FI_NAC * F16_FI_G3A_STRIDE, sd = F16_N_B * F16_FI_NAC * F16_FI_G3A_STRIDE;
    for (int t = 0; t < 3; t++)  // Cx, Cz, Cm
      o[t] = mix(l1, mix(lb, fd(p, t, la), fd(p + sb_, t, la)), mix(lb, fd(p + sd, t, la), fd(p + sd + sb_, t, la)));
    const d2 e = ld2(img + F16_FI_ETA + 2 * i1);
    o[42] = fma(l1, e.y, e.x);
  }
  {
    const double* p = img + F16_FI_G3B + ((i2 * F16_N_B + ib) * F16_FI_NAC + ia) * F16_FI_G3B_STRIDE;
    const int sb_ = F16_FI_NAC * F16_FI_G3B_STRIDE, sd = F16_N_B * F16_FI_NAC * F16_FI_G3B_STRIDE;
    for (int t = 0; t < 2; t++)  // Cn, Cl
      o[4 + t] = mix(l2, mix(lb, fd(p, t, la), fd(p + sb_, t, la)), mix(lb, fd(p + sd, t, la), fd(p + sd + sb_, t, la)));
  }
  {
    const double* n0 = img + F16_FI_G2 + (ib * F16_FI_NAC + ia) * F16_FI_G2_STRIDE;
    const double* n1 = n0 + F16_FI_NAC * F16_FI_G2_STRIDE;
    // f16_hifi_probe slot of each FG2 table
    const int dst[FG2_COUNT] = {15, 16, 17, 3, 18, 33, 34, 30, 19, 35, 36, 31, 20, 37, 38, 32};
    for (int t = 0; t < FG2_COUNT; t++) o[dst[t]] = mix(lb, fd(n0, t, la), fd(n1, t, la));
  }
  {
    const double* p = img + F16_FI_G1 + ia * F16_FI_G1_STRIDE;
    // FG1 order: Cxq dCxq_lef Czq Cmq dCmq_lef dCm Cyr dCyr_lef Cyp dCyp_lef Cnr dCnr_lef Cnp dCnp_lef dCnbeta Clr dClr_lef Clp dClp_lef dClbeta
    const int dst[FG1_COUNT] = {6, 21, 9, 12, 27, 41, 7, 22, 8, 23, 13, 28, 14, 29, 39, 10, 25, 11, 26, 40};
    for (int t = 0; t < FG1_COUNT; t++) o[dst[t]] = fd(p, t, la);
  }
}

// ------------------------------------------------------------------------------------------------------
// The lofi (Stevens-Lewis) model on the same arithmetic: env.py::_calc_xdot with fi_flag = 0.  `img` is the 7 KB lofi
// step image: the lofi tables of f16_tables.h (F16_LOFI_*, 792 doubles) followed by the 48 x 2 centre table of
// half_rho().  Look-ups as lofi_F16_AeroData.c:12-368 (5-degree alpha grid with linear extrapolation, |beta| grid 0:5:30,
// elevator grid -24:12:24), totals as nlplant.c:258-286,333-377 with every leading-edge-flap term zero (:256,295-319).
// alpha is not confined to the hifi tables here, so it takes the reduced sincos like the Euler angles.
// The prologue (trig, atmosphere, reciprocals, kinematics) and the epilogue (accelerations, moments, actuators) repeat
// calc_xdot_hifi's on purpose: the hifi function is the headline kernel's loop body, and its schedule (168 registers, no
// spills, 64 % of the FP64 peak) does not survive being cut into shared pieces -- ptxas is that sensitive here (DESIGN.md 7).
// ------------------------------------------------------------------------------------------------------
#define F16_LOFI_STEP_IMG_DOUBLES (F16_IMG_LOFI_DOUBLES + 2 * F16_FI_NPOW)

struct LofiA {
  int k, L;    // zero-based columns of the two alpha neighbours
  double ada;  // |alpha / 5 - k|
};
F16_FD double lrow(const double* row, const LofiA& A) {
  const double lo = row[A.k];
  return fma(A.ada, row[A.L] - lo, lo);
}

template <bool LIBM_TRIG, bool NLP = false, bool AUX = false>
F16_FD bool calc_xdot_lofi(const double* img, const double (&x)[18], const double (&uc)[4], double xcg, double (&xd)[18],
                           double* aux = nullptr) {
  const double B = 30.0, S = 300.0, cbar = 11.32, xcgr = K.c0_35;
  const double alpha = x[7] * K.r2d, beta = x[8] * K.r2d, el = x[13];
  if (!(fabs(beta) <= 30.0)) return false;  // lofi_envelope(): dmomdcon indexes past its arrays beyond 30 deg

  double sa, ca, sb, cb, st, ct, sphi, cphi, spsi, cpsi;
  sincos_quarter(x[8], sb, cb);
  if (LIBM_TRIG) {
    sincos_libm(x[7], &sa, &ca);
    sincos_libm(x[4], &st, &ct);
    sincos_libm(x[3], &sphi, &cphi);
    sincos_libm(x[5], &spsi, &cpsi);
  } else {
    double r7, r4, r3, r5;
    const int q7 = reduce_pio2(x[7], r7), q4 = reduce_pio2(x[4], r4), q3 = reduce_pio2(x[3], r3), q5 = reduce_pio2(x[5], r5);
    sincos_quarter(r7, sa, ca);
    sincos_quarter(r4, st, ct);
    sincos_quarter(r3, sphi, cphi);
    sincos_quarter(r5, spsi, cpsi);
    if (((q7 | q4 | q3 | q5) & 3) != 0) {
      quadrant_fix(q7, sa, ca);
      quadrant_fix(q4, st, ct);
      quadrant_fix(q3, sphi, cphi);
      quadrant_fix(q5, spsi, cpsi);
    }
  }

  double vt = x[6];
  if (at_most_0_01(vt)) vt = K.c0_01;  // nlplant.c:104
  const double P = x[9], Q = x[10], R = x[11], T = x[12];
  const double tfac = fma(K.tlapse, x[2], 1.0);
  const double temp = at_or_above_35000(x[2]) ? 390.0 : 519.0 * tfac;
  const double hrho = half_rho(img + F16_IMG_LOFI_DOUBLES - F16_FI_POW, tfac);
  const double qbar = hrho * (vt * vt);
  const double vc = vt * cb, tc = ct * temp;
  const double rr = rcp_nr(vc * tc);
  const double inv_vc = rr * tc, inv_tc = rr * vc;
  const double inv_vt = inv_vc * cb, inv_ct = inv_tc * temp, inv_temp = inv_tc * ct;
  const double dail = x[14] * K.inv21_5, drud = x[15] * K.inv30;

  // navigation + kinematics, nlplant.c:148-176
  const double U = vc * ca, V = vt * sb, W = vc * sa;
  {
    const double sphi_cpsi = sphi * cpsi, cphi_spsi = cphi * spsi, sphi_spsi = sphi * spsi, cphi_cpsi = cphi * cpsi,
                 cphi_st = cphi * st;
    xd[0] = fma(U, ct * cpsi, fma(V, fma(sphi_cpsi, st, -cphi_spsi), W * fma(cphi_st, cpsi, sphi_spsi)));
    xd[1] = fma(U, ct * spsi, fma(V, fma(sphi_spsi, st, cphi_cpsi), W * fma(cphi_st, spsi, -sphi_cpsi)));
    xd[2] = fma(U, st, -fma(V, sphi * ct, W * (cphi * ct)));
  }
  const double qr = fma(Q, sphi, R * cphi);
  xd[3] = fma(st * inv_ct, qr, P);
  xd[4] = fma(Q, cphi, -(R * sphi));
  xd[5] = qr * inv_ct;
  const double qQ = K.half_cbar * inv_vt * Q, bR = (0.5 * B) * inv_vt * R, bP = (0.5 * B) * inv_vt * P;

  // ---- look-ups ----
  LofiA A;
  {
    const double s = 0.2 * alpha;  // lofi:31-45
    int k = (int)s;                // fix(): truncation toward zero
    k = k <= -2 ? -1 : (k >= 9 ? 8 : k);
    const double da = s - (double)k;
    A.L = k + ((da > 0) - (da < 0)) + 2;
    A.k = k + 2;
    A.ada = fabs(da);
  }
  const double ab = 0.2 * fabs(beta);
  const int mb = (int)ab;  // 0..6
  double Cl_tot, Cn_tot;
  {  // dmomdcon (lofi:59-183): rows m, m + 1 of ALA, ALR, ANA, ANR
    const int m = mb >= 7 ? 6 : mb;
    const double db = ab - (double)m;
    double r[4];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int t = 0; t < 4; t++) {
      const double* Tt = img + F16_LOFI_DMOM + t * 96 + m * 12;
      const double v = lrow(Tt, A);
      r[t] = fma(db, lrow(Tt + 12, A) - v, v);
    }
    Cl_tot = fma(r[1], drud, r[0] * dail);  // dCl_a20 dail + dCl_r30 drud, nlplant.c:270-273,370-377
    Cn_tot = fma(r[3], drud, r[2] * dail);
  }
  {  // clcn (lofi:185-262), odd in beta
    const int m = mb == 0 ? 1 : (mb >= 6 ? 5 : mb);
    const double db = ab - (double)m;
    const int n = m + ((db > 0) - (db < 0));
    const double adb = fabs(db);
    const double* TL = img + F16_LOFI_CLCN;
    const double* TN = TL + 84;
    double v = lrow(TL + m * 12, A);
    const double cl = fma(adb, lrow(TL + n * 12, A) - v, v);
    v = lrow(TN + m * 12, A);
    const double cn = fma(adb, lrow(TN + n * 12, A) - v, v);
    const bool neg = beta < 0.0, zero = beta == 0.0;
    Cl_tot += zero ? 0.0 : (neg ? -cl : cl);
    Cn_tot += zero ? 0.0 : (neg ? -cn : cn);
  }
  double Cx_tot, Cm_tot;
  {  // cxcm (lofi:265-336)
    const double s = el * (1.0 / 12.0);
    int m = (int)s;
    m = m <= -2 ? -1 : (m >= 2 ? 1 : m);
    const double de = s - (double)m;
    const int n = m + ((de > 0) - (de < 0)) + 2;
    m += 2;
    const double ade = fabs(de);
    const double* TX = img + F16_LOFI_CXCM;
    const double* TM = TX + 60;
    double v = lrow(TX + m * 12, A);
    Cx_tot = fma(ade, lrow(TX + n * 12, A) - v, v);
    v = lrow(TM + m * 12, A);
    Cm_tot = fma(ade, lrow(TM + n * 12, A) - v, v);
  }
  // cz (lofi:339-368) and Cy (nlplant.c:283)
  const double b573 = beta * (1.0 / 57.3);
  double Cz_tot = fma(lrow(img + F16_LOFI_CZ, A), fma(-b573, b573, 1.0), -(0.19 / 25.0) * el);
  double Cy_tot = fma(0.086, drud, fma(0.021, dail, -0.02 * beta));
  {  // damping (lofi:12-56), nlplant.c:333-377 with dlef = 0
    const double* D = img + F16_LOFI_DAMP;
    Cx_tot = fma(qQ, lrow(D + 0 * 12, A), Cx_tot);
    Cz_tot = fma(qQ, lrow(D + 3 * 12, A), Cz_tot);
    Cm_tot = fma(qQ, lrow(D + 6 * 12, A), Cm_tot);
    Cm_tot = fma(Cz_tot, xcgr - xcg, Cm_tot);
    Cy_tot = fma(bR, lrow(D + 1 * 12, A), Cy_tot);
    Cy_tot = fma(bP, lrow(D + 2 * 12, A), Cy_tot);
    Cn_tot = fma(bR, lrow(D + 7 * 12, A), Cn_tot);
    Cn_tot = fma(bP, lrow(D + 8 * 12, A), Cn_tot);
    Cn_tot = fma(Cy_tot, (xcg - xcgr) * K.xcg_arm, Cn_tot);
    Cl_tot = fma(bR, lrow(D + 4 * 12, A), Cl_tot);
    Cl_tot = fma(bP, lrow(D + 5 * 12, A), Cl_tot);
  }

  // body-axis accelerations, nlplant.c:383-387
  const double qS_m = qbar * K.S_m;
  const double gct = K.g * ct;
  const double Udot = fma(T, K.inv_m, fma(qS_m, Cx_tot, fma(-K.g, st, fma(R, V, -(Q * W)))));
  const double Vdot = fma(qS_m, Cy_tot, fma(gct, sphi, fma(P, W, -(R * U))));
  const double Wdot = fma(qS_m, Cz_tot, fma(gct, cphi, fma(Q, U, -(P * V))));
  const double vtd = fma(ca * cb, Udot, fma(sb, Vdot, (sa * cb) * Wdot));
  xd[6] = vtd;
  xd[7] = fma(ca, Wdot, -(sa * Udot)) * inv_vc;
  xd[8] = fma(-sb, vtd, Vdot) * inv_vc;

  // moments, nlplant.c:413-436 (Heng = 0)
  const double qSb = qbar * (S * B);
  const double L_tot = Cl_tot * qSb, N_tot = Cn_tot * qSb, M_tot = Cm_tot * (qbar * (S * cbar));
  const double PQ = P * Q, QR = Q * R;
  xd[9] = fma(K.ixx_l, L_tot, fma(K.ixx_n, N_tot, fma(K.ixx_qr, QR, K.ixx_pq * PQ)));
  xd[10] = fma(K.inv_Jy, M_tot, fma(K.iyy_pr, P * R, K.iyy_p2 * fma(P, P, -(R * R))));
  xd[11] = fma(K.izz_n, N_tot, fma(K.izz_l, L_tot, fma(K.izz_pq, PQ, K.izz_qr * QR)));

  if (NLP) {
    nlplant_extra_rows(x[6], vt, sa, ca, sb, cb, st, ct, sphi, cphi, P, Q, R, qbar, hrho, temp, inv_temp, xd);
    return true;
  }
  // actuators and leading-edge flap, utils.py:289-330 (the flap states evolve in the lofi model too; Nlplant ignores them)
  const double atmos_out = (x[6] * x[6]) * inv_temp * K.lef_q;
  // utils.py:292 forms x[7] * 180 / pi; x[7] * (180 / pi) is the same angle to two ulp, but a forward difference of the flap rate
  // over eps = 1e-5 turns two ulp of a 20-degree alpha into 1.4e-8 of dA[16][7] (measured on the cfg-4 grid): keep the first product
  const double alpha_deg = (x[7] * 180.0) * K.inv_pi;
  actuator_rows(x, uc, atmos_out, alpha_deg, xd);
  if (AUX) { aux[0] = atmos_out; aux[1] = alpha_deg; }
  return true;
}

// K fused Euler steps of env.py::step from step k; stops (k < K on return) at the first state that fails step_ok or
// leaves the tables.  The state is not advanced on the failing step.
// The bound check of env.py:117 -- the reference exit()s there; we freeze this aircraft -- is asked about the NEW state at the
// bottom of the loop body (integer screen first, the exact comparison only for a state the screen is not sure about): its ~40
// integer instructions sit in the same basic block as the FP64 tail of the step that produced the state and issue in its
// shadow, instead of forming a block of their own at the top.  The state after the last step is screened for nothing.
template <bool LQR, bool LIBM_TRIG, int FI = 1, int COLMASK = 0>
F16_FD int run_steps(const double* img, double (&x)[18], const double (&u_in)[4], const LqrDense* lqr, double xcg, double dt,
                     int k, int K) {
  double uc[4];
  if (!LQR) clip_commands(u_in, uc);
  if (k >= K) return k;
  bool ok = step_screen<LIBM_TRIG>(x);
  if (!ok) ok = step_ok<LIBM_TRIG>(x);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
  while (ok) {
    double xd[18];
    if (LQR) {
      double u[4];
      lqr_action_dense<COLMASK>(*lqr, x, u_in, u);
      clip_commands(u, uc);
    }
    if (!(FI ? calc_xdot_hifi<LIBM_TRIG>(img, x, uc, xcg, xd) : calc_xdot_lofi<LIBM_TRIG>(img, x, uc, xcg, xd))) break;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < 18; i++) x[i] = fma(xd[i], dt, x[i]);  // env.py:126
    k++;
    ok = step_screen<LIBM_TRIG>(x);
    if (!ok) ok = step_ok<LIBM_TRIG>(x);
    ok &= k < K;
  }
  return k;
}

template <int FI = 1>
F16_FD unsigned exact_status(const double (&x)[18], const double (&u_in)[4]) {
  unsigned st = step_bounds(x, u_in);
  const double a = x[7] * (180.0 / 3.141592653589793), b = x[8] * (180.0 / 3.141592653589793);
  if (!st) st = FI ? hifi_envelope(a, b, x[13]) : lofi_envelope(a, b, x[13]);
  return st;
}

// the whole step_batch semantics for one aircraft: returns the status word, k = steps taken
template <bool LQR, int FI = 1, int COLMASK = 0>
F16_FD unsigned step_aircraft(const double* img, double (&x)[18], const double (&u_in)[4], const LqrDense* lqr, double xcg,
                              double dt, int K, int& k) {
  k = 0;
  if (either_nan(u_in[0], u_in[1]) || either_nan(u_in[2], u_in[3])) return K > 0 ? step_bounds(x, u_in) : 0u;
  k = run_steps<LQR, false, FI, COLMASK>(img, x, u_in, lqr, xcg, dt, 0, K);
  if (k == K) return 0u;
  unsigned st = exact_status<FI>(x, u_in);  // stopped early: the exact status word of the frozen state
  if (st) return st;
  // none of the reference's stop conditions: an Euler angle beyond 2^30 rad -- carry on with libm's trig
  k = run_steps<LQR, true, FI, COLMASK>(img, x, u_in, lqr, xcg, dt, k, K);
  return k == K ? 0u : exact_status<FI>(x, u_in);
}

}  // namespace fastmath
}  // namespace f16

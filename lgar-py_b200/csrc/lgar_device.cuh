// =====================================================================================
// lgar_device.cuh -- device-side LGAR column physics for sm_100a (fp64).
//
// One THREAD owns one soil column; one WARP owns a tile of 32 columns.  The variable-length
// wetting-front list of every column lives in shared memory as a flat array
// (field-major, thread fastest: element (field f, front i, thread t) at (f*FM + i)*NT + t,
// which is bank-conflict free for ANY per-lane front index).  The reference keeps one Python
// list per soil layer; here the global order is the concatenation of those lists and the
// per-layer list lengths are kept in `cnt` (list membership) separately from the front's own
// `layer_num` attribute, because the reference lets the two disagree transiently while a front
// crosses a layer boundary (physics/layers/Layer.py:965-1008 then :951-963).
//
// The Green-Ampt capillary drive Geff (physics/lgar/green_ampt.py:19-99; 120-interval
// trapezoid = 480 pow) is evaluated ONE REQUEST PER LANE: the requests of a phase are written
// to a per-warp queue (GeffQueue) and every lane runs one whole request through the
// reference's literal loop, so the result is bit-identical to a scalar evaluation and the
// cost does not depend on which lanes of the warp own the requests (divergent front counts).
//
// All citations are relative to /root/reference/dpLGAR/.  Quirk numbers (Qn) refer to
// SURVEY.md section 8(a).
// =====================================================================================
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/lgar_b200.h"
#include "lgar_pow.cuh"
#include "lgar_rounded.cuh"  // advance_rounded(): exact result of k rounded additions (host-testable)
#include "lgar_var.cuh"
#include <type_traits>

namespace lgar {

constexpr int NT = 128;          // threads per CTA (4 warps, each warp an independent tile)
constexpr int WARPS = NT / 32;
// doubles of per-warp scratch, which holds the Geff request queue.  The queue needs 96; the other 40 are kept because
// the size sets the kernels' shared-memory layout and L1 carve-out, so shrinking it is a change to measure on its own.
// (The taped pass returns its five partials per request through global scratch.)
constexpr int NODEBUF = 136;
constexpr int MAXL = LGAR_MAX_LAYERS;
constexpr int NGIUH = LGAR_MAX_GIUH;
constexpr int NOUT = LGAR_NUM_OUTPUTS;

enum Field { F_DEPTH = 0, F_THETA = 1, F_PSI = 2, F_K = 3, F_DZDT = 4 };

// work counters (per thread, flushed once per chunk when counting is enabled)
enum Cnt { C_GEFF = 0, C_THETA_H = 1, C_H_SE = 2, C_K_SE = 3, C_SE_H = 4, C_ROOT = 5, C_COLMASS = 6, C_SUB = 7 };

struct Soil {  // one layer of one column: Layer.attributes + alpha/n/ksat (Layer.py:48-57)
  double alpha, n, m, inv_m, ninv_m, inv_n, ksat, the, thr;
};

struct Ctx {  // per-thread execution context
  int st;               // lgar_status, first error wins
  unsigned cnt[8];      // work counters
  unsigned br[3];       // branch-coverage counters (counting kernels): 0 dry-over-wet fixes (A17), 1 insert_water equality
                        // fall-through (Q8), 2 calc_bottom_sum_f_p with the free-drainage front in layer >= 2 (Q18)
  long long iter_cap;
  unsigned long long ph[4];  // phase timers (clock64 deltas; counting kernels only): 0 insert-water Geff, 1 move sweep +
                             // merge/cross/fix/update_psi, 2 dry-depth Geff + surficial front, 3 calc_dzdt (Geff per front)
};

__device__ __forceinline__ void raise(Ctx& c, int code) {
  if (c.st == 0) c.st = code;
}

// ------------------------------------------------------------------------------------
// van Genuchten closures (physics/utils.py).
//
// Register discipline: the out-of-line functions below are PURE functions of scalar arguments
// (no Ctx&, no Soil&), so neither the status/counter block nor the soil parameters are forced
// into local memory by a call.  (With by-reference arguments the 1.2 KB/thread stack thrashed
// L1 -- the kernel got slower when the shared-memory carve-out was raised -- see DESIGN.md.)
// The reference's guards (safe_pow / error_check raising ValueError) are evaluated inline by the
// forceinline wrappers, on the same quantities.
// pow is the table-driven routine of lgar_pow.cuh; the CUDA math library's pow is only the
// out-of-range fallback.
// ------------------------------------------------------------------------------------
__device__ __noinline__ double pow_slow(double a, double b) { return pow(a, b); }  // specials / range ends
__device__ __noinline__ double pow_f64(double a, double b) {
  bool ok;
  const double r = pow_core(a, b, ok);  // lgar_pow.cuh: ~0.50 ulp
  return ok ? r : pow_slow(a, b);
}
__device__ __noinline__ double2 pow_log_slow(double a, double b) { return make_double2(pow(a, b), log(a)); }  // cold
// a^b together with log(a) (by-product of the pow core): derivative weights of the reverse kernel
__device__ __noinline__ double2 pow_log_f64(double a, double b) {
  const double xv[1] = {a}, yv[1] = {b};
  double r[1], lg[1];
  bool ok[1];
  pow_core_v<1>(xv, yv, r, ok, lg);
  if (!ok[0]) return pow_log_slow(a, b);
  return make_double2(r[0], lg[0]);
}
// two INDEPENDENT pows from one call (fewer calls; ptxas keeps the two chains back to back, see DESIGN.md 4.1)
__device__ __noinline__ double2 pow_x2(double x0, double y0, double x1, double y1) {
  bool ok0, ok1;
  double a = pow_core(x0, y0, ok0);
  double b = pow_core(x1, y1, ok1);
  if (!ok0) a = pow_slow(x0, y0);
  if (!ok1) b = pow_slow(x1, y1);
  return make_double2(a, b);
}

struct D4 {
  double a, b, c, d;
};
// two independent pows WITH their logs (a = x0^y0, b = log x0, c = x1^y1, d = log x1): the taped trapezoid nodes
__device__ __noinline__ D4 pow_log_x2(double x0, double y0, double x1, double y1) {
  const double xv[2] = {x0, x1}, yv[2] = {y0, y1};
  double r[2], lg[2];
  bool ok[2];
  pow_core_v<2>(xv, yv, r, ok, lg);
  if (!ok[0]) { const double2 q = pow_log_slow(x0, y0); r[0] = q.x; lg[0] = q.y; }  // (out of line: the hot loop of the
  if (!ok[1]) { const double2 q = pow_log_slow(x1, y1); r[1] = q.x; lg[1] = q.y; }  // taped Geff stays small)
  D4 o;
  o.a = r[0]; o.b = lg[0]; o.c = r[1]; o.d = lg[1];
  return o;
}

// utils.py:12-32 safe_pow guards: NaN input or negative base raise ValueError
__device__ __forceinline__ void guard_pow(double base, double e, Ctx& c) {
  if (isnan(base) || isnan(e)) raise(c, LGAR_ST_NAN);
  else if (base < 0.0) raise(c, LGAR_ST_NEG_POW);
}
__device__ __forceinline__ double safe_pow(double base, double e, Ctx& c) {
  guard_pow(base, e, c);
  return pow_f64(base, e);
}
__device__ __forceinline__ double error_check(double r, Ctx& c) {  // utils.py:177-185
  if (isnan(r)) raise(c, LGAR_ST_NAN);
  return r;
}

// ---- pure cores -----------------------------------------------------------------------
// utils.py:35-51   theta = theta_r + (theta_e - theta_r) / (1 + (alpha h)^n)^m
__device__ __noinline__ double theta_h_core(double h, double alpha, double n, double m, double the, double thr) {
  const double outer = pow_f64(1.0 + pow_f64(alpha * h, n), m);
  return (1.0 / outer * (the - thr)) + thr;
}
__device__ __noinline__ double2 theta_h_core_x2(double h0, double al0, double n0, double m0, double the0, double thr0,
                                                double h1, double al1, double n1, double m1, double the1, double thr1) {
  const double2 p = pow_x2(al0 * h0, n0, al1 * h1, n1);
  const double2 q = pow_x2(1.0 + p.x, m0, 1.0 + p.y, m1);
  return make_double2((1.0 / q.x * (the0 - thr0)) + thr0, (1.0 / q.y * (the1 - thr1)) + thr1);
}
// utils.py:159-174   h = (Se^(-1/m) - 1)^(1/n) / alpha ; returns NaN-coded guard via *bad
__device__ __noinline__ double h_se_core(double se, double alpha, double ninv_m, double inv_n, int* bad) {
  double base = pow_f64(se, ninv_m) - 1.0;
  if (fabs(base) <= 1e-8) base = base + 1e-12;  // torch.isclose(base, 0, 1e-12) == |base| <= 1e-8 (Q2)
  *bad = isnan(base) ? LGAR_ST_NAN : (base < 0.0 ? LGAR_ST_NEG_POW : 0);
  return 1.0 / alpha * pow_f64(base, inv_n);
}
// utils.py:134-156   K = Ks sqrt(Se) (1 - (1 - Se^(1/m))^m)^2 ; pow(x, 2) == x*x bit-for-bit in glibc
__device__ __noinline__ double k_se_core(double se, double ksat, double m, double inv_m, int* bad) {
  double base = 1.0 - pow_f64(se, inv_m);
  if (fabs(base) <= 1e-8) base = base + 1e-12;
  int b = isnan(base) ? LGAR_ST_NAN : (base < 0.0 ? LGAR_ST_NEG_POW : 0);
  const double t = 1.0 - pow_f64(base, m);
  if (!b) b = isnan(t) ? LGAR_ST_NAN : (t < 0.0 ? LGAR_ST_NEG_POW : 0);
  *bad = b;
  return ksat * sqrt(se) * (t * t);
}
// psi = h(Se) and K = K(Se) for the same Se: two independent chains interleaved
__device__ __noinline__ double2 psi_k_core(double se, double alpha, double ninv_m, double inv_n, double ksat, double m,
                                           double inv_m, int* bad) {
  const double2 p = pow_x2(se, ninv_m, se, inv_m);
  double bh = p.x - 1.0;
  if (fabs(bh) <= 1e-8) bh = bh + 1e-12;
  double bk = 1.0 - p.y;
  if (fabs(bk) <= 1e-8) bk = bk + 1e-12;
  int b = (isnan(bh) || isnan(bk)) ? LGAR_ST_NAN : ((bh < 0.0 || bk < 0.0) ? LGAR_ST_NEG_POW : 0);
  const double2 o = pow_x2(bh, inv_n, bk, m);
  const double t = 1.0 - o.y;
  if (!b) b = isnan(t) ? LGAR_ST_NAN : (t < 0.0 ? LGAR_ST_NEG_POW : 0);
  *bad = b;
  return make_double2(1.0 / alpha * o.x, ksat * sqrt(se) * (t * t));
}
// two h(Se) with the same soil (Geff end points)
__device__ __noinline__ double2 h_se_core_x2(double se0, double se1, double alpha, double ninv_m, double inv_n, int* bad) {
  const double2 p = pow_x2(se0, ninv_m, se1, ninv_m);
  double b0 = p.x - 1.0, b1 = p.y - 1.0;
  if (fabs(b0) <= 1e-8) b0 = b0 + 1e-12;
  if (fabs(b1) <= 1e-8) b1 = b1 + 1e-12;
  *bad = (isnan(b0) || isnan(b1)) ? LGAR_ST_NAN : ((b0 < 0.0 || b1 < 0.0) ? LGAR_ST_NEG_POW : 0);
  const double2 o = pow_x2(b0, inv_n, b1, inv_n);
  return make_double2(1.0 / alpha * o.x, 1.0 / alpha * o.y);
}
// K(Se(h)) at two trapezoid nodes of one Geff request (green_ampt.py:75-81): se_from_h (utils.py:115-131,
// constant 1.0 for |h| < 0.1, Q12) then k_from_se
__device__ __noinline__ double2 k_nodes_core_x2(double h0, double h1, double alpha, double n, double m, double inv_m,
                                                double ksat, int* bad) {
  const bool w0 = fabs(h0) < 1.0e-01, w1 = fabs(h1) < 1.0e-01;
  const double a0 = w0 ? 1.0 : alpha * h0, a1 = w1 ? 1.0 : alpha * h1;
  int b = (isnan(a0) || isnan(a1)) ? LGAR_ST_NAN : ((a0 < 0.0 || a1 < 0.0) ? LGAR_ST_NEG_POW : 0);
  const double2 p = pow_x2(a0, n, a1, n);
  const double2 d = pow_x2(1.0 + p.x, m, 1.0 + p.y, m);
  double se0 = 1.0 / d.x, se1 = 1.0 / d.y;
  if (!b && (isnan(se0) || isnan(se1))) b = LGAR_ST_NAN;
  if (w0) se0 = 1.0;
  if (w1) se1 = 1.0;
  const double2 sp = pow_x2(se0, inv_m, se1, inv_m);
  double b0 = 1.0 - sp.x, b1 = 1.0 - sp.y;
  if (fabs(b0) <= 1e-8) b0 = b0 + 1e-12;
  if (fabs(b1) <= 1e-8) b1 = b1 + 1e-12;
  if (!b) b = (isnan(b0) || isnan(b1)) ? LGAR_ST_NAN : ((b0 < 0.0 || b1 < 0.0) ? LGAR_ST_NEG_POW : 0);
  const double2 o = pow_x2(b0, m, b1, m);
  const double t0 = 1.0 - o.x, t1 = 1.0 - o.y;
  if (!b) b = (isnan(t0) || isnan(t1)) ? LGAR_ST_NAN : ((t0 < 0.0 || t1 < 0.0) ? LGAR_ST_NEG_POW : 0);
  *bad = b;
  return make_double2(ksat * sqrt(se0) * (t0 * t0), ksat * sqrt(se1) * (t1 * t1));
}

// ---- guarded wrappers (inline) ----------------------------------------------------------
__device__ __forceinline__ double theta_from_h(double h, const Soil& s, Ctx& c) {
  c.cnt[C_THETA_H]++;
  guard_pow(s.alpha * h, s.n, c);
  return error_check(theta_h_core(h, s.alpha, s.n, s.m, s.the, s.thr), c);
}
// two theta_from_h; `both` == false: only the first result is meaningful
__device__ __forceinline__ double2 theta_from_h_x2(double h0, const Soil& s0, double h1, const Soil& s1, bool both, Ctx& c) {
  c.cnt[C_THETA_H] += both ? 2 : 1;
  guard_pow(s0.alpha * h0, s0.n, c);
  if (both) guard_pow(s1.alpha * h1, s1.n, c);
  const double2 r = theta_h_core_x2(h0, s0.alpha, s0.n, s0.m, s0.the, s0.thr, both ? h1 : 1.0, s1.alpha, s1.n, s1.m,
                                    s1.the, s1.thr);
  if (isnan(r.x) || (both && isnan(r.y))) raise(c, LGAR_ST_NAN);
  return r;
}
// variants for the root-finder loop of the move sweep: the theta cores are inlined at the call site (one call level
// less per iteration: the loop's instruction stream is dominated by call/return fetch bubbles; +3 % throughput),
// pow_x2 / pow_f64 stay out of line (inlining them too costs 20 %: register pressure)
__device__ __forceinline__ double2 theta_from_h_x2_inl(double h0, const Soil& s0, double h1, const Soil& s1, bool both, Ctx& c) {
  c.cnt[C_THETA_H] += both ? 2 : 1;
  guard_pow(s0.alpha * h0, s0.n, c);
  if (both) guard_pow(s1.alpha * h1, s1.n, c);
  const double2 p = pow_x2(s0.alpha * h0, s0.n, s1.alpha * (both ? h1 : 1.0), s1.n);
  const double2 q = pow_x2(1.0 + p.x, s0.m, 1.0 + p.y, s1.m);
  const double2 r = make_double2((1.0 / q.x * (s0.the - s0.thr)) + s0.thr, (1.0 / q.y * (s1.the - s1.thr)) + s1.thr);
  if (isnan(r.x) || (both && isnan(r.y))) raise(c, LGAR_ST_NAN);
  return r;
}
__device__ __forceinline__ double theta_from_h_inl(double h, const Soil& s, Ctx& c) {
  c.cnt[C_THETA_H]++;
  guard_pow(s.alpha * h, s.n, c);
  const double outer = pow_f64(1.0 + pow_f64(s.alpha * h, s.n), s.m);
  return error_check((1.0 / outer * (s.the - s.thr)) + s.thr, c);
}
// utils.py:102-112
__device__ __forceinline__ double se_from_theta(double theta, const Soil& s, Ctx& c) {
  return error_check((theta - s.thr) / (s.the - s.thr), c);
}
__device__ __forceinline__ double k_from_se(double se, double ksat, double m, double inv_m, Ctx& c) {
  c.cnt[C_K_SE]++;
  guard_pow(se, inv_m, c);
  int bad;
  const double r = k_se_core(se, ksat, m, inv_m, &bad);
  if (bad) raise(c, bad);
  return error_check(r, c);
}
__device__ __forceinline__ double h_from_se(double se, const Soil& s, Ctx& c) {
  c.cnt[C_H_SE]++;
  guard_pow(se, s.ninv_m, c);
  int bad;
  const double r = h_se_core(se, s.alpha, s.ninv_m, s.inv_n, &bad);
  if (bad) raise(c, bad);
  return error_check(r, c);
}
__device__ __forceinline__ double2 psi_k_from_se(double se, const Soil& s, Ctx& c) {
  c.cnt[C_H_SE]++;
  c.cnt[C_K_SE]++;
  guard_pow(se, s.ninv_m, c);
  int bad;
  const double2 r = psi_k_core(se, s.alpha, s.ninv_m, s.inv_n, s.ksat, s.m, s.inv_m, &bad);
  if (bad) raise(c, bad);
  if (isnan(r.x) || isnan(r.y)) raise(c, LGAR_ST_NAN);
  return r;
}
__device__ __forceinline__ double2 h_from_se_x2(double se0, double se1, const Soil& s, Ctx& c) {
  c.cnt[C_H_SE] += 2;
  guard_pow(se0, s.ninv_m, c);
  guard_pow(se1, s.ninv_m, c);
  int bad;
  const double2 r = h_se_core_x2(se0, se1, s.alpha, s.ninv_m, s.inv_n, &bad);
  if (bad) raise(c, bad);
  if (isnan(r.x) || isnan(r.y)) raise(c, LGAR_ST_NAN);
  return r;
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
// maximum of v over the warp (butterfly); warp-convergent
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}

// torch.min / torch.minimum semantics (NaN propagates, unlike fmin)
__device__ __forceinline__ double tmin(double a, double b) {
  if (isnan(a) || isnan(b)) return a + b;
  return (b < a) ? b : a;
}

// ------------------------------------------------------------------------------------
// Closed-form capillary drive (cfg.data.use_closed_form_G, green_ampt.py:85-98), per lane (three pows, no queue
// needed).  Literal restatement, including the swapped roles of theta_1 / theta_2 and the operator
// precedence of the published line (sic):
//   se_f = Se(theta_1), se_i = Se(theta_2);  h_c = psib (2 + 3 lambda) / (1 + 3 lambda);  e = 3 + 1 / lambda
//   geff = h_c * se_i^e - se_f^e / (1 - se_f^e);  inf or NaN -> h_c
// with the Brooks-Corey estimates of generate_soil_metrics (data/utils.py:85-87, utils.py:54-99):
//   p = 1 + 2/m;  lambda = 2 / (p - 3);  psib = (p + 3)(147.8 + 8.1 p + 0.092 p^2) / (2 alpha p (p - 1)(55.6 + 7.4 p + p^2))
// P == true also returns the partials w.r.t. theta_1, theta_2, alpha and m (reference autograd: gradient flows
// through lambda(m) and psib(alpha, m); torch's pow has zero exponent-gradient at base 0).
// Evaluated through geff_closedR where nint < 0 (substep passes nint = -1 when the flag is set).
// ------------------------------------------------------------------------------------
struct GeffClosed {
  double v, d_t1, d_t2, d_alpha, d_m;
  int st;
};
__device__ __forceinline__ double bc_psib(double alpha, double m) {
  const double p_ = 1.0 + (2.0 / m);
  return (p_ + 3.0) * (147.8 + 8.1 * p_ + 0.092 * p_ * p_) / (2.0 * alpha * p_ * (p_ - 1.0) * (55.6 + 7.4 * p_ + p_ * p_));
}
template <bool P>
__device__ __noinline__ GeffClosed geff_closed_core(double theta_1, double theta_2, double alpha, double m, double the,
                                                    double thr) {
  GeffClosed r;
  r.v = r.d_t1 = r.d_t2 = r.d_alpha = r.d_m = 0.0;
  int st = 0;
  const double span = the - thr;
  const double se_f = (theta_1 - thr) / span;
  if (isnan(se_f)) st = LGAR_ST_NAN;
  const double se_i = (theta_2 - thr) / span;
  if (!st && isnan(se_i)) st = LGAR_ST_NAN;
  const double p_ = 1.0 + (2.0 / m);
  const double lam = 2.0 / (p_ - 3.0);
  const double psib = bc_psib(alpha, m);
  const double h_c = psib * (2.0 + 3.0 * lam) / (1.0 + 3.0 * lam);
  const double e = 3.0 + 1.0 / lam;
  // safe_pow guards (utils.py:12-32) in call order: se_i^e, se_f^e, se_f^e
  if (!st) st = (isnan(se_i) || isnan(e)) ? LGAR_ST_NAN : (se_i < 0.0 ? LGAR_ST_NEG_POW : 0);
  if (!st) st = isnan(se_f) ? LGAR_ST_NAN : (se_f < 0.0 ? LGAR_ST_NEG_POW : 0);
  double A, Bq, lse_i = 0.0, lse_f = 0.0;
  if (P) {
    const double2 a = pow_log_f64(se_i, e), b = pow_log_f64(se_f, e);
    A = a.x; lse_i = a.y; Bq = b.x; lse_f = b.y;
  } else {
    const double2 ab = pow_x2(se_i, e, se_f, e);
    A = ab.x; Bq = ab.y;
  }
  const double D = 1.0 - Bq;
  double geff = h_c * A - Bq / D;
  const bool fallback = isinf(geff) || isnan(geff);
  if (fallback) geff = h_c;
  r.v = geff;
  r.st = st;
  if (P) {
    const double dg_dhc = fallback ? 1.0 : A;
    double dg_de = 0.0;
    if (!fallback) {
      dg_de = ((se_i == 0.0) ? 0.0 : h_c * A * lse_i) - ((se_f == 0.0) ? 0.0 : Bq * lse_f / (D * D));
      r.d_t2 = ((se_i == 0.0) ? 0.0 : h_c * e * A / se_i) / span;
      r.d_t1 = -((se_f == 0.0) ? 0.0 : (e * Bq / se_f) / (D * D)) / span;
    }
    const double q3 = 1.0 + 3.0 * lam;
    const double dhc_dpsib = (2.0 + 3.0 * lam) / q3;
    const double dhc_dlam = -3.0 * psib / (q3 * q3);
    const double de_dlam = -1.0 / (lam * lam);
    const double dlam_dp = -2.0 / ((p_ - 3.0) * (p_ - 3.0));
    const double dp_dm = -2.0 / (m * m);
    const double N1 = p_ + 3.0, N2 = 147.8 + 8.1 * p_ + 0.092 * p_ * p_;
    const double D3 = 55.6 + 7.4 * p_ + p_ * p_;
    const double dlnN = 1.0 / N1 + (8.1 + 0.184 * p_) / N2;
    const double dlnD = 1.0 / p_ + 1.0 / (p_ - 1.0) + (7.4 + 2.0 * p_) / D3;
    const double dpsib_dp = psib * (dlnN - dlnD);
    const double dg_dlam = dg_dhc * dhc_dlam + dg_de * de_dlam;
    r.d_alpha = dg_dhc * dhc_dpsib * (-psib / alpha);
    r.d_m = (dg_dhc * dhc_dpsib * dpsib_dp + dg_dlam * dlam_dp) * dp_dm;
  }
  return r;
}

// ------------------------------------------------------------------------------------
// Scalar-generic layer: R = double (forward kernel) or R = Var (taped pass of the reverse kernel).
// ------------------------------------------------------------------------------------
template <class R>
struct SoilT;
template <>
struct SoilT<double> : Soil {
  __device__ __forceinline__ double ksatR() const { return ksat; }
};
template <>
struct SoilT<Var> : Soil {
  int id_alpha, id_n, id_m, id_ksat;  // tape ids of the differentiable parameters (m = 1 - 1/n is derived on tape)
  __device__ __forceinline__ Var ksatR() const { return Var(ksat, id_ksat); }
};

// ---- theta(h)
__device__ __forceinline__ double thetaR(double h, const SoilT<double>& s, Ctx& c) { return theta_from_h(h, s, c); }
struct P4 {
  double a, b, c, d;
};
// partials of theta(h; alpha, n, m): x = alpha h; ap = x^n; u = 1 + ap; o = u^m; theta = (the - thr)/o + thr
__device__ __noinline__ P4 theta_partials(double h, double alpha, double n, double m, double span) {
  const double x = alpha * h;
  const double ap = pow_f64(x, n);
  const double u = 1.0 + ap;
  const double o = pow_f64(u, m);
  const double dth_do = -span / (o * o);
  const double do_du = m * o / u;
  const double dap_dx = (x == 0.0) ? 0.0 : n * ap / x;
  const double dap_dn = (x == 0.0) ? 0.0 : ap * log(x);
  const double g = dth_do * do_du;
  P4 r;
  r.a = g * dap_dx * alpha;  // d/dh
  r.b = g * dap_dx * h;      // d/dalpha
  r.c = g * dap_dn;          // d/dn
  r.d = dth_do * o * log(u); // d/dm
  return r;
}
__device__ __forceinline__ Var thetaR(const Var& h, const SoilT<Var>& s, Ctx& c) {
  const double v = theta_from_h(h.v, s, c);
  const P4 q = theta_partials(h.v, s.alpha, s.n, s.m, s.the - s.thr);
  const int ids[4] = {h.id, s.id_alpha, s.id_n, s.id_m};
  const double d[4] = {q.a, q.b, q.c, q.d};
  return tape_record_n(v, 4, ids, d);
}
// ---- Se(theta)
__device__ __forceinline__ double se_thetaR(double theta, const SoilT<double>& s, Ctx& c) { return se_from_theta(theta, s, c); }
__device__ __forceinline__ Var se_thetaR(const Var& theta, const SoilT<Var>& s, Ctx& c) {
  return tape_record(se_from_theta(theta.v, s, c), theta.id, 1.0 / (s.the - s.thr), -1, 0.0);
}
// ---- h(Se) partials: sp = se^(-1/m); base = sp - 1; op = base^(1/n); h = op / alpha
__device__ __noinline__ P4 h_se_partials_core(double se, double alpha, double ninv_m, double inv_m, double inv_n,
                                              double hval) {
  const double sp = pow_f64(se, ninv_m);
  double base = sp - 1.0;
  if (fabs(base) <= 1e-8) base = base + 1e-12;
  const double op = hval * alpha;
  const double dop_dbase = inv_n * op / base;
  const double dsp_dse = (se == 0.0) ? 0.0 : ninv_m * sp / se;
  const double dsp_dm = (se == 0.0) ? 0.0 : sp * log(se) * (inv_m * inv_m);  // d(-1/m)/dm = 1/m^2
  const double dop_dn = (base == 0.0) ? 0.0 : op * log(base) * (-(inv_n * inv_n));
  P4 r;
  r.a = dop_dbase * dsp_dse / alpha;  // d/dse
  r.b = -hval / alpha;                // d/dalpha
  r.c = dop_dn / alpha;               // d/dn
  r.d = dop_dbase * dsp_dm / alpha;   // d/dm
  return r;
}
__device__ __forceinline__ void h_se_partials(double se, const Soil& s, double hval, double* d_se, double* d_alpha,
                                              double* d_n, double* d_m) {
  const P4 r = h_se_partials_core(se, s.alpha, s.ninv_m, s.inv_m, s.inv_n, hval);
  *d_se = r.a;
  *d_alpha = r.b;
  *d_n = r.c;
  *d_m = r.d;
}
__device__ __forceinline__ double h_seR(double se, const SoilT<double>& s, Ctx& c) { return h_from_se(se, s, c); }
__device__ __forceinline__ Var h_seR(const Var& se, const SoilT<Var>& s, Ctx& c) {
  const double v = h_from_se(se.v, s, c);
  double d_se, d_a, d_n, d_m;
  h_se_partials(se.v, s, v, &d_se, &d_a, &d_n, &d_m);
  const int ids[4] = {se.id, s.id_alpha, s.id_n, s.id_m};
  const double d[4] = {d_se, d_a, d_n, d_m};
  return tape_record_n(v, 4, ids, d);
}
// ---- K(Se) partials: sp = se^(1/m); base = 1 - sp; op = base^m; t = 1 - op; K = ksat sqrt(se) t^2
__device__ __noinline__ P4 k_se_partials_core(double se, double ksat, double m, double inv_m);
__device__ __forceinline__ void k_se_partials(double se, double ksat, double m, double inv_m, double* d_se, double* d_ksat,
                                              double* d_m) {
  const P4 r = k_se_partials_core(se, ksat, m, inv_m);
  *d_se = r.a;
  *d_ksat = r.b;
  *d_m = r.c;
}
__device__ __noinline__ P4 k_se_partials_core(double se, double ksat, double m, double inv_m) {
  const double sp = pow_f64(se, inv_m);
  double base = 1.0 - sp;
  if (fabs(base) <= 1e-8) base = base + 1e-12;
  const double op = pow_f64(base, m);
  const double t = 1.0 - op;
  const double rs = sqrt(se);
  const double sp_over = (se == 0.0) ? 0.0 : sp / se;
  // -dop/dse = op sp / (base se);  dop/dm = op ln(base) + op sp ln(se) / (base m)
  const double ndop_dse = op * sp_over / base;
  const double lnse = (se == 0.0) ? 0.0 : log(se);
  const double dop_dm = op * log(base) + op * sp * lnse / (base * m);
  P4 r;
  r.a = ksat * ((rs == 0.0 ? 0.0 : t * t / (2.0 * rs)) + 2.0 * t * rs * ndop_dse);  // d/dse
  r.b = rs * (t * t);                                                                // d/dksat
  r.c = ksat * rs * 2.0 * t * (-dop_dm);                                             // d/dm
  r.d = 0.0;
  return r;
}
__device__ __forceinline__ double k_seR(double se, const SoilT<double>& s, Ctx& c) {
  return k_from_se(se, s.ksat, s.m, s.inv_m, c);
}
__device__ __forceinline__ Var k_seR(const Var& se, const SoilT<Var>& s, Ctx& c) {
  const double v = k_from_se(se.v, s.ksat, s.m, s.inv_m, c);
  double d_se, d_k, d_m;
  k_se_partials(se.v, s.ksat, s.m, s.inv_m, &d_se, &d_k, &d_m);
  const int ids[3] = {se.id, s.id_ksat, s.id_m};
  const double d[3] = {d_se, d_k, d_m};
  return tape_record_n(v, 3, ids, d);
}
// ---- psi and K from the same Se
template <class R>
struct Pair {
  R x, y;
};
__device__ __forceinline__ Pair<double> psi_kR(double se, const SoilT<double>& s, Ctx& c) {
  const double2 r = psi_k_from_se(se, s, c);
  Pair<double> p;
  p.x = r.x;
  p.y = r.y;
  return p;
}
__device__ __forceinline__ Pair<Var> psi_kR(const Var& se, const SoilT<Var>& s, Ctx& c) {
  const double2 r = psi_k_from_se(se.v, s, c);  // same values as the forward kernel
  double d_se, d_a, d_n, d_m, e_se, e_k, e_m;
  h_se_partials(se.v, s, r.x, &d_se, &d_a, &d_n, &d_m);
  k_se_partials(se.v, s.ksat, s.m, s.inv_m, &e_se, &e_k, &e_m);
  const int ids[4] = {se.id, s.id_alpha, s.id_n, s.id_m};
  const double d[4] = {d_se, d_a, d_n, d_m};
  const int ids2[3] = {se.id, s.id_ksat, s.id_m};
  const double d2[3] = {e_se, e_k, e_m};
  Pair<Var> p;
  p.x = tape_record_n(r.x, 4, ids, d);
  p.y = tape_record_n(r.y, 3, ids2, d2);
  return p;
}

// ---- closed-form Geff of this lane's request (0 when need == false); the taped form records one entry with the
//      partials w.r.t. theta_1, theta_2, alpha and m
__device__ __forceinline__ double geff_closedR(bool need, double theta_1, double theta_2, const SoilT<double>& s, Ctx& c) {
  if (!need) return 0.0;
  const GeffClosed g = geff_closed_core<false>(theta_1, theta_2, s.alpha, s.m, s.the, s.thr);
  if (g.st) raise(c, g.st);
  return g.v;
}
__device__ Var geff_closedR(bool need, const Var& theta_1, const Var& theta_2, const SoilT<Var>& s, Ctx& c) {
  if (!need) return Var(0.0);
  const GeffClosed g = geff_closed_core<true>(theta_1.v, theta_2.v, s.alpha, s.m, s.the, s.thr);
  if (g.st) raise(c, g.st);
  const int ids[4] = {theta_1.id, theta_2.id, s.id_alpha, s.id_m};
  const double d[4] = {g.d_t1, g.d_t2, g.d_alpha, g.d_m};
  return tape_record_n(g.v, 4, ids, d);
}

// Node 0 of a taped Geff request (geff_batch_eval_taped), from ONE evaluation of the four pows: K (the same
// operations as k_nodes_core_x2, hence the same bits as the forward kernel) and the partials of
// K(Se(h; alpha, n, m); ksat, m); the logs come out of the pow cores.  K_0 = K(Se_i) is a direct function of Se_i in
// the reference graph (green_ampt.py:75), so with node0 Se is overridden by se0 after the guards of the first half
// and the partial w.r.t. Se is reported instead of the h / alpha / n ones.  The other nodes of the request go
// through k_node_full_x2, two at a time.
struct NodeFull {
  double K, dk_se, dk_h, dk_a, dk_n, dk_m;
  int bad;
};
__device__ __noinline__ NodeFull k_node_full(double h, bool node0, double se0, double alpha, double n, double m,
                                             double inv_m, double ksat) {
  NodeFull r;
  const bool w = fabs(h) < 1.0e-01;
  const double x = w ? 1.0 : alpha * h;
  int b = isnan(x) ? LGAR_ST_NAN : (x < 0.0 ? LGAR_ST_NEG_POW : 0);
  const double2 pa = pow_log_f64(x, n);  // ap, log x
  const double u = 1.0 + pa.x;
  const double2 pu = pow_log_f64(u, m);  // u^m, log u
  double se = 1.0 / pu.x;
  if (!b && isnan(se)) b = LGAR_ST_NAN;
  double dse_dh = 0.0, dse_da = 0.0, dse_dn = 0.0, dse_dm = 0.0;
  if (w) {
    se = 1.0;
  } else {
    const double dse_du = -m * se / u;
    const double dap_dx = (x == 0.0) ? 0.0 : n * pa.x / x;
    dse_dh = dse_du * dap_dx * alpha;
    dse_da = dse_du * dap_dx * h;
    dse_dn = (x == 0.0) ? 0.0 : dse_du * pa.x * pa.y;
    dse_dm = -se * pu.y;
  }
  if (node0) {
    se = se0;
    dse_dh = dse_da = dse_dn = dse_dm = 0.0;
  }
  const double2 ps = pow_log_f64(se, inv_m);  // sp, log se
  double base = 1.0 - ps.x;
  if (fabs(base) <= 1e-8) base = base + 1e-12;
  if (!b) b = isnan(base) ? LGAR_ST_NAN : (base < 0.0 ? LGAR_ST_NEG_POW : 0);
  const double2 po = pow_log_f64(base, m);  // op, log base
  const double t = 1.0 - po.x;
  if (!b) b = isnan(t) ? LGAR_ST_NAN : (t < 0.0 ? LGAR_ST_NEG_POW : 0);
  const double rs = sqrt(se);
  r.K = ksat * rs * (t * t);
  if (!b && isnan(r.K)) b = LGAR_ST_NAN;
  r.bad = b;
  // -dop/dse = op sp / (base se);  dop/dm = op ln(base) + op sp ln(se) / (base m)   (k_se_partials_core)
  const double sp_over = (se == 0.0) ? 0.0 : ps.x / se;
  const double ndop_dse = po.x * sp_over / base;
  const double lnse = (se == 0.0) ? 0.0 : ps.y;
  const double dop_dm = po.x * po.y + po.x * ps.x * lnse / (base * m);
  const double dk_se = ksat * ((rs == 0.0 ? 0.0 : t * t / (2.0 * rs)) + 2.0 * t * rs * ndop_dse);
  const double dk_m = ksat * rs * 2.0 * t * (-dop_dm);
  r.dk_se = dk_se;
  r.dk_h = dk_se * dse_dh;
  r.dk_a = dk_se * dse_da;
  r.dk_n = dk_se * dse_dn;
  r.dk_m = dk_se * dse_dm + dk_m;
  return r;
}

// ------------------------------------------------------------------------------------
// Batched Geff: ONE LANE PER REQUEST (green_ampt.py:19-84, trapezoid branch).
//
// A sub-step of a 32-column tile issues ~60 independent Geff(theta_1, theta_2; layer) requests in calc_dzdt (one
// per moving front of every column) -- ~90 % of all requests -- plus at most one per column in insert_water and in
// calc_dry_depth.  The requests of a phase are known before any of them is evaluated, so they are written to a
// per-warp queue of 32 slots (calc_dzdt: batches of 32 in queue order; the other two: slot = lane, through
// geff_one_per_lane) and every lane evaluates ONE whole request with the literal loop of the reference
// (`h2 = h2 + dh`, `geff = geff + (k1 + k2) * (dh / 2)`), two nodes per pass through the out-of-line pair evaluator
// k_nodes_core_x2.  Values are bit-identical to a scalar evaluation (same operations on the same operands in the
// same order), and the cost of a batch does not depend on which lanes own the requests.  The soil parameters of
// the requesting column are fetched with warp shuffles (owner lane, list layer).
// ------------------------------------------------------------------------------------
struct GeffQueue {         // SoA over the 32 slots of a batch; lives in the per-warp scratch
  double a[32];            // in: theta_1                    out: Geff
  double b[32];            // in: theta_2
  int meta[32];            // in: owner lane | list layer << 8; -1 = empty slot
  int st[32];              // out: lgar_status raised inside calc_geff (0 = none)
};
static_assert(sizeof(GeffQueue) <= NODEBUF * sizeof(double), "the queue lives in the per-warp scratch");
// taped pass only: d Geff / d(theta_1, theta_2, alpha, n, m) of the 32 slots, [5][32] doubles per warp.  Kept in GLOBAL
// scratch (the warp's adjoint array, idle during the taped recompute): 1.25 KB more shared memory per warp would cost
// the reverse kernel its second CTA per SM.
__shared__ double* g_geffq_partials[NT / 32];

// gather the soil of (owner lane, list layer) from the lanes' own parameter arrays; warp-convergent
template <class ST>
__device__ __forceinline__ Soil gather_soil(const ST* soil, int L, int owner, int lay) {
  Soil q;
  q.alpha = q.n = q.m = q.inv_m = q.ninv_m = q.inv_n = q.ksat = q.the = q.thr = 1.0;
  for (int l = 0; l < L; l++) {
    const ST& sl = soil[l];
    const double v0 = shfl_d(sl.alpha, owner), v1 = shfl_d(sl.n, owner), v2 = shfl_d(sl.m, owner);
    const double v3 = shfl_d(sl.inv_m, owner), v4 = shfl_d(sl.ninv_m, owner), v5 = shfl_d(sl.inv_n, owner);
    const double v6 = shfl_d(sl.ksat, owner), v7 = shfl_d(sl.the, owner), v8 = shfl_d(sl.thr, owner);
    if (l == lay) {
      q.alpha = v0; q.n = v1; q.m = v2; q.inv_m = v3; q.ninv_m = v4; q.inv_n = v5; q.ksat = v6; q.the = v7; q.thr = v8;
    }
  }
  return q;
}

// The start of one request, common to both batch evaluators: Se and h at both ends, the node spacing dh, K at node 0
// and the status raised so far
struct GeffStart {
  double se_i, se_f, h_i, h_f, dh, k1;
  int st;
};
__device__ __forceinline__ GeffStart geff_start(double theta_1, double theta_2, const Soil& s, int nint) {
  Ctx c;
  c.st = 0;
  GeffStart g;
  g.se_i = se_from_theta(theta_1, s, c);
  g.se_f = se_from_theta(theta_2, s, c);
  const double2 hh = h_from_se_x2(g.se_i, g.se_f, s, c);
  g.h_i = hh.x;
  g.h_f = hh.y;
  // "Checkpoint" calls green_ampt.py:61-63: results unused, only their guards can matter
  if (fabs(g.h_i) >= 0.1 && s.alpha * g.h_i < 0.0) raise(c, LGAR_ST_NEG_POW);
  if (fabs(g.h_f) >= 0.1 && s.alpha * g.h_f < 0.0) raise(c, LGAR_ST_NEG_POW);
  g.dh = (g.h_f - g.h_i) / (double)nint;
  g.k1 = k_from_se(g.se_i, s.ksat, s.m, s.inv_m, c);
  g.st = c.st;
  return g;
}

// Forward (values only).  Every lane of the warp calls it; lane s evaluates slot s.
template <class ST>
__device__ __noinline__ void geff_batch_eval(GeffQueue* q, const ST* soil, int L, int nint) {
  const int lane = threadIdx.x & 31;
  const int meta = q->meta[lane];
  const bool have = meta >= 0;
  const Soil s = gather_soil(soil, L, have ? (meta & 31) : lane, have ? ((meta >> 8) & 7) : 0);
  if (have) {
    const GeffStart g0 = geff_start(q->a[lane], q->b[lane], s, nint);
    const double dh = g0.dh;
    double k1 = g0.k1;
    const double half = dh / 2.0;
    double geff = 0.0;
    double h2 = g0.h_i + dh;
    int st = g0.st;
    // two nodes per pass through the SAME out-of-line pair evaluator as everything else (k_nodes_core_x2 -> pow_x2):
    // the kernel is instruction-fetch sensitive (DESIGN.md), so the hot loops share one small body of pow code
#pragma unroll 1
    for (int i = 0; i < nint; i += 2) {
      const double ha = h2, hb = ha + dh;
      h2 = hb + dh;
      int bad;
      const double2 kk = k_nodes_core_x2(ha, (i + 1 < nint) ? hb : ha, s.alpha, s.n, s.m, s.inv_m, s.ksat, &bad);
      geff = geff + ((k1 + kk.x) * half);
      k1 = kk.x;
      if (i + 1 < nint) {
        geff = geff + ((k1 + kk.y) * half);
        k1 = kk.y;
      }
      if (st == 0) {  // per-node guards: first node in sequence wins (bad covers the pair in node order)
        if (bad) st = bad;
        else if (isnan(kk.x) || (i + 1 < nint && isnan(kk.y))) st = LGAR_ST_NAN;
      }
    }
    q->a[lane] = fabs(geff / s.ksat);
    q->st[lane] = st;
  }
  __syncwarp();
}

// Two trapezoid nodes with everything the reverse kernel needs (k_node_full, two chains interleaved through the one
// shared pow_log_x2 body): K and the partials of K(Se(h; alpha, n, m); ksat, m) w.r.t. h, alpha, n, m.
struct NodeFull2 {
  double K[2], dk_h[2], dk_a[2], dk_n[2], dk_m[2];
  int bad[2];
};
__device__ __noinline__ NodeFull2 k_node_full_x2(double h0, double h1, double alpha, double n, double m, double inv_m,
                                                 double ksat) {
  NodeFull2 r;
  const double h[2] = {h0, h1};
  bool w[2];
  double x[2], ap[2], lx[2], u[2], um[2], lu[2], se[2], sp[2], lse[2], base[2], op[2], lb[2];
#pragma unroll
  for (int e = 0; e < 2; e++) {
    w[e] = fabs(h[e]) < 1.0e-01;
    x[e] = w[e] ? 1.0 : alpha * h[e];
    r.bad[e] = isnan(x[e]) ? LGAR_ST_NAN : (x[e] < 0.0 ? LGAR_ST_NEG_POW : 0);
  }
  D4 q = pow_log_x2(x[0], n, x[1], n);
  ap[0] = q.a; lx[0] = q.b; ap[1] = q.c; lx[1] = q.d;
  u[0] = 1.0 + ap[0];
  u[1] = 1.0 + ap[1];
  q = pow_log_x2(u[0], m, u[1], m);
  um[0] = q.a; lu[0] = q.b; um[1] = q.c; lu[1] = q.d;
  // The VALUE path (se, base, K) repeats the forward kernel's operations bit for bit.  The partials only have to
  // meet the gradient tolerance, so they use reciprocals (one MUFU + Newton step each) instead of IEEE divisions,
  // and 1 / se = u^m, 1 / sqrt(se) = sqrt(se) u^m come for free: three reciprocals per node instead of seven divisions.
  double dse_dh[2], dse_da[2], dse_dn[2], dse_dm[2], inv_se[2];
#pragma unroll
  for (int e = 0; e < 2; e++) {
    se[e] = 1.0 / um[e];
    if (!r.bad[e] && isnan(se[e])) r.bad[e] = LGAR_ST_NAN;
    if (w[e]) {
      se[e] = 1.0;
      inv_se[e] = 1.0;
      dse_dh[e] = dse_da[e] = dse_dn[e] = dse_dm[e] = 0.0;
    } else {
      inv_se[e] = um[e];
      const double dse_du = -m * se[e] * __drcp_rn(u[e]);
      const double dap_dx = (x[e] == 0.0) ? 0.0 : n * ap[e] * __drcp_rn(x[e]);
      dse_dh[e] = dse_du * dap_dx * alpha;
      dse_da[e] = dse_du * dap_dx * h[e];
      dse_dn[e] = (x[e] == 0.0) ? 0.0 : dse_du * ap[e] * lx[e];
      dse_dm[e] = -se[e] * lu[e];
    }
  }
  q = pow_log_x2(se[0], inv_m, se[1], inv_m);
  sp[0] = q.a; lse[0] = q.b; sp[1] = q.c; lse[1] = q.d;
#pragma unroll
  for (int e = 0; e < 2; e++) {
    base[e] = 1.0 - sp[e];
    if (fabs(base[e]) <= 1e-8) base[e] = base[e] + 1e-12;
    if (!r.bad[e]) r.bad[e] = isnan(base[e]) ? LGAR_ST_NAN : (base[e] < 0.0 ? LGAR_ST_NEG_POW : 0);
  }
  q = pow_log_x2(base[0], m, base[1], m);
  op[0] = q.a; lb[0] = q.b; op[1] = q.c; lb[1] = q.d;
#pragma unroll
  for (int e = 0; e < 2; e++) {
    const double t = 1.0 - op[e];
    if (!r.bad[e]) r.bad[e] = isnan(t) ? LGAR_ST_NAN : (t < 0.0 ? LGAR_ST_NEG_POW : 0);
    const double rs = sqrt(se[e]);
    r.K[e] = ksat * rs * (t * t);
    if (!r.bad[e] && isnan(r.K[e])) r.bad[e] = LGAR_ST_NAN;
    // -dop/dse = op sp / (base se);  dop/dm = op ln(base) + op sp ln(se) / (base m)   (k_se_partials_core)
    const bool se0 = (se[e] == 0.0);
    const double rbase = __drcp_rn(base[e]);
    const double sp_over = se0 ? 0.0 : sp[e] * inv_se[e];
    const double ndop_dse = op[e] * sp_over * rbase;
    const double lnse = se0 ? 0.0 : lse[e];
    const double dop_dm = op[e] * lb[e] + op[e] * sp[e] * lnse * (rbase * inv_m);
    const double dk_se = ksat * ((se0 ? 0.0 : 0.5 * (t * t) * (rs * inv_se[e])) + 2.0 * t * rs * ndop_dse);
    const double dkm = ksat * rs * 2.0 * t * (-dop_dm);
    r.dk_h[e] = dk_se * dse_dh[e];
    r.dk_a[e] = dk_se * dse_da[e];
    r.dk_n[e] = dk_se * dse_dn[e];
    r.dk_m[e] = dk_se * dse_dm[e] + dkm;
  }
  return r;
}

// Taped pass: value (the forward kernel's bits) and the partials of Geff w.r.t. theta_1, theta_2, alpha, n, m of
// one request per lane.  G = dh sum_k w_k K_k, geff = |G / ksat| (d geff / d ksat = 0: K is proportional to ksat);
// K_k = K(Se(h_k)), h_k = h_i + k dh; node 0 is K(Se_i), a direct function of Se_i in the reference graph
// (green_ampt.py:75).  The owner lane turns the five partials into one tape entry.
template <class ST>
__device__ __noinline__ void geff_batch_eval_taped(GeffQueue* q, const ST* soil, int L, int nint) {
  const int lane = threadIdx.x & 31;
  const int meta = q->meta[lane];
  const bool have = meta >= 0;
  const Soil s = gather_soil(soil, L, have ? (meta & 31) : lane, have ? ((meta >> 8) & 7) : 0);
  if (have) {
    const GeffStart g0 = geff_start(q->a[lane], q->b[lane], s, nint);
    const double h_i = g0.h_i, dh = g0.dh;
    double k1 = g0.k1;
    const P4 pi = h_se_partials_core(g0.se_i, s.alpha, s.ninv_m, s.inv_m, s.inv_n, h_i);
    const P4 pf = h_se_partials_core(g0.se_f, s.alpha, s.ninv_m, s.inv_m, s.inv_n, g0.h_f);
    const NodeFull n0 = k_node_full(h_i, true, g0.se_i, s.alpha, s.n, s.m, s.inv_m, s.ksat);
    int st = g0.st;
    if (st == 0 && n0.bad) st = n0.bad;
    double S = 0.5 * k1, Csei = 0.5 * n0.dk_se, Ahi = 0.0, Ahf = 0.0, Ca = 0.0, Cn = 0.0, Cm = 0.5 * n0.dk_m;
    const double half = dh / 2.0;
    const double inv_nint = 1.0 / (double)nint;
    double geff = 0.0;
    double h2 = h_i + dh;
#pragma unroll 1
    for (int i = 0; i < nint; i += 2) {
      const double ha = h2, hb = ha + dh;
      h2 = hb + dh;
      const NodeFull2 nf = k_node_full_x2(ha, (i + 1 < nint) ? hb : ha, s.alpha, s.n, s.m, s.inv_m, s.ksat);
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int node = i + e + 1;
        if (node <= nint) {
          if (st == 0 && nf.bad[e]) st = nf.bad[e];
          geff = geff + ((k1 + nf.K[e]) * half);
          k1 = nf.K[e];
          const double wgt = (node == nint) ? 0.5 : 1.0;
          const double frac = (double)node * inv_nint;
          S += wgt * nf.K[e];
          Ahi += wgt * nf.dk_h[e] * (1.0 - frac);
          Ahf += wgt * nf.dk_h[e] * frac;
          Ca += wgt * nf.dk_a[e];
          Cn += wgt * nf.dk_n[e];
          Cm += wgt * nf.dk_m[e];
        }
      }
    }
    const double value = fabs(geff / s.ksat);
    const double G = dh * S;
    const double sg = (G / s.ksat > 0.0) ? 1.0 : ((G / s.ksat < 0.0) ? -1.0 : 0.0);
    const double f = sg / s.ksat;
    const double dG_dhi = -S * inv_nint + dh * Ahi;
    const double dG_dhf = S * inv_nint + dh * Ahf;
    const double inv_span = 1.0 / (s.the - s.thr);
    q->a[lane] = value;
    q->st[lane] = st;
    double* dq = g_geffq_partials[threadIdx.x >> 5] + lane;
    dq[0 * 32] = f * (dG_dhi * pi.a + dh * Csei) * inv_span;
    dq[1 * 32] = f * (dG_dhf * pf.a) * inv_span;
    dq[2 * 32] = f * (dh * Ca + dG_dhi * pi.b + dG_dhf * pf.b);
    dq[3 * 32] = f * (dh * Cn + dG_dhi * pi.c + dG_dhf * pf.c);
    dq[4 * 32] = f * (dh * Cm + dG_dhi * pi.d + dG_dhf * pf.d);
  }
  __syncwarp();
}

// ---- queue protocol shared by the three call sites of a sub-step ------------------------------------------------
__device__ __forceinline__ void geffq_put(GeffQueue* q, int slot, int owner, int layer, double t1, double t2) {
  q->a[slot] = t1;
  q->b[slot] = t2;
  q->meta[slot] = owner | (layer << 8);
}
// result of slot `slot`, owned by this lane (value + status; the taped pass records one entry with five partials).
// geffq_take counts the request's work and raises its status.
__device__ __forceinline__ void geffq_take(const GeffQueue* q, int slot, int nint, Ctx& c) {
  c.cnt[C_GEFF]++;
  c.cnt[C_H_SE] += 2;
  c.cnt[C_K_SE] += 1 + nint;
  c.cnt[C_SE_H] += nint;
  const int st = q->st[slot];
  if (st) raise(c, st);
}
__device__ __forceinline__ double geffq_get(GeffQueue* q, int slot, double /*t1*/, double /*t2*/, const SoilT<double>&, int nint,
                                            Ctx& c) {
  geffq_take(q, slot, nint, c);
  return q->a[slot];
}
__device__ __forceinline__ Var geffq_get(GeffQueue* q, int slot, const Var& t1, const Var& t2, const SoilT<Var>& s, int nint,
                                         Ctx& c) {
  geffq_take(q, slot, nint, c);
  const int ids[5] = {t1.id, t2.id, s.id_alpha, s.id_n, s.id_m};
  const double* dq = g_geffq_partials[threadIdx.x >> 5] + slot;
  const double d[5] = {dq[0 * 32], dq[1 * 32], dq[2 * 32], dq[3 * 32], dq[4 * 32]};
  return tape_record_n(q->a[slot], 5, ids, d);
}
// evaluate the batch in the queue: values (forward) or values and partials (taped pass)
__device__ __forceinline__ void geffq_eval(GeffQueue* q, const SoilT<double>* soil, int L, int nint) {
  geff_batch_eval(q, soil, L, nint);
}
__device__ __forceinline__ void geffq_eval(GeffQueue* q, const SoilT<Var>* soil, int L, int nint) {
  geff_batch_eval_taped(q, soil, L, nint);
}

// At most one request per lane (insert_water, calc_dry_depth): slot = lane.  Warp-convergent.
// GM (Geff mode) = 0: trapezoid only (the production forward kernel: the closed form is compiled out of the call
// sites); GM = 2: run-time switch, nint < 0 selects the closed form.
template <int GM, class R>
__device__ __forceinline__ R geff_one_per_lane(bool need, const R& theta_1, const R& theta_2, int layer, const SoilT<R>* soil,
                                               int L, int nint, GeffQueue* q, Ctx& c) {
  if (GM == 2 && nint < 0)  // closed form: per lane, no queue
    return geff_closedR(need, theta_1, theta_2, soil[need ? layer : 0], c);
  if (!__any_sync(0xffffffffu, need)) return R(0.0);
  const int lane = threadIdx.x & 31;
  q->meta[lane] = -1;
  if (need) geffq_put(q, lane, lane, layer, val(theta_1), val(theta_2));
  __syncwarp();
  geffq_eval(q, soil, L, nint);
  R r(0.0);
  if (need) r = geffq_get(q, lane, theta_1, theta_2, soil[layer], nint, c);
  __syncwarp();
  return r;
}

// ------------------------------------------------------------------------------------
// Column: per-thread view of the front list in shared memory + scalar state in registers.
// R = double: forward kernel.  R = Var: taped pass (values in the same shared-memory array, tape
// ids of the five fields in a parallel int array).
// ------------------------------------------------------------------------------------
template <int FM, class R, int LM = 0>
struct Column {
  static constexpr bool TAPED = !std::is_same<R, double>::value;
  double* fb;        // this thread's slot in the field array
  short* ib;         // this thread's slot in the 16-bit tape-id array (TAPED only; ids < 32768)
  uint8_t* gb;       // this thread's slot in the flag array: bits 0-2 layer_num attr, bit 7 to_bottom
  int L;             // number of layers
  int n;             // total number of fronts
  unsigned cntpk;    // per-layer list lengths, 8 bits each
  SoilT<R> soil[MAXL];
  double cum[MAXL];  // cumulative layer thickness (GlobalParams.py:103-110)
  double thick[MAXL];
  double pdm;        // ponded_depth_max
  int id_pdm;        // TAPED: tape id of ponded_depth_max when its gradient is requested (dpLGAR.py:48), else -1
  __device__ __forceinline__ R pdmR() const {
    if constexpr (TAPED) return Var(pdm, id_pdm);
    else return pdm;
  }
  R psi_wp;          // AET: capillary head at which AET = 0.5 PET (aet.py:37-43); column constant
  R ponded_water, ending_volume;
  double previous_precip;
  R giuh[NGIUH];
  bool empty_list;   // set by mass_balance() when a layer list is empty (IndexError in the reference)
  // Search log (reverse pass): the two root finders of a sub-step (Layer.theta_mass_balance, Layer.check_column_mass)
  // only STEER psi / the depth by constants -- they never appear on the tape (Q14) -- so the forward kernel, when it
  // stores checkpoints, also logs where every search ended (one double per search, per lane and chunk, in program
  // order) and the taped recompute of the reverse kernel reads the end point instead of searching again: no
  // upper-layer sums (P1), no iterations (P2).  A lane whose log is exhausted searches as usual.
  double* logp;      // this lane's log of the current chunk: entry k at logp[k * log_stride]; nullptr = no log
  int log_pos;       // entries written / consumed so far
  int log_valid;     // write mode: capacity; read mode: entries the forward pass stored (<= capacity)
  static constexpr int log_mode = LM;  // 0 off (production forward: compiled out), 1 write (forward with checkpoints),
                                       // 2 read (taped recompute)
  int log_stride;

  static constexpr unsigned long long LOG_NAN = 0x7ff8000000000000ULL;
  enum LogMark { LOG_SINGLE = 1, LOG_NONE = 2, LOG_SCALE = 16 };
  __device__ __forceinline__ void log_put(double v) {
    if (log_pos < log_valid) logp[(size_t)log_pos * log_stride] = v;
    log_pos++;
  }
  __device__ __forceinline__ void log_put_mark(int mark) { log_put(__longlong_as_double((long long)(LOG_NAN | (unsigned)mark))); }
  __device__ __forceinline__ bool log_get(double& v) {
    if (log_pos >= log_valid) {
      log_pos = 0x40000000;  // exhausted: search from here on (and never come back to the log of this chunk)
      log_valid = 0;
      return false;
    }
    v = __ldcg(logp + (size_t)log_pos * log_stride);
    log_pos++;
    return true;
  }

  __device__ __forceinline__ double& f(int fld, int i) { return fb[(fld * FM + i) * NT]; }
  __device__ __forceinline__ short& fid(int fld, int i) { return ib[(fld * FM + i) * NT]; }
  // generic get / set of a field as R
  __device__ __forceinline__ R g(int fld, int i) {
    if constexpr (TAPED) return Var(f(fld, i), (int)fid(fld, i));
    else return f(fld, i);
  }
  __device__ __forceinline__ void s(int fld, int i, const R& x) {
    if constexpr (TAPED) {
      f(fld, i) = x.v;
      fid(fld, i) = (short)x.id;
    } else {
      f(fld, i) = x;
    }
  }
  template <class Q>
  __device__ __forceinline__ Q gq(int fld, int i) {
    if constexpr (std::is_same<Q, double>::value) return f(fld, i);
    else return g(fld, i);
  }
  __device__ __forceinline__ int lay(int i) const { return gb[i * NT] & 7; }
  __device__ __forceinline__ bool tb(int i) const { return (gb[i * NT] & 0x80) != 0; }
  __device__ __forceinline__ void set_flag(int i, int layer, bool to_bottom) {
    gb[i * NT] = (uint8_t)((layer & 7) | (to_bottom ? 0x80 : 0));
  }
  __device__ __forceinline__ int cnt(int l) const { return (cntpk >> (8 * l)) & 0xff; }
  __device__ __forceinline__ void add_cnt(int l, int d) { cntpk += (unsigned)d << (8 * l); }
  __device__ __forceinline__ int off(int l) const {
    int o = 0;
    for (int k = 0; k < l; k++) o += cnt(k);
    return o;
  }
  __device__ __forceinline__ void copy_front(int dst, int src) {
#pragma unroll
    for (int k = 0; k < 5; k++) {
      f(k, dst) = f(k, src);
      if constexpr (TAPED) fid(k, dst) = fid(k, src);
    }
    gb[dst * NT] = gb[src * NT];
  }
  // list.insert(0, front) on layer list l
  __device__ __forceinline__ bool insert_at(int pos, int l, Ctx& c) {
    if (n >= FM) {
      raise(c, LGAR_ST_FRONT_OVERFLOW);
      return false;
    }
    for (int i = n; i > pos; i--) copy_front(i, i - 1);
    n++;
    add_cnt(l, 1);
    return true;
  }
  // list.pop(i) on the list holding flat index pos
  __device__ __forceinline__ void erase_at(int pos, int l) {
    for (int i = pos; i < n - 1; i++) copy_front(i, i + 1);
    n--;
    add_cnt(l, -1);
  }
  // WettingFront.is_equal (WettingFront.py:76-84): value equality on depth, psi, dzdt (Q3)
  __device__ __forceinline__ bool is_equal(int a, int b) {
    return f(F_DEPTH, a) == f(F_DEPTH, b) && f(F_PSI, a) == f(F_PSI, b) && f(F_DZDT, a) == f(F_DZDT, b);
  }
  // list layer of flat front index i
  __device__ __forceinline__ int list_layer(int i) const {
    int l = 0, o = cnt(0);
    while (i >= o && l < MAXL - 1) {
      l++;
      o += cnt(l);
    }
    return l;
  }
  // Layer.get_len_layers (Layer.py:1145-1155)
  __device__ __forceinline__ int len_layers(int l) const { return (l < L - 1) ? cnt(l) : cnt(l) - 1; }

  // ---- Layer.mass_balance (Layer.py:795-824); association S0 + (S1 + (S2 ...)).
  //      Q = double evaluates values only (root-finder loops), Q = R is on the tape.
  //      layer_water_t: the inner sum of layer l, whose list starts at flat index o (the soil-moisture output W_l,
  //      lgar_b200.h); 0 for an empty list.
  template <class Q>
  __device__ __forceinline__ Q layer_water_t(int l, int o) {
    const double base = (l == 0) ? 0.0 : (cum[l] - thick[l]);
    const int nf = cnt(l);
    Q sum(0.0);
    for (int i = 0; i < nf - 1; i++)
      sum = sum + (gq<Q>(F_DEPTH, o + i) - base) * (gq<Q>(F_THETA, o + i) - gq<Q>(F_THETA, o + i + 1));
    if (nf > 0) sum = sum + (gq<Q>(F_DEPTH, o + nf - 1) - base) * gq<Q>(F_THETA, o + nf - 1);
    return sum;
  }
  template <class Q>
  __device__ Q mass_balance_t() {
    Q s_l[MAXL];
    empty_list = false;
    int o = 0;
    for (int l = 0; l < L; l++) {
      const int nf = cnt(l);
      s_l[l] = layer_water_t<Q>(l, o);
      if (nf == 0) empty_list = true;  // wetting_fronts[0] of an empty list: IndexError in the reference
      o += nf;
    }
    return layer_sum(s_l);
  }
  __device__ __forceinline__ R mass_balance() { return mass_balance_t<R>(); }
  // sum of per-layer terms in the reference's association x[0] + (x[1] + (... + x[L-1]))
  template <class Q>
  __device__ __forceinline__ Q layer_sum(const Q* x) const {
    Q tot = x[L - 1];
    for (int l = L - 2; l >= 0; l--) tot = x[l] + tot;
    return tot;
  }

  // ---- soil-moisture output theta(z) (lgar_b200.h): flat index of the first front of the list of the layer holding
  //      depth z (cum[l-1] < z <= cum[l]) whose depth >= z; -1 if z lies below the column or no front qualifies.
  //      A selection: no arithmetic, nothing on the tape.
  __device__ __forceinline__ int front_at_depth(double z) const {
    int o = 0;
    for (int l = 0; l < L; l++) {
      const int nf = cnt(l);
      if (z <= cum[l]) {
        for (int i = o; i < o + nf; i++)
          if (fb[(F_DEPTH * FM + i) * NT] >= z) return i;
        return -1;
      }
      o += nf;
    }
    return -1;
  }

  // ---- free-drainage front (models/dpLGAR.py:328-338, Layer.py:134-162): arg-min psi, ties ->
  //      deeper; else-branch torch.isclose(psi_i, psi, atol=1e-8) with default rtol 1e-5
  __device__ int free_drainage_front() {
    int w = 0;
    double psi = f(F_PSI, 0);
    for (int i = 0; i < n; i++) {
      const double p = f(F_PSI, i);
      if (p <= psi) {
        psi = p;
        w = i;
      } else {
        bool close;
        if (isfinite(p) && isfinite(psi)) close = fabs(p - psi) <= 1e-8 + 1e-5 * fabs(psi);
        else close = (p == psi);
        if (close) {
          psi = p;
          w = i;
        }
      }
    }
    return w;
  }

  // ---- Layer.check_column_mass (Layer.py:655-701): if the free-drainage front is saturated, its
  //      depth is stepped by +/-0.01*factor (factor *= 0.001 at every down-switch) until the column
  //      mass error lies in [0, 2e-12].  The column mass is monotone in that depth, so long runs of
  //      equal steps are crossed with doubling/halving probes on depths computed by
  //      advance_rounded(): the visited depths are exactly the reference's.  Autograd: the depth is
  //      shifted by constants only, so the tape id of the depth is kept (straight-through, Q14).
  __device__ void check_column_mass(int fd, double old_mass, double percolation, double aet, Ctx& c) {
    const double theta_e_k1 = soil[lay(fd)].the;
    const double mass_timestep = (old_mass + percolation) - (aet + 0.0);
    if (fabs(f(F_THETA, fd) - theta_e_k1) < 1e-12) {
      double current_mass = mass_balance_t<double>();
      double err = fabs(current_mass - mass_timestep);
      bool switched = false;
      double factor = 1.0;
      double depth_new = f(F_DEPTH, fd);
      long long it = 0;
      int run_len = 0;
      bool run_up = false;
      if (log_mode == 2 && fabs(err - 1e-12) > 1e-12) {  // the forward pass logged where this search ended
        double v;
        if (log_get(v)) {
          f(F_DEPTH, fd) = v;
          return;
        }
      }
      while (fabs(err - 1e-12) > 1e-12) {
        if (++it > c.iter_cap) {
          raise(c, LGAR_ST_ITER_CAP);
          break;
        }
        c.cnt[C_COLMASS]++;
        const bool up = current_mass < mass_timestep;
        const double fac_before = factor;
        if (up) {
          depth_new = depth_new + 0.01 * factor;
          switched = false;
        } else {
          if (!switched) {
            switched = true;
            factor = factor * 0.001;
          }
          depth_new = depth_new - (0.01 * factor);
        }
        f(F_DEPTH, fd) = depth_new;
        current_mass = mass_balance_t<double>();
        err = fabs(current_mass - mass_timestep);
        if (up == run_up && factor == fac_before) run_len++;
        else {
          run_len = 1;
          run_up = up;
        }
        if (run_len >= 3 && fabs(err - 1e-12) > 1e-12 && (current_mass < mass_timestep) == run_up &&
            fabs(depth_new) >= 64.0 * (0.01 * factor)) {
          run_len = 0;  // re-armed after three more regular steps of the same run
          const double step = 0.01 * factor;
          long long stride = 4;
          bool shrinking = false;
          while (stride >= 2) {
            c.cnt[C_COLMASS]++;
            const double cand = advance_rounded(depth_new, up ? step : -step, stride);
            f(F_DEPTH, fd) = cand;
            const double m = mass_balance_t<double>();
            const double e = fabs(m - mass_timestep);
            // (mass monotone in the depth: the iterates in between lie between the two end points.  Either the mass
            // moves by more than the rounding noise per step, or both end points are far (> 1e-11, a hundred times the
            // rounding noise of a column mass) from the [0, 2e-12] window the loop stops in, or the step has fallen
            // below the spacing of the depth (cand == depth_new: nothing can change any more) -- the FLAT case: theta
            // of the free-drainage front equals theta of
            // the front below, the mass does not depend on the depth, the reference never leaves the loop
            // (Layer.py:681-701 has no stall guard) and this column ends with ITER_CAP.  Without the second clause
            // such a column walked its million iterations one by one: 1.7 s of a warp, 2.5 % of the bench shard's
            // work and, when it happened in the last rows of the record, the tail of the whole pass.)
            const bool cont = (up ? (m < mass_timestep) : !(m < mass_timestep)) && (fabs(e - 1e-12) > 1e-12) &&
                              (fabs(cand) >= 64.0 * step) && ((cand < 0.0) == (depth_new < 0.0)) &&
                              (fabs(m - current_mass) >= 1e-13 * (double)stride || (e > 1e-11 && err > 1e-11) || cand == depth_new);
            if (cont) {  // identical to `stride` regular iterations of this run
              depth_new = cand;
              current_mass = m;
              err = e;
              it += stride;
              if (it > c.iter_cap) break;  // (a flat run never ends: the outer loop raises ITER_CAP)
              stride = shrinking ? (stride >> 1) : (stride << 1);
              if (stride > (1LL << 40)) stride = 1LL << 40;
            } else {
              shrinking = true;
              stride >>= 1;
            }
          }
          f(F_DEPTH, fd) = depth_new;
        }
      }
      if (log_mode == 1 && it > 0) log_put(depth_new);
    }
  }

  // ---- Layer.move_wetting_fronts (Layer.py:1254-1307): sweep from the deepest front to the top,
  //      WARP-CONVERGENT: every lane of the warp calls it.  Round r handles, in every lane, the r-th
  //      front counted from the bottom of that lane's column.  All pow-heavy work runs in batched,
  //      convergent phases:
  //        P1  upper-layer sums of compute_wetting_front_mass (:561-644) / populate_delta_thickness
  //            (:177-209)
  //        P2  Layer.theta_mass_balance (:242-318) + recalculate_mass (:211-240): one root-finder
  //            iteration per warp pass for every lane that has a request; the sequence of psi values
  //            a lane visits is exactly the reference's
  //        P3  psi = h(Se(theta)) tail
  //      previous_state[i] of the reference equals the state at entry of this sweep (nothing modifies
  //      fronts between copy_states() and here), and only the OLD theta/psi of the front below
  //      (previous_next_front) and the front's own old values are read, so the snapshot is carried in
  //      registers instead of a copy of the list.
  //      Autograd (Q14): P1 and P2 only steer the search for psi, which is shifted by constants, so they
  //      run on plain values; the tape sees theta = theta_l(scale * psi_in + const).
  enum Kind { K_NONE = 0, K_DEEPEST = 1, K_INLAYER0 = 2, K_INLAYER_DEEP = 3, K_BASE = 4 };

  __device__ void move_wetting_fronts_warp(bool go, int fd, const R& infiltration, const R& aet, const R& old_mass,
                                           double dt, Ctx& c) {
    const unsigned FULL = 0xffffffffu;
    go = go && (c.st == 0);
    const int num_wf = go ? n : 0;
    const int rmax = warp_max(num_wf);
    R old_theta_below(0.0), old_psi_below(0.0);  // previous_state of front i+1
    int l = L - 1;
    int o = go ? n - cnt(L - 1) : 0;  // flat offset of list l
    for (int r = 0; r < rmax; r++) {
      const int i = num_wf - 1 - r;
      const bool mine = go && (i >= 0) && (c.st == 0);
      int kind = K_NONE, lyr = 0, nup = 0;
      bool add_flux = false;
      double psi_cm = 0.0, psi_old = 0.0, psi_below = 0.0, psi_below_old = 0.0;
      double prior_mass = 0.0, new_mass = 0.0, own_dth = 0.0, own_dtk = 0.0;
      R old_depth(0.0), old_theta(0.0), old_psi(0.0), psi_in(0.0);
      if (mine) {
        while (i < o) {  // step to the list above
          l--;
          o -= cnt(l);
        }
        lyr = l;
        const int last = o + cnt(l) - 1;  // wetting_fronts[-1] of this list
        old_depth = g(F_DEPTH, i);
        old_theta = g(F_THETA, i);
        old_psi = g(F_PSI, i);
        if (i < num_wf - 1) {
          if (is_equal(i, last)) {
            // deepest_layer_front (Layer.py:389-418): theta = theta_l(psi of the front below)
            if (!(i < last || l < L - 1)) raise(c, LGAR_ST_NULL_NEIGHBOUR);
            kind = K_DEEPEST;
            psi_in = g(F_PSI, i + 1);
            psi_cm = val(psi_in);
          } else {
            // wetting_front_in_layer (Layer.py:420-547); i < last, so next is in the same list
            const R dzdt = g(F_DZDT, i);
            if (l == 0) {
              kind = K_INLAYER0;
              R pm = old_depth * (old_theta - old_theta_below);
              if (is_equal(fd, i)) pm = pm + (infiltration - (0.0 + aet));
              R depth = old_depth + (dzdt * dt);
              depth = tmin(depth, cum[L - 1]);
              s(F_DEPTH, i, depth);
              const bool zero_dzdt = vabs(dzdt) <= 1e-8;  // isclose(dzdt, 0, rtol=1e-8) (Q2)
              if (!(zero_dzdt && !tb(i))) {
                R potential_theta = (pm / depth) + g(F_THETA, i + 1);
                s(F_THETA, i, tmin(soil[0].the, potential_theta));
              }
            } else {
              kind = K_INLAYER_DEEP;
              const double plt = cum[l - 1];
              const R depth = old_depth + (dzdt * dt);
              s(F_DEPTH, i, depth);
              psi_in = old_psi;
              psi_old = val(old_psi);
              psi_below_old = val(old_psi_below);
              psi_cm = val(old_psi);
              psi_below = f(F_PSI, i + 1);
              prior_mass = (val(old_depth) - plt) * (val(old_theta) - val(old_theta_below));
              new_mass = (val(depth) - plt) * (val(old_theta) - f(F_THETA, i + 1));
              nup = l;
              own_dth = f(F_THETA, i + 1);
              own_dtk = val(depth) - plt;
              add_flux = is_equal(fd, i);
            }
          }
        }
        if (num_wf == L && l == L - 1) {
          // base_case (Layer.py:320-387): one front per layer, this is the bottom one
          kind = K_BASE;
          const R depth = g(F_DEPTH, i) + g(F_DZDT, i) * dt;
          s(F_DEPTH, i, depth);
          psi_in = g(F_PSI, i);
          psi_old = val(old_psi);
          psi_cm = val(psi_in);
          const double base = (l > 0) ? cum[l - 1] : 0.0;
          prior_mass = (val(old_depth) - base) * (val(old_theta) - 0.0);
          new_mass = (val(depth) - base) * (f(F_THETA, i) - 0.0);
          if (L < 2) raise(c, LGAR_ST_NULL_NEIGHBOUR);
          nup = L - 1;
          own_dth = 0.0;
          own_dtk = val(depth) - base;
          add_flux = (lay(fd) == l);
        }
      }
      // ---- search log (taped recompute): the end point of this front's search, if the forward pass logged it
      bool log_hit = false, log_single = false, log_have = false;
      double log_psi = 0.0, log_scale = 1.0;
      if (log_mode == 2 && mine && kind >= K_INLAYER_DEEP && c.st == 0) {
        double v;
        if (log_get(v)) {
          int mark = isnan(v) ? (int)((unsigned long long)__double_as_longlong(v) & 0xffffULL) : 0;
          if (mark >= LOG_SCALE) {  // psi was scaled by 0.1^k on the way (the `psi < 0` guard): same product chain
            for (int k = LOG_SCALE; k < mark; k++) log_scale = log_scale * 0.1;
            log_get(v);
            mark = 0;
          }
          log_hit = true;
          log_single = (mark == LOG_SINGLE);
          log_have = (mark == 0);
          log_psi = v;
          nup = 0;  // no upper-layer sums, no iterations for this lane
          add_flux = false;
        }
      }
      // ---- P1: sums over the layers above (convergent, values only)
      double dth[MAXL - 1], dtk[MAXL - 1];
      const int nupmax = warp_max(nup);
#pragma unroll
      for (int k = 0; k < MAXL - 1; k++) {
        dth[k] = 0.0;
        dtk[k] = 0.0;
        if (k < nupmax) {
          if (k < nup) {
            const Soil& sk = soil[k];
            if (kind == K_INLAYER_DEEP) {
              const double2 ob = theta_from_h_x2(psi_old, sk, psi_below_old, sk, true, c);
              double local_delta_old = ob.x - ob.y;
              double layer_thickness = cum[k] - 0.0;  // sic (Q5): cumulative thickness
              prior_mass = prior_mass + (layer_thickness * local_delta_old);
              const double2 nb2 = theta_from_h_x2(psi_cm, sk, psi_below, sk, true, c);
              new_mass = new_mass + (layer_thickness * (nb2.x - nb2.y));
              dth[k] = nb2.y;
              dtk[k] = layer_thickness;
            } else {  // K_BASE
              const double2 on = theta_from_h_x2(psi_old, sk, psi_cm, sk, true, c);
              prior_mass = prior_mass + thick[k] * (on.x - 0.0);
              new_mass = new_mass + thick[k] * (on.y - 0.0);
              dth[k] = 0.0;
              dtk[k] = thick[k];
            }
          }
        }
      }
      if (add_flux) prior_mass = prior_mass + val(infiltration) - (0.0 + val(aet));

      // ---- P2: batched theta_mass_balance (values only)
      const double tol = 1e-12;
      const Soil own = soil[lyr];  // hoisted into registers for the iteration loop
      const Soil up0 = soil[0];
      const Soil up1 = soil[(MAXL > 2) ? 1 : 0];
      double delta_mass = fabs(new_mass - prior_mass);
      double theta = 0.0;
      double psi_scale = 1.0;   // d psi_final / d psi_in: 0.1 per `psi = psi_prev * 0.1` guard hit
      bool have_theta = false;  // theta already holds theta_l(psi_cm) (value)
      const bool wants = mine && (kind == K_DEEPEST || kind >= K_INLAYER_DEEP) && (c.st == 0);
      // early return `delta_mass <= tolerance` (and the deepest-front case): one evaluation
      const bool single = wants && (kind == K_DEEPEST || (log_hit ? log_single : (delta_mass <= tol)));
      bool active = wants && kind >= K_INLAYER_DEEP && !log_hit && (delta_mass > tol);
      if (log_hit && log_have) {
        psi_cm = log_psi;
        psi_scale = log_scale;
        have_theta = true;
      }
      {
        bool switched = false;
        double factor = 1.0;
        double psi_prev = psi_cm;
        double prev_scale = 1.0;
        double delta_mass_prev = delta_mass;
        int count_no_mass_change = 0;
        long long it = 0;
        // run tracking for the exact jump: a "run" is a maximal sequence of iterations that step psi
        // in the same direction with the same step.  Only the coarse runs (step 0.1 or 0.01) can be
        // long (psi travelling hundreds of cm after a wetting/drying event); they are crossed by
        // doubling/halving probes on psi values computed with advance_rounded(), so the lane lands on
        // exactly the psi the reference's one-step-at-a-time loop reaches before the run ends.
        int run_len = 0;        // regular iterations taken so far in the current run
        bool run_up = false;
        long long stride = 0;   // > 0: next pass is a probe `stride` steps ahead
        bool shrinking = false;
        // predictive probe: after the single up-step that ends a decade, the next down-run (10x finer step)
        // needs k <= 10 steps to cross again; k is estimated by the secant through the last two evaluations
        // and the lane probes k-1 steps ahead at once.  Acceptance is the same exact test as for galloping
        // probes, so a wrong estimate only costs one evaluation.
        bool pred = false;
        while (__any_sync(FULL, active)) {
          if (active) {
            if (it > c.iter_cap) {
              raise(c, LGAR_ST_ITER_CAP);
              active = false;
            }
          }
          if (active) {
            c.cnt[C_ROOT]++;
            const bool probe = stride >= 2;
            const bool up = probe ? run_up : (new_mass > prior_mass);
            double step;
            double psi_try, psi_prev_try = psi_prev;
            double scale_try = psi_scale, prev_scale_try = prev_scale;
            bool sw = switched;
            double fac = factor;
            if (probe) {
              if (pred) fac = factor * 0.1;  // the first step of a down-run after an up-step shrinks the factor
              step = 0.1 * fac;
              psi_try = advance_rounded(psi_cm, up ? step : -step, stride);
              if (!up) psi_prev_try = advance_rounded(psi_cm, -step, stride - 1);
              if (!up) prev_scale_try = psi_scale;
            } else if (up) {
              step = 0.1 * factor;
              psi_try = psi_cm + step;
              sw = false;
            } else {
              if (!sw) {
                sw = true;
                fac = fac * 0.1;
              }
              step = 0.1 * fac;
              psi_prev_try = psi_cm;
              prev_scale_try = psi_scale;
              psi_try = psi_cm - step;
              if (psi_try < 0.0 && psi_prev_try != 0.0) {
                psi_try = psi_prev_try * 0.1;
                scale_try = prev_scale_try * 0.1;
              }
            }
            Ctx cc;  // guards raised by a rejected probe must not kill the column
            cc.st = 0;
            cc.cnt[C_THETA_H] = 0;
            // own layer + first upper layer evaluated as an interleaved pair; further upper layers singly
            const double2 t01 = theta_from_h_x2_inl(psi_try, own, psi_try, up0, nup > 0, cc);
            const double th = t01.x;
            double mass_layers = 0.0 + (own_dtk * (th - own_dth));
            if (nup > 0) mass_layers = mass_layers + dtk[0] * (t01.y - dth[0]);
            if (nup > 1) {
              double theta_layer = theta_from_h_inl(psi_try, up1, cc);
              mass_layers = mass_layers + dtk[1] * (theta_layer - dth[1]);
            }
#pragma unroll
            for (int k = 2; k < MAXL - 1; k++) {
              if (k < nup) {
                double theta_layer = theta_from_h(psi_try, soil[k], cc);
                mass_layers = mass_layers + dtk[k] * (theta_layer - dth[k]);
              }
            }
            c.cnt[C_THETA_H] += cc.cnt[C_THETA_H];
            const double dm = fabs(mass_layers - prior_mass);
            if (probe) {
              const bool cont = up ? (mass_layers > prior_mass) : (mass_layers <= prior_mass);
              const bool ok = cont && cc.st == 0 && dm > tol && (psi_try > 64.0 * step) &&
                              fabs(mass_layers - new_mass) >= 1e-13 * (double)stride;  // 100x the stall guard
              if (ok) {  // identical to `stride` regular iterations of this run
                psi_cm = psi_try;
                psi_prev = psi_prev_try;
                prev_scale = prev_scale_try;
                theta = th;
                have_theta = true;
                new_mass = mass_layers;
                delta_mass = dm;
                delta_mass_prev = dm;
                count_no_mass_change = 0;
                it += stride;
                if (pred) {  // the run has started: factor was shrunk by its first step
                  switched = true;
                  factor = fac;
                  run_len = 1;
                  run_up = false;
                  stride = 0;
                } else {
                  stride = shrinking ? (stride >> 1) : (stride << 1);
                  if (stride > (1LL << 40)) stride = 1LL << 40;
                }
              } else if (pred) {
                stride = 0;  // estimate too optimistic: step normally
              } else {
                shrinking = true;
                stride >>= 1;
              }
              pred = false;
              if (stride < 2) stride = 0;
            } else {
              it++;
              if (cc.st) raise(c, cc.st);  // the reference raised inside theta_from_h
              const double psi_a = psi_cm, mass_a = new_mass;  // previous evaluation (for the secant estimate)
              if (up == run_up && fac == factor) run_len++;
              else {
                run_len = 1;
                run_up = up;
              }
              psi_cm = psi_try;
              psi_prev = psi_prev_try;
              psi_scale = scale_try;
              prev_scale = prev_scale_try;
              switched = sw;
              factor = fac;
              theta = th;
              have_theta = true;
              new_mass = mass_layers;
              delta_mass = dm;
              bool stop = !(delta_mass > tol);
              if (c.st) stop = true;
              if (fabs(psi_cm - psi_prev) < 1e-15 && factor < 1e-13) stop = true;
              if (fabs(delta_mass - delta_mass_prev) < 1e-15) count_no_mass_change++;
              else count_no_mass_change = 0;
              if (count_no_mass_change == 5) stop = true;
              if (psi_cm <= 0.0 && psi_prev < 1e-50) stop = true;
              delta_mass_prev = delta_mass;
              if (stop) active = false;
              // start probing if the run goes on: same direction next, coarse step, far from psi = 0
              else if (run_len >= 3 && factor >= 0.05 && (new_mass > prior_mass) == run_up &&
                       count_no_mass_change == 0 && psi_cm > 64.0 * (0.1 * factor)) {
                stride = 4;
                shrinking = false;
                run_len = 0;  // re-armed after three more regular steps of the same run
              } else if (up && !(new_mass > prior_mass) && mass_layers != mass_a) {
                // an up-step just crossed below prior_mass: the next iteration starts a down-run with step s2
                const double s2 = 0.1 * (factor * 0.1);
                const double psi_star = psi_cm - (mass_layers - prior_mass) * (psi_cm - psi_a) / (mass_layers - mass_a);
                const double kest = (psi_cm - psi_star) / s2;
                // (skip when one fine step changes the mass by less than the probe's monotonicity margin)
                if (kest >= 3.0 && kest <= 4096.0 && psi_cm > 128.0 * s2 && fabs(mass_layers - mass_a) >= 4e-12) {
                  stride = (long long)kest - 1;  // one step of margin before the estimated crossing
                  pred = true;
                  run_up = false;
                  shrinking = false;
                }
              }
            }
          }
        }
      }
      if (log_mode == 1 && wants && kind >= K_INLAYER_DEEP) {  // forward with checkpoints: log the end point
        if (single) log_put_mark(LOG_SINGLE);
        else if (have_theta) {
          if (psi_scale != 1.0) {
            int k = 0;
            for (double sc = 1.0; sc != psi_scale && k < 300; k++) sc = sc * 0.1;
            log_put_mark(LOG_SCALE + k);
          }
          log_put(psi_cm);
        } else log_put_mark(LOG_NONE);
      }
      // ---- P3: theta = theta_l(psi_final) on the tape, psi = h(Se(theta)) tail
      if (mine && c.st == 0 && (kind == K_DEEPEST || kind >= K_INLAYER_DEEP)) {
        R thR(0.0);  // NaN delta_mass: the reference returns its initial theta = 0.0
        if (single) {
          thR = thetaR(psi_in, soil[lyr], c);
        } else if (have_theta) {
          if constexpr (TAPED) thR = thetaR(scaled_shift(psi_in, psi_cm, psi_scale), soil[lyr], c);
          else thR = theta;  // the loop's last evaluation is theta_l(psi_final)
        }
        if (kind == K_DEEPEST) {
          s(F_THETA, i, thR);
          s(F_PSI, i, psi_in);
        } else {
          s(F_THETA, i, tmin(thR, soil[lyr].the));
        }
      }
      if (mine && kind >= K_INLAYER0 && c.st == 0) {
        R se = se_thetaR(g(F_THETA, i), soil[lyr], c);
        s(F_PSI, i, h_seR(se, soil[lyr], c));
      }
      if (mine) {
        if (i == 0 && c.st == 0) check_column_mass(fd, val(old_mass), val(infiltration), val(aet), c);
        old_theta_below = old_theta;
        old_psi_below = old_psi;
      }
    }
  }

  // next_to_next of get_extended_neighbors (Layer.py:733-758) for list l, list index j
  // (flat index o + j).  Returns -1 for None, -2 if the reference would raise AttributeError.
  __device__ int next_to_next(int l, int o, int j) {
    const int nf = cnt(l);
    const int i = o + j;
    if (j < nf - 2) return i + 2;
    const bool has_next = (j < nf - 1) || (l < L - 1);
    if (!has_next) return -1;
    const int nx = i + 1;
    if (lay(nx) != lay(i)) {
      if (l >= L - 1) return -2;  // self.next_layer is None
      const int o1 = o + nf;      // first front of list l+1
      if (cnt(l + 1) > 1) return o1 + 1;
      if (l + 1 < L - 1) return o1 + cnt(l + 1);
      return -1;
    }
    if (l < L - 1) return o + nf;
    return -1;
  }

  // ---- Layer.merge_wetting_fronts (Layer.py:838-892): at most one merge per layer list per call
  __device__ void merge_wetting_fronts(Ctx& c) {
    int o = 0;
    for (int l = 0; l < L; l++) {
      const int lf = len_layers(l);
      for (int j = 0; j < lf; j++) {
        const int i = o + j, nx = i + 1;
        const bool passing = (f(F_DEPTH, i) > f(F_DEPTH, nx)) && (lay(i) == lay(nx)) && !tb(nx);
        if (passing) {
          const int n2 = next_to_next(l, o, j);
          if (n2 < 0) {
            raise(c, LGAR_ST_NULL_NEIGHBOUR);  // Q10
            break;
          }
          const SoilT<R>& sl = soil[l];
          const R th_c = g(F_THETA, i), th_n = g(F_THETA, nx), th_2 = g(F_THETA, n2);
          R mass = g(F_DEPTH, i) * (th_c - th_n) + g(F_DEPTH, nx) * (th_n - th_2);
          s(F_DEPTH, i, mass / (th_c - th_2));
          R se = se_thetaR(th_c, sl, c);
          s(F_PSI, i, h_seR(se, sl, c));
          s(F_K, i, k_seR(se, sl, c));
          // delete_front (:888-892): pop the first front of THIS list that is value-equal to next
          const int nf = cnt(l);
          for (int q = 0; q < nf; q++) {
            if (is_equal(o + q, nx)) {
              erase_at(o + q, l);
              break;
            }
          }
          break;
        }
      }
      o += cnt(l);
    }
  }

  // ---- Layer.wetting_fronts_cross_layer_boundary (Layer.py:894-1008) + check_wetting_front
  __device__ void cross_layer_boundary(Ctx& c) {
    int o = 0;
    for (int l = 0; l < L; l++) {
      const int lf = len_layers(l);
      const SoilT<R>& sl = soil[l];
      for (int j = 0; j < lf; j++) {
        const int i = o + j, nx = i + 1;
        const bool deeper = f(F_DEPTH, i) > cum[l];
        const bool next_at_boundary = f(F_DEPTH, nx) == cum[l];
        if (deeper && next_at_boundary) {
          const R overshot = g(F_DEPTH, i) - g(F_DEPTH, nx);
          R se = se_thetaR(g(F_THETA, i), sl, c);
          const R psi_c = h_seR(se, sl, c);
          s(F_PSI, i, psi_c);
          s(F_K, i, k_seR(se, sl, c));
          if (l >= L - 1) {  // recalibrate dereferences self.next_layer (None): Q9
            raise(c, LGAR_ST_BOTTOM_REACHED);
            return;
          }
          const int n2 = next_to_next(l, o, j);
          R theta_new = thetaR(psi_c, soil[l + 1], c);
          R mbal = overshot * (g(F_THETA, i) - g(F_THETA, nx));
          if (n2 < 0) {
            raise(c, LGAR_ST_NULL_NEIGHBOUR);
            return;
          }
          R mbal_z = mbal / (theta_new - g(F_THETA, n2));
          R depth_new = cum[l] + mbal_z;
          s(F_DEPTH, i, R(cum[l]));
          s(F_THETA, nx, theta_new);
          s(F_PSI, nx, psi_c);
          s(F_DEPTH, nx, depth_new);
          s(F_DZDT, nx, g(F_DZDT, i));
          s(F_DZDT, i, R(0.0));
          set_flag(nx, l + 1, false);
          set_flag(i, lay(i), true);
        }
      }
      o += cnt(l);
    }
    // update_wetting_fronts / check_wetting_front (:939-963): fronts whose layer_num attribute
    // exceeds their list's layer move to the head of the next list
    o = 0;
    for (int l = 0; l < L; l++) {
      bool again = true;
      while (again) {
        again = false;
        const int nf = cnt(l);
        for (int j = 0; j < nf; j++) {
          if (lay(o + j) > l) {
            if (l >= L - 1) {
              raise(c, LGAR_ST_NULL_NEIGHBOUR);
              return;
            }
            // pop(j) from list l and insert at the head of list l+1: rotate [o+j, o+nf)
            const int from = o + j, to = o + nf - 1;
            if (from != to) {
              R t5[5];
#pragma unroll
              for (int k = 0; k < 5; k++) t5[k] = g(k, from);
              uint8_t tg = gb[from * NT];
              for (int q = from; q < to; q++) copy_front(q, q + 1);
#pragma unroll
              for (int k = 0; k < 5; k++) s(k, to, t5[k]);
              gb[to * NT] = tg;
            }
            add_cnt(l, -1);
            add_cnt(l + 1, 1);
            again = true;
            break;
          }
        }
      }
      o += cnt(l);
    }
  }

  // ---- Layer.wetting_front_cross_domain_boundary (Layer.py:1010-1053): a front without a
  //      next_to_next neighbour that lies below its layer leaves the domain: its water becomes the
  //      bottom flux, the front below inherits its theta (psi, K recomputed with THIS layer's
  //      parameters, sic) and it is popped.  Reachable for the last front of layer L-2 when the
  //      last layer holds a single front.  The loop bound is evaluated before the pops, like
  //      Python's range(): an index past the shortened list raises IndexError.
  __device__ R cross_domain_boundary(Ctx& c) {
    R fl[MAXL];
    int o = 0;
    for (int l = 0; l < L; l++) {
      fl[l] = R(0.0);
      const int lf = len_layers(l);
      const SoilT<R>& sl = soil[l];
      for (int j = 0; j < lf; j++) {
        if (j >= cnt(l)) {
          raise(c, LGAR_ST_INDEX_ERROR);
          return R(0.0);
        }
        const int n2 = next_to_next(l, o, j);
        if (n2 == -2) {
          raise(c, LGAR_ST_NULL_NEIGHBOUR);
          return R(0.0);
        }
        R tmp(0.0);
        const int i = o + j;
        if (n2 == -1 && f(F_DEPTH, i) > cum[l]) {
          const bool has_next = (j < cnt(l) - 1) || (l < L - 1);
          if (!has_next) {
            raise(c, LGAR_ST_NULL_NEIGHBOUR);
            return R(0.0);
          }
          const int nx = i + 1;
          tmp = (g(F_THETA, i) - g(F_THETA, nx)) * (g(F_DEPTH, i) - g(F_DEPTH, nx));
          s(F_THETA, nx, g(F_THETA, i));
          R se_k = se_thetaR(g(F_THETA, i), sl, c);
          s(F_PSI, nx, h_seR(se_k, sl, c));
          s(F_K, nx, k_seR(se_k, sl, c));
          erase_at(i, l);
        }
        fl[l] = fl[l] + tmp;
      }
      o += cnt(l);
    }
    return layer_sum(fl);
  }

  // ---- Layer.fix_dry_over_wet_fronts (Layer.py:1055-1143): one fix per layer list per call
  __device__ R fix_dry_over_wet(Ctx& c) {
    R mc[MAXL];
    int o = 0;
    for (int l = 0; l < L; l++) {
      mc[l] = R(0.0);
      const int nf = cnt(l);
      for (int j = 0; j < nf; j++) {
        const int i = o + j;
        const bool has_next = (j < nf - 1) || (l < L - 1);
        if (!has_next) continue;
        const int nx = i + 1;
        if (f(F_THETA, i) <= f(F_THETA, nx) && lay(i) == lay(nx)) {
          c.br[0]++;
          const R mass_before = mass_balance();
          const int popped_layer = lay(i);
          erase_at(i, l);  // the former next front now sits at flat index i
          if (popped_layer > 0) cleanup_wetting_fronts(i, c);
          const R mass_after = mass_balance();
          mc[l] = mc[l] + abs_(mass_after - mass_before);
          break;
        }
      }
      o += cnt(l);
    }
    return layer_sum(mc);
  }
  // cleanup_wetting_fronts (:1098-1115): the search is by VALUE from the top of the column
  __device__ void cleanup_wetting_fronts(int nx, Ctx& c) {
    int o = 0;
    for (int l = 0; l < L; l++) {
      const int nf = cnt(l);
      for (int j = 0; j < nf; j++) {
        const int i = o + j;
        if (is_equal(i, nx)) {
          const SoilT<R>& sl = soil[l];
          R se_k = se_thetaR(g(F_THETA, i), sl, c);
          s(F_PSI, i, h_seR(se_k, sl, c));
          // update_layer_fronts (:1117-1143, Q15): every front of every list above dry.layer_num
          const int dry_layer = lay(i);
          const R dry_theta = g(F_THETA, i), dry_psi = g(F_PSI, i);
          int o2 = 0;
          for (int l2 = 0; l2 < L && l2 < dry_layer; l2++) {
            const SoilT<R>& s2 = soil[l2];
            const int nf2 = cnt(l2);
            for (int q = 0; q < nf2; q++) {
              R se_l = se_thetaR(dry_theta, s2, c);
              s(F_PSI, o2 + q, h_seR(se_l, s2, c));
              s(F_THETA, o2 + q, thetaR(dry_psi, s2, c));
            }
            o2 += nf2;
          }
          return;
        }
      }
      o += nf;
    }
    raise(c, LGAR_ST_INDEX_ERROR);
  }

  // ---- Layer.update_psi (Layer.py:1157-1174): psi, K from theta for every front except the deepest
  //      of the domain.  Warp-convergent flat loop over the front index.
  __device__ void update_psi_warp(bool go, Ctx& c) {
    go = go && (c.st == 0);
    const int my_n = go ? n - 1 : 0;
    const int nmax = warp_max(my_n);
    int l = 0, o_next = go ? cnt(0) : 0;
    for (int i = 0; i < nmax; i++) {
      if (i < my_n) {
        while (i >= o_next) {
          l++;
          o_next += cnt(l);
        }
        const SoilT<R>& sl = soil[l];
        R se = se_thetaR(g(F_THETA, i), sl, c);
        const Pair<R> pk = psi_kR(se, sl, c);
        s(F_PSI, i, pk.x);
        s(F_K, i, pk.y);
      }
    }
  }

  // ---- Layer.calc_bottom_sum (Layer.py:1557-1582) from list l0 upward in index
  __device__ R calc_bottom_sum(int l0, R bottom_sum, const R& psi, int front_layer, Ctx& c) {
    for (int k = l0;; k++) {
      const SoilT<R>& sk = soil[k];
      R theta_prev = thetaR(psi, sk, c);
      R se_prev = se_thetaR(theta_prev, sk, c);
      R kk = k_seR(se_prev, sk, c);
      double plt = (k != 0) ? cum[k - 1] : 0.0;
      bottom_sum = bottom_sum + ((cum[k] - plt) / kk);
      if (k + 1 >= L) {
        raise(c, LGAR_ST_NULL_NEIGHBOUR);
        return bottom_sum;
      }
      if (k + 1 == front_layer) return bottom_sum;
    }
  }

  // ---- dpLGAR.move_wetting_front (models/dpLGAR.py:340-367); returns the bottom flux.
  //      Warp-convergent (every lane calls; `go` selects the lanes that actually move fronts).
  __device__ R move_wetting_front_warp(bool go, int fd, const R& infiltration, R& AET_sub, const R& old_mass, double dt,
                                       Ctx& c) {
    move_wetting_fronts_warp(go, fd, infiltration, AET_sub, old_mass, dt, c);
    R bottom_flux(0.0);
    if (go && c.st == 0) {
      merge_wetting_fronts(c);
      cross_layer_boundary(c);
      merge_wetting_fronts(c);
      bottom_flux = 0.0 + cross_domain_boundary(c);
      // a layer list emptied by the pop above: the very next neighbour lookup of the reference
      // (fix_dry_over_wet_fronts -> get_neighboring_fronts / mass_balance) raises IndexError
      for (int l = 0; l < L; l++)
        if (cnt(l) == 0) raise(c, LGAR_ST_INDEX_ERROR);
      R mass_change(0.0);
      if (c.st == 0) mass_change = fix_dry_over_wet(c);
      if (vabs(mass_change) > 1e-7) AET_sub = AET_sub - mass_change;
    }
    update_psi_warp(go, c);
    return bottom_flux;
  }
};

}  // namespace lgar

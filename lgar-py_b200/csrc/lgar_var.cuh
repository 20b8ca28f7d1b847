// =====================================================================================
// lgar_var.cuh -- tape-recording scalar for the hand-written reverse-mode kernel.
//
// The column physics (lgar_device.cuh / lgar_forward.cuh) is written once, templated on the
// scalar type R.  R = double is the forward kernel.  R = Var records, for ONE sub-step of one
// column, every differentiable operation as a tape entry {a, b, da, db}: "the adjoint of this
// value flows to value a with weight da and to value b with weight db".  The reverse sweep of
// lgar_backward.cuh then walks the entries backwards.  The local derivatives mirror the
// reference's torch.autograd graph (SURVEY.md Q12-Q14):
//   * torch.min / torch.minimum split the gradient 0.5 / 0.5 at ties; torch.clamp passes 1 at the
//     boundary; torch.abs has gradient sgn(x);
//   * the root finders shift psi / depth by CONSTANTS, so they are straight-through: only the final
//     theta(psi) evaluation is on the tape (with d psi_final / d psi_in = 0.1^k from the psi < 0 guard);
//   * branch predicates carry no gradient; calc_se_from_h returns a constant for |h| < 0.1.
// Expensive closures (theta(h), h(Se), K(Se), Geff) are single macro entries with analytic partials;
// their VALUES come from the same cores as the forward kernel, so the taped pass takes exactly the
// same branches as the forward pass.
// =====================================================================================
#pragma once
#include <cuda_runtime.h>

namespace lgar {

struct Var {
  double v;
  int id;  // < 0: constant (no gradient)
  __device__ __forceinline__ Var() : v(0.0), id(-1) {}
  __device__ __forceinline__ Var(double x) : v(x), id(-1) {}
  __device__ __forceinline__ Var(double x, int i) : v(x), id(i) {}
};

struct TapeEntry {
  int a, b;
  double da, db;
};
struct TapeCtl {          // per thread
  TapeEntry* base;        // entry k of this lane at base[k * 32]
  int n;                  // entries recorded (may exceed cap: overflow)
  int cap;
  int first_id;           // id of entry 0 (= number of leaf ids)
};
constexpr int TAPE_NT = 128;
__shared__ TapeCtl g_tapectl[TAPE_NT];

__device__ __forceinline__ double val(double x) { return x; }
__device__ __forceinline__ double val(const Var& x) { return x.v; }

__device__ __forceinline__ Var tape_record(double v, int a, double da, int b, double db) {
  if (a < 0 && b < 0) return Var(v);
  TapeCtl& t = g_tapectl[threadIdx.x];
  const int k = t.n;
  t.n = k + 1;
  if (k >= t.cap) return Var(v);  // overflow: detected by the kernel through n > cap
  TapeEntry e;
  e.a = a; e.b = b; e.da = da; e.db = db;
  t.base[(size_t)k * 32] = e;
  return Var(v, t.first_id + k);
}
// one entry "copy of x" even when x is a constant (a < 0): callers that find entries by their position on the tape
__device__ __forceinline__ void tape_append(const Var& x) {
  TapeCtl& t = g_tapectl[threadIdx.x];
  const int k = t.n;
  t.n = k + 1;
  if (k >= t.cap) return;  // overflow: detected by the kernel through n > cap
  TapeEntry e;
  e.a = x.id; e.b = -1; e.da = 1.0; e.db = 0.0;
  t.base[(size_t)k * 32] = e;
}
// value = sum_j d_j * x_j over up to 6 inputs (macro closures)
__device__ __forceinline__ Var tape_record_n(double v, int n, const int* ids, const double* d) {
  Var acc(0.0);
  bool any = false;
  for (int j = 0; j < n; j += 2) {
    const int a = ids[j], b = (j + 1 < n) ? ids[j + 1] : -1;
    const double da = d[j], db = (j + 1 < n) ? d[j + 1] : 0.0;
    if (a < 0 && b < 0) continue;
    Var pair = tape_record(0.0, a, da, b, db);
    if (!any) { acc = pair; any = true; }
    else acc = tape_record(0.0, acc.id, 1.0, pair.id, 1.0);
  }
  acc.v = v;
  return acc;
}

// ---- arithmetic ------------------------------------------------------------------------
__device__ __forceinline__ Var operator+(const Var& a, const Var& b) { return tape_record(a.v + b.v, a.id, 1.0, b.id, 1.0); }
__device__ __forceinline__ Var operator-(const Var& a, const Var& b) { return tape_record(a.v - b.v, a.id, 1.0, b.id, -1.0); }
__device__ __forceinline__ Var operator*(const Var& a, const Var& b) { return tape_record(a.v * b.v, a.id, b.v, b.id, a.v); }
__device__ __forceinline__ Var operator/(const Var& a, const Var& b) {
  return tape_record(a.v / b.v, a.id, 1.0 / b.v, b.id, -a.v / (b.v * b.v));
}
__device__ __forceinline__ Var operator-(const Var& a) { return tape_record(-a.v, a.id, -1.0, -1, 0.0); }
__device__ __forceinline__ Var operator+(const Var& a, double b) { return Var(a.v + b, a.id); }  // same adjoint: reuse id
__device__ __forceinline__ Var operator+(double a, const Var& b) { return Var(a + b.v, b.id); }
__device__ __forceinline__ Var operator-(const Var& a, double b) { return Var(a.v - b, a.id); }
__device__ __forceinline__ Var operator-(double a, const Var& b) { return tape_record(a - b.v, b.id, -1.0, -1, 0.0); }
__device__ __forceinline__ Var operator*(const Var& a, double b) { return tape_record(a.v * b, a.id, b, -1, 0.0); }
__device__ __forceinline__ Var operator*(double a, const Var& b) { return tape_record(a * b.v, b.id, a, -1, 0.0); }
__device__ __forceinline__ Var operator/(const Var& a, double b) { return tape_record(a.v / b, a.id, 1.0 / b, -1, 0.0); }
__device__ __forceinline__ Var operator/(double a, const Var& b) { return tape_record(a / b.v, b.id, -a / (b.v * b.v), -1, 0.0); }

// comparisons look at values only (branch predicates carry no gradient)
#define LGAR_VAR_CMP(op)                                                                              \
  __device__ __forceinline__ bool operator op(const Var& a, const Var& b) { return a.v op b.v; }      \
  __device__ __forceinline__ bool operator op(const Var& a, double b) { return a.v op b; }            \
  __device__ __forceinline__ bool operator op(double a, const Var& b) { return a op b.v; }
LGAR_VAR_CMP(<) LGAR_VAR_CMP(>) LGAR_VAR_CMP(<=) LGAR_VAR_CMP(>=) LGAR_VAR_CMP(==) LGAR_VAR_CMP(!=)
#undef LGAR_VAR_CMP

__device__ __forceinline__ bool isnan_(double x) { return isnan(x); }
__device__ __forceinline__ bool isnan_(const Var& x) { return isnan(x.v); }
__device__ __forceinline__ double vabs(double x) { return fabs(x); }       // |x| for predicates (no tape)
__device__ __forceinline__ double vabs(const Var& x) { return fabs(x.v); }

// differentiable abs / sqrt / min / clamp with torch's sub-gradient conventions
__device__ __forceinline__ double abs_(double x) { return fabs(x); }
__device__ __forceinline__ Var abs_(const Var& x) {
  return tape_record(fabs(x.v), x.id, (x.v > 0.0) ? 1.0 : ((x.v < 0.0) ? -1.0 : 0.0), -1, 0.0);
}
__device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
__device__ __forceinline__ Var sqrt_(const Var& x) {
  const double r = sqrt(x.v);
  return tape_record(r, x.id, 1.0 / (2.0 * r), -1, 0.0);
}
__device__ __forceinline__ Var tmin(const Var& a, const Var& b) {
  if (isnan(a.v) || isnan(b.v)) return Var(a.v + b.v);
  if (b.v < a.v) return b;
  if (a.v < b.v) return a;
  return tape_record(a.v, a.id, 0.5, b.id, 0.5);
}
__device__ __forceinline__ Var tmin(const Var& a, double b) { return tmin(a, Var(b)); }
__device__ __forceinline__ Var tmin(double a, const Var& b) { return tmin(Var(a), b); }
// torch.clamp(x, min=lo): gradient 1 where x >= lo (NaN propagates)
__device__ __forceinline__ double clamp_min_(double x, double lo) { return (x < lo) ? lo : x; }
__device__ __forceinline__ Var clamp_min_(const Var& x, double lo) { return (x.v < lo) ? Var(lo) : x; }
// torch.clamp(x, min=lo, max=hi)
__device__ __forceinline__ double clamp_(double x, double lo, double hi) {
  double r = (x < lo) ? lo : x;
  return (r > hi) ? hi : r;
}
__device__ __forceinline__ Var clamp_(const Var& x, double lo, double hi) {
  if (x.v < lo) return Var(lo);
  if (x.v > hi) return Var(hi);
  return x;
}
// x + c and c * x helpers that keep ids when possible are the operators above.
// a value shifted by a CONSTANT (root finders): same adjoint, new value
__device__ __forceinline__ double shifted(double /*x*/, double newv) { return newv; }
__device__ __forceinline__ Var shifted(const Var& x, double newv) { return Var(newv, x.id); }
// psi_final = scale * psi_in + const (scale = 0.1^k from the `psi < 0` guard of theta_mass_balance)
__device__ __forceinline__ double scaled_shift(double /*x*/, double newv, double /*scale*/) { return newv; }
__device__ __forceinline__ Var scaled_shift(const Var& x, double newv, double scale) {
  if (scale == 1.0) return Var(newv, x.id);
  return tape_record(newv, x.id, scale, -1, 0.0);
}
// torch.pow(x, 3.0) with a constant exponent (aet.py:45)
__device__ __forceinline__ Var pow3_(const Var& x, double value) { return tape_record(value, x.id, 3.0 * (x.v * x.v), -1, 0.0); }

}  // namespace lgar

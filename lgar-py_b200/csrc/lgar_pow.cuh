// =====================================================================================
// lgar_pow.cuh -- table-driven double-double pow(x, y) for the LGAR kernels.
//
// Why not the CUDA math library's pow: (a) accuracy -- libdevice's pow is a <= 2 ulp routine,
// the reference runs on glibc's ~0.52 ulp pow, and the LGAR root finders amplify ulp-level
// differences (measured: 2.9e-9 relative on per-step AET over a year, above the 1e-9 bar);
// (b) cost -- libdevice's pow occupies ~150 FP64-pipe issue slots and has a 926-cycle dependent
// latency on B200 (tools/fp64_microbench.cu); this routine needs ~55 FP64 operations, two small
// table look-ups (6 KB, L1-resident), and inlines so that independent evaluations overlap.
//
// Lineage: the structure is that of the pow in glibc >= 2.28 / ARM Optimized Routines (Szabolcs Nagy, `pow.c` +
// `pow_log_data.c` / `exp_data.c`: 128-entry `invc / logc / logctail` table indexed by the leading mantissa bits,
// log1p polynomial on the exact residual r, `tail`-corrected 2^(k/128) table with `sbits` exponent reconstruction) --
// i.e. the very routine the reference's torch.pow ends up in on the CPU, which is why its accuracy class is the
// target.  No code or table was copied: the interval layout, polynomial degrees and error handling are written for
// this kernel (fast path only, specials delegated) and all tables and coefficients are generated here with mpmath
// (tools/gen_pow_tables.py).
//
// Algorithm (tables from tools/gen_pow_tables.py, mpmath 200 bit):
//   log:  x = 2^k z; i = sub-interval of z (128 in mantissa-bit space, 1.0 at the centre of
//         interval 64); r = z*invc_i - 1 as an exact two-term sum (p = fl(z*invc), e = fma error);
//         log x = k ln2 + log c_i + log1p(r) evaluated as hi + lo with |err| ~ 2^-66 relative.
//   mul:  ehi + elo = y * (hi + lo)      (fma for the exact product error)
//   exp:  exp(ehi + elo) = 2^(k'/128) * (1 + tail + r + r^2/2 + ...), k' = rint(ehi*128/ln2)
// Fast path: x positive normal, result comfortably inside the normal range; everything else
// (zero, negative, inf, NaN, subnormal, overflow/underflow) goes to the library pow so all
// special-value semantics are the library's.
//
// The same source compiles as plain C++ for the CPU accuracy harness (tools/pow_accuracy.cpp):
// every operation is an IEEE fp64 add/mul/fma, so CPU and GPU results are bit-identical.
// =====================================================================================
#pragma once
#include <cstdint>
#include <cstring>
#include <cmath>
#include "lgar_pow_tables.h"

#ifdef __CUDACC__
#define LGAR_HD __host__ __device__ __forceinline__
#else
#define LGAR_HD inline
#endif

namespace lgar {

struct PowLogEntry { double invc, logc, logctail, pad; };
struct PowExpEntry { double t, tail; };

#ifdef __CUDACC__
__device__ const PowLogEntry g_pow_log_table[LGAR_POW_N] = {LGAR_POW_LOG_TABLE};
__device__ const PowExpEntry g_pow_exp_table[LGAR_POW_N] = {LGAR_POW_EXP_TABLE};
// Table placement (measured on B200, tools/ + DESIGN.md): the look-ups are data-dependent (a warp touches up to
// 32 different rows).  The 2 KB exp table is copied to shared memory by every kernel (pow_tables_to_shared(), once
// per CTA, before its first pow); the 4 KB log table stays in global memory / L1: a shared-memory copy shortens a
// lone warp's pow by ~3 % but costs 5 % THROUGHPUT at full occupancy (two 16-byte LDS per pow with random rows
// serialise on bank conflicts), and throughput is what the ensemble runs are bound by.
__shared__ double2 s_pow_exp_table[LGAR_POW_N];
#define LGAR_POW_LOG_ROW(i2) __ldg(reinterpret_cast<const double2*>(g_pow_log_table) + (i2))
#define LGAR_POW_EXP_ROW(j) s_pow_exp_table[j]
__device__ __forceinline__ void pow_tables_to_shared() {
  for (int i = threadIdx.x; i < LGAR_POW_N; i += blockDim.x)
    s_pow_exp_table[i] = reinterpret_cast<const double2*>(g_pow_exp_table)[i];
  __syncthreads();
}
#endif
static const PowLogEntry h_pow_log_table[LGAR_POW_N] = {LGAR_POW_LOG_TABLE};
static const PowExpEntry h_pow_exp_table[LGAR_POW_N] = {LGAR_POW_EXP_TABLE};

// Scalar constants.  On the device they live in __constant__ memory so that FP64 instructions take them as
// constant-bank operands instead of materialising each 64-bit immediate with two moves.
enum PowConst { PC_LN2HI, PC_LN2LO, PC_INVLN2N, PC_LN2N_HI, PC_LN2N_LO, PC_A3, PC_A4, PC_A5, PC_A6, PC_A7, PC_A8, PC_A9,
                PC_C2, PC_C3, PC_C4, PC_C5, PC_C6, PC_SHIFT, PC_COUNT };
#define LGAR_POW_CONSTS {LGAR_LN2HI, LGAR_LN2LO, LGAR_INVLN2N, -LGAR_LN2N_HI, -LGAR_LN2N_LO, LGAR_LOG_A3, LGAR_LOG_A4, \
                         LGAR_LOG_A5, LGAR_LOG_A6, LGAR_LOG_A7, LGAR_LOG_A8, LGAR_LOG_A9, LGAR_EXP_C2, LGAR_EXP_C3, \
                         LGAR_EXP_C4, LGAR_EXP_C5, LGAR_EXP_C6, 0x1.8p52}
#ifdef __CUDACC__
static __constant__ double c_pow_consts[PC_COUNT] = LGAR_POW_CONSTS;
#endif
static const double h_pow_consts[PC_COUNT] = LGAR_POW_CONSTS;
#ifdef __CUDA_ARCH__
#define PCK(i) c_pow_consts[i]
#else
#define PCK(i) h_pow_consts[i]
#endif

LGAR_HD uint64_t pow_bits(double x) {
#ifdef __CUDA_ARCH__
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t u; std::memcpy(&u, &x, 8); return u;
#endif
}
LGAR_HD double pow_from_bits(uint64_t u) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)u);
#else
  double d; std::memcpy(&d, &u, 8); return d;
#endif
}
LGAR_HD double pow_fma(double a, double b, double c) {
#ifdef __CUDA_ARCH__
  return __fma_rn(a, b, c);
#else
  return std::fma(a, b, c);
#endif
}

// Branch-free core, written for N independent evaluations at once: every statement is applied to all N
// arguments before the next one, so the N dependent chains are interleaved IN SOURCE ORDER.  (Calling a scalar
// core N times in a row does not do it: ptxas keeps the chains back to back -- checked in the SASS -- and a warp
// then waits out the full FP64 latency of one chain after the other.)  Per element the operations are exactly the
// same IEEE operations in the same order, so pow_core_v<N> is bit-identical to N scalar calls.
// Sets ok[k] = false when the arguments are outside the fast path (the caller then uses the library pow).
// lg (optional): log(x[k]) to double precision -- a by-product of the log stage, used by the derivative weights of
// the reverse kernel (d x^y / dy = x^y log x) instead of a separate log() call.
template <int N>
LGAR_HD void pow_core_v(const double (&x)[N], const double (&y)[N], double (&res)[N], bool (&ok)[N],
                        double* lg = nullptr) {
  bool x_ok[N];
  int ki_[N];
  double z[N], kd[N], invc[N], logc[N], logctail[N];
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int e = 0; e < N; e++) {
    const uint64_t ix = pow_bits(x[e]);
    // x must be a positive normal number
    x_ok[e] = (ix - 0x0010000000000000ULL) < (0x7ff0000000000000ULL - 0x0010000000000000ULL);
    // ---- log(x) = hi + lo
    const uint64_t tmp = ix - LGAR_POW_OFF;
    const int i = (int)((tmp >> 45) & (LGAR_POW_N - 1));
    const int k = (int)((int64_t)tmp >> 52);
    z[e] = pow_from_bits(ix - (tmp & 0xfff0000000000000ULL));
    kd[e] = (double)k;
#ifdef __CUDA_ARCH__
    const double2 le0 = LGAR_POW_LOG_ROW(2 * i);
    const double2 le1 = LGAR_POW_LOG_ROW(2 * i + 1);
    invc[e] = le0.x; logc[e] = le0.y; logctail[e] = le1.x;
#else
    invc[e] = h_pow_log_table[i].invc; logc[e] = h_pow_log_table[i].logc; logctail[e] = h_pow_log_table[i].logctail;
#endif
  }
#define LGAR_V(stmt)                        \
  _Pragma("unroll") for (int e = 0; e < N; e++) { stmt; }
  double p[N], rl[N], r[N], t1[N], t2[N], lo2[N], lo1[N], ar[N], ar2[N], lo3[N], hi[N], lo4[N], r2[N], q[N];
  LGAR_V(p[e] = z[e] * invc[e])
  LGAR_V(rl[e] = pow_fma(z[e], invc[e], -p[e]))  // exact: z*invc = p + rl
  LGAR_V(r[e] = p[e] - 1.0)                      // exact (Sterbenz)
  LGAR_V(t1[e] = pow_fma(kd[e], PCK(PC_LN2HI), logc[e]))  // exact: both are multiples of 2^-42 below 2^10
  // Fast2Sum t1 + r: exact because t1 == 0 (interval 64, k = 0) or |t1| >= |log c_63| = 0.0059 > |r|
  LGAR_V(t2[e] = t1[e] + r[e])
  LGAR_V(lo2[e] = (t1[e] - t2[e]) + r[e])
  LGAR_V(lo1[e] = pow_fma(kd[e], PCK(PC_LN2LO), logctail[e]))
  // -r^2/2 in two terms
  LGAR_V(ar[e] = -0.5 * r[e])
  LGAR_V(ar2[e] = r[e] * ar[e])
  LGAR_V(lo3[e] = pow_fma(ar[e], r[e], -ar2[e]))
  LGAR_V(hi[e] = t2[e] + ar2[e])
  LGAR_V(lo4[e] = (t2[e] - hi[e]) + ar2[e])
  LGAR_V(r2[e] = r[e] * r[e])
  // log1p(r) - r + r^2/2 = r^3 (A3 + A4 r + ... + A9 r^6): |r| <= 0.0046, truncation < 2^-70 relative
  LGAR_V(q[e] = pow_fma(r[e], PCK(PC_A9), PCK(PC_A8)))
  LGAR_V(q[e] = pow_fma(r[e], q[e], PCK(PC_A7)))
  LGAR_V(q[e] = pow_fma(r[e], q[e], PCK(PC_A6)))
  LGAR_V(q[e] = pow_fma(r[e], q[e], PCK(PC_A5)))
  LGAR_V(q[e] = pow_fma(r[e], q[e], PCK(PC_A4)))
  LGAR_V(q[e] = pow_fma(r[e], q[e], PCK(PC_A3)))
  double pl[N], lo5[N], lo[N], lhi[N], llo[N], ehi[N], elo[N], aeh[N];
  LGAR_V(pl[e] = (r2[e] * r[e]) * q[e])
  // contribution of the product rounding error rl: rl * d/dr log1p(r) = rl (1 - r + r^2)
  LGAR_V(lo5[e] = pow_fma(rl[e], r2[e] - r[e], rl[e]))
  LGAR_V(lo[e] = ((lo1[e] + lo2[e]) + (lo3[e] + lo4[e])) + (pl[e] + lo5[e]))
  LGAR_V(lhi[e] = hi[e] + lo[e])
  LGAR_V(llo[e] = (hi[e] - lhi[e]) + lo[e])
  if (lg) {
    LGAR_V(lg[e] = lhi[e])
  }
  // ---- ehi + elo = y * log(x)
  LGAR_V(ehi[e] = y[e] * lhi[e])
  LGAR_V(elo[e] = pow_fma(y[e], llo[e], pow_fma(y[e], lhi[e], -ehi[e])))
  // result must stay well inside the normal range (also rejects NaN / inf in y)
  LGAR_V(aeh[e] = ehi[e] < 0.0 ? -ehi[e] : ehi[e])
  LGAR_V(ok[e] = x_ok[e] && (aeh[e] < 700.0))
  // ---- exp(ehi + elo)
  double zz[N], kf[N], rr[N], tj[N], tailj[N], scale[N], rr2[N], e2[N], e4[N], tmp2[N];
  LGAR_V(zz[e] = ehi[e] * PCK(PC_INVLN2N))
  LGAR_V(kf[e] = (zz[e] + PCK(PC_SHIFT)) - PCK(PC_SHIFT))  // rint(zz), |zz| < 2^17
  LGAR_V(ki_[e] = ok[e] ? (int)kf[e] : 0)
  LGAR_V(rr[e] = pow_fma(kf[e], PCK(PC_LN2N_HI), ehi[e]))  // exact: kf*LN2N_HI has <= 52 bits
  LGAR_V(rr[e] = pow_fma(kf[e], PCK(PC_LN2N_LO), rr[e]))
  LGAR_V(rr[e] = rr[e] + elo[e])
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int e = 0; e < N; e++) {
    const int j = (int)(ki_[e] & (LGAR_POW_N - 1));
#ifdef __CUDA_ARCH__
    const double2 ee = LGAR_POW_EXP_ROW(j);
    tj[e] = ee.x; tailj[e] = ee.y;
#else
    tj[e] = h_pow_exp_table[j].t; tailj[e] = h_pow_exp_table[j].tail;
#endif
    const uint64_t sbits = pow_bits(tj[e]) + ((uint64_t)(int64_t)(ki_[e] >> 7) << 52);
    scale[e] = pow_from_bits(sbits);
  }
  LGAR_V(rr2[e] = rr[e] * rr[e])
  LGAR_V(e2[e] = pow_fma(rr[e], PCK(PC_C3), PCK(PC_C2)))
  LGAR_V(e4[e] = pow_fma(rr[e], PCK(PC_C5), PCK(PC_C4)))
  LGAR_V(e4[e] = pow_fma(rr2[e], PCK(PC_C6), e4[e]))
  LGAR_V(tmp2[e] = tailj[e] + (rr[e] + (rr2[e] * e2[e] + (rr2[e] * rr2[e]) * e4[e])))
  // |y log x| tiny: pow = 1 + y log x to well below half an ulp
  LGAR_V(res[e] = (aeh[e] < 0x1p-60) ? (1.0 + ehi[e]) : pow_fma(scale[e], tmp2[e], scale[e]))
#undef LGAR_V
}

// scalar form (the CPU accuracy harness and the single-evaluation closures)
LGAR_HD double pow_core(double x, double y, bool& ok) {
  const double xv[1] = {x}, yv[1] = {y};
  double rv[1];
  bool okv[1];
  pow_core_v<1>(xv, yv, rv, okv);
  ok = okv[0];
  return rv[0];
}

// returns true and sets *out on the fast path; false -> caller must use the library pow
LGAR_HD bool pow_fast(double x, double y, double* out) {
  bool ok;
  *out = pow_core(x, y, ok);
  return ok;
}

}  // namespace lgar

// thrl_device.cuh — device-side building blocks shared by the scan kernels.
//
// Arithmetic contract (DESIGN.md "Arithmetic"): every f64/f32 operation below is one IEEE round-to-nearest-even
// operation in the reference's order.  The translation unit is compiled with --fmad=false and the order-critical
// expressions also spell out the _rn intrinsics, so no FMA is ever formed.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/thrl.h"

namespace thrl {

constexpr unsigned kFull = 0xffffffffu;
__host__ __device__ constexpr int align16(int x) { return (x + 15) & ~15; }

// ---------------------------------------------------------------- Philox4x32-10 (DESIGN.md "Philox streams")
enum : uint32_t { kStreamAct = 0, kStreamEnv = 1, kStreamInitQ = 2, kStreamInitP = 3 };

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&o)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    c0 = h1 ^ c1 ^ k0;
    c1 = l1;
    c2 = h0 ^ c3 ^ k1;
    c3 = l0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}
// 53-bit uniform in [0,1): 32 bits of hi, top 21 bits of lo (exact: integer < 2^53 times 2^-53)
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
  const unsigned long long m = ((unsigned long long)hi << 21) | (unsigned long long)(lo >> 11);
  return __dmul_rn(__ull2double_rn(m), 1.0 / 9007199254740992.0);
}

// 32-bit uniform in [0,1) for the exploration test (exact: integer < 2^32 times 2^-32)
__device__ __forceinline__ double u32_unit(uint32_t x) { return __dmul_rn((double)x, 1.0 / 4294967296.0); }
// The same test in integers: u32_unit(x) < eps  <=>  x < u32_unit_threshold(eps), for every x and every eps (NaN and
// infinities included).  Proof: u32_unit(x) is x * 2^-32 exactly, and y = eps * 2^32 is exact in f64 (a power-of-two
// scaling; +-inf on overflow, which still orders correctly), so u32_unit(x) < eps <=> x < y.  For an integer x,
// x < y <=> x < ceil(y).  y <= 0 or NaN: no x qualifies (threshold 0); y > 2^32 - 1: every x does (threshold 2^32, hence
// 64 bits); otherwise ceil(y) lies in [1, 2^32 - 1].  Computed once per epsilon, it replaces a convert, a multiply and a
// compare in f64 per draw by one integer compare.
__device__ __forceinline__ unsigned long long u32_unit_threshold(double eps) {
  const double y = __dmul_rn(eps, 4294967296.0);
  if (!(y > 0.0)) return 0ull;
  if (y > 4294967295.0) return 1ull << 32;
  return (unsigned long long)ceil(y);
}

// ---------------------------------------------------------------- state encodes (th_rl/agents.py:47-49)
// float32 encode of the state handed to sample_action (trainer.py:53): rint_f32(f32(p) / f32(max_state) * f32(states))
__device__ __forceinline__ int act_row(double price, float max_state_f, float states_f) {
  const float x = __fmul_rn(__fdiv_rn(__double2float_rn(price), max_state_f), states_f);
  return __float2int_rn(x);
}
// float64 encode of the states stored in the replay buffer (agents.py:62,66)
__device__ __forceinline__ int upd_row(double price, double max_state, double states) {
  return __double2int_rn(__dmul_rn(__ddiv_rn(price, max_state), states));
}
// QTable.scale (agents.py:51-57): k / (actions - 1.0) * (hi - lo) + lo
__device__ __forceinline__ double scale_action(int k, int actions, double lo, double hi) {
  return __dadd_rn(__dmul_rn(__ddiv_rn((double)k, __dsub_rn((double)actions, 1.0)), __dsub_rn(hi, lo)), lo);
}

// ---------------------------------------------------------------- warp-wide row max / first argmax
// Lane l owns columns l, l+32, ... of every row, both for reading and for writing; a lane therefore only ever
// re-reads cells it wrote itself and the update loop needs no intra-warp memory fence.
__device__ __forceinline__ float warp_max(float v) {
  float m;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(v));
  return m;
}
__device__ __forceinline__ unsigned long long dkey(double v) {  // order-preserving map f64 -> u64
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double dunkey(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ double warp_max(double v) {
  const unsigned long long k = dkey(v);
  const unsigned hi = (unsigned)(k >> 32);
  const unsigned mh = __reduce_max_sync(kFull, hi);
  const unsigned lo = hi == mh ? (unsigned)k : 0u;
  const unsigned ml = __reduce_max_sync(kFull, lo);
  return dunkey(((unsigned long long)mh << 32) | ml);
}
template <typename T> struct NegInf;
template <> struct NegInf<float> { __device__ static float v() { return __int_as_float(0xff800000); } };
template <> struct NegInf<double> { __device__ static double v() { return __longlong_as_double(0xfff0000000000000ll); } };

// numpy.max(table[row]) (agents.py:71)
template <typename T>
__device__ __forceinline__ T row_max(const T* row, int actions, int lane) {
  T m = NegInf<T>::v();
  for (int k = lane; k < actions; k += 32) {
    const T v = row[k];
    m = v > m ? v : m;
  }
  return warp_max(m);
}
// numpy.argmax(table[row]) (agents.py:88): FIRST maximal index
template <typename T>
__device__ __forceinline__ int row_argmax(const T* row, int actions, int lane) {
  T m = NegInf<T>::v();
  int best = 0x7fffffff;
  for (int k = lane; k < actions; k += 32) {
    const T v = row[k];
    if (v > m || best == 0x7fffffff) { m = v; best = k; }
  }
  const T wm = warp_max(m);
  const unsigned cand = (best != 0x7fffffff && m == wm) ? (unsigned)best : 0xffffffffu;
  return (int)__reduce_min_sync(kFull, cand);
}

__device__ __forceinline__ double shfl_d(double v, int src) {
  const long long b = __double_as_longlong(v);
  const int lo = __shfl_sync(kFull, (int)b, src), hi = __shfl_sync(kFull, (int)(b >> 32), src);
  return __longlong_as_double(((long long)hi << 32) | (unsigned)lo);
}

__device__ __forceinline__ float shfl_t(float v, int src) { return __shfl_sync(kFull, v, src); }
__device__ __forceinline__ double shfl_t(double v, int src) { return shfl_d(v, src); }
__device__ __forceinline__ float shfl_xor_t(float v, int off) { return __shfl_xor_sync(kFull, v, off); }
__device__ __forceinline__ double shfl_xor_t(double v, int off) {
  const long long b = __double_as_longlong(v);
  const int lo = __shfl_xor_sync(kFull, (int)b, off), hi = __shfl_xor_sync(kFull, (int)(b >> 32), off);
  return __longlong_as_double(((long long)hi << 32) | (unsigned)lo);
}

// environments.py:27 `Q = sum(A)` as CPython >= 3.12 evaluates it (oracle/thrl_oracle.c py_sum_quantities): Neumaier-
// compensated over the leading exact-float items (the MLP agents' scaled actions), plain left-to-right addition from the
// first numpy.float64 item (a QTable agent) on.  lead <= 2 is the naive sum.  aq(i) returns agent i's scaled quantity.
__device__ __forceinline__ int lead_exact_floats(const ThrlGame& G) {
  int m = 0;
  while (m < G.n_agents && G.agent[m].kind != THRL_AGENT_QTABLE) ++m;
  return m;
}
template <typename F>
__device__ __forceinline__ double py_sum_quantities(int n, int lead, F aq) {
  if (lead <= 2) {
    double q = 0.0;
    for (int i = 0; i < n; ++i) q = __dadd_rn(q, aq(i));
    return q;
  }
  double f = __dadd_rn(0.0, aq(0)), c = 0.0;
  int i = 1;
  for (; i < lead; ++i) {
    const double x = aq(i), t = __dadd_rn(f, x);
    c = __dadd_rn(c, fabs(f) >= fabs(x) ? __dadd_rn(__dsub_rn(f, t), x) : __dadd_rn(__dsub_rn(x, t), f));
    f = t;
  }
  if (c != 0.0 && isfinite(c)) f = __dadd_rn(f, c);
  for (; i < n; ++i) f = __dadd_rn(f, aq(i));
  return f;
}

// fixed-point statistics (include/thrl.h THRL_STATS_*): exact integer sums, independent of run order and sharding
__device__ __forceinline__ long long fx_round(double x) { return __double2ll_rn(x); }

}  // namespace thrl

// Shared device helpers: Philox4x32-10, the uniform -> Poisson / categorical maps, error plumbing.
// The arithmetic here is restated op-for-op (fp32) in oracle/rng.py; keep the two in sync.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <math.h>
#include "../../include/ctdd.h"

namespace ctdd {

// ------------------------------------------------------------------------------------------------
// error / launch accounting (host side)
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
#define CTDD_CHECK_LAUNCH(name)                                                          \
  do {                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) {                                                            \
      ctdd::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));           \
      return 1;                                                                          \
    }                                                                                    \
    ctdd::count_launch();                                                                \
  } while (0)

// ------------------------------------------------------------------------------------------------
// RNG streams (Philox counter word c3)
enum : uint32_t {
  STREAM_JUMP = 0,      // per-row tau-leap draws, per chunk of 32 states: call 0 word 0 = total count, further words = picks
  STREAM_JUMP_COUNT = 1, // S <= JUMP_SHARED_MAX_S: uniform of a row's total jump count, one call per 4 consecutive rows
  STREAM_ROW = 2,       // one 32-bit uniform per row (Euler categorical draw)
  STREAM_INIT = 3,      // initial samples
  STREAM_NOISE_XT = 4,  // forward noising x_t
  STREAM_TILDE_DIM = 5, // x~: which dimension
  STREAM_TILDE_VAL = 6  // x~: new value
};

struct Philox4 { uint32_t w[4]; };

__host__ __device__ __forceinline__ void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__) && !defined(CTDD_PHILOX_WIDE)
  lo = a * b;
  hi = __umulhi(a, b);
#else
  uint64_t p = (uint64_t)a * b;
  lo = (uint32_t)p;
  hi = (uint32_t)(p >> 32);
#endif
}

// Standard Philox4x32-10 (Salmon et al. 2011): same constants/round function as Random123 / cuRAND.
__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                         uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(M0, c0, hi0, lo0);
    philox_mulhilo(M1, c2, hi1, lo1);
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  Philox4 o; o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
  return o;
}

// Round keys of Philox4x32-10 for `seed` (key of round r: pk[2r], pk[2r+1]); the launchers make them once on the host
// and pass them in the kernel arguments.
inline void philox_key_schedule(unsigned long long seed, uint32_t (&pk)[20]) {
  for (int r = 0; r < 10; ++r) {
    pk[2 * r] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
    pk[2 * r + 1] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
  }
}
#ifdef __CUDACC__
// Philox4x32-10 with the round keys read from the kernel arguments (constant bank operands): the same function as
// philox4x32_10(c0, c1, c2, c3, seed_lo, seed_hi), 4 instructions per round instead of 6.
__device__ __forceinline__ Philox4 philox_keyed(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t (&pk)[20]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ pk[2 * r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ pk[2 * r + 1];
    c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
  }
  Philox4 o; o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
  return o;
}

// Logits of the reverse step are fp32 or bf16 (ctdd_step_params::logits_dtype), and so are the truncated-logistic head's
// (mu, log_scale) and incoming gradient.  Widening bf16 to fp32 is exact (the 16 bits are the upper half of the fp32
// pattern), so a kernel that widens on load and then runs its fp32 code returns the results of the same call on the
// widened inputs bit for bit.
__device__ __forceinline__ float ld_logit(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_logit(const __nv_bfloat16* p) {
  return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}
// 4 consecutive bf16 (element 0 in the low half of w.x) -> fp32
__device__ __forceinline__ void widen_bf16x4(uint2 w, float& v0, float& v1, float& v2, float& v3) {
  v0 = __uint_as_float(w.x << 16); v1 = __uint_as_float(w.x & 0xFFFF0000u);
  v2 = __uint_as_float(w.y << 16); v3 = __uint_as_float(w.y & 0xFFFF0000u);
}
#endif

// Tau-leap draws of one GLOBAL row: the states are cut into chunks of JUMP_CHUNK consecutive states; chunk q draws its
// own total and picks from Philox calls (q << 16) + c of the row's stream, counter = (call, grow, offset_lo, stream | ...).
//   call 0 word 0     -> uniform of the chunk's TOTAL jump count K ~ Poisson(sum of the chunk's lam_s)
//   call 0 words 1..3 -> uniforms of picks 0..2;  call 1 + (j-3)/4 word (j-3)%4 -> pick j >= 3
// Each pick chooses its target state ~ Categorical(lam_s / sum) by inverse CDF: S independent Poisson counts through
// the superposition identity, chunks independent of one another (oracle/rng.py poisson_rows is the op-for-op
// restatement).  One warp of the tensor-path epilogue owns one chunk of a row, so no warp waits for another's total.
// State spaces of at most JUMP_SHARED_MAX_S states (one chunk; a row is 4*S + 8 bytes, a Philox call per row would be the
// whole cost of the step): the TOTAL's uniform of row g is word g & 3 of the call (0, g >> 2, offset, STREAM_JUMP_COUNT)
// shared by 4 consecutive rows (philox_row_word); the picks still come from the row's own calls, words 1..3 of call 0 first.
constexpr int JUMP_PICK_CAP = 4096;
constexpr int JUMP_CHUNK = 32;
constexpr int JUMP_SHARED_MAX_S = 8;
__host__ __device__ __forceinline__ Philox4 philox_rowjump(uint64_t grow, uint32_t call, uint64_t offset, uint64_t seed) {
  return philox4x32_10(call, (uint32_t)grow, (uint32_t)offset,
                       STREAM_JUMP | (((uint32_t)(offset >> 32) & 0xFFFFu) << 8) | (((uint32_t)(grow >> 32) & 0xFFu) << 24),
                       (uint32_t)seed, (uint32_t)(seed >> 32));
}
__host__ __device__ __forceinline__ uint32_t philox_word(const Philox4& p, int i) {   // register-only select
  return i == 0 ? p.w[0] : (i == 1 ? p.w[1] : (i == 2 ? p.w[2] : p.w[3]));
}

// Per-row 32-bit draw: one Philox call serves 4 consecutive global rows: counter = (sub, grow >> 2, ...).
__host__ __device__ __forceinline__ Philox4 philox_row_call(uint64_t grow, uint32_t sub, uint64_t offset,
                                                           uint32_t stream, uint64_t seed) {
  return philox4x32_10(sub, (uint32_t)(grow >> 2), (uint32_t)offset,
                       stream | (((uint32_t)(offset >> 32) & 0xFFFFu) << 8) | (((uint32_t)(grow >> 34) & 0xFFu) << 24),
                       (uint32_t)seed, (uint32_t)(seed >> 32));
}
__host__ __device__ __forceinline__ uint32_t philox_row_word(uint64_t grow, uint32_t sub, uint64_t offset,
                                                            uint32_t stream, uint64_t seed) {
  const Philox4 p = philox_row_call(grow, sub, offset, stream, seed);
  return p.w[grow & 3];
}

// 32 random bits -> v in (0, 1]:  v = (word + 0.5) * 2^-32 evaluated in fp32 (one rounding).
__host__ __device__ __forceinline__ float u32_to_unit(uint32_t w) {
#ifdef __CUDA_ARCH__
  return __fmaf_rn(__uint2float_rn(w), 2.3283064365386963e-10f, 1.1641532182693481e-10f);
#else
  return fmaf((float)w, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
#endif
}

// P(K >= 1) for K ~ Poisson(lam): 1 - exp(-lam), via a 3-term series below 2^-6 (no cancellation).
__host__ __device__ __forceinline__ float poisson_sf0(float lam) {
  if (lam < 0.015625f) {
    float t = fmaf(lam, -0.16666667f, 0.5f);
    float u = fmaf(-lam, t, 1.0f);
    return lam * u;
  }
  return 1.0f - expf(-lam);
}

// lam > 64: Cornish-Fisher normal approximation of the upper-tail quantile (kept out of line: it is rare and its
// register footprint would otherwise be charged to every caller)
__host__ __device__ __noinline__ inline int poisson_large_rate(float lam, float v) {
  if (lam > 1.0e9f) lam = 1.0e9f;
  // z = upper-tail normal quantile of v
#ifdef __CUDA_ARCH__
  float z = -normcdfinvf(v);
#else
  float z = 0.0f;  // host build never evaluates this branch (oracle has its own implementation)
#endif
  float k = lam + sqrtf(lam) * z + (z * z - 1.0f) * 0.16666667f;
  k = rintf(k);
  if (!(k > 1.0f)) k = 1.0f;
  if (k > 2.0e9f) k = 2.0e9f;
  return (int)k;
}

// Upper-tail inverse CDF: k = #{ j >= 0 : v < P(K > j) }, v in (0,1] small <=> many jumps.
// lam <= 64: exact pmf recurrence in fp32 (capped); lam > 64: Cornish-Fisher normal approximation.
// Callers may skip the call when v >= lam, because P(K>=1) <= lam.
__host__ __device__ __forceinline__ int poisson_from_unit(float lam, float v) {
  if (!(lam > 0.0f)) return 0;
  float sf = poisson_sf0(lam);
  if (v >= sf) return 0;
  if (lam <= 64.0f) {
    float p = expf(-lam);
    int kmax = (int)(lam + 10.0f * sqrtf(lam) + 12.0f);
    int k = 1;
    while (k < kmax) {
      p = p * lam / (float)k;   // pmf(k)
      sf -= p;                  // P(K > k)
      if (v >= sf) break;
      ++k;
    }
    return k;
  }
  return poisson_large_rate(lam, v);
}

// Inverse-CDF categorical draw from unnormalised weights: first index whose sequential fp32 cumulative
// sum exceeds v * total; falls back to the last positive weight. v in (0,1].
template <class F>
__device__ __forceinline__ int inv_cdf(int n, float v, F weight) {
  float tot = 0.f;
  for (int s = 0; s < n; ++s) tot += weight(s);
  const float target = fminf(v, 0.99999994f) * tot;
  float cum = 0.f;
  int last = 0;
  for (int s = 0; s < n; ++s) {
    const float w = weight(s);
    cum += w;
    if (w > 0.f) last = s;
    if (cum > target) return s;
  }
  return last;
}

// Tau-leap of one row in the oracle's op order (sequential fp32 sums), chunk by chunk (JUMP_CHUNK states share one
// superposition draw): lam(s) must return the row's rate * h with the entry s == x zeroed, rounded the same way on
// every call. Returns (sum_j (s_j - x), sum over the chunks of min(K_chunk, cap)).
template <class F>
__device__ __forceinline__ int2 tau_leap_row_seq(int S, int x, uint64_t grow, uint64_t offset, uint64_t seed, F lam) {
  int jump = 0, Ksum = 0;
  for (int c0 = 0, chunk = 0; c0 < S; c0 += JUMP_CHUNK, ++chunk) {
    const int c1 = (c0 + JUMP_CHUNK < S) ? c0 + JUMP_CHUNK : S;
    const uint32_t cbase = (uint32_t)chunk << 16;
    float tot = 0.f;
    for (int s = c0; s < c1; ++s) tot = __fadd_rn(tot, lam(s));
    const Philox4 p0 = philox_rowjump(grow, cbase, offset, seed);
    const uint32_t w0 = S <= JUMP_SHARED_MAX_S ? philox_row_word(grow, 0, offset, STREAM_JUMP_COUNT, seed) : p0.w[0];
    int K = poisson_from_unit(tot, u32_to_unit(w0));
    if (K <= 0) continue;
    if (K > JUMP_PICK_CAP) K = JUMP_PICK_CAP;
    Ksum += K;
    Philox4 pc = p0;
    for (int j = 0; j < K; ++j) {
      uint32_t w;
      if (j < 3) {
        w = philox_word(p0, 1 + j);
      } else {
        const int i = j - 3;
        if ((i & 3) == 0) pc = philox_rowjump(grow, cbase + 1u + (uint32_t)(i >> 2), offset, seed);
        w = philox_word(pc, i & 3);
      }
      const float target = __fmul_rn(fminf(u32_to_unit(w), 0.99999994f), tot);
      float cum = 0.f;
      int last = c0, pick = -1;
      for (int s = c0; s < c1; ++s) {
        const float v = lam(s);
        cum = __fadd_rn(cum, v);
        if (v > 0.f) last = s;
        if (cum > target) { pick = s; break; }
      }
      if (pick < 0) pick = last;
      jump += pick - x;
    }
  }
  return make_int2(jump, Ksum);
}

// per-thread statistics counters (CTDD_STAT_* order) and the common end of every jump update
struct RowStats { int changed_base, nonzero, changed_eval, jumped, multi; };

__device__ __forceinline__ int finalize_jump(int xb, int xe, int jump, int cnt, int reject_multi, int S,
                                             RowStats& st) {
  st.jumped += (cnt > 0);
  st.multi += (cnt > 1);
  if (reject_multi && cnt > 1) jump = 0;
  st.nonzero += (jump != 0);
  int xn = xb + jump;
  xn = xn < 0 ? 0 : (xn > S - 1 ? S - 1 : xn);
  st.changed_base += (xn != xb);
  st.changed_eval += (xn != xe);
  return xn;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace ctdd

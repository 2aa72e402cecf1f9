// CUDA-core reverse-step kernels.
//   step_small_kernel<S>  S <= 8 (C1: S=2, C2: S=3): one thread owns 8 consecutive rows, everything in
//                         registers, float4 logits loads — HBM-bound by construction.
//   step_block_kernel     any S: one CTA owns 8 consecutive rows, threads span the state axis. This is the
//                         general path and the on-GPU cross-check of the tcgen05 path at S=256.
// Both implement every CTDD_MODE_* / CTDD_BRANCH_* and draw exactly the same per-row Philox uniforms as the tensor
// path (superposition map, ctdd_common.cuh), so the three are interchangeable up to fp32 rounding of the rates.
// Reference arithmetic: lib/sampling/sampling.py:31-78 (rates), :127-160 (tau-leap), :278-293 (Euler),
// :423-453 / :459-503 (midpoint), :170-221 (corrector); lib/models/model_utils.py:30-60.
#define CTDD_PHILOX_WIDE 1   // this file is issue-bound on the Philox rounds: one 32x32->64 multiply per round half
#include "ctdd_common.cuh"

namespace ctdd {

// softmax pieces of the small-S kernel: ex2.approx / rcp.approx (<= 2 ulp; the parity bar on the rates is 1e-4 relative)
__device__ __forceinline__ float fast_exp(float v) {       // v <= 0; flushes results below 2^-126 to zero
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v * 1.4426950408889634f));
  return r;
}
__device__ __forceinline__ float fast_rcp(float v) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

struct StepArgs {
  int mode, branch, D, S, reject_multi;
  long long rows;        // N*D
  long long row_offset;  // multiple of 8
  const void* logits;    // fp32 or bf16 (the kernel's logits-type template argument)
  long long ld, batch_stride;
  const int* x_eval;
  const int* x_base;
  const float* Q;
  const float* QT;
  const float* Rb;
  const float* RbT;
  float beta, h, eps;
  unsigned long long seed, offset;
  int* x_out;
  float* rr_out;
  float* ratio_out;
  unsigned long long* stats;
  uint32_t pk[20];       // Philox key schedule of `seed` (key of round r: pk[2r], pk[2r+1]), made once on the host
};

// Tau-leap of one row with S <= 8 states (one chunk of the superposition map): the draws, thresholds and sums of
// tau_leap_row_seq (ctdd_common.cuh) with the row's Philox counter words prepared by the caller.  Out of line: one
// copy serves the 8 unrolled rows of a thread (the kernel was stalling on instruction fetch).
//   c1 = low word of the global row, c2 = low word of the offset, c3 = stream word (philox_rowjump)
//   tot = sequential fp32 sum of lam from 0, v0 = the uniform of the total count (shared call, JUMP_SHARED_MAX_S);
//   the caller has already handled the common case v0 >= tot, i.e. no jump
// words of the per-row uniforms of 8 consecutive global rows starting at g0 (a multiple of 8): 2 calls
__device__ __forceinline__ void row_words8(uint64_t g0, uint32_t stream, uint64_t offset, const uint32_t (&pk)[20], uint32_t (&rw)[8]) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const uint64_t gq = g0 + 4 * q;
    const Philox4 pq = philox_keyed(0u, (uint32_t)(gq >> 2), (uint32_t)offset,
                                    stream | (((uint32_t)(offset >> 32) & 0xFFFFu) << 8) | (((uint32_t)(gq >> 34) & 0xFFu) << 24), pk);
#pragma unroll
    for (int i = 0; i < 4; ++i) rw[4 * q + i] = pq.w[i];
  }
}

template <int S> struct LamVec { float v[S]; };
template <int S>
__device__ __noinline__ int2 tau_leap_small(LamVec<S> lam, float tot, float v0, int x, uint32_t c1, uint32_t c2,
                                            uint32_t c3, uint32_t k0, uint32_t k1) {
  const Philox4 p0 = philox4x32_10(0u, c1, c2, c3, k0, k1);      // words 1..3: picks 0..2
  int K = poisson_from_unit(tot, v0);
  if (K <= 0) return make_int2(0, 0);
  if (K > JUMP_PICK_CAP) K = JUMP_PICK_CAP;
  int jump = 0;
  Philox4 pc = p0;
  for (int j = 0; j < K; ++j) {
    uint32_t w;
    if (j < 3) {
      w = philox_word(p0, 1 + j);
    } else {
      const int i = j - 3;
      if ((i & 3) == 0) pc = philox4x32_10(1u + (uint32_t)(i >> 2), c1, c2, c3, k0, k1);
      w = philox_word(pc, i & 3);
    }
    const float target = __fmul_rn(fminf(u32_to_unit(w), 0.99999994f), tot);
    float cum = 0.f;
    int last = 0, pick = -1;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      cum = __fadd_rn(cum, lam.v[s]);
      if (lam.v[s] > 0.f) last = s;
      if (pick < 0 && cum > target) pick = s;
    }
    if (pick < 0) pick = last;
    jump += pick - x;
  }
  return make_int2(jump, K);
}

template <typename LT>
__device__ __forceinline__ const LT* logits_row(const StepArgs& a, long long r) {
  const long long n = r / a.D, d = r - n * a.D;
  return static_cast<const LT*>(a.logits) + n * a.batch_stride + d * a.ld;
}

__device__ __forceinline__ void flush_stats(const RowStats& st, unsigned long long* stats) {
  if (!stats) return;
  int v[5] = {st.changed_base, st.nonzero, st.changed_eval, st.jumped, st.multi};
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    int s = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(stats + i, (unsigned long long)s);
  }
}

// The same counters summed per CTA in shared memory first: one global atomic per counter and CTA instead of one per warp
// (the small-S kernels run tens of thousands of warps per launch onto the same 5 addresses).  Every thread of the CTA
// must call it.
__device__ __forceinline__ void flush_stats_cta(const RowStats& st, unsigned long long* stats) {
  if (!stats) return;            // uniform: a kernel argument
  __shared__ int s_cnt[5];
  if (threadIdx.x < 5) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  int v[5] = {st.changed_base, st.nonzero, st.changed_eval, st.jumped, st.multi};
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    int s = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(&s_cnt[i], s);
  }
  __syncthreads();
  if (threadIdx.x < 5 && s_cnt[threadIdx.x]) atomicAdd(stats + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------
// small S: thread per 8 rows
// MODE / BRANCH >= 0: the launch's mode and branch as compile-time constants (the two BASELINE configurations: every other
// mode's code drops out of the instruction stream); -1: read from the arguments at run time.
// The S = 2 lean instantiation is compiled for 8 CTAs of 128 threads per SM (64 registers) and runs as a grid-stride
// kernel on a capped grid (a CTA pays its table prologue once for several groups of rows): 3.0 -> 3.2 TB/s at 33 M rows.
// The S = 3 one measured 7 % slower that way (4.4 vs 4.8 TB/s) and keeps one group per thread.
constexpr int SMALL_MINB = 8;
constexpr unsigned SMALL_GRIDCAP = 64u;   // CTAs per SM of the capped grid
// LEAN: the launch has dense logits and no rr_out / ratio_out (the samplers' call): the strided-row loads and the
// (predicated, but issued) rate stores drop out as well.
// LT: element type of the logits, float or __nv_bfloat16 (widened on load; everything after the load is the fp32 code).
template <int S, int MODE = -1, int BRANCH = -1, bool LEAN = false, typename LT = float>
__global__ void __launch_bounds__(128, (LEAN && S == 2 && MODE == CTDD_MODE_TAU_LEAP) ? SMALL_MINB : 0) step_small_kernel(StepArgs a_in) {
  StepArgs a = a_in;
  if (MODE >= 0) a.mode = MODE;
  if (BRANCH >= 0) a.branch = BRANCH;
  if (LEAN) { a.rr_out = nullptr; a.ratio_out = nullptr; a.ld = S; a.batch_stride = (long long)a.D * S; }
  // TABLE (lean tauLDR launches without corrector): everything of h * rate[s] that does not depend on the logits is
  // folded, once per CTA, into sT[x][k][s] = h * beta * Rb[s][x] * q[k][s] / (q[k][x] + eps), zero at s == x, so that
  // h * rate[s] = (sum_k e_k sT[x][k][s]) / sum_k e_k: S*S FMAs and S multiplies per row
  constexpr bool TABLE = LEAN && S == 2 && BRANCH == CTDD_BRANCH_TAULDR && (MODE == CTDD_MODE_TAU_LEAP || MODE == CTDD_MODE_EULER);
  constexpr bool ONE = TABLE && S == 2 && MODE == CTDD_MODE_TAU_LEAP;   // one jump target per row: only its rate is made
  constexpr int TQ = (S * S + 3) / 4;                    // float4 per x
  __shared__ float sQ[S * S], sRb[S * S], sQi[S * S];   // sRb = beta * R_b (every use is that product); sQi = 1 / (q_t|0 + eps)
  __shared__ float4 sT4[TABLE ? S * TQ : 1];
  for (int i = threadIdx.x; i < S * S; i += blockDim.x) {
    const float q = a.Q[i];
    sQ[i] = q; sRb[i] = a.beta * a.Rb[i]; sQi[i] = 1.0f / (q + a.eps);
  }
  __syncthreads();
  if (TABLE) {
    float* sT = reinterpret_cast<float*>(sT4);
    for (int i = threadIdx.x; i < S * TQ * 4; i += blockDim.x) {
      const int x = i / (TQ * 4), ks = i - x * (TQ * 4), k = ks / S, t = ks - k * S;
      sT[i] = (ks < S * S && t != x) ? (sRb[t * S + x] * (sQ[k * S + t] * sQi[k * S + x])) * a.h : 0.f;
    }
    __syncthreads();
    if (ONE) {       // S = 2: the only target of x is 1 - x; sT[x] = {T[x][0][1-x], T[x][1][1-x], -, -}
      float v = 0.f;
      const int x = threadIdx.x >> 2, k = threadIdx.x & 3;
      if (threadIdx.x < 8 && k < 2) v = sT[x * 4 + k * 2 + (1 - x)];
      __syncthreads();
      if (threadIdx.x < 8) sT[threadIdx.x] = v;
      __syncthreads();
    }
  }
  const float hh = TABLE ? 1.0f : a.h;      // TABLE: rate[][] already holds h * rate
  RowStats st = {0, 0, 0, 0, 0};
  // STRIDE: grid-stride over groups of 8 rows on a capped grid; otherwise one group per thread
  constexpr bool STRIDE = LEAN && S == 2 && MODE == CTDD_MODE_TAU_LEAP;
  long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  do {
    const long long r0 = g * 8;
    if (r0 >= a.rows) break;
    g += (long long)gridDim.x * blockDim.x;
    const int nr = (a.rows - r0) < 8 ? (int)(a.rows - r0) : 8;
    float lg[8][S];
    // (bf16: the 16-byte loads also need a 16-byte aligned tensor; r0 * S * 2 is a multiple of 16)
    const bool contiguous = (a.ld == S) && (a.batch_stride == (long long)a.D * S) && nr == 8 &&
                            (sizeof(LT) == 4 || (reinterpret_cast<uintptr_t>(a.logits) & 15) == 0);
    if (contiguous) {
      if constexpr (sizeof(LT) == 2) {     // 8 rows of S bf16: S 16-byte loads
        const uint4* p = reinterpret_cast<const uint4*>(static_cast<const LT*>(a.logits) + r0 * S);
        uint4 buf[S];
#pragma unroll
        for (int i = 0; i < S; ++i) buf[i] = __ldg(p + i);
        float f[8 * S];
#pragma unroll
        for (int i = 0; i < S; ++i) {
          widen_bf16x4(make_uint2(buf[i].x, buf[i].y), f[8 * i], f[8 * i + 1], f[8 * i + 2], f[8 * i + 3]);
          widen_bf16x4(make_uint2(buf[i].z, buf[i].w), f[8 * i + 4], f[8 * i + 5], f[8 * i + 6], f[8 * i + 7]);
        }
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
          for (int s = 0; s < S; ++s) lg[r][s] = f[r * S + s];
      } else {
        const float4* p = reinterpret_cast<const float4*>(static_cast<const LT*>(a.logits) + r0 * S);
        float4 buf[2 * S];
#pragma unroll
        for (int i = 0; i < 2 * S; ++i) buf[i] = __ldg(p + i);
        const float* f = reinterpret_cast<const float*>(buf);
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
          for (int s = 0; s < S; ++s) lg[r][s] = f[r * S + s];
      }
    } else {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const LT* p = LEAN ? static_cast<const LT*>(a.logits) + (r0 + (r < nr ? r : 0)) * S : logits_row<LT>(a, r0 + (r < nr ? r : 0));
#pragma unroll
        for (int s = 0; s < S; ++s) lg[r][s] = ld_logit(p + s);
      }
    }
    int xe[8], xb[8];
    const bool vec_x = nr == 8 && ((reinterpret_cast<uintptr_t>(a.x_eval) | reinterpret_cast<uintptr_t>(a.x_base) |
                                    reinterpret_cast<uintptr_t>(a.x_out)) & 15) == 0;   // r0 is a multiple of 8
    if (vec_x) {
      const int4 e0 = __ldg(reinterpret_cast<const int4*>(a.x_eval + r0)), e1 = __ldg(reinterpret_cast<const int4*>(a.x_eval + r0) + 1);
      xe[0] = e0.x; xe[1] = e0.y; xe[2] = e0.z; xe[3] = e0.w; xe[4] = e1.x; xe[5] = e1.y; xe[6] = e1.z; xe[7] = e1.w;
      if (a.x_base) {
        const int4 b0 = __ldg(reinterpret_cast<const int4*>(a.x_base + r0)), b1 = __ldg(reinterpret_cast<const int4*>(a.x_base + r0) + 1);
        xb[0] = b0.x; xb[1] = b0.y; xb[2] = b0.z; xb[3] = b0.w; xb[4] = b1.x; xb[5] = b1.y; xb[6] = b1.z; xb[7] = b1.w;
      } else {
#pragma unroll
        for (int r = 0; r < 8; ++r) xb[r] = xe[r];
      }
    } else {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const long long rr_ = r0 + (r < nr ? r : 0);
        xe[r] = a.x_eval[rr_];
        xb[r] = a.x_base ? a.x_base[rr_] : xe[r];
      }
    }
    // per-row 32-bit uniforms (Euler / exact posterior: the row's draw; tau-leaping with S <= 8: the uniform of the
    // row's total jump count): one Philox call serves 4 consecutive global rows, and the 8 rows of a thread start at a
    // multiple of 8 (row_offset is one too), so 2 calls serve the thread
    uint32_t rw[8];
    static_assert(S <= JUMP_SHARED_MAX_S, "the small-S kernel takes the jump count's uniform from the shared call");
    if (a.mode == CTDD_MODE_EXACT || a.mode == CTDD_MODE_EULER || a.mode == CTDD_MODE_EULER_CORR)
      row_words8((uint64_t)(a.row_offset + r0), STREAM_ROW, a.offset, a.pk, rw);
    int xn_out[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) xn_out[r] = 0;
    // rates: rate[r][s] holds rr with the s==x entry zeroed (the quantity every mode consumes)
    float rate[8][S];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int x = xe[r];
      float m = lg[r][0];
#pragma unroll
      for (int s = 1; s < S; ++s) m = fmaxf(m, lg[r][s]);
      float e[S], sum = 0.f;
      if (S == 2) {      // the larger logit's term is exp(0) = 1 exactly
        const float d = lg[r][1] - lg[r][0];
        const float es = fast_exp(-fabsf(d));
        e[0] = d > 0.f ? es : 1.0f;
        e[S - 1] = d > 0.f ? 1.0f : es;
        sum = 1.0f + es;
      } else {
#pragma unroll
        for (int s = 0; s < S; ++s) { e[s] = fast_exp(lg[r][s] - m); sum += e[s]; }
      }
      const float inv_sum = fast_rcp(sum);     // sum in [1, S]
      if (a.mode == CTDD_MODE_EXACT) {
        // sampling.py:1008-1052: weight[s'] = (sum_k p_k q_{t-h|0}[k,s']) * q_{t|t-h}[s', x]  (second factor: a.RbT[x][s'])
        float wgt[S];
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float acc = 0.f;
#pragma unroll
          for (int k = 0; k < S; ++k) acc = fmaf(e[k] * inv_sum, sQ[k * S + s], acc);
          wgt[s] = acc * __ldg(a.RbT + (size_t)x * S + s);
        }
        const float v = u32_to_unit(rw[r]);
        const int xn = inv_cdf(S, v, [&](int s) {
          float w = 0.f;
#pragma unroll
          for (int q = 0; q < S; ++q) w = (q == s) ? wgt[q] : w;
          return w;
        });
        xn_out[r] = xn;
        if (r < nr) {
          st.changed_base += (xn != xb[r]);
          st.changed_eval += (xn != x);
        }
#pragma unroll
        for (int s = 0; s < S; ++s) rate[r][s] = 0.f;
        continue;
      }
      if (ONE) {
        const float4 t4 = sT4[x];
        rate[r][0] = fmaf(e[S - 1], t4.y, fmaf(e[0], t4.x, 0.f)) * inv_sum;      // h * rate of the state 1 - x
        rate[r][S - 1] = 0.f;
        continue;
      }
      if (TABLE) {
        float T[TQ * 4];
#pragma unroll
        for (int i = 0; i < TQ; ++i) {
          const float4 t4 = sT4[x * TQ + i];
          T[4 * i] = t4.x; T[4 * i + 1] = t4.y; T[4 * i + 2] = t4.z; T[4 * i + 3] = t4.w;
        }
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float acc = 0.f;
#pragma unroll
          for (int k = 0; k < S; ++k) acc = fmaf(e[k], T[k * S + s], acc);
          rate[r][s] = acc * inv_sum;
        }
        continue;
      }
      float ratio[S], rfull[S];
      if (a.branch == CTDD_BRANCH_TAULDR) {
        float w[S];
#pragma unroll
        for (int k = 0; k < S; ++k) w[k] = (e[k] * inv_sum) * sQi[k * S + x];
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float acc = 0.f;
#pragma unroll
          for (int k = 0; k < S; ++k) acc = fmaf(w[k], sQ[k * S + s], acc);
          ratio[s] = acc;
          rfull[s] = sRb[s * S + x] * acc;
        }
      } else {
        float ll[S];
        const float lse = m + logf(sum);
#pragma unroll
        for (int s = 0; s < S; ++s) {
          if (a.branch == CTDD_BRANCH_SDDM_DIRECT) {
            ll[s] = lg[r][s] - lse;
          } else if (a.branch == CTDD_BRANCH_SDDM_REVERSE_PROB) {
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < S; ++k) acc = fmaf(e[k] * inv_sum, sQ[k * S + s], acc);
            ll[s] = logf(acc + 1e-35f);
          } else {
            float t[S], tm = -INFINITY;
#pragma unroll
            for (int k = 0; k < S; ++k) {
              const float q = sQ[k * S + s];
              t[k] = (lg[r][k] - lse) + (q <= 1e-35f ? -1e9f : logf(q));
              tm = fmaxf(tm, t[k]);
            }
            float ts = 0.f;
#pragma unroll
            for (int k = 0; k < S; ++k) ts += expf(t[k] - tm);
            ll[s] = tm + logf(ts);
          }
        }
        float llx = 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) llx = (s == x) ? ll[s] : llx;
#pragma unroll
        for (int s = 0; s < S; ++s) {
          ratio[s] = expf(ll[s] - llx);
          rfull[s] = ratio[s] * sRb[x * S + s];
        }
      }
      if (r < nr) {
        if (a.rr_out) {
#pragma unroll
          for (int s = 0; s < S; ++s) a.rr_out[(r0 + r) * S + s] = rfull[s];
        }
        if (a.ratio_out) {
#pragma unroll
          for (int s = 0; s < S; ++s) a.ratio_out[(r0 + r) * S + s] = ratio[s];
        }
      }
      const bool corr = (a.mode == CTDD_MODE_TAU_LEAP_CORR || a.mode == CTDD_MODE_EULER_CORR);
#pragma unroll
      for (int s = 0; s < S; ++s) {
        float v = rfull[s];
        if (corr) v = v + sRb[x * S + s];
        rate[r][s] = (s == x) ? 0.f : v;
      }
    }
    if (a.mode == CTDD_MODE_TAU_LEAP || a.mode == CTDD_MODE_TAU_LEAP_CORR || a.mode == CTDD_MODE_MIDPOINT_JUMP) {
      // the thread's 8 global rows share everything of the Philox counter but the low 3 bits of the row
      const uint64_t g0 = (uint64_t)(a.row_offset + r0);
      const uint32_t c3 = STREAM_JUMP | (((uint32_t)(a.offset >> 32) & 0xFFFFu) << 8) | (((uint32_t)(g0 >> 32) & 0xFFu) << 24);
      row_words8(g0, STREAM_JUMP_COUNT, a.offset, a.pk, rw);       // uniforms of the 8 rows' total jump counts
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        if (r >= nr) continue;
        LamVec<S> lam;
        float tot = 0.f;
        if (ONE) {       // 0 + lam_0 + lam_1 with one of them zero
          tot = rate[r][0];
          lam.v[0] = xe[r] == 0 ? 0.f : tot;
          lam.v[S - 1] = xe[r] == 0 ? tot : 0.f;
        } else {
#pragma unroll
          for (int s = 0; s < S; ++s) lam.v[s] = TABLE ? rate[r][s] : __fmul_rn(rate[r][s], a.h);
#pragma unroll
          for (int s = 0; s < S; ++s) tot = __fadd_rn(tot, lam.v[s]);
        }
        const float v0 = u32_to_unit(rw[r]);
        if (v0 >= tot) {       // P(K >= 1) <= tot: no jump (the common case) - finalize_jump(xb, xe, 0, 0, ...)
          const int xn = xb[r] < 0 ? 0 : (xb[r] > S - 1 ? S - 1 : xb[r]);
          st.changed_base += (xn != xb[r]);
          st.changed_eval += (xn != xe[r]);
          xn_out[r] = xn;
        } else {
          const int2 jc = tau_leap_small<S>(lam, tot, v0, xe[r], (uint32_t)g0 | (uint32_t)r, (uint32_t)a.offset, c3,
                                            (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
          xn_out[r] = finalize_jump(xb[r], xe[r], jc.x, jc.y, a.reject_multi, S, st);
        }
      }
    } else if (a.mode == CTDD_MODE_MIDPOINT_DRIFT) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float acc = 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) acc += rate[r][s] * (float)(s - xe[r]);
        const int ch = (int)rintf(0.5f * a.h * acc);
        int xn = xe[r] + ch;
        xn = xn < 0 ? 0 : (xn > S - 1 ? S - 1 : xn);
        xn_out[r] = xn;
        if (r < nr) {
          st.changed_base += (xn != xe[r]);
          st.changed_eval += (xn != xe[r]);
          st.nonzero += (ch != 0);
        }
      }
    } else if (a.mode == CTDD_MODE_EULER || a.mode == CTDD_MODE_EULER_CORR) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float tot = 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) tot += rate[r][s];
        const float diag = fmaxf(0.f, 1.f - hh * tot);
        const int x = xe[r];
        const float v = u32_to_unit(rw[r]);
        float P[S];
#pragma unroll
        for (int s = 0; s < S; ++s) P[s] = (s == x) ? diag : rate[r][s] * hh;
        const int xn = inv_cdf(S, v, [&](int s) {
          float w = 0.f;
#pragma unroll
          for (int q = 0; q < S; ++q) w = (q == s) ? P[q] : w;
          return w;
        });
        xn_out[r] = xn;
        if (r < nr) {
          st.changed_base += (xn != xb[r]);
          st.changed_eval += (xn != x);
        }
      }
    }
    if (a.mode == CTDD_MODE_RATES_ONLY) {
      // no state update
    } else if (vec_x) {
      int4* o = reinterpret_cast<int4*>(a.x_out + r0);
      o[0] = make_int4(xn_out[0], xn_out[1], xn_out[2], xn_out[3]);
      o[1] = make_int4(xn_out[4], xn_out[5], xn_out[6], xn_out[7]);
    } else {
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < nr) a.x_out[r0 + r] = xn_out[r];
    }
  } while (STRIDE);
  flush_stats_cta(st, a.stats);
}

// ------------------------------------------------------------------------------------------------
// any S: CTA per 8 rows, threads over states.  smem: A[8][S] (operand rows, later reused for per-state
// terms), small per-row scalars.
constexpr int BLK_ROWS = 8;

// LT: element type of the logits, float or __nv_bfloat16 (every logits load goes through ld_logit)
template <typename LT = float>
__global__ void __launch_bounds__(256) step_block_kernel(StepArgs a) {
  extern __shared__ float smem[];
  const int S = a.S;
  float* sA = smem;                 // [8][S]
  float* sT = smem + BLK_ROWS * S;  // [8][S] per-state terms (rates / P)
  __shared__ int s_xe[BLK_ROWS], s_xb[BLK_ROWS];
  __shared__ float s_llx[BLK_ROWS], s_lse[BLK_ROWS];
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nth >> 5;
  const long long r0 = (long long)blockIdx.x * BLK_ROWS;
  const int nr = (a.rows - r0) < BLK_ROWS ? (int)(a.rows - r0) : BLK_ROWS;
  if (tid < BLK_ROWS) {
    const long long r = r0 + (tid < nr ? tid : 0);
    s_xe[tid] = a.x_eval[r];
    s_xb[tid] = a.x_base ? a.x_base[r] : s_xe[tid];
    s_llx[tid] = 0.f;
  }
  __syncthreads();
  // 1. softmax statistics and operand rows: warp w handles rows w, w+nwarp, ...
  for (int r = warp; r < BLK_ROWS; r += nwarp) {
    const LT* lp = logits_row<LT>(a, r0 + (r < nr ? r : 0));
    const int x = s_xe[r];
    float m = -INFINITY;
    for (int k = lane; k < S; k += 32) m = fmaxf(m, ld_logit(lp + k));
    m = warp_max(m);
    float sum = 0.f;
    for (int k = lane; k < S; k += 32) sum += expf(ld_logit(lp + k) - m);
    sum = warp_sum(sum);
    if (lane == 0) s_lse[r] = m + logf(sum);
    for (int k = lane; k < S; k += 32) {
      const float p = expf(ld_logit(lp + k) - m) / sum;
      float v;
      if (a.mode == CTDD_MODE_EXACT) v = p;
      else if (a.branch == CTDD_BRANCH_TAULDR) v = p / (a.QT[(size_t)x * S + k] + a.eps);
      else if (a.branch == CTDD_BRANCH_SDDM_REVERSE_LOGSCALE) v = ld_logit(lp + k) - (m + logf(sum));  // log p
      else v = p;
      sA[r * S + k] = v;
    }
  }
  __syncthreads();
  // 2. contraction over k for this thread's states; 3. rates
  for (int s = tid; s < S; s += nth) {
    float acc[BLK_ROWS];
#pragma unroll
    for (int r = 0; r < BLK_ROWS; ++r) acc[r] = 0.f;
    if (a.mode == CTDD_MODE_EXACT || a.branch == CTDD_BRANCH_TAULDR || a.branch == CTDD_BRANCH_SDDM_REVERSE_PROB) {
      for (int k = 0; k < S; ++k) {
        const float q = __ldg(a.Q + (size_t)k * S + s);
#pragma unroll
        for (int r = 0; r < BLK_ROWS; ++r) acc[r] = fmaf(sA[r * S + k], q, acc[r]);
      }
    } else if (a.mode != CTDD_MODE_EXACT && a.branch == CTDD_BRANCH_SDDM_REVERSE_LOGSCALE) {
      float mx[BLK_ROWS];
#pragma unroll
      for (int r = 0; r < BLK_ROWS; ++r) mx[r] = -INFINITY;
      for (int k = 0; k < S; ++k) {
        const float q = __ldg(a.Q + (size_t)k * S + s);
        const float lq = q <= 1e-35f ? -1e9f : logf(q);
#pragma unroll
        for (int r = 0; r < BLK_ROWS; ++r) mx[r] = fmaxf(mx[r], sA[r * S + k] + lq);
      }
      for (int k = 0; k < S; ++k) {
        const float q = __ldg(a.Q + (size_t)k * S + s);
        const float lq = q <= 1e-35f ? -1e9f : logf(q);
#pragma unroll
        for (int r = 0; r < BLK_ROWS; ++r) acc[r] += expf(sA[r * S + k] + lq - mx[r]);
      }
#pragma unroll
      for (int r = 0; r < BLK_ROWS; ++r) acc[r] = mx[r] + logf(acc[r]);  // ll[s]
    }
    if (a.mode == CTDD_MODE_EXACT) {   // weight[s] = (p Q)[s] * q_{t|t-h}[s, x]
#pragma unroll
      for (int r = 0; r < BLK_ROWS; ++r) sT[r * S + s] = acc[r] * __ldg(a.RbT + (size_t)s_xe[r] * S + s);
      continue;
    }
#pragma unroll
    for (int r = 0; r < BLK_ROWS; ++r) {
      float v = acc[r];
      if (a.branch == CTDD_BRANCH_SDDM_REVERSE_PROB) v = logf(v + 1e-35f);
      else if (a.branch == CTDD_BRANCH_SDDM_DIRECT) v = ld_logit(logits_row<LT>(a, r0 + (r < nr ? r : 0)) + s) - s_lse[r];
      sT[r * S + s] = v;  // tauLDR: ratio; SDDM: ll
      if (a.branch != CTDD_BRANCH_TAULDR && s == s_xe[r]) s_llx[r] = v;
    }
  }
  __syncthreads();
  if (a.mode == CTDD_MODE_EXACT) {
    RowStats st = {0, 0, 0, 0, 0};
    if (tid < nr) {
      const int r = tid, x = s_xe[r];
      const float v = u32_to_unit(philox_row_word((uint64_t)(a.row_offset + r0 + r), 0, a.offset, STREAM_ROW, a.seed));
      const float* rowp = sT + r * S;
      const int xn = inv_cdf(S, v, [&](int s) { return rowp[s]; });
      a.x_out[r0 + r] = xn;
      st.changed_base += (xn != s_xb[r]);
      st.changed_eval += (xn != x);
    }
    flush_stats(st, a.stats);
    return;
  }
  const bool corr = (a.mode == CTDD_MODE_TAU_LEAP_CORR || a.mode == CTDD_MODE_EULER_CORR);
  for (int s = tid; s < S; s += nth) {
#pragma unroll
    for (int r = 0; r < BLK_ROWS; ++r) {
      const int x = s_xe[r];
      float ratio, rfull;
      if (a.branch == CTDD_BRANCH_TAULDR) {
        ratio = sT[r * S + s];
        rfull = a.beta * __ldg(a.RbT + (size_t)x * S + s) * ratio;
      } else {
        ratio = expf(sT[r * S + s] - s_llx[r]);
        rfull = ratio * (a.beta * __ldg(a.Rb + (size_t)x * S + s));
      }
      if (r < nr) {
        if (a.rr_out) a.rr_out[(r0 + r) * S + s] = rfull;
        if (a.ratio_out) a.ratio_out[(r0 + r) * S + s] = ratio;
      }
      float v = rfull;
      if (corr) v = v + a.beta * __ldg(a.Rb + (size_t)x * S + s);
      sA[r * S + s] = (s == x) ? 0.f : v;  // zeroed rates (sA is free again)
    }
  }
  __syncthreads();
  RowStats st = {0, 0, 0, 0, 0};
  if (a.mode == CTDD_MODE_TAU_LEAP || a.mode == CTDD_MODE_TAU_LEAP_CORR || a.mode == CTDD_MODE_MIDPOINT_JUMP) {
    // one thread per row, oracle op order (this path doubles as the on-GPU cross-check of the tensor path)
    if (tid < nr) {
      const int r = tid;
      const float h = a.h;
      const float* rowp = sA + r * S;
      const int2 jc = tau_leap_row_seq(S, s_xe[r], (uint64_t)(a.row_offset + r0 + r), a.offset, a.seed,
                                       [&](int s) { return __fmul_rn(rowp[s], h); });
      a.x_out[r0 + r] = finalize_jump(s_xb[r], s_xe[r], jc.x, jc.y, a.reject_multi, S, st);
    }
  } else if (a.mode == CTDD_MODE_MIDPOINT_DRIFT) {
    // deterministic: warp r reduces row r in a fixed order
    for (int r = warp; r < BLK_ROWS; r += nwarp) {
      float acc = 0.f;
      for (int s = lane; s < S; s += 32) acc += sA[r * S + s] * (float)(s - s_xe[r]);
      acc = warp_sum(acc);
      if (lane == 0 && r < nr) {
        const int ch = (int)rintf(0.5f * a.h * acc);
        int xn = s_xe[r] + ch;
        xn = xn < 0 ? 0 : (xn > S - 1 ? S - 1 : xn);
        a.x_out[r0 + r] = xn;
        st.changed_base += (xn != s_xe[r]);
        st.changed_eval += (xn != s_xe[r]);
        st.nonzero += (ch != 0);
      }
    }
  } else if (a.mode == CTDD_MODE_EULER || a.mode == CTDD_MODE_EULER_CORR) {
    if (tid < nr) {
      const int r = tid, x = s_xe[r];
      float tot = 0.f;
      for (int s = 0; s < S; ++s) tot += sA[r * S + s];
      const float diag = fmaxf(0.f, 1.f - a.h * tot);
      const float v = u32_to_unit(philox_row_word((uint64_t)(a.row_offset + r0 + r), 0, a.offset, STREAM_ROW, a.seed));
      const float h = a.h;
      const float* rowp = sA + r * S;
      const int xn = inv_cdf(S, v, [&](int s) { return s == x ? diag : rowp[s] * h; });
      a.x_out[r0 + r] = xn;
      st.changed_base += (xn != s_xb[r]);
      st.changed_eval += (xn != x);
    }
  }
  flush_stats(st, a.stats);
}

// The small-S dispatch table, the same for both logits types.
template <typename LT>
void launch_step_small(const StepArgs& a, int S, bool lean, unsigned blocks, int threads, cudaStream_t st) {
  switch (S) {
    case 2:   // C1: S = 2, tau-leaping on the tauLDR branch
      if (a.mode == CTDD_MODE_TAU_LEAP && a.branch == CTDD_BRANCH_TAULDR && lean)    // grid-stride instantiation
        step_small_kernel<2, CTDD_MODE_TAU_LEAP, CTDD_BRANCH_TAULDR, true, LT>
            <<<blocks > 148u * SMALL_GRIDCAP ? 148u * SMALL_GRIDCAP : blocks, threads, 0, st>>>(a);
      else if (lean && a.branch == CTDD_BRANCH_TAULDR && a.mode == CTDD_MODE_TAU_LEAP_CORR)   // PCTauL's corrector step
        step_small_kernel<2, CTDD_MODE_TAU_LEAP_CORR, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else if (lean && a.branch == CTDD_BRANCH_TAULDR && a.mode == CTDD_MODE_EULER)
        step_small_kernel<2, CTDD_MODE_EULER, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else if (lean && a.branch == CTDD_BRANCH_TAULDR && a.mode == CTDD_MODE_EULER_CORR)
        step_small_kernel<2, CTDD_MODE_EULER_CORR, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else
        step_small_kernel<2, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a);
      break;
    case 3:   // C2: S = 3, Euler (LBJF) on the tauLDR branch
      if (a.mode == CTDD_MODE_EULER && a.branch == CTDD_BRANCH_TAULDR && lean)
        step_small_kernel<3, CTDD_MODE_EULER, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else if (lean && a.branch == CTDD_BRANCH_TAULDR && a.mode == CTDD_MODE_EULER_CORR)      // LBJF's corrector step
        step_small_kernel<3, CTDD_MODE_EULER_CORR, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else if (lean && a.branch == CTDD_BRANCH_TAULDR && a.mode == CTDD_MODE_TAU_LEAP)
        step_small_kernel<3, CTDD_MODE_TAU_LEAP, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else if (lean && a.branch == CTDD_BRANCH_TAULDR && a.mode == CTDD_MODE_TAU_LEAP_CORR)
        step_small_kernel<3, CTDD_MODE_TAU_LEAP_CORR, CTDD_BRANCH_TAULDR, true, LT><<<blocks, threads, 0, st>>>(a);
      else
        step_small_kernel<3, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a);
      break;
    case 4: step_small_kernel<4, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a); break;
    case 5: step_small_kernel<5, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a); break;
    case 6: step_small_kernel<6, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a); break;
    case 7: step_small_kernel<7, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a); break;
    default: step_small_kernel<8, -1, -1, false, LT><<<blocks, threads, 0, st>>>(a); break;
  }
}

int launch_step_simt(const ctdd_step_params* p, cudaStream_t st) {
  StepArgs a;
  a.mode = p->mode; a.branch = p->branch; a.D = p->D; a.S = p->S; a.reject_multi = p->reject_multi;
  a.rows = (long long)p->N * p->D; a.row_offset = p->row_offset;
  a.logits = p->logits; a.ld = p->ld_logits; a.batch_stride = p->batch_stride_logits;
  a.x_eval = p->x_eval; a.x_base = p->x_base; a.Q = p->Q; a.QT = p->QT; a.Rb = p->Rb; a.RbT = p->RbT;
  a.beta = p->beta; a.h = p->h; a.eps = p->eps; a.seed = p->seed; a.offset = p->offset;
  a.x_out = p->x_out; a.rr_out = p->rr_out; a.ratio_out = p->ratio_out;
  a.stats = reinterpret_cast<unsigned long long*>(p->stats_out);
  philox_key_schedule(p->seed, a.pk);
  const bool bf16 = p->logits_dtype == CTDD_DTYPE_BF16;
  const int S = p->S;
  if (S <= 8 && S >= 2) {
    const long long groups = (a.rows + 7) / 8;
    const int threads = 128;
    unsigned blocks = (unsigned)((groups + threads - 1) / threads);
    const bool lean = !a.rr_out && !a.ratio_out && a.ld == S && a.batch_stride == (long long)a.D * S;
    if (bf16) launch_step_small<__nv_bfloat16>(a, S, lean, blocks, threads, st);
    else launch_step_small<float>(a, S, lean, blocks, threads, st);
    CTDD_CHECK_LAUNCH("step_small_kernel");
    return 0;
  }
  const size_t smem = (size_t)2 * BLK_ROWS * S * sizeof(float);
  if (smem > 200 * 1024) { set_error("ctdd_reverse_step: S=%d too large for the block path", S); return 2; }
  static unsigned long long attr_done = 0ull;   // function attributes live in the device's context: a bit per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !((attr_done >> dev) & 1ull)) {
    cudaFuncSetAttribute(step_block_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(step_block_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (dev >= 0 && dev < 64) attr_done |= 1ull << dev;
  }
  int threads = ((S + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  if (threads < 64) threads = 64;
  const unsigned blocks = (unsigned)((a.rows + BLK_ROWS - 1) / BLK_ROWS);
  if (bf16) step_block_kernel<__nv_bfloat16><<<blocks, threads, smem, st>>>(a);
  else step_block_kernel<float><<<blocks, threads, smem, st>>>(a);
  CTDD_CHECK_LAUNCH("step_block_kernel");
  return 0;
}

}  // namespace ctdd

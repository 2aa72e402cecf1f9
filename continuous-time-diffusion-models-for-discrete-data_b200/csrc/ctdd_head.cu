// Truncated-logistic output head: (mu, log_scale) per dimension -> logits over S bins of [-1, 1].
// Replaces sample_logistic (reference lib/models/models.py:28-74; inline copy :248-282) with one HBM-bound pass.
//
// With z_j = (edge_j - mu) * exp(2 - log_scale) for the S+1 bin edges, u = sigmoid(z), v = sigmoid(-z),
// w = z_{s+1} - z_s and kappa = 1 - exp(-w), the reference's
//     logits_1 = logsig(z_{s+1}) + log1p(-exp(logsig(z_s) - logsig(z_{s+1})) + 1e-6)
// equals   log u_{s+1} + log(kappa * v_s + 1e-6)   exactly (1 - u_s/u_{s+1} = v_s * kappa), and the mirrored
//     logits_2 = log v_s + log(kappa * u_{s+1} + 1e-6).
// This form has no cancellation (the reference's 1 - exp(.) has), so it sits inside the reference's own fp32 noise
// around the fp64 value (tests/golden/head.npz keeps both).
#include "ctdd_common.cuh"

namespace ctdd {
namespace {

// log sigmoid(z), log sigmoid(-z), sigmoid(z), sigmoid(-z): stable for every z (e <= 1, no overflow, no cancellation)
__device__ __forceinline__ void logsig_pair(float z, float& log_u, float& log_v, float& u, float& v) {
  const float e = __expf(-fabsf(z));
  const float d = 1.0f + e;
  const float r = __fdividef(1.0f, d);
  const float ld = __logf(d);
  const bool pos = z >= 0.f;
  u = pos ? r : e * r;
  v = pos ? e * r : r;
  log_u = fminf(z, 0.f) - ld;
  log_v = fminf(-z, 0.f) - ld;
}

// Stores of the forward kernel: fp32, or bf16 rounded once to nearest even (VEC = 4: one 16-byte / one 8-byte store).
__device__ __forceinline__ void st_logits4(float* p, const float (&o)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
}
__device__ __forceinline__ void st_logits4(__nv_bfloat16* p, const float (&o)[4]) {
  const __nv_bfloat162 lo = __halves2bfloat162(__float2bfloat16_rn(o[0]), __float2bfloat16_rn(o[1]));
  const __nv_bfloat162 hi = __halves2bfloat162(__float2bfloat16_rn(o[2]), __float2bfloat16_rn(o[3]));
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}
__device__ __forceinline__ void st_logit(float* p, float o) { *p = o; }
__device__ __forceinline__ void st_logit(__nv_bfloat16* p, float o) { *p = __float2bfloat16_rn(o); }

// Incoming gradient of the backward kernel, widened on load: VEC = 4 reads one 16-byte (fp32) or 8-byte (bf16) word.
__device__ __forceinline__ void ld_grad4(const float* p, float (&gr)[4]) {
  const float4 q = __ldg(reinterpret_cast<const float4*>(p));
  gr[0] = q.x; gr[1] = q.y; gr[2] = q.z; gr[3] = q.w;
}
__device__ __forceinline__ void ld_grad4(const __nv_bfloat16* p, float (&gr)[4]) {
  widen_bf16x4(__ldg(reinterpret_cast<const uint2*>(p)), gr[0], gr[1], gr[2], gr[3]);
}

// one thread per VEC consecutive states of a row (VEC + 1 bin edges); row scalars are recomputed per thread.
// IT: type of mu / log_scale, OT: type of the logits (float or __nv_bfloat16); bf16 inputs are widened on load (exact),
// every logit is computed in fp32 as for fp32 inputs, and a bf16 output is that value rounded once at the store.
template <int VEC, typename IT, typename OT>
__global__ void __launch_bounds__(256) logistic_logits_kernel(const IT* __restrict__ mu, const IT* __restrict__ log_scale,
                                                              long long rows, int D, long long batch_stride, int S, int fix,
                                                              OT* __restrict__ out) {
  const int per_row = S / VEC;
  const long long total = rows * per_row;
  const float bw = 2.0f / (float)S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long g = i / per_row;
    const int s0 = (int)(i - g * per_row) * VEC;
    long long src = g;
    if (batch_stride != (long long)D) {
      const long long n = g / D;
      src = n * batch_stride + (g - n * D);
    }
    const float m = ld_logit(mu + src);
    const float inv = expf(2.0f - ld_logit(log_scale + src));
    const float kap = -expm1f(-inv * bw);
    float lu[VEC + 1], lv[VEC + 1], u[VEC + 1], v[VEC + 1];
#pragma unroll
    for (int k = 0; k <= VEC; ++k) {
      // bin edges are exact in fp32 (multiples of 2/S), like the reference's centers -/+ bin_width/2
      const float z = (fmaf((float)(s0 + k), bw, -1.0f) - m) * inv;
      logsig_pair(z, lu[k], lv[k], u[k], v[k]);
    }
    float o[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      o[k] = lu[k + 1] + __logf(fmaf(kap, v[k], 1e-6f));
      if (fix) o[k] = fminf(o[k], lv[k] + __logf(fmaf(kap, u[k + 1], 1e-6f)));
    }
    if constexpr (VEC == 4) {
      st_logits4(out + g * S + s0, o);
    } else {
#pragma unroll
      for (int k = 0; k < VEC; ++k) st_logit(out + g * S + s0 + k, o[k]);
    }
  }
}

// Backward of the head: d mu = sum_s g_s dlogit_s/dmu, d log_scale = sum_s g_s dlogit_s/dlog_scale.  One warp per row,
// lane-strided 128-bit reads of the incoming gradient (each read once), butterfly reduce.  With z' = dz/dmu = -inv,
// dz/dlog_scale = -z, dkappa/dlog_scale = -w (1 - kappa), d log u/dz = v, d log v/dz = -u, dv/dz = -u v, du/dz = u v:
//   logits_1 = log u_{s+1} + log A,  A = kappa v_s + 1e-6
//     d/dmu = inv (-v_{s+1} + kappa u_s v_s / A),   d/dls = -z_{s+1} v_{s+1} + (kappa u_s v_s z_s - w (1-kappa) v_s) / A
//   logits_2 = log v_s + log B,      B = kappa u_{s+1} + 1e-6
//     d/dmu = inv (u_s - kappa u_{s+1} v_{s+1} / B), d/dls = z_s u_s - (kappa u_{s+1} v_{s+1} z_{s+1} + w (1-kappa) u_{s+1}) / B
// IT: type of mu / log_scale, GT: type of grad_logits (float or __nv_bfloat16), both widened on load.  A bf16 gradient is
// read with the VEC, lane -> state assignment and accumulation order of the fp32 one, so the results equal those of the
// fp32 kernel on the widened tensors bit for bit.  dmu / dls are fp32.
template <int VEC, typename IT, typename GT>
__global__ void __launch_bounds__(256) logistic_backward_kernel(const IT* __restrict__ mu, const IT* __restrict__ log_scale,
                                                                const GT* __restrict__ grad_logits, long long rows, int D,
                                                                long long batch_stride, int S, int fix,
                                                                float* __restrict__ dmu, float* __restrict__ dls) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const float bw = 2.0f / (float)S;
  for (long long g = warp0; g < rows; g += nwarps) {
    long long src = g;
    if (batch_stride != (long long)D) {
      const long long n = g / D;
      src = n * batch_stride + (g - n * D);
    }
    const float m = ld_logit(mu + src);
    const float inv = expf(2.0f - ld_logit(log_scale + src));
    const float w = inv * bw;
    const float kap = -expm1f(-w);
    const float wk = w * (1.0f - kap);
    float acc_mu = 0.f, acc_ls = 0.f;
    for (int s0 = lane * VEC; s0 < S; s0 += 32 * VEC) {
      float gr[VEC];
      if constexpr (VEC == 4) {
        ld_grad4(grad_logits + g * S + s0, gr);
      } else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) gr[k] = ld_logit(grad_logits + g * S + s0 + k);
      }
      float z[VEC + 1], lu[VEC + 1], lv[VEC + 1], u[VEC + 1], v[VEC + 1];
#pragma unroll
      for (int k = 0; k <= VEC; ++k) {
        z[k] = (fmaf((float)(s0 + k), bw, -1.0f) - m) * inv;
        logsig_pair(z[k], lu[k], lv[k], u[k], v[k]);
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const float uv_l = u[k] * v[k], uv_r = u[k + 1] * v[k + 1];
        const float A = fmaf(kap, v[k], 1e-6f);
        float d_mu = -v[k + 1] + kap * uv_l / A;
        float d_ls = -z[k + 1] * v[k + 1] + (kap * uv_l * z[k] - wk * v[k]) / A;
        if (fix) {
          const float B = fmaf(kap, u[k + 1], 1e-6f);
          const float l1 = lu[k + 1] + __logf(A), l2 = lv[k] + __logf(B);
          if (l2 < l1) {
            d_mu = u[k] - kap * uv_r / B;
            d_ls = z[k] * u[k] - (kap * uv_r * z[k + 1] + wk * u[k + 1]) / B;
          }
        }
        acc_mu = fmaf(gr[k], d_mu, acc_mu);
        acc_ls = fmaf(gr[k], d_ls, acc_ls);
      }
    }
    acc_mu = warp_sum(acc_mu);
    acc_ls = warp_sum(acc_ls);
    if (lane == 0) {
      dmu[src] = acc_mu * inv;
      dls[src] = acc_ls;
    }
  }
}

template <typename IT, typename OT>
void launch_logits(const void* mu, const void* log_scale, long long rows, int D, int64_t batch_stride, int S, int fix,
                   void* out, bool vec4, unsigned blocks, cudaStream_t st) {
  const IT* m = static_cast<const IT*>(mu);
  const IT* l = static_cast<const IT*>(log_scale);
  if (vec4)
    logistic_logits_kernel<4, IT, OT><<<blocks, 256, 0, st>>>(m, l, rows, D, batch_stride, S, fix, static_cast<OT*>(out));
  else
    logistic_logits_kernel<1, IT, OT><<<blocks, 256, 0, st>>>(m, l, rows, D, batch_stride, S, fix, static_cast<OT*>(out));
}

template <typename IT, typename GT>
void launch_backward(const void* mu, const void* log_scale, const void* grad, long long rows, int D, int64_t batch_stride,
                     int S, int fix, float* dmu, float* dls, bool vec4, unsigned blocks, cudaStream_t st) {
  const IT* m = static_cast<const IT*>(mu);
  const IT* l = static_cast<const IT*>(log_scale);
  const GT* g = static_cast<const GT*>(grad);
  if (vec4)
    logistic_backward_kernel<4, IT, GT><<<blocks, 256, 0, st>>>(m, l, g, rows, D, batch_stride, S, fix, dmu, dls);
  else
    logistic_backward_kernel<1, IT, GT><<<blocks, 256, 0, st>>>(m, l, g, rows, D, batch_stride, S, fix, dmu, dls);
}

bool known_dtype(int t) { return t == CTDD_DTYPE_F32 || t == CTDD_DTYPE_BF16; }
size_t dtype_bytes(int t) { return t == CTDD_DTYPE_BF16 ? 2 : 4; }

}  // namespace
}  // namespace ctdd

extern "C" int ctdd_logistic_logits_ex(const void* mu, const void* log_scale, int in_dtype, int N, int D,
                                       int64_t batch_stride, int S, int fix_logistic, void* logits_out, int out_dtype,
                                       void* stream) {
  using namespace ctdd;
  if (!mu || !log_scale || !logits_out) { set_error("ctdd_logistic_logits: null pointer"); return 2; }
  if (!known_dtype(in_dtype) || !known_dtype(out_dtype)) {
    set_error("ctdd_logistic_logits: unknown dtype in=%d out=%d (CTDD_DTYPE_F32 = 0, CTDD_DTYPE_BF16 = 1)", in_dtype, out_dtype);
    return 2;
  }
  if (N <= 0 || D <= 0 || S < 2 || batch_stride < D) { set_error("ctdd_logistic_logits: bad sizes N=%d D=%d S=%d stride=%lld", N, D, S, (long long)batch_stride); return 2; }
  const long long rows = (long long)N * D, total = rows * S;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // VEC = 4 stores 4 logits at once: 16 bytes (fp32) or 8 bytes (bf16), so the output must be aligned to that
  const bool vec4 = (S % 4 == 0) && ((reinterpret_cast<uintptr_t>(logits_out) & (4 * dtype_bytes(out_dtype) - 1)) == 0);
  long long blocks = ((vec4 ? total / 4 : total) + 255) / 256;
  if (blocks > (long long)sms * 16) blocks = (long long)sms * 16;
  auto launch = (in_dtype == CTDD_DTYPE_BF16)
                    ? (out_dtype == CTDD_DTYPE_BF16 ? launch_logits<__nv_bfloat16, __nv_bfloat16> : launch_logits<__nv_bfloat16, float>)
                    : (out_dtype == CTDD_DTYPE_BF16 ? launch_logits<float, __nv_bfloat16> : launch_logits<float, float>);
  launch(mu, log_scale, rows, D, batch_stride, S, fix_logistic, logits_out, vec4, (unsigned)blocks, (cudaStream_t)stream);
  CTDD_CHECK_LAUNCH("logistic_logits_kernel");
  return 0;
}

extern "C" int ctdd_logistic_logits(const float* mu, const float* log_scale, int N, int D, int64_t batch_stride, int S,
                                    int fix_logistic, float* logits_out, void* stream) {
  return ctdd_logistic_logits_ex(mu, log_scale, CTDD_DTYPE_F32, N, D, batch_stride, S, fix_logistic, logits_out, CTDD_DTYPE_F32, stream);
}

extern "C" int ctdd_logistic_logits_backward_ex(const void* mu, const void* log_scale, int in_dtype, const void* grad_logits,
                                                int grad_dtype, int N, int D, int64_t batch_stride, int S, int fix_logistic,
                                                float* grad_mu, float* grad_log_scale, void* stream) {
  using namespace ctdd;
  if (!mu || !log_scale || !grad_logits || !grad_mu || !grad_log_scale) { set_error("ctdd_logistic_logits_backward: null pointer"); return 2; }
  if (!known_dtype(in_dtype) || !known_dtype(grad_dtype)) {
    set_error("ctdd_logistic_logits_backward: unknown dtype in=%d grad=%d (CTDD_DTYPE_F32 = 0, CTDD_DTYPE_BF16 = 1)", in_dtype, grad_dtype);
    return 2;
  }
  if (N <= 0 || D <= 0 || S < 2 || batch_stride < D) { set_error("ctdd_logistic_logits_backward: bad sizes N=%d D=%d S=%d stride=%lld", N, D, S, (long long)batch_stride); return 2; }
  const long long rows = (long long)N * D;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  long long blocks = (rows + 7) / 8;      // 8 warps per block, one row per warp per iteration
  if (blocks > (long long)sms * 8) blocks = (long long)sms * 8;
  // VEC = 4 reads 4 gradient entries at once: 16 bytes (fp32) or 8 bytes (bf16)
  const bool vec4 = (S % 4 == 0) && ((reinterpret_cast<uintptr_t>(grad_logits) & (4 * dtype_bytes(grad_dtype) - 1)) == 0);
  auto launch = (in_dtype == CTDD_DTYPE_BF16)
                    ? (grad_dtype == CTDD_DTYPE_BF16 ? launch_backward<__nv_bfloat16, __nv_bfloat16> : launch_backward<__nv_bfloat16, float>)
                    : (grad_dtype == CTDD_DTYPE_BF16 ? launch_backward<float, __nv_bfloat16> : launch_backward<float, float>);
  launch(mu, log_scale, grad_logits, rows, D, batch_stride, S, fix_logistic, grad_mu, grad_log_scale, vec4, (unsigned)blocks,
         (cudaStream_t)stream);
  CTDD_CHECK_LAUNCH("logistic_backward_kernel");
  return 0;
}

extern "C" int ctdd_logistic_logits_backward(const float* mu, const float* log_scale, const float* grad_logits, int N, int D,
                                             int64_t batch_stride, int S, int fix_logistic, float* grad_mu,
                                             float* grad_log_scale, void* stream) {
  return ctdd_logistic_logits_backward_ex(mu, log_scale, CTDD_DTYPE_F32, grad_logits, CTDD_DTYPE_F32, N, D, batch_stride, S,
                                          fix_logistic, grad_mu, grad_log_scale, stream);
}

// Fused loss terms (forward + backward w.r.t. the logits) for the three loss families of lib/losses/losses.py:
//   CTDD_LOSS_CTELBO  tauLDR CT-ELBO   losses.py:108-286  (CTElbo, NLL, CTElboLambda, CondCTElbo)
//   CTDD_LOSS_SDDM    SDDM ELBO        losses.py:1345-1500 (ScoreElbo), :389-544 (SDDMElbo)
//   CTDD_LOSS_CRM     ratio matching   losses.py:794-890 (CatRM), :1146-1242 (CatRMNLL)
// One CTA owns ROWS rows (b, d..d+ROWS-1) of ONE sample, so the per-sample q_{t|0} is shared by the CTA; threads span
// the state axis. The (rows x S)(S x S) contractions against the per-sample Q run on CUDA cores in this round
// (2*B*D*S^2 FLOP forward, 4*B*D*S^2 backward: the backward recomputes u instead of saving a (B,D,S) tensor).
// S == 256 uses ROWS = 32 and a 16-row x 2-state register tile per thread: each Q element fetched from L2 feeds 16 FMAs
// and each 128-bit shared-memory operand load 8 (the ROWS = 8 / one-state-per-thread form streamed the 256 KB per-sample
// Q once per 8 rows and was L2-bandwidth bound at ~15 TFLOP/s); other S keep ROWS = 8.  The k order of every dot
// product is the same in both forms, so the results are bit-identical.
// Per-sample reductions are returned as [B] vectors; the final means / weights are combined by the Python classes.
// Logits and their gradient are fp32, bf16 or fp16 (ctdd_loss_params::logits_dtype; template argument LT of every kernel
// that touches them).  The 2-byte types are widened on load, which is exact, and the fp32 code runs unchanged; the
// gradient is rounded once (round-to-nearest-even) when it is stored.  A bf16 or fp16 call therefore returns the
// per-sample terms of the same call on the widened logits (bit for bit up to the order of the cross-CTA atomicAdds) and
// that call's gradient rounded to the logits' type.
#include "ctdd_common.cuh"

namespace ctdd {
namespace loss {


struct Args {
  int kind, logit_type, crm_type, B, D, S;
  const void* logits;  // [B][D][S] of LT
  const float* Q;
  const float* QT;
  const float* Rb;
  const float* beta;
  const int* x0;
  const int* xt;       // state the ratio/reg terms are evaluated at (CTELBO: reg_x; SDDM/CRM: state of the logits)
  const int* x_tilde;  // CTELBO: signal-term state; SDDM: == xt
  const float* G;      // CTELBO: [B][x][k] = beta * sum_s Rb[s,x][s!=x] Q[k,s] / (Q[k,x]+eps)
  const float* baseZ;  // [B] sum_d z_b[x_tilde_d]
  const float* RbT;    // [x][s] = Rb[s][x]: the per-(row, s) terms read a COLUMN of Rb per row (coalesced through the transpose)
  const float* RbD;    // [s] = Rb[s][s]
  float eps;
  float* out_a; float* out_b; float* out_c; float* out_d; float* out_nll;
  const float* ga; const float* gb; const float* gd; const float* gn;
  void* grad;          // [B][D][S] of LT
  float* bufA;         // tensor-core path (S == 256): [B][D][S] GEMM operand p, later the cotangent V
  float* bufU;         // tensor-core path: [B][D][S] u = p Q (kept from forward to backward), later dp = V Q^T
  float* lse;          // tensor-core path: [B][D] log-sum-exp of every logits row (kept from forward to backward)
  float* fix;          // tensor-core path: [B][D] cotangent of u at the evaluation state that comes through ll_x (backward)
};

__device__ __forceinline__ float log1mexp_ref(float v) {  // lib/utils/utils.py:86-91
  const float x = -fabsf(v);
  return x > -0.693f ? logf(-expm1f(x)) : log1pf(-expf(x));
}

// G[b][x][k] = beta_b * (sum_s RzT[x][s] * QT_b[s][k]) / (QT_b[x][k] + eps), RzT[x][s] = Rb[s][x] (s != x)
// 64 x 64 output tile per CTA, 4 x 4 register tile per thread (rows x = x0 + ty + 16a, columns k = k0 + 4tx .. +3);
// the s order of every dot product is ascending.
__global__ void __launch_bounds__(256) ctelbo_table_kernel(const float* __restrict__ QT, const float* __restrict__ Rb,
                                                          const float* __restrict__ beta, int S, float eps,
                                                          float* __restrict__ G) {
  __shared__ __align__(16) float sA[16][64];    // [s][x]
  __shared__ __align__(16) float sB[16][64];    // [s][k]
  const int b = blockIdx.z, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int x0 = blockIdx.y * 64, k0 = blockIdx.x * 64;
  const float* qt = QT + (size_t)b * S * S;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
  for (int s0 = 0; s0 < S; s0 += 16) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + 256 * e, sl = idx >> 6, col = idx & 63;
      const int sg = s0 + sl, x = x0 + col, k = k0 + col;
      sA[sl][col] = (sg < S && x < S && sg != x) ? Rb[(size_t)sg * S + x] : 0.f;
      sB[sl][col] = (sg < S && k < S) ? qt[(size_t)sg * S + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const float4 bv = *reinterpret_cast<const float4*>(&sB[m][4 * tx]);
      const float bq[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float av = sA[m][ty + 16 * a];
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(av, bq[c], acc[a][c]);
      }
    }
    __syncthreads();
  }
  const float bt = beta[b];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int x = x0 + ty + 16 * a;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int k = k0 + 4 * tx + c;
      if (x < S && k < S) G[((size_t)b * S + x) * S + k] = bt * acc[a][c] / (qt[(size_t)x * S + k] + eps);
    }
  }
}

__global__ void basez_kernel(const float* __restrict__ Rb, const float* __restrict__ beta, const int* __restrict__ x_tilde,
                             int D, int S, float* __restrict__ baseZ) {
  const int b = blockIdx.x;
  float acc = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const int x = x_tilde[(size_t)b * D + d];
    acc += -beta[b] * Rb[(size_t)x * S + x];
  }
  acc = warp_sum(acc);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) baseZ[b] = v;
  }
}

// out[r][c] = epi(r, c, sum_j in[r][j] * M[j][c]) for the CTA's ROWS rows; `in` / `out` are [ROWS][S] shared-memory
// arrays, M a row-major S x S matrix in global memory (L2-resident).  The j order is sequential in every variant.
// RbT[x][s] = Rb[s][x], RbD[s] = Rb[s][s] (built by the forward call into the workspace)
__global__ void __launch_bounds__(256) rb_tables_kernel(const float* __restrict__ Rb, int S, float* __restrict__ RbT,
                                                        float* __restrict__ RbD) {
  __shared__ float tile[16][17];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int x = blockIdx.x * 16 + tx, y = blockIdx.y * 16 + ty;
  tile[ty][tx] = (x < S && y < S) ? Rb[(size_t)y * S + x] : 0.f;
  __syncthreads();
  const int ox = blockIdx.y * 16 + tx, oy = blockIdx.x * 16 + ty;
  if (ox < S && oy < S) RbT[(size_t)oy * S + ox] = tile[tx][ty];
  if (blockIdx.x == blockIdx.y && ty == tx && x < S) RbD[x] = tile[ty][tx];
}

template <int ROWS, class Epi>
__device__ __forceinline__ void rows_times_matrix(const float* __restrict__ in, const float* __restrict__ M, int S, Epi epi) {
  const int tid = threadIdx.x, nth = blockDim.x;
  if (ROWS == 32 && S == 256 && nth == 256) {
    // 16 rows x 2 adjacent columns per thread; a warp reads one 256-byte run of M per j and broadcasts the operand
    constexpr int RT = 16;
    const int c = 2 * (tid & 127), r0 = RT * (tid >> 7);
    float acc0[RT], acc1[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) acc0[r] = acc1[r] = 0.f;
    const float* mp = M + c;
    const float* ip = in + r0 * 256;
    // the four matrix rows of step j + 4 are requested before the FMAs of step j (L2 latency off the critical path)
    float2 q0 = __ldg(reinterpret_cast<const float2*>(mp));
    float2 q1 = __ldg(reinterpret_cast<const float2*>(mp + 256));
    float2 q2 = __ldg(reinterpret_cast<const float2*>(mp + 512));
    float2 q3 = __ldg(reinterpret_cast<const float2*>(mp + 768));
#pragma unroll 1
    for (int j = 0; j < 256; j += 4) {
      const int jn = (j + 4 < 256) ? j + 4 : j;
      const float2 n0 = __ldg(reinterpret_cast<const float2*>(mp + (size_t)jn * 256));
      const float2 n1 = __ldg(reinterpret_cast<const float2*>(mp + (size_t)(jn + 1) * 256));
      const float2 n2 = __ldg(reinterpret_cast<const float2*>(mp + (size_t)(jn + 2) * 256));
      const float2 n3 = __ldg(reinterpret_cast<const float2*>(mp + (size_t)(jn + 3) * 256));
#pragma unroll
      for (int r = 0; r < RT; ++r) {
        const float4 av = *reinterpret_cast<const float4*>(ip + r * 256 + j);
        acc0[r] = fmaf(av.w, q3.x, fmaf(av.z, q2.x, fmaf(av.y, q1.x, fmaf(av.x, q0.x, acc0[r]))));
        acc1[r] = fmaf(av.w, q3.y, fmaf(av.z, q2.y, fmaf(av.y, q1.y, fmaf(av.x, q0.y, acc1[r]))));
      }
      q0 = n0; q1 = n1; q2 = n2; q3 = n3;
    }
#pragma unroll
    for (int r = 0; r < RT; ++r) { epi(r0 + r, c, acc0[r]); epi(r0 + r, c + 1, acc1[r]); }
    return;
  }
  const bool vec4 = (S & 3) == 0;   // rows of the smem operands are 16-byte aligned only then
  for (int c = tid; c < S; c += nth) {
    for (int rb = 0; rb < ROWS; rb += 8) {
      float acc[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) acc[r] = 0.f;
      int j = 0;
      for (; vec4 && j + 4 <= S; j += 4) {   // 4 contraction steps per 128-bit shared-memory load of every row's operand
        const float q0 = __ldg(M + (size_t)j * S + c), q1 = __ldg(M + (size_t)(j + 1) * S + c);
        const float q2 = __ldg(M + (size_t)(j + 2) * S + c), q3 = __ldg(M + (size_t)(j + 3) * S + c);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const float4 av = *reinterpret_cast<const float4*>(in + (rb + r) * S + j);
          acc[r] = fmaf(av.w, q3, fmaf(av.z, q2, fmaf(av.y, q1, fmaf(av.x, q0, acc[r]))));
        }
      }
      for (; j < S; ++j) {
        const float q = __ldg(M + (size_t)j * S + c);
#pragma unroll
        for (int r = 0; r < 8; ++r) acc[r] = fmaf(in[(rb + r) * S + j], q, acc[r]);
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) epi(rb + r, c, acc[r]);
    }
  }
}

// One logits element as fp32.  fp32 keeps a plain load (ld_logit's __ldg would change the fp32 kernels' code); bf16 and
// fp16 are widened by ld_logit.
template <typename LT>
__device__ __forceinline__ float logit_at(const LT* p) {
  if constexpr (sizeof(LT) == 4) return *p;
  else return ld_logit(p);
}
// One gradient element: fp32 stored as it is, bf16 and fp16 rounded to nearest even.
__device__ __forceinline__ void st_grad(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_grad(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void st_grad(__half* p, float v) { *p = __float2half_rn(v); }

template <bool BWD, int ROWS, typename LT = float>
__global__ void __launch_bounds__(256, ROWS == 32 ? 2 : 1) loss_kernel(const Args a) {
  extern __shared__ __align__(16) float smem[];
  const int S = a.S;
  float* sP = smem;                 // [ROWS][S] softmax p
  float* sA = smem + ROWS * S;      // [ROWS][S] GEMM operand (p * a, or p), later dp
  float* sU = smem + 2 * ROWS * S;  // [ROWS][S] u, later the s-space cotangent
  __shared__ int s_x0[ROWS], s_xr[ROWS], s_xt[ROWS];
  __shared__ float s_llx[ROWS], s_lse[ROWS], s_row_a[ROWS], s_row_b[ROWS], s_row_c[ROWS], s_row_d[ROWS], s_row_n[ROWS];
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nth >> 5;
  const int b = blockIdx.y;
  const int d0 = blockIdx.x * ROWS;
  const int nr = (a.D - d0) < ROWS ? (a.D - d0) : ROWS;
  const float* Q = a.Q + (size_t)b * S * S;
  const float* QT = a.QT + (size_t)b * S * S;
  const float beta = a.beta[b];
  const bool ctelbo = a.kind == CTDD_LOSS_CTELBO;
  const bool direct = !ctelbo && a.logit_type == CTDD_BRANCH_SDDM_DIRECT;
  // reverse_prob: ll = log(u + 1e-35) (model_utils.py:41-46).  reverse_logscale (model_utils.py:49-54) is the log-sum-exp
  // form of the same contraction without the guard: ll = log(u), and -1e9 where no term survives (log q = -1e9 there)
  const float lle = (!ctelbo && a.logit_type == CTDD_BRANCH_SDDM_REVERSE_LOGSCALE) ? 0.f : 1e-35f;
  auto ll_of = [&](float u) { const float v = u + lle; return v > 0.f ? __logf(v) : -1e9f; };
  if (tid < ROWS) {
    const size_t r = (size_t)b * a.D + d0 + (tid < nr ? tid : 0);
    s_x0[tid] = a.x0[r];
    s_xr[tid] = a.xt[r];
    s_xt[tid] = a.x_tilde ? a.x_tilde[r] : a.xt[r];
    s_row_a[tid] = s_row_b[tid] = s_row_c[tid] = s_row_d[tid] = s_row_n[tid] = 0.f;
  }
  __syncthreads();
  // 1. softmax, GEMM operand
  for (int r = warp; r < ROWS; r += nwarp) {
    const LT* lp = static_cast<const LT*>(a.logits) + ((size_t)b * a.D + d0 + (r < nr ? r : 0)) * S;
    float m = -INFINITY;
    for (int k = lane; k < S; k += 32) m = fmaxf(m, logit_at(lp + k));
    m = warp_max(m);
    float sum = 0.f;
    for (int k = lane; k < S; k += 32) {      // one exp per element: the numerators are parked in sP
      const float e = expf(logit_at(lp + k) - m);
      sP[r * S + k] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float lse = m + logf(sum);
    if (lane == 0) { s_lse[r] = lse; s_row_n[r] = lse - logit_at(lp + s_x0[r]); }
    const int xt = s_xt[r];
    const float rsum = 1.f / sum;
    for (int k = lane; k < S; k += 32) {
      const float p = sP[r * S + k] * rsum;
      sP[r * S + k] = p;
      sA[r * S + k] = ctelbo ? __fdividef(p, QT[(size_t)xt * S + k] + a.eps) : p;
    }
  }
  __syncthreads();
  // 2. u[r][s] = sum_k A[r][k] Q[k][s]
  if (!direct) {
    rows_times_matrix<ROWS>(sA, Q, S, [&](int r, int c, float v) { sU[r * S + c] = v; });
  } else {
    for (int s = tid; s < S; s += nth)
#pragma unroll
      for (int r = 0; r < ROWS; ++r)
        sU[r * S + s] = logit_at(static_cast<const LT*>(a.logits) + ((size_t)b * a.D + d0 + (r < nr ? r : 0)) * S + s) - s_lse[r];  // ll directly
  }
  __syncthreads();
  // SDDM / CRM: ll[s] and ll at the evaluation state
  if (!ctelbo) {
    if (tid < ROWS) {
      const float ux = sU[tid * S + s_xr[tid]];
      s_llx[tid] = direct ? ux : (ux + lle > 0.f ? logf(ux + lle) : -1e9f);
    }
    __syncthreads();
  }
  // 3. per-(row, s) terms; row reductions by warp r
  const float baseZ = (a.kind != CTDD_LOSS_CRM) ? a.baseZ[b] : 0.f;
  for (int r = warp; r < ROWS; r += nwarp) {
    const int x0 = s_x0[r], xr = s_xr[r], xt = s_xt[r];
    const float ga = BWD ? a.ga[b] : 0.f, gb = BWD ? a.gb[b] : 0.f, gd = BWD ? a.gd[b] : 0.f;
    float ra = 0.f, rb = 0.f, rc = 0.f, wsum = 0.f;
    if (ctelbo) {
      const float inv_den = 1.f / (Q[(size_t)x0 * S + xt] + a.eps);   // per row: the per-element divisions become products
      const float zt = -beta * a.Rb[(size_t)xt * S + xt];
      const float* Gr = a.G + ((size_t)b * S + xr) * S;
      const float* rcol = a.RbT + (size_t)xt * S;      // Rb[., xt]
      for (int s = lane; s < S; s += 32) {
        const float u = sU[r * S + s];
        const float w = (s == xt) ? 0.f : beta * rcol[s] * Q[(size_t)x0 * S + s] * inv_den;
        const float Z = baseZ - zt + (-beta * a.RbD[s]);
        rb += w * __logf(u + a.eps);
        rc += __fdividef(w, Z);
        ra += sP[r * S + s] * Gr[s];                 // reg: sum_k p_k G[x_reg][k]   (index s doubles as k)
        if (BWD) sU[r * S + s] = __fdividef(gb * w, u + a.eps);  // cotangent of u
      }
    } else {
      const float llx = s_llx[r];
      const float inv_den = 1.f / (Q[(size_t)x0 * S + xr] + a.eps);
      const float inv_ex = expf(-llx);          // reverse_prob: exp(ll_s - ll_x) = (u_s + 1e-35) * exp(-ll_x)
      const float zt = -beta * a.Rb[(size_t)xr * S + xr];
      const float* rcol = a.RbT ? a.RbT + (size_t)xr * S : nullptr;      // Rb[., xr] (SDDM only)
      for (int s = lane; s < S; s += 32) {
        const float uraw = sU[r * S + s];
        const float ll = direct ? uraw : ll_of(uraw);
        float dll = 0.f;
        if (a.kind == CTDD_LOSS_SDDM) {
          const float rs = (s == xr) ? 0.f : beta * rcol[s];
          const float e = direct ? __expf(ll - llx) : (uraw + lle) * inv_ex;
          const float w = (s == xr) ? 0.f : rs * Q[(size_t)x0 * S + s] * inv_den;
          const float Z = baseZ - zt + (-beta * a.RbD[s]);
          ra += e * rs;
          rb += w * (ll - llx);
          rc += __fdividef(w, Z);
          wsum += w;
          dll = ga * e * rs + gb * w;
        } else {  // CRM
          if (a.crm_type == 1) {          // mle
            ra += -log1mexp_ref(ll);
            const float el = expf(ll);
            dll = (s == xr) ? 0.f : ga * el / (1.f - el);
          } else if (a.crm_type == 2) {   // elbo
            if (s != xr) {
              const float e = expf(ll - llx);
              const float qsx = QT[(size_t)xr * S + s], qxs = Q[(size_t)xr * S + s];   // Q[s][xr] through the transpose
              ra += e * qsx - (llx - ll) * qxs;
              wsum += e * qsx + qxs;
              dll = ga * (e * qsx + qxs);
            }
          }
        }
        if (BWD) sU[r * S + s] = direct ? dll : (uraw + lle > 0.f ? __fdividef(dll, uraw + lle) : 0.f);   // cotangent of u (or of ll for direct)
      }
    }
    ra = warp_sum(ra); rb = warp_sum(rb); rc = warp_sum(rc); wsum = warp_sum(wsum);
    float rd = 0.f;
    if (!ctelbo) {
      const float llx = s_llx[r];
      float dllx;
      if (a.kind == CTDD_LOSS_SDDM) {
        dllx = -ga * ra - gb * wsum;
      } else {
        if (a.crm_type == 0) { ra = -llx; dllx = -ga; }
        else if (a.crm_type == 1) { ra = -((float)(S - 1) * llx) + ra + log1mexp_ref(llx); dllx = -ga * (float)(S - 1); }
        else { dllx = -ga * wsum; }
      }
      rd = -llx;
      dllx -= gd;
      if (BWD) {
        __syncwarp();
        // the cotangent at the evaluation state also receives d/d ll_x; for reverse_prob u_x + 1e-35 = exp(ll_x)
        if (lane == 0) sU[r * S + xr] += dllx / (direct ? 1.f : expf(llx));
      }
    }
    if (lane == 0) { s_row_a[r] = ra; s_row_b[r] = rb; s_row_c[r] = rc; s_row_d[r] = rd; }
  }
  __syncthreads();
  if (!BWD) {
    if (tid == 0) {
      float A = 0.f, Bv = 0.f, C = 0.f, Dd = 0.f, Nn = 0.f;
      for (int r = 0; r < nr; ++r) { A += s_row_a[r]; Bv += s_row_b[r]; C += s_row_c[r]; Dd += s_row_d[r]; Nn += s_row_n[r]; }
      atomicAdd(a.out_a + b, A);
      atomicAdd(a.out_b + b, Bv);
      atomicAdd(a.out_c + b, C);
      atomicAdd(a.out_d + b, Dd);
      atomicAdd(a.out_nll + b, Nn);
    }
    return;
  }
  // 4. dp[r][k] = a[k] * sum_s V[r][s] Q[k][s]  (+ reg part)  — threads over k, QT[s][k] coalesced
  const float gn = a.gn[b];
  {
    const float ga_b = a.ga[b];
    auto store_dp = [&](int r, int k, float dp) {
      if (ctelbo) dp = dp / (QT[(size_t)s_xt[r] * S + k] + a.eps) + ga_b * a.G[((size_t)b * S + s_xr[r]) * S + k];
      sA[r * S + k] = dp;
    };
    if (!direct) {
      rows_times_matrix<ROWS>(sU, QT, S, store_dp);
    } else {
      for (int k = tid; k < S; k += nth)
        for (int r = 0; r < ROWS; ++r) store_dp(r, k, 0.f);
    }
  }
  __syncthreads();
  // 5. softmax Jacobian + cross-entropy gradient
  for (int r = warp; r < ROWS; r += nwarp) {
    if (r >= nr) continue;
    float dot = 0.f;
    if (direct) {
      for (int k = lane; k < S; k += 32) dot += sU[r * S + k];          // sum_s dll_s
    } else {
      for (int k = lane; k < S; k += 32) dot += sP[r * S + k] * sA[r * S + k];
    }
    dot = warp_sum(dot);
    LT* gp = static_cast<LT*>(a.grad) + ((size_t)b * a.D + d0 + r) * S;
    const int x0 = s_x0[r];
    for (int k = lane; k < S; k += 32) {
      const float p = sP[r * S + k];
      float g = direct ? (sU[r * S + k] - p * dot) : p * (sA[r * S + k] - dot);
      g += gn * (p - (k == x0 ? 1.f : 0.f));
      st_grad(gp + k, g);
    }
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Tensor-core path (S == 256, SDDM / CRM kinds, reverse_prob / reverse_logscale): the two contractions run on tcgen05
// (ctdd_bgemm256_tc); what is left of loss_kernel are three streaming passes, one warp per row, lane l owns the states
// 4l..4l+3 and 128+4l..+3 (two coalesced 128-bit accesses per array), no shared-memory staging:
//   tc_pre_kernel   softmax p -> bufA, lse -> a.lse, cross-entropy sum                       (forward)
//   tc_terms_kernel u from bufU: the per-(row, s) terms and their per-sample sums            (forward)
//                   or the cotangent V = dL/du -> bufA                                        (backward)
//   tc_post_kernel  dp = V Q^T from bufU: softmax Jacobian + cross-entropy gradient -> grad   (backward)
// The arithmetic per element is loss_kernel's (phases 1, 3 and 5).  With bf16 or fp16 logits (LT) tc_pre_kernel and
// tc_post_kernel read a row as two 8-byte loads per lane and tc_post_kernel stores the gradient as two 8-byte stores of
// packed 2-byte values; lanes own the same states, and the scratch (bufA, bufU, lse, fix) stays fp32.
constexpr int TC_S = 256;
constexpr int TC_ROWS = 32;      // rows of ONE sample per CTA (8 warps x 4 rows): one atomicAdd per CTA and output

struct Row8 { float v[8]; };
__device__ __forceinline__ Row8 load_row8(const float* p, int lane) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p) + lane), b = __ldg(reinterpret_cast<const float4*>(p + 128) + lane);
  return Row8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
__device__ __forceinline__ void store_row8(float* p, int lane, const float (&v)[8]) {
  reinterpret_cast<float4*>(p)[lane] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p + 128)[lane] = make_float4(v[4], v[5], v[6], v[7]);
}
template <typename LT>
__device__ __forceinline__ Row8 load_row8(const LT* p, int lane) {     // the 2-byte types
  const uint2 a = __ldg(reinterpret_cast<const uint2*>(p) + lane), b = __ldg(reinterpret_cast<const uint2*>(p + 128) + lane);
  Row8 r;
  widen2x4<LT>(a, r.v[0], r.v[1], r.v[2], r.v[3]);
  widen2x4<LT>(b, r.v[4], r.v[5], r.v[6], r.v[7]);
  return r;
}
// two values rounded to nearest even, packed (lo -> low half)
__device__ __forceinline__ uint32_t pack2(__nv_bfloat16*, float lo, float hi) {
  return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(lo)) | ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(hi)) << 16);
}
__device__ __forceinline__ uint32_t pack2(__half*, float lo, float hi) {
  return (uint32_t)__half_as_ushort(__float2half_rn(lo)) | ((uint32_t)__half_as_ushort(__float2half_rn(hi)) << 16);
}
template <typename LT>
__device__ __forceinline__ void store_row8(LT* p, int lane, const float (&v)[8]) {     // the 2-byte types
  reinterpret_cast<uint2*>(p)[lane] = make_uint2(pack2(p, v[0], v[1]), pack2(p, v[2], v[3]));
  reinterpret_cast<uint2*>(p + 128)[lane] = make_uint2(pack2(p, v[4], v[5]), pack2(p, v[6], v[7]));
}
__device__ __forceinline__ int state_of(int lane, int e) { return (e < 4 ? 0 : 128) + 4 * lane + (e & 3); }
// value of element `s` of a row held as Row8 across the warp
__device__ __forceinline__ float row_elem(const float (&v)[8], int s, int lane) {
  const int e = ((s >> 7) << 2) | (s & 3), src = (s & 127) >> 2;
  float x = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) x = (k == e) ? v[k] : x;
  return __shfl_sync(0xffffffffu, x, src);
}
// sum over the CTA's warps of up to 5 per-warp values, then one atomicAdd each (thread 0)
__device__ __forceinline__ void block_accumulate(float (&acc)[5], float* const (&dst)[5], int n) {
  __shared__ float s_part[8][5];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
    for (int k = 0; k < n; ++k) s_part[warp][k] = acc[k];
  __syncthreads();
  if (threadIdx.x < n) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += s_part[w][threadIdx.x];
    atomicAdd(dst[threadIdx.x], t);
  }
}

template <typename LT = float>
__global__ void __launch_bounds__(256) tc_pre_kernel(const Args a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.y;
  float nll = 0.f;
  for (int r = warp; r < TC_ROWS; r += 8) {
    const int d = blockIdx.x * TC_ROWS + r;
    if (d >= a.D) break;
    const size_t row = (size_t)b * a.D + d;
    const Row8 l = load_row8(static_cast<const LT*>(a.logits) + row * TC_S, lane);
    float m = l.v[0];
#pragma unroll
    for (int e = 1; e < 8; ++e) m = fmaxf(m, l.v[e]);
    m = warp_max(m);
    float ex[8], sum = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { ex[e] = expf(l.v[e] - m); sum += ex[e]; }
    sum = warp_sum(sum);
    const float lse = m + logf(sum), rsum = 1.f / sum;
#pragma unroll
    for (int e = 0; e < 8; ++e) ex[e] *= rsum;
    store_row8(a.bufA + row * TC_S, lane, ex);
    const float lx0 = row_elem(l.v, a.x0[row], lane);
    if (lane == 0) { a.lse[row] = lse; nll += lse - lx0; }
  }
  float acc[5] = {nll, 0.f, 0.f, 0.f, 0.f};
  float* const dst[5] = {a.out_nll + b, nullptr, nullptr, nullptr, nullptr};
  block_accumulate(acc, dst, 1);
}

template <bool BWD>
__global__ void __launch_bounds__(256) tc_terms_kernel(const Args a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.y;
  const float* Q = a.Q + (size_t)b * TC_S * TC_S;
  const float* QT = a.QT + (size_t)b * TC_S * TC_S;
  const float beta = a.beta[b];
  const float lle = (a.logit_type == CTDD_BRANCH_SDDM_REVERSE_LOGSCALE) ? 0.f : 1e-35f;   // see loss_kernel
  const float baseZ = (a.kind != CTDD_LOSS_CRM) ? a.baseZ[b] : 0.f;
  const float ga = BWD ? a.ga[b] : 0.f, gb = BWD ? a.gb[b] : 0.f, gd = BWD ? a.gd[b] : 0.f;
  float sa = 0.f, sb = 0.f, sc = 0.f, sd = 0.f;      // per-warp sums over its rows (forward)
  for (int r = warp; r < TC_ROWS; r += 8) {
    const int d = blockIdx.x * TC_ROWS + r;
    if (d >= a.D) break;
    const size_t row = (size_t)b * a.D + d;
    const int x0 = a.x0[row], xr = a.xt[row];
    const Row8 u = load_row8(a.bufU + row * TC_S, lane);
    const float ux = row_elem(u.v, xr, lane);
    const float llx = ux + lle > 0.f ? logf(ux + lle) : -1e9f;
    float ra = 0.f, rb = 0.f, rc = 0.f, wsum = 0.f;
    float V[8];
    if (a.kind == CTDD_LOSS_SDDM) {
      const Row8 rcol = load_row8(a.RbT + (size_t)xr * TC_S, lane);       // Rb[., xr]
      const Row8 qx0 = load_row8(Q + (size_t)x0 * TC_S, lane);            // Q[x0, .]
      const Row8 zd = load_row8(a.RbD, lane);                             // Rb[s, s]
      const float inv_den = 1.f / (Q[(size_t)x0 * TC_S + xr] + a.eps);
      const float inv_ex = expf(-llx);
      const float zt = -beta * a.Rb[(size_t)xr * TC_S + xr];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int s = state_of(lane, e);
        const float uraw = u.v[e];
        const float ll = uraw + lle > 0.f ? __logf(uraw + lle) : -1e9f;
        const float rs = (s == xr) ? 0.f : beta * rcol.v[e];
        const float ev = (uraw + lle) * inv_ex;
        const float w = (s == xr) ? 0.f : rs * qx0.v[e] * inv_den;
        const float Z = baseZ - zt + (-beta * zd.v[e]);
        ra += ev * rs;
        rb += w * (ll - llx);
        rc += __fdividef(w, Z);
        wsum += w;
        const float dll = ga * ev * rs + gb * w;
        V[e] = (uraw + lle > 0.f) ? __fdividef(dll, uraw + lle) : 0.f;
      }
    } else {      // CRM
      Row8 qsx, qxs;
      if (a.crm_type == 2) { qsx = load_row8(QT + (size_t)xr * TC_S, lane); qxs = load_row8(Q + (size_t)xr * TC_S, lane); }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int s = state_of(lane, e);
        const float uraw = u.v[e];
        const float ll = uraw + lle > 0.f ? __logf(uraw + lle) : -1e9f;
        float dll = 0.f;
        if (a.crm_type == 1) {          // mle
          ra += -log1mexp_ref(ll);
          const float el = expf(ll);
          dll = (s == xr) ? 0.f : ga * el / (1.f - el);
        } else if (a.crm_type == 2) {   // elbo
          if (s != xr) {
            const float ev = expf(ll - llx);
            ra += ev * qsx.v[e] - (llx - ll) * qxs.v[e];
            wsum += ev * qsx.v[e] + qxs.v[e];
            dll = ga * (ev * qsx.v[e] + qxs.v[e]);
          }
        }
        V[e] = (uraw + lle > 0.f) ? __fdividef(dll, uraw + lle) : 0.f;
      }
    }
    ra = warp_sum(ra); rb = warp_sum(rb); rc = warp_sum(rc); wsum = warp_sum(wsum);
    float dllx;
    if (a.kind == CTDD_LOSS_SDDM) {
      dllx = -ga * ra - gb * wsum;
    } else {
      if (a.crm_type == 0) { ra = -llx; dllx = -ga; }
      else if (a.crm_type == 1) { ra = -((float)(TC_S - 1) * llx) + ra + log1mexp_ref(llx); dllx = -ga * (float)(TC_S - 1); }
      else { dllx = -ga * wsum; }
    }
    dllx -= gd;
    if (BWD) {
      // The cotangent at the evaluation state also receives d/d ll_x (u_x + lle = exp(ll_x)).  That one-hot part is kept
      // OUT of the tensor-core product: it is the large, cancelling term of the softmax Jacobian, and its contribution
      // dp[k] += fix * Q[k][x] is one exact fp32 row gather in tc_post_kernel instead of a 3 x BF16 product.
      if (lane == 0) a.fix[row] = dllx / expf(llx);
      store_row8(a.bufA + row * TC_S, lane, V);
    } else {
      sa += ra; sb += rb; sc += rc; sd += -llx;
    }
  }
  if (!BWD) {
    float acc[5] = {sa, sb, sc, sd, 0.f};
    float* const dst[5] = {a.out_a + b, a.out_b + b, a.out_c + b, a.out_d + b, nullptr};
    block_accumulate(acc, dst, 4);
  }
}

template <typename LT = float>
__global__ void __launch_bounds__(256) tc_post_kernel(const Args a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.y;
  const float gn = a.gn[b];
  for (int r = warp; r < TC_ROWS; r += 8) {
    const int d = blockIdx.x * TC_ROWS + r;
    if (d >= a.D) break;
    const size_t row = (size_t)b * a.D + d;
    const Row8 l = load_row8(static_cast<const LT*>(a.logits) + row * TC_S, lane);
    Row8 dp = load_row8(a.bufU + row * TC_S, lane);
    const float lse = a.lse[row], fix = a.fix[row];
    const int x0 = a.x0[row];
    const Row8 qx = load_row8(a.QT + ((size_t)b * TC_S + a.xt[row]) * TC_S, lane);     // Q[k][x] over k
    float p[8], dot = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      dp.v[e] = fmaf(fix, qx.v[e], dp.v[e]);
      p[e] = expf(l.v[e] - lse);
      dot += p[e] * dp.v[e];
    }
    dot = warp_sum(dot);
    float g[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) g[e] = p[e] * (dp.v[e] - dot) + gn * (p[e] - (state_of(lane, e) == x0 ? 1.f : 0.f));
    store_row8(static_cast<LT*>(a.grad) + row * TC_S, lane, g);
  }
}

}  // namespace loss
}  // namespace ctdd

namespace {
template <typename LT>
void reserve_loss_smem() {
  using ctdd::loss::loss_kernel;
  cudaFuncSetAttribute(loss_kernel<false, 8, LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(loss_kernel<true, 8, LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(loss_kernel<false, 32, LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(loss_kernel<true, 32, LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
}

template <typename LT>
void launch_loss_kernel(const ctdd::loss::Args& a, bool bwd, int ROWS, dim3 grid, int threads, size_t smem, cudaStream_t st) {
  using ctdd::loss::loss_kernel;
  if (ROWS == 32) {
    if (bwd) loss_kernel<true, 32, LT><<<grid, threads, smem, st>>>(a);
    else loss_kernel<false, 32, LT><<<grid, threads, smem, st>>>(a);
  } else {
    if (bwd) loss_kernel<true, 8, LT><<<grid, threads, smem, st>>>(a);
    else loss_kernel<false, 8, LT><<<grid, threads, smem, st>>>(a);
  }
}

int run_loss(const ctdd_loss_params* p, void* stream, bool bwd) {
  using namespace ctdd;
  using namespace ctdd::loss;
  if (!p) { set_error("ctdd_loss: null params"); return 2; }
  if (p->B <= 0 || p->D <= 0 || p->S < 2) { set_error("ctdd_loss: bad sizes"); return 2; }
  if (p->kind < CTDD_LOSS_CTELBO || p->kind > CTDD_LOSS_SDDM) { set_error("ctdd_loss: unknown kind %d", p->kind); return 2; }
  if (p->logits_dtype != CTDD_DTYPE_F32 && p->logits_dtype != CTDD_DTYPE_BF16 && p->logits_dtype != CTDD_DTYPE_F16) {
    set_error("ctdd_loss: unknown logits_dtype %d (CTDD_DTYPE_F32 = 0, CTDD_DTYPE_BF16 = 1, CTDD_DTYPE_F16 = 2)", p->logits_dtype);
    return 2;
  }
  if (!p->logits || !p->Q || !p->QT || !p->Rb || !p->beta || !p->x0 || !p->xt) { set_error("ctdd_loss: null input"); return 2; }
  if (p->kind != CTDD_LOSS_CTELBO && !(p->logit_type == CTDD_BRANCH_SDDM_DIRECT || p->logit_type == CTDD_BRANCH_SDDM_REVERSE_PROB ||
                                       p->logit_type == CTDD_BRANCH_SDDM_REVERSE_LOGSCALE)) {
    set_error("ctdd_loss: unknown logit_type %d", p->logit_type);
    return 3;
  }
  if (p->kind == CTDD_LOSS_CTELBO && !p->x_tilde) { set_error("ctdd_loss: x_tilde required"); return 2; }
  if (bwd && (!p->ga || !p->gb || !p->gd || !p->gn || !p->grad_logits)) { set_error("ctdd_loss_backward: null gradient pointer"); return 2; }
  if (!bwd && (!p->out_a || !p->out_b || !p->out_c || !p->out_d || !p->out_nll)) { set_error("ctdd_loss_forward: null output pointer"); return 2; }
  // S == 256, SDDM / CRM kinds with a scratch buffer: the tensor-core path (below).  Its streaming kernels read the logits
  // and write the gradient in 16-byte (fp32) / 8-byte (bf16, fp16) pieces per lane: both must be 16-byte aligned.
  const int dt = p->logits_dtype;
  const bool tc_path = p->S == 256 && p->tc_scratch && p->kind != CTDD_LOSS_CTELBO && p->logit_type != CTDD_BRANCH_SDDM_DIRECT;
  if (tc_path && ((reinterpret_cast<uintptr_t>(p->logits) | (bwd ? reinterpret_cast<uintptr_t>(p->grad_logits) : 0)) & 15)) {
    set_error("ctdd_loss: logits and grad_logits must be 16-byte aligned on the tensor-core path (S = 256, tc_scratch)");
    return 2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int S = p->S;
  const int ROWS = (S == 256) ? 32 : 8;
  const size_t smem = (size_t)3 * ROWS * S * sizeof(float);
  if (smem > 200 * 1024) { set_error("ctdd_loss: S=%d too large", S); return 2; }
  static unsigned long long attr_done = 0ull;   // function attributes live in the device's context: a bit per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !((attr_done >> dev) & 1ull)) {
    reserve_loss_smem<float>();
    reserve_loss_smem<__nv_bfloat16>();
    reserve_loss_smem<__half>();
    if (dev >= 0 && dev < 64) attr_done |= 1ull << dev;
  }
  Args a;
  a.kind = p->kind; a.logit_type = p->logit_type; a.crm_type = p->crm_type; a.B = p->B; a.D = p->D; a.S = S;
  a.logits = p->logits; a.Q = p->Q; a.QT = p->QT; a.Rb = p->Rb; a.beta = p->beta;
  a.x0 = p->x0; a.xt = p->xt; a.x_tilde = p->x_tilde; a.eps = p->eps;
  // workspace: [G: B*S*S, CTELBO only][baseZ: B, padded to a multiple of 4][RbT: S*S][RbD: S]
  a.G = reinterpret_cast<const float*>(p->workspace);
  a.baseZ = p->workspace ? reinterpret_cast<const float*>(p->workspace) + (p->kind == CTDD_LOSS_CTELBO ? (size_t)p->B * S * S : 0) : nullptr;
  a.RbT = (a.baseZ && p->kind != CTDD_LOSS_CRM) ? a.baseZ + ((p->B + 3) & ~3) : nullptr;   // 16-byte aligned rows
  a.RbD = a.RbT ? a.RbT + (size_t)S * S : nullptr;
  a.out_a = p->out_a; a.out_b = p->out_b; a.out_c = p->out_c; a.out_d = p->out_d; a.out_nll = p->out_nll;
  a.ga = p->ga; a.gb = p->gb; a.gd = p->gd; a.gn = p->gn; a.grad = p->grad_logits;
  if (p->kind != CTDD_LOSS_CRM) {
    if (!p->workspace) { set_error("ctdd_loss: workspace required (ctdd_loss_workspace_bytes)"); return 2; }
    if (!bwd) {  // tables are built by the forward call and reused by the backward call (same workspace)
      if (p->kind == CTDD_LOSS_CTELBO) {
        const int tiles = (S + 63) / 64;
        dim3 grid(tiles, tiles, p->B), block(256);
        ctelbo_table_kernel<<<grid, block, 0, st>>>(p->QT, p->Rb, p->beta, S, p->eps, const_cast<float*>(a.G));
        CTDD_CHECK_LAUNCH("ctelbo_table_kernel");
      }
      const int rt = (S + 15) / 16;
      rb_tables_kernel<<<dim3(rt, rt), 256, 0, st>>>(p->Rb, S, const_cast<float*>(a.RbT), const_cast<float*>(a.RbD));
      CTDD_CHECK_LAUNCH("rb_tables_kernel");
      basez_kernel<<<p->B, 256, 0, st>>>(p->Rb, p->beta, p->x_tilde ? p->x_tilde : p->xt, p->D, S, const_cast<float*>(a.baseZ));
      CTDD_CHECK_LAUNCH("basez_kernel");
    }
  }
  // S == 256, SDDM / CRM kinds with a scratch buffer: the two contractions run on tcgen05 (ctdd_bgemm256_tc) between three
  // streaming kernels.  u = p Q and the rows' log-sum-exp are kept in the scratch from the forward to the backward call.
  // (CT-ELBO stays on the fp32 CUDA-core contraction: its operand p / (Q[k,x~] + eps) spans 9 decades and the softmax
  // Jacobian cancels to ~1e-4 of its terms, which takes the 3 x BF16 product error past the gradient parity bar.)
  if (tc_path) {
    if (reinterpret_cast<uintptr_t>(p->tc_scratch) & 15) { set_error("ctdd_loss: tc_scratch must be 16-byte aligned"); return 2; }
    const size_t n = (size_t)p->B * p->D * S;
    a.bufA = reinterpret_cast<float*>(p->tc_scratch);
    a.bufU = a.bufA + n;
    a.lse = a.bufU + n;
    a.fix = a.lse + (size_t)p->B * p->D;
    dim3 tgrid((p->D + TC_ROWS - 1) / TC_ROWS, p->B);
    if (!bwd) {
      if (dt == CTDD_DTYPE_BF16) tc_pre_kernel<__nv_bfloat16><<<tgrid, 256, 0, st>>>(a);
      else if (dt == CTDD_DTYPE_F16) tc_pre_kernel<__half><<<tgrid, 256, 0, st>>>(a);
      else tc_pre_kernel<<<tgrid, 256, 0, st>>>(a);
      CTDD_CHECK_LAUNCH("tc_pre_kernel");
      if (int rc = ctdd_bgemm256_tc(a.bufA, p->QT, p->B, p->D, a.bufU, stream)) return rc;      // u[s] = sum_k p[k] Q[k][s]
      tc_terms_kernel<false><<<tgrid, 256, 0, st>>>(a);
      CTDD_CHECK_LAUNCH("tc_terms_kernel");
    } else {
      tc_terms_kernel<true><<<tgrid, 256, 0, st>>>(a);
      CTDD_CHECK_LAUNCH("tc_terms_kernel<bwd>");
      if (p->kind == CTDD_LOSS_CRM && p->crm_type == 0) {      // ratio matching 'rm': the cotangent is the one-hot part only
        cudaMemsetAsync(a.bufU, 0, n * sizeof(float), st);
      } else {
        if (int rc = ctdd_bgemm256_tc(a.bufA, p->Q, p->B, p->D, a.bufU, stream)) return rc;     // dp[k] = sum_s V[s] Q[k][s]
      }
      if (dt == CTDD_DTYPE_BF16) tc_post_kernel<__nv_bfloat16><<<tgrid, 256, 0, st>>>(a);
      else if (dt == CTDD_DTYPE_F16) tc_post_kernel<__half><<<tgrid, 256, 0, st>>>(a);
      else tc_post_kernel<<<tgrid, 256, 0, st>>>(a);
      CTDD_CHECK_LAUNCH("tc_post_kernel");
    }
    return 0;
  }
  a.bufA = a.bufU = a.lse = a.fix = nullptr;
  int threads = ((S + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  if (threads < 64) threads = 64;
  dim3 grid((p->D + ROWS - 1) / ROWS, p->B);
  if (dt == CTDD_DTYPE_BF16) launch_loss_kernel<__nv_bfloat16>(a, bwd, ROWS, grid, threads, smem, st);
  else if (dt == CTDD_DTYPE_F16) launch_loss_kernel<__half>(a, bwd, ROWS, grid, threads, smem, st);
  else launch_loss_kernel<float>(a, bwd, ROWS, grid, threads, smem, st);
  CTDD_CHECK_LAUNCH("loss_kernel");
  return 0;
}
}  // namespace

extern "C" int64_t ctdd_loss_workspace_bytes(int kind, int B, int S) {
  const int64_t Bp = (B + 3) & ~3;
  if (kind == CTDD_LOSS_CTELBO) return ((int64_t)B * S * S + Bp + (int64_t)S * S + S) * 4;
  if (kind == CTDD_LOSS_SDDM) return (Bp + (int64_t)S * S + S) * 4;
  return 0;
}
extern "C" int64_t ctdd_loss_tc_scratch_bytes(int B, int D, int S) {
  return S == 256 ? ((int64_t)2 * B * D * S + (int64_t)2 * B * D + 4) * 4 : 0;
}
extern "C" int ctdd_loss_forward(const ctdd_loss_params* p, void* stream) { return run_loss(p, stream, false); }
extern "C" int ctdd_loss_backward(const ctdd_loss_params* p, void* stream) { return run_loss(p, stream, true); }

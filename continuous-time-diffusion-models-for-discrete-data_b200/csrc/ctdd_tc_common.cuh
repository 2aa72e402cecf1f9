// Shared pieces of the three tcgen05 kernels: the reverse-step kernels (ctdd_step_tc.cu: Euler modes, ctdd_step_tcq.cu:
// every other mode) and the per-sample contraction of the losses (ctdd_bgemm_tc.cu).  Table-blob layout and kernel
// arguments of the step kernels, PTX wrappers (mbarrier, tcgen05, bulk copies, packed fp32 pairs), the bf16 hi/mid split,
// the CTA-pair plumbing all three share (operand rows, MMA issue, relay, teardown, launch geometry) and the softmax
// numerators of the truncated-logistic head.
#pragma once
#include "ctdd_common.cuh"
#include <cuda_bf16.h>

namespace ctdd {
namespace tc {

constexpr int S = 256;
constexpr int TMEM_COLS = 512;
constexpr int TM_QH = 0, TM_QM = 128, TM_ACC = 256;  // TMEM column map: A operand hi / mid, accumulator b at TM_ACC + b * NT

// per-time-point table blob (ctdd_prep_tc_tables)
constexpr size_t TAB_QH_OFF = 0;                                 // uint32 [256][128]  bf16 pairs of Q^T hi
constexpr size_t TAB_QM_OFF = TAB_QH_OFF + (size_t)S * 128 * 4;  // uint32 [256][128]  bf16 pairs of Q^T mid
constexpr size_t TAB_A_OFF = TAB_QM_OFF + (size_t)S * 128 * 4;   // float [x][k]  tauLDR: 1/(Q[k,x]+eps); SDDM: Q[k,x]
constexpr size_t TAB_BYTES = TAB_A_OFF + (size_t)S * S * 4;
// static blob (ctdd_prep_tc_static); the caller places it on a ST_ALIGN boundary, so that "blob + offset" never carries
// into the upper address word (the epilogue adds 32-bit offsets to a constant upper word)
constexpr size_t ST_ALIGN = (size_t)2 << 20;
constexpr size_t ST_RBZT_OFF = 0;                                // float [x][s] = Rb[s][x], zero at s == x
constexpr size_t ST_RBZ_OFF = (size_t)S * S * 4;                 // float [x][s] = Rb[x][s], zero at s == x
constexpr size_t ST_RBT_OFF = 2 * (size_t)S * S * 4;             // float [x][s] = Rb[s][x], diagonal kept (rates output)
constexpr size_t ST_RB_OFF = 3 * (size_t)S * S * 4;              // float [x][s] = Rb[x][s], diagonal kept
constexpr size_t ST_ZERO_OFF = 4 * (size_t)S * S * 4;            // float [S] zeros: the "row" read for chunks outside the band
constexpr size_t ST_BANDT_OFF = ST_ZERO_OFF + (size_t)S * 4;     // int [x] = lo | hi << 8: first / last s with Rbzt[x][s] != 0
constexpr size_t ST_BANDR_OFF = ST_BANDT_OFF + (size_t)S * 4;    // int [x], same for Rbz[x][s]   (empty: lo = 255, hi = 0)
constexpr size_t ST_BYTES = ST_BANDR_OFF + (size_t)S * 4;
static_assert(ST_BYTES <= ST_ALIGN, "static blob larger than its alignment");

// step_q_kernel modes (the Euler modes run on step_tc_kernel); the corrector variant adds h * R_t[x,:] to the rates
enum { KM_JUMP = 0, KM_CORR = 1, KM_RATES = 2, KM_DRIFT = 3 };
__host__ __device__ constexpr bool km_corr(int km) { return km == KM_CORR; }

struct Args {
  int branch, D, reject_multi;
  long long rows, row_offset;
  const void* logits;        // fp32 or bf16 (the kernel's logits-type template argument)
  long long ld, batch_stride;
  const int* x_eval;
  const int* x_base;
  const uint8_t* tab;     // per-time-point blob
  const uint8_t* stat;    // static blob
  float beta, h;
  unsigned long long seed, offset;
  int* x_out;
  float* rr_out;
  float* ratio_out;
  unsigned long long* stats;
  int num_tiles;
  int head_fix;              // fused truncated-logistic head (HEAD kernels): fix_logistic
  const void* head_mu;       // fp32 or bf16 (HEAD kernels: the logits-type template argument names the head's type)
  const void* head_ls;
  long long head_bs;         // elements between consecutive n
};

// the kernel arguments of a step; num_tiles depends on the kernel's tile size and is left to the launcher
inline Args make_args(const ctdd_step_params* p) {
  Args a;
  a.branch = p->branch; a.D = p->D; a.reject_multi = p->reject_multi;
  a.rows = (long long)p->N * p->D; a.row_offset = p->row_offset;
  a.logits = p->logits; a.ld = p->ld_logits; a.batch_stride = p->batch_stride_logits;
  a.x_eval = p->x_eval; a.x_base = p->x_base;
  a.tab = reinterpret_cast<const uint8_t*>(p->tc_tables);
  a.stat = reinterpret_cast<const uint8_t*>(p->tc_static);
  a.beta = p->beta; a.h = p->h; a.seed = p->seed; a.offset = p->offset;
  a.x_out = p->x_out; a.rr_out = p->rr_out; a.ratio_out = p->ratio_out;
  a.stats = reinterpret_cast<unsigned long long*>(p->stats_out);
  a.head_fix = p->head == CTDD_HEAD_LOGISTIC_FIX;
  a.head_mu = p->head_mu; a.head_ls = p->head_log_scale; a.head_bs = p->head_batch_stride;
  a.num_tiles = 0;
  return a;
}

// ---------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory object in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on a barrier addressed in the cluster window (own or partner CTA). RELEASE: the arriving thread's earlier
// writes (and, through __syncwarp, its warp's) are visible to whoever acquires the phase; RELAXED: pure signalling
// (tensor-memory reads already fenced with tcgen05.fence, or buffers whose values were consumed before the arrive).
__device__ __forceinline__ void mbar_arrive_cluster_release(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// wait for a phase: one try_wait (which suspends in hardware for a short, implementation-defined time), then a
// sleep / try_wait loop - a warp that has to wait longer must not eat issue slots of the warps it is waiting for.
// SLEEP_NS: pause between polls; roles whose waits are long (a whole tile) and whose wake-up is not on the critical path
// use a longer one.
constexpr uint32_t POLL_NS = 96;
template <uint32_t SLEEP_NS = POLL_NS>
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra DONE_%=;\n"
      "WAIT_%=:\n"
      "nanosleep.u32 %3;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@!p bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"(0x989680u), "r"(SLEEP_NS)
      : "memory");
}
// same, for phases completed by arrivals from the partner CTA: acquire at cluster scope once the phase has flipped
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  mbar_wait(bar, parity);
  // the phase has flipped: one test_wait with acquire semantics at CLUSTER scope (it succeeds at once) orders this
  // thread after the partner's release-arrive - cheaper than a stand-alone fence.acq_rel.cluster
  asm volatile(
      "{\n.reg .pred p;\n"
      "mbarrier.test_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"((uint32_t)TMEM_COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"((uint32_t)TMEM_COLS) : "memory");
}
// signal the barrier at this smem offset in BOTH CTAs of the pair when all prior MMAs of this thread have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc] over the CTA pair (kind::f16, bf16 inputs, fp32 accumulate); the descriptor
// is passed as two 32-bit halves so that the 48 per-tile variants are one 32-bit add each
__device__ __forceinline__ void umma_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint32_t bdesc_lo, uint32_t bdesc_hi, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 bd;\n"
      "mov.b64 bd, {%2, %3};\n"
      "setp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], bd, %4, p;\n"
      "}\n" ::"r"(d_tmem), "r"(a_tmem), "r"(bdesc_lo), "r"(bdesc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major, SWIZZLE_128B operand descriptor: LBO = 1 (unused), SBO = 1024 B (8 rows x 128 B), version 1
__device__ __forceinline__ uint64_t make_b_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// instruction descriptor: fp32 accumulate, bf16 A and B, K-major both, N = n, M = 256 (CTA pair)
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float4 ld_stream(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// 32 bytes of read-only table data per lane in one request (one sector; the address must be 32-byte aligned)
__device__ __forceinline__ void ldg256(const uint8_t* p, float* v) {
  asm("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
      : "l"(p));
}
// the same when `on`, eight zeros otherwise
__device__ __forceinline__ void ldg256_pred(const uint8_t* p, float* v, bool on) {
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = 0.f;
  asm("{\n.reg .pred q;\nsetp.ne.u32 q, %9, 0;\n@q ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n}\n"
      : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7])
      : "l"(p), "r"((uint32_t)on));
}
// explicit shared-space accesses (the compiler emits generic LD/ST for pointers it cannot prove to be shared)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// remote store that reports its bytes to an mbarrier of the destination CTA when it has landed (no fence needed)
__device__ __forceinline__ void st_async_cluster_f32(uint32_t cluster_addr, float v, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(cluster_addr),
               "r"(__float_as_uint(v)), "r"(cluster_mbar)
               : "memory");
}
__device__ __forceinline__ void st_async_cluster_b32(uint32_t cluster_addr, uint32_t v, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(cluster_addr), "r"(v),
               "r"(cluster_mbar)
               : "memory");
}
__device__ __forceinline__ void st_async_cluster_v2(uint32_t cluster_addr, uint32_t v0, uint32_t v1, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];" ::"r"(cluster_addr),
               "r"(v0), "r"(v1), "r"(cluster_mbar)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void l2_prefetch_bulk(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// bulk copy global -> this CTA's shared memory; the bytes are reported to `bar` (expect_tx armed by the caller)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// bulk copy this CTA's shared memory -> shared memory of a CTA of the cluster; bytes reported to an mbarrier there
__device__ __forceinline__ void bulk_s2cluster(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t mbar_cluster) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_cluster),
               "r"(src_cta), "r"(bytes), "r"(mbar_cluster)
               : "memory");
}
// non-blocking phase test
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(ok)
               : "r"(smem_u32(bar)), "r"(parity)
               : "memory");
  return ok != 0;
}

// packed fp32 pairs (Blackwell: one issue slot for two lanes of an FMA / ADD / MUL / SUB)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rc, rd;\nmov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nmov.b64 rc, {%6, %7};\n"
      "fma.rn.f32x2 rd, ra, rb, rc;\nmov.b64 {%0, %1}, rd;\n}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rd;\nmov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nadd.rn.f32x2 rd, ra, rb;\nmov.b64 {%0, %1}, rd;\n}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rd;\nmov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nsub.rn.f32x2 rd, ra, rb;\nmov.b64 {%0, %1}, rd;\n}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rd;\nmov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nmul.rn.f32x2 rd, ra, rb;\nmov.b64 {%0, %1}, rd;\n}\n"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

// bf16 hi/mid split of two floats, packed (element 0 in the low half)
__device__ __forceinline__ void split2(float a0, float a1, uint32_t& hi, uint32_t& mid) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a0, a1);
  hi = *reinterpret_cast<uint32_t*>(&h);
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 1000
  const float2 r = fsub2(make_float2(a0, a1), make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xFFFF0000u)));
  __nv_bfloat162 m = __floats2bfloat162_rn(r.x, r.y);
#else
  const float r0 = a0 - __uint_as_float(hi << 16);
  const float r1 = a1 - __uint_as_float(hi & 0xFFFF0000u);
  __nv_bfloat162 m = __floats2bfloat162_rn(r0, r1);
#endif
  mid = *reinterpret_cast<uint32_t*>(&m);
}

// ---------------------------------------------------------------------------------------------- CTA-pair plumbing
// Each kernel runs on CTA pairs (cluster of 2, cta_group::2).  The A operand, one CTA's 128-row half of a 256 x 256 matrix
// split into bf16 hi and mid, stays in tensor memory at TM_QH / TM_QM.  The B operand is a smem stage of the CTA's rows
// of a tile, K-major and 128B-swizzled: the hi split, then the mid split (SPLIT_BYTES each), each 4 K blocks of
// KBLOCK_BYTES = rows x 128 B.

// One operand row of a producer half-warp: lane l16 holds k = 64c + 4*l16 .. +3 (c = 0..3) of row r, which lives in
// K block c, 16-byte chunk l16/2 (XOR-swizzled by the row), half l16&1 (the layout make_b_desc describes).
template <int KBLOCK_BYTES, int SPLIT_BYTES>
__device__ __forceinline__ void store_operand_row(uint32_t stage, int r, int l16, const float (&v)[16]) {
  const uint32_t off = (uint32_t)r * 128 + (uint32_t)((((l16 >> 1) ^ (r & 7)) << 4) | ((l16 & 1) << 3));
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t h0, m0, h1, m1;
    split2(v[4 * c], v[4 * c + 1], h0, m0);
    split2(v[4 * c + 2], v[4 * c + 3], h1, m1);
    sts64(stage + c * KBLOCK_BYTES + off, h0, h1);
    sts64(stage + SPLIT_BYTES + c * KBLOCK_BYTES + off, m0, m1);
  }
}

// The 48 tcgen05.mma of one tile: 3 passes Qh*ah + Qh*am + Qm*ah of 16 K steps into the accumulator at d_tmem.  One
// descriptor per tile; the 48 instructions differ only by compile-time offsets (16-byte units, low word).
template <int KBLOCK_BYTES, int SPLIT_BYTES, uint32_t IDESC>
__device__ __forceinline__ void issue_tile(uint32_t tmem, uint32_t d_tmem, uint32_t stage) {
  const uint64_t bd0 = make_b_desc(stage);
  const uint32_t bd_lo = (uint32_t)bd0, bd_hi = (uint32_t)(bd0 >> 32);
#pragma unroll 1
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t a_tmem = tmem + (pass == 2 ? TM_QM : TM_QH);
    const uint32_t lo = bd_lo + (pass == 1 ? (uint32_t)(SPLIT_BYTES >> 4) : 0u);
#pragma unroll
    for (int k16 = 0; k16 < 16; ++k16) {
      const uint32_t boff = (uint32_t)((k16 >> 2) * KBLOCK_BYTES + (k16 & 3) * 32) >> 4;
      umma_ts_pair(d_tmem, a_tmem + k16 * 8, lo + boff, bd_hi, IDESC, (pass | k16) ? 1u : 0u);
    }
  }
}

// Partner CTA: relay "my producer warps have filled stage st" (full_local) to the leader's full barrier as ONE
// cluster-scope arrival per tile (this thread has no memory traffic of its own, so its release costs nothing).
template <int STAGES, uint32_t SLEEP_NS>
__device__ __forceinline__ void relay_full(uint64_t* full_local, uint64_t* full, int my_tiles) {
  const uint32_t full_addr = mapa(smem_u32(full), 0);
  for (int i = 0; i < my_tiles; ++i) {
    const int st = i % STAGES;
    mbar_wait<SLEEP_NS>(&full_local[st], (i / STAGES) & 1);
    mbar_arrive_cluster_release(full_addr + (uint32_t)st * 8u);
  }
}

// The step kernels' A operand: this CTA's 128-state half of Q^T (bf16 hi + mid pairs of the table blob) -> tensor
// memory, loaded by warps 0 .. LOAD_WARPS - 1 (a multiple of 4).  A warp reaches the TMEM lanes [32q, 32q+32) of its
// quadrant q = warp & 3; the quadrant's 8 pieces of 32 columns (4 per bf16 split) are dealt to the loading warps of that
// quadrant.  step_q_kernel lets all its warps load, so that the whole 128 KB is requested at once.  step_tc_kernel keeps
// its four loading warps (each loads its quadrant's 8 pieces): dealt to all 20 of its warps, its Euler step at the C4
// shape (tools/kernel_zoo.py) took 1.747-1.750 ms instead of 1.724-1.736 ms (three alternated runs each, one B200 with
// a 1000 W power limit).
template <int LOAD_WARPS>
__device__ __forceinline__ void load_qt_half(const uint8_t* tab, uint32_t tmem, uint32_t rank, int warp, int lane) {
  const int q = warp & 3;
  const int srow = (int)rank * 128 + q * 32 + lane;
  constexpr int WPQ = LOAD_WARPS / 4;              // loading warps per quadrant
#pragma unroll 1
  for (int piece = warp >> 2; piece < 8; piece += WPQ) {
    const int split = piece >> 2, c = (piece & 3) * 32;
    const uint4* src = reinterpret_cast<const uint4*>(tab + (split ? TAB_QM_OFF : TAB_QH_OFF)) + (size_t)srow * 32;
    uint32_t r[32];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint4 v = __ldg(src + (c >> 2) + i);
      r[4 * i] = v.x; r[4 * i + 1] = v.y; r[4 * i + 2] = v.z; r[4 * i + 3] = v.w;
    }
    tmem_st32(tmem + ((uint32_t)(q * 32) << 16) + (split ? TM_QM : TM_QH) + c, r);
  }
  tmem_st_wait();
}

// End of a pair kernel: no CTA of the pair may exit (or free tensor memory) while the other can still reach it.
// `alloc_warp`: the warp that allocated the tensor memory frees it.
__device__ __forceinline__ void pair_teardown(bool alloc_warp, uint32_t tmem) {
  tc_fence_before();
  cluster_sync_all();
  if (alloc_warp) {
    tc_fence_after();
    tmem_dealloc(tmem);
  }
}

// Host side of a pair-kernel launcher.  Function attributes live in the device's context, so each launcher reserves its
// kernels' dynamic shared memory once per device ordinal (a bit of `attr_done`) and reads the SM count then.
struct PairLaunchState {
  int num_sms[64] = {0};
  unsigned long long attr_done = 0ull;
};
// Makes that reservation for every kernel of `kerns` on the current device if it has not been made, and returns the number
// of CTA pairs of the grid for num_tiles tiles: one pair per TPC, at most one per tile, at least one.  Returns 0 with the
// error set (in the name of `who`) when the reservation fails.
template <typename Kernel, size_t N>
inline int pair_count(PairLaunchState& ls, const char* who, const Kernel (&kerns)[N], size_t smem_bytes, long long num_tiles) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!(dev >= 0 && dev < 64 && ((ls.attr_done >> dev) & 1ull))) {
    cudaDeviceGetAttribute(&ls.num_sms[dev & 63], cudaDevAttrMultiProcessorCount, dev);
    for (size_t i = 0; i < N; ++i)
      if (cudaFuncSetAttribute(kerns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes) != cudaSuccess) {
        set_error("%s: cannot reserve %zu bytes of shared memory for the tcgen05 kernel", who, smem_bytes);
        cudaGetLastError();
        return 0;
      }
    if (dev >= 0 && dev < 64) ls.attr_done |= 1ull << dev;
  }
  long long pairs = ls.num_sms[dev & 63] / 2;
  if (pairs > num_tiles) pairs = num_tiles;
  return pairs < 1 ? 1 : (int)pairs;
}

__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Softmax numerators of the truncated-logistic head (reference lib/models/models.py:28-74, :248-282) for the 16 states
// k = 64c + 4*l16 .. +3 (c = 0..3) of one row.  With z_j = (edge_j - mu) * exp(2 - log_scale), u = sigmoid(z),
// v = sigmoid(-z) and kappa = 1 - exp(-(z_{j+1} - z_j)):   exp(logits_1[s]) = u_{s+1} * (kappa * v_s + 1e-6)  and the
// fix_logistic variant exp(min(logits_1, logits_2)[s]) = kappa * u_{s+1} * v_s + 1e-6 * min(u_{s+1}, v_s)  (identities,
// not approximations; no cancellation, unlike the 1 - exp(.) of the reference's log_minus_exp).  Rows whose edges all lie
// on one side of mu (|mu| > 1: outside what tanh emits, but legal input) are rescaled by exp(+-c) so that the numerators
// cannot all underflow; softmax is invariant to the common factor.
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// The part of it that depends on the row only (8 floats): made once per row - by the loader warp in ctdd_step_tcq.cu, by
// every lane in ctdd_step_tc.cu.
struct HeadRec { float mu, sc, off0, kap, A, B, c, pad; };
__device__ __forceinline__ HeadRec head_row_record(float mu, float ls, bool fix) {
  constexpr float L2E = 1.4426950408889634f, BW = 2.0f / S;
  const float inv = expf(2.0f - ls);
  HeadRec h;
  h.mu = mu;
  h.kap = -expm1f(-inv * BW);
  const float z_first = (-1.0f - mu) * inv, z_last = (1.0f - mu) * inv;
  float c = 0.f;
  if (z_last < 0.f) c = -z_last; else if (fix && z_first > 0.f) c = -z_first;
  h.c = c;
  h.A = c > 0.f ? expf(-c) : 1.0f;
  h.B = c < 0.f ? expf(c) : 1.0f;
  h.sc = -inv * L2E;             // exponent (base 2) of e_j = exp(-z_j - c) for edge j = 64c + 4*l16 + k:  t_c * sc + off[k]
  h.off0 = -c * L2E;
  h.pad = 0.f;
  return h;
}
__device__ __forceinline__ void head_numerators_rec(const HeadRec& h, bool fix, int l16, float (&P)[16]) {
  constexpr float BW = 2.0f / S, EPS = 1e-6f;
  const float sc = h.sc, A = h.A, B = h.B, kap = h.kap, c = h.c;
  float off[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) off[k] = fmaf((float)k * BW, sc, h.off0);
  // select of the 1e-6 term:  no fix / c > 0 -> u,  fix and c == 0 -> min(u, v),  fix and c < 0 -> v
  const float bu = (fix && c < 0.f) ? 3.0e38f : 0.f;
  const float bv = (!fix || c > 0.f) ? 3.0e38f : 0.f;
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    const float t = (fmaf((float)(64 * cc + 4 * l16), BW, -1.0f)) - h.mu;       // edge - mu (the edge is exact in fp32)
    float u[5], vv[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const float e = ex2_approx(fminf(fmaf(t, sc, off[k]), 126.0f));
      u[k] = rcp_approx(fmaf(B, e, A));
      vv[k] = e * u[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (fix) {
        const float m = fminf(fmaxf(u[k + 1], bu), fmaxf(vv[k], bv));
        P[4 * cc + k] = fmaf(kap * u[k + 1], vv[k], EPS * m);
      } else {
        P[4 * cc + k] = u[k + 1] * fmaf(kap, vv[k], EPS);
      }
    }
  }
}
__device__ __forceinline__ void head_numerators(float mu, float ls, bool fix, int l16, float (&P)[16]) {
  head_numerators_rec(head_row_record(mu, ls, fix), fix, l16, P);
}

}  // namespace tc
}  // namespace ctdd

// tcgen05 reverse-step kernel for S == 256, Euler modes (lib/sampling/sampling.py:278-341, with and without the
// corrector rates): the (N*D x S)(S x S) contraction of sampling.py:57 on 5th-generation tensor cores, fused with softmax,
// the q_{t|0} denominators, the forward-rate multiply and one categorical draw per row over
// {h * rate_s (s != x), max(0, 1 - h * sum)}.  That draw needs the row's total rate before its pick, so each row is
// sampled with all 256 states in one place; every other mode runs on step_q_kernel (ctdd_step_tcq.cu).
//
// One CTA PAIR (thread-block cluster of 2, tcgen05 cta_group::2) owns a sequence of 64-row tiles:
//   D[s, row] = sum_k Q^T[s, k] * a[row, k]        M = 256 states (128 per CTA), N = 64 rows, K = 256
//   * M side = state s. Each CTA keeps ITS 128-state half of Q^T (bf16 hi + mid split, 2 x 128 TMEM columns)
//     resident in tensor memory as the A operand (TS form) for the whole kernel; 4 accumulators of 64 columns.
//   * N side = data rows. Each CTA's 8 producer warps build 32 of the tile's 64 rows, two rows per pass with 16 lanes
//     per row: raw fp32 or bf16 logits arrive through a per-warp smem ring filled by cp.async.bulk (HBM -> L2 prefetch eight
//     tiles ahead), row softmax by half-warp butterflies, gathered reciprocal denominators 1/(Q[k,x]+eps), bf16 hi/mid
//     split, K-major 128B-swizzled smem stage.  Every row is produced exactly once.
//   * Count warp (lane = row): the row's Euler uniform (Philox, STREAM_ROW).
//   * 3 tensor passes  Qh*ah + Qh*am + Qm*ah  accumulate in fp32 TMEM (48 tcgen05.mma per tile).
//   * Epilogue phase A: each CTA reads its 128 states x 64 rows with tcgen05.ld and scatters them (local st.shared /
//     remote st.async with mbarrier complete_tx) into the [row][state] gather buffer of the CTA that OWNS the row, so
//     that each owner sees all 256 states of its 32 rows.  Two gather buffers: phase A of tile i+1 runs before the
//     sampling of tile i.
//   * Row sampler (the same 8 warps, one warp per row, two rows in flight): lam_s = D_s * c * Rbz[s,x], warp prefix
//     sum, the stay probability added at x, one inverse-CDF pick per row, statistics, x_out.  The side record and the
//     R_b table rows (L2 gathers) of the NEXT row pair are requested while the current pair is searched; the first
//     pair's before phase A of the next tile, which hides their latency.
//   * Producers finish the row reductions (sum e, and sum e*Q[.,x] for SDDM) and the side record of a pass in the head of
//     the NEXT pass, next to its row-maximum butterfly; only the operand rows are completed inside the pass.
//   * The MMA-issue thread acquires the partner CTA's release-arrive with ONE mbarrier.test_wait.acquire.cluster on the
//     already flipped barrier; a stand-alone fence.acq_rel.cluster there cost 0.2 ms per launch.
// Warp roles per CTA (5 warpgroups, setmaxnreg 104 / 64): 8 epilogue/sampler warps, 8 producer warps, and a light
// group with the MMA-issue warp (leader CTA issues; the partner's relays its producers' arrivals), the count warp and
// 2 idle warps.  profiles/r1_step_tc_summary.md has the measured per-role timeline.
#include "ctdd_tc_common.cuh"

namespace ctdd {
namespace tc {

constexpr int NH = 32;                 // rows produced and sampled by one CTA per tile
constexpr int NT = 2 * NH;             // rows per pair tile (= UMMA N)
constexpr int STAGES = 3;              // smem operand stages
constexpr int ACC = 4;                 // TMEM accumulator buffers (NT columns each)
constexpr int GBUF = 2;                // gather buffers: phase A of tile i+1 overlaps the sampling of tile i
constexpr int RING = 16;               // per-tile side-info ring (> STAGES + ACC + GBUF + 2)
constexpr int NUM_EPI_WARPS = 8;       // warps 0-7: TMEM quadrant w&3, column half w>>2 (= owner CTA of those rows)
constexpr int FIRST_PROD_WARP = 8;     // warps 8-15
constexpr int NUM_PROD_WARPS = 8;
constexpr int MMA_WARP = 16;           // warps 16-19 form the light warpgroup: MMA issue / relay, count warp, 2 idle
constexpr int COUNT_WARP = 17;         // draws the Euler uniforms of a tile, lane = row
constexpr int NUM_THREADS = 20 * 32;   // 640: register allocation is per 4-warp group, so 18 warps cost the same
// setmaxnreg targets: samplers + producers / the light warpgroup.  The registers handed out by .inc are the ones the
// CTA's own warps released with .dec: 16 * HEAVY + 4 * LIGHT must not exceed 20 * 96 (the launch allocation), or
// the .inc never returns.
constexpr int REGS_HEAVY = 104;
constexpr int REGS_LIGHT = 64;
constexpr int ROWS_PER_PROD = NH / NUM_PROD_WARPS;                   // 4
constexpr int ROWS_PER_SAMPLER = NH / NUM_EPI_WARPS;                 // 4
constexpr int KBLOCK_BYTES = NH * 128;         // one 64-wide K block of one split: NH rows x 128 B
constexpr int SPLIT_BYTES = 4 * KBLOCK_BYTES;  // K = 256 -> 4 blocks
constexpr int STAGE_BYTES = 2 * SPLIT_BYTES;   // hi + mid
constexpr int PREFETCH_TILES = 8;      // HBM -> L2 bulk-prefetch distance (tiles of this pair's sequence)
constexpr int LRING = 2;               // per-producer-warp ring of raw logits row pairs filled by cp.async.bulk
constexpr uint32_t IDESC = make_idesc(NT);

// per-row hand-over producer -> count warp -> sampler: rate scale, state (x < 0: row past the end), Euler uniform
struct __align__(16) Side { float c1, c0; int x; uint32_t w; };

struct Smem {
  alignas(1024) uint8_t stage[STAGES][STAGE_BYTES];
  alignas(16) float gather[GBUF][NH][S];   // [row owned by this CTA][state]: accumulator values, then prefix sums
  Side side[RING][NH];
  alignas(16) float lring[NUM_PROD_WARPS][LRING][2][S];   // raw logits rows, one pass ahead of their use (2-byte: the
                                                          // row pair packed into the first half of the slot)
  alignas(8) uint64_t full[STAGES];  // leader CTA: its 8 producer warps + 1 relayed arrival for the partner's 8
  uint64_t full_local[STAGES];       // partner CTA: its 8 producer warps; the partner's idle MMA warp relays the phase
  uint64_t empty[STAGES];            // multicast tcgen05.commit
  uint64_t pre_full[RING];           // local producers -> count warp (row scalars written)
  uint64_t side_full[RING];          // count warp -> local samplers (Euler uniforms written)
  uint64_t lring_full[NUM_PROD_WARPS][LRING];   // cp.async.bulk complete_tx of one row pair
  uint64_t tmem_full[ACC];           // multicast tcgen05.commit
  uint64_t tmem_empty[ACC];          // used in the leader CTA: 8 local + 8 remote epilogue warps
  uint64_t gather_full[GBUF];        // 4 local epilogue warps + the bytes of the partner's 4 warps (st.async complete_tx)
  uint64_t gather_free_local[GBUF];  // the 8 local sampler warps are done with this CTA's gather buffer
  uint64_t gather_free_remote[GBUF]; // the 8 sampler warps of the PARTNER are done with the partner's buffer
  uint32_t tmem_base;
};

static_assert(sizeof(Smem) + 1024 <= 232448, "shared memory budget of one CTA (227 KB) exceeded");


// First index whose inclusive prefix sum (256 floats at shared address P) exceeds T: three rounds of INDEPENDENT loads
// (7 splitters of stride 32, 7 of stride 4, 3 neighbours) instead of eight dependent binary-search steps.
__device__ __forceinline__ int prefix_search(uint32_t P, float T) {
  int c1 = 0;
#pragma unroll
  for (int m = 0; m < 7; ++m) c1 += (lds32(P + 4 * (32 * m + 31)) <= T) ? 1 : 0;
  const uint32_t P1 = P + 128 * c1;
  int c2 = 0;
#pragma unroll
  for (int n = 0; n < 7; ++n) c2 += (lds32(P1 + 4 * (4 * n + 3)) <= T) ? 1 : 0;
  const uint32_t P2 = P1 + 16 * c2;
  const int c3 = ((lds32(P2) <= T) ? 1 : 0) + ((lds32(P2 + 4) <= T) ? 1 : 0) + ((lds32(P2 + 8) <= T) ? 1 : 0);
  return 32 * c1 + 4 * c2 + c3;
}

// (mu, log_scale) of the fused head as the producers carry them: fp32, or the raw bits of a bf16 value (exact widening)
__device__ __forceinline__ float widen_head(float v) { return v; }
__device__ __forceinline__ float widen_head(unsigned short v) { return __uint_as_float((uint32_t)v << 16); }

// ---------------------------------------------------------------------------------------------- the kernel
// TAULDR: tauLDR rates (else SDDM reverse_prob); CORR: the corrector variant adds h * R_t[x,:] to the rates;
// HEAD: the rows' softmax numerators come from the truncated-logistic head (mu, log_scale per row) instead of logits;
// LT: element type of the logits, float, __nv_bfloat16 or __half (a 2-byte row pair travels packed, 2*S bytes per row,
// and is widened on the producers' shared-memory load; the arithmetic after that load is the fp32 kernel's).  A HEAD
// kernel reads no logits: LT is then the type of (mu, log_scale), float or __nv_bfloat16, widened on the producers' load
template <bool TAULDR, bool CORR, bool HEAD, typename LT = float>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) step_tc_kernel(const Args a) {
  static_assert(!(HEAD && std::is_same<LT, __half>::value), "the fused head takes fp32 or bf16 (mu, log_scale)");
  constexpr uint32_t ROW_BYTES = S * sizeof(LT);
  extern __shared__ uint8_t smem_raw[];
  // aligned by offsetting the shared array itself (not through an integer): the compiler keeps `sm` a shared-space
  // pointer, so its accesses are 32-bit LDS/STS and no 64-bit generic base stays live (that base was spilled at 96 registers)
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();       // state half owned by this CTA; rank 0 issues the MMAs
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  const int my_tiles = (a.num_tiles > pair) ? (a.num_tiles - pair + npairs - 1) / npairs : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&sm.full[i], NUM_PROD_WARPS + 1);
      mbar_init(&sm.full_local[i], NUM_PROD_WARPS);
      mbar_init(&sm.empty[i], 1);
    }
    for (int i = 0; i < RING; ++i) { mbar_init(&sm.pre_full[i], NUM_PROD_WARPS); mbar_init(&sm.side_full[i], 1); }
    for (int w = 0; w < NUM_PROD_WARPS; ++w)
      for (int i = 0; i < LRING; ++i) mbar_init(&sm.lring_full[w][i], 1);
    for (int i = 0; i < ACC; ++i) { mbar_init(&sm.tmem_full[i], 1); mbar_init(&sm.tmem_empty[i], 2 * NUM_EPI_WARPS); }
    for (int i = 0; i < GBUF; ++i) {
      mbar_init(&sm.gather_full[i], NUM_EPI_WARPS / 2);
      mbar_init(&sm.gather_free_local[i], NUM_EPI_WARPS);
      mbar_init(&sm.gather_free_remote[i], NUM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  if (warp < 4) load_qt_half<4>(a.tab, tmem, rank, warp, lane);
  tc_fence_before();
  cluster_sync_all();    // barriers initialised and both A halves resident before any cross-CTA traffic
  tc_fence_after();

  // register budget per role (whole 4-warp groups): the light group hands its registers to samplers and producers
  if (warp >= FIRST_PROD_WARP && warp < MMA_WARP) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_HEAVY));
    // ======================================================================== producers: 16 lanes per row, 2 rows per pass
    const int pw = warp - FIRST_PROD_WARP;
    const int half = lane >> 4, l16 = lane & 15;
    // lane owns k = 64c + 4*l16 .. +3 for c = 0..3; each softmax reduction is a 4-step butterfly inside the half-warp
    // (two independent rows per warp keep the pipes busy).  The raw logits rows arrive through a small smem ring that
    // cp.async.bulk fills two passes ahead, so no global-memory latency sits on the warp's critical path.
    const float* tabA = reinterpret_cast<const float*>(a.tab + TAB_A_OFF) + 4 * l16;
    const float hb = a.h * a.beta;
    const bool contiguous = (a.ld == S) && (a.batch_stride == (long long)a.D * S);
    uint64_t* const full_bar = rank == 0 ? &sm.full[0] : &sm.full_local[0];
    constexpr int PASSES = ROWS_PER_PROD / 2;                    // passes per tile; warp pw builds rows ROWS_PER_PROD*pw ..
    const int npass = my_tiles * PASSES;

    const LT* const logits = static_cast<const LT*>(a.logits);
    auto row_ptr = [&](long long g) -> const LT* {
      if (contiguous) return logits + g * S;
      const uint32_t n = (uint32_t)g / (uint32_t)a.D, d = (uint32_t)g - n * (uint32_t)a.D;
      return logits + (long long)n * a.batch_stride + (long long)d * a.ld;
    };
    // Running state of the fetch stream (two passes ahead of the compute stream): first row of the pair, pass-in-tile,
    // ring slot.  Everything advances by additions only - no index arithmetic on the warp's critical path.
    const long long tile_step = (long long)npairs * NT - 2 * (PASSES - 1);
    long long gf = (long long)pair * NT + (long long)rank * NH + ROWS_PER_PROD * pw;
    int f_left = npass, f_ps = 0, f_slot = 0;
    // lane 0 starts the bulk copy of the next row pair (rows past the end are replaced by row 0: never used; adjacent
    // rows of a contiguous logits tensor travel as one 2 KB copy); every lane fetches the state of its half's row
    // HEAD: head parameters of the row fetch() just visited.  They reach their use two passes later in their stored type
    // (bf16 as its raw 16 bits) and are widened only there: a widening at the load would wait for the load right away and
    // put its latency on the warp's critical path
    using HeadRaw = typename std::conditional<sizeof(LT) == 2, unsigned short, float>::type;
    HeadRaw f_mu = 0, f_ls = 0;
    auto fetch = [&]() -> int {
      int xv = -1;
      if (f_left > 0) {
        if (HEAD) {
          const long long g = gf + half;
          if (g < a.rows) {
            long long src = g;
            if (a.head_bs != (long long)a.D) {   // (N, 2D) network output viewed as two (N, D) halves
              // 32-bit division whenever the row index fits (a 64-bit one is ~100 instructions on the warp's critical path)
              const long long n = (a.rows <= 0xFFFFFFFFLL) ? (long long)((uint32_t)g / (uint32_t)a.D) : g / a.D;
              src = n * a.head_bs + (g - n * a.D);
            }
            f_mu = __ldg(static_cast<const HeadRaw*>(a.head_mu) + src);
            f_ls = __ldg(static_cast<const HeadRaw*>(a.head_ls) + src);
          }
        } else if (lane == 0) {
          uint64_t* bar = &sm.lring_full[pw][f_slot];
          mbar_arrive_expect_tx(bar, 2 * ROW_BYTES);
          uint8_t* const dst = reinterpret_cast<uint8_t*>(&sm.lring[pw][f_slot][0][0]);   // row hf of the pair at hf * ROW_BYTES
          if (contiguous && gf + 1 < a.rows) {
            bulk_g2s(dst, logits + gf * S, 2 * ROW_BYTES, bar);
          } else {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const long long gg = (gf + hf < a.rows) ? gf + hf : 0;
              bulk_g2s(dst + hf * ROW_BYTES, row_ptr(gg), ROW_BYTES, bar);
            }
          }
        }
        if (gf + half < a.rows) xv = __ldg(a.x_eval + gf + half);
        if (!HEAD && contiguous && f_ps == 0 && lane == 0) {   // pull this warp's 4 rows of a later tile from HBM into L2
          const long long r0 = gf + (long long)PREFETCH_TILES * npairs * NT;
          if (r0 + ROWS_PER_PROD <= a.rows) l2_prefetch_bulk(logits + r0 * S, ROWS_PER_PROD * ROW_BYTES);
        }
        --f_left;
        f_slot = (f_slot + 1 == LRING) ? 0 : f_slot + 1;
        if (++f_ps == PASSES) { f_ps = 0; gf += tile_step; } else { gf += 2; }
      }
      return xv;
    };

    int x_cur = fetch();
    HeadRaw mu_cur = f_mu, ls_cur = f_ls;
    int x_n1 = fetch();
    HeadRaw mu_n1 = f_mu, ls_n1 = f_ls;
    float4 t4[4];
    {
      const size_t xo = (size_t)(x_cur < 0 ? 0 : x_cur) << 8;
#pragma unroll
      for (int c = 0; c < 4; ++c) t4[c] = __ldg(reinterpret_cast<const float4*>(tabA + xo + 64 * c));
    }
    // The row reductions (sum e, sum e*a) and the row scalars of a pass are FINISHED IN THE NEXT PASS: its per-lane
    // partial sums are carried over, their butterflies run next to the next pass's row-maximum butterfly (independent
    // shuffle chains instead of one after the other), and the side record / pre_full arrival follow there.
    // Only the operand rows (what the MMA waits for) are completed inside the pass itself.
    float p_sum = 1.f, p_dot = 0.f;
    int p_x = 0, p_r = 0, p_slot = 0;
    bool p_have = false, p_close = false;
    auto finish_prev = [&]() {          // p_sum / p_dot hold the reduced values
      if (!p_have) return;
      const float rs = __frcp_rn(p_sum);
      float c1, c0;
      if (TAULDR) {
        c1 = hb * rs;                                            // lam_s = D_s * c1 * Rb[s,x]
        c0 = 0.f;
      } else {
        const float inv = __frcp_rn(fmaf(p_dot, rs, 1e-35f));    // 1 / (pQ[x] + 1e-35)
        c1 = hb * rs * inv;                                      // lam_s = (D_s * c1 + c0) * Rb[x,s]
        c0 = hb * 1e-35f * inv;
      }
      // row scalars for the count warp and the samplers (one lane per half-warp); the count warp adds the uniform
      if (l16 == 0) sm.side[p_slot][p_r] = Side{c1, c0, p_x, 0u};
      if (p_close) {                    // that pass closed its tile: the tile's row scalars are complete now
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.pre_full[p_slot]);
      }
      p_have = false;
    };
    // running state of the compute stream
    int ps = 0, st = 0, slot = 0, rslot = 0;
    uint32_t st_par = 1, ring_par = 0;      // parity to wait for on empty[st] / lring_full[rslot]
#pragma unroll 1
    for (int pi = 0; pi < npass; ++pi) {
      const bool ok = x_cur >= 0;
      if (ps == 0) mbar_wait(&sm.empty[st], st_par);
      const uint32_t stage_s = smem_u32(sm.stage[st]);
      if (!HEAD) mbar_wait(&sm.lring_full[pw][rslot], ring_par);
      const int r = ROWS_PER_PROD * pw + 2 * ps + half;
      float v[16];
      float ml = 0.f;
      if (HEAD) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {     // previous pass's reductions: independent of the head arithmetic below
          p_sum += __shfl_xor_sync(0xffffffffu, p_sum, o);
          if (!TAULDR) p_dot += __shfl_xor_sync(0xffffffffu, p_dot, o);
        }
        head_numerators(widen_head(mu_cur), widen_head(ls_cur), a.head_fix != 0, l16, v);
      } else {
        if constexpr (sizeof(LT) == 2) {
          // lane l16 widens the same elements 64c + 4*l16 .. +3 as in the fp32 kernel, one 64-bit load each
          const uint32_t src = smem_u32(&sm.lring[pw][rslot][0][0]) + half * ROW_BYTES + 8 * l16;
#pragma unroll
          for (int c = 0; c < 4; ++c) widen2x4<LT>(lds64(src + 128 * c), v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        } else {
          const uint32_t src = smem_u32(&sm.lring[pw][rslot][half][4 * l16]);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 q4 = lds128(src + 256 * c);
            v[4 * c] = q4.x; v[4 * c + 1] = q4.y; v[4 * c + 2] = q4.z; v[4 * c + 3] = q4.w;
          }
        }
        float m4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) m4[c] = fmaxf(fmaxf(v[4 * c], v[4 * c + 1]), fmaxf(v[4 * c + 2], v[4 * c + 3]));
        float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {     // this pass's row maximum next to the previous pass's reductions
          m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
          p_sum += __shfl_xor_sync(0xffffffffu, p_sum, o);
          if (!TAULDR) p_dot += __shfl_xor_sync(0xffffffffu, p_dot, o);
        }
        ml = -m * 1.4426950408889634f;
      }
      finish_prev();
      // four independent accumulation chains of packed pairs
      float2 sum2[4], dot2[4];
      const float2 l2e2 = make_float2(1.4426950408889634f, 1.4426950408889634f), ml2 = make_float2(ml, ml);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        sum2[c] = make_float2(0.f, 0.f); dot2[c] = make_float2(0.f, 0.f);
#pragma unroll
        for (int e = 0; e < 4; e += 2) {
          const float2 tq = e == 0 ? make_float2(t4[c].x, t4[c].y) : make_float2(t4[c].z, t4[c].w);
          float2 ex = make_float2(v[4 * c + e], v[4 * c + e + 1]);                 // HEAD: already the numerators
          if (!HEAD) {
            const float2 arg = ffma2(ex, l2e2, ml2);
            ex = make_float2(ex2_approx(arg.x), ex2_approx(arg.y));                // exp(v - max)
          }
          sum2[c] = fadd2(sum2[c], ex);
          if (!TAULDR) dot2[c] = ffma2(ex, tq, dot2[c]);
          const float2 op = TAULDR ? fmul2(ex, tq) : ex;   // tauLDR operand: e_k / (Q[k,x] + eps); 1/sum applied by the sampler
          v[4 * c + e] = op.x; v[4 * c + e + 1] = op.y;
        }
      }
      const float2 s01 = fadd2(sum2[0], sum2[1]), s23 = fadd2(sum2[2], sum2[3]), sall = fadd2(s01, s23);
      float sum = sall.x + sall.y;
      float dot = 0.f;
      if (!TAULDR) {
        const float2 d01 = fadd2(dot2[0], dot2[1]), d23 = fadd2(dot2[2], dot2[3]), dall = fadd2(d01, d23);
        dot = dall.x + dall.y;
      }
      // the table row of the NEXT pass is requested as soon as this pass's has been consumed
      {
        const size_t xo = (size_t)(x_n1 < 0 ? 0 : x_n1) << 8;
#pragma unroll
        for (int c = 0; c < 4; ++c) t4[c] = __ldg(reinterpret_cast<const float4*>(tabA + xo + 64 * c));
      }
      // rows past the end (the last tile only) contribute zero operand rows
      if (!ok) {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = 0.f;
      }
      store_operand_row<KBLOCK_BYTES, SPLIT_BYTES>(stage_s, r, l16, v);
      // this pass's partial sums and row identity travel to the next pass (finish_prev)
      p_sum = sum; p_dot = dot;
      p_x = x_cur; p_r = r; p_slot = slot; p_close = (ps + 1 == PASSES); p_have = true;
      if (++rslot == LRING) { rslot = 0; ring_par ^= 1u; }
      __syncwarp();            // every lane is done with this pass's ring slot: refill it for the pass after next
      x_cur = x_n1;
      if (HEAD) { mu_cur = mu_n1; ls_cur = ls_n1; }
      x_n1 = fetch();
      if (HEAD) { mu_n1 = f_mu; ls_n1 = f_ls; }
      if (++ps == PASSES) {     // last pass of the tile
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar + st);   // operand rows are in place (the row scalars follow in finish_prev)
        ps = 0;
        slot = (slot + 1) & (RING - 1);
        if (++st == STAGES) { st = 0; st_par ^= 1u; }
      }
    }
    // the last pass's reductions and row scalars
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      p_sum += __shfl_xor_sync(0xffffffffu, p_sum, o);
      if (!TAULDR) p_dot += __shfl_xor_sync(0xffffffffu, p_dot, o);
    }
    finish_prev();
  } else if (warp > COUNT_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));   // idle warps of the light group
  } else if (warp == COUNT_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));
    // ======================================================================== count warp: lane = row of the tile
    // one categorical draw per valid row: its uniform from the per-row Euler stream
    for (int i = 0; i < my_tiles; ++i) {
      const int tile = pair + i * npairs, slot = i % RING;
      const long long g0 = (long long)tile * NT + (long long)rank * NH;
      mbar_wait(&sm.pre_full[slot], (i / RING) & 1);
      if (sm.side[slot][lane].x >= 0)
        sm.side[slot][lane].w = philox_row_word((uint64_t)(a.row_offset + g0 + lane), 0, a.offset, STREAM_ROW, a.seed);
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.side_full[slot]);
    }
  } else if (warp == MMA_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));
    // ======================================================================== MMA issue (one thread of the leader CTA)
    if (rank == 0 && lane == 0) {
      for (int i = 0; i < my_tiles; ++i) {
        const int st = i % STAGES, b = i % ACC;
        mbar_wait_cluster(&sm.full[st], (i / STAGES) & 1);
        mbar_wait(&sm.tmem_empty[b], ((i / ACC) & 1) ^ 1);
        tc_fence_after();
        issue_tile<KBLOCK_BYTES, SPLIT_BYTES, IDESC>(tmem, tmem + TM_ACC + b * NT, smem_u32(sm.stage[st]));
        umma_commit_pair(&sm.empty[st]);
        umma_commit_pair(&sm.tmem_full[b]);
      }
    } else if (rank != 0 && lane == 0) {
      relay_full<STAGES, POLL_NS>(sm.full_local, sm.full, my_tiles);
    }
    __syncwarp();
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_HEAVY));
    // ======================================================================== epilogue + row sampler
    const int q = warp & 3;                       // TMEM quadrant -> states rank*128 + 32q + lane
    const uint32_t owner = (uint32_t)(warp >> 2); // accumulator columns [32*owner, 32*owner+32) belong to CTA `owner`
    const int s_mine = (int)rank * 128 + q * 32 + lane;
    const uint32_t gather_dst = mapa(smem_u32(&sm.gather[0][0][0]), owner) + (uint32_t)s_mine * 4u;
    const uint32_t gfull_dst = mapa(smem_u32(&sm.gather_full[0]), owner);
    const uint32_t tempty_dst = mapa(smem_u32(&sm.tmem_empty[0]), 0);
    const uint32_t gfree_remote_dst = mapa(smem_u32(&sm.gather_free_remote[0]), rank ^ 1u);
    uint64_t* const gfree_wait = (owner == rank) ? &sm.gather_free_local[0] : &sm.gather_free_remote[0];
    const float* tabE = reinterpret_cast<const float*>(a.stat + (TAULDR ? ST_RBZT_OFF : ST_RBZ_OFF)) + 8 * lane;
    const float* tabC = reinterpret_cast<const float*>(a.stat + ST_RBZ_OFF) + 8 * lane;   // corrector add: Rb[x][s], zero diag
    const float hb = a.h * a.beta;
    RowStats stt = {0, 0, 0, 0, 0};

    // phase A of tile i: accumulator (this CTA's 128 states x this warp's 32 rows) -> gather buffer of the rows' owner
    auto phase_a = [&](int i) {
      const int b = i % ACC, gb = i % GBUF;
      mbar_wait(&sm.tmem_full[b], (i / ACC) & 1);
      mbar_wait(gfree_wait + gb, ((i / GBUF) & 1) ^ 1);
      tc_fence_after();
      uint32_t acc[32];
      tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + TM_ACC + b * NT + owner * NH, acc);
      tmem_ld_wait();
      if (owner == rank) {
        const uint32_t dst = smem_u32(&sm.gather[gb][0][s_mine]);
#pragma unroll
        for (int j = 0; j < 32; ++j) sts32(dst + (uint32_t)j * (S * 4), __uint_as_float(acc[j]));
      } else {
        // the partner's barrier counts these bytes as they land: nothing to fence, nothing to wait for here
        const uint32_t dst = gather_dst + (uint32_t)gb * (NH * S * 4);
        const uint32_t bar = gfull_dst + (uint32_t)gb * 8u;
#pragma unroll
        for (int j = 0; j < 32; ++j) st_async_cluster_f32(dst + (uint32_t)j * (S * 4), __uint_as_float(acc[j]), bar);
      }
      tc_fence_before();   // accumulator has been read: hand the buffer back to the MMA warp
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_cluster_relaxed(tempty_dst + (uint32_t)b * 8u);
        if (owner == rank) {
          // warp 0 also announces the bytes the partner's four warps will deliver for this phase
          if (q == 0) mbar_arrive_expect_tx(&sm.gather_full[gb], (NUM_EPI_WARPS / 2) * 32 * NH * 4);
          else mbar_arrive(&sm.gather_full[gb]);
        }
      }
    };

    if (my_tiles > 0) phase_a(0);
    for (int i = 0; i < my_tiles; ++i) {
      // ---- phase B: sample the rows this CTA owns (warp w: rows 4w .. 4w+3 of the CTA's 32)
      const int tile = pair + i * npairs;
      const int slot = i % RING, gb = i % GBUF;
      mbar_wait(&sm.side_full[slot], (i / RING) & 1);
      const long long g0 = (long long)tile * NT + (long long)rank * NH;
      // the warp's rows that exist, processed two per iteration
      uint32_t todo = __ballot_sync(0xffffffffu, lane < ROWS_PER_SAMPLER && sm.side[slot][warp * ROWS_PER_SAMPLER + lane].x >= 0);
      // The side record + rate-table rows (L2 gathers) of the NEXT pair are requested while the current pair is searched;
      // the first pair's before the wait for the accumulator rows.  The table registers are dead between the rate
      // computation and the next iteration.
      int rrow[2] = {0, 0};
      bool two = false;
      Side si[2];
      float4 e0[2], e1[2], c0v[2], c1v[2];
      auto load_pair = [&]() {
        rrow[0] = __ffs(todo) - 1;
        todo &= todo - 1;
        two = todo != 0;
        rrow[1] = two ? __ffs(todo) - 1 : rrow[0];
        todo &= todo - 1;   // no-op when todo == 0
#pragma unroll
        for (int u = 0; u < 2; ++u) si[u] = sm.side[slot][warp * ROWS_PER_SAMPLER + rrow[u]];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const size_t xo = (size_t)si[u].x << 8;
          // lane owns states 4*lane .. +3 (elements 0-3) and 128 + 4*lane .. +3 (elements 4-7): every 128-bit access of
          // the warp to a gather row is then one contiguous 512-byte run (no bank conflicts)
          e0[u] = __ldg(reinterpret_cast<const float4*>(tabE - 4 * lane + xo));
          e1[u] = __ldg(reinterpret_cast<const float4*>(tabE - 4 * lane + xo + 128));
          if (CORR) {
            c0v[u] = __ldg(reinterpret_cast<const float4*>(tabC - 4 * lane + xo));
            c1v[u] = __ldg(reinterpret_cast<const float4*>(tabC - 4 * lane + xo + 128));
          }
        }
      };
      bool have = todo != 0;
      if (have) load_pair();
      // the next tile's accumulator is moved now: the cross-CTA hand-shakes of tile i and the L2 latency of the first
      // pair's table rows complete in its shadow
      if (i + 1 < my_tiles) phase_a(i + 1);
      mbar_wait(&sm.gather_full[gb], (i / GBUF) & 1);
      // two rows in flight per iteration (independent dependency chains hide the shuffle / smem latency)
#pragma unroll 1
      while (have) {
        // the current pair's identifiers survive the preload of the next pair
        const int rc0 = rrow[0], rc1 = rrow[1];
        const bool two_c = two;
        const int xc0 = si[0].x, xc1 = si[1].x;
        uint32_t gp[2];   // shared-space address of the row's gather slot
        float d[2][8];
        float total[2];
        gp[0] = smem_u32(&sm.gather[gb][warp * ROWS_PER_SAMPLER + rc0][0]);
        gp[1] = smem_u32(&sm.gather[gb][warp * ROWS_PER_SAMPLER + rc1][0]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float4 d0 = lds128(gp[u] + 16 * lane);
          const float4 d1 = lds128(gp[u] + 512 + 16 * lane);
          const float dv[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
          const float ev[8] = {e0[u].x, e0[u].y, e0[u].z, e0[u].w, e1[u].x, e1[u].y, e1[u].z, e1[u].w};
          // lam_s (zero at s == x through the zero-diagonal tables)
#pragma unroll
          for (int e = 0; e < 8; ++e) d[u][e] = fmaf(dv[e], si[u].c1, si[u].c0) * ev[e];
          if (CORR) {
            const float cv[8] = {c0v[u].x, c0v[u].y, c0v[u].z, c0v[u].w, c1v[u].x, c1v[u].y, c1v[u].z, c1v[u].w};
#pragma unroll
            for (int e = 0; e < 8; ++e) d[u][e] = fmaf(hb, cv[e], d[u][e]);
          }
          // inclusive prefix sums over the 256 states: in-lane per 4-state group, then across lanes per half
#pragma unroll
          for (int e = 1; e < 4; ++e) { d[u][e] += d[u][e - 1]; d[u][4 + e] += d[u][3 + e]; }
        }
        float incl[2][2] = {{d[0][3], d[0][7]}, {d[1][3], d[1][7]}};   // [row][half]
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const float n = __shfl_up_sync(0xffffffffu, incl[u][hf], o);
              if (lane >= o) incl[u][hf] += n;
            }
        }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          float excl_a = __shfl_up_sync(0xffffffffu, incl[u][0], 1);
          float excl_b = __shfl_up_sync(0xffffffffu, incl[u][1], 1);
          const float tot_a = __shfl_sync(0xffffffffu, incl[u][0], 31);
          const float tot_b = __shfl_sync(0xffffffffu, incl[u][1], 31);
          if (lane == 0) { excl_a = 0.f; excl_b = 0.f; }
          excl_b += tot_a;
          total[u] = tot_a + tot_b;
#pragma unroll
          for (int e = 0; e < 4; ++e) { d[u][e] += excl_a; d[u][4 + e] += excl_b; }
          // stay-probability max(0, 1 - sum) enters the cumulative sums at position x
          const float diag = fmaxf(0.f, 1.0f - total[u]);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            d[u][e] += (4 * lane + e >= si[u].x) ? diag : 0.f;
            d[u][4 + e] += (128 + 4 * lane + e >= si[u].x) ? diag : 0.f;
          }
          total[u] += diag;
          if (u == 0 || two_c) {
            sts128(gp[u] + 16 * lane, make_float4(d[u][0], d[u][1], d[u][2], d[u][3]));
            sts128(gp[u] + 512 + 16 * lane, make_float4(d[u][4], d[u][5], d[u][6], d[u][7]));
          }
        }
        __syncwarp();
        have = todo != 0;
        if (have) load_pair();      // next pair: side record and table rows in flight during the search below
        // lane 0 picks for the first row, lane 1 for the second: the first state whose prefix sum exceeds v * total.
        // The other lanes get a target below every prefix sum and walk the second row's (broadcast) addresses instead of
        // scattering random shared-memory reads over the banks.
        const int u = lane == 0 ? 0 : 1;
        const bool active = lane == 0 || (lane == 1 && two_c);
        const int r = warp * ROWS_PER_SAMPLER + (u ? rc1 : rc0);
        const uint32_t w = sm.side[slot][r].w;
        const float T = active ? fminf(u32_to_unit(w), 0.99999994f) * (u ? total[1] : total[0]) : -1.0f;
        const int xn = prefix_search(u ? gp[1] : gp[0], T);   // the pick IS the new state
        if (active) {
          const long long g = g0 + r;
          const int x = u ? xc1 : xc0;
          const int xb = a.x_base ? a.x_base[g] : x;
          a.x_out[g] = xn;
          stt.changed_base += (xn != xb);
          stt.changed_eval += (xn != x);
        }
      }
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&sm.gather_free_local[gb]);
        mbar_arrive_cluster_relaxed(gfree_remote_dst + (uint32_t)gb * 8u);
      }
    }
    if (a.stats) {
      const int v[5] = {stt.changed_base, stt.nonzero, stt.changed_eval, stt.jumped, stt.multi};
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const int tot = warp_sum_int(v[k]);
        if (lane == 0 && tot) atomicAdd(a.stats + k, (unsigned long long)tot);
      }
    }
  }
  pair_teardown(warp == MMA_WARP, tmem);
}

// ---------------------------------------------------------------------------------------------- table prep
__global__ void prep_tables_kernel(const float* __restrict__ QT, int T, float eps, int branch, uint8_t* __restrict__ out) {
  const int t = blockIdx.y;
  const float* qt = QT + (size_t)t * S * S;
  uint8_t* blob = out + (size_t)t * TAB_BYTES;
  uint32_t* qh = reinterpret_cast<uint32_t*>(blob + TAB_QH_OFF);
  uint32_t* qm = reinterpret_cast<uint32_t*>(blob + TAB_QM_OFF);
  float* ta = reinterpret_cast<float*>(blob + TAB_A_OFF);
  // QT[s][k] = Q[k][s]: the A operand row s holds K contiguous -> pairs (k, k+1)
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * 128; i += gridDim.x * blockDim.x) {
    const float a0 = qt[2 * i], a1 = qt[2 * i + 1];
    uint32_t hi, mid;
    split2(a0, a1, hi, mid);
    qh[i] = hi;
    qm[i] = mid;
  }
  // TAB_A[x][k] = f(Q[k][x]) = f(QT[x][k])
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * S; i += gridDim.x * blockDim.x) {
    const float q = qt[i];
    ta[i] = (branch == CTDD_BRANCH_TAULDR) ? 1.0f / (q + eps) : q;
  }
}

__global__ void prep_static_kernel(const float* __restrict__ Rb, uint8_t* __restrict__ out) {
  float* rbzt = reinterpret_cast<float*>(out + ST_RBZT_OFF);
  float* rbz = reinterpret_cast<float*>(out + ST_RBZ_OFF);
  float* rbt = reinterpret_cast<float*>(out + ST_RBT_OFF);
  float* rbf = reinterpret_cast<float*>(out + ST_RB_OFF);
  float* zero = reinterpret_cast<float*>(out + ST_ZERO_OFF);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * S; i += gridDim.x * blockDim.x) {
    const int x = i / S, s = i % S;
    const float t = Rb[(size_t)s * S + x], r = Rb[i];
    rbzt[i] = (s == x) ? 0.f : t;
    rbz[i] = (s == x) ? 0.f : r;
    rbt[i] = t;
    rbf[i] = r;
    if (i < S) zero[i] = 0.f;
  }
  int* bandT = reinterpret_cast<int*>(out + ST_BANDT_OFF);
  int* bandR = reinterpret_cast<int*>(out + ST_BANDR_OFF);
  for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < S; x += gridDim.x * blockDim.x) {
    int loT = S - 1, hiT = 0, loR = S - 1, hiR = 0;   // exact zero pattern of column x / row x without the diagonal
    for (int s = 0; s < S; ++s) {
      if (s == x) continue;
      const float r = Rb[(size_t)x * S + s], c = Rb[(size_t)s * S + x];
      if (r != 0.f) { loR = s < loR ? s : loR; hiR = s > hiR ? s : hiR; }
      if (c != 0.f) { loT = s < loT ? s : loT; hiT = s > hiT ? s : hiT; }
    }
    bandT[x] = loT | (hiT << 8);
    bandR[x] = loR | (hiR << 8);
  }
}

}  // namespace tc

bool tc_supports(const ctdd_step_params* p) {
  if (p->S != tc::S) return false;
  if (!(p->branch == CTDD_BRANCH_TAULDR || p->branch == CTDD_BRANCH_SDDM_REVERSE_PROB)) return false;
  if (!(p->mode == CTDD_MODE_TAU_LEAP || p->mode == CTDD_MODE_TAU_LEAP_CORR || p->mode == CTDD_MODE_MIDPOINT_JUMP ||
        p->mode == CTDD_MODE_MIDPOINT_DRIFT || p->mode == CTDD_MODE_EULER || p->mode == CTDD_MODE_EULER_CORR ||
        p->mode == CTDD_MODE_RATES_ONLY))
    return false;
  if (!p->tc_tables || !p->tc_static) return false;
  // rows are bulk-copied: 16-byte aligned (4 fp32 or 8 bf16 / fp16 elements)
  const int64_t row_align = (int64_t)(16 / dtype_bytes(p->logits_dtype)) - 1;
  if (p->head == CTDD_HEAD_LOGITS &&
      ((p->ld_logits & row_align) || (p->batch_stride_logits & row_align) || (reinterpret_cast<uintptr_t>(p->logits) & 15)))
    return false;
  if (p->mode == CTDD_MODE_RATES_ONLY &&
      ((reinterpret_cast<uintptr_t>(p->rr_out) & 15) || (reinterpret_cast<uintptr_t>(p->ratio_out) & 15)))
    return false;
  return true;
}

long long tc_workspace_bytes(long long rows, int S) {
  (void)rows; (void)S;
  return 0;   // every row is finished inside the kernel (no cross-kernel partials)
}

// Euler modes (one categorical draw per row over all 256 states); ctdd_reverse_step sends every other mode to
// launch_step_tcq.
int launch_step_tc(const ctdd_step_params* p, cudaStream_t st) {
  using namespace tc;
  static PairLaunchState launch_state;
  const size_t smem_bytes = sizeof(Smem) + 1024;
  typedef void (*kern_t)(const Args);
#define CTDD_TC_ROW(T, H, LT) step_tc_kernel<T, false, H, LT>, step_tc_kernel<T, true, H, LT>
  static const kern_t kerns[20] = {CTDD_TC_ROW(false, false, float), CTDD_TC_ROW(true, false, float),
                                     CTDD_TC_ROW(false, true, float), CTDD_TC_ROW(true, true, float),
                                     CTDD_TC_ROW(false, false, __nv_bfloat16), CTDD_TC_ROW(true, false, __nv_bfloat16),
                                     CTDD_TC_ROW(false, true, __nv_bfloat16), CTDD_TC_ROW(true, true, __nv_bfloat16),
                                     CTDD_TC_ROW(false, false, __half), CTDD_TC_ROW(true, false, __half)};
#undef CTDD_TC_ROW
  Args a = make_args(p);
  a.num_tiles = (int)((a.rows + NT - 1) / NT);
  const int pairs = pair_count(launch_state, "ctdd_reverse_step", kerns, smem_bytes, a.num_tiles);
  if (!pairs) return 1;
  // rows of kerns: fp32 logits, fused head on fp32 (mu, log_scale), bf16 logits, fused head on bf16 (mu, log_scale),
  // fp16 logits (the head takes no fp16: ctdd_reverse_step refuses it)
  const int dt = p->head != CTDD_HEAD_LOGITS ? p->head_dtype : p->logits_dtype;
  const int ki = ((p->branch == CTDD_BRANCH_TAULDR) ? 1 : 0) + (p->head != CTDD_HEAD_LOGITS ? 2 : 0) +
                 (dt == CTDD_DTYPE_BF16 ? 4 : (dt == CTDD_DTYPE_F16 ? 8 : 0));
  const int kj = (p->mode == CTDD_MODE_EULER_CORR) ? 1 : 0;
  kerns[2 * ki + kj]<<<2 * pairs, NUM_THREADS, smem_bytes, st>>>(a);
  CTDD_CHECK_LAUNCH("step_tc_kernel");
  return 0;
}

}  // namespace ctdd

extern "C" int64_t ctdd_tc_tables_bytes(int S) { return S == ctdd::tc::S ? (int64_t)ctdd::tc::TAB_BYTES : 0; }
extern "C" int64_t ctdd_tc_static_bytes(int S) { return S == ctdd::tc::S ? (int64_t)ctdd::tc::ST_BYTES : 0; }
extern "C" int64_t ctdd_tc_static_align(void) { return (int64_t)ctdd::tc::ST_ALIGN; }

extern "C" int ctdd_prep_tc_tables(const float* Q, const float* QT, const float* Rb, int T, int S, float eps,
                                   int branch, void* tables_out, void* stream) {
  using namespace ctdd;
  (void)Q; (void)Rb;
  if (S != tc::S) { set_error("ctdd_prep_tc_tables: the tcgen05 path needs S == 256 (got %d)", S); return 2; }
  if (!QT || !tables_out || T <= 0) { set_error("ctdd_prep_tc_tables: bad arguments"); return 2; }
  for (int t0 = 0; t0 < T; t0 += 32768) {
    const int nt = (T - t0) < 32768 ? (T - t0) : 32768;
    uint8_t* out = reinterpret_cast<uint8_t*>(tables_out) + (size_t)t0 * tc::TAB_BYTES;
    dim3 grid(32, nt);
    tc::prep_tables_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(QT + (size_t)t0 * S * S, nt, eps, branch, out);
    CTDD_CHECK_LAUNCH("prep_tables_kernel");
  }
  return 0;
}

extern "C" int ctdd_prep_tc_static(const float* Rb, int S, void* static_out, void* stream) {
  using namespace ctdd;
  if (S != tc::S) { set_error("ctdd_prep_tc_static: the tcgen05 path needs S == 256 (got %d)", S); return 2; }
  if (!Rb || !static_out) { set_error("ctdd_prep_tc_static: null pointer"); return 2; }
  if (reinterpret_cast<uintptr_t>(static_out) % tc::ST_ALIGN) {
    set_error("ctdd_prep_tc_static: static_out must be aligned to ctdd_tc_static_align() = %zu bytes", tc::ST_ALIGN);
    return 2;
  }
  tc::prep_static_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(Rb, reinterpret_cast<uint8_t*>(static_out));
  CTDD_CHECK_LAUNCH("prep_static_kernel");
  return 0;
}

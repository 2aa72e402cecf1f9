// tcgen05 reverse-step kernel for S == 256 (configs C3/C4/C5), every mode except the Euler ones: the (N*D x S)(S x S)
// contraction of lib/sampling/sampling.py:57 on 5th-generation tensor cores, fused with softmax, the q_{t|0}
// denominators, the forward-rate multiply and the Philox state update (tau-leap / corrector sampling.py:127-221,
// midpoint :423-503, rates only :31-78).
//
// One CTA PAIR (thread-block cluster of 2, tcgen05 cta_group::2) owns a sequence of 128-row tiles:
//   D[s, row] = sum_k Q^T[s, k] * a[row, k]        M = 256 states (128 per CTA), N = 128 rows, K = 256
//   * M side = state s. Each CTA keeps ITS 128-state half of Q^T (bf16 hi + mid split, 2 x 128 TMEM columns) resident
//     in tensor memory as the A operand (TS form) for the whole kernel; 2 accumulators of 128 columns.  With N = 128
//     an instruction sits on the 64-cycle floor of the TS form (the A slice is read from tensor memory at 64 B/cycle).
//   * N side = data rows; each CTA produces 64 rows of a tile.  Producer warps work on two rows per pass, 16 lanes per
//     row: raw fp32 or bf16 logits from a per-warp ring of two 2 KB slots, row softmax by half-warp butterflies, gathered reciprocal
//     denominators 1/(Q[k,x]+eps), bf16 hi/mid split, K-major 128B-swizzled smem stage.  The passes of a tile are dealt
//     round-robin to the producer warps; one pass counter per warp, every position derives from it.
//   * A loader warp issues what the producers would otherwise stall on: per GROUP of 4 producer warps (one per SM
//     sub-partition; their 4 consecutive passes are 8 consecutive rows) ONE 8 KB cp.async.bulk per round into the group's
//     ring slots, and per tile two DSMEM bulk copies that forward the 64 row-scalar records (rate scale, state, band of
//     non-zero base rates) to the partner CTA.
//   * 3 tensor passes  Qh*ah + Qh*am + Qm*ah  accumulate in fp32 TMEM (48 tcgen05.mma of N = 128 per tile).
//   * Epilogue: warp (q, h) reads its 32 states x 32 rows with tcgen05.ld (lane = state; two batches per tile).  In the
//     load's shadow lane = ROW fetches the 32 base-rate entries R_b[chunk states, x_row] of its own row (128 bytes of the
//     zero-diagonal [x][s] table; the zero row when the chunk lies outside the band of x) and the row's Philox call.  A
//     4.3 KB per-warp scratch transposes the accumulator to lane = row.  A warp's 32 states are one CHUNK of the chunked
//     superposition map (ctdd_common.cuh): each chunk of a row draws its own jump count K ~ Poisson(chunk total) and its
//     own picks, so no warp ever waits for another warp's total and all 32 rows of a batch are sampled in parallel:
//     sequential fp32 prefix sums in registers (the oracle's summation order, one FMA per state), inverse-CDF count,
//     picks by 31 register compares per pick when the batch's largest K is <= 3, else dealt to the 32 lanes over the prefix
//     sums parked in the scratch.
//   * The per-(row, chunk) result is one 32-bit record (sum of jumps << 2 | min(K, 3), or the partial drift); it goes to
//     the CTA that produced the row (plain st.shared or st.async + complete_tx), whose two finalizer warps (lane = row) add
//     the 8 chunks, apply the clamp / rejection rule and write x_out coalesced.
// Nothing but those records and the row scalars crosses between the CTAs of a pair.
// Warp roles per CTA: 8 epilogue warps, NPW producer warps, and a light group with the MMA-issue warp (leader CTA
// issues; the partner's relays its producers' arrivals), the loader warp and the 2 finalizer warps.
// Measurements, the hardware ceiling of the MMA stream and the variants that were tried and dropped:
// profiles/r2_step_tcq_summary.md.
#include "ctdd_tc_common.cuh"

namespace ctdd {
namespace tcq {
using namespace tc;

constexpr int NH = 64;                 // rows of a tile produced and finalized by one CTA
constexpr int NT = 2 * NH;             // rows per pair tile (= UMMA N)
constexpr int STAGES = 2;              // smem operand stages (64 KB each)
constexpr int ACC = 2;                 // TMEM accumulator buffers (NT columns each)
constexpr int CBUF = 2;                // contribution buffers (epilogue -> finalizer)
constexpr int RING = 7;                // per-tile row-scalar ring (> STAGES + ACC + CBUF)
constexpr int NUM_EPI_WARPS = 8;       // epilogue warp e: TMEM quadrant e&3, column half e>>2 (= CTA that owns those rows)
constexpr int NPW = 12;                // producer warps (a multiple of 4: register budgets are per 4-warp group)
constexpr int FIRST_PROD_WARP = NUM_EPI_WARPS;
constexpr int FIRST_EPI_WARP = 0;
constexpr int MMA_WARP = NUM_EPI_WARPS + NPW;   // light group: MMA issue / relay, idle, 2 finalizer warps
constexpr int FIN_WARP0 = MMA_WARP + 2;
constexpr int NUM_THREADS = (NUM_EPI_WARPS + NPW + 4) * 32;
// setmaxnreg targets.  The registers handed out by .inc are the ones the CTA's own warps released with .dec:
// 8 * EPI + NPW * PROD + 4 * LIGHT must not exceed (12 + NPW) * (launch allocation), or the .inc never returns.
constexpr int REGS_LAUNCH = (65536 / NUM_THREADS) & ~7;          // what __launch_bounds__ gives every thread (80)
constexpr int REGS_LIGHT = 48;
constexpr int REGS_PROD = REGS_LAUNCH;                           // producers keep the launch allocation
constexpr int REGS_EPI = 96;
static_assert(NUM_EPI_WARPS * REGS_EPI + NPW * REGS_PROD + 4 * REGS_LIGHT <= (NUM_EPI_WARPS + NPW + 4) * REGS_LAUNCH,
              "setmaxnreg budget exceeds the launch allocation");
constexpr int PASSES_PER_TILE = NH / 2;                          // 32 two-row passes per tile and CTA
constexpr int KBLOCK_BYTES = NH * 128;         // one 64-wide K block of one split: NH rows x 128 B
constexpr int SPLIT_BYTES = 4 * KBLOCK_BYTES;  // K = 256 -> 4 blocks
constexpr int STAGE_BYTES = 2 * SPLIT_BYTES;   // hi + mid
// The logits ring is refilled per GROUP of 4 producer warps 4g .. 4g+3 (one per SM sub-partition, the same rank in each
// scheduler's priority order, so they advance together): their 4 consecutive passes are 8 consecutive rows of one tile = one
// 8 KB bulk copy per group and round.
constexpr int GSZ = 4, NSUB = NPW / GSZ;   // (4 divides 32: passes of a group never cross a tile boundary)
constexpr int REGPICK_MAX = 3;         // largest per-(row, chunk) jump count of a batch that is resolved from registers
constexpr int LRING = 2;               // per-producer-warp slots of raw logits row pairs filled by cp.async.bulk: refilled for the
                                       // warp's next pass as soon as this pass has its values in registers (rows are L2 hits)
constexpr int SCR_LD = 34;             // floats per row of an epilogue warp's transposing scratch (conflict-free 64-bit reads; 32 states + the jump-sum column)
constexpr uint32_t IDESC = make_idesc(NT);
constexpr uint32_t POLL_LONG = 512;    // ns between polls of the roles that wait for a whole tile (producers on a free stage, finalizers)
constexpr int NCHUNK = S / JUMP_CHUNK;                           // 8 chunks of 32 states per row
constexpr uint32_t SCAL_TX_BYTES = NH * 12;                      // row scalars the partner sends per tile
constexpr uint32_t CONTRIB_TX_BYTES = (NUM_EPI_WARPS / 2) * 2 * 32 * 4;   // records the partner's 4 warps send per tile

struct Smem {
  alignas(1024) uint8_t stage[STAGES][STAGE_BYTES];
  alignas(16) float lring[LRING][NPW][2][S];   // raw logits rows, LRING passes of every producer warp ahead of their use
                                               // (2-byte: a round's 8 rows packed into the first half of its group's slots)
  alignas(16) float2 scal_c[RING][NT];         // (c1, c0) of the tile's rows: rows 0..63 from CTA 0, 64..127 from CTA 1
  uint32_t scal_x[RING][NT];                   // chunk mask of the band (bits 0-7) | valid << 8 | x << 10 (= table-row byte offset)
  alignas(16) float scratch[NUM_EPI_WARPS][32][SCR_LD];   // per epilogue warp: lam[row][state of the chunk] (lane = state -> lane = row)
  alignas(16) int contrib[CBUF][NCHUNK][NH];   // per (chunk, row of THIS CTA): sum of jumps << 2 | min(jump count, 3), or the drift's float bits
  uint8_t band[S];                             // per state x: which of the 8 chunks hold a non-zero base rate (this launch's branch / mode)
  alignas(8) uint64_t full[STAGES];            // leader CTA: its NPW producer warps + 1 relayed arrival for the partner's
  uint64_t full_local[STAGES];                 // partner CTA: its NPW producer warps; the partner's idle MMA warp relays the phase
  uint64_t empty[STAGES];                      // multicast tcgen05.commit
  uint64_t scal_local[RING];                   // NPW local producer warps: this CTA's 64 rows of the tile have their scalars
  uint64_t scal_full[RING];                    // the local loader's arrival (scal_local seen) + the partner's bytes (DSMEM bulk copy)
  uint64_t lring_full_g[LRING][NSUB];          // one round of a 4-warp group: the bytes of its bulk copy
  uint64_t lring_free_g[LRING][NSUB];          // its 4 warps have their values in registers: the loader may refill the slots
  uint64_t tmem_full[ACC];                     // multicast tcgen05.commit
  uint64_t tmem_empty[ACC];                    // used in the leader CTA: 8 local + 8 remote epilogue warps
  uint64_t contrib_full[CBUF];                 // 4 local epilogue warps + the bytes of the partner's 4 warps
  uint64_t contrib_free_local[CBUF];           // the 2 local finalizer warps are done with this CTA's buffer
  uint64_t contrib_free_remote[CBUF];          // the 2 finalizer warps of the PARTNER are done with the partner's buffer
  uint32_t tmem_base;
};

static_assert(sizeof(Smem) + 1024 <= 232448, "shared memory budget of one CTA (227 KB) exceeded");
static_assert(NPW <= PASSES_PER_TILE, "every producer warp must own a pass in every tile");
static_assert(RING > STAGES + ACC + CBUF, "row-scalar ring shorter than the pipeline");

// TAULDR: tauLDR rates (else SDDM reverse_prob); KM: KM_JUMP / KM_CORR / KM_RATES / KM_DRIFT;
// HEAD: the rows' softmax numerators come from the truncated-logistic head (mu, log_scale per row) instead of logits;
// LT: element type of the logits, float, __nv_bfloat16 or __half (2-byte rows travel packed, 2*S bytes each, and are
// widened on the producers' shared-memory load; the arithmetic after that load is the fp32 kernel's).  A HEAD kernel reads
// no logits: LT is then the type of (mu, log_scale), float or __nv_bfloat16, widened on the loader warp's load
template <bool TAULDR, int KM, bool HEAD, typename LT = float>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) step_q_kernel(const Args a) {
  static_assert(!(HEAD && std::is_same<LT, __half>::value), "the fused head takes fp32 or bf16 (mu, log_scale)");
  constexpr uint32_t ROW_BYTES = S * sizeof(LT);
  extern __shared__ uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();       // state half owned by this CTA; rank 0 issues the MMAs
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  const int my_tiles = (a.num_tiles > pair) ? (a.num_tiles - pair + npairs - 1) / npairs : 0;
  constexpr bool SAMPLES = (KM != KM_RATES);     // contributions + finalizers exist

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&sm.full[i], NPW + 1);
      mbar_init(&sm.full_local[i], NPW);
      mbar_init(&sm.empty[i], 1);
    }
    for (int i = 0; i < RING; ++i) { mbar_init(&sm.scal_local[i], NPW); mbar_init(&sm.scal_full[i], 1); }
    for (int i = 0; i < LRING; ++i)
      for (int g = 0; g < NSUB; ++g) { mbar_init(&sm.lring_full_g[i][g], 1); mbar_init(&sm.lring_free_g[i][g], GSZ); }
    for (int i = 0; i < ACC; ++i) { mbar_init(&sm.tmem_full[i], 1); mbar_init(&sm.tmem_empty[i], 2 * NUM_EPI_WARPS); }
    for (int i = 0; i < CBUF; ++i) {
      mbar_init(&sm.contrib_full[i], NUM_EPI_WARPS / 2);
      mbar_init(&sm.contrib_free_local[i], 2);
      mbar_init(&sm.contrib_free_remote[i], 2);
    }
    fence_barrier_init();
  }
  // band of non-zero base rates of every state (exact zero pattern of the gathered table rows, union for the corrector)
  for (int x = threadIdx.x; x < S; x += NUM_THREADS) {
    const int bt = reinterpret_cast<const int*>(a.stat + ST_BANDT_OFF)[x];
    const int br = reinterpret_cast<const int*>(a.stat + ST_BANDR_OFF)[x];
    int lo, hi;
    if (TAULDR && km_corr(KM)) {
      lo = min(bt & 255, br & 255);
      hi = max((bt >> 8) & 255, (br >> 8) & 255);
    } else {
      const int b = TAULDR ? bt : br;
      lo = b & 255; hi = (b >> 8) & 255;
    }
    if (KM == KM_RATES) { lo = 0; hi = S - 1; }   // the rates output keeps the diagonal: every chunk is read
    uint32_t mask = 0;
    for (int c = 0; c < NCHUNK; ++c)
      if (hi >= c * JUMP_CHUNK && lo <= c * JUMP_CHUNK + JUMP_CHUNK - 1) mask |= 1u << c;
    sm.band[x] = (uint8_t)mask;
  }
  if (warp == MMA_WARP) tmem_alloc(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  load_qt_half<NUM_THREADS / 32>(a.tab, tmem, rank, warp, lane);
  tc_fence_before();
  cluster_sync_all();    // barriers initialised and both A halves resident before any cross-CTA traffic
  tc_fence_after();

  if (warp >= FIRST_PROD_WARP && warp < FIRST_PROD_WARP + NPW) {
    // ======================================================================== producers: 16 lanes per row, 2 rows per pass
    const int pw = warp - FIRST_PROD_WARP;
    const int half = lane >> 4, l16 = lane & 15;
    // lane owns k = 64c + 4*l16 .. +3 for c = 0..3; each softmax reduction is a 4-step butterfly inside the half-warp
    // (two independent rows per warp keep the pipes busy).  The raw logits rows arrive through a small smem ring that
    // cp.async.bulk fills two passes ahead, so no global-memory latency sits on the warp's critical path.
    const float* tabA = reinterpret_cast<const float*>(a.tab + TAB_A_OFF) + 4 * l16;
    uint64_t* const full_bar = rank == 0 ? &sm.full[0] : &sm.full_local[0];
    // passes of this CTA: pass P = 32 * tl + ps builds rows 2 ps, 2 ps + 1 of the CTA's 64 rows of its tl-th tile; warp pw
    // takes P = pw, pw + NPW, ..  The states are fetched two passes of the warp ahead;
    // every position is derived from the one pass counter (row indices fit 32 bits: a row is 1 KB of logits).
    const int total_passes = my_tiles * PASSES_PER_TILE;
    const uint32_t tile_rows = (uint32_t)npairs * NT;
    const uint32_t row00 = (uint32_t)pair * NT + rank * NH;      // first row of this CTA's half of its first tile
    const uint32_t rows32 = (uint32_t)a.rows;
    auto row_of = [&](int Pq) -> uint32_t { return row00 + (uint32_t)(Pq >> 5) * tile_rows + 2u * (uint32_t)(Pq & 31); };
    const uint32_t scal_c_p = smem_u32(&sm.scal_c[0][0]), scal_x_p = smem_u32(&sm.scal_x[0][0]);

    // States: two passes of this warp ahead, into registers.
    auto fetch = [&](int Pq) -> int {
      int xv = -1;
      if (Pq < total_passes) {
        const uint32_t g = row_of(Pq) + half;
        if (g < rows32) xv = __ldg(a.x_eval + g);
      }
      return xv;
    };
    // Logits (HEAD: the rows' head records): the loader warp (light group) refills the ring slots of this warp's group as
    // soon as its 4 warps report that the current pass has its values in registers (lring_free_g).
    int P = pw;
    int x_cur = fetch(P);
    int x_n1 = fetch(P + NPW);
    float4 t4[4];
    {
      const size_t xo = (size_t)(x_cur < 0 ? 0 : x_cur) << 8;
#pragma unroll
      for (int c = 0; c < 4; ++c) t4[c] = __ldg(reinterpret_cast<const float4*>(tabA + xo + 64 * c));
    }
    // The row reductions (sum e, sum e*Q[.,x]) and the row scalars of a pass are FINISHED IN THE NEXT PASS: its per-lane
    // partial sums are carried over, their butterflies run next to the next pass's row-maximum butterfly, and the
    // scalar records follow there.  Only the operand rows (what the MMA waits for) are completed inside the pass itself.
    // Barrier arrivals (operands: full, scalars: scal_full) happen once per warp and tile, after the warp's last pass in it.
    float p_sum = 1.f, p_dot = 0.f;
    int p_x = 0, p_idx = 0, p_slot = 0;
    bool p_ok = false, p_have = false, p_last = false;
    auto finish_prev = [&]() {          // p_sum / p_dot hold the reduced values
      if (!p_have) return;
      if (l16 == 0) {   // one lane per half-warp: the row's RAW sums and state; the loader warp turns the tile's 64 records
                        // into the row scalars (reciprocals, rate scale, band mask) and forwards them to the partner CTA
        const uint32_t sx = (p_ok ? (1u << 8) : 0u) | ((uint32_t)p_x << 10);
        sts64(scal_c_p + (uint32_t)p_idx * 8u, __float_as_uint(p_sum), __float_as_uint(p_dot));
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(scal_x_p + (uint32_t)p_idx * 4u), "r"(sx) : "memory");
      }
      if (p_last) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.scal_local[p_slot]);
      }
      p_have = false;
    };
    int ring_n = 0;              // passes of this warp so far: slot ring_n % LRING, phase ring_n / LRING
    int last_tl = -1;
#pragma unroll 1
    while (P < total_passes) {
      const int tl = P >> 5, ps = P & 31;
      const int st = tl % STAGES;
      const int slot = tl % RING;
      const bool ok = x_cur >= 0;
      const int x = ok ? x_cur : 0;
      const bool last_in_tile = ps + NPW >= PASSES_PER_TILE;     // this warp's next pass belongs to another tile
      const int rslot = ring_n % LRING;
      mbar_wait(&sm.lring_full_g[rslot][pw / GSZ], (uint32_t)((ring_n / LRING) & 1));
      const int r = 2 * ps + half;
      float v[16];
      float ml = 0.f;
      if (HEAD) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {     // previous pass's reductions: independent of the head arithmetic below
          p_sum += __shfl_xor_sync(0xffffffffu, p_sum, o);
          if (!TAULDR) p_dot += __shfl_xor_sync(0xffffffffu, p_dot, o);
        }
        // the row's head record (8 floats made by the loader warp): two broadcast 128-bit loads per half-warp
        const uint32_t hsrc = smem_u32(&sm.lring[rslot][pw][half][0]);
        const float4 h0 = lds128(hsrc), h1 = lds128(hsrc + 16);
        ++ring_n;
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.lring_free_g[rslot][pw / GSZ]);
        const HeadRec hr = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        head_numerators_rec(hr, a.head_fix != 0, l16, v);
      } else {
        if constexpr (sizeof(LT) == 2) {
          // the round's 8 2-byte rows lie packed from the group's first slot: this half's row is number 2 * (pw % GSZ) + half;
          // lane l16 widens the same elements 64c + 4*l16 .. +3 as in the fp32 kernel, one 64-bit load each
          const uint32_t src = smem_u32(&sm.lring[rslot][pw - pw % GSZ][0][0]) + (uint32_t)(2 * (pw % GSZ) + half) * ROW_BYTES +
                               8 * l16;
#pragma unroll
          for (int c = 0; c < 4; ++c) widen2x4<LT>(lds64(src + 128 * c), v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        } else {
          const uint32_t src = smem_u32(&sm.lring[rslot][pw][half][4 * l16]);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 q4 = lds128(src + 256 * c);
            v[4 * c] = q4.x; v[4 * c + 1] = q4.y; v[4 * c + 2] = q4.z; v[4 * c + 3] = q4.w;
          }
        }
        ++ring_n;
        __syncwarp();            // every lane has its values: the group's slots may be refilled once its 4 warps say so
        if (lane == 0) mbar_arrive(&sm.lring_free_g[rslot][pw / GSZ]);
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
      if (tl != last_tl) {       // first pass of this warp in a new tile: the tile's operand stage must be free
        mbar_wait<POLL_LONG>(&sm.empty[st], (uint32_t)(((tl / STAGES) & 1) ^ 1));
        last_tl = tl;
      }
      const uint32_t stage_s = smem_u32(sm.stage[st]);
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
          const float2 op = TAULDR ? fmul2(ex, tq) : ex;   // tauLDR operand: e_k / (Q[k,x] + eps); 1/sum applied by the epilogue
          v[4 * c + e] = op.x; v[4 * c + e + 1] = op.y;
        }
      }
      const float2 s01 = fadd2(sum2[0], sum2[1]), s23 = fadd2(sum2[2], sum2[3]), sall = fadd2(s01, s23);
      const float sum = sall.x + sall.y;
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
      if (__any_sync(0xffffffffu, !ok)) {
        if (!ok) {
#pragma unroll
          for (int k = 0; k < 16; ++k) v[k] = 0.f;
        }
      }
      store_operand_row<KBLOCK_BYTES, SPLIT_BYTES>(stage_s, r, l16, v);
      // this pass's partial sums and row identity travel to the next pass (finish_prev)
      p_sum = sum; p_dot = dot;
      p_x = x; p_ok = ok; p_idx = slot * NT + (int)rank * NH + r; p_slot = slot; p_last = last_in_tile; p_have = true;
      if (last_in_tile) {      // the warp's operand rows of this tile are in place
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar + st);
      }
      x_cur = x_n1;
      x_n1 = fetch(P + 2 * NPW);
      P += NPW;
    }
    // the last pass's reductions and row scalars
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      p_sum += __shfl_xor_sync(0xffffffffu, p_sum, o);
      if (!TAULDR) p_dot += __shfl_xor_sync(0xffffffffu, p_dot, o);
    }
    finish_prev();
  } else if (warp == MMA_WARP + 1) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));
    // ======================================================================== loader: everything the producers would otherwise
    // issue themselves.  Lane g < NSUB serves producer warps 4g .. 4g+3: ONE 8 KB bulk copy per round into their four ring
    // slots as soon as all four have released them (a bulk-copy issue costs the issuing thread a few hundred cycles: off
    // the producers' critical path).  Lane 31 forwards each finished tile's 64 row-scalar records to the partner CTA as
    // two DSMEM bulk copies.  Nobody blocks: the warp polls, every lane acts on what is ready.
    {
      const bool contiguous = (a.ld == S) && (a.batch_stride == (long long)a.D * S);
      const LT* const logits = static_cast<const LT*>(a.logits);
      auto row_ptr = [&](long long g) -> const LT* {
        if (contiguous) return logits + g * S;
        const uint32_t n = (uint32_t)g / (uint32_t)a.D, d = (uint32_t)g - n * (uint32_t)a.D;
        return logits + (long long)n * a.batch_stride + (long long)d * a.ld;
      };
      const uint32_t scal_c_p = smem_u32(&sm.scal_c[0][rank * NH]), scal_x_p = smem_u32(&sm.scal_x[0][rank * NH]);
      const uint32_t scal_c_remote = mapa(scal_c_p, rank ^ 1u), scal_x_remote = mapa(scal_x_p, rank ^ 1u);
      const uint32_t scal_full_remote = mapa(smem_u32(&sm.scal_full[0]), rank ^ 1u);
      const long long tile_rows = (long long)npairs * NT;
      const long long row00 = (long long)pair * NT + (int)rank * NH;      // first row of this CTA's half of its first tile
      const int total = my_tiles * PASSES_PER_TILE;
      const bool group_lane = !HEAD && lane < NSUB;
      // HEAD: lanes 8g .. 8g+7 make the head records of the 8 rows of group g's round (lane & 7 = row of the round); the
      // (mu, log_scale) of the next round are loaded one round ahead
      const bool head_lane = HEAD && lane < 2 * GSZ * NSUB;
      const int hg = lane / (2 * GSZ), hi = lane % (2 * GSZ);
      float h_mu = 0.f, h_ls = 0.f;
      auto head_load = [&](int round) {
        h_mu = 0.f; h_ls = 0.f;
        const int Pq = round * NPW + GSZ * hg + (hi >> 1);
        if (!head_lane || Pq >= total) return;
        const long long g = row00 + (long long)(Pq >> 5) * tile_rows + 2 * (Pq & 31) + (hi & 1);
        if (g >= a.rows) return;
        long long src = g;
        if (a.head_bs != (long long)a.D) {   // (N, 2D) network output viewed as two (N, D) halves
          const uint32_t n = (uint32_t)g / (uint32_t)a.D;
          src = (long long)n * a.head_bs + ((uint32_t)g - n * (uint32_t)a.D);
        }
        h_mu = ld_logit(static_cast<const LT*>(a.head_mu) + src);
        h_ls = ld_logit(static_cast<const LT*>(a.head_ls) + src);
      };
      if (HEAD) head_load(0);
      int grp = 0;               // (lanes < NSUB) next round of the lane's group: passes NPW * grp + 4 * lane .. + 3
      int fwd = 0;               // (lane 31) next tile whose scalars go to the partner
      while (true) {
        const bool more_f = lane == 31 && fwd < my_tiles;
        const bool more_g = group_lane && grp * NPW + GSZ * lane < total;
        const bool more_h = head_lane && grp * NPW + GSZ * hg < total;
        if (!__any_sync(0xffffffffu, more_f || more_g || more_h) && fwd >= my_tiles) break;
        bool did = false;
        if (HEAD) {
          // every group's slot of this round must be free (the three groups advance in lockstep here: one test each)
          const int hslot = grp % LRING;
          const bool free_ok = !more_h || grp < LRING || mbar_test(&sm.lring_free_g[hslot][hg], (uint32_t)((grp / LRING - 1) & 1));
          if (__any_sync(0xffffffffu, more_h) && __all_sync(0xffffffffu, free_ok)) {
            if (more_h) {
              const HeadRec hr = head_row_record(h_mu, h_ls, a.head_fix != 0);
              const uint32_t dst = smem_u32(&sm.lring[hslot][GSZ * hg + (hi >> 1)][hi & 1][0]);
              sts128(dst, make_float4(hr.mu, hr.sc, hr.off0, hr.kap));
              sts128(dst + 16, make_float4(hr.A, hr.B, hr.c, 0.f));
            }
            head_load(grp + 1);
            __syncwarp();
            if (more_h && hi == 0) mbar_arrive(&sm.lring_full_g[hslot][hg]);
            ++grp;
            did = true;
          }
        }
        const int gslot = grp % LRING;
        if (more_g && (grp < LRING || mbar_test(&sm.lring_free_g[gslot][lane], (uint32_t)((grp / LRING - 1) & 1)))) {
          // round grp of group `lane`: passes P0 .. P0 + 3 (4-aligned: never across a tile boundary) = 8 consecutive rows;
          // rows past the end of the batch are not copied
          const int P0 = grp * NPW + GSZ * lane;
          auto seg_rows = [&](long long r0) -> long long {
            long long nrows = 2LL * GSZ;
            if (r0 + nrows > a.rows) nrows = a.rows > r0 ? a.rows - r0 : 0;
            return nrows;
          };
          const long long rA = row00 + (long long)(P0 >> 5) * tile_rows + 2 * (P0 & 31);
          const long long nA = seg_rows(rA);
          uint64_t* gbar = &sm.lring_full_g[gslot][lane];
          mbar_arrive_expect_tx(gbar, (uint32_t)nA * ROW_BYTES);
          uint8_t* dA = reinterpret_cast<uint8_t*>(&sm.lring[gslot][GSZ * lane][0][0]);   // row rr of the round at rr * ROW_BYTES
          if (contiguous) {
            if (nA > 0) bulk_g2s(dA, logits + rA * S, (uint32_t)nA * ROW_BYTES, gbar);
          } else {               // strided logits: one copy per row
            for (long long rr = 0; rr < nA; ++rr) bulk_g2s(dA + rr * ROW_BYTES, row_ptr(rA + rr), ROW_BYTES, gbar);
          }
          ++grp;
          did = true;
        }
        // (fwd is kept by every lane; every lane tests the barrier itself - its own acquire of the producers' records - and all
        // lanes turn the raw records into the row scalars; lane 31 issues the copies)
        const int fslot = fwd % RING;
        const bool f_ready = fwd < my_tiles && __all_sync(0xffffffffu, mbar_test(&sm.scal_local[fslot], (uint32_t)((fwd / RING) & 1)));
        if (f_ready) {
          const float hb = (KM == KM_RATES) ? 1.0f : a.h * a.beta;   // rates-only ignores the step length
#pragma unroll
          for (int rr = 0; rr < NH / 32; ++rr) {
            const uint32_t idx = (uint32_t)fslot * NT + (uint32_t)(32 * rr + lane);       // (scal_*_p already point at this CTA's half)
            float p_sum, p_dot;
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(p_sum), "=f"(p_dot) : "r"(scal_c_p + idx * 8u));
            uint32_t sx;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(sx) : "r"(scal_x_p + idx * 4u));
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
            sx |= (uint32_t)sm.band[(sx >> 10) & 255u];
            sts64(scal_c_p + idx * 8u, __float_as_uint(c1), __float_as_uint(c0));
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(scal_x_p + idx * 4u), "r"(sx) : "memory");
          }
          fence_proxy_async();     // the records are read by a bulk copy (async proxy)
          __syncwarp();
        }
        if (more_f) {
          const int slot = fslot;
          if (f_ready) {
            // local consumers: this arrival + the partner's 768 bytes complete the phase
            mbar_arrive_expect_tx(&sm.scal_full[slot], SCAL_TX_BYTES);
            const uint32_t bar = scal_full_remote + (uint32_t)slot * 8u;
            bulk_s2cluster(scal_c_remote + (uint32_t)slot * (NT * 8u), scal_c_p + (uint32_t)slot * (NT * 8u), NH * 8u, bar);
            bulk_s2cluster(scal_x_remote + (uint32_t)slot * (NT * 4u), scal_x_p + (uint32_t)slot * (NT * 4u), NH * 4u, bar);
          }
        }
        if (f_ready) { ++fwd; did = true; }
        if (!__any_sync(0xffffffffu, did)) asm volatile("nanosleep.u32 32;");
      }
    }
    __syncwarp();
  } else if (warp >= FIN_WARP0) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));
    // ======================================================================== finalizers: lane = row of this CTA
    if constexpr (SAMPLES) {
      const int r = (warp - FIN_WARP0) * 32 + lane;          // row of the tile's 64 that this CTA produced
      const uint32_t cfree_remote = mapa(smem_u32(&sm.contrib_free_remote[0]), rank ^ 1u);
      RowStats stt = {0, 0, 0, 0, 0};
      for (int i = 0; i < my_tiles; ++i) {
        const int tile = pair + i * npairs, slot = i % RING, cb = i % CBUF;
        const long long g = (long long)tile * NT + (long long)rank * NH + r;
        mbar_wait<POLL_LONG>(&sm.scal_full[slot], (i / RING) & 1);
        const uint32_t sx = sm.scal_x[slot][rank * NH + r];
        const int x = (int)((sx >> 10) & 255u);
        const bool valid = (sx >> 8) & 1u;
        int xb = x;
        if (a.x_base && valid) xb = __ldg(a.x_base + g);
        mbar_wait<POLL_LONG>(&sm.contrib_full[cb], (i / CBUF) & 1);
        int jump = 0, cnt = 0;
        float drift = 0.f;
#pragma unroll
        for (int c = 0; c < NCHUNK; ++c) {
          const int v = sm.contrib[cb][c][r];
          // (the count of a chunk is saturated at 3: only "none / one / several" of the row's total matters downstream)
          if (KM == KM_DRIFT) drift += __int_as_float(v); else { jump += v >> 2; cnt += v & 3; }
        }
        if (valid) {
          if (KM == KM_DRIFT) {
            // sampling.py:433-453: x' = clip(x + round_half_even(h/2 * sum_s rr_s (s - x)))
            const int ch = (int)rintf(0.5f * drift);
            int xn = x + ch;
            xn = xn < 0 ? 0 : (xn > S - 1 ? S - 1 : xn);
            a.x_out[g] = xn;
            stt.changed_base += (xn != x);
            stt.changed_eval += (xn != x);
            stt.nonzero += (ch != 0);
          } else {
            a.x_out[g] = finalize_jump(xb, x, jump, cnt, a.reject_multi, S, stt);
          }
        }
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&sm.contrib_free_local[cb]);
          mbar_arrive_cluster_relaxed(cfree_remote + (uint32_t)cb * 8u);
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
      relay_full<STAGES, POLL_LONG>(sm.full_local, sm.full, my_tiles);
    }
    __syncwarp();
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
    // ======================================================================== epilogue: lane = state
    const int ew = warp - FIRST_EPI_WARP;         // (FIRST_EPI_WARP is a multiple of 4: ew & 3 is the warp's TMEM quadrant)
    const int q = ew & 3;                         // TMEM quadrant -> states rank*128 + 32q + lane = one chunk of the map
    const uint32_t h = (uint32_t)(ew >> 2);       // accumulator columns [64h, 64h+64) are the rows CTA h produced
    const int chunk = (int)rank * 4 + q;
    const int cs = chunk * JUMP_CHUNK;            // first state of the chunk
    const int s_mine = cs + lane;
    const uint32_t cbase = (uint32_t)chunk << 16; // Philox call base of this chunk
    const uint32_t tempty_dst = mapa(smem_u32(&sm.tmem_empty[0]), 0);
    // record slot of this chunk: shared::cta address when this CTA produced the rows, else in the partner's window
    const uint32_t contrib_dst = (h == rank) ? smem_u32(&sm.contrib[0][chunk][0]) : mapa(smem_u32(&sm.contrib[0][chunk][0]), h);
    const uint32_t cfull_dst = mapa(smem_u32(&sm.contrib_full[0]), h);
    uint64_t* const cfree_wait = (h == rank) ? &sm.contrib_free_local[0] : &sm.contrib_free_remote[0];
    // Table rows are addressed as static blob + 32-bit offset: the blob is 2 MiB aligned, so the upper address word is
    // a constant and the lower word is one add.  Offset of a row = table + x * 1024 (the row scalar carries x << 10):
    // zero-diagonal R_b^T / R_b for the rates (the diagonal-keeping copies for the rates output), R_b[x][.] for the
    // corrector add, the zero row for chunks outside the band of x.
    const float* stat_lane = reinterpret_cast<const float*>(a.stat) + s_mine;
    constexpr uint32_t TAB_R = (uint32_t)((KM == KM_RATES) ? (TAULDR ? ST_RBT_OFF : ST_RB_OFF) : (TAULDR ? ST_RBZT_OFF : ST_RBZ_OFF));
    auto stat_ptr = [&](uint32_t off) -> const float* { return stat_lane + (off >> 2); };   // one widening multiply-add
    const uint32_t chunkbit = 1u << chunk;
    const uint32_t scr_p = smem_u32(&sm.scratch[ew][0][0]);
    const float hb = a.h * a.beta;

    for (int i = 0; i < my_tiles; ++i) {
      const int tile = pair + i * npairs;
      const int slot = i % RING, b = i % ACC, cb = i % CBUF;
      mbar_wait(&sm.scal_full[slot], (i / RING) & 1);
      mbar_wait(&sm.tmem_full[b], (i / ACC) & 1);
      tc_fence_after();
      if (SAMPLES) mbar_wait(cfree_wait + cb, ((i / CBUF) & 1) ^ 1);
#pragma unroll 1
      for (int bb = 0; bb < 2; ++bb) {
        const int col = (int)h * NH + 32 * bb;                         // tile column (= tile row) of this batch's row 0
        const long long g0 = (long long)tile * NT + col;               // its global row
        const uint32_t sx_p = smem_u32(&sm.scal_x[slot][col]);
        const uint32_t sc_p = smem_u32(&sm.scal_c[slot][col]);
        uint32_t acc[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + TM_ACC + b * NT + col, acc);
        uint32_t sxl;            // row scalar of row `lane` of the batch
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(sxl) : "r"(sx_p + 4 * lane));
        if constexpr (KM == KM_RATES) {
          // rates output: lane = state.  Base-rate entries R[s_mine, x_row] of the 32 rows: 32 coalesced 128-byte loads
          // (lane L prepares the table offset of row L, a shuffle hands it to all).
          const uint32_t offl = TAB_R + (sxl & 0x3FC00u);
          float R[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) R[j] = __ldg(stat_ptr(__shfl_sync(0xffffffffu, offl, j)));
          tmem_ld_wait();
          if (bb == 1) {           // the accumulator has been read: hand the buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster_relaxed(tempty_dst + (uint32_t)b * 8u);
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float c1, c0;
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(c1), "=f"(c0) : "r"(sc_p + 8 * j));
            const float ratio = fmaf(__uint_as_float(acc[j]), c1, c0);
            const float rfull = TAULDR ? a.beta * R[j] * ratio : ratio * (a.beta * R[j]);
            const long long g = g0 + j;
            if (g < a.rows) {
              if (a.rr_out) a.rr_out[g * S + s_mine] = rfull;
              if (a.ratio_out) a.ratio_out[g * S + s_mine] = ratio;
            }
          }
        } else {
          // Sampling modes work with lane = ROW: lane L reads the 32 base-rate entries of ITS row's state for this chunk
          // (one 128-byte piece of the zero-diagonal table row x, four 256-bit loads; the zero row when the chunk lies
          // outside the band of non-zero rates of x), the accumulator is transposed through the warp's scratch, and
          // lam[row, s] = D[s, row] * R[x_row][s] is formed where the prefix sums need it.
          constexpr bool UNSCALED = TAULDR && !km_corr(KM);
          const bool inband = (sxl & chunkbit) != 0u;
          float R[32];
          {
            const uint8_t* rrow = a.stat + (inband ? TAB_R + (sxl & 0x3FC00u) : (uint32_t)ST_ZERO_OFF) + cs * 4;
#pragma unroll
            for (int c = 0; c < 4; ++c) ldg256(rrow + 32 * c, &R[8 * c]);
          }
          // the row's Philox draw (count uniform + first three pick uniforms) does not depend on the data: computed in the
          // shadow of the loads
          const uint64_t grow = (uint64_t)(a.row_offset + g0 + lane);
          Philox4 p0 = {{0u, 0u, 0u, 0u}};
          if constexpr (KM == KM_JUMP || KM == KM_CORR) p0 = philox_rowjump(grow, cbase, a.offset, a.seed);
          tmem_ld_wait();
          if (bb == 1) {           // the accumulator has been read: hand the buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster_relaxed(tempty_dst + (uint32_t)b * 8u);
          }
          // transpose through the warp's scratch: lane = state -> lane = row (row `lane` of the batch, the chunk's 32 states)
          __syncwarp();          // the previous batch's reads of the scratch are done
#pragma unroll
          for (int j = 0; j < 32; ++j) sts32(scr_p + (uint32_t)(j * SCR_LD + lane) * 4u, __uint_as_float(acc[j]));
          __syncwarp();
          float p[32];
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(p[2 * c]), "=f"(p[2 * c + 1]) : "r"(scr_p + (uint32_t)(lane * SCR_LD + 2 * c) * 4u));
          }
          // lam[s, row] (zero at s == x through the zero-diagonal tables).  tauLDR without corrector: the row's scale c1
          // is applied to the chunk total only (the picks are scale-invariant); otherwise per element.
          float sc1 = 0.f, sc0 = 0.f;
          asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(sc1), "=f"(sc0) : "r"(sc_p + 8 * lane));
          if constexpr (!UNSCALED) {
#pragma unroll
            for (int s2 = 0; s2 < 32; ++s2) p[s2] = fmaf(p[s2], sc1, sc0) * R[s2];
            if constexpr (km_corr(KM)) {
              const uint8_t* crow = a.stat + (inband ? (uint32_t)ST_RBZ_OFF + (sxl & 0x3FC00u) : (uint32_t)ST_ZERO_OFF) + cs * 4;
#pragma unroll
              for (int c = 0; c < 4; ++c) ldg256(crow + 32 * c, &R[8 * c]);
#pragma unroll
              for (int s2 = 0; s2 < 32; ++s2) p[s2] = fmaf(hb, R[s2], p[s2]);
            }
          }
          const int xl = (int)((sxl >> 10) & 255u);
          int2 rec = make_int2(0, 0);
          if constexpr (KM == KM_DRIFT) {
            // sum_s rr_s (s - x) over this chunk (sampling.py:433-453)
            float dsum = 0.f;
#pragma unroll
            for (int s2 = 0; s2 < 32; ++s2) {
              const float lam = UNSCALED ? p[s2] * R[s2] : p[s2];
              dsum = fmaf(lam, (float)(cs + s2 - xl), dsum);
            }
            if constexpr (UNSCALED) dsum *= sc1;
            rec.x = __float_as_int(dsum);
          } else {
            // sequential fp32 prefix sums over the chunk's states (the oracle's summation order)
            if constexpr (UNSCALED) {     // product and running sum in one fused multiply-add per state
              p[0] *= R[0];
#pragma unroll
              for (int s2 = 1; s2 < 32; ++s2) p[s2] = fmaf(p[s2], R[s2], p[s2 - 1]);
            } else {
#pragma unroll
              for (int s2 = 1; s2 < 32; ++s2) p[s2] += p[s2 - 1];
            }
            float tot = p[31];
            if constexpr (UNSCALED) tot *= sc1;
            int K = poisson_from_unit(tot, u32_to_unit(p0.w[0]));
            K = K > JUMP_PICK_CAP ? JUMP_PICK_CAP : K;
            rec.y = K;
            // Picks: first state whose prefix sum exceeds v * total.  The picks of the batch's 32 rows are dealt to the
            // 32 lanes (a row with K picks would otherwise keep 31 lanes idle for K rounds): lane = row parks its prefix
            // sums in its scratch row, a warp scan of K numbers the picks, and lane i resolves pick base + i of whatever
            // row it belongs to (row found by a 5-shuffle search over the scan, uniforms fetched from the row's lane).
            int jump = 0;
            const uint32_t any = __ballot_sync(0xffffffffu, K > 0);
            // Few picks per row (the common case once the schedule has left its first tenth): every lane resolves the
            // picks of ITS row from the prefix sums it holds in registers - the pick is the number of prefix sums <= the
            // target, 31 independent compares, no shared memory, no shuffles; one round per pick, uniforms of call 0.
            int maxK = 0;
            if (any) maxK = __reduce_max_sync(0xffffffffu, K);
            if (any && maxK <= REGPICK_MAX) {
              const float ptot = p[31];
#pragma unroll
              for (int j = 0; j < REGPICK_MAX; ++j) {
                if (j < maxK) {
                  const uint32_t w = p0.w[1 + j];   // the three pick uniforms of the row's Philox call
                  float T = fminf(u32_to_unit(w), 0.99999994f) * ptot;
                  // the product can round up to the total itself: then the pick is the last state with a positive rate
                  if (T >= ptot) T = __uint_as_float(__float_as_uint(ptot) - 1u);
                  int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#pragma unroll
                  for (int s2 = 0; s2 < 28; s2 += 4) {
                    c0 += (p[s2] <= T) ? 1 : 0; c1 += (p[s2 + 1] <= T) ? 1 : 0;
                    c2 += (p[s2 + 2] <= T) ? 1 : 0; c3 += (p[s2 + 3] <= T) ? 1 : 0;
                  }
                  c0 += (p[28] <= T) ? 1 : 0; c1 += (p[29] <= T) ? 1 : 0; c2 += (p[30] <= T) ? 1 : 0;
                  if (K > j) jump += cs + (c0 + c1) + (c2 + c3) - xl;
                }
              }
            } else if (any) {
              __syncwarp();
#pragma unroll
              for (int c = 0; c < 16; ++c)
                sts64(scr_p + (uint32_t)(lane * SCR_LD + 2 * c) * 4u, __float_as_uint(p[2 * c]), __float_as_uint(p[2 * c + 1]));
              // column 32 of the scratch row: the row's jump sum (shared-memory reduction target)
              asm volatile("st.shared.u32 [%0], %1;" ::"r"(scr_p + (uint32_t)(lane * SCR_LD + 32) * 4u), "r"(0) : "memory");
              int incl = K;
#pragma unroll
              for (int o = 1; o < 32; o <<= 1) {
                const int n = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += n;
              }
              const int npick = __shfl_sync(0xffffffffu, incl, 31);
              __syncwarp();
              for (int base = 0; base < npick; base += 32) {
                const int idx = base + lane;
                // row of pick idx: the first lane whose inclusive count exceeds idx
                int r = 0;
#pragma unroll
                for (int stp = 16; stp >= 1; stp >>= 1) {
                  const int v = __shfl_sync(0xffffffffu, incl, (r + stp - 1) & 31);
                  if (v <= idx) r += stp;
                }
                r &= 31;                                  // lanes beyond the last pick (idx >= npick) walk a valid row
                const int j = idx - (__shfl_sync(0xffffffffu, incl, r) - __shfl_sync(0xffffffffu, K, r));
                const uint32_t w1 = __shfl_sync(0xffffffffu, p0.w[1], r), w2 = __shfl_sync(0xffffffffu, p0.w[2], r),
                               w3 = __shfl_sync(0xffffffffu, p0.w[3], r);
                if (idx < npick) {
                  uint32_t w = j == 0 ? w1 : (j == 1 ? w2 : w3);
                  if (j >= 3) {
                    const int jj = j - 3;
                    const Philox4 pc = philox_rowjump((uint64_t)(a.row_offset + g0 + r), cbase + 1u + (uint32_t)(jj >> 2), a.offset, a.seed);
                    w = philox_word(pc, jj & 3);
                  }
                  const uint32_t prow = scr_p + (uint32_t)(r * SCR_LD) * 4u;
                  const float ptot = lds32(prow + 31 * 4);
                  float T = fminf(u32_to_unit(w), 0.99999994f) * ptot;
                  // the product can round up to the total itself: then the pick is the last state with a positive rate
                  if (T >= ptot) T = __uint_as_float(__float_as_uint(ptot) - 1u);
                  // two rounds of independent loads: 7 splitters of stride 4, then the 3 entries below the next one
                  int c1 = 0;
#pragma unroll
                  for (int m = 0; m < 7; ++m) c1 += (lds32(prow + 4 * (4 * m + 3)) <= T) ? 1 : 0;
                  const uint32_t p2 = prow + 16 * c1;
                  const int c2 = ((lds32(p2) <= T) ? 1 : 0) + ((lds32(p2 + 4) <= T) ? 1 : 0) + ((lds32(p2 + 8) <= T) ? 1 : 0);
                  uint32_t sxr;
                  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(sxr) : "r"(sx_p + 4 * r));
                  const int dj = cs + 4 * c1 + c2 - (int)((sxr >> 10) & 255u);
                  asm volatile("red.shared.add.s32 [%0], %1;" ::"r"(prow + 32 * 4), "r"(dj) : "memory");
                }
              }
              __syncwarp();
              asm volatile("ld.shared.s32 %0, [%1];" : "=r"(jump) : "r"(scr_p + (uint32_t)(lane * SCR_LD + 32) * 4u));
            }
            rec.x = jump;
          }
          // the record of (row `lane`, this chunk) goes to the CTA that produced the row
          const uint32_t roff = (uint32_t)cb * (NCHUNK * NH * 4) + (uint32_t)(32 * bb + lane) * 4u;
          const uint32_t word = (KM == KM_DRIFT) ? (uint32_t)rec.x : (((uint32_t)rec.x << 2) | (uint32_t)(rec.y > 3 ? 3 : rec.y));
          if (h == rank) {
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(contrib_dst + roff), "r"(word) : "memory");
          } else {
            st_async_cluster_b32(contrib_dst + roff, word, cfull_dst + (uint32_t)cb * 8u);
          }
        }
      }
      if (SAMPLES && h == rank) {
        __syncwarp();
        if (lane == 0) {
          // warp 0 also announces the bytes the partner's four warps will deliver for this tile
          if (q == 0) mbar_arrive_expect_tx(&sm.contrib_full[cb], CONTRIB_TX_BYTES);
          else mbar_arrive(&sm.contrib_full[cb]);
        }
      }
    }
  }
  pair_teardown(warp == MMA_WARP, tmem);
}

}  // namespace tcq

int launch_step_tcq(const ctdd_step_params* p, cudaStream_t st) {
  using namespace tcq;
  static tc::PairLaunchState launch_state;
  const size_t smem_bytes = sizeof(Smem) + 1024;
  typedef void (*kern_t)(const tc::Args);
#define CTDD_TCQ_ROW(T, H, LT)                                                                                            \
  step_q_kernel<T, tc::KM_JUMP, H, LT>, step_q_kernel<T, tc::KM_CORR, H, LT>, step_q_kernel<T, tc::KM_RATES, H, LT>,    \
      step_q_kernel<T, tc::KM_DRIFT, H, LT>
  static const kern_t kerns[40] = {CTDD_TCQ_ROW(false, false, float), CTDD_TCQ_ROW(true, false, float),
                                     CTDD_TCQ_ROW(false, true, float), CTDD_TCQ_ROW(true, true, float),
                                     CTDD_TCQ_ROW(false, false, __nv_bfloat16), CTDD_TCQ_ROW(true, false, __nv_bfloat16),
                                     CTDD_TCQ_ROW(false, true, __nv_bfloat16), CTDD_TCQ_ROW(true, true, __nv_bfloat16),
                                     CTDD_TCQ_ROW(false, false, __half), CTDD_TCQ_ROW(true, false, __half)};
#undef CTDD_TCQ_ROW
  if (reinterpret_cast<uintptr_t>(p->tc_static) % tc::ST_ALIGN) {
    set_error("ctdd_reverse_step: tc_static must be aligned to ctdd_tc_static_align() = %zu bytes", tc::ST_ALIGN);
    return 2;
  }
  tc::Args a = tc::make_args(p);
  if (a.rows >= (1LL << 31)) {      // the producers index rows with 32 bits (2^31 rows would be 2 TB of logits)
    set_error("ctdd_reverse_step: N * D = %lld rows exceed the tensor path's 2^31 - 1", a.rows);
    return 2;
  }
  a.num_tiles = (int)((a.rows + NT - 1) / NT);
  const int pairs = tc::pair_count(launch_state, "ctdd_reverse_step", kerns, smem_bytes, a.num_tiles);
  if (!pairs) return 1;
  // rows of kerns: fp32 logits, fused head on fp32 (mu, log_scale), bf16 logits, fused head on bf16 (mu, log_scale),
  // fp16 logits (the head takes no fp16: ctdd_reverse_step refuses it)
  const int dt = p->head != CTDD_HEAD_LOGITS ? p->head_dtype : p->logits_dtype;
  const int ki = ((p->branch == CTDD_BRANCH_TAULDR) ? 1 : 0) + (p->head != CTDD_HEAD_LOGITS ? 2 : 0) +
                 (dt == CTDD_DTYPE_BF16 ? 4 : (dt == CTDD_DTYPE_F16 ? 8 : 0));
  int kj = 0;
  if (p->mode == CTDD_MODE_RATES_ONLY) kj = 2;
  else if (p->mode == CTDD_MODE_TAU_LEAP_CORR) kj = 1;
  else if (p->mode == CTDD_MODE_MIDPOINT_DRIFT) kj = 3;
  kerns[4 * ki + kj]<<<2 * pairs, NUM_THREADS, smem_bytes, st>>>(a);
  CTDD_CHECK_LAUNCH("step_q_kernel");
  return 0;
}

}  // namespace ctdd

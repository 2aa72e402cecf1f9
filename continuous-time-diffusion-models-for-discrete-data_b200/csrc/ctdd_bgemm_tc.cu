// Per-sample contraction on tcgen05 for the loss terms (S == 256):
//     out[b, d, n] = sum_k X[b, d, k] * M[b, n, k]          b < B samples, d < D rows per sample, n, k < 256
// fp32 in and out, 3 x BF16 split precision (hi*hi + hi*mid + mid*hi), fp32 accumulation in tensor memory.
// This is the two/three (B*D x S)(S x S) products with a PER-SAMPLE q_{t|0} of the CT-ELBO / SDDM-ELBO / ratio-matching
// losses (reference lib/losses/losses.py:121-181, lib/models/model_utils.py:41-46): forward u = A Q (M = Q^T) and
// backward dL/dA = dL/du Q^T (M = Q).
//
// Same skeleton as the reverse-step kernel (ctdd_step_tcq.cu): one CTA pair per TPC, tcgen05 cta_group::2, M side =
// output column n (128 per CTA) with the sample's matrix resident in tensor memory as the A operand (TS form), N side =
// data rows (128-row tiles, 64 produced per CTA), 2 operand stages of 64 KB, 2 accumulators of 128 columns.
//   * A pair owns a contiguous range of the global tile list (tiles of sample 0, tiles of sample 1, ..), so the matrix
//     in tensor memory changes only when the range crosses a sample boundary: the epilogue warps then convert the next
//     sample's fp32 matrix half to bf16 hi / mid and tcgen05.st it, after the last MMA of the old sample has completed;
//     the MMA thread waits for that (q_ready) before the first MMA of the new sample.
//   * Producers (12 warps, two rows per pass, 16 lanes per row): rows arrive by cp.async.bulk, are split into bf16 hi /
//     mid and stored K-major, 128B-swizzled.
//   * Epilogue (8 warps, lane = output column): tcgen05.ld 32 columns x 32 rows, coalesced 128-byte stores per row.
#include "ctdd_tc_common.cuh"

namespace ctdd {
namespace bgemm {
using namespace tc;

constexpr int NH = 64;                 // rows of a tile produced by one CTA
constexpr int NT = 2 * NH;             // rows per pair tile (= UMMA N)
constexpr int STAGES = 2;
constexpr int ACC = 2;
constexpr int NUM_EPI_WARPS = 8;       // warps 0-7: TMEM quadrant w&3, column half w>>2 (= CTA that produced those rows)
constexpr int FIRST_PROD_WARP = 8;
constexpr int NPW = 12;
constexpr int MMA_WARP = FIRST_PROD_WARP + NPW;   // light group: MMA issue / relay + 3 idle warps
constexpr int NUM_THREADS = (FIRST_PROD_WARP + NPW + 4) * 32;
constexpr int REGS_LIGHT = 48;
constexpr int PASSES_PER_TILE = NH / 2;
constexpr int KBLOCK_BYTES = NH * 128;
constexpr int SPLIT_BYTES = 4 * KBLOCK_BYTES;
constexpr int STAGE_BYTES = 2 * SPLIT_BYTES;
constexpr uint32_t IDESC = make_idesc(NT);

struct Smem {
  alignas(1024) uint8_t stage[STAGES][STAGE_BYTES];
  alignas(16) float lring[NPW][2][S];          // raw fp32 row pairs, refilled one pass ahead
  alignas(8) uint64_t full[STAGES];            // leader CTA: its NPW producer warps + 1 relayed arrival for the partner's
  uint64_t full_local[STAGES];
  uint64_t empty[STAGES];                      // multicast tcgen05.commit
  uint64_t lring_full[NPW];
  uint64_t tmem_full[ACC];                     // multicast tcgen05.commit
  uint64_t tmem_empty[ACC];                    // leader CTA: 8 local + 8 remote epilogue warps
  uint64_t q_ready;                            // leader CTA: 8 local + 8 remote epilogue warps have stored the new matrix
  uint32_t tmem_base;
};
static_assert(sizeof(Smem) + 1024 <= 232448, "shared memory budget exceeded");

struct GemmArgs {
  const float* X;      // [B][D][256]
  const float* M;      // [B][256][256]  (row n, column k)
  float* out;          // [B][D][256]
  int B, D;
  int tiles_per_sample;
  long long num_tiles;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) bgemm_kernel(const GemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  // this pair's contiguous range of the global tile list
  const int g_begin = (int)(a.num_tiles * pair / npairs), g_end = (int)(a.num_tiles * (pair + 1) / npairs);
  const int my_tiles = g_end - g_begin;
  const int TPS = a.tiles_per_sample;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&sm.full[i], NPW + 1);
      mbar_init(&sm.full_local[i], NPW);
      mbar_init(&sm.empty[i], 1);
    }
    for (int w = 0; w < NPW; ++w) mbar_init(&sm.lring_full[w], 1);
    for (int i = 0; i < ACC; ++i) { mbar_init(&sm.tmem_full[i], 1); mbar_init(&sm.tmem_empty[i], 2 * NUM_EPI_WARPS); }
    mbar_init(&sm.q_ready, 2 * NUM_EPI_WARPS);
    fence_barrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();

  if (warp >= FIRST_PROD_WARP && warp < MMA_WARP) {
    // ======================================================================== producers
    const int pw = warp - FIRST_PROD_WARP;
    const int half = lane >> 4, l16 = lane & 15;
    uint64_t* const full_bar = rank == 0 ? &sm.full[0] : &sm.full_local[0];
    // pass P = 32 * tl + ps of this CTA: rows 2 ps, 2 ps + 1 of the CTA's 64 rows of its tl-th tile
    auto pass_rows = [&](int tl, int ps, long long& x_off, int& nvalid) {
      const int g = g_begin + tl;
      const int b = g / TPS;
      const int d0 = (g - b * TPS) * NT + (int)rank * NH + 2 * ps;          // first row of the pair within the sample
      nvalid = a.D - d0;                                                     // <= 0: both rows past the end
      x_off = ((long long)b * a.D + d0) * S;
    };
    auto fetch_rows = [&](int tl, int ps) {
      if (tl >= my_tiles) return;
      long long x_off; int nvalid;
      pass_rows(tl, ps, x_off, nvalid);
      if (lane == 0) {
        uint64_t* bar = &sm.lring_full[pw];
        mbar_arrive_expect_tx(bar, 2 * S * 4);
        if (nvalid >= 2) {
          bulk_g2s(&sm.lring[pw][0][0], a.X + x_off, 2 * S * 4, bar);
        } else {      // ragged end of a sample: rows past it are replaced by row 0 of the tensor (never used)
          bulk_g2s(&sm.lring[pw][0][0], a.X + (nvalid >= 1 ? x_off : 0), S * 4, bar);
          bulk_g2s(&sm.lring[pw][1][0], a.X, S * 4, bar);
        }
      }
    };
    int f_tl = 0, f_ps = pw;
    fetch_rows(f_tl, f_ps);
    uint32_t ring_par = 0;
    int last_tl = -1;
    int tl = 0, ps = pw;
#pragma unroll 1
    while (tl < my_tiles) {
      const int st = tl % STAGES;
      long long x_off; int nvalid;
      pass_rows(tl, ps, x_off, nvalid);
      const bool ok = half < nvalid;
      const bool last_in_tile = ps + NPW >= PASSES_PER_TILE;
      mbar_wait(&sm.lring_full[pw], ring_par);
      ring_par ^= 1u;
      float v[16];
      const uint32_t src = smem_u32(&sm.lring[pw][half][4 * l16]);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float4 q4 = lds128(src + 256 * c);
        v[4 * c] = q4.x; v[4 * c + 1] = q4.y; v[4 * c + 2] = q4.z; v[4 * c + 3] = q4.w;
      }
      __syncwarp();            // every lane has its values: the slot is refilled for the warp's next pass
      f_ps += NPW;
      if (f_ps >= PASSES_PER_TILE) { f_ps -= PASSES_PER_TILE; ++f_tl; }
      fetch_rows(f_tl, f_ps);
      if (tl != last_tl) {
        mbar_wait(&sm.empty[st], (uint32_t)(((tl / STAGES) & 1) ^ 1));
        last_tl = tl;
      }
      if (!ok) {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = 0.f;
      }
      store_operand_row<KBLOCK_BYTES, SPLIT_BYTES>(smem_u32(sm.stage[st]), 2 * ps + half, l16, v);
      if (last_in_tile) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar + st);
      }
      ps += NPW;
      if (ps >= PASSES_PER_TILE) { ps -= PASSES_PER_TILE; ++tl; }
    }
  } else if (warp > MMA_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));
  } else if (warp == MMA_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LIGHT));
    // ======================================================================== MMA issue (one thread of the leader CTA)
    if (rank == 0 && lane == 0) {
      int nq = 0;          // matrices loaded so far
      for (int i = 0; i < my_tiles; ++i) {
        const int st = i % STAGES, b = i % ACC;
        const int g = g_begin + i;
        if (i == 0 || g % TPS == 0) {      // first tile of a sample in this range: its matrix must be in tensor memory
          mbar_wait_cluster(&sm.q_ready, nq & 1);
          ++nq;
        }
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
    // ======================================================================== epilogue + matrix loads: lane = output column
    const int q = warp & 3;
    const uint32_t h = (uint32_t)(warp >> 2);
    const int n_mine = (int)rank * 128 + q * 32 + lane;          // output column (= row of M) of this lane
    const uint32_t tempty_dst = mapa(smem_u32(&sm.tmem_empty[0]), 0);
    const uint32_t qready_dst = mapa(smem_u32(&sm.q_ready), 0);

    // row n_mine of sample b's matrix -> tensor memory, bf16 hi / mid split; warp h of the quadrant takes k in [128 h, 128 h + 128)
    auto load_matrix = [&](int b) {
      const float4* src = reinterpret_cast<const float4*>(a.M + ((size_t)b * S + n_mine) * S + 128 * h);
#pragma unroll 1
      for (int c = 0; c < 64; c += 32) {        // 32 TMEM columns (= 64 k) per step
        uint32_t rh[32], rm[32];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float4 v = __ldg(src + (c >> 1) + i);
          split2(v.x, v.y, rh[2 * i], rm[2 * i]);
          split2(v.z, v.w, rh[2 * i + 1], rm[2 * i + 1]);
        }
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
        tmem_st32(lane_base + TM_QH + 64 * h + c, rh);
        tmem_st32(lane_base + TM_QM + 64 * h + c, rm);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster_release(qready_dst);
    };

    if (my_tiles > 0) load_matrix(g_begin / TPS);
    for (int i = 0; i < my_tiles; ++i) {
      const int b_acc = i % ACC;
      const int g = g_begin + i;
      const int bs = g / TPS;
      const int d_tile = (g - bs * TPS) * NT;
      mbar_wait(&sm.tmem_full[b_acc], (i / ACC) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int bb = 0; bb < 2; ++bb) {
        uint32_t acc[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + TM_ACC + b_acc * NT + h * NH + 32 * bb, acc);
        tmem_ld_wait();
        if (bb == 1) {           // the accumulator has been read: hand the buffer back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster_relaxed(tempty_dst + (uint32_t)b_acc * 8u);
        }
        const int d0 = d_tile + (int)h * NH + 32 * bb;
        float* dst = a.out + ((size_t)bs * a.D + d0) * S + n_mine;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (d0 + j < a.D) dst[(size_t)j * S] = __uint_as_float(acc[j]);
      }
      // the next tile starts a new sample: its matrix replaces this one now - the last MMA that reads the old matrix (tile
      // i) has completed, and the MMA thread does not start tile i + 1 before q_ready
      if ((i + 1 < my_tiles) && ((g + 1) % TPS == 0)) load_matrix(bs + 1);
    }
  }
  pair_teardown(warp == MMA_WARP, tmem);
}

}  // namespace bgemm
}  // namespace ctdd

extern "C" int ctdd_bgemm256_tc(const float* X, const float* M, int B, int D, float* out, void* stream) {
  using namespace ctdd;
  using namespace ctdd::bgemm;
  if (!X || !M || !out || B <= 0 || D <= 0) { set_error("ctdd_bgemm256_tc: bad arguments"); return 2; }
  if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(M) & 15)) {
    set_error("ctdd_bgemm256_tc: X and M must be 16-byte aligned");
    return 2;
  }
  static tc::PairLaunchState launch_state;
  void (*const kerns[1])(const GemmArgs) = {bgemm_kernel};
  const size_t smem_bytes = sizeof(Smem) + 1024;
  GemmArgs a;
  a.X = X; a.M = M; a.out = out; a.B = B; a.D = D;
  a.tiles_per_sample = (D + NT - 1) / NT;
  a.num_tiles = (long long)B * a.tiles_per_sample;
  const int pairs = tc::pair_count(launch_state, "ctdd_bgemm256_tc", kerns, smem_bytes, a.num_tiles);
  if (!pairs) return 1;
  bgemm_kernel<<<2 * pairs, NUM_THREADS, smem_bytes, (cudaStream_t)stream>>>(a);
  CTDD_CHECK_LAUNCH("bgemm_kernel");
  return 0;
}

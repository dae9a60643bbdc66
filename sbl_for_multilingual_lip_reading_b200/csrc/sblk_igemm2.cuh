// sblk_igemm2.cuh — CTA-pair (cta_group::2) variant of the persistent tcgen05 implicit GEMM of sblk_igemm.cuh.
//
// Why: ncu on the 1-CTA kernel at the BASELINE shape (profiles/r01f_*) shows the 3x3 convs of ResNet layers 2-4 stalled
// on L2->SM operand delivery (479-631 MB per launch at ~12 TB/s, tensor pipe 41-58 % busy): a 128 x BLOCK_N tile
// fetches 16 KB of A plus BLOCK_N*128 B of B per 64-wide K block.  Here two CTAs of a cluster (the two SMs of a TPC)
// compute one 256 x BLOCK_N tile with tcgen05.mma.cta_group::2: each CTA stages its own 128 A rows and only HALF of the
// B tile, the tensor cores read both halves, so operand bytes per FLOP drop by 1.5x (BLOCK_N = 256) to 2x.
//
// Same roles as the 1-CTA kernel (192 threads: warp 0 TMA producer, warp 1 MMA issuer / TMEM owner, warps 2-5
// epilogue), same fused epilogue.  Protocol differences (CTA rank 0 = leader):
//   * full barriers live in the LEADER: its producer posts expect_tx for both CTAs' bytes, the peer's TMA loads
//     (cp.async.bulk.tensor...cta_group::2) complete_tx on the leader's barrier through its shared::cluster address
//   * only the leader issues MMAs; tcgen05.commit...multicast::cluster arrives on the empty / accumulator-full
//     barriers of BOTH CTAs (same smem offsets)
//   * accumulator-empty barrier lives in the leader and counts the epilogue warps of both CTAs (remote arrive)
//   * TMEM is allocated / freed with cta_group::2 by warp 1 of each CTA; cluster barriers bracket the kernel and the
//     producer drains its empty barriers before exit so no multicast arrive can land in a retired CTA's smem.
// Reference call sites: BasicBlock convs + downsample, SBL/transformer/video_frontend.py:10-12,28-41,68-72.
#pragma once
#include "sblk_common.cuh"
#include "sblk_igemm.cuh"

namespace sblk {

// ------------------------------------------------------------------ cluster / cta_group::2 PTX wrappers
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // relaxed: the only data handed over is the TMEM accumulator, ordered by tcgen05.fence::before_thread_sync on this
  // side and ::after_thread_sync on the waiter's; .release.cluster compiled to MEMBAR.ALL.GPU + ERRBAR in front of
  // every arrive (ncu: 16 % of all stall samples of flatconv2, on the accumulator-release critical path)
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// TMA loads whose completion is signalled on an mbarrier given by its shared::cluster address (may be the peer's)
__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* d, uint32_t bar_cluster_addr, int c0,
                                             int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(d)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma2_load_im2col_4d(void* smem_dst, const CUtensorMap* d, uint32_t bar_cluster_addr,
                                                    int c, int w, int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(d)), "r"(bar_cluster_addr), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all previously issued MMAs retired) on the barrier at this smem offset in both CTAs of the pair
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}

// Coalesced store of a [32 rows x 128 B] block held one row per lane: the block goes through a per-warp swizzled
// staging tile and comes back transposed, so one instruction writes 4 complete 128-byte row segments instead of
// 32 x 16 B scattered over 32 rows (LSU-bound).  Row r is written at gbase + row_off(r) (element offset owned by lane
// r, fetched by shuffle: the flat output layout has no constant row pitch); rows with ok(r) == false are skipped.
__device__ __forceinline__ void warp_store_rows128_idx(uint8_t* stg, const uint4 (&d)[8], uint8_t* gbase,
                                                       unsigned long long my_row_off_bytes, bool my_row_ok, int lane) {
#pragma unroll
  for (int c = 0; c < 8; ++c) *reinterpret_cast<uint4*>(stg + lane * 128 + ((c ^ (lane & 7)) << 4)) = d[c];
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3), c = lane & 7;
    const unsigned long long off = __shfl_sync(0xffffffffu, my_row_off_bytes, r);
    const int ok = __shfl_sync(0xffffffffu, my_row_ok ? 1 : 0, r);
    const uint4 v = *reinterpret_cast<const uint4*>(stg + r * 128 + ((c ^ (r & 7)) << 4));
    if (ok) *reinterpret_cast<uint4*>(gbase + off + c * 16) = v;
  }
  __syncwarp();
}

// 64-byte-row variant (2 KB per warp): one instruction writes 8 half-line row segments
__device__ __forceinline__ void warp_store_rows64_idx(uint8_t* stg, const uint4 (&d)[4], uint8_t* gbase,
                                                      unsigned long long my_row_off_bytes, bool my_row_ok, int lane) {
#pragma unroll
  for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4*>(stg + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4)) = d[c];
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i * 8 + (lane >> 2), c = lane & 3;
    const unsigned long long off = __shfl_sync(0xffffffffu, my_row_off_bytes, r);
    const int ok = __shfl_sync(0xffffffffu, my_row_ok ? 1 : 0, r);
    const uint4 v = *reinterpret_cast<const uint4*>(stg + r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
    if (ok) *reinterpret_cast<uint4*>(gbase + off + c * 16) = v;
  }
  __syncwarp();
}

template <int BLOCK_N, bool DUAL = false>
struct Igemm2Cfg {
  static constexpr int BLOCK_M = 128;                 // rows per CTA; the pair computes 256
  static constexpr int PAIR_M = 256;
  static constexpr int BLOCK_K = 64;
  static constexpr int BH = BLOCK_N / 2;              // B rows staged by each CTA
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = BH * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + (DUAL ? 2 : 1) * B_BYTES;
  // per-warp staging tiles of the 8 epilogue warps (32 rows x 128 B for BLOCK_N = 256, x 64 B for 128) for coalesced
  // epilogue stores.  They take the place of the LAST ring stage: the L2-latency-bound shapes (strided block heads of
  // layers 3-4) lose 14 % with one stage less, but the whole frontend graph measured 607 us with staged stores against
  // 644 us with direct per-thread stores and the full ring.
  static constexpr int STG_WARP_BYTES = BLOCK_N == 256 ? 4096 : 2048;
  static constexpr int STG_BYTES = 8 * STG_WARP_BYTES;
  static constexpr int STAGES = (227 * 1024 - 2048) / STAGE_BYTES;
  static_assert(STG_BYTES <= STAGE_BYTES, "staging must fit in one ring stage");
  static constexpr int ACC_STAGES = 2;
  static constexpr int TMEM_COLS = (DUAL ? 2 : 1) * ACC_STAGES * BLOCK_N;
  static constexpr int OFF_STG = (STAGES - 1) * STAGE_BYTES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;
  static constexpr int EPI_WARPS = 8;   // two warps per TMEM lane quarter, each takes half of the tile's columns
  static constexpr int THREADS = 64 + EPI_WARPS * 32;
};

template <int BLOCK_N, bool IM2COL, bool DUAL = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Igemm2Cfg<BLOCK_N, DUAL>::THREADS, 1)
igemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
              const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmA2,
              const IgemmParams p) {
  using Cfg = Igemm2Cfg<BLOCK_N, DUAL>;
  static_assert(BLOCK_N == 128 || BLOCK_N == 256, "BLOCK_N");
  static_assert(!DUAL || (IM2COL && BLOCK_N == 128), "DUAL needs im2col and BLOCK_N = 128");
  static_assert(Cfg::TMEM_COLS <= 512, "TMEM");
  constexpr int STAGES = Cfg::STAGES - 1;   // ring stages: the last stage's bytes hold the staging tiles
  constexpr uint32_t IDESC = make_idesc_bf16(Cfg::PAIR_M, BLOCK_N);

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[STAGES];
  __shared__ uint64_t empty_bar[STAGES];
  __shared__ uint64_t tfull_bar[Cfg::ACC_STAGES];
  __shared__ uint64_t tempty_bar[Cfg::ACC_STAGES];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float bias_s[(DUAL ? 2 : 1) * BLOCK_N];   // bias (| bias2) of the current tile's columns

  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  const int n_tiles = p.N / BLOCK_N;
  const int m_pairs = (p.M + Cfg::PAIR_M - 1) / Cfg::PAIR_M;
  const int num_tiles = m_pairs * n_tiles;
  const int num_kb_main = p.taps_r * p.taps_s * p.cblocks;
  // K-extension (IgemmParams::ext_cblocks): k-blocks of a second (activation, filter) pair behind the conv's own
  const int num_kb = num_kb_main + ((IM2COL && !DUAL) ? p.ext_cblocks : 0);
  const int pair_id = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (DUAL || (IM2COL && p.ext_cblocks > 0)) tma_prefetch_desc(&tmB2);
    if (IM2COL && !DUAL && p.ext_cblocks > 0) tma_prefetch_desc(&tmA2);
#pragma unroll
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);    // used in the leader only: one expect_tx arrive covering both CTAs' bytes
      mbar_init(&empty_bar[i], 1);   // one multicast commit per use
    }
#pragma unroll
    for (int i = 0; i < Cfg::ACC_STAGES; ++i) {
      mbar_init(&tfull_bar[i], 1);   // one multicast commit per tile
      mbar_init(&tempty_bar[i], 2 * Cfg::EPI_WARPS);  // used in the leader only: epilogue warps x 2 CTAs
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2cta(&tmem_base_slot, Cfg::TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();   // barrier inits of both CTAs are visible cluster-wide before any remote arrive / TMA signal
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_slot, 0);

  grid_dep_launch();  // PDL: let the next kernel start its prologue now; its own wait orders the data
  // griddepcontrol.wait is executed by the roles that touch the previous kernel's data (producer: A tiles; epilogue:
  // residual / output)

  if (warp == 0) {
    // ------------------------------------------------ TMA producer (both CTAs): own A rows, own half of the B tile
    int stage = 0;
    uint32_t phase = 0;
    // (issuing the first weight tiles ahead of the PDL wait was tried: the A tiles then queue behind ~100 KB of B
    // loads and the first MMA starts ~3.7k cycles later; with one CTA per SM there is no earlier launch to gain)
    grid_dep_wait();
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
      const int m_blk = tile / n_tiles;
      const int n_blk = tile - m_blk * n_tiles;
      const int m0 = m_blk * Cfg::PAIR_M + static_cast<int>(rank) * Cfg::BLOCK_M;
      const int n0 = n_blk * BLOCK_N + static_cast<int>(rank) * Cfg::BH;
      int img = 0, base_w = 0, base_h = 0, ext_w = 0, ext_h = 0;
      if (IM2COL) {
        const int pq = p.P * p.Q;
        img = m0 / pq;
        const int rem = m0 - img * pq;
        const int ph = rem / p.Q;
        const int qw = rem - ph * p.Q;
        base_w = qw * p.stride - p.pad;
        base_h = ph * p.stride - p.pad;
        ext_w = qw * p.ext_stride;   // the extension is a 1x1 / pad 0 view onto the same output grid
        ext_h = ph * p.ext_stride;
      }
      int cb = 0, r = 0, s = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u, 0x0401);
        uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
        uint8_t* b_dst = a_dst + Cfg::A_BYTES;
        const bool centre = DUAL && r == p.taps_r / 2 && s == p.taps_s / 2;
        const bool ext = IM2COL && !DUAL && kb >= num_kb_main;
        const uint32_t bar = mapa_u32(smem_u32(&full_bar[stage]), 0);   // the leader's barrier
        if (elect_one()) {
          if (leader)
            mbar_arrive_expect_tx(&full_bar[stage], 2u * (Cfg::A_BYTES + Cfg::B_BYTES + (centre ? Cfg::B_BYTES : 0)));
          if (centre) tma2_load_2d(b_dst + Cfg::B_BYTES, &tmB2, bar, cb * 64, n0);
          if (ext) {
            tma2_load_im2col_4d(a_dst, &tmA2, bar, (kb - num_kb_main) * 64, ext_w, ext_h, img, 0, 0);
            tma2_load_2d(b_dst, &tmB2, bar, (kb - num_kb_main) * 64, n0);
          } else if (IM2COL) {
            tma2_load_im2col_4d(a_dst, &tmA, bar, cb * 64, base_w, base_h, img, static_cast<uint16_t>(s),
                                static_cast<uint16_t>(r));
          } else {
            tma2_load_2d(a_dst, &tmA, bar, kb * 64, m0);
          }
          if (!ext) tma2_load_2d(b_dst, &tmB, bar, kb * 64, n0);
        }
        __syncwarp();
        if (++cb == p.cblocks) {
          cb = 0;
          if (++s == p.taps_s) { s = 0; ++r; }
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
    // drain: every slot this CTA filled has been released (no multicast arrive can land after this CTA retires)
    for (int i = 0; i < STAGES; ++i) {
      mbar_wait(&empty_bar[stage], phase ^ 1u, 0x0405);
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer: leader CTA only (one elected lane issues)
    if (leader) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u, 0x0402);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BLOCK_N);
        const uint32_t d_tmem2 = tmem_base + static_cast<uint32_t>((Cfg::ACC_STAGES + acc) * BLOCK_N);
        const int centre_kb0 = ((p.taps_r / 2) * p.taps_s + p.taps_s / 2) * p.cblocks;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase, 0x0403);
          tc_fence_after_sync();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t da = make_desc_sw128(a_addr);
          const uint64_t db = make_desc_sw128(a_addr + Cfg::A_BYTES);
          const uint32_t da_lo = static_cast<uint32_t>(da), db_lo = static_cast<uint32_t>(db);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < Cfg::BLOCK_K / 16; ++k) {
              umma2_bf16(d_tmem, desc_with_lo(da, da_lo + 2 * k), desc_with_lo(db, db_lo + 2 * k), IDESC,
                         (kb > 0 || k > 0) ? 1u : 0u);
            }
            if (DUAL && kb >= centre_kb0 && kb < centre_kb0 + p.cblocks) {
#pragma unroll
              for (int k = 0; k < Cfg::BLOCK_K / 16; ++k)
                umma2_bf16(d_tmem2, desc_with_lo(da, da_lo + 2 * k),
                           desc_with_lo(db, db_lo + static_cast<uint32_t>(Cfg::B_BYTES / 16 + 2 * k)), IDESC,
                           (kb > centre_kb0 || k > 0) ? 1u : 0u);
            }
            umma2_commit_mc(&empty_bar[stage]);                      // frees the slot in both CTAs
            if (kb == num_kb - 1) umma2_commit_mc(&tfull_bar[acc]);  // accumulators complete in both CTAs
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (++acc == Cfg::ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ------------------------------------------------ epilogue warps (TMEM lane quarter = warp % 4), both CTAs.
    // Layers 3-4 give a CTA pair one or two tiles, so the LAST tile's epilogue is exposed at the end of the kernel:
    // eight warps (half of the columns each) and the residual slice requested before the accumulator is waited for
    // keep that tail short (it was 8 chunks x (TMEM load -> dependent global residual load -> store) per thread).
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int half = ew >> 2;
    const int row = quarter * 32 + lane;
    const int etid = static_cast<int>(threadIdx.x) - 64;
    constexpr int NCH = BLOCK_N / 32 / 2;          // 32-column chunks per warp
    constexpr int NB = (DUAL ? 2 : 1) * BLOCK_N;   // bias floats per tile
    const int c_begin = half * NCH;
    uint8_t* const stg = smem + Cfg::OFF_STG + ew * Cfg::STG_WARP_BYTES;
    int acc = 0;
    uint32_t acc_phase = 0;
    int cur_nblk = -1;
    grid_dep_wait();
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
      const int m_blk = tile / n_tiles;
      const int n_blk = tile - m_blk * n_tiles;
      const int m = m_blk * Cfg::PAIR_M + static_cast<int>(rank) * Cfg::BLOCK_M + row;
      const bool row_ok = m < p.M;
      const int ncol0 = n_blk * BLOCK_N + c_begin * 32;   // first output column of this warp
      // while the tile's MMAs run: stage its bias slice in shared memory (only when the column block changes: a
      // block-uniform decision) and request this thread's residual slice
      if (n_blk != cur_nblk) {
        if (cur_nblk >= 0) asm volatile("bar.sync 1, 256;" ::: "memory");   // everyone is done with the old slice
        cur_nblk = n_blk;
        float* bw = bias_s;
        for (int e = etid; e < NB; e += Cfg::EPI_WARPS * 32) {
          float bv = 0.0f;
          if (e < BLOCK_N) {
            if (p.bias != nullptr) bv = __ldg(p.bias + n_blk * BLOCK_N + e);
          } else if (DUAL) {
            bv = __ldg(p.bias2 + n_blk * BLOCK_N + (e - BLOCK_N));
          }
          bw[e] = bv;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // bias slice visible to all epilogue warps
      }
      const float* bs = bias_s;
      uint4 res[NCH * 4];
      if (p.residual != nullptr && row_ok) {
        const uint4* rp = reinterpret_cast<const uint4*>(p.residual + static_cast<size_t>(m) * p.ldo + ncol0);
#pragma unroll
        for (int j = 0; j < NCH * 4; ++j) res[j] = __ldg(rp + j);
      } else {
#pragma unroll
        for (int j = 0; j < NCH * 4; ++j) res[j] = make_uint4(0u, 0u, 0u, 0u);
      }
      mbar_wait(&tfull_bar[acc], acc_phase, 0x0404);
      tc_fence_after_sync();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                             static_cast<uint32_t>(acc * BLOCK_N + c_begin * 32);
      size_t out_row = static_cast<size_t>(m);
      if (IM2COL && p.flat_out) {
        const int pq = p.P * p.Q;
        const int fr = m / pq;
        const int rem = m - fr * pq;
        const int y = rem / p.Q;
        out_row = (static_cast<size_t>(fr) * (p.P + 1) + 1 + y) * (p.Q + 2) + 1 + (rem - y * p.Q);
      }
      const unsigned long long row_off_b = static_cast<unsigned long long>(out_row) * p.ldo * 2ull;   // bf16 bytes
#pragma unroll
      for (int c2 = 0; c2 < NCH / 2; ++c2) {        // 64-column blocks: two TMEM loads in flight, one coalesced store
        uint32_t v2[2][32];
        tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c2 * 64), v2[0]);
        tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c2 * 64 + 32), v2[1]);
        tmem_ld_wait();
        uint4 o[8];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int cl = (c_begin + c2 * 2 + hh) * 32;   // column inside the tile
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 b0 = *reinterpret_cast<const float4*>(&bs[cl + 8 * j]);
            const float4 b1 = *reinterpret_cast<const float4*>(&bs[cl + 8 * j + 4]);
            const uint4 r4 = res[(c2 * 2 + hh) * 4 + j];   // zeros when there is no residual
            float f[8];
            f[0] = __uint_as_float(v2[hh][8 * j + 0]) + b0.x + bf16_lo(r4.x);
            f[1] = __uint_as_float(v2[hh][8 * j + 1]) + b0.y + bf16_hi(r4.x);
            f[2] = __uint_as_float(v2[hh][8 * j + 2]) + b0.z + bf16_lo(r4.y);
            f[3] = __uint_as_float(v2[hh][8 * j + 3]) + b0.w + bf16_hi(r4.y);
            f[4] = __uint_as_float(v2[hh][8 * j + 4]) + b1.x + bf16_lo(r4.z);
            f[5] = __uint_as_float(v2[hh][8 * j + 5]) + b1.y + bf16_hi(r4.z);
            f[6] = __uint_as_float(v2[hh][8 * j + 6]) + b1.z + bf16_lo(r4.w);
            f[7] = __uint_as_float(v2[hh][8 * j + 7]) + b1.w + bf16_hi(r4.w);
            if (p.relu) {
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.0f);
            }
            o[hh * 4 + j].x = pack_bf16x2(f[0], f[1]);
            o[hh * 4 + j].y = pack_bf16x2(f[2], f[3]);
            o[hh * 4 + j].z = pack_bf16x2(f[4], f[5]);
            o[hh * 4 + j].w = pack_bf16x2(f[6], f[7]);
          }
        }
        const int n0 = ncol0 + c2 * 64;
        if (p.out_bf16 != nullptr) {
          if (BLOCK_N == 256) {
            warp_store_rows128_idx(stg, o, reinterpret_cast<uint8_t*>(p.out_bf16 + n0), row_off_b, row_ok, lane);
          } else {
            const uint4 (&o0)[4] = *reinterpret_cast<const uint4 (*)[4]>(&o[0]);
            const uint4 (&o1)[4] = *reinterpret_cast<const uint4 (*)[4]>(&o[4]);
            warp_store_rows64_idx(stg, o0, reinterpret_cast<uint8_t*>(p.out_bf16 + n0), row_off_b, row_ok, lane);
            warp_store_rows64_idx(stg, o1, reinterpret_cast<uint8_t*>(p.out_bf16 + n0 + 32), row_off_b, row_ok, lane);
          }
        }
      }
      if (DUAL) {
        // downsample branch: accumulator 2, + bias2, no ReLU, no residual
        const uint32_t t_row2 = t_row + static_cast<uint32_t>(Cfg::ACC_STAGES * BLOCK_N);
#pragma unroll
        for (int c2 = 0; c2 < NCH / 2; ++c2) {
          uint32_t v2[2][32];
          tmem_ld_32x32b_x32(t_row2 + static_cast<uint32_t>(c2 * 64), v2[0]);
          tmem_ld_32x32b_x32(t_row2 + static_cast<uint32_t>(c2 * 64 + 32), v2[1]);
          tmem_ld_wait();
          uint4 o[8];
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int cl = BLOCK_N + (c_begin + c2 * 2 + hh) * 32;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b0 = *reinterpret_cast<const float4*>(&bs[cl + 8 * j]);
              const float4 b1 = *reinterpret_cast<const float4*>(&bs[cl + 8 * j + 4]);
              o[hh * 4 + j].x = pack_bf16x2(__uint_as_float(v2[hh][8 * j + 0]) + b0.x, __uint_as_float(v2[hh][8 * j + 1]) + b0.y);
              o[hh * 4 + j].y = pack_bf16x2(__uint_as_float(v2[hh][8 * j + 2]) + b0.z, __uint_as_float(v2[hh][8 * j + 3]) + b0.w);
              o[hh * 4 + j].z = pack_bf16x2(__uint_as_float(v2[hh][8 * j + 4]) + b1.x, __uint_as_float(v2[hh][8 * j + 5]) + b1.y);
              o[hh * 4 + j].w = pack_bf16x2(__uint_as_float(v2[hh][8 * j + 6]) + b1.z, __uint_as_float(v2[hh][8 * j + 7]) + b1.w);
            }
          }
          const uint4 (&o0)[4] = *reinterpret_cast<const uint4 (*)[4]>(&o[0]);
          const uint4 (&o1)[4] = *reinterpret_cast<const uint4 (*)[4]>(&o[4]);
          uint8_t* g2 = reinterpret_cast<uint8_t*>(p.out2_bf16 + ncol0 + c2 * 64);
          warp_store_rows64_idx(stg, o0, g2, row_off_b, row_ok, lane);
          warp_store_rows64_idx(stg, o1, g2 + 64, row_off_b, row_ok, lane);
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[acc]), 0));   // the leader's barrier
      if (++acc == Cfg::ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();   // both CTAs are done with each other's smem / TMEM / barriers
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc_2cta(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace sblk

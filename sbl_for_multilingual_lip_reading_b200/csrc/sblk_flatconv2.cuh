// sblk_flatconv2.cuh — stride-1 3x3 convolution C -> C (C = 64 or 128) over the zero-haloed flat layout, as a
// CTA-PAIR (tcgen05 cta_group::2) shifted-window implicit GEMM.
// Reference: BasicBlock conv1/bn1/relu and conv2/bn2/+=residual/relu of ResNet layer1 (64 ch, 22x22) and layer2
//            (128 ch, 11x11), SBL/transformer/video_frontend.py:10-12,28-41.
//
// Why not the im2col kernel (sblk_igemm.cuh): with N = 64 a 128 x 64 tile re-fetches 9 shifted copies of its
// activations plus the whole filter from L2 (216 KB per tile, at the L2 -> SM fabric limit).  Here activations live in
// a zero-haloed flat layout: pixel (f, y, x) lives at row (f*(H+1) + 1 + y)*(W+2) + 1 + x of a [rows, C] bf16 matrix
// whose other rows are zero (one zero row between frames, zero columns left / right), so tap (r, s) of 128 consecutive
// output rows is the SAME staged pixel run shifted by (r-1)*(W+2) + (s-1) rows; each run is staged once (TMA,
// SWIZZLE_128B) and the 9 taps are UMMA descriptors with start addresses shifted by whole 128-byte rows (the swizzle is a
// function of the absolute smem address, so row-shifted descriptors read the staged pixels correctly).  Outputs that
// fall on halo positions are written as zeros, so the result is again a valid flat layout.  Further:
//   * two CTAs (one TPC) compute 256 rows x C with ONE tcgen05.mma.cta_group::2 stream: each CTA stages its own 128-row
//     pixel run but only HALF of the filter rows, so the shared-memory operand bytes per MMA drop from A+B to A+B/2
//     (the N = 64 MMA of layer1 is bound by exactly that fetch: 6 KB -> 5 KB per M128xN64xK16) and layer2 gets the
//     9x cut in L2->SM activation traffic the im2col kernel cannot give (ncu: 418 MB per launch at the L2 fabric limit).
//   * C = 128: the filter (288 KB) does not fit next to the activations, so its 64-row halves stream through a small
//     ring, one 8 KB tile per (tap, channel block); C = 64: the 36 KB half filter stays resident.
//   * the residual tile is TMA-loaded into the buffer the epilogue uses as its store-staging tile: + bias, + residual,
//     ReLU and the halo mask happen in fp32 in place (one rounding to bf16), and the tile leaves with a TMA store.
//   * the epilogue is two independent groups of 4 warps working on alternate tiles (own staging buffer each), so the
//     TMEM-load -> math -> store latency chain of one tile overlaps the next tile's.
// Roles: warp 0 activation loader, warp 1 MMA issuer (leader CTA) + TMEM owner, 8 (C = 128) or 12 (C = 64) epilogue
// warps, then the filter loader warp and the store + residual warp.  Barrier protocol as in sblk_igemm2.cuh (full barriers in the leader).
#pragma once
#include "sblk_common.cuh"
#include "sblk_igemm2.cuh"

namespace sblk {

template <int CB>
struct Fc2Cfg {
  static constexpr int C = 64 * CB;                 // Cin == Cout
  static constexpr int TILE_M = 128;                // rows per CTA (256 per pair)
  static constexpr int BOX_PIX = CB == 1 ? 192 : 160;   // staged pixel run: 128 + 2*(Wp+1) rows (Wp <= 31 / 15)
  static constexpr int A_BOX_BYTES = BOX_PIX * 128;
  static constexpr int A_STAGE_BYTES = CB * A_BOX_BYTES;          // 24 KB / 40 KB
  static constexpr int A_STAGES = CB == 1 ? 5 : 2;    // a stage lasts a whole tile (>= one L2 round trip)
  static constexpr int R_BOX_BYTES = TILE_M * 128;                // one 64-channel block of the residual / output tile
  static constexpr int R_BYTES = CB * R_BOX_BYTES;                // 16 KB / 32 KB
  // residual / store-staging tiles: C = 64 has room for two per epilogue group, so the residual of the group's NEXT
  // tile is already in flight while the current one is still being stored (else: load latency on the critical path)
  static constexpr int R_BUFS = CB == 1 ? 4 : 2;
  static constexpr int BH = C / 2;                                // filter rows staged per CTA
  static constexpr int B_TILE_BYTES = BH * 128;                   // one (tap, channel block) k-block: 4 KB / 8 KB
  static constexpr int B_TILES = 9 * CB;                          // k-blocks per tile
  static constexpr bool B_RESIDENT = CB == 1;
  static constexpr int B_SLOTS = B_RESIDENT ? B_TILES : 10;   // one slot lasts 4 MMAs: cover the L2 latency
  static constexpr int OFF_B = 0;
  static constexpr int OFF_A = ((B_SLOTS * B_TILE_BYTES + 1023) / 1024) * 1024;
  static constexpr int OFF_R = OFF_A + A_STAGES * A_STAGE_BYTES;
  static constexpr int SMEM_BYTES = OFF_R + R_BUFS * R_BYTES + 1024;
  static constexpr int ACC_STAGES = 4;
  static constexpr int TMEM_COLS = ACC_STAGES * C;                // 256 / 512
  // epilogue groups of 4 warps (one TMEM lane quarter each) working on successive tiles.  Two are enough: the C = 64
  // kernel is SHARED-MEMORY-BANDWIDTH bound (per 128-row tile the 36 N=64 MMAs fetch 180 KB of operands, the
  // residual / staging / TMA traffic adds 88 KB: ~2100 cycles at 128 B/clk vs ~2550 measured), so a third group
  // (measured: 36.4 vs 35.5 us) only adds contention
  static constexpr int EPI_GROUPS = 2;
  static constexpr int EPI_WARPS = 4 * EPI_GROUPS;
  static constexpr int THREADS = 64 + EPI_WARPS * 32 + 64;        // + filter loader warp + residual loader warp
};

// shared -> global TMA store of one box (bulk async group of the issuing thread)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* d, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(d)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}


struct FlatConv2Params {
  int m_total;       // rows of the flat activation matrix = (F*(H+1) + 1) * (W+2)
  int num_tiles;     // pair tiles = ceil(m_total / 256)
  int H, W;
  int relu;
  int has_res;
  const float* bias;           // [C] folded BN shift
  // 1 = every CTA pair walks its tile range from the last tile to the first.  Consecutive convs of a stage alternate the
  // direction: the activation rows a pair wrote (and read) LAST in one conv are the first it reads in the next, i.e. the
  // ones most likely still in L2 (a layer-1 tensor is 65.6 MB, conv + residual + output 197 MB against 126 MB of L2).
  // Same tiles, same arithmetic: bit-identical.
  int reverse;
};

template <int CB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Fc2Cfg<CB>::THREADS, 1)
flatconv2_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
                 const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmO,
                 const FlatConv2Params p) {
  using Cfg = Fc2Cfg<CB>;
  constexpr int C = Cfg::C;
  constexpr int A_STAGES = Cfg::A_STAGES;
  constexpr int B_SLOTS = Cfg::B_SLOTS;
  constexpr int ACC_STAGES = Cfg::ACC_STAGES;
  constexpr uint32_t IDESC = make_idesc_bf16(256, C);

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t a_full[A_STAGES];      // leader: pixel runs of both CTAs landed
  __shared__ uint64_t a_empty[A_STAGES];     // both CTAs: slot released by the MMAs (multicast commit)
  __shared__ uint64_t b_full[B_SLOTS];       // leader: filter k-block halves of both CTAs landed (resident: slot 0 only)
  __shared__ uint64_t b_empty[B_SLOTS];      // both CTAs (streaming only)
  __shared__ uint64_t r_full[Cfg::R_BUFS];   // local: staging tile may be used (residual landed / previous store read out)
  __shared__ uint64_t s_ready[Cfg::R_BUFS];  // local: the 4 warps of an epilogue group finished writing the tile
  __shared__ uint64_t tfull_bar[ACC_STAGES];
  __shared__ uint64_t tempty_bar[ACC_STAGES];   // leader: 4 epilogue warps (one group) x 2 CTAs
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float bias_s[C];

  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  const uint32_t smem_base = smem_u32(smem);
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int Wp = p.W + 2;

  // contiguous, balanced range of pair tiles for this CTA pair
  const int pair_id = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int base_cnt = p.num_tiles / num_pairs;
  const int rem = p.num_tiles - base_cnt * num_pairs;
  const int my_cnt = base_cnt + (pair_id < rem ? 1 : 0);
  const int tile_begin = pair_id * base_cnt + min(pair_id, rem);
  const int tile_end = tile_begin + my_cnt;
  // j-th tile of this pair (every role walks j = 0 .. my_cnt-1)
  const int tile_first = p.reverse ? tile_end - 1 : tile_begin;
  const int tile_step = p.reverse ? -1 : 1;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmR);
    tma_prefetch_desc(&tmO);
#pragma unroll
    for (int i = 0; i < A_STAGES; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
#pragma unroll
    for (int i = 0; i < B_SLOTS; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
#pragma unroll
    for (int i = 0; i < Cfg::R_BUFS; ++i) {
      mbar_init(&r_full[i], 1);
      mbar_init(&s_ready[i], 4);
    }
#pragma unroll
    for (int i = 0; i < ACC_STAGES; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 8);   // the 4 warps of one epilogue group x 2 CTAs
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2cta(&tmem_base_slot, Cfg::TMEM_COLS);
  if (threadIdx.x >= 64 && threadIdx.x < 64 + C) bias_s[threadIdx.x - 64] = __ldg(p.bias + (threadIdx.x - 64));
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_slot, 0);

  grid_dep_launch();  // PDL: let the next kernel start its prologue now; its own wait orders the data
  // (the filter loader below starts before grid_dep_wait: weights do not depend on the previous kernel)

  if (warp == 0) {
    // ------------------------------------------------ activation / residual loader (both CTAs)
    grid_dep_wait();
    int stage = 0;
    uint32_t phase = 0;
    for (int j = 0; j < my_cnt; ++j) {
      const int tile = tile_first + j * tile_step;
      const int row0 = tile * 256 + static_cast<int>(rank) * Cfg::TILE_M;   // first output row of this CTA
      mbar_wait(&a_empty[stage], phase ^ 1u, 0x0701);
      uint8_t* a_dst = smem + Cfg::OFF_A + stage * Cfg::A_STAGE_BYTES;
      const uint32_t bar = mapa_u32(smem_u32(&a_full[stage]), 0);
      if (elect_one()) {
        if (leader) mbar_arrive_expect_tx(&a_full[stage], 2u * Cfg::A_STAGE_BYTES);
#pragma unroll
        for (int cb = 0; cb < CB; ++cb)   // may start before row 0 / run past the end: TMA zero-fills
          tma2_load_2d(a_dst + cb * Cfg::A_BOX_BYTES, &tmX, bar, cb * 64, row0 - (Wp + 1));
      }
      __syncwarp();
      if (++stage == A_STAGES) { stage = 0; phase ^= 1u; }
    }
    for (int i = 0; i < A_STAGES; ++i) {   // drain (see sblk_igemm2.cuh)
      mbar_wait(&a_empty[stage], phase ^ 1u, 0x0703);
      if (++stage == A_STAGES) { stage = 0; phase ^= 1u; }
    }
  } else if (warp == 3 + Cfg::EPI_WARPS) {
    // ------------------------------------------------ store + residual warp (both CTAs).  One lane owns every TMA store
    // of the CTA (bulk async-groups are per thread) and recycles the staging tiles: as soon as a store has been READ
    // out of shared memory the tile is handed back — with the residual of its next user already requested (has_res) or
    // as a plain arrive.  Nothing in the epilogue warps ever waits for a store, and a residual load is in flight two
    // (C = 64) tiles ahead of its use.  (Clock stamps before: the MMA issuer idled ~40 % on a_full because residual
    // waits sat in the activation loader's in-order loop, and the epilogue groups idled on their own store reads.)
    grid_dep_wait();
    if (lane == 0) {
      constexpr int R_BUFS = Cfg::R_BUFS;
      constexpr int LAG = R_BUFS / 2 - 1;      // stores allowed to be still reading when the next one is issued
      auto recycle = [&](int j_next) {         // staging tile j_next % R_BUFS is free again: prepare it for tile j_next
        if (j_next >= my_cnt) return;
        const int rb = j_next % R_BUFS;
        if (p.has_res) {
          const int row0 = (tile_first + j_next * tile_step) * 256 + static_cast<int>(rank) * Cfg::TILE_M;
          uint8_t* r_dst = smem + Cfg::OFF_R + rb * Cfg::R_BYTES;
          mbar_arrive_expect_tx(&r_full[rb], Cfg::R_BYTES);
#pragma unroll
          for (int cb = 0; cb < CB; ++cb)
            tma_load_2d(r_dst + cb * Cfg::R_BOX_BYTES, &tmR, &r_full[rb], cb * 64, row0);
        } else {
          mbar_arrive(&r_full[rb]);
        }
      };
      if (p.has_res)
        for (int j = 0; j < R_BUFS; ++j) recycle(j);   // first round: the tiles are free, only the residuals are missing
      for (int j = 0; j < my_cnt; ++j) {
        const int rb = j % R_BUFS;
        const int row0 = (tile_first + j * tile_step) * 256 + static_cast<int>(rank) * Cfg::TILE_M;
        mbar_wait(&s_ready[rb], static_cast<uint32_t>(j / R_BUFS) & 1u, 0x0702);
        const uint8_t* stg = smem + Cfg::OFF_R + rb * Cfg::R_BYTES;
#pragma unroll
        for (int cb = 0; cb < CB; ++cb)        // rows past the end of the tensor are clipped by TMA
          tma_store_2d(&tmO, stg + cb * Cfg::R_BOX_BYTES, cb * 64, row0);
        bulk_commit_group();
        if (LAG == 1) bulk_wait_group_read1(); else bulk_wait_group_read0();
        if (j >= LAG) recycle(j - LAG + R_BUFS);
      }
      bulk_wait_group0();                      // all output bytes are in global memory before the CTA retires
    }
    __syncwarp();
  } else if (warp == 2 + Cfg::EPI_WARPS) {
    // ------------------------------------------------ filter loader (both CTAs): own half of the output channels
    const int n0 = static_cast<int>(rank) * Cfg::BH;
    if (Cfg::B_RESIDENT) {
      const uint32_t bar = mapa_u32(smem_u32(&b_full[0]), 0);
      if (elect_one()) {
        if (leader) mbar_arrive_expect_tx(&b_full[0], 2u * Cfg::B_TILES * Cfg::B_TILE_BYTES);
#pragma unroll
        for (int t = 0; t < Cfg::B_TILES; ++t)
          tma2_load_2d(smem + Cfg::OFF_B + t * Cfg::B_TILE_BYTES, &tmW, bar, t * 64, n0);
      }
      __syncwarp();
    } else {
      int slot = 0;
      uint32_t phase = 0;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        for (int kb = 0; kb < Cfg::B_TILES; ++kb) {   // k-block kb = (channel block, tap) in MMA order
          const int cb = kb / 9;
          const int t = kb - cb * 9;
          mbar_wait(&b_empty[slot], phase ^ 1u, 0x0704);
          const uint32_t bar = mapa_u32(smem_u32(&b_full[slot]), 0);
          if (elect_one()) {
            if (leader) mbar_arrive_expect_tx(&b_full[slot], 2u * Cfg::B_TILE_BYTES);
            tma2_load_2d(smem + Cfg::OFF_B + slot * Cfg::B_TILE_BYTES, &tmW, bar, (t * CB + cb) * 64, n0);
          }
          __syncwarp();
          if (++slot == B_SLOTS) { slot = 0; phase ^= 1u; }
        }
      }
      for (int i = 0; i < B_SLOTS; ++i) {   // drain
        mbar_wait(&b_empty[slot], phase ^ 1u, 0x0705);
        if (++slot == B_SLOTS) { slot = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer: leader CTA only (one elected lane issues)
    if (leader) {
      int stage = 0;
      uint32_t phase = 0;
      int slot = 0;
      uint32_t bphase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint64_t db0 = make_desc_sw128(smem_base + Cfg::OFF_B);
      const uint32_t db0_lo = static_cast<uint32_t>(db0);
      uint32_t tap_off[9];   // (r*Wp + s) rows of 128 B, in descriptor units of 16 B
#pragma unroll
      for (int t = 0; t < 9; ++t) tap_off[t] = static_cast<uint32_t>(((t / 3) * Wp + (t % 3)) * 8);
      if (Cfg::B_RESIDENT) mbar_wait(&b_full[0], 0, 0x0706);
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        mbar_wait(&a_full[stage], phase, 0x0707);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u, 0x0708);
        tc_fence_after_sync();
        const uint64_t da0 = make_desc_sw128(smem_base + Cfg::OFF_A + stage * Cfg::A_STAGE_BYTES);
        const uint32_t da0_lo = static_cast<uint32_t>(da0);
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * C);
#pragma unroll 1
        for (int cb = 0; cb < CB; ++cb) {
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            uint32_t b_lo;
            if (Cfg::B_RESIDENT) {
              b_lo = db0_lo + static_cast<uint32_t>(t * (Cfg::B_TILE_BYTES / 16));
            } else {
              mbar_wait(&b_full[slot], bphase, 0x0709);
              tc_fence_after_sync();
              b_lo = db0_lo + static_cast<uint32_t>(slot * (Cfg::B_TILE_BYTES / 16));
            }
            const uint32_t a_lo = da0_lo + static_cast<uint32_t>(cb * (Cfg::A_BOX_BYTES / 16)) + tap_off[t];
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma2_bf16(d_tmem, desc_with_lo(da0, a_lo + static_cast<uint32_t>(2 * k)),
                           desc_with_lo(db0, b_lo + static_cast<uint32_t>(2 * k)), IDESC,
                           (cb > 0 || t > 0 || k > 0) ? 1u : 0u);
              if (!Cfg::B_RESIDENT) umma2_commit_mc(&b_empty[slot]);
            }
            __syncwarp();
            if (!Cfg::B_RESIDENT) {
              if (++slot == B_SLOTS) { slot = 0; bphase ^= 1u; }
            }
          }
        }
        if (elect_one()) {
          umma2_commit_mc(&tfull_bar[acc]);
          umma2_commit_mc(&a_empty[stage]);
        }
        __syncwarp();
        if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
        if (++stage == A_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    // ------------------------------------------------ epilogue (both CTAs): two groups of 4 warps, alternate tiles
    // thread = output row (TMEM lane), all C channels: + bias (+ residual, read from the staging tile the loader
    // filled), ReLU, halo rows -> 0, bf16 written back IN PLACE (16-byte chunk c of row r at c ^ (r & 7): the layout TMA
    // SWIZZLE_128B gave the residual and expects for the store), then one thread issues the TMA store of the tile.
    grid_dep_wait();
    const int ew = warp - 2;
    const int grp = ew >> 2;                   // epilogue group = staging buffer
    const int quarter = warp & 3;
    const int arow = quarter * 32 + lane;      // output row of this thread inside the CTA's 128-row tile
    const int Hp = p.H + 1;
    const uint32_t tempty_leader = mapa_u32(smem_u32(&tempty_bar[0]), 0);
    for (int j = grp; j < my_cnt; j += Cfg::EPI_GROUPS) {
      const int tile = tile_first + j * tile_step;
      const int row0 = tile * 256 + static_cast<int>(rank) * Cfg::TILE_M;
      const int acc = j & (ACC_STAGES - 1);
      const uint32_t acc_phase = static_cast<uint32_t>(j >> 2) & 1u;
      const int rb = j % Cfg::R_BUFS;
      const uint32_t rphase = static_cast<uint32_t>(j / Cfg::R_BUFS) & 1u;
      uint8_t* stg = smem + Cfg::OFF_R + rb * Cfg::R_BYTES;
      mbar_wait(&tfull_bar[acc], acc_phase, 0x070a);
      tc_fence_after_sync();
      // the staging tile is usable: residual landed (has_res), or its previous store has been read out (first round of a
      // residual-free conv: nothing to wait for, hence the inverted parity)
      mbar_wait(&r_full[rb], p.has_res ? rphase : (rphase ^ 1u), 0x070b);
      const int m = row0 + arow;
      const int R = m / Wp;
      const int cpos = m - R * Wp;
      const bool valid = cpos >= 1 && cpos <= p.W && R >= 1 && ((R - 1) % Hp) < p.H;   // else: halo row -> zeros
#pragma unroll 1
      for (int c64 = 0; c64 < C / 64; ++c64) {
        // both 32-column halves of the 64-channel block are requested before the first is used
        uint32_t v2[2][32];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                               static_cast<uint32_t>(acc * C + c64 * 64);
        tmem_ld_32x32b_x32(taddr, v2[0]);
        tmem_ld_32x32b_x32(taddr + 32u, v2[1]);
        tmem_ld_wait();
        uint8_t* rowp = stg + c64 * Cfg::R_BOX_BYTES + arow * 128;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t (&v)[32] = v2[hh];
          const int col0 = c64 * 64 + hh * 32;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 b0 = *reinterpret_cast<const float4*>(&bias_s[col0 + 8 * q]);
            const float4 b1 = *reinterpret_cast<const float4*>(&bias_s[col0 + 8 * q + 4]);
            float f[8];
            f[0] = __uint_as_float(v[8 * q + 0]) + b0.x; f[1] = __uint_as_float(v[8 * q + 1]) + b0.y;
            f[2] = __uint_as_float(v[8 * q + 2]) + b0.z; f[3] = __uint_as_float(v[8 * q + 3]) + b0.w;
            f[4] = __uint_as_float(v[8 * q + 4]) + b1.x; f[5] = __uint_as_float(v[8 * q + 5]) + b1.y;
            f[6] = __uint_as_float(v[8 * q + 6]) + b1.z; f[7] = __uint_as_float(v[8 * q + 7]) + b1.w;
            const int cc = hh * 4 + q;                               // 16-byte chunk inside the 128-byte row block
            uint4* slot = reinterpret_cast<uint4*>(rowp + ((cc ^ (arow & 7)) << 4));
            if (p.has_res) {
              const uint4 r4 = *slot;
              f[0] += bf16_lo(r4.x); f[1] += bf16_hi(r4.x); f[2] += bf16_lo(r4.y); f[3] += bf16_hi(r4.y);
              f[4] += bf16_lo(r4.z); f[5] += bf16_hi(r4.z); f[6] += bf16_lo(r4.w); f[7] += bf16_hi(r4.w);
            }
            if (p.relu) {
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.0f);
            }
            uint4 o;
            o.x = pack_bf16x2(f[0], f[1]);
            o.y = pack_bf16x2(f[2], f[3]);
            o.z = pack_bf16x2(f[4], f[5]);
            o.w = pack_bf16x2(f[6], f[7]);
            if (!valid) o = make_uint4(0u, 0u, 0u, 0u);   // halo positions stay zero for the next conv
            *slot = o;
          }
        }
      }
      // the accumulator is consumed: hand it back to the MMA issuer (leader's barrier)
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader + static_cast<uint32_t>(acc * 8));
      fence_proxy_async_smem();               // generic-proxy tile writes -> visible to the TMA store
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_ready[rb]);   // 4 warps -> the store warp issues the tile's TMA store
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc_2cta(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace sblk

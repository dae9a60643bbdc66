// sblk_igemm.cuh — persistent, warp-specialised tcgen05 implicit-GEMM for sm_100a.
//
// One kernel serves every dense contraction of the visual encoder except the Cin=1 Conv3d:
//   * 3x3 / 1x1 Conv2d over NHWC bf16 activations (A operand fetched by TMA *im2col* loads, so the
//     GEMM-M axis is the dense flattened (frame, y, x) output index and padding is hardware zero fill)
//     -> reference: BasicBlock convs + downsample, SBL/transformer/video_frontend.py:10-12,28-41,68-72
//   * Linear layers (A operand fetched by tiled 2-D TMA)
//     -> reference: nn.Linear call sites, SBL/transformer/attention.py:41-43,57, module.py:49, encoder.py:53
//
// D[M,N] = A[M,K] * W[N,K]^T, bf16 operands, fp32 accumulate in TMEM.
// Roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM owner), warps 2-5 = epilogue.
// Pipelines: smem ring full/empty (TMA <-> MMA) and a 2-deep TMEM accumulator ring (MMA <-> epilogue),
// so the epilogue of tile i overlaps the main loop of tile i+1.
// Epilogue (fused): + bias (folded BatchNorm shift / Linear bias), + residual, ReLU, bf16 and/or fp32 store.
#pragma once
#include "sblk_common.cuh"

namespace sblk {

struct IgemmParams {
  int M;          // GEMM rows: frames*P*Q for a conv, tokens for a linear
  int N;          // output channels / features (multiple of BLOCK_N)
  int taps_r;     // filter height (1 for linear)
  int taps_s;     // filter width
  int cblocks;    // K-blocks (of 64) per filter tap = Cin/64 ; for a linear: K/64
  int P, Q;       // conv output height / width (im2col only)
  int stride;     // conv traversal stride
  int pad;        // conv zero padding
  int relu;       // apply ReLU in the epilogue
  int ldo;        // row pitch (elements) of out / residual
  const float* bias;               // [N] fp32 or nullptr
  const __nv_bfloat16* residual;   // [M, ldo] bf16 or nullptr
  __nv_bfloat16* out_bf16;         // [M, ldo] or nullptr
  float* out_f32;                  // [M, ldo] or nullptr
  // sblk_igemm2.cuh's dual-head kernel only: the 1x1 / same-stride downsample conv of a BasicBlock shares the
  // centre-tap A tiles of conv1
  const float* bias2;              // [N] folded BN shift of the downsample branch
  __nv_bfloat16* out2_bf16;        // [M, ldo] downsample output (no ReLU)
  // split-K (linear layers at small M): K is cut into `splits` ranges, one tile per (split, m, n); split s writes its
  // fp32 partial to out_f32 + s * split_stride (bias added by split 0 only); the consumer sums the partials
  int splits;                      // >= 1
  long long split_stride;          // elements between partial outputs
  // CTA-pair kernel only: write out / out2 into the zero-haloed flat layout of sblk_flatconv2.cuh (halo rows are not
  // touched: the caller keeps them zero), output pixel (f, y, x) -> row (f*(P+1) + 1 + y)*(Q+2) + 1 + x
  int flat_out;
  // 16-bit float format of A, B, residual and out_bf16: 0 = bf16 (every conv), 1 = IEEE fp16 (the encoder's linear
  // layers, sblk_common.cuh "enc16"); both run as tcgen05 kind::f16 at the same rate
  int fp16;
  // CTA-pair im2col kernel only: K-extension.  After the conv's own taps*cblocks k-blocks, ext_cblocks more k-blocks
  // are accumulated into the SAME tile from a second activation tensor (tmA2: 1x1 / pad 0 / stride ext_stride im2col
  // view with the same P x Q output grid) and a second filter (tmB2: [N][ext_cblocks*64]).  This is how the 1x1
  // downsample branch of a BasicBlock is folded into the block's conv2: relu(conv2(y) + ds(x) + bias) in one fp32
  // accumulator, no bf16 round trip of the branch, no launch of its own.
  int ext_cblocks = 0;
  int ext_stride = 1;
};

template <int BLOCK_N>
struct IgemmCfg {
  static constexpr int BLOCK_M = 128;
  static constexpr int BLOCK_K = 64;
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BLOCK_N == 256) ? 4 : (BLOCK_N == 128) ? 6 : 8;
  static constexpr int ACC_STAGES = 2;
  static constexpr int TMEM_COLS = ACC_STAGES * BLOCK_N;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;  // + manual 1024-B alignment slack
  static constexpr int THREADS = 192;
};

template <int BLOCK_N, bool IM2COL>
__global__ void __launch_bounds__(192, 1)
igemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const IgemmParams p) {
  using Cfg = IgemmCfg<BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  const uint32_t IDESC = (!IM2COL && p.fp16) ? make_idesc_f16(Cfg::BLOCK_M, BLOCK_N)
                                              : make_idesc_bf16(Cfg::BLOCK_M, BLOCK_N);
  const bool out_fp16 = !IM2COL && p.fp16;
  static_assert(BLOCK_N == 64 || BLOCK_N == 128 || BLOCK_N == 256, "BLOCK_N");

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[STAGES];
  __shared__ uint64_t empty_bar[STAGES];
  __shared__ uint64_t tfull_bar[Cfg::ACC_STAGES];
  __shared__ uint64_t tempty_bar[Cfg::ACC_STAGES];
  __shared__ uint32_t tmem_base_slot;

  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  const int n_tiles = p.N / BLOCK_N;
  const int m_tiles = (p.M + Cfg::BLOCK_M - 1) / Cfg::BLOCK_M;
  const int mn_tiles = m_tiles * n_tiles;
  const int num_tiles = mn_tiles * p.splits;
  const int num_kb = p.taps_r * p.taps_s * p.cblocks / p.splits;   // k-blocks per tile

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
#pragma unroll
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
#pragma unroll
    for (int i = 0; i < Cfg::ACC_STAGES; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 4);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_slot, Cfg::TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_slot, 0);

  // Everything above overlaps the tail of the previous kernel under PDL; inputs are read below.
  grid_dep_launch();  // PDL: let the next kernel start its prologue now; its own wait orders the data
  grid_dep_wait();

  if (warp == 0) {
    // ------------------------------------------------ TMA producer (warp-uniform control flow, one elected lane issues)
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int split = tile / mn_tiles;
      const int mn = tile - split * mn_tiles;
      const int m_blk = mn / n_tiles;
      const int n_blk = mn - m_blk * n_tiles;
      const int m0 = m_blk * Cfg::BLOCK_M;
      const int kb0 = split * num_kb;   // first k-block of this split (linear layers only)
      int img = 0, base_w = 0, base_h = 0;
      if (IM2COL) {
        const int pq = p.P * p.Q;
        img = m0 / pq;
        const int rem = m0 - img * pq;
        const int ph = rem / p.Q;
        const int qw = rem - ph * p.Q;
        base_w = qw * p.stride - p.pad;
        base_h = ph * p.stride - p.pad;
      }
      int cb = 0, r = 0, s = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u, 0x0101);
        uint8_t* a_dst = smem + stage * Cfg::STAGE_BYTES;
        uint8_t* b_dst = a_dst + Cfg::A_BYTES;
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_bar[stage], Cfg::A_BYTES + Cfg::B_BYTES);
          if (IM2COL) {
            tma_load_im2col_4d(a_dst, &tmA, &full_bar[stage], cb * 64, base_w, base_h, img,
                               static_cast<uint16_t>(s), static_cast<uint16_t>(r));
          } else {
            tma_load_2d(a_dst, &tmA, &full_bar[stage], (kb0 + kb) * 64, m0);
          }
          tma_load_2d(b_dst, &tmB, &full_bar[stage], (kb0 + kb) * 64, n_blk * BLOCK_N);
        }
        __syncwarp();
        if (++cb == p.cblocks) {
          cb = 0;
          if (++s == p.taps_s) { s = 0; ++r; }
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer (warp-uniform, one elected lane issues)
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1u, 0x0102);
      tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BLOCK_N);
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase, 0x0103);
        tc_fence_after_sync();
        const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
        const uint64_t da = make_desc_sw128(a_addr);
        const uint64_t db = make_desc_sw128(a_addr + Cfg::A_BYTES);
        const uint32_t da_lo = static_cast<uint32_t>(da), db_lo = static_cast<uint32_t>(db);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < Cfg::BLOCK_K / 16; ++k) {
            // advance 16 bf16 = 32 B inside the 128-B swizzle atom: +2 in the (addr >> 4) field
            umma_bf16(d_tmem, desc_with_lo(da, da_lo + 2 * k), desc_with_lo(db, db_lo + 2 * k), IDESC,
                      (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees this smem slot once the MMAs above retire
          if (kb == num_kb - 1) umma_commit(&tfull_bar[acc]);  // accumulator complete -> epilogue
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (++acc == Cfg::ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
    }
  } else {
    // ------------------------------------------------ epilogue warps (TMEM lane quarter = warp % 4)
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int split = tile / mn_tiles;
      const int mn = tile - split * mn_tiles;
      const int m_blk = mn / n_tiles;
      const int n_blk = mn - m_blk * n_tiles;
      const int m = m_blk * Cfg::BLOCK_M + row;
      const bool row_ok = m < p.M;
      mbar_wait(&tfull_bar[acc], acc_phase, 0x0104);
      tc_fence_after_sync();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                             static_cast<uint32_t>(acc * BLOCK_N);
      const size_t row_off = static_cast<size_t>(m) * static_cast<size_t>(p.ldo);
#pragma unroll 1
      for (int c = 0; c < BLOCK_N / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(t_row + static_cast<uint32_t>(c * 32), v);
        tmem_ld_wait();
        if (row_ok) {
          const int n0 = n_blk * BLOCK_N + c * 32;
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          if (p.bias != nullptr && split == 0) {
            const float4* bp = reinterpret_cast<const float4*>(p.bias + n0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 b = __ldg(bp + j);
              f[4 * j + 0] += b.x; f[4 * j + 1] += b.y; f[4 * j + 2] += b.z; f[4 * j + 3] += b.w;
            }
          }
          if (p.residual != nullptr) {
            const uint4* rp = reinterpret_cast<const uint4*>(p.residual + row_off + n0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 r4 = __ldg(rp + j);
              const uint32_t rw[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                f[8 * j + 2 * q + 0] += out_fp16 ? f16_lo(rw[q]) : bf16_lo(rw[q]);
                f[8 * j + 2 * q + 1] += out_fp16 ? f16_hi(rw[q]) : bf16_hi(rw[q]);
              }
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.0f);
          }
          if (p.out_bf16 != nullptr) {
            uint4* op = reinterpret_cast<uint4*>(p.out_bf16 + row_off + n0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 o;
              if (out_fp16) {
                o.x = pack_f16x2(f[8 * j + 0], f[8 * j + 1]);
                o.y = pack_f16x2(f[8 * j + 2], f[8 * j + 3]);
                o.z = pack_f16x2(f[8 * j + 4], f[8 * j + 5]);
                o.w = pack_f16x2(f[8 * j + 6], f[8 * j + 7]);
              } else {
                o.x = pack_bf16x2(f[8 * j + 0], f[8 * j + 1]);
                o.y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
                o.z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
                o.w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
              }
              op[j] = o;
            }
          }
          if (p.out_f32 != nullptr) {
            float4* op = reinterpret_cast<float4*>(p.out_f32 + static_cast<size_t>(split) * p.split_stride + row_off + n0);
#pragma unroll
            for (int j = 0; j < 8; ++j) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (++acc == Cfg::ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace sblk

// sblk_conv3d.cuh — fused visual frontend stem for sm_100a:
//   Conv3d(1->64, k=(5,7,7), s=(1,2,2), p=(2,3,3), no bias) + BatchNorm3d(eval, folded) + ReLU
//   + MaxPool3d((1,3,3), s=(1,2,2), p=(0,1,1)), written as per-frame NHWC bf16 [F,22,22,64].
// Reference: Lipreading.frontend3D + the transpose/contiguous/view that follows it,
//            SBL/transformer/video_frontend.py:99-104,111-115.
//
// Implicit GEMM on tcgen05 with NO per-CTA operand expansion.  Cin = 1, so TMA im2col cannot build the A operand.
// Instead prep_clip (sblk_aux.cuh) writes the clip once as a row-Toeplitz array of 16-byte entries
//     X8[n][tp][pl][yy][x][j] = xpad[n][tp][2*yy + pl][2*x + j],  j = 0..7      (pl = row parity, 47x44 (+4 pad) entries/plane)
// so that the K-chunk (dt, r) of conv pixel m = y*44 + x is the entry at flat index  m + (r>>1)*44  of plane
// (tp = t + dt, pl = r & 1): the A operand of every (dt, r) is the SAME flat entry array at a shifted start.  A
// SWIZZLE_NONE K-major UMMA descriptor reads 8 consecutive entries as one core matrix (SBO = 128 B) and takes the
// second K-chunk of an MMA at an arbitrary byte distance (LBO), so one M128 x N64 x K16 tcgen05.mma consumes the
// filter rows (r, r+1) = (plane 0, plane 1) straight out of the staged entries.
//
// Per CTA (persistent over half frames):
//   * loader thread: per (group of 4 tiles, dt) two bulk copies (plane 0 / plane 1, 644 entries each) into a 4-stage ring
//   * MMA thread:    per stage 4 tiles x 4 MMAs (r pairs 01, 23, 45, 6+zero) into 4 TMEM accumulators; 2 accumulator sets
//   * 16 epilogue warps: TMEM -> +bias, ReLU -> bf16 -> swizzled smem ring of conv pixels, then the 3x3/s2 max-pool is
//     taken straight out of that ring with 16-byte loads and stored coalesced.  The 7.2 MB/clip un-pooled activation
//     never reaches HBM.
#pragma once
#include "sblk_common.cuh"

namespace sblk {

namespace c3d {
constexpr int IN_HW = 88;
constexpr int TPAD = 2;              // zero frames before/after each clip
constexpr int CONV_HW = 44;
constexpr int POOL_HW = 22;
constexpr int COUT = 64;
constexpr int PLANE_ROWS = 47;       // (3 + 88 + 3) / 2 row pairs
constexpr int PLANE_ENTRIES = PLANE_ROWS * CONV_HW + 4;  // 2068 entries of 16 B + 4 zero entries -> 128-B multiple
constexpr int FRAME_ENTRIES = 2 * PLANE_ENTRIES;     // two row-parity planes
constexpr int TAIL_PAD_ENTRIES = 256;                // over-read slack at the very end of X8
constexpr int KPAD = 320;            // packed weight row: 5 dt x 4 MMAs x 16
constexpr int TILES_PER_GROUP = 4;
constexpr int GROUP_PIX = TILES_PER_GROUP * 128;     // 512 conv pixels
constexpr int HALO_ENTRIES = 3 * CONV_HW + 4;        // filter rows 2..6 reach 1..3 entry-rows further (+4: 128-B multiple)
constexpr int STAGE_PLANE_ENTRIES = GROUP_PIX + HALO_ENTRIES;   // 648
constexpr int STAGE_PLANE_BYTES = STAGE_PLANE_ENTRIES * 16;     // 10368 = 81 * 128
constexpr int A_STAGE_BYTES = 2 * STAGE_PLANE_BYTES;            // 20736
constexpr int HALF1_ROW = 21;                                   // second half frame starts at conv row 21 ...
constexpr int HALF1_OFF = 4;                                    // ... loaded from flat pixel 920 = 21*44 - 4 (128-B aligned)
constexpr int A_STAGES = 4;
constexpr int B_BYTES = 5 * COUT * 128;                         // 40960
constexpr int RING_PIX = 768;
constexpr int RING_BYTES = RING_PIX * 128;                      // 98304
constexpr int OFF_B = 0;
constexpr int OFF_RING = OFF_B + B_BYTES;                       // 40960
constexpr int OFF_A = OFF_RING + RING_BYTES;                    // 139264
constexpr int SMEM_BYTES = OFF_A + A_STAGES * A_STAGE_BYTES + 1024;  // 222720
constexpr int GROUPS_PER_UNIT = 2;   // a half frame = 22/23 conv rows <= 1024 pixels
constexpr int EPI_WARPS = 16;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int THREADS = 64 + EPI_THREADS;  // loader warp, mma warp, 16 epilogue warps
constexpr int TMEM_COLS = 512;       // 2 sets x 4 tiles x 64 columns
}  // namespace c3d

// SWIZZLE_NONE K-major smem descriptor: core matrix = 8 rows x 16 B contiguous; SBO = byte distance between
// M-adjacent core matrices, LBO = byte distance between the two K-adjacent core matrices of one K16 MMA.
__device__ __forceinline__ uint64_t make_desc_kmajor_noswizzle(uint32_t smem_addr_bytes, uint32_t lbo_bytes,
                                                               uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr_bytes & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (Blackwell); layout type 0 = SWIZZLE_NONE
  return d;
}

// global -> shared bulk copy (contiguous bytes, multiple of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

struct Conv3dParams {
  int frames;                 // F = N*T
  int T;                      // frames per clip
  const uint4* x8;            // row-Toeplitz clip [N][T+4][2][47][44] entries of 8 bf16
  const float* bias;          // [64] folded BN shift
  __nv_bfloat16* out;         // [F,22,22,64], or the zero-haloed flat layout of sblk_flatconv2.cuh when flat_out
  int flat_out;               // 1: pixel (f,y,x) -> row (f*23 + 1 + y)*24 + 1 + x, halo rows/columns written as zeros
};

__global__ void __launch_bounds__(c3d::THREADS, 1)
conv3d_bn_relu_pool_kernel(const __grid_constant__ CUtensorMap tmW, const Conv3dParams p) {
  using namespace c3d;
  constexpr uint32_t IDESC = make_idesc_bf16(128, COUT);

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[A_STAGES];
  __shared__ uint64_t empty_bar[A_STAGES];
  __shared__ uint64_t tfull_bar[2];
  __shared__ uint64_t tempty_bar[2];
  __shared__ uint64_t weights_bar;
  __shared__ uint32_t tmem_base_slot;

  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  const uint32_t smem_base = smem_u32(smem);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int num_units = p.frames * 2;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmW);
#pragma unroll
    for (int i = 0; i < A_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(&tfull_bar[0], 1);
    mbar_init(&tfull_bar[1], 1);
    mbar_init(&tempty_bar[0], EPI_WARPS);
    mbar_init(&tempty_bar[1], EPI_WARPS);
    mbar_init(&weights_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_slot, 0);

  grid_dep_launch();  // PDL: let the next kernel start its prologue now; its own wait orders the data
  grid_dep_wait();

  if (warp == 0) {
    // ------------------------------------------------ loader: weights once, then (group, dt) stages
    if (elect_one()) {
      mbar_arrive_expect_tx(&weights_bar, B_BYTES);
#pragma unroll
      for (int j = 0; j < 5; ++j) tma_load_2d(smem + OFF_B + j * (COUT * 128), &tmW, &weights_bar, j * 64, 0);
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    const int TP = p.T + 2 * TPAD;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      const int f = u >> 1;
      const int half = u & 1;
      const int n = f / p.T;
      const int t = f - n * p.T;
      const int m_start = half ? HALF1_ROW * CONV_HW - HALF1_OFF : 0;
      for (int g = 0; g < GROUPS_PER_UNIT; ++g) {
        const int m0 = m_start + g * GROUP_PIX;
#pragma unroll 1
        for (int dt = 0; dt < 5; ++dt) {
          mbar_wait(&empty_bar[stage], phase ^ 1u, 0x0201);
          uint8_t* dst = smem + OFF_A + stage * A_STAGE_BYTES;
          const uint4* src = p.x8 + static_cast<size_t>(n * TP + t + dt) * FRAME_ENTRIES + m0;
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[stage], A_STAGE_BYTES);
            bulk_load(dst, src, STAGE_PLANE_BYTES, &full_bar[stage]);
            bulk_load(dst + STAGE_PLANE_BYTES, src + PLANE_ENTRIES, STAGE_PLANE_BYTES, &full_bar[stage]);
          }
          __syncwarp();
          if (++stage == A_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer (warp-uniform control flow, one elected lane issues)
    mbar_wait(&weights_bar, 0, 0x0202);
    int stage = 0;
    uint32_t phase = 0;
    int set = 0;
    uint32_t set_phase = 0;
    const uint64_t db0 = make_desc_sw128(smem_base + OFF_B);
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      for (int g = 0; g < GROUPS_PER_UNIT; ++g) {
        mbar_wait(&tempty_bar[set], set_phase ^ 1u, 0x0203);
        tc_fence_after_sync();
#pragma unroll 1
        for (int dt = 0; dt < 5; ++dt) {
          mbar_wait(&full_bar[stage], phase, 0x0204);
          tc_fence_after_sync();
          const uint32_t a_base = smem_base + OFF_A + stage * A_STAGE_BYTES;
          // descriptors differ only in the low word (start address >> 4): one 32-bit add per operand per MMA
          const uint64_t da0 = make_desc_kmajor_noswizzle(a_base, STAGE_PLANE_BYTES, 128);
          const uint32_t da0_lo = static_cast<uint32_t>(da0);
          const uint32_t db_lo = static_cast<uint32_t>(db0) + static_cast<uint32_t>((dt * COUT * 128) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < TILES_PER_GROUP; ++j) {
              const uint32_t d_tmem = tmem_base + static_cast<uint32_t>((set * TILES_PER_GROUP + j) * COUT);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                // filter rows (2q, 2q+1): plane 0 / plane 1 entries at flat offset q*44 ; q == 3: row 6 + zero weights
                umma_bf16(d_tmem, desc_with_lo(da0, da0_lo + static_cast<uint32_t>((j * 2048 + q * (CONV_HW * 16)) >> 4)),
                          desc_with_lo(db0, db_lo + static_cast<uint32_t>(2 * q)), IDESC, (dt > 0 || q > 0) ? 1u : 0u);
              }
            }
            umma_commit(&empty_bar[stage]);
            if (dt == 4) umma_commit(&tfull_bar[set]);
          }
          __syncwarp();
          if (++stage == A_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (++set == 2) { set = 0; set_phase ^= 1u; }
      }
    }
  } else {
    // ------------------------------------------------ epilogue + fused max-pool (warps 2..17, 512 threads)
    const int ew = warp - 2;              // 0..15
    const int quarter = warp & 3;         // TMEM lane quarter this warp may read
    const int cq = ew >> 2;               // which 16 of the 64 channels
    const int etid = threadIdx.x - 64;    // 0..511
    int set = 0;
    uint32_t set_phase = 0;
    float bias_r[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) bias_r[j] = __ldg(p.bias + cq * 16 + j);
    uint8_t* ring = smem + OFF_RING;
    const uint32_t ring_u32 = smem_base + OFF_RING;

    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      const int f = u >> 1;
      const int half = u & 1;
      const int y_base = half ? HALF1_ROW : 0;
      const int pix_off = half ? HALF1_OFF : 0;   // ring slot of conv pixel (y_base, 0)
      const int nrows = half ? 23 : 22;
      const int py_end = half ? 22 : 11;
      int py_next = half ? 11 : 0;
      for (int g = 0; g < GROUPS_PER_UNIT; ++g) {
        mbar_wait(&tfull_bar[set], set_phase, 0x0205);
        tc_fence_after_sync();
        uint32_t v[TILES_PER_GROUP][16];
#pragma unroll
        for (int j = 0; j < TILES_PER_GROUP; ++j) {
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                 static_cast<uint32_t>((set * TILES_PER_GROUP + j) * COUT + cq * 16);
          tmem_ld_32x32b_x16(taddr, v[j]);
        }
        tmem_ld_wait();
        // the accumulators are in registers: hand the TMEM set back to the MMA thread before the slow part
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[set]);
        if (++set == 2) { set = 0; set_phase ^= 1u; }
#pragma unroll
        for (int j = 0; j < TILES_PER_GROUP; ++j) {
          const int pm = g * GROUP_PIX + j * 128 + quarter * 32 + lane;  // conv pixel index local to the unit
          const int slot = (pm >= RING_PIX) ? pm - RING_PIX : pm;
          uint8_t* dst_row = ring + slot * 128;
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            float gq[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) gq[e] = fmaxf(__uint_as_float(v[j][q * 8 + e]) + bias_r[q * 8 + e], 0.0f);
            uint4 o;
            o.x = pack_bf16x2(gq[0], gq[1]);
            o.y = pack_bf16x2(gq[2], gq[3]);
            o.z = pack_bf16x2(gq[4], gq[5]);
            o.w = pack_bf16x2(gq[6], gq[7]);
            const int chunk = cq * 2 + q;
            *reinterpret_cast<uint4*>(dst_row + ((chunk ^ (slot & 7)) << 4)) = o;
          }
        }

        // conv pixels of this group are in the ring; pool every pooled row whose 3 conv rows are complete
        asm volatile("bar.sync 1, 512;" ::: "memory");
        const int rows_done =
            (g == GROUPS_PER_UNIT - 1) ? nrows : min(nrows, (GROUP_PIX * (g + 1) - pix_off) / CONV_HW);
        int py_stop = py_next;
        while (py_stop < py_end && min(2 * py_stop + 1, CONV_HW - 1) - y_base < rows_done) ++py_stop;
        const int wcols = p.flat_out ? POOL_HW + 2 : POOL_HW;   // flat layout: zero halo column on each side
        const int items = (py_stop - py_next) * (wcols * 8);
        for (int it = etid; it < items; it += EPI_THREADS) {
          const int c = it & 7;                  // 8-channel chunk
          const int pp = it >> 3;
          const int pyo = pp / wcols;
          const int pxp = pp - pyo * wcols;
          const int px = p.flat_out ? pxp - 1 : pxp;
          const int py = py_next + pyo;
          uint4 o = make_uint4(0u, 0u, 0u, 0u);
          if (px >= 0 && px < POOL_HW) {
            // clamped 3x3 window: a clamped tap repeats an in-range pixel, which leaves the max unchanged
            int rowoff[3], col[3];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
              rowoff[i] = (min(max(2 * py - 1 + i, 0), CONV_HW - 1) - y_base) * CONV_HW + pix_off;
              col[i] = min(max(2 * px - 1 + i, 0), CONV_HW - 1);
            }
            __nv_bfloat162 b0 = __floats2bfloat162_rn(0.0f, 0.0f);  // post-ReLU values are >= 0
            __nv_bfloat162 b1 = b0, b2 = b0, b3 = b0;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
              for (int k = 0; k < 3; ++k) {
                int s2 = rowoff[i] + col[k];
                s2 = (s2 >= RING_PIX) ? s2 - RING_PIX : s2;
                uint4 w;
                const uint32_t addr = ring_u32 + s2 * 128 + ((c ^ (s2 & 7)) << 4);
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "r"(addr));
                b0 = __hmax2(b0, *reinterpret_cast<const __nv_bfloat162*>(&w.x));
                b1 = __hmax2(b1, *reinterpret_cast<const __nv_bfloat162*>(&w.y));
                b2 = __hmax2(b2, *reinterpret_cast<const __nv_bfloat162*>(&w.z));
                b3 = __hmax2(b3, *reinterpret_cast<const __nv_bfloat162*>(&w.w));
              }
            }
            o.x = *reinterpret_cast<uint32_t*>(&b0);
            o.y = *reinterpret_cast<uint32_t*>(&b1);
            o.z = *reinterpret_cast<uint32_t*>(&b2);
            o.w = *reinterpret_cast<uint32_t*>(&b3);
          }
          const size_t opix = p.flat_out
              ? (static_cast<size_t>(f) * (POOL_HW + 1) + 1 + py) * (POOL_HW + 2) + pxp
              : (static_cast<size_t>(f) * POOL_HW + py) * POOL_HW + px;
          *reinterpret_cast<uint4*>(p.out + opix * COUT + c * 8) = o;
        }
        py_next = py_stop;
        // the next group's ring writes may overwrite pixels this group's pooling just read
        asm volatile("bar.sync 2, 512;" ::: "memory");
      }
      if (p.flat_out) {
        // zero row between frames (written by the frame's second half) and the leading zero row (frame 0)
        const int zrow = half ? (f + 1) * (POOL_HW + 1) : (f == 0 ? 0 : -1);
        if (zrow >= 0 && etid < (POOL_HW + 2) * 8)
          *reinterpret_cast<uint4*>(p.out + (static_cast<size_t>(zrow) * (POOL_HW + 2)) * COUT + etid * 8) =
              make_uint4(0u, 0u, 0u, 0u);
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace sblk

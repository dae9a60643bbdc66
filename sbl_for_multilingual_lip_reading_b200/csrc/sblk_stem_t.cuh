// sblk_stem_t.cuh — the visual frontend stem, "transposed" form with the filter resident in TENSOR MEMORY:
//   Conv3d(1->64, k=(5,7,7), s=(1,2,2), p=(2,3,3), no bias) + BatchNorm3d(eval, folded) + ReLU
//   + MaxPool3d((1,3,3), s=(1,2,2), p=(0,1,1)), written as per-frame NHWC bf16 (or the zero-haloed flat layout).
// Reference: Lipreading.frontend3D + the transpose/contiguous/view that follows it,
//            SBL/transformer/video_frontend.py:99-104,111-115.  Same inputs / outputs as sblk_conv3d.cuh.
//
// Why a second form.  With 64 output channels the pixel-major kernel (sblk_conv3d.cuh) issues M128 x N64 x K16 MMAs:
// each one reads 4 KB of pixels + 2 KB of filter from shared memory for 32 cycles of math, 192 B/clk against the
// 128 B/clk an SM's shared memory delivers, and its pooling ring adds as much again — ncu: tensor pipe 42 % active,
// 36 % of the bf16 peak.  Here the GEMM is transposed and two output frames share every pixel operand:
//     D[(j, co), px] = sum_k  W[(j, co), k] * X[px, k]        j = 0, 1: output frames t0 and t0 + 1 of one clip
//   * A = the folded filter, M = 128 rows = 2 temporal offsets x 64 channels, lives in TMEM for the whole kernel
//     (tcgen05.mma with a tensor-memory A operand: 24 K16 chunks x 8 columns = 192 columns, written once with
//     tcgen05.st).  An input frame tp feeds frame t0 with the filter slice dt = tp - t0 + 2 and frame t0 + 1 with
//     dt - 1, so ONE pixel operand is used by both row halves of A.
//   * B = the row-Toeplitz entries of sblk_aux.cuh::prep_clip (K-major, SWIZZLE_NONE, second K-half = the other
//     row-parity plane through LBO), N = 96 conv pixels = two conv rows (88) + 8 ignored: the only shared-memory
//     operand, 3 KB per 48-cycle MMA = 64 B/clk.
//   * D = [128 lanes = (j, co)] x [96 pixel columns] fp32, three accumulator buffers (288 columns).
//   * Epilogue: one thread per (frame, channel) lane.  It reads its 88 pixels (two complete conv rows) from TMEM and
//     does the WHOLE 3x3 / stride-2 max-pool in registers: horizontal 3-max per row, vertical max with the previous
//     tile's last row carried in registers (tiles of one frame pair are processed top to bottom by the same CTA).  No
//     pooling ring, no shared-memory traffic; bias + ReLU are applied to the 22 pooled values only
//     (max commutes with the monotone  x -> relu(x + b)).
// Work = (frame pair, row-pair tile) steps in one flat order, cut into equal contiguous ranges per CTA; a range that
// starts inside a frame pair recomputes one tile to get its carry row.
#pragma once
#include "sblk_common.cuh"
#include "sblk_conv3d.cuh"

namespace sblk {

namespace stt {
constexpr int CONV_HW = c3d::CONV_HW;            // 44
constexpr int POOL_HW = c3d::POOL_HW;            // 22
constexpr int COUT = c3d::COUT;                  // 64
constexpr int TILE_PX = 2 * CONV_HW;             // 88 conv pixels = two conv rows = one pooled row
constexpr int TILE_N = 96;                       // MMA N (multiple of 16): 88 + 8 ignored columns
constexpr int TILES_PER_UNIT = POOL_HW;          // 22 row pairs per frame
constexpr int G = 4;                             // tiles staged per group
constexpr int WIN_ENTRIES = TILE_PX * G + (TILE_N - TILE_PX) + 3 * CONV_HW;   // 492: filter rows reach 3 entry-rows further
constexpr int WIN_BYTES = WIN_ENTRIES * 16;      // 7872
constexpr int NP = 6;                            // input frames feeding a pair of output frames
constexpr int STAGE_BYTES = NP * 2 * WIN_BYTES;  // 94464: [p][plane][entries]
constexpr int STAGES = 2;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;
constexpr int ACC_BUFS = 3;
constexpr int A_COL0 = ACC_BUFS * TILE_N;        // 288: first TMEM column of the filter
constexpr int A_CHUNK_COLS = 8;                  // K16 bf16 = 8 x 32-bit columns
constexpr int TMEM_COLS = 512;                   // 288 accumulator + 192 filter columns
constexpr int EPI_WARPS = 8;
constexpr int MMA_WARPS = 2;                     // two issuing threads take alternate tile steps (see the MMA section)
constexpr int THREADS = 64 + EPI_WARPS * 32 + 32;   // loader, MMA issuer 0, 8 epilogue warps (two per TMEM lane quarter), MMA issuer 1
// FUSED form: the row-Toeplitz entries are not read from a prepped copy of the clip (sblk_aux.cuh::prep_clip) but built
// in shared memory by producer warps straight from the fp32 clip / the raw uint8 frames — no 70 MB round trip through
// HBM, one launch less
constexpr int PROD_WARPS = 9;                    // warp 0 (the loader of the unfused form) + 8 more
constexpr int THREADS_FUSED = THREADS + (PROD_WARPS - 1) * 32;
constexpr int PROD_BATCH = 3;                    // work items (4 entries each) a producer thread keeps in flight
static_assert(A_COL0 + NP * 4 * A_CHUNK_COLS <= TMEM_COLS, "TMEM budget");
}  // namespace stt

// D[tmem] (+)= A[tmem] * B[smem]^T : the A operand is read from tensor memory (lane = row, 2 bf16 per 32-bit column)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// registers -> TMEM: this warp's 32 lanes x 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

struct StemTParams {
  int N, T;                   // clips, frames per clip
  const uint4* x8;            // row-Toeplitz clip [N][T+4][2][47*44+4] entries of 8 bf16 (prep_clip); unused when FUSED
  // FUSED sources (exactly one is non-null): the reference-layout fp32 clip [N,1,T,88,88], or raw uint8 gray frames
  // [N,T_in,H0,W0] with the 256-entry bf16 normalisation table and the crop offsets of sblk_prep_clip_u8 (frames
  // T_in .. T-1 are zero padding in normalised space)
  const float* x_f32;
  const uint8_t* x_u8;
  const uint16_t* lut_bf16;
  const int* crop_yx;
  int crop_y0, crop_x0, T_in, H0, W0;
  const __nv_bfloat16* wp;    // packed filter [64][320] bf16, BN folded (sblk_pack_conv3d)
  const float* bias;          // [64] folded BN shift
  __nv_bfloat16* out;         // [F,22,22,64], or the zero-haloed flat layout when flat_out
  int flat_out;
};

// Epilogue of one warp: pooled columns [11 * HALF, 11 * HALF + 11) of every tile step, for the 32 (frame, channel) lanes
// of this warp's TMEM quarter.  The two conv rows of a tile are accumulator columns [0, 44) and [44, 88); this half
// needs conv columns 22 * HALF - 1 .. 22 * HALF + 21 of each, loaded as two 32-column windows starting at column
// 12 * HALF (so that every register index below is a compile-time constant).
// Work partition.  A tile step of frame pair t0 costs one MMA group per EXISTING input frame (3..6 of t0-2 .. t0+3)
// against a roughly constant epilogue, so CTA b starts at the tile step where the running weight
// sum(max(4, frames)) reaches b / grid of the total (clip-periodic: closed form over clips, a short loop over pairs).
__device__ __forceinline__ int stem_t_pair_weight(int t0, int T) {
  const int cnt = min(T, t0 + 4) - max(0, t0 - 2);
  return max(cnt, 4);
}
__device__ __forceinline__ int stem_t_cut(int b, int grid, int N, int T) {
  using namespace stt;
  const int ppc = (T + 1) >> 1;
  if (b >= grid) return N * ppc * TILES_PER_UNIT;
  int clip_w = 0;
  for (int pi = 0; pi < ppc; ++pi) clip_w += stem_t_pair_weight(2 * pi, T);
  const long long clip_cost = static_cast<long long>(clip_w) * TILES_PER_UNIT;
  const long long tgt = clip_cost * N * b / grid;
  const int n = static_cast<int>(tgt / clip_cost);
  int rem = static_cast<int>(tgt - static_cast<long long>(n) * clip_cost);
  int pi = 0, tile = 0;
  for (; pi < ppc; ++pi) {
    const int w = stem_t_pair_weight(2 * pi, T);
    if (rem < w * TILES_PER_UNIT) { tile = rem / w; break; }
    rem -= w * TILES_PER_UNIT;
  }
  return (n * ppc + pi) * TILES_PER_UNIT + tile;
}

template <int HALF>
__device__ __forceinline__ void stem_t_epilogue(const StemTParams& p, uint32_t tmem_base, uint64_t* accfull_bar,
                                                uint64_t* accempty_bar, int s_begin, int s_own, int s_end, int warp,
                                                int lane) {
  using namespace stt;
  constexpr int HP = POOL_HW / 2;          // 11 pooled columns per half
  constexpr int C0 = 12 * HALF;            // first accumulator column of the 32-column window (per conv row)
  const int quarter = warp & 3;
  const int L = quarter * 32 + lane;
  const int j = L >> 6, co = L & 63;
  const int T = p.T;
  const int ppc = (T + 1) >> 1;
  const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(C0);
  const float bias = __ldg(p.bias + co);
  int buf = 0;
  uint32_t buf_phase = 0;
  float carry[HP];
#pragma unroll
  for (int x = 0; x < HP; ++x) carry[x] = -INFINITY;
  const unsigned short zero16 = 0;
  unsigned short* const out16 = reinterpret_cast<unsigned short*>(p.out) + co;
  for (int s = s_begin; s < s_end; ++s) {
    const int u = s / TILES_PER_UNIT;
    const int i = s - u * TILES_PER_UNIT;
    const int n = u / ppc;
    const int t0 = (u - n * ppc) * 2;
    mbar_wait(&accfull_bar[buf], buf_phase, 0x0904);
    tc_fence_after_sync();
    uint32_t r0[32], r1[32];
    const uint32_t taddr = t_lane + static_cast<uint32_t>(buf * TILE_N);
    tmem_ld_32x32b_x32(taddr, r0);
    tmem_ld_32x32b_x32(taddr + static_cast<uint32_t>(CONV_HW), r1);
    tmem_ld_wait();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(&accempty_bar[buf]);
    if (++buf == ACC_BUFS) { buf = 0; buf_phase ^= 1u; }

    float o[HP];
#pragma unroll
    for (int x = 0; x < HP; ++x) {
      const int c = 2 * (x + HP * HALF) - C0;           // window index of conv column 2 * px
      float h0 = fmaxf(__uint_as_float(r0[c]), __uint_as_float(r0[c + 1]));
      float h1 = fmaxf(__uint_as_float(r1[c]), __uint_as_float(r1[c + 1]));
      if (c > 0) {                                       // px == 0: the left neighbour is padding (-inf)
        h0 = fmaxf(h0, __uint_as_float(r0[c > 0 ? c - 1 : 0]));
        h1 = fmaxf(h1, __uint_as_float(r1[c > 0 ? c - 1 : 0]));
      }
      const float top = i == 0 ? -INFINITY : carry[x];   // MaxPool3d pads with -inf above the first conv row
      o[x] = fmaxf(fmaxf(top, h0), h1);
      carry[x] = h1;
    }
    const bool store = s >= s_own && (t0 + j) < T;
    if (store) {
      const long long f = static_cast<long long>(n) * T + t0 + j;
      if (p.flat_out) {
        unsigned short* row = out16 + ((f * (POOL_HW + 1) + 1 + i) * (POOL_HW + 2) + 1 + HP * HALF) * COUT;
        if (HALF == 0) row[-COUT] = zero16;              // left halo column
#pragma unroll
        for (int x = 0; x < HP; ++x)
          row[x * COUT] = __bfloat16_as_ushort(__float2bfloat16_rn(fmaxf(o[x] + bias, 0.0f)));
        if (HALF == 1) row[HP * COUT] = zero16;          // right halo column
        if (i == TILES_PER_UNIT - 1) {                   // zero row between frames
          unsigned short* z = out16 + ((f + 1) * (POOL_HW + 1) * (POOL_HW + 2) + (HP + 1) * HALF) * COUT;
#pragma unroll
          for (int x = 0; x < HP + 1; ++x) z[x * COUT] = zero16;
        }
        if (i == 0 && f == 0) {                          // leading zero row of the whole buffer
          unsigned short* z = out16 + ((HP + 1) * HALF) * COUT;
#pragma unroll
          for (int x = 0; x < HP + 1; ++x) z[x * COUT] = zero16;
        }
      } else {
        unsigned short* row = out16 + ((f * POOL_HW + i) * POOL_HW + HP * HALF) * COUT;
#pragma unroll
        for (int x = 0; x < HP; ++x)
          row[x * COUT] = __bfloat16_as_ushort(__float2bfloat16_rn(fmaxf(o[x] + bias, 0.0f)));
      }
    }
  }
}


// ------------------------------------------------ entry producers of the FUSED forms (SRC 1: fp32 clip, 2: uint8 frames).
// A stage holds, per existing input frame pp and row-parity plane pl, the entries of plane rows
// 2*i0 .. 2*i0 + 2*gn + 3 (44 entries of 16 bytes per row): entry (yy, cx) = the 8 pixels 2cx-3 .. 2cx+4 of input row
// 2*yy + pl - 3, zero outside the frame (sblk_aux.cuh::prep_clip).  Work item = FOUR consecutive entries of one row
// (cx = 4q .. 4q+3, q < 11): the thread loads the 16 pixels 8q-4 .. 8q+11 (four aligned 16-byte loads of the fp32 clip, or
// 16 bytes of the uint8 frame through the normalisation table), packs them to eight bf16 pairs P0..P7 and funnel-shifts
// neighbours, F_k = (P_k >> 16) | (P_{k+1} << 16): entry e is (F_e, F_e+1, F_e+2, F_e+3).  The items of all existing frames
// are spread over all producer threads; PROD_BATCH items per thread are requested before the first one is used.
// Bank conflicts: every item's 64 bytes start at a multiple of 64, so threads storing the same entry index would hit the
// same four banks (4-way); the store order is rotated by rho = (item >> 1) & 3 — a per-thread constant because the
// thread stride is a multiple of 8 — which makes every quarter-warp store 8 distinct 16-byte slots.
template <int SRC>
__device__ __forceinline__ void stem_t_produce(const StemTParams& p, uint8_t* smem, const uint16_t* lut_s,
                                               uint64_t* full_bar, uint64_t* empty_bar, int s_begin, int s_end,
                                               int ptid, int lane) {
  using namespace stt;
  constexpr int PROD_THREADS = PROD_WARPS * 32;
  static_assert(PROD_THREADS % 8 == 0, "the rotation must be a per-thread constant");
  const int T = p.T;
  const int ppc = (T + 1) >> 1;
  const int rho = (ptid >> 1) & 3;
  int stage = 0;
  uint32_t phase = 0;
  int s = s_begin;
  while (s < s_end) {
    const int u = s / TILES_PER_UNIT;
    const int i0 = s - u * TILES_PER_UNIT;
    int gn = TILES_PER_UNIT - i0;
    if (gn > G) gn = G;
    if (gn > s_end - s) gn = s_end - s;
    const int n = u / ppc;
    const int t0 = (u - n * ppc) * 2;
    const int nrows = 2 * gn + 4;                      // plane rows per (frame, plane) window; the last one holds 8 entries
    const int pp_lo = max(0, 2 - t0);
    const int pp_hi = min(NP - 1, T + 1 - t0);         // existing frames t0 - 2 + pp, pp_lo <= pp <= pp_hi
    const int rows2 = 2 * nrows;                       // 12, 16, 20 or 24
    const uint32_t rcp = (65536u + rows2 - 1) / rows2; // x / rows2 == (x * rcp) >> 16 for x < 144
    const int n_items = (pp_hi - pp_lo + 1) * rows2 * 11;
    mbar_wait(&empty_bar[stage], phase ^ 1u, 0x0906);
    uint8_t* const sbase = smem + stage * STAGE_BYTES;
    for (int it0 = ptid; it0 < n_items; it0 += PROD_THREADS * PROD_BATCH) {
      uint32_t dsto[PROD_BATCH];        // byte offset of the item's first entry in the stage
      bool item[PROD_BATCH];            // the item exists (inside the window)
      bool edge0[PROD_BATCH], edge3[PROD_BATCH];   // pixels -4..-1 / 88..91 of the row: padding
      bool rowok[PROD_BATCH];           // the row holds data (else: zero entries)
      float4 vf[PROD_BATCH][4];
      uint32_t vb[PROD_BATCH][4];       // uint8 input: 16 table indices, four per word
#pragma unroll
      for (int b = 0; b < PROD_BATCH; ++b) {
        const int it = it0 + b * PROD_THREADS;
        const int plr_all = it / 11;
        const int q = it - plr_all * 11;
        const int fi = static_cast<int>((static_cast<uint32_t>(plr_all) * rcp) >> 16);
        const int plr = plr_all - fi * rows2;
        const int pl = plr >= nrows ? 1 : 0;
        const int r = plr - pl * nrows;
        const int pp = pp_lo + fi;
        const int tp = t0 - 2 + pp;
        const int y = 2 * (2 * i0 + r) + pl - 3;
        item[b] = it < n_items && !(r == nrows - 1 && q >= 2);
        dsto[b] = static_cast<uint32_t>((pp * 2 + pl) * WIN_BYTES + (r * CONV_HW + 4 * q) * 16);
        edge0[b] = q == 0;
        edge3[b] = q == 10;
        bool row = item[b] && y >= 0 && y < c3d::IN_HW;   // else: zero entries
        if (SRC == 1) {
          const float4* src = reinterpret_cast<const float4*>(
                                  p.x_f32 + ((static_cast<size_t>(n) * T + tp) * c3d::IN_HW + y) * c3d::IN_HW) + (2 * q - 1);
          const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
          vf[b][0] = (row && !edge0[b]) ? __ldg(src) : z;
          vf[b][1] = row ? __ldg(src + 1) : z;
          vf[b][2] = row ? __ldg(src + 2) : z;
          vf[b][3] = (row && !edge3[b]) ? __ldg(src + 3) : z;
        } else {
          row = row && tp < p.T_in;
          const size_t fr = static_cast<size_t>(n) * p.T_in + (row ? tp : 0);
          const int cy = (row && p.crop_yx != nullptr) ? __ldg(p.crop_yx + 2 * fr) : p.crop_y0;
          const int cx = (row && p.crop_yx != nullptr) ? __ldg(p.crop_yx + 2 * fr + 1) : p.crop_x0;
          const uint8_t* src = p.x_u8 + (fr * p.H0 + (cy + y)) * p.W0 + cx + (8 * q - 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const bool ok = row && !(k == 0 && edge0[b]) && !(k == 3 && edge3[b]);
            uint32_t w = 0;
            if (ok) {
#pragma unroll
              for (int m = 0; m < 4; ++m) w |= static_cast<uint32_t>(__ldg(src + 4 * k + m)) << (8 * m);
            }
            vb[b][k] = w;
          }
        }
        rowok[b] = row;
      }
#pragma unroll
      for (int b = 0; b < PROD_BATCH; ++b) {
        uint32_t P[8];
        if (SRC == 1) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            P[2 * k] = pack_bf16x2(vf[b][k].x, vf[b][k].y);
            P[2 * k + 1] = pack_bf16x2(vf[b][k].z, vf[b][k].w);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t w = vb[b][k];
            const bool ok = rowok[b] && !(k == 0 && edge0[b]) && !(k == 3 && edge3[b]);
            const uint32_t lo = static_cast<uint32_t>(lut_s[w & 0xFFu]) | (static_cast<uint32_t>(lut_s[(w >> 8) & 0xFFu]) << 16);
            const uint32_t hi = static_cast<uint32_t>(lut_s[(w >> 16) & 0xFFu]) | (static_cast<uint32_t>(lut_s[w >> 24]) << 16);
            P[2 * k] = ok ? lo : 0u;
            P[2 * k + 1] = ok ? hi : 0u;
          }
        }
        uint32_t F[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) F[k] = __funnelshift_r(P[k], P[k + 1], 16);
        // entries in the rotated order: step st stores entry (st + rho) & 3
        uint4 E[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) E[e] = make_uint4(F[e], F[e + 1], F[e + 2], F[e + 3]);
        if (rho & 1) { const uint4 t = E[0]; E[0] = E[1]; E[1] = E[2]; E[2] = E[3]; E[3] = t; }
        if (rho & 2) { uint4 t = E[0]; E[0] = E[2]; E[2] = t; t = E[1]; E[1] = E[3]; E[3] = t; }
        if (item[b]) {
          uint8_t* const dst = sbase + dsto[b];
#pragma unroll
          for (int st = 0; st < 4; ++st) *reinterpret_cast<uint4*>(dst + (((st + rho) & 3) << 4)) = E[st];
        }
      }
    }
    fence_proxy_async_smem();   // generic-proxy entry writes -> visible to the tensor core's operand reads
    __syncwarp();
    if (lane == 0) mbar_arrive(&full_bar[stage]);
    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    s += gn;
  }
}

template <int SRC>   // input: 0 = prepped copy of the clip (prep_clip), 1 = fp32 clip, 2 = raw uint8 frames
__global__ void __launch_bounds__(SRC != 0 ? stt::THREADS_FUSED : stt::THREADS, 1)
stem_t_kernel(const StemTParams p) {
  using namespace stt;
  constexpr bool FUSED = SRC != 0;
  constexpr uint32_t IDESC = make_idesc_bf16(128, TILE_N);

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[STAGES];
  __shared__ uint64_t empty_bar[STAGES];
  __shared__ uint64_t accfull_bar[ACC_BUFS];
  __shared__ uint64_t accempty_bar[ACC_BUFS];
  __shared__ uint64_t filter_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ uint16_t lut_s[256];                              // FUSED, uint8 input: normalisation table

  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  const uint32_t smem_base = smem_u32(smem);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int T = p.T;
  const int TP = T + 2 * c3d::TPAD;
  const int ppc = (T + 1) >> 1;                      // frame pairs per clip (the last one is half empty when T is odd)
  const int s_own = stem_t_cut(blockIdx.x, gridDim.x, p.N, T);          // first tile step this CTA stores
  const int s_end = stem_t_cut(blockIdx.x + 1, gridDim.x, p.N, T);
  const int s_begin = s_own - ((s_own % TILES_PER_UNIT) != 0 ? 1 : 0);   // + one recomputed tile for the carry row

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], FUSED ? PROD_WARPS : 1);
      mbar_init(&empty_bar[s], MMA_WARPS);
    }
#pragma unroll
    for (int b = 0; b < ACC_BUFS; ++b) {
      mbar_init(&accfull_bar[b], 1);
      mbar_init(&accempty_bar[b], EPI_WARPS);
    }
    mbar_init(&filter_bar, EPI_WARPS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_slot, 0);

  grid_dep_launch();  // PDL: let the next kernel start its prologue now; its own wait orders the data

  if (warp >= 2 && warp < 2 + EPI_WARPS) {
    // the filter goes to TMEM once: lane (j, co) holds, for every (input frame p, filter-row pair q), the 16 taps
    // W[dt][2q .. 2q+1][0..7] with dt = p - j (zero when that temporal offset does not exist).  Warps (ew, ew + 4) of
    // a lane quarter write three input frames each; only the MMA warp waits for it (filter_bar), the loader does not.
    const int quarter = warp & 3;
    const int L = quarter * 32 + lane;
    const int j = L >> 6, co = L & 63;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const int pp0 = warp < 6 ? 0 : 3;
    uint4 wa[12], wb[12];
#pragma unroll
    for (int c = 0; c < 12; ++c) {
      const int dt = pp0 + (c >> 2) - j;
      const bool ok = dt >= 0 && dt < 5;
      const uint4* src = reinterpret_cast<const uint4*>(p.wp + co * c3d::KPAD + (ok ? dt : 0) * 64 + (c & 3) * 16);
      wa[c] = ok ? __ldg(src) : make_uint4(0u, 0u, 0u, 0u);
      wb[c] = ok ? __ldg(src + 1) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int c = 0; c < 12; ++c) {
      const uint32_t w[8] = {wa[c].x, wa[c].y, wa[c].z, wa[c].w, wb[c].x, wb[c].y, wb[c].z, wb[c].w};
      tmem_st_32x32b_x8(t_lane + static_cast<uint32_t>(A_COL0 + ((pp0 + (c >> 2)) * 4 + (c & 3)) * A_CHUNK_COLS), w);
    }
    tmem_st_wait();
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(&filter_bar);
  }

  if (SRC == 2) {   // normalisation table (an input of the launch, not of the previous kernel)
    if (threadIdx.x < 256) lut_s[threadIdx.x] = __ldg(p.lut_bf16 + threadIdx.x);
    __syncthreads();
  }
  grid_dep_wait();

  if (warp == 0 && !FUSED) {
    // ------------------------------------------------ loader: per group of <= G tiles, the entry windows of the
    // (up to) six input frames, two row-parity planes each
    int stage = 0;
    uint32_t phase = 0;
    int s = s_begin;
    while (s < s_end) {
      const int u = s / TILES_PER_UNIT;
      const int i0 = s - u * TILES_PER_UNIT;
      int gn = TILES_PER_UNIT - i0;
      if (gn > G) gn = G;
      if (gn > s_end - s) gn = s_end - s;
      const int n = u / ppc;
      const int t0 = (u - n * ppc) * 2;
      const uint32_t bytes = static_cast<uint32_t>(TILE_PX * gn + (TILE_N - TILE_PX) + 3 * CONV_HW) * 16u;
      int nvalid = 0;
#pragma unroll
      for (int pp = 0; pp < NP; ++pp) {
        const int tp = t0 - 2 + pp;
        nvalid += (tp >= 0 && tp < T) ? 1 : 0;
      }
      mbar_wait(&empty_bar[stage], phase ^ 1u, 0x0901);
      if (elect_one()) {
        mbar_arrive_expect_tx(&full_bar[stage], static_cast<uint32_t>(2 * nvalid) * bytes);
#pragma unroll 1
        for (int pp = 0; pp < NP; ++pp) {
          const int tp = t0 - 2 + pp;
          if (tp < 0 || tp >= T) continue;   // zero padding frames contribute nothing: no load, no MMA
          const uint4* src = p.x8 + static_cast<size_t>(n * TP + t0 + pp) * c3d::FRAME_ENTRIES + i0 * TILE_PX;
          uint8_t* dst = smem + stage * STAGE_BYTES + pp * (2 * WIN_BYTES);
          bulk_load(dst, src, bytes, &full_bar[stage]);
          bulk_load(dst + WIN_BYTES, src + c3d::PLANE_ENTRIES, bytes, &full_bar[stage]);
        }
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      s += gn;
    }
  } else if (FUSED && (warp == 0 || warp >= 3 + EPI_WARPS)) {
    stem_t_produce<SRC>(p, smem, lut_s, full_bar, empty_bar, s_begin, s_end,
                        (warp == 0 ? 0 : (warp - (2 + EPI_WARPS)) * 32) + lane, lane);
  } else if (warp == 1 || warp == 2 + EPI_WARPS) {
    // ------------------------------------------------ MMA issuers.  One thread cannot keep the tensor pipe fed here: a
    // tile step is 24 short MMAs (48 cycles each) whose descriptors differ, ~7 uniform-datapath instructions per MMA
    // (measured: 59 cycles per MMA with one issuer).  Two warps therefore take alternate tile steps; every barrier
    // phase is derived from the tile / group counters, so the two warps share no state.
    const int me = warp == 1 ? 0 : 1;
    const uint64_t db0 = make_desc_kmajor_noswizzle(smem_base, WIN_BYTES, 128);
    mbar_wait(&filter_bar, 0, 0x0905);
    tc_fence_after_sync();
    const uint32_t db0_lo = static_cast<uint32_t>(db0);
    const uint32_t a_tmem = tmem_base + static_cast<uint32_t>(A_COL0);
    int s = s_begin;
    int c = 0;        // tile steps of this CTA so far: accumulator buffer c % 3, issuer c & 1
    int grp = 0;      // groups so far: stage grp % STAGES
    while (s < s_end) {
      const int u = s / TILES_PER_UNIT;
      const int i0 = s - u * TILES_PER_UNIT;
      int gn = TILES_PER_UNIT - i0;
      if (gn > G) gn = G;
      if (gn > s_end - s) gn = s_end - s;
      const int n = u / ppc;
      const int t0 = (u - n * ppc) * 2;
      const int stage = grp % STAGES;
      const uint32_t phase = static_cast<uint32_t>(grp / STAGES) & 1u;
      // which of the six input frames exist (zero padding frames contribute nothing: no load, no MMA)
      uint32_t vmask = 0;
#pragma unroll
      for (int pp = 0; pp < NP; ++pp) {
        const int tp = t0 - 2 + pp;
        if (tp >= 0 && tp < T) vmask |= 1u << pp;
      }
      const int first_pp = __ffs(static_cast<int>(vmask)) - 1;
      bool waited = false, mine = false;
      for (int k = 0; k < gn; ++k, ++c) {
        if ((c & 1) != me) continue;
        mine = true;
        const int buf = c % ACC_BUFS;
        mbar_wait(&accempty_bar[buf], (static_cast<uint32_t>(c / ACC_BUFS) & 1u) ^ 1u, 0x0902);
        if (!waited) {
          mbar_wait(&full_bar[stage], phase, 0x0903);
          waited = true;
        }
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(buf * TILE_N);
        const uint32_t b_lo = db0_lo + static_cast<uint32_t>((stage * STAGE_BYTES + k * (TILE_PX * 16)) >> 4);
        bool last_mine = k == gn - 1 || k == gn - 2;   // no later tile of this group is this warp's
        if (elect_one()) {
#pragma unroll
          for (int pp = 0; pp < NP; ++pp) {
            if (vmask & (1u << pp)) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                umma_bf16_ts(d_tmem, a_tmem + static_cast<uint32_t>((pp * 4 + q) * A_CHUNK_COLS),
                             desc_with_lo(db0, b_lo + static_cast<uint32_t>((pp * (2 * WIN_BYTES) + q * CONV_HW * 16) >> 4)),
                             IDESC, (pp == first_pp && q == 0) ? 0u : 1u);
              }
            }
          }
          umma_commit(&accfull_bar[buf]);
          if (last_mine) umma_commit(&empty_bar[stage]);   // the stage is free once BOTH issuers' MMAs on it are done
        }
        __syncwarp();
      }
      if (!mine) {   // a one-tile group that was the other issuer's
        if (elect_one()) mbar_arrive(&empty_bar[stage]);
        __syncwarp();
      }
      ++grp;
      s += gn;
    }
  } else {
    // ------------------------------------------------ epilogue: warp pairs (ew, ew + 4) share a TMEM lane quarter;
    // thread = one (frame j, channel co) lane and one half of the 22 pooled columns
    if (warp < 6) stem_t_epilogue<0>(p, tmem_base, accfull_bar, accempty_bar, s_begin, s_own, s_end, warp, lane);
    else stem_t_epilogue<1>(p, tmem_base, accfull_bar, accempty_bar, s_begin, s_own, s_end, warp, lane);
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace sblk

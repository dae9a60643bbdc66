// sblk_aux.cuh — the memory-bound kernels of the visual encoder (HBM roofline, not tensor):
//   clip prep (fp32 -> padded bf16), weight packers (BN fold), global average pool,
//   residual + LayerNorm (+ positional encoding, + pad mask), fp32 -> bf16 / fp16 cast.
#pragma once
#include "sblk_common.cuh"
#include "sblk_conv3d.cuh"

namespace sblk {

// --------------------------------------------------------------------------------------------
// Clip prep: x fp32 [N,1,T,88,88] -> row-Toeplitz bf16 entries X8[N][T+4][2][47][44][8] (layout: sblk_conv3d.cuh):
//   X8[n][tp][pl][yy][x][j] = xpad[n][tp - 2][2*yy + pl - 3][2*x + j - 3]   (zero outside the clip)
// i.e. the Conv3d zero padding (2 frames, 3 px) is materialised and every 16-byte entry already holds the 8
// consecutive input pixels one (dt, r) filter row multiplies for conv pixel x, so the stem kernel streams its A
// operand with plain bulk copies.  Reference: input layout of Lipreading.forward, SBL/transformer/video_frontend.py:
// 119-121 (+ Conv3d padding=(2,3,3), stride (1,2,2), :100).
// --------------------------------------------------------------------------------------------
// One WARP per plane row (n, tp, pl, yy): the 88-pixel input row is read once with coalesced 16-byte loads into a
// zero-bordered shared-memory line, every lane then assembles its entries (8 consecutive pixels at even offsets)
// from that line and the warp stores 512 contiguous bytes.
__global__ void __launch_bounds__(256)
prep_clip_kernel(const float* __restrict__ x, uint4* __restrict__ out, int N, int T) {
  using namespace c3d;
  __shared__ __align__(16) float line[8][104];   // [warp][3 zero | 88 pixels | zeros up to 2*43 + 8 = 94 (+ slack)]
  const int TP = T + 2 * TPAD;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long rows = static_cast<long long>(N) * TP * 2 * PLANE_ROWS;
  float* ln = line[warp];
  for (int i = lane; i < 104; i += 32) ln[i] = 0.0f;   // borders stay zero for the whole kernel
  __syncwarp();
  for (long long row = static_cast<long long>(blockIdx.x) * 8 + warp; row < rows;
       row += static_cast<long long>(gridDim.x) * 8) {
    const int yy = static_cast<int>(row % PLANE_ROWS);
    long long r = row / PLANE_ROWS;
    const int pl = static_cast<int>(r & 1);
    r >>= 1;
    const int tp = static_cast<int>(r % TP);
    const int n = static_cast<int>(r / TP);
    const int t = tp - TPAD;
    const int y = 2 * yy + pl - 3;
    const bool inside = t >= 0 && t < T && y >= 0 && y < IN_HW;   // warp-uniform
    uint4* dst = out + ((static_cast<long long>(n) * TP + tp) * 2 + pl) * PLANE_ENTRIES + yy * CONV_HW;
    if (inside) {
      if (lane < IN_HW / 4) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(
                                   x + ((static_cast<long long>(n) * T + t) * IN_HW + y) * IN_HW) + lane);
        ln[3 + 4 * lane + 0] = v.x; ln[3 + 4 * lane + 1] = v.y; ln[3 + 4 * lane + 2] = v.z; ln[3 + 4 * lane + 3] = v.w;
      }
      __syncwarp();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cx = lane + 32 * h;
        if (cx < CONV_HW) {
          const float2* src = reinterpret_cast<const float2*>(ln + 2 * cx);
          const float2 a = src[0], b = src[1], c = src[2], d = src[3];
          uint4 o;
          o.x = pack_bf16x2(a.x, a.y);
          o.y = pack_bf16x2(b.x, b.y);
          o.z = pack_bf16x2(c.x, c.y);
          o.w = pack_bf16x2(d.x, d.y);
          dst[cx] = o;
        }
      }
      __syncwarp();   // the line is rewritten by the next row
    } else {
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      dst[lane] = z;
      if (lane + 32 < CONV_HW) dst[lane + 32] = z;
    }
    if (yy == PLANE_ROWS - 1 && lane < PLANE_ENTRIES - PLANE_ROWS * CONV_HW)
      dst[CONV_HW + lane] = make_uint4(0u, 0u, 0u, 0u);   // the 4 zero entries that pad the plane to 128 bytes
  }
}

// --------------------------------------------------------------------------------------------
// Fused input pipeline: raw uint8 gray frames -> the same row-Toeplitz bf16 layout, in one pass.
// Reference (SBL/data_gen.py:122-125,276-296 + cvtransforms.py:7-20,44-48): np.load(uint8 [T,H0,W0]) / 255. ->
// ColorNormalize ((x - 0.413621) / 0.1700239) -> CenterCrop / RandomCrop to 88x88 (per-frame offsets) -> zero-pad the
// clip to T_out frames (zeros in NORMALISED space) -> float32 tensor -> model.  Here the host ships the uint8 frames
// (4x fewer PCIe / host-memory bytes than the fp32 tensor the reference builds on the CPU) and the normalisation is
// a 256-entry table lut[u] = bf16(float32((u / 255. - mean) / std)) evaluated in float64 on the host exactly like
// numpy does, so the result is BIT-IDENTICAL to prep_clip(reference-normalised fp32 clip).
// crop_yx: optional int32 [N*T_in][2] per-frame (y1, x1) offsets (RandomCrop), else the uniform (crop_y0, crop_x0).
// One warp per plane row, like prep_clip_kernel.
__global__ void __launch_bounds__(256)
prep_clip_u8_kernel(const uint8_t* __restrict__ x, const uint16_t* __restrict__ lut_bf16,
                    const int* __restrict__ crop_yx, int crop_y0, int crop_x0, uint4* __restrict__ out, int N, int T_in,
                    int T_out, int H0, int W0) {
  using namespace c3d;
  __shared__ uint16_t lut[256];
  __shared__ __align__(16) uint16_t line[8][104];   // [warp][3 zero | 88 pixels (bf16 bits) | zeros ...]
  const int TP = T_out + 2 * TPAD;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  lut[threadIdx.x] = lut_bf16[threadIdx.x];
  const long long rows = static_cast<long long>(N) * TP * 2 * PLANE_ROWS;
  uint16_t* ln = line[warp];
  for (int i = lane; i < 104; i += 32) ln[i] = 0;   // borders stay zero for the whole kernel
  __syncthreads();
  for (long long row = static_cast<long long>(blockIdx.x) * 8 + warp; row < rows;
       row += static_cast<long long>(gridDim.x) * 8) {
    const int yy = static_cast<int>(row % PLANE_ROWS);
    long long r = row / PLANE_ROWS;
    const int pl = static_cast<int>(r & 1);
    r >>= 1;
    const int tp = static_cast<int>(r % TP);
    const int n = static_cast<int>(r / TP);
    const int t = tp - TPAD;
    const int y = 2 * yy + pl - 3;
    const bool inside = t >= 0 && t < T_in && y >= 0 && y < IN_HW;   // warp-uniform (frames >= T_in are zero padding)
    uint4* dst = out + ((static_cast<long long>(n) * TP + tp) * 2 + pl) * PLANE_ENTRIES + yy * CONV_HW;
    if (inside) {
      const long long fr = static_cast<long long>(n) * T_in + t;
      const int cy = crop_yx != nullptr ? __ldg(crop_yx + 2 * fr) : crop_y0;
      const int cx0 = crop_yx != nullptr ? __ldg(crop_yx + 2 * fr + 1) : crop_x0;
      const uint8_t* src = x + (fr * H0 + (cy + y)) * W0 + cx0;
      for (int i = lane; i < IN_HW; i += 32) ln[3 + i] = lut[__ldg(src + i)];
      __syncwarp();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cx = lane + 32 * h;
        if (cx < CONV_HW) {
          const uint32_t* s32 = reinterpret_cast<const uint32_t*>(ln + 2 * cx);   // even index: 4-byte aligned
          dst[cx] = make_uint4(s32[0], s32[1], s32[2], s32[3]);
        }
      }
      __syncwarp();   // the line is rewritten by the next row
    } else {
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      dst[lane] = z;
      if (lane + 32 < CONV_HW) dst[lane + 32] = z;
    }
    if (yy == PLANE_ROWS - 1 && lane < PLANE_ENTRIES - PLANE_ROWS * CONV_HW)
      dst[CONV_HW + lane] = make_uint4(0u, 0u, 0u, 0u);   // the 4 zero entries that pad the plane to 128 bytes
  }
}

// --------------------------------------------------------------------------------------------
// Weight packers.  Eval-mode BatchNorm y = (x - mean) * gamma / sqrt(var + eps) + beta is folded:
//   w' = w * gamma / sqrt(var + eps)   (per output channel), bias' = beta - mean * gamma / sqrt(var + eps)
// Reference BN call sites: video_frontend.py:21,24,71,101 (eps = 1e-5 PyTorch default).
// --------------------------------------------------------------------------------------------
// Conv2d weight fp32 [Co,Ci,R,S] -> bf16 [Co][R][S][Ci] (K-major for the implicit GEMM), bias fp32 [Co].
__global__ void __launch_bounds__(256)
pack_conv2d_kernel(const float* __restrict__ w, const float* __restrict__ gamma, const float* __restrict__ beta,
                   const float* __restrict__ mean, const float* __restrict__ var, float eps,
                   __nv_bfloat16* __restrict__ wp, float* __restrict__ bias, int Co, int Ci, int R, int S) {
  const int total = Co * Ci * R * S;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ci = i % Ci;
    int r = i / Ci;
    const int s = r % S;
    r /= S;
    const int rr = r % R;
    const int co = r / R;
    const float scale = (gamma != nullptr) ? gamma[co] / sqrtf(var[co] + eps) : 1.0f;
    wp[i] = __float2bfloat16_rn(w[((co * Ci + ci) * R + rr) * S + s] * scale);
    if (ci == 0 && s == 0 && rr == 0 && bias != nullptr) {
      bias[co] = (gamma != nullptr) ? beta[co] - mean[co] * scale : 0.0f;
    }
  }
}

// Conv3d stem weight fp32 [64,1,5,7,7] -> bf16 [64][320] in the MMA order of sblk_conv3d.cuh:
//   k = dt*64 + q*16 + h*8 + s  with filter row r = 2q + h ; r == 7 and s == 7 are zero.
__global__ void __launch_bounds__(256)
pack_conv3d_kernel(const float* __restrict__ w, const float* __restrict__ gamma, const float* __restrict__ beta,
                   const float* __restrict__ mean, const float* __restrict__ var, float eps,
                   __nv_bfloat16* __restrict__ wp, float* __restrict__ bias) {
  const int total = c3d::COUT * c3d::KPAD;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i % c3d::KPAD;
    const int co = i / c3d::KPAD;
    const float scale = gamma[co] / sqrtf(var[co] + eps);
    float v = 0.0f;
    const int dt = k >> 6;
    const int r = ((k >> 4) & 3) * 2 + ((k >> 3) & 1);
    const int s = k & 7;
    if (r < 7 && s < 7) v = w[((co * 5 + dt) * 7 + r) * 7 + s] * scale;
    wp[i] = __float2bfloat16_rn(v);
    if (k == 0) bias[co] = beta[co] - mean[co] * scale;
  }
}

// fp32 -> bf16 / fp16 cast (Linear weights, encoder input).  n must be a multiple of 4.
__global__ void __launch_bounds__(256)
cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n4, int fp16) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    uint2 o;
    o.x = fp16 ? pack_f16x2(v.x, v.y) : pack_bf16x2(v.x, v.y);
    o.y = fp16 ? pack_f16x2(v.z, v.w) : pack_bf16x2(v.z, v.w);
    reinterpret_cast<uint2*>(dst)[i] = o;
  }
}

// L2 prefetch of one read-only range (packed weights of the layers that run later in the same forward):
// prefetch.global.L2 of every 128-byte line, no shared memory and few registers, so the few CTAs co-reside with the
// persistent conv kernels.  The bench flushes L2 between steps, so without it every kernel's first weight tiles (and
// the whole dependent chain of the encoder stack) pay DRAM latency.
__global__ void __launch_bounds__(256)
l2_prefetch_kernel(const uint8_t* base, long long lines) {   // base 128-byte aligned
#pragma unroll 1
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < lines;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(base + i * 128));
}

// --------------------------------------------------------------------------------------------
// One-shot all-gather of the per-GPU encoder outputs over NVLink / NVSwitch peer memory (one process per GPU).
// Reference: nn.DataParallel's gather of the replicas' outputs, SBL/train.py:114-115.  Every rank holds, for each
// peer, a mapped pointer to that peer's gather buffer [world][n] and flag array [world] (CUDA IPC).  One kernel:
//   1. each thread reads 16 bytes of the local block once and stores them into slot `rank` of EVERY rank's buffer
//      (peer stores travel over NVLink; the peers are visited in a rank-staggered order),
//   2. the last CTA to finish (device-scope counter after a system-scope fence) publishes flag[rank] = epoch in every
//      rank's flag array with a system-scope release store,
//   3. and then waits (acquire loads, wall-clock watchdog) until all `world` flags of ITS OWN array carry the epoch:
//      when the kernel completes, every peer's block has landed in the local buffer — the completion semantics of
//      ncclAllGather, without its ~60 us of latency for 8 x 1.9 MB.
// Epochs increase by one per call; callers alternate two buffers so a peer that runs one step ahead never overwrites
// a block that may still be read.
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
p2p_gather_kernel(const uint4* __restrict__ local, uint4* const* __restrict__ peer_bufs,
                  unsigned int* const* __restrict__ peer_flags, unsigned int* __restrict__ counter, int rank, int world,
                  long long n16, unsigned int epoch, unsigned long long timeout_ns) {
  __shared__ int is_last;
  const long long slot = static_cast<long long>(rank) * n16;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n16;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 v = __ldg(local + i);
    for (int k = 0; k < world; ++k) {
      uint4* dst = peer_bufs[(rank + k) % world];
      dst[slot + i] = v;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  if (threadIdx.x == 0) *counter = 0u;   // ready for the next call (stream-ordered)
  if (threadIdx.x < world) {
    __threadfence_system();
    unsigned int* f = peer_flags[threadIdx.x] + rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(epoch) : "memory");
    const unsigned int* mine = peer_flags[rank] + threadIdx.x;
    unsigned int seen;
    unsigned long long t0 = 0;
    unsigned int polls = 0;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(mine) : "memory");
      if (static_cast<int>(seen - epoch) >= 0) break;
      if ((++polls & 255u) == 0u) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        if (now - t0 > timeout_ns) {   // a peer did not show up (sblk_set_p2p_timeout_ms; a data-loader stall is not an error)
          unsigned int* wd = g_sblk_watchdog_ptr;
          if (wd != nullptr) {
            atomicCAS_system(wd, 0u, 0x0901u | 0x80000000u);
            __threadfence_system();
          }
          __trap();
        }
      }
    } while (true);
  }
}

// --------------------------------------------------------------------------------------------
// Global average pool: bf16 NHWC [F, HW, C] -> fp32 [F, C] (+ optional bf16 copy), optionally times a per-element
// fp32 factor [F, C] (the always-on dropout of Lipreading.forward, video_frontend.py:122, with its mask * 1/(1-p)
// drawn ahead of time: mean * (mask * 2) == (mean * mask) * 2 bit for bit).
// Reference: ResNet.avgpool + view, SBL/transformer/video_frontend.py:87-88.
// One thread per (frame, channel pair).
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
avgpool_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ scale, float* __restrict__ out_f32,
               __nv_bfloat16* __restrict__ out_bf16, int F, int HW, int C, int out_fp16) {
  const int C2 = C >> 1;
  const long long total = static_cast<long long>(F) * C2;
  const float inv = 1.0f / static_cast<float>(HW);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c2 = static_cast<int>(i % C2);
    const long long f = i / C2;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(x) + f * HW * C2 + c2;
    float a = 0.0f, b = 0.0f;
    for (int q = 0; q < HW; ++q) {
      const uint32_t u = __ldg(src + static_cast<long long>(q) * C2);
      a += bf16_lo(u);
      b += bf16_hi(u);
    }
    a *= inv;
    b *= inv;
    if (scale != nullptr) {
      const float2 m = __ldg(reinterpret_cast<const float2*>(scale) + i);
      a *= m.x;
      b *= m.y;
    }
    if (out_f32 != nullptr) reinterpret_cast<float2*>(out_f32)[i] = make_float2(a, b);
    if (out_bf16 != nullptr)
      reinterpret_cast<uint32_t*>(out_bf16)[i] = out_fp16 ? pack_f16x2(a, b) : pack_bf16x2(a, b);
  }
}

// Same pooling, one thread per (frame, 8 channels): 16-byte loads (nine of them in flight per thread for the 3x3 maps
// of layer 4), 16/32-byte stores; the per-channel summation order is that of avgpool_kernel (bit-identical).
// PDL-enabled: it is the launch between the last conv and the encoder stack.
__global__ void __launch_bounds__(256)
avgpool8_kernel(const uint4* __restrict__ x, const float* __restrict__ scale, float* __restrict__ out_f32,
                void* __restrict__ out_16, int F, int HW, int C8, int out_fp16) {
  grid_dep_launch();
  grid_dep_wait();
  const long long total = static_cast<long long>(F) * C8;
  const float inv = 1.0f / static_cast<float>(HW);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % C8);
    const long long f = i / C8;
    const uint4* src = x + f * HW * C8 + c8;
    float a[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] = 0.0f;
#pragma unroll 9
    for (int q = 0; q < HW; ++q) {
      const uint4 u = __ldg(src + static_cast<long long>(q) * C8);
      a[0] += bf16_lo(u.x); a[1] += bf16_hi(u.x); a[2] += bf16_lo(u.y); a[3] += bf16_hi(u.y);
      a[4] += bf16_lo(u.z); a[5] += bf16_hi(u.z); a[6] += bf16_lo(u.w); a[7] += bf16_hi(u.w);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] *= inv;
    if (scale != nullptr) {
      const float4 m0 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * i);
      const float4 m1 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * i + 1);
      a[0] *= m0.x; a[1] *= m0.y; a[2] *= m0.z; a[3] *= m0.w;
      a[4] *= m1.x; a[5] *= m1.y; a[6] *= m1.z; a[7] *= m1.w;
    }
    if (out_f32 != nullptr) {
      reinterpret_cast<float4*>(out_f32)[2 * i] = make_float4(a[0], a[1], a[2], a[3]);
      reinterpret_cast<float4*>(out_f32)[2 * i + 1] = make_float4(a[4], a[5], a[6], a[7]);
    }
    if (out_16 != nullptr) {
      uint4 o;
      if (out_fp16) {
        o.x = pack_f16x2(a[0], a[1]); o.y = pack_f16x2(a[2], a[3]);
        o.z = pack_f16x2(a[4], a[5]); o.w = pack_f16x2(a[6], a[7]);
      } else {
        o.x = pack_bf16x2(a[0], a[1]); o.y = pack_bf16x2(a[2], a[3]);
        o.z = pack_bf16x2(a[4], a[5]); o.w = pack_bf16x2(a[6], a[7]);
      }
      reinterpret_cast<uint4*>(out_16)[i] = o;
    }
  }
}

// --------------------------------------------------------------------------------------------
// y = LayerNorm(x + residual) * gamma + beta  (+ pe[t])  (* pad_mask[b,t]),  D = 512, eps = 1e-5.
// Reference: attention.py:58, module.py:51, encoder.py:53-55 (+PE), encoder.py:86,89 (mask).
// One warp per row; the row lives in registers (16 values per lane); two-pass mean / variance in fp32.
// Writes the fp32 residual stream and the 16-bit (enc16_t) copy the next GEMM consumes.
// --------------------------------------------------------------------------------------------
struct LnParams {
  const float* x;         // [nparts][M, 512] GEMM output (split-K partials are summed here; bias added if given)
  int nparts;             // >= 1
  long long part_stride;  // elements between partials
  const float* bias;      // [512] or nullptr
  const float* residual;  // [M, 512] or nullptr
  const float* gamma;     // [512]
  const float* beta;      // [512]
  const float* pe;        // [>=T, 512] or nullptr ; row t = m % T
  const int* lengths;     // [M / T] or nullptr ; rows with t >= lengths[b] are zeroed
  float* out_f32;         // [M, 512] or nullptr
  enc16_t* out_bf16;        // [M, 512] or nullptr (encoder operand format, sblk_common.cuh)
  int M;
  int T;
  float eps;
};

__global__ void __launch_bounds__(256)
add_layernorm512_kernel(const LnParams p) {
  grid_dep_launch();  // PDL: let the next kernel start its prologue now; its own wait orders the data
  grid_dep_wait();
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  for (int m = blockIdx.x * warps_per_block + (threadIdx.x >> 5); m < p.M; m += gridDim.x * warps_per_block) {
    const float4* xr = reinterpret_cast<const float4*>(p.x + static_cast<size_t>(m) * 512);
    float v[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 a = __ldg(xr + j * 32 + lane);
      v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
    }
    for (int s = 1; s < p.nparts; ++s) {
      const float4* xs = reinterpret_cast<const float4*>(p.x + s * p.part_stride + static_cast<size_t>(m) * 512);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 a = __ldg(xs + j * 32 + lane);
        v[4 * j] += a.x; v[4 * j + 1] += a.y; v[4 * j + 2] += a.z; v[4 * j + 3] += a.w;
      }
    }
    if (p.bias != nullptr) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(p.bias) + j * 32 + lane);
        v[4 * j] += a.x; v[4 * j + 1] += a.y; v[4 * j + 2] += a.z; v[4 * j + 3] += a.w;
      }
    }
    if (p.residual != nullptr) {
      const float4* rr = reinterpret_cast<const float4*>(p.residual + static_cast<size_t>(m) * 512);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 a = __ldg(rr + j * 32 + lane);
        v[4 * j] += a.x; v[4 * j + 1] += a.y; v[4 * j + 2] += a.z; v[4 * j + 3] += a.w;
      }
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += v[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.0f / 512.0f);
    float q = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float d = v[j] - mean;
      q += d * d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q * (1.0f / 512.0f) + p.eps);
    const int t = m % p.T;
    float keep = 1.0f;
    if (p.lengths != nullptr && t >= __ldg(p.lengths + m / p.T)) keep = 0.0f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col4 = j * 32 + lane;
      const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma) + col4);
      const float4 b = __ldg(reinterpret_cast<const float4*>(p.beta) + col4);
      float4 y;
      y.x = (v[4 * j] - mean) * rstd * g.x + b.x;
      y.y = (v[4 * j + 1] - mean) * rstd * g.y + b.y;
      y.z = (v[4 * j + 2] - mean) * rstd * g.z + b.z;
      y.w = (v[4 * j + 3] - mean) * rstd * g.w + b.w;
      if (p.pe != nullptr) {
        const float4 e = __ldg(reinterpret_cast<const float4*>(p.pe + static_cast<size_t>(t) * 512) + col4);
        y.x += e.x; y.y += e.y; y.z += e.z; y.w += e.w;
      }
      y.x *= keep; y.y *= keep; y.z *= keep; y.w *= keep;
      if (p.out_f32 != nullptr)
        reinterpret_cast<float4*>(p.out_f32 + static_cast<size_t>(m) * 512)[col4] = y;
      if (p.out_bf16 != nullptr) {
        uint2 o;
        o.x = pack_e16x2(y.x, y.y);
        o.y = pack_e16x2(y.z, y.w);
        reinterpret_cast<uint2*>(p.out_bf16 + static_cast<size_t>(m) * 512)[col4] = o;
      }
    }
  }
}

// --------------------------------------------------------------------------------------------
// Co-scheduling gate (one thread): returns once `count` more CTAs have bumped gate[0] than the running target gate[1]
// records, or after timeout_ns (the gate only ORDERS the placement of two concurrent kernel chains; results never depend
// on it, so giving up is safe).  gate[1] advances by `count` either way, so late arrivals of this round are accounted for
// when the next round starts (rounds are stream-ordered: all CTAs of a round have run before the next gate launch).
__global__ void gate_wait_kernel(unsigned int* gate, unsigned int count, unsigned long long timeout_ns) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const unsigned int target = gate[1] + count;
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    unsigned int v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(gate) : "memory");
    if (static_cast<int>(v - target) >= 0) break;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > timeout_ns) break;
    __nanosleep(200);
  }
  gate[1] = target;
}

}  // namespace sblk

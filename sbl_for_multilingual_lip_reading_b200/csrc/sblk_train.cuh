// sblk_train.cuh — the memory-bound kernels of the TRAINING path (forward with batch statistics + backward).
//
// Reference behaviour being reproduced: `model.train()` + `loss.backward()` through the hot path,
//   VSR_visual_frontend_pretraining_on_LRW_LRW1000_classify/train.py:107-146 and SBL/train.py:177-210:
//   BatchNorm2d/3d in training mode (batch statistics, biased variance for the normalisation, running statistics updated
//   with momentum 0.1 and the unbiased variance: video_frontend.py:21,24,71,101), ReLU, MaxPool3d((1,3,3),(1,2,2),(0,1,1)),
//   AdaptiveAvgPool2d, LayerNorm, scaled-dot-product attention with dropout on the probabilities (attention.py:72-83).
// Every contraction of the backward pass (dgrad, wgrad, Linear backward) runs on the tcgen05 GEMM / conv kernels of the
// forward path: dgrad of a stride-1 3x3 conv IS a 3x3 conv with the flipped, transposed filter; dgrad of a stride-2 conv is
// that conv over the zero-stuffed gradient; wgrad is a split-K GEMM dY^T [Cout, M] x col^T [9 Cin, M]^T whose operands are
// produced K-major by the transposing kernels below.  What lives here is everything around them: layout changes
// (transpose, im2col, zero-stuffing), per-channel reductions, and the elementwise / row-wise derivative formulas, all
// fp32 math on bf16 (convolutional trunk, every gradient) or enc16 (saved encoder activations) storage.
#pragma once
#include "sblk_common.cuh"

namespace sblk {

__device__ __forceinline__ float ld16(const uint16_t* p, int fp16) {
  const uint16_t u = *p;
  return fp16 ? __half2float(__ushort_as_half(u)) : __uint_as_float(static_cast<uint32_t>(u) << 16);
}
__device__ __forceinline__ float lo16(uint32_t u, int fp16) { return fp16 ? f16_lo(u) : bf16_lo(u); }
__device__ __forceinline__ float hi16(uint32_t u, int fp16) { return fp16 ? f16_hi(u) : bf16_hi(u); }

// ----------------------------------------------------------------------------------------------------------------
// 16-bit transpose: in [R, C] (row pitch ld_in elements) -> out [C, ld_out] with out[c][r] = in[r][c] for r < R and 0 for
// R <= r < ld_out (K padding of the wgrad GEMMs).  convert = 1 re-rounds IEEE fp16 input to bf16 (saved enc16
// activations feeding a bf16 gradient GEMM).  64 x 64 tiles through shared memory, coalesced both ways.
// ----------------------------------------------------------------------------------------------------------------
// Shared 64 x 64 tile of 16-bit values, 128-byte rows, 16-byte chunk c of row r stored at chunk c ^ ((r >> 3) & 7):
// load: thread -> (row, 8-column chunk) as one 16-byte store (a quarter-warp covers one row: conflict-free);
// store: thread -> (column, 8-row chunk) gathered with 8 halfword reads (lanes of a warp differ in the row group, i.e. in
// the swizzled chunk position: conflict-free) and written to global memory as one 16-byte access.
struct Tile64 {
  uint16_t v[64 * 64];
};
__device__ __forceinline__ uint4* tile_chunk(Tile64& t, int row, int chunk) {
  return reinterpret_cast<uint4*>(&t.v[row * 64 + ((chunk ^ ((row >> 3) & 7)) << 3)]);
}
__device__ __forceinline__ uint4 tile_gather_col8(const Tile64& t, int col, int row0) {   // row0 % 8 == 0
  const int off = (((col >> 3) ^ ((row0 >> 3) & 7)) << 3) + (col & 7);
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    w[j] = static_cast<uint32_t>(t.v[(row0 + 2 * j) * 64 + off]) |
           (static_cast<uint32_t>(t.v[(row0 + 2 * j + 1) * 64 + off]) << 16);
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ uint4 cvt8_f16_to_bf16(uint4 u) {
  uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) w[j] = pack_bf16x2(f16_lo(w[j]), f16_hi(w[j]));
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// Requires C % 8 == 0, ld_in % 8 == 0, ld_out % 8 == 0 and 16-byte aligned bases (checked by the C ABI).
__global__ void __launch_bounds__(256)
transpose16_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, long long R, int C, long long ld_in,
                   long long ld_out, int convert) {
  __shared__ __align__(16) Tile64 tile;
  const long long tiles_r = (ld_out + 63) / 64;
  const int tiles_c = (C + 63) / 64;
  const long long total = tiles_r * tiles_c;
  for (long long tI = blockIdx.x; tI < total; tI += gridDim.x) {
    const long long tr = tI / tiles_c;
    const int tc = static_cast<int>(tI - tr * tiles_c);
    const long long r0 = tr * 64;
    const int c0 = tc * 64;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = threadIdx.x + 256 * i;      // 512 chunks: 64 rows x 8 chunks
      const int rr = idx >> 3, ch = idx & 7;
      const long long r = r0 + rr;
      const int c = c0 + ch * 8;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (r < R && c < C) {
        v = __ldg(reinterpret_cast<const uint4*>(in + r * ld_in + c));
        if (convert) v = cvt8_f16_to_bf16(v);
      }
      *tile_chunk(tile, rr, ch) = v;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = threadIdx.x + 256 * i;      // 512 chunks: 64 columns x 8 row-chunks
      const int cc = idx >> 3, rc = idx & 7;
      const int c = c0 + cc;
      const long long r = r0 + rc * 8;
      if (c < C && r < ld_out)
        *reinterpret_cast<uint4*>(out + static_cast<long long>(c) * ld_out + r) = tile_gather_col8(tile, cc, rc * 8);
    }
    __syncthreads();
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Transposed im2col of an NHWC bf16 tensor for the wgrad GEMM of a Conv2d (R x S taps, stride, pad):
//   out[(tap * C + c)][m] = x[f, p*stride + r - pad, q*stride + s - pad, c]   (0 outside the image and for m >= M),
//   m = (f * P + p) * Q + q, tap = r * S + s, out row pitch ld_out >= M.
// One block = 64 output pixels x 64 channels of one tap, transposed through shared memory.
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
im2col_t_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ out, int F, int H, int W, int C, int P, int Q,
                int R, int S, int stride, int pad, long long ld_out) {
  __shared__ __align__(16) Tile64 tile;
  const long long M = static_cast<long long>(F) * P * Q;
  const long long tiles_m = (ld_out + 63) / 64;
  const int tiles_c = C / 64;
  const int taps = R * S;
  const long long total = tiles_m * tiles_c * taps;
  for (long long tI = blockIdx.x; tI < total; tI += gridDim.x) {
    const long long tm = tI / (tiles_c * taps);
    const int rest = static_cast<int>(tI - tm * (tiles_c * taps));
    const int tap = rest / tiles_c;
    const int tc = rest - tap * tiles_c;
    const int r = tap / S, s = tap - r * S;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = threadIdx.x + 256 * i;      // 64 pixels x 8 channel chunks
      const int mm = idx >> 3, ch = idx & 7;
      const long long m = tm * 64 + mm;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (m < M) {
        const int q = static_cast<int>(m % Q);
        const long long t2 = m / Q;
        const int pp = static_cast<int>(t2 % P);
        const long long f = t2 / P;
        const int y = pp * stride + r - pad, xx = q * stride + s - pad;
        if (y >= 0 && y < H && xx >= 0 && xx < W)
          v = __ldg(reinterpret_cast<const uint4*>(x + ((f * H + y) * W + xx) * static_cast<long long>(C) + tc * 64 + ch * 8));
      }
      *tile_chunk(tile, mm, ch) = v;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int idx = threadIdx.x + 256 * i;      // 64 channels x 8 pixel chunks
      const int cc = idx >> 3, mc = idx & 7;
      const long long m = tm * 64 + mc * 8;
      if (m < ld_out)
        *reinterpret_cast<uint4*>(out + (static_cast<long long>(tap) * C + tc * 64 + cc) * ld_out + m) =
            tile_gather_col8(tile, cc, mc * 8);
    }
    __syncthreads();
  }
}

// ----------------------------------------------------------------------------------------------------------------
// im2col of the Conv3d stem (Cin = 1, 5x7x7 taps, stride (1,2,2), pad (2,3,3), video_frontend.py:100):
//   x fp32 [N, T, 88, 88];  k = (dt*7 + r)*7 + s < 245, zero-padded to 256;  m = ((n*T + t)*44 + y)*44 + xo.
//   transposed == 0: col [M, 256] bf16 (forward GEMM A operand)     transposed == 1: colT [256, ld_out] (wgrad B operand)
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float stem_tap(const float* __restrict__ x, int T, long long n, int t, int y, int xo, int k) {
  if (k >= 245) return 0.0f;
  const int dt = k / 49, rs = k - dt * 49, r = rs / 7, s = rs - r * 7;
  const int tt = t + dt - 2, yy = 2 * y + r - 3, xx = 2 * xo + s - 3;
  if (tt < 0 || tt >= T || yy < 0 || yy >= 88 || xx < 0 || xx >= 88) return 0.0f;
  return __ldg(x + ((n * T + tt) * 88 + yy) * 88 + xx);
}

// transposed == 0: blockIdx.x = output row (f, y); threads = 44 pixels x 32 chunks of 8 taps, 16-byte stores
// transposed == 1: blockIdx.x = tap k (256), blockIdx.y = frame slot (1936 consecutive m); 2-pixel 4-byte stores
__global__ void __launch_bounds__(256)
stem_im2col_kernel(const float* __restrict__ x, uint16_t* __restrict__ out, int N, int T, int transposed,
                   long long ld_out) {
  const long long M = static_cast<long long>(N) * T * 44 * 44;
  if (!transposed) {
    const int fy = blockIdx.x;                  // f * 44 + y
    const int y = fy % 44;
    const int f = fy / 44;
    const int t = f % T;
    const long long n = f / T;
    uint4* dst = reinterpret_cast<uint4*>(out) + static_cast<long long>(fy) * 44 * 32;
    for (int i = threadIdx.x; i < 44 * 32; i += blockDim.x) {
      const int xo = i >> 5;
      const int k0 = (i & 31) * 8;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = stem_tap(x, T, n, t, y, xo, k0 + j);
      uint4 o;
      o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
      o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
      dst[i] = o;
    }
  } else {
    const int k = blockIdx.x;
    const long long m0 = static_cast<long long>(blockIdx.y) * 1936;
    const int f = blockIdx.y;
    const bool real = k < 245 && f < N * T;
    const int t = real ? f % T : 0;
    const long long n = real ? f / T : 0;
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + static_cast<long long>(k) * ld_out + m0);
    for (int i = threadIdx.x; i < 968; i += blockDim.x) {      // 968 pixel pairs of one frame
      const long long m = m0 + 2 * i;
      if (m >= ld_out) break;
      float a = 0.0f, b = 0.0f;
      if (real) {
        const int px = 2 * i;
        const int y = px / 44, xo = px - y * 44;              // 44 is even: both pixels in the same row
        a = stem_tap(x, T, n, t, y, xo, k);
        b = stem_tap(x, T, n, t, y, xo + 1, k);
      }
      if (m + 1 < ld_out) dst[i] = pack_bf16x2(a, b);
      else *reinterpret_cast<uint16_t*>(dst + i) = static_cast<uint16_t>(pack_bf16x2(a, 0.0f) & 0xFFFFu);
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------
// The same im2col straight from the training loader's raw uint8 gray frames x [N, T_in, H0, W0]: the clip value at
// (n, t, y, x) is lut[x[n, t, cy + y, cx + (flip[n] ? 87 - x : x)]] for t < T_in and 0 for T_in <= t < T (frame
// zero-padding in normalised space), with (cy, cx) = crop_yx[n*T_in + t] clamped into [0, H0-88] x [0, W0-88] (the
// offsets live in device memory, where the C ABI cannot check them), or (crop_y0, crop_x0) when crop_yx is null.
// lut[u] = bf16(float32((u/255 - mean)/std)) is what pack_bf16x2 makes of the reference loader's fp32 clip, so the
// output is bit-identical to stem_im2col_kernel on that clip.  Same grids and output layouts as stem_im2col_kernel.
// ----------------------------------------------------------------------------------------------------------------
struct StemU8Src {
  const uint8_t* x;
  const uint16_t* lut;   // bf16 bits [256]
  const int* crop_yx;    // [N*T_in][2] (y, x) or nullptr
  const int* flip;       // [N] or nullptr
  int crop_y0, crop_x0, N, T_in, T, H0, W0;
};

// top-left pixel of the 88x88 crop of clip frame (n, t), t < T_in
__device__ __forceinline__ const uint8_t* stem_u8_crop(const StemU8Src& s, long long n, int t) {
  const long long fr = n * s.T_in + t;
  int cy = s.crop_y0, cx = s.crop_x0;
  if (s.crop_yx != nullptr) {
    cy = min(max(__ldg(s.crop_yx + 2 * fr), 0), s.H0 - 88);
    cx = min(max(__ldg(s.crop_yx + 2 * fr + 1), 0), s.W0 - 88);
  }
  return s.x + (fr * s.H0 + cy) * s.W0 + cx;
}

// transposed == 0: blockIdx.x = output row (f, y); the 5 frames x 7 rows x 94 columns (88 + the 3-pixel halo on either
//   side) its 44 x 245 taps read are normalised once into shared memory, then the taps are stored as in stem_im2col_kernel
// transposed == 1: blockIdx.x = temporal tap dt (5: the zero rows 245..255), blockIdx.y = frame slot; the one source frame
//   the 49 taps (dt, r, s) read is normalised (and mirrored) once into a zero-haloed 94 x 94 tile in shared memory, then
//   each of the 49 output rows gets the slot's 1936 pixels as 2-pixel 4-byte stores
constexpr int kStemU8Tile = 94 * 96;       // uint16 elements: the transposed tile (row pitch 96); holds the 35 x 96 window
__global__ void __launch_bounds__(256)
stem_im2col_u8_kernel(StemU8Src s, uint16_t* __restrict__ out, int transposed, long long ld_out) {
  __shared__ uint16_t lut[256];
  __shared__ __align__(16) uint16_t tile[kStemU8Tile];
  __shared__ const uint8_t* crop[5];          // transposed == 0: crops of the frames t-2 .. t+2 (nullptr: zero frame)
  lut[threadIdx.x] = __ldg(s.lut + threadIdx.x);
  if (!transposed) {
    uint16_t (*win)[96] = reinterpret_cast<uint16_t (*)[96]>(tile);   // [5 * 7][96]
    const int fy = blockIdx.x;                  // f * 44 + y
    const int y = fy % 44;
    const int f = fy / 44;
    const int t = f % s.T;
    const long long n = f / s.T;
    if (threadIdx.x < 5) {
      const int tt = t + static_cast<int>(threadIdx.x) - 2;
      crop[threadIdx.x] = (tt >= 0 && tt < s.T_in) ? stem_u8_crop(s, n, tt) : nullptr;
    }
    __syncthreads();
    const bool mirror = s.flip != nullptr && __ldg(s.flip + n) != 0;
    for (int i = threadIdx.x; i < 5 * 7 * 94; i += blockDim.x) {
      const int row = i / 94, col = i - row * 94;
      const int dt = row / 7, r = row - dt * 7;
      const int yy = 2 * y + r - 3, xx = col - 3;
      const uint8_t* src = crop[dt];
      uint16_t v = 0;
      if (src != nullptr && yy >= 0 && yy < 88 && xx >= 0 && xx < 88)
        v = lut[__ldg(src + yy * s.W0 + (mirror ? 87 - xx : xx))];
      win[row][col] = v;
    }
    __syncthreads();
    uint4* dst = reinterpret_cast<uint4*>(out) + static_cast<long long>(fy) * 44 * 32;
    for (int i = threadIdx.x; i < 44 * 32; i += blockDim.x) {
      const int xo = i >> 5;
      const int k0 = (i & 31) * 8;
      uint32_t w[4];
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        uint32_t h[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int k = k0 + j + e;
          const int dt = k / 49, rs = k - dt * 49, r = rs / 7, sx = rs - r * 7;
          h[e] = k < 245 ? win[dt * 7 + r][2 * xo + sx] : 0u;
        }
        w[j >> 1] = h[0] | (h[1] << 16);
      }
      dst[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  } else {
    const int dt = blockIdx.x;
    const int f = blockIdx.y;
    const long long m0 = static_cast<long long>(f) * 1936;
    const int t = f % s.T;
    const int tt = t + dt - 2;
    const bool real = dt < 5 && f < s.N * s.T && tt >= 0 && tt < s.T_in;   // block-uniform
    __syncthreads();
    if (real) {
      const long long n = f / s.T;
      const uint8_t* src = stem_u8_crop(s, n, tt);
      const bool mirror = s.flip != nullptr && __ldg(s.flip + n) != 0;
      for (int i = threadIdx.x; i < 94 * 94; i += blockDim.x) {
        const int yy = i / 94 - 3, xx = i - (yy + 3) * 94 - 3;
        uint16_t v = 0;
        if (yy >= 0 && yy < 88 && xx >= 0 && xx < 88) v = lut[__ldg(src + yy * s.W0 + (mirror ? 87 - xx : xx))];
        tile[(yy + 3) * 96 + xx + 3] = v;
      }
      __syncthreads();
    }
    const int k0 = dt * 49;
    const int rows = dt < 5 ? 49 : 256 - 245;
    for (int rr = 0; rr < rows; ++rr) {
      const int r = rr / 7, sx = rr - r * 7;
      uint32_t* dst = reinterpret_cast<uint32_t*>(out + static_cast<long long>(k0 + rr) * ld_out + m0);
      for (int i = threadIdx.x; i < 968; i += blockDim.x) {      // 968 pixel pairs of one frame
        const long long m = m0 + 2 * i;
        if (m >= ld_out) break;
        uint32_t a = 0u, b = 0u;
        if (real) {
          const int px = 2 * i;
          const int y = px / 44, xo = px - y * 44;              // 44 is even: both pixels in the same row
          const uint16_t* p = tile + (2 * y + r) * 96 + 2 * xo + sx;
          a = p[0];
          b = p[2];
        }
        if (m + 1 < ld_out) dst[i] = a | (b << 16);
        else *reinterpret_cast<uint16_t*>(dst + i) = static_cast<uint16_t>(a);
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Per-channel (column) reductions over the rows of a [M, C] matrix, deterministic two-stage: every block writes its
// partial sums to part[block][2][C], colreduce_finish_kernel adds the blocks in order.  Modes:
//   0  x 16-bit                    -> (sum x, sum x^2)                          BatchNorm batch statistics
//   1  dy 16-bit, out 16-bit, x 16-bit, mean/rstd -> (sum dz, sum dz * xhat), dz = dy * (out > 0 or no mask)   BN backward
//   2  x fp32                      -> (sum x, -)                                bias gradients of fp32 rows
//   4  x 16-bit                    -> (sum x, -)                                bias gradients of 16-bit rows
// ----------------------------------------------------------------------------------------------------------------
struct ColReduceParams {
  const void* a;        // x / dy
  const void* b;        // mode 1: BN output (ReLU mask) or nullptr ; mode 3: z
  const void* c;        // mode 1: raw conv output x
  const float* mean;    // mode 1: [C]
  const float* rstd;    // mode 1: [C]
  const int* lengths;   // mode 3: pad mask (rows with t >= lengths[m / T] contribute nothing), or nullptr
  float* part;          // [gridDim.x][2][C]
  long long M;
  int C;
  int mode;
  int fp16;             // 16-bit inputs are IEEE fp16 (else bf16)
  int T;                // mode 3
  float eps;            // mode 3
};

// A thread owns 8 adjacent channels (one 16-byte load per operand and row); blockDim = (C/8 capped at 64) x rows in
// flight.  C % 8 == 0 and (C/8 <= 64 with 256 % (C/8) == 0, or C/8 % 64 == 0).
__global__ void __launch_bounds__(256)
colreduce_kernel(const ColReduceParams p) {
  extern __shared__ float red[];   // [256 threads][16]
  const int cols8 = p.C / 8;
  const int cpb = cols8 < 64 ? cols8 : 64;          // 8-channel chunks per block pass
  const int rif = blockDim.x / cpb;                 // rows in flight
  const int cx = threadIdx.x % cpb, ry = threadIdx.x / cpb;
  for (int cbase = 0; cbase < cols8; cbase += cpb) {
    const int c8 = cbase + cx;
    float s0[8], s1[8], mean[8], rstd[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { s0[e] = 0.0f; s1[e] = 0.0f; mean[e] = 0.0f; rstd[e] = 0.0f; }
    if (p.mode == 1) {
#pragma unroll
      for (int e = 0; e < 8; ++e) { mean[e] = __ldg(p.mean + 8 * c8 + e); rstd[e] = __ldg(p.rstd + 8 * c8 + e); }
    }
    for (long long m = static_cast<long long>(blockIdx.x) * rif + ry; m < p.M; m += static_cast<long long>(gridDim.x) * rif) {
      const long long idx = m * cols8 + c8;
      if (p.mode == 2) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(p.a) + 2 * idx);
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.a) + 2 * idx + 1);
        s0[0] += a.x; s0[1] += a.y; s0[2] += a.z; s0[3] += a.w; s0[4] += b.x; s0[5] += b.y; s0[6] += b.z; s0[7] += b.w;
      } else {
        const uint4 ua = __ldg(reinterpret_cast<const uint4*>(p.a) + idx);
        const uint32_t wa[4] = {ua.x, ua.y, ua.z, ua.w};
        if (p.mode == 0 || p.mode == 4) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float a0 = lo16(wa[j], p.fp16), a1 = hi16(wa[j], p.fp16);
            s0[2 * j] += a0; s0[2 * j + 1] += a1;
            if (p.mode == 0) { s1[2 * j] += a0 * a0; s1[2 * j + 1] += a1 * a1; }
          }
        } else {   // mode 1
          uint4 uo = make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);   // "positive": no mask
          if (p.b != nullptr) uo = __ldg(reinterpret_cast<const uint4*>(p.b) + idx);
          const uint4 ux = __ldg(reinterpret_cast<const uint4*>(p.c) + idx);
          const uint32_t wo[4] = {uo.x, uo.y, uo.z, uo.w}, wx[4] = {ux.x, ux.y, ux.z, ux.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float d0 = bf16_lo(wo[j]) > 0.0f ? bf16_lo(wa[j]) : 0.0f;
            const float d1 = bf16_hi(wo[j]) > 0.0f ? bf16_hi(wa[j]) : 0.0f;
            s0[2 * j] += d0; s0[2 * j + 1] += d1;
            s1[2 * j] += d0 * ((bf16_lo(wx[j]) - mean[2 * j]) * rstd[2 * j]);
            s1[2 * j + 1] += d1 * ((bf16_hi(wx[j]) - mean[2 * j + 1]) * rstd[2 * j + 1]);
          }
        }
      }
    }
    float* my = red + threadIdx.x * 16;
#pragma unroll
    for (int e = 0; e < 8; ++e) { my[e] = s0[e]; my[8 + e] = s1[e]; }
    __syncthreads();
    if (ry == 0) {
      for (int r = 1; r < rif; ++r) {
        const float* o = red + (r * cpb + cx) * 16;
#pragma unroll
        for (int e = 0; e < 8; ++e) { s0[e] += o[e]; s1[e] += o[8 + e]; }
      }
      float* dst = p.part + static_cast<long long>(blockIdx.x) * 2 * p.C;
#pragma unroll
      for (int e = 0; e < 8; ++e) { dst[8 * c8 + e] = s0[e]; dst[p.C + 8 * c8 + e] = s1[e]; }
    }
    __syncthreads();
  }
}

// out[j] = sum over blocks of part[block][j], j < 2*C, in a fixed order (deterministic): a CTA owns 32 columns, thread
// (cx, sy) adds the blocks sy, sy + 8, ... of column cx in order, the eight slice sums are then added in slice order.
// (One thread per column walking all ~600 partial blocks was a chain of dependent L2 round trips: ~40 us per call, the
// fixed cost of every BatchNorm statistic / bias-gradient reduction of the training step.)  Launch: ceil(n / 32) CTAs.
__global__ void __launch_bounds__(256)
colreduce_finish_kernel(const float* __restrict__ part, float* __restrict__ out, int nblocks, int n) {
  __shared__ float red[8][32];
  const int cx = threadIdx.x & 31, sy = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + cx;
  float s = 0.0f;
  if (j < n)
    for (int b = sy; b < nblocks; b += 8) s += part[static_cast<long long>(b) * n + j];
  red[sy][cx] = s;
  __syncthreads();
  if (sy == 0 && j < n) {
    float t = red[0][cx];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += red[k][cx];
    out[j] = t;
  }
}

// BatchNorm training statistics from (sum, sumsq): mean, rstd = 1/sqrt(biased var + eps), and the running-stat update
// running = (1 - momentum) * running + momentum * (mean | unbiased var)   (torch.nn.BatchNorm semantics)
__global__ void bn_finalize_kernel(const float* __restrict__ sums, float* __restrict__ mean, float* __restrict__ rstd,
                                   float* __restrict__ running_mean, float* __restrict__ running_var, int C,
                                   float count, float eps, float momentum) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float m = sums[c] / count;
  float var = sums[C + c] / count - m * m;
  var = fmaxf(var, 0.0f);
  mean[c] = m;
  rstd[c] = rsqrtf(var + eps);
  if (running_mean != nullptr) {
    running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * m;
    const float unbiased = count > 1.0f ? var * (count / (count - 1.0f)) : var;
    running_var[c] = (1.0f - momentum) * running_var[c] + momentum * unbiased;
  }
}

// ----------------------------------------------------------------------------------------------------------------
// BatchNorm apply (training forward): out = act((x - mean) * rstd * gamma + beta (+ residual)), bf16 in / out, 8 channels
// per thread.  C % 8 == 0.
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
bn_apply_kernel(const uint4* __restrict__ x, const uint4* __restrict__ residual, const float* __restrict__ mean,
                const float* __restrict__ rstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                uint4* __restrict__ out, long long total8, int C, int relu) {
  const int c8n = C / 8;
  // the grid stride (gridDim.x * 256) is a multiple of C/8 (a power of two <= 64: checked by the launcher), so a thread
  // sees the same 8 channels in every trip: their statistics / affine parameters are loaded once (they were 32 scalar
  // loads per 16-byte vector)
  const long long i0 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const int c0 = static_cast<int>(i0 % c8n) * 8;
  float mn[8], rs[8], gm[8], bt[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    mn[e] = __ldg(mean + c0 + e); rs[e] = __ldg(rstd + c0 + e); gm[e] = __ldg(gamma + c0 + e); bt[e] = __ldg(beta + c0 + e);
  }
  for (long long i = i0; i < total8; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 u = __ldg(x + i);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    uint4 r4 = make_uint4(0u, 0u, 0u, 0u);
    if (residual != nullptr) r4 = __ldg(residual + i);
    const uint32_t rw[4] = {r4.x, r4.y, r4.z, r4.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a = (bf16_lo(w[j]) - mn[2 * j]) * rs[2 * j] * gm[2 * j] + bt[2 * j];
      float b = (bf16_hi(w[j]) - mn[2 * j + 1]) * rs[2 * j + 1] * gm[2 * j + 1] + bt[2 * j + 1];
      if (residual != nullptr) { a += bf16_lo(rw[j]); b += bf16_hi(rw[j]); }
      if (relu) { a = fmaxf(a, 0.0f); b = fmaxf(b, 0.0f); }
      o[j] = pack_bf16x2(a, b);
    }
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// BatchNorm backward (training): dz = dy * (out > 0 if masked);  dx = gamma * rstd * (dz - sum_dz / M - xhat * sum_dzx / M)
// Optionally also writes dz itself (the gradient of the residual branch of `relu(bn2(conv2) + residual)`).
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ out_act, const uint4* __restrict__ x,
                    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ gamma,
                    const float* __restrict__ sums, uint4* __restrict__ dx, uint4* __restrict__ dres, long long total8,
                    int C, float inv_count) {
  const int c8n = C / 8;
  // per-thread constant channels (see bn_apply_kernel): statistics, scale and the two reduction sums loaded once
  const long long i0 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const int c0 = static_cast<int>(i0 % c8n) * 8;
  float mn[8], rsv[8], gm[8], sm0[8], sm1[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    mn[e] = __ldg(mean + c0 + e); rsv[e] = __ldg(rstd + c0 + e); gm[e] = __ldg(gamma + c0 + e);
    sm0[e] = __ldg(sums + c0 + e); sm1[e] = __ldg(sums + C + c0 + e);
  }
  for (long long i = i0; i < total8; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 ud = __ldg(dy + i), ux = __ldg(x + i);
    uint4 uo = make_uint4(0u, 0u, 0u, 0u);
    if (out_act != nullptr) uo = __ldg(out_act + i);
    const uint32_t wd[4] = {ud.x, ud.y, ud.z, ud.w}, wx[4] = {ux.x, ux.y, ux.z, ux.w}, wo[4] = {uo.x, uo.y, uo.z, uo.w};
    uint32_t o[4], oz[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float d[2] = {bf16_lo(wd[j]), bf16_hi(wd[j])};
      const float xv[2] = {bf16_lo(wx[j]), bf16_hi(wx[j])};
      if (out_act != nullptr) {
        if (!(bf16_lo(wo[j]) > 0.0f)) d[0] = 0.0f;
        if (!(bf16_hi(wo[j]) > 0.0f)) d[1] = 0.0f;
      }
      float g[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = 2 * j + e;
        const float rs = rsv[c];
        const float xh = (xv[e] - mn[c]) * rs;
        g[e] = gm[c] * rs * (d[e] - sm0[c] * inv_count - xh * sm1[c] * inv_count);
      }
      o[j] = pack_bf16x2(g[0], g[1]);
      oz[j] = pack_bf16x2(d[0], d[1]);
    }
    dx[i] = make_uint4(o[0], o[1], o[2], o[3]);
    if (dres != nullptr) dres[i] = make_uint4(oz[0], oz[1], oz[2], oz[3]);
  }
}

// ----------------------------------------------------------------------------------------------------------------
// MaxPool 3x3 / stride 2 / pad 1 over NHWC bf16 [F, H, W, C] -> [F, P, Q, C] (P = (H-1)/2 + 1), forward and backward.
// Backward: every INPUT pixel looks at the <= 4 windows covering it and takes the window's gradient iff it is that
// window's FIRST maximum in row-major scan order (PyTorch's tie rule) — no atomics, one write per element.
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
maxpool3x3s2_fwd_kernel(const uint32_t* __restrict__ x, uint32_t* __restrict__ out, int F, int H, int W, int C2, int P,
                        int Q) {
  const long long total = static_cast<long long>(F) * P * Q * C2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C2);
    long long t = i / C2;
    const int q = static_cast<int>(t % Q); t /= Q;
    const int pp = static_cast<int>(t % P);
    const long long f = t / P;
    float a = -INFINITY, b = -INFINITY;
    for (int r = 0; r < 3; ++r) {
      const int y = 2 * pp + r - 1;
      if (y < 0 || y >= H) continue;
      for (int s = 0; s < 3; ++s) {
        const int xx = 2 * q + s - 1;
        if (xx < 0 || xx >= W) continue;
        const uint32_t u = __ldg(x + ((f * H + y) * W + xx) * C2 + c);
        a = fmaxf(a, bf16_lo(u));
        b = fmaxf(b, bf16_hi(u));
      }
    }
    out[i] = pack_bf16x2(a, b);
  }
}

// `pooled` is the forward output.  A pixel receives a window's gradient iff it equals the window maximum and no EARLIER
// pixel of the window (row-major scan order, PyTorch's tie rule) does; only candidates (x == max) scan their window.
// Non-positive pixels take no gradient: the pooled tensor is a ReLU output, so its gradient is masked there anyway.
__global__ void __launch_bounds__(256)
maxpool3x3s2_bwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ pooled, const uint4* __restrict__ dy,
                        uint4* __restrict__ dx, int F, int H, int W, int C8, int P, int Q) {
  const long long total = static_cast<long long>(F) * H * W * C8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C8);
    long long t = i / C8;
    const int xx = static_cast<int>(t % W); t /= W;
    const int y = static_cast<int>(t % H);
    const long long f = t / H;
    const uint4 self = __ldg(x + i);
    const uint32_t sw[4] = {self.x, self.y, self.z, self.w};
    float v[8], g[8];
    bool any_pos = false;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] = bf16_lo(sw[j]); v[2 * j + 1] = bf16_hi(sw[j]);
      g[2 * j] = 0.0f; g[2 * j + 1] = 0.0f;
      any_pos = any_pos || v[2 * j] > 0.0f || v[2 * j + 1] > 0.0f;
    }
    if (any_pos) {
      for (int pp = (y >> 1); pp <= ((y + 1) >> 1); ++pp) {
        if (pp >= P) continue;
        for (int q = (xx >> 1); q <= ((xx + 1) >> 1); ++q) {
          if (q >= Q) continue;
          const long long widx = ((f * P + pp) * Q + q) * C8 + c;
          const uint4 mx = __ldg(pooled + widx);
          const uint32_t mw[4] = {mx.x, mx.y, mx.z, mx.w};
          bool cand[8];
          bool any = false;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            cand[2 * j] = v[2 * j] > 0.0f && v[2 * j] == bf16_lo(mw[j]);
            cand[2 * j + 1] = v[2 * j + 1] > 0.0f && v[2 * j + 1] == bf16_hi(mw[j]);
            any = any || cand[2 * j] || cand[2 * j + 1];
          }
          if (!any) continue;
          // tie check: an equal value EARLIER in the window's row-major scan order wins
          for (int r = 0; r < 3; ++r) {
            const int y2 = 2 * pp + r - 1;
            if (y2 < 0 || y2 > y) continue;
            for (int s2 = 0; s2 < 3; ++s2) {
              const int x2 = 2 * q + s2 - 1;
              if (x2 < 0 || x2 >= W) continue;
              if (!(y2 < y || x2 < xx)) continue;
              const uint4 u = __ldg(x + ((f * H + y2) * W + x2) * C8 + c);
              const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (bf16_lo(uw[j]) == v[2 * j]) cand[2 * j] = false;
                if (bf16_hi(uw[j]) == v[2 * j + 1]) cand[2 * j + 1] = false;
              }
            }
          }
          const uint4 gy = __ldg(dy + widx);
          const uint32_t gw[4] = {gy.x, gy.y, gy.z, gy.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (cand[2 * j]) g[2 * j] += bf16_lo(gw[j]);
            if (cand[2 * j + 1]) g[2 * j + 1] += bf16_hi(gw[j]);
          }
        }
      }
    }
    dx[i] = make_uint4(pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]), pack_bf16x2(g[6], g[7]));
  }
}

// AdaptiveAvgPool2d(1) backward: dx[f, hw, c] = dfeat[f, c] / HW  (fp32 in, bf16 out)
__global__ void __launch_bounds__(256)
avgpool_bwd_kernel(const float2* __restrict__ dfeat, uint32_t* __restrict__ dx, long long F, int HW, int C2) {
  const long long total = F * HW * C2;
  const float inv = 1.0f / static_cast<float>(HW);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C2);
    const long long f = i / (static_cast<long long>(HW) * C2);
    const float2 g = __ldg(dfeat + f * C2 + c);
    dx[i] = pack_bf16x2(g.x * inv, g.y * inv);
  }
}

// Zero-stuffing for the dgrad of a stride-2 conv: out [F, H, W, C] = 0 except out[f, 2p, 2q, :] = dy[f, p, q, :]
__global__ void __launch_bounds__(256)
zero_stuff2_kernel(const uint4* __restrict__ dy, uint4* __restrict__ out, int F, int H, int W, int C8, int P, int Q) {
  const long long total = static_cast<long long>(F) * H * W * C8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C8);
    long long t = i / C8;
    const int xx = static_cast<int>(t % W); t /= W;
    const int y = static_cast<int>(t % H);
    const long long f = t / H;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (!(y & 1) && !(xx & 1) && (y >> 1) < P && (xx >> 1) < Q)
      v = __ldg(dy + ((f * P + (y >> 1)) * Q + (xx >> 1)) * C8 + c);
    out[i] = v;
  }
}

// dh *= (h > 0)   (ReLU backward of the FFN hidden layer; dh bf16 in place, h enc16)
__global__ void __launch_bounds__(256)
relu_bwd_kernel(uint32_t* __restrict__ dh, const uint32_t* __restrict__ h, long long total2, int h_fp16) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total2;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t u = dh[i], v = __ldg(h + i);
    const float a = lo16(v, h_fp16) > 0.0f ? bf16_lo(u) : 0.0f;
    const float b = hi16(v, h_fp16) > 0.0f ? bf16_hi(u) : 0.0f;
    dh[i] = pack_bf16x2(a, b);
  }
}

// ----------------------------------------------------------------------------------------------------------------
// LayerNorm(512) backward, one warp per row.  z fp32 [M, 512] is the pre-normalisation sum the forward saved; mean / rstd
// are recomputed.  y = xhat * gamma + beta (* keep):  dxhat = dy * keep * gamma ;
//   dz = rstd * (dxhat - mean(dxhat) - xhat * mean(dxhat * xhat)).   dz fp32 (residual stream gradient) and / or bf16.
// dgamma / dbeta partials: part[block][2][512] = (sum dy*keep*xhat, sum dy*keep) over the block's rows (finished by
// colreduce_finish_kernel).
// ----------------------------------------------------------------------------------------------------------------
struct LnBwdParams {
  const float* dy;       // [M, 512]
  const float* z;        // [M, 512]
  const float* gamma;    // [512]
  const int* lengths;    // or nullptr
  float* dz_f32;         // [M, 512] or nullptr
  uint16_t* dz_bf16;     // [M, 512] or nullptr
  float* part;           // [gridDim.x][2][512]
  int M, T;
  float eps;
};

__global__ void __launch_bounds__(256)
ln_bwd_kernel(const LnBwdParams p) {
  __shared__ float acc[8][2][512];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  float dg[16], db[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) { dg[j] = 0.0f; db[j] = 0.0f; }
  for (int m = blockIdx.x * warps_per_block + warp; m < p.M; m += gridDim.x * warps_per_block) {
    float keep = 1.0f;
    if (p.lengths != nullptr && (m % p.T) >= __ldg(p.lengths + m / p.T)) keep = 0.0f;
    const float4* zr = reinterpret_cast<const float4*>(p.z + static_cast<size_t>(m) * 512);
    const float4* dr = reinterpret_cast<const float4*>(p.dy + static_cast<size_t>(m) * 512);
    float v[16], d[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 a = __ldg(zr + j * 32 + lane);
      v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
      const float4 b = __ldg(dr + j * 32 + lane);
      d[4 * j] = b.x * keep; d[4 * j + 1] = b.y * keep; d[4 * j + 2] = b.z * keep; d[4 * j + 3] = b.w * keep;
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += v[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.0f / 512.0f);
    float q = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) { const float e = v[j] - mean; q += e * e; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q * (1.0f / 512.0f) + p.eps);
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(p.gamma) + j * 32 + lane);
      const float gg[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float xh = (v[4 * j + e] - mean) * rstd;
        dg[4 * j + e] += d[4 * j + e] * xh;
        db[4 * j + e] += d[4 * j + e];
        v[4 * j + e] = xh;
        d[4 * j + e] *= gg[e];           // dxhat
        s1 += d[4 * j + e];
        s2 += d[4 * j + e] * xh;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    s1 *= (1.0f / 512.0f); s2 *= (1.0f / 512.0f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float4 o;
      o.x = rstd * (d[4 * j] - s1 - v[4 * j] * s2);
      o.y = rstd * (d[4 * j + 1] - s1 - v[4 * j + 1] * s2);
      o.z = rstd * (d[4 * j + 2] - s1 - v[4 * j + 2] * s2);
      o.w = rstd * (d[4 * j + 3] - s1 - v[4 * j + 3] * s2);
      if (p.dz_f32 != nullptr) reinterpret_cast<float4*>(p.dz_f32 + static_cast<size_t>(m) * 512)[j * 32 + lane] = o;
      if (p.dz_bf16 != nullptr) {
        uint2 w;
        w.x = pack_bf16x2(o.x, o.y);
        w.y = pack_bf16x2(o.z, o.w);
        reinterpret_cast<uint2*>(p.dz_bf16 + static_cast<size_t>(m) * 512)[j * 32 + lane] = w;
      }
    }
  }
  // block-level sum of the per-warp dgamma / dbeta accumulators (fixed order: deterministic)
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      acc[warp][0][(j * 32 + lane) * 4 + e] = dg[4 * j + e];
      acc[warp][1][(j * 32 + lane) * 4 + e] = db[4 * j + e];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 1024; i += blockDim.x) {
    const int which = i >> 9, col = i & 511;
    float s = 0.0f;
    for (int w = 0; w < warps_per_block; ++w) s += acc[w][which][col];
    p.part[static_cast<long long>(blockIdx.x) * 1024 + i] = s;
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Scaled-dot-product self-attention, TRAINING forward + backward for short clips (T <= 64, d_k = 64), one CTA per
// (clip, head), fp32 math in shared memory (0.05 % of the encoder's FLOPs).  attention.py:72-83 with the dropout on the
// probabilities made explicit: `drop` = mask / (1 - p) drawn by the caller ([H*N, T, T] fp32, or nullptr).
//   forward : P = softmax(Q K^T * scale, keys >= len masked) ; O = (P * drop) V       -> O enc16, P fp32 (saved)
//   backward: dV = (P*drop)^T dO ; dPd = dO V^T ; dP = dPd * drop ; dS = P * (dP - rowsum(dP * P)) * scale ;
//             dQ = dS K ; dK = dS^T Q                                                  -> dqkv bf16 [M, 3*H*64]
// qkv enc16 [N*T, 3*H*64] (q | k | v thirds, head h at columns h*64), probs index (h*N + b) like the reference.
// ----------------------------------------------------------------------------------------------------------------
struct AttnTrainParams {
  const uint16_t* qkv;   // enc16
  const float* drop;     // or nullptr
  float* probs;          // forward: written; backward: read
  uint16_t* out;         // forward: O enc16 [N*T, H*64]
  const uint16_t* dout;  // backward: dO bf16 [N*T, H*64]
  uint16_t* dqkv;        // backward: bf16 [N*T, 3*H*64]
  const int* lengths;
  int N, T, H;
  float scale;
  int fp16;              // qkv / out storage is IEEE fp16 (else bf16)
};

template <bool BWD>
__global__ void __launch_bounds__(256)
attn_train_kernel(const AttnTrainParams p) {
  extern __shared__ float sm[];
  const int T = p.T, D = 64;
  const int b = blockIdx.x / p.H, h = blockIdx.x - b * p.H;
  const int ld = 3 * p.H * D;
  float* sQ = sm;                 // [T][65]
  float* sK = sQ + T * 65;
  float* sV = sK + T * 65;
  float* sP = sV + T * 65;        // [T][T+1]
  float* sG = sP + T * (T + 1);   // BWD: dO [T][65]
  float* sS = sG + (BWD ? T * 65 : 0);   // BWD: dS [T][T+1]
  const int len = (p.lengths != nullptr) ? min(max(__ldg(p.lengths + b), 0), T) : T;
  const uint16_t* base = p.qkv + static_cast<size_t>(b) * T * ld + h * D;
  for (int i = threadIdx.x; i < T * D; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    sQ[t * 65 + d] = ld16(base + static_cast<size_t>(t) * ld + d, p.fp16);
    sK[t * 65 + d] = ld16(base + static_cast<size_t>(t) * ld + p.H * D + d, p.fp16);
    sV[t * 65 + d] = ld16(base + static_cast<size_t>(t) * ld + 2 * p.H * D + d, p.fp16);
    if (BWD) sG[t * 65 + d] = ld16(p.dout + (static_cast<size_t>(b) * T + t) * (p.H * D) + h * D + d, 0);
  }
  float* probs = p.probs + (static_cast<size_t>(h) * p.N + b) * T * T;
  const float* drop = p.drop != nullptr ? p.drop + (static_cast<size_t>(h) * p.N + b) * T * T : nullptr;
  __syncthreads();
  if (!BWD) {
    // S = Q K^T * scale, masked; one warp per query row: softmax with shuffles
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int qi = warp; qi < T; qi += nw) {
      float sc[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int kj = lane + 32 * e;
        if (kj < T && kj < len) {
          float a = 0.0f;
          for (int d = 0; d < D; ++d) a += sQ[qi * 65 + d] * sK[kj * 65 + d];
          sc[e] = a * p.scale;
        }
      }
      float mx = fmaxf(sc[0], sc[1]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float e0 = __expf(sc[0] - mx), e1 = __expf(sc[1] - mx);   // all-masked row: NaN like the reference softmax
      float sum = e0 + e1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float inv = 1.0f / sum;
      if (lane < T) { sP[qi * (T + 1) + lane] = e0 * inv; probs[qi * T + lane] = e0 * inv; }
      if (lane + 32 < T) { sP[qi * (T + 1) + lane + 32] = e1 * inv; probs[qi * T + lane + 32] = e1 * inv; }
    }
    __syncthreads();
    uint16_t* out = p.out + static_cast<size_t>(b) * T * (p.H * D) + h * D;
    for (int i = threadIdx.x; i < T * D; i += blockDim.x) {
      const int t = i >> 6, d = i & 63;
      float a = 0.0f;
      for (int j = 0; j < T; ++j) {
        float pj = sP[t * (T + 1) + j];
        if (drop != nullptr) pj *= __ldg(drop + t * T + j);
        a += pj * sV[j * 65 + d];
      }
      const uint32_t w = p.fp16 ? pack_f16x2(a, 0.0f) : pack_bf16x2(a, 0.0f);
      out[static_cast<size_t>(t) * (p.H * D) + d] = static_cast<uint16_t>(w & 0xFFFFu);
    }
  } else {
    for (int i = threadIdx.x; i < T * T; i += blockDim.x) sP[(i / T) * (T + 1) + (i % T)] = __ldg(probs + i);
    __syncthreads();
    // dP = (dO V^T) * drop ; row statistics ; dS
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int qi = warp; qi < T; qi += nw) {
      float dp[2] = {0.0f, 0.0f}, pv[2] = {0.0f, 0.0f};
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int kj = lane + 32 * e;
        if (kj < T) {
          float a = 0.0f;
          for (int d = 0; d < D; ++d) a += sG[qi * 65 + d] * sV[kj * 65 + d];
          if (drop != nullptr) a *= __ldg(drop + qi * T + kj);
          dp[e] = a;
          pv[e] = sP[qi * (T + 1) + kj];
        }
      }
      float dot = dp[0] * pv[0] + dp[1] * pv[1];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      if (lane < T) sS[qi * (T + 1) + lane] = pv[0] * (dp[0] - dot) * p.scale;
      if (lane + 32 < T) sS[qi * (T + 1) + lane + 32] = pv[1] * (dp[1] - dot) * p.scale;
    }
    __syncthreads();
    uint16_t* dq = p.dqkv + static_cast<size_t>(b) * T * ld + h * D;
    for (int i = threadIdx.x; i < T * D; i += blockDim.x) {
      const int t = i >> 6, d = i & 63;
      float aq = 0.0f, ak = 0.0f, av = 0.0f;
      for (int j = 0; j < T; ++j) {
        aq += sS[t * (T + 1) + j] * sK[j * 65 + d];          // dQ[t] = sum_j dS[t][j] K[j]
        ak += sS[j * (T + 1) + t] * sQ[j * 65 + d];          // dK[t] = sum_j dS[j][t] Q[j]
        float pj = sP[j * (T + 1) + t];
        if (drop != nullptr) pj *= __ldg(drop + j * T + t);
        av += pj * sG[j * 65 + d];                           // dV[t] = sum_j (P*drop)[j][t] dO[j]
      }
      dq[static_cast<size_t>(t) * ld + d] = static_cast<uint16_t>(pack_bf16x2(aq, 0.0f) & 0xFFFFu);
      dq[static_cast<size_t>(t) * ld + p.H * D + d] = static_cast<uint16_t>(pack_bf16x2(ak, 0.0f) & 0xFFFFu);
      dq[static_cast<size_t>(t) * ld + 2 * p.H * D + d] = static_cast<uint16_t>(pack_bf16x2(av, 0.0f) & 0xFFFFu);
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Scaled-dot-product attention, TRAINING forward + backward for short sequences (Lq, Lk <= 64, d_k = 64), with separate
// query and key / value sources and an optional causal mask: the decoder's self-attention over the prefix (Lq = Lk = L,
// causal in its first layer) and its decoder-encoder attention (Lq = L, Lk = t_enc).  One CTA per (clip, head), fp32 math in shared memory.  The encoder
// keeps attn_train_kernel above: this kernel computes the same values on its shape (bit for bit) but measured 0.8 %
// slower there (DESIGN.md §9).
// attention.py:72-83 with the dropout on the probabilities made explicit: `drop` = mask / (1 - p) drawn by the caller
// ([H*N, Lq, Lk] fp32, or nullptr).
//   forward : P = softmax(Q K^T * scale, keys j >= klens[b] and (causal) j > i masked) ; O = (P * drop) V
//             -> O enc16, P fp32 (saved)
//   backward: dV = (P*drop)^T dO ; dPd = dO V^T ; dP = dPd * drop ; dS = P * (dP - rowsum(dP * P)) * scale ;
//             dQ = dS K ; dK = dS^T Q                                                  -> dQ, dK, dV bf16
// Q rows at q + (b*Lq + i)*ldq + h*64, K / V rows at k|v + (b*Lk + j)*ldk|ldv + h*64 (enc16); O / dO / dQ rows with the
// query pitches ldo / lddo / lddq, dK / dV rows with lddk / lddv.  probs / drop index (h*N + b) like the reference.
// ----------------------------------------------------------------------------------------------------------------
struct XAttnTrainParams {
  const uint16_t* q;     // enc16
  const uint16_t* k;
  const uint16_t* v;
  const float* drop;     // or nullptr
  float* probs;          // forward: written; backward: read
  uint16_t* out;         // forward: O enc16
  const uint16_t* dout;  // backward: dO bf16
  uint16_t* dq;          // backward: bf16
  uint16_t* dk;
  uint16_t* dv;
  const int* klens;      // [N] valid keys or nullptr
  int ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv;
  int N, Lq, Lk, H, causal;
  float scale;
  int fp16;              // q / k / v / out storage is IEEE fp16 (else bf16)
};

template <bool BWD>
__global__ void __launch_bounds__(256)
xattn_train_kernel(const XAttnTrainParams p) {
  extern __shared__ float sm[];
  const int Lq = p.Lq, Lk = p.Lk, D = 64;
  const int b = blockIdx.x / p.H, h = blockIdx.x - b * p.H;
  float* sQ = sm;                        // [Lq][65]
  float* sK = sQ + Lq * 65;              // [Lk][65]
  float* sV = sK + Lk * 65;              // [Lk][65]
  float* sP = sV + Lk * 65;              // [Lq][Lk+1]
  float* sG = sP + Lq * (Lk + 1);        // BWD: dO [Lq][65]
  float* sS = sG + (BWD ? Lq * 65 : 0);  // BWD: dS [Lq][Lk+1]
  const int klen = (p.klens != nullptr) ? min(max(__ldg(p.klens + b), 0), Lk) : Lk;
  for (int i = threadIdx.x; i < Lq * D; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    const size_t row = static_cast<size_t>(b) * Lq + t;
    sQ[t * 65 + d] = ld16(p.q + row * p.ldq + h * D + d, p.fp16);
    if (BWD) sG[t * 65 + d] = ld16(p.dout + row * p.lddo + h * D + d, 0);
  }
  for (int i = threadIdx.x; i < Lk * D; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    const size_t row = static_cast<size_t>(b) * Lk + t;
    sK[t * 65 + d] = ld16(p.k + row * p.ldk + h * D + d, p.fp16);
    sV[t * 65 + d] = ld16(p.v + row * p.ldv + h * D + d, p.fp16);
  }
  float* probs = p.probs + (static_cast<size_t>(h) * p.N + b) * Lq * Lk;
  const float* drop = p.drop != nullptr ? p.drop + (static_cast<size_t>(h) * p.N + b) * Lq * Lk : nullptr;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (!BWD) {
    // S = Q K^T * scale, masked; one warp per query row: softmax with shuffles
    for (int qi = warp; qi < Lq; qi += nw) {
      float sc[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int kj = lane + 32 * e;
        if (kj < klen && !(p.causal && kj > qi)) {
          float a = 0.0f;
          for (int d = 0; d < D; ++d) a += sQ[qi * 65 + d] * sK[kj * 65 + d];
          sc[e] = a * p.scale;
        }
      }
      float mx = fmaxf(sc[0], sc[1]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float e0 = __expf(sc[0] - mx), e1 = __expf(sc[1] - mx);   // all-masked row: NaN like the reference softmax
      float sum = e0 + e1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float inv = 1.0f / sum;
      if (lane < Lk) { sP[qi * (Lk + 1) + lane] = e0 * inv; probs[qi * Lk + lane] = e0 * inv; }
      if (lane + 32 < Lk) { sP[qi * (Lk + 1) + lane + 32] = e1 * inv; probs[qi * Lk + lane + 32] = e1 * inv; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < Lq * D; i += blockDim.x) {
      const int t = i >> 6, d = i & 63;
      float a = 0.0f;
      for (int j = 0; j < Lk; ++j) {
        float pj = sP[t * (Lk + 1) + j];
        if (drop != nullptr) pj *= __ldg(drop + t * Lk + j);
        a += pj * sV[j * 65 + d];
      }
      const uint32_t w = p.fp16 ? pack_f16x2(a, 0.0f) : pack_bf16x2(a, 0.0f);
      p.out[(static_cast<size_t>(b) * Lq + t) * p.ldo + h * D + d] = static_cast<uint16_t>(w & 0xFFFFu);
    }
  } else {
    for (int i = threadIdx.x; i < Lq * Lk; i += blockDim.x) sP[(i / Lk) * (Lk + 1) + (i % Lk)] = __ldg(probs + i);
    __syncthreads();
    // dP = (dO V^T) * drop ; row statistics ; dS
    for (int qi = warp; qi < Lq; qi += nw) {
      float dp[2] = {0.0f, 0.0f}, pv[2] = {0.0f, 0.0f};
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int kj = lane + 32 * e;
        if (kj < Lk) {
          float a = 0.0f;
          for (int d = 0; d < D; ++d) a += sG[qi * 65 + d] * sV[kj * 65 + d];
          if (drop != nullptr) a *= __ldg(drop + qi * Lk + kj);
          dp[e] = a;
          pv[e] = sP[qi * (Lk + 1) + kj];
        }
      }
      float dot = dp[0] * pv[0] + dp[1] * pv[1];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      if (lane < Lk) sS[qi * (Lk + 1) + lane] = pv[0] * (dp[0] - dot) * p.scale;
      if (lane + 32 < Lk) sS[qi * (Lk + 1) + lane + 32] = pv[1] * (dp[1] - dot) * p.scale;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < Lq * D; i += blockDim.x) {   // dQ[t] = sum_j dS[t][j] K[j]
      const int t = i >> 6, d = i & 63;
      float aq = 0.0f;
      for (int j = 0; j < Lk; ++j) aq += sS[t * (Lk + 1) + j] * sK[j * 65 + d];
      p.dq[(static_cast<size_t>(b) * Lq + t) * p.lddq + h * D + d] = static_cast<uint16_t>(pack_bf16x2(aq, 0.0f) & 0xFFFFu);
    }
    for (int i = threadIdx.x; i < Lk * D; i += blockDim.x) {   // dK[t] = sum_j dS[j][t] Q[j], dV[t] = sum_j (P*drop)[j][t] dO[j]
      const int t = i >> 6, d = i & 63;
      float ak = 0.0f, av = 0.0f;
      for (int j = 0; j < Lq; ++j) {
        ak += sS[j * (Lk + 1) + t] * sQ[j * 65 + d];
        float pj = sP[j * (Lk + 1) + t];
        if (drop != nullptr) pj *= __ldg(drop + j * Lk + t);
        av += pj * sG[j * 65 + d];
      }
      const size_t row = static_cast<size_t>(b) * Lk + t;
      p.dk[row * p.lddk + h * D + d] = static_cast<uint16_t>(pack_bf16x2(ak, 0.0f) & 0xFFFFu);
      p.dv[row * p.lddv + h * D + d] = static_cast<uint16_t>(pack_bf16x2(av, 0.0f) & 0xFFFFu);
    }
  }
}

}  // namespace sblk

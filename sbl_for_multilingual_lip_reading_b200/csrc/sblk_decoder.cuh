// sblk_decoder.cuh — the small kernels of the SBL bidirectional decoder (SURVEY.md 8f.1):
//   * general multi-head attention for short sequences with separate Q and K/V sources (decoder self-attention with or
//     without the subsequent mask, decoder-encoder attention over cached encoder keys / values),
//   * token embedding + positional encoding,
//   * the synchronous bidirectional mixing of the two directions' hidden states,
//   * for the training path: the backward of the mixing and of the embedding (the attention's training forward /
//     backward is xattn_train_kernel in sblk_train.cuh, shared with the encoder).
// Reference: SBL/transformer/decoder.py:301-385 (recognize_beam), :79-191 (forward), DecoderLayer :388-408,
//            attention.py:32-83, module.py:8-32, utils.py:116-124 (get_subsequent_mask).
// Every projection / FFN GEMM and every residual + LayerNorm of the decoder runs on the encoder's tcgen05 kernels
// (sblk_gemm_fwd, sblk_gemm_splitk_fwd + sblk_sum_layernorm_fwd, sblk_gemm_ln_fwd); these kernels are the glue.
#pragma once
#include "sblk_common.cuh"
#include "sblk_train.cuh"

namespace sblk {

// ----------------------------------------------------------------------------------------------------------------
// out[b, q, h*64 + d] = sum_k softmax_k(Q[b,q,h] . K[b,k,h] * scale, masked) V[b,k,h,d]
// Q rows at q + (b*Lq + i)*ldq + h*64, K / V rows at k|v + (b*Lk + j)*ldk|ldv + h*64 (enc16), out enc16 row pitch ldo.
// mask: causal (key j > query i, get_subsequent_mask) and / or key lengths (j >= klens[b]).  One CTA per (b, h), fp32
// math in shared memory: Lq <= 32, Lk <= 128 (decoder prefixes are <= 17 tokens, encoder outputs <= 128 frames).
// ----------------------------------------------------------------------------------------------------------------
struct XAttnParams {
  const uint16_t* q;
  const uint16_t* k;
  const uint16_t* v;
  uint16_t* out;
  const int* klens;      // [N] valid keys or nullptr
  int ldq, ldk, ldv, ldo;
  int N, Lq, Lk, H;
  int causal;
  float scale;
  int fp16;
};

__global__ void __launch_bounds__(128)
xattention_kernel(const XAttnParams p) {
  extern __shared__ float xs[];
  grid_dep_launch();
  grid_dep_wait();
  const int b = blockIdx.x / p.H, h = blockIdx.x - b * p.H;
  const int Lq = p.Lq, Lk = p.Lk;
  float* sQ = xs;                    // [Lq][65]
  float* sK = sQ + Lq * 65;          // [Lk][65]
  float* sV = sK + Lk * 65;          // [Lk][65]
  float* sP = sV + Lk * 65;          // [Lq][Lk + 1]
  const int klen = (p.klens != nullptr) ? min(max(__ldg(p.klens + b), 0), Lk) : Lk;
  for (int i = threadIdx.x; i < Lq * 64; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    sQ[t * 65 + d] = ld16(p.q + (static_cast<size_t>(b) * Lq + t) * p.ldq + h * 64 + d, p.fp16);
  }
  for (int i = threadIdx.x; i < Lk * 64; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    sK[t * 65 + d] = ld16(p.k + (static_cast<size_t>(b) * Lk + t) * p.ldk + h * 64 + d, p.fp16);
    sV[t * 65 + d] = ld16(p.v + (static_cast<size_t>(b) * Lk + t) * p.ldv + h * 64 + d, p.fp16);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int qi = warp; qi < Lq; qi += nw) {
    float sc[4];
    float mx = -INFINITY;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int kj = lane + 32 * e;
      sc[e] = -INFINITY;
      if (kj < klen && !(p.causal && kj > qi)) {
        float a = 0.0f;
        for (int d = 0; d < 64; ++d) a += sQ[qi * 65 + d] * sK[kj * 65 + d];
        sc[e] = a * p.scale;
      }
      mx = fmaxf(mx, sc[e]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float ex[4], sum = 0.0f;
#pragma unroll
    for (int e = 0; e < 4; ++e) { ex[e] = __expf(sc[e] - mx); sum += ex[e]; }   // all-masked row: NaN like the reference
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.0f / sum;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int kj = lane + 32 * e;
      if (kj < Lk) sP[qi * (Lk + 1) + kj] = ex[e] * inv;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < Lq * 64; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    float a = 0.0f;
    for (int j = 0; j < Lk; ++j) a += sP[t * (Lk + 1) + j] * sV[j * 65 + d];
    const uint32_t w = p.fp16 ? pack_f16x2(a, 0.0f) : pack_bf16x2(a, 0.0f);
    p.out[(static_cast<size_t>(b) * Lq + t) * p.ldo + h * 64 + d] = static_cast<uint16_t>(w & 0xFFFFu);
  }
}

// x[n, l, :] = emb[tok[n * ld_tok + l], :] * scale + pe[l, :]   -> fp32 and enc16 copies ([N*L, D], D % 4 == 0)
// decoder.py:323-327: self.tgt_word_emb(ys) * self.x_logit_scale + self.positional_encoding(ys)
__global__ void __launch_bounds__(256)
embed_pe_kernel(const long long* __restrict__ tok, int ld_tok, const float* __restrict__ emb,
                const float* __restrict__ pe, float* __restrict__ out_f32, uint16_t* __restrict__ out_16, int rows, int L,
                int D, int vocab, float scale, int fp16) {
  const int d4 = D / 4;
  const long long total = static_cast<long long>(rows) * d4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % d4);
    const int r = static_cast<int>(i / d4);
    long long t = tok[static_cast<long long>(r / L) * ld_tok + (r % L)];
    t = t < 0 ? 0 : (t >= vocab ? vocab - 1 : t);
    const float4 e = __ldg(reinterpret_cast<const float4*>(emb + t * D) + c);
    const float4 q = __ldg(reinterpret_cast<const float4*>(pe + static_cast<long long>(r % L) * D) + c);
    const float4 o = make_float4(e.x * scale + q.x, e.y * scale + q.y, e.z * scale + q.z, e.w * scale + q.w);
    reinterpret_cast<float4*>(out_f32)[i] = o;
    if (out_16 != nullptr) {
      uint2 w;
      w.x = fp16 ? pack_f16x2(o.x, o.y) : pack_bf16x2(o.x, o.y);
      w.y = fp16 ? pack_f16x2(o.z, o.w) : pack_bf16x2(o.z, o.w);
      reinterpret_cast<uint2*>(out_16)[i] = w;
    }
  }
}

// Synchronous bidirectional mixing, decoder.py:336-346,358-362 (the reference updates both tensors IN PLACE through
// aliases: `dec_output_left = dec_output_l2r` ... so the second loop already sees the updated left stream):
//   l2r'[n, i] = l2r[n, i] + r2l[n, L-1-i]
//   r2l'[n, i] = r2l[n, i] + l2r'[n, L-1-i] = 2 * r2l[n, i] + l2r[n, L-1-i]
// fp32 in -> fp32 + enc16 out (new buffers).
__global__ void __launch_bounds__(256)
bidir_mix_kernel(const float* __restrict__ l2r, const float* __restrict__ r2l, float* __restrict__ l2r_out,
                 float* __restrict__ r2l_out, uint16_t* __restrict__ l2r_16, uint16_t* __restrict__ r2l_16, int N, int L,
                 int D, int fp16) {
  const int d4 = D / 4;
  const long long total = static_cast<long long>(N) * L * d4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % d4);
    const long long row = i / d4;
    const int pos = static_cast<int>(row % L);
    const long long n = row / L;
    const long long mirror = (n * L + (L - 1 - pos)) * d4 + c;
    const float4 a = __ldg(reinterpret_cast<const float4*>(l2r) + i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(r2l) + i);
    const float4 am = __ldg(reinterpret_cast<const float4*>(l2r) + mirror);
    const float4 bm = __ldg(reinterpret_cast<const float4*>(r2l) + mirror);
    const float4 lo = make_float4(a.x + bm.x, a.y + bm.y, a.z + bm.z, a.w + bm.w);
    // r2l' = r2l + l2r'[mirror] with l2r'[mirror] = l2r[mirror] + r2l[this]  (same summation order as the reference)
    const float4 ro = make_float4(b.x + (am.x + b.x), b.y + (am.y + b.y), b.z + (am.z + b.z), b.w + (am.w + b.w));
    reinterpret_cast<float4*>(l2r_out)[i] = lo;
    reinterpret_cast<float4*>(r2l_out)[i] = ro;
    uint2 w;
    w.x = fp16 ? pack_f16x2(lo.x, lo.y) : pack_bf16x2(lo.x, lo.y);
    w.y = fp16 ? pack_f16x2(lo.z, lo.w) : pack_bf16x2(lo.z, lo.w);
    reinterpret_cast<uint2*>(l2r_16)[i] = w;
    w.x = fp16 ? pack_f16x2(ro.x, ro.y) : pack_bf16x2(ro.x, ro.y);
    w.y = fp16 ? pack_f16x2(ro.z, ro.w) : pack_bf16x2(ro.z, ro.w);
    reinterpret_cast<uint2*>(r2l_16)[i] = w;
  }
}

// ----------------------------------------------------------------------------------------------------------------
// Training-path backward kernels of the decoder glue.
// ----------------------------------------------------------------------------------------------------------------
// Backward of bidir_mix_kernel, fp32, given the gradients g_a / g_b of l2r' / r2l':
//   d_l2r[n, i] = g_a[n, i] + g_b[n, L-1-i]
//   d_r2l[n, i] = g_b[n, i] + (g_a[n, L-1-i] + g_b[n, i])
// The second line is the order in which autograd through the aliased loops adds the two paths into r2l (the direct one
// and the one through l2r'[L-1-i]); g_a + 2 g_b would round differently.  __fadd_rn: no contraction, bit-exact.
__global__ void __launch_bounds__(256)
bidir_mix_bwd_kernel(const float* __restrict__ ga, const float* __restrict__ gb, float* __restrict__ d_l2r,
                     float* __restrict__ d_r2l, int N, int L, int D) {
  const int d4 = D / 4;
  const long long total = static_cast<long long>(N) * L * d4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % d4);
    const long long row = i / d4;
    const int pos = static_cast<int>(row % L);
    const long long n = row / L;
    const long long mirror = (n * L + (L - 1 - pos)) * d4 + c;
    const float4 a = __ldg(reinterpret_cast<const float4*>(ga) + i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(gb) + i);
    const float4 am = __ldg(reinterpret_cast<const float4*>(ga) + mirror);
    const float4 bm = __ldg(reinterpret_cast<const float4*>(gb) + mirror);
    reinterpret_cast<float4*>(d_l2r)[i] = make_float4(__fadd_rn(a.x, bm.x), __fadd_rn(a.y, bm.y), __fadd_rn(a.z, bm.z),
                                                      __fadd_rn(a.w, bm.w));
    reinterpret_cast<float4*>(d_r2l)[i] = make_float4(
        __fadd_rn(b.x, __fadd_rn(am.x, b.x)), __fadd_rn(b.y, __fadd_rn(am.y, b.y)),
        __fadd_rn(b.z, __fadd_rn(am.z, b.z)), __fadd_rn(b.w, __fadd_rn(am.w, b.w)));
  }
}

// Embedding backward: demb[v, :] = scale * sum of dx[r, :] over the rows r whose (clamped, as in embed_pe_kernel) token
// id is v, rows in the token layout of embed_pe_kernel.  Deterministic without atomics: CTA (v, 128-column slice); warp
// s adds the rows r = s, s + 8, ... in order (lane = 4 columns), the 8 warp sums are then added in warp order.  Every
// CTA scans the token ids (staged 1024 at a time in shared memory) and reads only its own rows of dx.
constexpr int kEmbedBwdIds = 1024;
__global__ void __launch_bounds__(256)
embed_bwd_kernel(const long long* __restrict__ tok, int ld_tok, const float* __restrict__ dx, float* __restrict__ demb,
                 int rows, int L, int D, int vocab, float scale) {
  __shared__ int ids[kEmbedBwdIds];
  __shared__ float4 part[8][32];
  const int v = blockIdx.x;
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int d4 = D / 4;
  const int c4 = blockIdx.y * 32 + lane;
  float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (int r0 = 0; r0 < rows; r0 += kEmbedBwdIds) {
    const int nr = min(kEmbedBwdIds, rows - r0);
    for (int i = threadIdx.x; i < nr; i += blockDim.x) {
      const int r = r0 + i;
      long long t = __ldg(tok + static_cast<long long>(r / L) * ld_tok + (r % L));
      t = t < 0 ? 0 : (t >= vocab ? vocab - 1 : t);
      ids[i] = static_cast<int>(t);
    }
    __syncthreads();
    if (c4 < d4) {
      for (int i = slice; i < nr; i += 8) {
        if (ids[i] != v) continue;
        const float4 g = __ldg(reinterpret_cast<const float4*>(dx) + static_cast<long long>(r0 + i) * d4 + c4);
        acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
      }
    }
    __syncthreads();
  }
  part[slice][lane] = acc;
  __syncthreads();
  if (slice == 0 && c4 < d4) {
    float4 s = part[0][lane];
#pragma unroll
    for (int k = 1; k < 8; ++k) { s.x += part[k][lane].x; s.y += part[k][lane].y; s.z += part[k][lane].z; s.w += part[k][lane].w; }
    reinterpret_cast<float4*>(demb)[static_cast<long long>(v) * d4 + c4] =
        make_float4(s.x * scale, s.y * scale, s.z * scale, s.w * scale);
  }
}

}  // namespace sblk

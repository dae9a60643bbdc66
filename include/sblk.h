/* sblk.h — C ABI of libsblk.so: the B200 (sm_100a) kernel library behind the drop-in visual encoder
 * (Conv3d frontend -> per-frame ResNet-18 trunk -> transformer Encoder) of SBL_For_Multilingual_Lip_Reading.
 *
 * The reference has no native code and no plugin ABI for this path: every call below replaces a stock
 * torch.nn call site of the reference (cited per function, paths relative to
 * SBL_Multilingual_Lip_reading/).  Conventions:
 *   - every pointer is a raw CUDA device pointer on the caller's CURRENT device; `stream` is a cudaStream_t
 *   - functions only enqueue work (no sync, no allocation) and are CUDA-graph capturable
 *   - return 0 = OK, < 0 = argument / shape / alignment error (unsupported configurations fail loudly,
 *     there is no CPU or library fallback), > 0 = cudaError_t of the failed launch
 *   - sblk_last_error() returns a thread-local description of the last failure
 *   - convolutional activations / weights are bf16 (NHWC / K-major); the transformer encoder's 16-bit operands
 *     ("enc16": x_in, every encoder weight, the qkv / attention / hidden workspaces) are IEEE fp16 when
 *     sblk_enc16_format() == 1 (default build) and bf16 when it is 0 — same bytes, same tcgen05 kind::f16 rate,
 *     3 more mantissa bits for LayerNorm-bounded values; accumulation, normalisation and the residual stream are fp32.
 *     Parameters documented as "bf16" in the encoder section below mean "enc16".
 *   - sblk_set_pdl / sblk_set_sm_limit are per calling host thread (nn.DataParallel replicas launch from worker threads)
 */
#ifndef SBLK_H_
#define SBLK_H_

#ifdef __cplusplus
extern "C" {
#endif

#define SBLK_VERSION 200

int sblk_version(void);
const char* sblk_last_error(void);
/* Number of SMs of the current device (>0) or a negative error. Also performs the one-time per-device setup. */
int sblk_init(void);
/* Device-side pipeline watchdog word (0 = never fired); survives a trapped launch. */
unsigned int sblk_watchdog_code(void);
/* Enable (1) / disable (0) programmatic dependent launch for the CALLING THREAD's subsequent launches (a CUDA graph
 * keeps whatever was set while it was captured).  Returns the previous value. */
int sblk_set_pdl(int enable);
/* Size the persistent grids of the calling thread's subsequent launches for at most max_sms SMs (rounded down to an
 * even count; 0 = all SMs).  Used to run independent kernel chains (halves of a clip batch) concurrently on disjoint
 * SM sets.  Returns the previous limit. */
int sblk_set_sm_limit(int max_sms);
/* Which kernel sblk_conv3d_bn_relu_pool_fwd launches for the CALLING THREAD: 0 (default) = the transposed stem with
 * the filter resident in tensor memory (csrc/sblk_stem_t.cuh), 1 = the pixel-major stem of round 1
 * (csrc/sblk_conv3d.cuh, kept for A/B measurements).  Same inputs, same outputs.  Returns the previous value. */
int sblk_set_stem_variant(int variant);
/* Number of kernels launched by this library since load (all threads). */
long long sblk_launch_count(void);

/* ---- packers (one-time, per weight version) ------------------------------------------------------- */
/* Conv3d(1,64,(5,7,7)) weight [64,1,5,7,7] fp32 + BatchNorm3d(eval) -> bf16 [64][320] (k = dt*64 + (r/2)*16 +
 * (r%2)*8 + s, zero elsewhere) + fp32 bias[64].
 * replaces: nn.Conv3d / nn.BatchNorm3d parameters, transformer/video_frontend.py:100-101 */
int sblk_pack_conv3d(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
                     float eps, void* w_packed_bf16, float* bias, void* stream);
/* Conv2d weight [Co,Ci,R,S] fp32 + BatchNorm2d(eval) -> bf16 [Co][R][S][Ci] + fp32 bias[Co].
 * gamma == NULL packs without folding (bias, if given, is zero-filled).
 * replaces: conv3x3 / downsample conv + bn parameters, transformer/video_frontend.py:10-12,20-24,68-72 */
int sblk_pack_conv2d(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
                     float eps, void* w_packed_bf16, float* bias, int Co, int Ci, int R, int S, void* stream);
/* fp32 -> bf16 cast of n elements (n % 4 == 0). Linear weights [out,in] are already K-major. */
int sblk_cast_f32_bf16(const float* src, void* dst_bf16, long long n, void* stream);
/* 16-bit operand format of the transformer-encoder entry points: 1 = IEEE fp16 (default), 0 = bf16. */
int sblk_enc16_format(void);
/* fp32 -> enc16 cast of n elements (n % 4 == 0; fp16 conversions saturate at +-65504): encoder weights and inputs. */
int sblk_cast_f32_enc16(const float* src, void* dst_enc16, long long n, void* stream);
/* Hint: pull the n ranges [ptrs[i], ptrs[i] + bytes[i]) into L2 (prefetch.global.L2 per 128-byte line; no data is
 * produced; ptrs / bytes are HOST arrays).  Used on a side stream for the packed weights of the layers that run later in
 * the same forward. */
int sblk_l2_prefetch(const void* const* ptrs, const long long* bytes, int n, void* stream);
/* Co-scheduling gate for two concurrent kernel chains (runner.PipelinedVisualEncoderPlan: the encoder stack of batch
 * i-1 next to the clip prep + stem of batch i).  Enqueues a one-thread kernel that returns once `count` more CTAs have
 * bumped gate[0] (sblk_encoder_stack_args.resident_counter) than gate[1] accounts for, or after timeout_us; gate[1] then
 * advances by `count`.  Kernels enqueued behind it on `stream` therefore start only when the other chain's clusters have
 * been placed.  A scheduling hint only: results never depend on it.  No reference counterpart. */
int sblk_gate_wait(void* gate_u32x2, int count, int timeout_us, void* stream);

/* ---- visual frontend ------------------------------------------------------------------------------ */
/* Number of bf16 elements the prepped clip of sblk_prep_clip needs (includes the over-read slack). */
long long sblk_prep_clip_elems(int N, int T);
/* x fp32 [N,1,T,88,88] -> bf16 row-Toeplitz entries [N][T+4][2][47][44][8] (zero temporal (2) and spatial (3)
 * borders materialised; entry (pl,yy,x) = the 8 input pixels 2x-3.. of padded row 2yy+pl).
 * replaces: the implicit zero padding / stride-2 window walk of nn.Conv3d(stride=(1,2,2), padding=(2,3,3)),
 * transformer/video_frontend.py:100 */
int sblk_prep_clip(const float* x, void* x_prepped_bf16, int N, int T, void* stream);
/* Fused input pipeline (SURVEY.md 8f.3): raw uint8 gray frames [N, T_in, H0, W0] -> the prepped layout of
 * sblk_prep_clip for clips of T_out >= T_in frames (trailing frames are zero padding in normalised space), cropping
 * every frame to 88x88 at (crop_y0, crop_x0) or at the per-frame offsets crop_yx int32 [N*T_in][2] (y1, x1), and
 * normalising through lut_bf16: 256 bf16 values, lut[u] = bf16((u / 255. - 0.413621) / 0.1700239) evaluated on the
 * host.  Bit-identical to sblk_prep_clip of the reference-normalised fp32 clip.
 * replaces: load_file / ColorNormalize / CenterCrop / RandomCrop / frame zero-padding of the reference loader,
 * SBL/data_gen.py:122-125,276-296 ; SBL/cvtransforms.py:7-33,44-48 */
int sblk_prep_clip_u8(const void* x_u8, const void* lut_bf16, const int* crop_yx, int crop_y0, int crop_x0, void* out,
                      int N, int T_in, int T_out, int H0, int W0, void* stream);
/* Conv3d + BN3d(eval) + ReLU + MaxPool3d((1,3,3),(1,2,2),(0,1,1)) + transpose(1,2).contiguous().view:
 * prepped clip -> bf16 NHWC [N*T,22,22,64] (flat_out = 0) or the flat layout below (flat_out = 1).
 * replaces: Lipreading.frontend3D and _frontend_forward's relayout, transformer/video_frontend.py:99-104,111-115 */
int sblk_conv3d_bn_relu_pool_fwd(const void* x_prepped_bf16, const void* w_packed_bf16, const float* bias,
                                 void* out_bf16, int N, int T, int flat_out, void* stream);
/* The same stem WITHOUT the prepped copy of the clip: producer warps of the (transposed, tensor-memory-filter) stem
 * kernel build the row-Toeplitz entries in shared memory straight from the input — exactly one of
 *   x_f32  fp32 clips [N,1,T,88,88] (reference layout; T_out == T_in), or
 *   x_u8   raw uint8 gray frames [N,T_in,H0,W0] + lut_bf16 / crop_yx / (crop_y0, crop_x0) as in sblk_prep_clip_u8,
 *          clips zero-padded (in normalised space) to T_out frames.
 * Bit-identical to sblk_prep_clip[_u8] + sblk_conv3d_bn_relu_pool_fwd; saves the 70 MB round trip through HBM and a launch.
 * replaces: the loader transforms (u8) + Lipreading.frontend3D + relayout, SBL/data_gen.py:122-125,276-296,
 * transformer/video_frontend.py:99-104,111-115 */
int sblk_stem_fused_fwd(const float* x_f32, const void* x_u8, const void* lut_bf16, const int* crop_yx, int crop_y0,
                        int crop_x0, const void* w_packed_bf16, const float* bias, void* out_bf16, int N, int T_in,
                        int T_out, int H0, int W0, int flat_out, void* stream);
/* Rows of the zero-haloed flat activation layout for F frames of H x W pixels:
 * pixel (f,y,x) -> row (f*(H+1) + 1 + y)*(W+2) + 1 + x of a [rows, C] bf16 matrix; all other rows are zero. */
long long sblk_flat_rows(int F, int H, int W);
/* Stride-1 3x3 / pad 1 Conv2d (C -> C, C == 64 or 128) + folded BN (+ residual) (+ ReLU) over the flat layout
 * (flat_out of sblk_conv3d_bn_relu_pool_fwd / sblk_conv2d_dual_igemm_fwd or a previous call); output is again flat
 * with zero halos.  w_packed_bf16 is [C][10*C]: the 9 taps of sblk_pack_conv2d's [C][3][3][C] followed by a CxC
 * identity.  Those last C columns are not read; they are kept so that the packed layout does not change.
 * W + 2 <= 31 for C == 64, <= 15 for C == 128.  CTA-pair (cta_group::2) shifted-window implicit GEMM.
 * replaces: the stride-1 convs of ResNet layer1 and layer2, transformer/video_frontend.py:10-12,28-41 */
int sblk_flatconv3x3_fwd(const void* x_flat, const void* w_packed_bf16, const float* bias, const void* residual_flat,
                         void* out_flat, int F, int H, int W, int C, int relu, void* stream);
/* Same conv with the tile order chosen by the caller: reverse != 0 makes every CTA pair walk its contiguous tile range
 * from the last tile to the first.  Consecutive convs of a stage alternate the direction, so that the rows a pair wrote
 * (and read as residual) last in one conv — the ones most likely still resident in L2 — are the first it reads in the
 * next (a layer-1 tensor is 65.6 MB at the BASELINE batch: a conv with residual touches 197 MB against 126 MB of L2).
 * Bit-identical to sblk_flatconv3x3_fwd. */
int sblk_flatconv3x3_dir_fwd(const void* x_flat, const void* w_packed_bf16, const float* bias,
                             const void* residual_flat, void* out_flat, int F, int H, int W, int C, int relu,
                             int reverse, void* stream);
/* Implicit-GEMM Conv2d (3x3 pad 1 or 1x1 pad 0, stride 1 or 2) over bf16 NHWC [F,H,W,Cin] with folded BN:
 * out = act(conv(x, w) + bias (+ residual)), bf16 NHWC [F,P,Q,Cout].  Cin % 64 == 0, Cout % 64 == 0.
 * in_row_pitch / in_frame_pitch (pixels, 0 = dense) let x point at pixel (0,0,0) of a pitched layout such as the
 * flat one (pass x_flat + (W+3)*Cin elements, W+2, (H+1)*(W+2)).
 * replaces: BasicBlock.forward conv1/bn1/relu, conv2/bn2/+=residual/relu and the downsample branch,
 * transformer/video_frontend.py:28-41,68-72 */
int sblk_conv2d_igemm_fwd(const void* x_bf16, const void* w_packed_bf16, const float* bias,
                          const void* residual_bf16, void* out_bf16, int F, int H, int W, int Cin, int Cout,
                          int R, int S, int stride, int pad, int relu, int in_row_pitch, int in_frame_pitch,
                          void* stream);
/* sblk_conv2d_igemm_fwd with a K-extension: out = act(conv(x, w) + conv1x1_stride2(x2, w2) + bias (+ residual)).
 * x2 is bf16 NHWC [F,H2,W2,Cin2] (pitches as for x), w2 bf16 [Cout][Cin2]; the 1x1 / pad 0 / stride2 view of x2 must
 * give the conv's own P x Q output grid.  Both contractions accumulate in ONE fp32 tensor-memory tile (the k-blocks
 * of (x2, w2) follow the conv's own in the same TMA ring), so a BasicBlock with a downsample branch runs as
 *   y   = sblk_conv2d_igemm_fwd(x, conv1, stride 2)                                  (256-wide pair tiles)
 *   out = sblk_conv2d_igemm_ext_fwd(y, conv2, bias2 + bias_ds, x2 = x, w2 = w_ds)    (relu(bn2(conv2 y) + bn_ds(ds x)))
 * with the branch never rounded to bf16 and no launch of its own.  Cout % 128 == 0 (CTA-pair kernel).
 * replaces: BasicBlock.forward conv2/bn2, downsample(x), += residual, relu, transformer/video_frontend.py:35-41,68-72 */
int sblk_conv2d_igemm_ext_fwd(const void* x_bf16, const void* w_packed_bf16, const float* bias,
                              const void* residual_bf16, void* out_bf16, int F, int H, int W, int Cin, int Cout,
                              int R, int S, int stride, int pad, int relu, int in_row_pitch, int in_frame_pitch,
                              const void* x2_bf16, const void* w2_bf16, int H2, int W2, int Cin2, int stride2,
                              int x2_row_pitch, int x2_frame_pitch, void* stream);
/* A whole BasicBlock of ResNet layer 3 (Cout = 256) or layer 4 (Cout = 512) in ONE launch:
 *   y1  = relu(conv3x3_stride(x, w1) + bias1)                                   (workspace y1_ws, bf16 [F,P,Q,Cout])
 *   out = relu(conv3x3(y1, w2) + bias2 + (w_ds ? conv1x1_stride(x, w_ds) : x))   (bias2 includes the downsample shift)
 * Pair tiles are made of whole frames, so conv2 of a tile depends on conv1 of the same frames only: every CTA pair runs
 * conv1 over its work units, then conv2 over the same units — no grid-wide synchronisation, no second launch.  Cout =
 * 256: one unit per frame group, a pair-wide mbarrier per tile.  Cout = 512: two column tiles per frame group on
 * neighbouring CTA pairs, which meet at a self-resetting counter pair in flags_ws (uint32 [sblk_conv_block_flag_words],
 * zeroed ONCE by the caller; one workspace per stream).  The grid never exceeds the SMs of sblk_set_sm_limit, which is
 * what keeps the waiting pairs deadlock-free next to a co-running kernel.  Bit-identical to sblk_conv2d_igemm_fwd +
 * sblk_conv2d_igemm[_ext]_fwd.  w_ds must be given exactly when the block changes shape; x may be pitched (flat layout)
 * only then.  Returns -2 (nothing launched) when a CTA pair would own more than 32 units: launch the convs one by one.
 * replaces: BasicBlock.forward of ResNet layer3 / layer4, transformer/video_frontend.py:28-41,68-72 */
int sblk_conv_block_flag_words(int F, int H, int W, int stride);
int sblk_conv_block_fwd(const void* x_bf16, const void* w1_packed_bf16, const float* bias1, const void* w2_packed_bf16,
                        const float* bias2, const void* w_ds_packed_bf16, void* y1_ws, void* flags_ws, void* out_bf16,
                        int F, int H, int W, int Cin, int Cout, int stride, int in_row_pitch, int in_frame_pitch,
                        void* stream);
/* BasicBlock head of layers 2-4 in one launch: out = relu(conv3x3_stride_s(x) + bias) and the downsample branch
 * out_ds = conv1x1_stride_s(x) + bias_ds.  The 1x1 conv reads exactly the centre-tap A tiles of the 3x3 conv, so
 * both share one pass over x (second TMEM accumulator).  w_ds_packed is [Cout][1][1][Cin]; Cout % 128 == 0.
 * replaces: BasicBlock.conv1/bn1/relu + downsample(conv1x1, bn), transformer/video_frontend.py:30-32,35-36,68-72
 * flat_out = 1 writes both outputs into the zero-haloed flat layout (pixel rows only: the caller provides buffers
 * whose halo rows are already zero), so a stride-1 sblk_flatconv3x3_fwd can consume them directly. */
int sblk_conv2d_dual_igemm_fwd(const void* x_bf16, const void* w_packed_bf16, const float* bias,
                               const void* w_ds_packed_bf16, const float* bias_ds, void* out_bf16, void* out_ds_bf16,
                               int F, int H, int W, int Cin, int Cout, int stride, int relu, int in_row_pitch,
                               int in_frame_pitch, int flat_out, void* stream);
/* bf16 NHWC [F,HW,C] -> mean over HW: fp32 [F,C] and/or bf16 [F,C] (either may be NULL).
 * replaces: nn.AdaptiveAvgPool2d(1) + view, transformer/video_frontend.py:87-88 */
int sblk_avgpool_fwd(const void* x_bf16, float* out_f32, void* out_bf16, int F, int HW, int C, void* stream);
/* Same, times a per-element fp32 factor scale[F,C] (NULL = none): the always-on F.dropout(x, p=0.5) of
 * Lipreading.forward (transformer/video_frontend.py:122) applied in the pooling pass, with the factor (mask / (1-p))
 * drawn ahead of time by the caller; bit-identical to pooling followed by that dropout.  out16_enc != 0 writes the
 * 16-bit output in the encoder's operand format (it is then x_in of sblk_encoder_stack_fwd) instead of bf16. */
int sblk_avgpool_scale_fwd(const void* x_bf16, const float* scale, float* out_f32, void* out_16, int F, int HW, int C,
                           int out16_enc, void* stream);

/* ---- transformer encoder -------------------------------------------------------------------------- */
/* out = act(A[M,K] * W[N,K]^T + bias (+ residual_bf16)); bf16 operands, fp32 accumulate; writes bf16 and/or fp32.
 * K % 64 == 0, N % 64 == 0.
 * replaces: nn.Linear call sites, transformer/attention.py:41-43,57 ; module.py:49 ; encoder.py:53 */
int sblk_gemm_fwd(const void* a_bf16, const void* w_bf16, const float* bias, const void* residual_bf16,
                  void* out_bf16, float* out_f32, int M, int N, int K, int relu, void* stream);
/* Split-K plan for a Linear at small M: the number of K ranges (1, 2, 4 or 8) that fills the SMs with one tile each
 * (negative on error).  The caller allocates [splits, M, N] fp32 for sblk_gemm_splitk_fwd. */
int sblk_gemm_splitk_plan(int M, int N, int K);
/* Split-K Linear: partial s = A[:, K_s] W[:, K_s]^T (+ bias for s == 0) -> out_partials[s] fp32 [M,N]; the partials
 * are summed by sblk_sum_layernorm_fwd (deterministic: no atomics).  (K / 64) % splits == 0.
 * replaces: nn.Linear call sites whose output feeds a LayerNorm, attention.py:57 ; module.py:49 ; encoder.py:53 */
int sblk_gemm_splitk_fwd(const void* a_bf16, const void* w_bf16, const float* bias, float* out_partials, int M, int N,
                         int K, int splits, void* stream);
/* sblk_add_layernorm_fwd over the sum of nparts partial inputs x_parts[nparts][M,512] (+ bias[512]). */
int sblk_sum_layernorm_fwd(const float* x_parts, int nparts, const float* bias, const float* residual,
                           const float* gamma, const float* beta, const float* pe, const int* lengths,
                           float* out_f32, void* out_bf16, int M, int T, int D, float eps, void* stream);
/* y = LayerNorm(x + residual) * gamma + beta (+ pe[m % T]) (* (m % T < lengths[m / T])), D must be 512.
 * residual, pe, lengths, out_f32, out_bf16 may be NULL.
 * replaces: nn.LayerNorm call sites attention.py:58, module.py:51, encoder.py:53-55 (+PositionalEncoding,
 * module.py:26-32) and the non_pad_mask multiplies, encoder.py:86,89 + utils.py:98-113 */
int sblk_add_layernorm_fwd(const float* x, const float* residual, const float* gamma, const float* beta,
                           const float* pe, const int* lengths, float* out_f32, void* out_bf16, int M, int T,
                           int D, float eps, void* stream);
/* Fused self-attention on a packed projection qkv bf16 [N*T, 3*H*64] (q|k|v): softmax(QK^T * scale, keys >=
 * lengths[b] masked) V -> bf16 [N*T, H*64].  probs (optional) fp32 [H*N, T, T] with batch index h*N + b.
 * d_k must be 64, T <= 128.
 * replaces: ScaledDotProductAttention.forward + head split/merge, transformer/attention.py:45-55,72-83 and
 * get_attn_pad_mask, transformer/utils.py:140-147 */
int sblk_attention_fwd(const void* qkv_bf16, void* out_bf16, float* probs, const int* lengths, int N, int T,
                       int H, int d_k, float scale, void* stream);

/* One launch for Linear(K -> 512) + bias + fp32 residual + LayerNorm(512) (+ pe[m % T]) (* pad mask):
 * y = LN(A[M,K] W[512,K]^T + bias + residual) * gamma + beta (+ pe) (* (m % T < lengths[m / T])).
 * A, W bf16; accumulation, statistics (two-pass) and the residual stream fp32.  N must be 512, K % 64 == 0.
 * A cluster of 4 CTAs owns each 128-row tile and combines the row statistics through distributed shared memory.
 * replaces: fc + layer_norm(out + residual) attention.py:57-58 ; w_2 + layer_norm(out + x) module.py:49-51 ;
 * layer_norm_in(linear_in(x)) + positional_encoding encoder.py:53-55 ; `*= non_pad_mask` encoder.py:86,89 */
int sblk_gemm_ln_fwd(const void* a_bf16, const void* w_bf16, const float* bias, const float* residual_f32,
                     const float* gamma, const float* beta, const float* pe, const int* lengths, float* out_f32,
                     void* out_bf16, int M, int N, int K, int T, float eps, void* stream);
/* Clips per 128-row tile used by sblk_qkv_attention_fwd for T frames per clip (-1 if T is unsupported). */
int sblk_qkv_group_clips(int T);
/* One launch for the q/k/v projections + scaled-dot-product self-attention of all heads:
 * x bf16 [N*T, K]; w_heads bf16 [H*192, K] head-major (rows h*192 + [0,64) = w_qs rows of head h, [64,128) = w_ks,
 * [128,192) = w_vs); bias_heads fp32 [H*192] in the same order -> out bf16 [N*T, H*64] (heads concatenated).
 * d_k must be 64, T <= 128, K % 64 == 0.
 * replaces: MultiHeadAttention.forward up to the head merge, attention.py:41-55, ScaledDotProductAttention.forward,
 * attention.py:72-83, and get_attn_pad_mask, utils.py:140-147 (attention maps are not produced by this entry point:
 * use sblk_gemm_fwd + sblk_attention_fwd when return_attns is requested) */
int sblk_qkv_attention_fwd(const void* x_bf16, const void* w_heads_bf16, const float* bias_heads, const int* lengths,
                           void* out_bf16, int N, int T, int H, int d_k, int K, float scale, void* stream);

/* The whole transformer encoder stack in ONE launch (eval mode):
 *   x = LayerNorm(x_in W_in^T + b_in) + pe[t];  n_layers x { x = LN(fc(attn(x)) + x) * keep ; x = LN(w_2 relu(w_1 x) + x) * keep }
 * A thread-block cluster owns a group of floor(128 / T) whole clips and runs it through every layer without any
 * inter-group synchronisation; each CTA of the cluster computes 1 / cluster_size of every step's output features.
 * All per-layer tensors are STACKED along their first dimension:
 *   w_heads bf16 [L*1536, 512] (per layer the head-major q_h|k_h|v_h rows of sblk_qkv_attention_fwd), b_heads fp32 [L*1536],
 *   w_fc bf16 [L*512, 512], b_fc / ln1_gamma / ln1_beta fp32 [L*512], w_1 bf16 [L*d_inner, 512], b_1 fp32 [L*d_inner],
 *   w_2 bf16 [L*512, d_inner], b_2 / ln2_gamma / ln2_beta fp32 [L*512].
 * x_in bf16 [N*T, d_in]; w_in bf16 [512, d_in]; pe fp32 [>= T, 512]; lengths int32 [N] or NULL; out fp32 [N*T, 512];
 * workspace: sblk_encoder_stack_workspace_bytes(N, T, d_inner) bytes of device memory (contents irrelevant).
 * Implemented for n_head = 8, d_k = d_v = 64, d_model = 512, T <= 128, d_in % 128 == 0, d_inner % 1024 == 0 and <= 2048;
 * anything else returns < 0 (callers then use the per-step entry points above).
 * replaces: Encoder.forward transformer/encoder.py:36-67 ; EncoderLayer.forward encoder.py:83-91 ;
 * MultiHeadAttention.forward attention.py:32-60 ; ScaledDotProductAttention.forward attention.py:72-83 ;
 * PositionwiseFeedForward.forward module.py:47-52 ; get_non_pad_mask / get_attn_pad_mask utils.py:98-113,140-147 */
typedef struct sblk_encoder_stack_args {
  const void* x_in;
  const void* w_in;
  const float* b_in;
  const float* ln_in_gamma;
  const float* ln_in_beta;
  const float* pe;
  const void* w_heads;
  const float* b_heads;
  const void* w_fc;
  const float* b_fc;
  const float* ln1_gamma;
  const float* ln1_beta;
  const void* w_1;
  const float* b_1;
  const void* w_2;
  const float* b_2;
  const float* ln2_gamma;
  const float* ln2_beta;
  const int* lengths;
  float* out;
  void* workspace;
  int N, T, n_layers, n_head, d_k, d_model, d_in, d_inner;
  float scale; /* 1 / temperature */
  float eps;   /* LayerNorm eps (shared by all LayerNorms of the stack) */
  int cluster_size;   /* 0 = automatic (16 CTAs per cluster when <= 7 clusters, else 8), or 8 / 16 */
  void* debug_stamps; /* NULL, or device uint64 [(1 + 4*n_layers)*8 + 2*groups]: per-stage clock64 stamps of CTA 0, then
                       * (start, end) globaltimer ns of every cluster (profiling aid) */
  void* resident_counter; /* NULL, or device uint32[2] (zero-initialised once): every CTA adds 1 to word 0 when it starts
                           * running, i.e. when its cluster owns its SMs (see sblk_gate_wait) */
  int no_multicast;   /* 0 = activation tiles are loaded once per cluster and TMA-multicast (default); 1 = every CTA loads
                       * its own copy (bit-identical; A/B timing and tests) */
  int groups_per_cluster; /* 0 / 1 = one clip group per cluster; 2 = every cluster runs two clip groups through the stack
                           * alternately, the loads / MMAs of one hidden behind the epilogues / cluster barriers of the
                           * other (half the SMs for little more than the time of one group; bit-identical) */
} sblk_encoder_stack_args;
long long sblk_encoder_stack_workspace_bytes(int N, int T, int d_inner);
int sblk_encoder_stack_fwd(const sblk_encoder_stack_args* args, void* stream);


/* ---- training path: forward with batch statistics + backward (BASELINE configs[3]) ---------------------------------
 * replaces: `model.train()` + `loss.backward()` through the hot path,
 * VSR_visual_frontend_pretraining_on_LRW_LRW1000_classify/train.py:107-146 and SBL/train.py:177-210 (autograd of the stock
 * nn.Conv3d / Conv2d / BatchNorm / ReLU / MaxPool3d / AdaptiveAvgPool2d / Linear / LayerNorm / softmax call sites cited
 * above).  Every contraction of the backward pass runs on the forward tcgen05 kernels: dgrad of a stride-1 3x3 conv is
 * sblk_conv2d_igemm_fwd with the flipped, transposed filter (stride 2: over the zero-stuffed gradient), wgrad and the
 * Linear backward are sblk_gemm_fmt_fwd over K-major operands produced by sblk_transpose16 / sblk_im2col_t.  Gradients
 * are bf16 (fp32 for parameters and the encoder's residual stream); saved encoder activations are enc16. */
/* sblk_gemm_fwd with an explicit 16-bit operand format (fp16 = 0: bf16, 1: IEEE fp16) and optional split-K:
 * splits == 1 -> out_16 and/or out_f32 [M,N]; splits > 1 -> out_f32 is [splits][M,N] raw partials ((K/64) % splits == 0). */
int sblk_gemm_fmt_fwd(const void* a, const void* w, const float* bias, const void* residual_16, void* out_16,
                      float* out_f32, int M, int N, int K, int relu, int splits, int fp16, void* stream);
/* out[c][r] = in[r][c] for 16-bit elements: in [R, C] (row pitch ld_in), out [C, ld_out], columns R..ld_out-1 zero
 * (K padding of the wgrad GEMMs).  convert = 1 re-rounds IEEE fp16 input to bf16.  C, ld_in, ld_out % 8 == 0. */
int sblk_transpose16(const void* in, void* out, long long R, int C, long long ld_in, long long ld_out, int convert,
                     void* stream);
/* Transposed im2col of NHWC bf16 [F,H,W,C] for an R x S / stride / pad conv: out[(r*S + s)*C + c][m] (row pitch ld_out,
 * zero outside the image and for m >= F*P*Q): the K-major B operand of the wgrad GEMM dW = dY^T col.  C % 64 == 0. */
int sblk_im2col_t(const void* x, void* out, int F, int H, int W, int C, int R, int S, int stride, int pad,
                  long long ld_out, void* stream);
/* im2col of the Conv3d stem (x fp32 [N,T,88,88]; k = (dt*7 + r)*7 + s, 245 taps zero-padded to 256):
 * transposed = 0 -> bf16 [N*T*44*44, 256] (A operand of the training-forward GEMM); 1 -> bf16 [256, ld_out] (wgrad). */
int sblk_stem_im2col(const float* x, void* out, int N, int T, int transposed, long long ld_out, void* stream);
/* im2col of the Conv3d stem straight from raw uint8 gray frames x_u8 [N, T_in, H0, W0]:
 * value = lut_bf16[x_u8[n, t, y1 + y, x1 + xm]], xm = flip[n] ? 87 - x : x, with (y1, x1) = crop_yx[n*T_in + t]
 * (or (crop_y0, crop_x0) for every frame when crop_yx == NULL); frames t >= T_in are zero (padding in normalised
 * space); flip may be NULL (no clip mirrored).  Same output layout as sblk_stem_im2col with T = T_out:
 * transposed = 0 -> bf16 [N*T_out*44*44, 256]; 1 -> bf16 [256, ld_out].
 * The crop comes first, in source coordinates; the flip mirrors the 88 x 88 crop (torch.flip(clip, dims=[-1])).
 * Per-frame offsets in crop_yx live in device memory and are not checked here: the kernel clamps each into
 * [0, H0-88] x [0, W0-88], so it never reads outside its frame.  A uniform crop outside the frame is an error.
 * With lut_bf16 = bf16(float32((u / 255. - mean) / std)) the output is bit-identical to sblk_stem_im2col of the clip
 * the reference loader builds on the host.
 * replaces: load_file / ColorNormalize / RandomCrop / HorizontalFlip / frame zero-padding of the training loader
 * + the stem's im2col, SBL/data_gen.py:122-125,276-296, cvtransforms.py:7-48 */
int sblk_stem_im2col_u8(const void* x_u8, const void* lut_bf16, const int* crop_yx, int crop_y0, int crop_x0,
                        const int* flip, void* out, int N, int T_in, int T_out, int H0, int W0, int transposed,
                        long long ld_out, void* stream);
/* Deterministic per-channel reductions over the rows of [M, C] -> out_2C = (first[C], second[C]):
 *   mode 0: a 16-bit -> (sum, sum of squares)        mode 2: a fp32 -> (sum, -)        mode 4: a 16-bit -> (sum, -)
 *   mode 1: BatchNorm backward sums (sum dz, sum dz * xhat): a = dy bf16, b = BN output bf16 (ReLU mask) or NULL,
 *           c = raw conv output bf16, mean / rstd [C].
 * workspace: sblk_colreduce_workspace_floats(C) floats.  fp16: 16-bit inputs of modes 0 / 4 are IEEE fp16. */
long long sblk_colreduce_workspace_floats(int C);
int sblk_colreduce(int mode, const void* a, const void* b, const void* c, const float* mean, const float* rstd,
                   long long M, int C, int fp16, float* workspace, float* out_2C, void* stream);
/* (sum, sumsq)[2C] over `count` rows -> mean, rstd = 1/sqrt(biased var + eps); running stats (may be NULL) updated with
 * `momentum` and the unbiased variance (torch.nn.BatchNorm training semantics). */
int sblk_bn_finalize(const float* sums_2C, float* mean, float* rstd, float* running_mean, float* running_var, int C,
                     float count, float eps, float momentum, void* stream);
/* out = act((x - mean) * rstd * gamma + beta (+ residual)), bf16 [M, C], C % 8 == 0. */
int sblk_bn_apply_fwd(const void* x, const void* residual, const float* mean, const float* rstd, const float* gamma,
                      const float* beta, void* out, long long M, int C, int relu, void* stream);
/* dz = dy * (out_act > 0) (out_act NULL: no ReLU); dx = gamma * rstd * (dz - sum_dz/M - xhat * sum_dzx/M) with sums_2C from
 * sblk_colreduce mode 1; dres (optional) receives dz (gradient of the residual branch). */
int sblk_bn_bwd(const void* dy, const void* out_act, const void* x, const float* mean, const float* rstd,
                const float* gamma, const float* sums_2C, void* dx, void* dres, long long M, int C, void* stream);
/* MaxPool 3x3 / stride 2 / pad 1 over NHWC bf16 (the spatial part of MaxPool3d((1,3,3),(1,2,2),(0,1,1))), and its backward
 * (gradient to the first maximum of every window, PyTorch's tie rule; `pooled` = the forward output; x is a ReLU output:
 * non-positive pixels take no gradient, which the ReLU backward would mask anyway). */
int sblk_maxpool3x3s2_fwd(const void* x, void* out, int F, int H, int W, int C, void* stream);
int sblk_maxpool3x3s2_bwd(const void* x, const void* pooled, const void* dy, void* dx, int F, int H, int W, int C,
                          void* stream);
/* AdaptiveAvgPool2d(1) backward: dx bf16 [F, HW, C] = dfeat fp32 [F, C] / HW. */
int sblk_avgpool_bwd(const float* dfeat, void* dx, long long F, int HW, int C, void* stream);
/* out [F,H,W,C] = 0 except out[f,2p,2q,:] = dy[f,p,q,:] (dgrad of a stride-2 conv = stride-1 conv over this). */
int sblk_zero_stuff2(const void* dy, void* out, int F, int H, int W, int C, int P, int Q, void* stream);
/* dh (bf16, in place) *= (h > 0), h enc16: ReLU backward of the FFN hidden layer. */
int sblk_relu_bwd(void* dh_bf16, const void* h_enc16, long long n, void* stream);
/* LayerNorm(512) backward from the saved pre-normalisation sum z fp32 [M,512]: dz (fp32 and/or bf16) and
 * dgamma_dbeta_1024 = (dgamma[512], dbeta[512]); rows with t >= lengths[m / T] carry no gradient (`*= non_pad_mask`). */
long long sblk_ln_bwd_workspace_floats(void);
int sblk_ln_bwd(const float* dy, const float* z, const float* gamma, const int* lengths, float* dz_f32, void* dz_bf16,
                float* dgamma_dbeta_1024, float* workspace, int M, int T, float eps, void* stream);
/* Training-mode scaled-dot-product self-attention (T <= 64, d_k = 64): qkv enc16 [N*T, 3*H*64], drop = dropout factor
 * mask/(1-p) fp32 [H*N,T,T] or NULL, probs fp32 [H*N,T,T] (written by fwd, read by bwd), out enc16 / dout bf16
 * [N*T, H*64], dqkv bf16 [N*T, 3*H*64].  replaces: ScaledDotProductAttention.forward + autograd, attention.py:72-83 */
int sblk_attention_train_fwd(const void* qkv, const float* drop, float* probs, void* out, const int* lengths, int N,
                             int T, int H, float scale, void* stream);
int sblk_attention_train_bwd(const void* qkv, const float* drop, const float* probs, const void* dout, void* dqkv,
                             const int* lengths, int N, int T, int H, float scale, void* stream);
/* Training-mode scaled-dot-product attention with separate query and key / value sources (Lq <= 64, Lk <= 64, d_k = 64,
 * head h at columns h*64): Q rows (b*Lq + i)*ldq, K / V rows (b*Lk + j)*ldk|ldv (enc16); mask = causal (key j > query
 * i) and / or key lengths klens[b] (NULL = all Lk); drop = dropout factor mask/(1-p) fp32 [H*N, Lq, Lk] applied to the
 * probabilities, or NULL; probs fp32 [H*N, Lq, Lk] (index h*N + b; written by fwd, read by bwd).  fwd: out enc16 rows
 * (b*Lq + i)*ldo.  bwd: dout bf16 rows with pitch lddo -> dq (pitch lddq), dk / dv (rows (b*Lk + j)*lddk|lddv), bf16,
 * every output written (dk / dv may be the two halves of one [N*Lk, 2*H*64] buffer, dq / dk / dv the thirds of one
 * [N*T, 3*H*64] buffer).  (The encoder's packed self-attention stays on sblk_attention_train_*: same values, faster
 * on its shape.)
 * replaces: ScaledDotProductAttention.forward + autograd in DecoderLayer, attention.py:72-83 */
int sblk_xattention_train_fwd(const void* q, const void* k, const void* v, const float* drop, float* probs, void* out,
                              const int* klens, int ldq, int ldk, int ldv, int ldo, int N, int Lq, int Lk, int H,
                              int causal, float scale, void* stream);
int sblk_xattention_train_bwd(const void* q, const void* k, const void* v, const float* drop, const float* probs,
                              const void* dout, void* dq, void* dk, void* dv, const int* klens, int ldq, int ldk,
                              int ldv, int lddo, int lddq, int lddk, int lddv, int N, int Lq, int Lk, int H, int causal,
                              float scale, void* stream);

/* ---- SBL bidirectional decoder glue (SURVEY.md 8f.1) ----------------------------------------------------------------
 * The decoder's projections, FFNs and residual + LayerNorms run on the encoder entry points above (sblk_gemm_fwd,
 * sblk_gemm_splitk_fwd + sblk_sum_layernorm_fwd, sblk_gemm_ln_fwd); these three add what the encoder does not have. */
/* Multi-head attention with separate query and key / value sources (enc16, d_k = 64, head h at columns h*64):
 * Q rows (b*Lq + i)*ldq, K / V rows (b*Lk + j)*ldk|ldv, out rows (b*Lq + i)*ldo; mask = causal (key j > query i) and / or
 * key lengths klens[b] (NULL = all Lk).  Lq <= 32, Lk <= 128.
 * replaces: MultiHeadAttention / ScaledDotProductAttention inside DecoderLayer (decoder.py:388-408, attention.py:32-83)
 * with get_subsequent_mask (utils.py:116-124) — self-attention over the decoded prefix and decoder-encoder attention */
int sblk_xattention_fwd(const void* q, const void* k, const void* v, void* out, const int* klens, int ldq, int ldk,
                        int ldv, int ldo, int N, int Lq, int Lk, int H, int causal, float scale, void* stream);
/* x[n*L + l, :] = emb[tokens[n*ld_tokens + l], :] * scale + pe[l, :] (tokens int64, rows = N*L): fp32 [rows, D] and
 * (optional) enc16.  Token ids outside [0, vocab) are clamped to 0 / vocab - 1 (no error is reported).
 * replaces: tgt_word_emb(ys) * x_logit_scale + positional_encoding(ys), decoder.py:323-327 */
int sblk_embed_pe_fwd(const void* tokens_i64, int ld_tokens, const float* emb, const float* pe, float* out_f32,
                      void* out_16, int rows, int L, int D, int vocab, float scale, void* stream);
/* Synchronous bidirectional mixing of the two directions' hidden states [N, L, D] fp32 (the reference's aliased in-place
 * loops): l2r' = l2r + flip_L(r2l); r2l' = r2l + flip_L(l2r') = 2 r2l + flip_L(l2r).  Writes fp32 + enc16 copies
 * (fp32 pointers 16-byte aligned, enc16 pointers 8-byte aligned; outputs must not alias inputs).
 * replaces: decoder.py:336-346,358-362 */
int sblk_bidir_mix_fwd(const float* l2r, const float* r2l, float* l2r_out, float* r2l_out, void* l2r_16, void* r2l_16,
                       int N, int L, int D, void* stream);
/* Training path: backward of sblk_bidir_mix_fwd, fp32 [N, L, D], from the gradients g_l2r / g_r2l of its outputs:
 * d_l2r = g_l2r + flip_L(g_r2l); d_r2l = g_r2l + (flip_L(g_l2r) + g_r2l) (autograd's order through the aliased loops,
 * bit for bit).  16-byte aligned, no aliasing. */
int sblk_bidir_mix_bwd(const float* g_l2r, const float* g_r2l, float* d_l2r, float* d_r2l, int N, int L, int D,
                       void* stream);
/* Training path: backward of sblk_embed_pe_fwd's embedding term.  demb fp32 [vocab, D] = scale * sum of dx fp32 [rows, D]
 * over the rows whose token id (same layout and clamping as sblk_embed_pe_fwd) is v; overwritten, rows no token
 * selects are zero.  Deterministic: fixed summation order, no atomics.  16-byte aligned dx / demb, D % 4 == 0. */
int sblk_embed_bwd(const void* tokens_i64, int ld_tokens, const float* dx, float* demb, int rows, int L, int D,
                   int vocab, float scale, void* stream);

/* ---- one-shot all-gather of the per-GPU outputs over NVLink / NVSwitch peer memory (one process per GPU) ----------
 * replaces: nn.DataParallel's gather of the replicas' outputs, SBL/train.py:114-115.
 * sblk_p2p_alloc: cudaMalloc + zero a buffer of its own and return its 64-byte CUDA IPC handle (exchange it with the
 * peers through any host channel); sblk_p2p_open maps a peer's handle; sblk_p2p_close unmaps (opened != 0) or frees.
 * sblk_p2p_gather_fwd: ONE kernel stores the local block (bytes_per_rank, multiple of 16) into slot `rank` of every
 * rank's gather buffer [world * bytes_per_rank], publishes flag[rank] = epoch in every rank's flag array
 * (unsigned [world]) and returns only when all `world` flags of its own array carry `epoch` (ncclAllGather completion
 * semantics).  peer_bufs_dev / peer_flags_dev: DEVICE arrays of `world` pointers (entry `rank` = the local buffers);
 * counter_dev: device unsigned, zero-initialised; epoch must increase by one per call on every rank.
 * sblk_set_p2p_timeout_ms: how long a gather kernel waits for its peers (default 30 s; a rank held up by its data
 * loader is not an error) before it records watchdog code 0x0901 and traps; returns the previous value. */
int sblk_p2p_alloc(long long bytes, void** dev_ptr, void* ipc_handle_64);
int sblk_p2p_open(const void* ipc_handle_64, void** dev_ptr);
int sblk_p2p_close(void* dev_ptr, int opened);
int sblk_p2p_gather_fwd(const void* local, const void* const* peer_bufs_dev, const void* const* peer_flags_dev,
                        void* counter_dev, int rank, int world, long long bytes_per_rank, unsigned int epoch,
                        void* stream);
unsigned int sblk_set_p2p_timeout_ms(unsigned int ms);

#ifdef __cplusplus
}
#endif
#endif /* SBLK_H_ */

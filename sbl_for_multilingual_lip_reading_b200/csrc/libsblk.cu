// libsblk.cu — the single translation unit of libsblk.so: C-ABI entry points (include/sblk.h),
// TMA tensor-map construction and kernel launches.  Build: nvcc -gencode arch=compute_100a,code=sm_100a.
#include <cuda_runtime.h>
#include <cuda.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "../../include/sblk.h"
#include "sblk_common.cuh"
#include "sblk_igemm.cuh"
#include "sblk_igemm2.cuh"
#include "sblk_igemm2_block.cuh"
#include "sblk_conv3d.cuh"
#include "sblk_stem_t.cuh"
#include "sblk_flatconv2.cuh"
#include "sblk_aux.cuh"
#include "sblk_attention.cuh"
#include "sblk_gemm_ln.cuh"
#include "sblk_qkv_attn.cuh"
#include "sblk_encoder_stack.cuh"
#include "sblk_train.cuh"
#include "sblk_decoder.cuh"

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};
// Launch settings are per HOST THREAD (nn.DataParallel replicas launch from worker threads, SURVEY.md 8b): a plan that
// captures with PDL on, or sizes grids for a co-running chain, never changes what another thread's launches do.
thread_local int g_pdl = 0;        // != 0: launches carry the programmatic-dependent-launch attribute
thread_local int g_sm_limit = 0;   // > 0: size persistent grids for at most this many SMs (concurrent kernel chains)
thread_local int g_stem_variant = 0;   // 0: transposed stem with the filter in tensor memory; 1: pixel-major stem

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return static_cast<int>(e) > 0 ? static_cast<int>(e) : 1;
}

// ---- driver entry points for tensor-map encoding (no link-time dependency on libcuda) ------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct DeviceState {
  bool ready = false;
  int num_sms = 0;
  unsigned int* wd_host = nullptr;
};

std::mutex g_mu;
DeviceState g_dev[64];
EncodeTiledFn g_encode_tiled = nullptr;
EncodeIm2colFn g_encode_im2col = nullptr;
int g_driver_version = 0;

template <typename K>
int set_smem(K kernel, int bytes) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
  return 0;
}

int ensure_init(int* num_sms_out) {
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  if (dev < 0 || dev >= 64) return fail(-1, "device ordinal %d out of range", dev);
  std::lock_guard<std::mutex> lk(g_mu);
  DeviceState& st = g_dev[dev];
  if (!st.ready) {
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
    if (prop.major != 10) {
      return fail(-2, "libsblk requires an sm_100a (Blackwell B200) device, found sm_%d%d: no fallback path exists",
                  prop.major, prop.minor);
    }
    st.num_sms = prop.multiProcessorCount;
    if (g_encode_tiled == nullptr) {
      cudaDriverEntryPointQueryResult q;
      void* fn = nullptr;
      e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
      if (e != cudaSuccess || fn == nullptr) return cuda_fail(e, "cudaGetDriverEntryPoint(cuTensorMapEncodeTiled)");
      g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
      fn = nullptr;
      e = cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q);
      if (e != cudaSuccess || fn == nullptr) return cuda_fail(e, "cudaGetDriverEntryPoint(cuTensorMapEncodeIm2col)");
      g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
      cudaDriverGetVersion(&g_driver_version);
    }
    // watchdog word in host-mapped memory: readable even after a trapped kernel killed the context
    unsigned int* wd = nullptr;
    e = cudaHostAlloc(reinterpret_cast<void**>(&wd), sizeof(unsigned int), cudaHostAllocMapped);
    if (e != cudaSuccess) return cuda_fail(e, "cudaHostAlloc(watchdog)");
    *wd = 0u;
    unsigned int* wd_dev = nullptr;
    e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&wd_dev), wd, 0);
    if (e != cudaSuccess) return cuda_fail(e, "cudaHostGetDevicePointer(watchdog)");
    e = cudaMemcpyToSymbol(sblk::g_sblk_watchdog_ptr, &wd_dev, sizeof(wd_dev));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyToSymbol(watchdog)");
    st.wd_host = wd;
    int rc;
    if ((rc = set_smem(sblk::igemm_kernel<64, true>, sblk::IgemmCfg<64>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm_kernel<128, true>, sblk::IgemmCfg<128>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm_kernel<256, true>, sblk::IgemmCfg<256>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm2_kernel<128, true>, sblk::Igemm2Cfg<128>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm2_kernel<256, true>, sblk::Igemm2Cfg<256>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm2_kernel<128, true, true>, sblk::Igemm2Cfg<128, true>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm2_block_kernel, sblk::Igemm2Cfg<256>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm_kernel<64, false>, sblk::IgemmCfg<64>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm_kernel<128, false>, sblk::IgemmCfg<128>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::igemm_kernel<256, false>, sblk::IgemmCfg<256>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::conv3d_bn_relu_pool_kernel, sblk::c3d::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::stem_t_kernel<0>, sblk::stt::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::stem_t_kernel<1>, sblk::stt::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::stem_t_kernel<2>, sblk::stt::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::flatconv2_kernel<1>, sblk::Fc2Cfg<1>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::flatconv2_kernel<2>, sblk::Fc2Cfg<2>::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::gemm_ln512_kernel, sblk::gln::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::qkv_attention_kernel<4>, sblk::qa::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::qkv_attention_kernel<8>, sblk::qa::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::qkv_attention_kernel<16>, sblk::qa::SMEM_BYTES))) return rc;
    if ((rc = set_smem(sblk::attention_kernel<4>, 100 * 1024))) return rc;
    if ((rc = set_smem(sblk::attention_kernel<8>, 100 * 1024))) return rc;
    if ((rc = set_smem(sblk::attention_kernel<16>, 100 * 1024))) return rc;
    if ((rc = set_smem(sblk::attn_train_kernel<false>, 104 * 1024))) return rc;
    if ((rc = set_smem(sblk::attn_train_kernel<true>, 104 * 1024))) return rc;
    if ((rc = set_smem(sblk::xattn_train_kernel<false>, 104 * 1024))) return rc;
    if ((rc = set_smem(sblk::xattn_train_kernel<true>, 104 * 1024))) return rc;
    if ((rc = set_smem(sblk::xattention_kernel, 100 * 1024))) return rc;
    st.ready = true;
  }
  if (num_sms_out != nullptr)
    *num_sms_out = (g_sm_limit > 0 && g_sm_limit < st.num_sms) ? g_sm_limit : st.num_sms;
  return 0;
}

int encode_tiled(CUtensorMap* tm, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                 const cuuint32_t* box, CUtensorMapSwizzle swz) {
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = g_encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank),
                              const_cast<void*>(ptr), dims, strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(-10, "cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
  return 0;
}

// Launch helper: optional programmatic-dependent-launch attribute.
template <typename... KArgs, typename... Args>
int launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl_capable,
           const char* name, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  int nattr = 0;
  if (pdl_capable && g_pdl != 0) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    nattr = 1;
  }
  cfg.attrs = attr;
  cfg.numAttrs = nattr;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
  if (e != cudaSuccess) return cuda_fail(e, name);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return 0;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int pick_block_n(int m_tiles, int N, int num_sms) {
  const int cand[3] = {256, 128, 64};
  for (int i = 0; i < 3; ++i) {
    const int bn = cand[i];
    if (N % bn != 0) continue;
    if (static_cast<long long>(m_tiles) * (N / bn) * 10 >= static_cast<long long>(num_sms) * 9) return bn;
  }
  for (int i = 2; i >= 0; --i)
    if (N % cand[i] == 0) return cand[i];
  return 0;
}

template <bool IM2COL>
int launch_igemm(int bn, const CUtensorMap& tmA, const CUtensorMap& tmB, sblk::IgemmParams p, int num_sms,
                 cudaStream_t stream) {
  const int m_tiles = (p.M + 127) / 128;
  const int tiles = m_tiles * (p.N / bn) * p.splits;
  const int grid = tiles < num_sms ? tiles : num_sms;
  switch (bn) {
    case 64:
      return launch(sblk::igemm_kernel<64, IM2COL>, dim3(grid), dim3(192), sblk::IgemmCfg<64>::SMEM_BYTES, stream,
                    true, "igemm_kernel<64>", tmA, tmB, p);
    case 128:
      return launch(sblk::igemm_kernel<128, IM2COL>, dim3(grid), dim3(192), sblk::IgemmCfg<128>::SMEM_BYTES, stream,
                    true, "igemm_kernel<128>", tmA, tmB, p);
    case 256:
      return launch(sblk::igemm_kernel<256, IM2COL>, dim3(grid), dim3(192), sblk::IgemmCfg<256>::SMEM_BYTES, stream,
                    true, "igemm_kernel<256>", tmA, tmB, p);
    default:
      return fail(-11, "no BLOCK_N for N=%d", p.N);
  }
}

int elementwise_grid(long long work_items, int block, int num_sms) {
  long long g = (work_items + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms) * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace

extern "C" {

int sblk_version(void) { return SBLK_VERSION; }
const char* sblk_last_error(void) { return g_err; }

int sblk_init(void) {
  int sms = 0;
  int rc = ensure_init(&sms);
  if (rc != 0) return rc < 0 ? rc : -rc;
  return sms;
}

unsigned int sblk_watchdog_code(void) {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  std::lock_guard<std::mutex> lk(g_mu);
  return g_dev[dev].wd_host ? *reinterpret_cast<volatile unsigned int*>(g_dev[dev].wd_host) : 0u;
}

int sblk_set_pdl(int enable) {
  const int prev = g_pdl;
  g_pdl = enable ? 1 : 0;
  return prev;
}
int sblk_set_sm_limit(int max_sms) {
  const int prev = g_sm_limit;
  g_sm_limit = max_sms > 0 ? (max_sms & ~1) : 0;   // even: CTA-pair kernels take whole TPCs
  return prev;
}
int sblk_set_stem_variant(int variant) {
  const int prev = g_stem_variant;
  g_stem_variant = variant == 1 ? 1 : 0;
  return prev;
}
long long sblk_launch_count(void) { return g_launches.load(); }

int sblk_pack_conv3d(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
                     float eps, void* wp, float* bias, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!w || !gamma || !beta || !mean || !var || !wp || !bias) return fail(-1, "sblk_pack_conv3d: null pointer");
  return launch(sblk::pack_conv3d_kernel, dim3(80), dim3(256), 0, static_cast<cudaStream_t>(stream), false,
                "pack_conv3d_kernel", w, gamma, beta, mean, var, eps, static_cast<__nv_bfloat16*>(wp), bias);
}

int sblk_pack_conv2d(const float* w, const float* gamma, const float* beta, const float* mean, const float* var,
                     float eps, void* wp, float* bias, int Co, int Ci, int R, int S, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!w || !wp) return fail(-1, "sblk_pack_conv2d: null pointer");
  if (gamma && (!beta || !mean || !var || !bias)) return fail(-1, "sblk_pack_conv2d: incomplete BatchNorm arguments");
  if (Co <= 0 || Ci <= 0 || R <= 0 || S <= 0) return fail(-1, "sblk_pack_conv2d: bad shape");
  const long long total = static_cast<long long>(Co) * Ci * R * S;
  return launch(sblk::pack_conv2d_kernel, dim3(elementwise_grid(total, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "pack_conv2d_kernel", w, gamma, beta, mean, var, eps,
                static_cast<__nv_bfloat16*>(wp), bias, Co, Ci, R, S);
}

static int cast_impl(const float* src, void* dst, long long n, int fp16, void* stream, const char* who) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!src || !dst) return fail(-1, "%s: null pointer", who);
  if (n <= 0 || (n & 3) != 0) return fail(-1, "%s: n=%lld must be a positive multiple of 4", who, n);
  if (!aligned16(src) || (reinterpret_cast<uintptr_t>(dst) & 7u)) return fail(-1, "%s: misaligned", who);
  return launch(sblk::cast_f32_bf16_kernel, dim3(elementwise_grid(n / 4, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "cast_f32_bf16_kernel", src,
                static_cast<__nv_bfloat16*>(dst), n / 4, fp16);
}

int sblk_cast_f32_bf16(const float* src, void* dst, long long n, void* stream) {
  return cast_impl(src, dst, n, 0, stream, "sblk_cast_f32_bf16");
}

int sblk_enc16_format(void) { return SBLK_ENC_FP16 ? 1 : 0; }

int sblk_cast_f32_enc16(const float* src, void* dst, long long n, void* stream) {
  return cast_impl(src, dst, n, SBLK_ENC_FP16 ? 1 : 0, stream, "sblk_cast_f32_enc16");
}

int sblk_l2_prefetch(const void* const* ptrs, const long long* bytes, int n, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!ptrs || !bytes || n <= 0) return fail(-1, "sblk_l2_prefetch: null pointer / no ranges");
  // Measured on B200 (tools/exp/l2_prefetch_check.py and the whole-path graph): prefetch.global.L2 hints are DROPPED when
  // tens of MB are requested in one burst (encoder stack after an L2 flush: cold 240 us, one 296-CTA burst 235 us,
  // throttled hints or demand loads 223 us, warm 221 us), while demand loads running next to the persistent conv kernels
  // slow the whole graph down (818 -> 980 us: their CTAs finish late and the join holds the encoder back).  One hint
  // launch PER RANGE keeps the bursts small (launch gaps let the memory system drain) and costs nothing when a hint
  // is dropped: whole path 820 -> 808 us.
  const long long cap = 2 * sms;
  const long long chunk_lines = (64ll << 20) / 128;   // one hint launch per range (<= 64 MB); smaller bursts only add launches (graph: 808 us per tensor, 816 at 4 MB, 871 at 1 MB)
  for (int i = 0; i < n; ++i) {
    if (!ptrs[i] || bytes[i] <= 0) return fail(-1, "sblk_l2_prefetch: null pointer / empty range %d", i);
    const uintptr_t a = reinterpret_cast<uintptr_t>(ptrs[i]);
    const uintptr_t base = a & ~static_cast<uintptr_t>(127);
    const long long lines = (static_cast<long long>(a - base) + bytes[i] + 127) / 128;
    for (long long l0 = 0; l0 < lines; l0 += chunk_lines) {
      const long long chunk = lines - l0 < chunk_lines ? lines - l0 : chunk_lines;
      long long grid = (chunk + 255) / 256;
      if (grid > cap) grid = cap;
      if (grid < 1) grid = 1;
      if ((rc = launch(sblk::l2_prefetch_kernel, dim3(static_cast<unsigned>(grid)), dim3(256), 0,
                       static_cast<cudaStream_t>(stream), false, "l2_prefetch_kernel",
                       reinterpret_cast<const uint8_t*>(base) + l0 * 128, chunk)))
        return rc;
    }
  }
  return 0;
}

int sblk_gate_wait(void* gate_u32x2, int count, int timeout_us, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!gate_u32x2 || count <= 0 || timeout_us < 0) return fail(-1, "sblk_gate_wait: bad arguments");
  if (reinterpret_cast<uintptr_t>(gate_u32x2) % 8 != 0) return fail(-1, "sblk_gate_wait: gate must be 8-byte aligned");
  return launch(sblk::gate_wait_kernel, dim3(1), dim3(32), 0, static_cast<cudaStream_t>(stream), false,
                "gate_wait_kernel", static_cast<unsigned int*>(gate_u32x2), static_cast<unsigned int>(count),
                static_cast<unsigned long long>(timeout_us) * 1000ull);
}

// ---- peer-memory plumbing for the one-shot output gather (one process per GPU) ------------------------------------
int sblk_p2p_alloc(long long bytes, void** dev_ptr, void* ipc_handle_64) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (bytes <= 0 || !dev_ptr || !ipc_handle_64) return fail(-1, "sblk_p2p_alloc: bad arguments");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, static_cast<size_t>(bytes));   // a whole allocation of its own: IPC handles map bases
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(p2p buffer)");
  e = cudaMemset(p, 0, static_cast<size_t>(bytes));
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemset(p2p buffer)");
  cudaIpcMemHandle_t h;
  e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return cuda_fail(e, "cudaIpcGetMemHandle"); }
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(ipc_handle_64, &h, 64);
  *dev_ptr = p;
  return 0;
}

int sblk_p2p_open(const void* ipc_handle_64, void** dev_ptr) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!ipc_handle_64 || !dev_ptr) return fail(-1, "sblk_p2p_open: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle_64, 64);
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return cuda_fail(e, "cudaIpcOpenMemHandle");
  *dev_ptr = p;
  return 0;
}

int sblk_p2p_close(void* dev_ptr, int opened) {
  if (!dev_ptr) return 0;
  cudaError_t e = opened ? cudaIpcCloseMemHandle(dev_ptr) : cudaFree(dev_ptr);
  return e == cudaSuccess ? 0 : cuda_fail(e, "sblk_p2p_close");
}

// how long a gather kernel waits for its peers before it gives up (process-wide; an atomic, read at every launch)
static std::atomic<unsigned int> g_p2p_timeout_ms{30000u};

unsigned int sblk_set_p2p_timeout_ms(unsigned int ms) {
  return g_p2p_timeout_ms.exchange(ms == 0 ? 1u : ms, std::memory_order_relaxed);
}

int sblk_p2p_gather_fwd(const void* local, const void* const* peer_bufs_dev, const void* const* peer_flags_dev,
                        void* counter_dev, int rank, int world, long long bytes_per_rank, unsigned int epoch,
                        void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!local || !peer_bufs_dev || !peer_flags_dev || !counter_dev) return fail(-1, "sblk_p2p_gather_fwd: null pointer");
  if (world < 1 || world > 64 || rank < 0 || rank >= world) return fail(-1, "sblk_p2p_gather_fwd: bad rank %d / world %d", rank, world);
  if (bytes_per_rank <= 0 || (bytes_per_rank & 15) || !aligned16(local))
    return fail(-1, "sblk_p2p_gather_fwd: block must be a positive multiple of 16 bytes, 16-byte aligned");
  const long long n16 = bytes_per_rank / 16;
  // 64 CTAs of 128 threads (8192 threads x 16 B x `world` stores in flight: enough for NVLink).  Small CTAs on purpose:
  // the gather runs next to the compute graph, whose persistent kernels hold every SM with one big CTA — a 128-thread
  // CTA with 40 registers per thread still fits beside a stem CTA (608 threads x 96 registers), a 256-thread one does not
  // and made the stem's CTAs on 32 SMs start late (2 GPUs: 0.650 -> see DESIGN.md 6 [r2d])
  long long grid = (n16 + 127) / 128;
  if (grid > 64) grid = 64;
  return launch(sblk::p2p_gather_kernel, dim3(static_cast<unsigned>(grid)), dim3(128), 0,
                static_cast<cudaStream_t>(stream), false, "p2p_gather_kernel", static_cast<const uint4*>(local),
                reinterpret_cast<uint4* const*>(const_cast<void* const*>(reinterpret_cast<const void* const*>(peer_bufs_dev))),
                reinterpret_cast<unsigned int* const*>(const_cast<void* const*>(reinterpret_cast<const void* const*>(peer_flags_dev))),
                static_cast<unsigned int*>(counter_dev), rank, world, n16, epoch,
                static_cast<unsigned long long>(g_p2p_timeout_ms.load(std::memory_order_relaxed)) * 1000000ull);
}

long long sblk_prep_clip_elems(int N, int T) {
  using namespace sblk::c3d;
  if (N <= 0 || T <= 0) return -1;
  return (static_cast<long long>(N) * (T + 2 * TPAD) * FRAME_ENTRIES + TAIL_PAD_ENTRIES) * 8;
}

int sblk_prep_clip(const float* x, void* out, int N, int T, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !out) return fail(-1, "sblk_prep_clip: null pointer");
  if (N <= 0 || T <= 0) return fail(-1, "sblk_prep_clip: bad shape N=%d T=%d", N, T);
  if (!aligned16(out)) return fail(-1, "sblk_prep_clip: output must be 16-byte aligned");
  const long long rows = static_cast<long long>(N) * (T + 2 * sblk::c3d::TPAD) * 2 * sblk::c3d::PLANE_ROWS;
  long long grid = (rows + 7) / 8;   // one warp per plane row, 8 warps per CTA
  if (grid > static_cast<long long>(sms) * 8) grid = static_cast<long long>(sms) * 8;
  return launch(sblk::prep_clip_kernel, dim3(static_cast<unsigned>(grid)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "prep_clip_kernel", x, static_cast<uint4*>(out), N, T);
}

int sblk_prep_clip_u8(const void* x_u8, const void* lut_bf16, const int* crop_yx, int crop_y0, int crop_x0, void* out,
                      int N, int T_in, int T_out, int H0, int W0, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x_u8 || !lut_bf16 || !out) return fail(-1, "sblk_prep_clip_u8: null pointer");
  if (N <= 0 || T_in <= 0 || T_out < T_in || H0 < 88 || W0 < 88)
    return fail(-1, "sblk_prep_clip_u8: bad shape N=%d T_in=%d T_out=%d H0=%d W0=%d (T_out >= T_in, frames >= 88x88)", N,
                T_in, T_out, H0, W0);
  if (!crop_yx && (crop_y0 < 0 || crop_x0 < 0 || crop_y0 + 88 > H0 || crop_x0 + 88 > W0))
    return fail(-1, "sblk_prep_clip_u8: crop offset (%d, %d) leaves the %dx%d frame", crop_y0, crop_x0, H0, W0);
  if (!aligned16(out)) return fail(-1, "sblk_prep_clip_u8: output must be 16-byte aligned");
  const long long rows = static_cast<long long>(N) * (T_out + 2 * sblk::c3d::TPAD) * 2 * sblk::c3d::PLANE_ROWS;
  long long grid = (rows + 7) / 8;   // one warp per plane row, 8 warps per CTA
  if (grid > static_cast<long long>(sms) * 8) grid = static_cast<long long>(sms) * 8;
  return launch(sblk::prep_clip_u8_kernel, dim3(static_cast<unsigned>(grid)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "prep_clip_u8_kernel", static_cast<const uint8_t*>(x_u8),
                static_cast<const uint16_t*>(lut_bf16), crop_yx, crop_y0, crop_x0, static_cast<uint4*>(out), N, T_in,
                T_out, H0, W0);
}

// launches the transposed stem (sblk_stem_t.cuh): q carries the input source (x8, or the FUSED sources)
static int launch_stem_t(sblk::StemTParams& q, const void* wp, const float* bias, void* out, int N, int T, int flat_out,
                         int sms, void* stream) {
  const long long steps = static_cast<long long>(N) * ((T + 1) / 2) * sblk::stt::TILES_PER_UNIT;
  if (steps > 0x7fffffffLL / 2) return fail(-1, "sblk stem: batch too large (N=%d T=%d)", N, T);
  q.N = N;
  q.T = T;
  q.wp = static_cast<const __nv_bfloat16*>(wp);
  q.bias = bias;
  q.out = static_cast<__nv_bfloat16*>(out);
  q.flat_out = flat_out ? 1 : 0;
  // every CTA gets an equal-cost contiguous share of the (frame pair, row pair) steps; at least two tiles per CTA
  long long g = steps / 2 < 1 ? 1 : steps / 2;
  if (g > sms) g = sms;
  if (q.x_f32 != nullptr)
    return launch(sblk::stem_t_kernel<1>, dim3(static_cast<unsigned>(g)), dim3(sblk::stt::THREADS_FUSED),
                  sblk::stt::SMEM_BYTES, static_cast<cudaStream_t>(stream), true, "stem_t_kernel<fp32 clip>", q);
  if (q.x_u8 != nullptr)
    return launch(sblk::stem_t_kernel<2>, dim3(static_cast<unsigned>(g)), dim3(sblk::stt::THREADS_FUSED),
                  sblk::stt::SMEM_BYTES, static_cast<cudaStream_t>(stream), true, "stem_t_kernel<uint8 frames>", q);
  return launch(sblk::stem_t_kernel<0>, dim3(static_cast<unsigned>(g)), dim3(sblk::stt::THREADS), sblk::stt::SMEM_BYTES,
                static_cast<cudaStream_t>(stream), true, "stem_t_kernel", q);
}

int sblk_stem_fused_fwd(const float* x_f32, const void* x_u8, const void* lut_bf16, const int* crop_yx, int crop_y0,
                        int crop_x0, const void* wp, const float* bias, void* out, int N, int T_in, int T_out, int H0,
                        int W0, int flat_out, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if ((x_f32 == nullptr) == (x_u8 == nullptr))
    return fail(-1, "sblk_stem_fused_fwd: exactly one of x_f32 / x_u8 must be given");
  if (!wp || !bias || !out) return fail(-1, "sblk_stem_fused_fwd: null pointer");
  if (N <= 0 || T_in <= 0 || T_out < T_in)
    return fail(-1, "sblk_stem_fused_fwd: bad shape N=%d T_in=%d T_out=%d", N, T_in, T_out);
  if (!aligned16(wp) || !aligned16(out) || (x_f32 && !aligned16(x_f32)))
    return fail(-1, "sblk_stem_fused_fwd: pointers must be 16-byte aligned");
  sblk::StemTParams q;
  memset(&q, 0, sizeof(q));
  if (x_f32 != nullptr) {
    if (T_out != T_in) return fail(-1, "sblk_stem_fused_fwd: fp32 clips carry their own frame count (T_out == T_in)");
    q.x_f32 = x_f32;
  } else {
    if (!lut_bf16) return fail(-1, "sblk_stem_fused_fwd: null normalisation table");
    if (H0 < 88 || W0 < 88) return fail(-1, "sblk_stem_fused_fwd: frames must be at least 88x88 (got %dx%d)", H0, W0);
    if (!crop_yx && (crop_y0 < 0 || crop_x0 < 0 || crop_y0 + 88 > H0 || crop_x0 + 88 > W0))
      return fail(-1, "sblk_stem_fused_fwd: crop offset (%d, %d) leaves the %dx%d frame", crop_y0, crop_x0, H0, W0);
    q.x_u8 = static_cast<const uint8_t*>(x_u8);
    q.lut_bf16 = static_cast<const uint16_t*>(lut_bf16);
    q.crop_yx = crop_yx;
    q.crop_y0 = crop_y0; q.crop_x0 = crop_x0; q.H0 = H0; q.W0 = W0;
  }
  q.T_in = T_in;
  return launch_stem_t(q, wp, bias, out, N, T_out, flat_out, sms, stream);
}

int sblk_conv3d_bn_relu_pool_fwd(const void* xp, const void* wp, const float* bias, void* out, int N, int T,
                                 int flat_out, void* stream) {
  using namespace sblk::c3d;
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!xp || !wp || !bias || !out) return fail(-1, "sblk_conv3d_bn_relu_pool_fwd: null pointer");
  if (N <= 0 || T <= 0) return fail(-1, "sblk_conv3d_bn_relu_pool_fwd: bad shape N=%d T=%d", N, T);
  if (!aligned16(xp) || !aligned16(wp) || !aligned16(out))
    return fail(-1, "sblk_conv3d_bn_relu_pool_fwd: pointers must be 16-byte aligned");
  if (g_stem_variant == 0) {
    sblk::StemTParams q;
    memset(&q, 0, sizeof(q));
    q.x8 = static_cast<const uint4*>(xp);
    return launch_stem_t(q, wp, bias, out, N, T, flat_out, sms, stream);
  }
  CUtensorMap tmW;
  {
    cuuint64_t dims[2] = {KPAD, COUT};
    cuuint64_t strides[1] = {KPAD * 2};
    cuuint32_t box[2] = {64, COUT};
    if ((rc = encode_tiled(&tmW, wp, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  sblk::Conv3dParams p;
  p.frames = N * T;
  p.T = T;
  p.x8 = static_cast<const uint4*>(xp);
  p.bias = bias;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.flat_out = flat_out ? 1 : 0;
  const int units = p.frames * 2;
  const int grid = units < sms ? units : sms;
  return launch(sblk::conv3d_bn_relu_pool_kernel, dim3(grid), dim3(THREADS), SMEM_BYTES,
                static_cast<cudaStream_t>(stream), true, "conv3d_bn_relu_pool_kernel", tmW, p);
}

long long sblk_flat_rows(int F, int H, int W) {
  if (F <= 0 || H <= 0 || W <= 0) return -1;
  return (static_cast<long long>(F) * (H + 1) + 1) * (W + 2);
}

extern "C++" {
template <int CB>
static int launch_flatconv2(const void* x, const void* wp, const float* bias, const void* residual, void* out,
                            long long rows, int H, int W, int relu, int sms, cudaStream_t stream, int reverse = 0) {
  using Cfg = sblk::Fc2Cfg<CB>;
  constexpr int C = Cfg::C;
  int rc;
  if (2 * (W + 3) + Cfg::TILE_M > Cfg::BOX_PIX)
    return fail(-1, "sblk_flatconv3x3_fwd: W=%d too wide for the %d-row staged run of the C=%d kernel", W,
                Cfg::BOX_PIX, C);
  CUtensorMap tmX, tmW, tmR, tmO;
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(C) * 2};
    cuuint32_t box[2] = {64, Cfg::BOX_PIX};
    if ((rc = encode_tiled(&tmX, x, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    cuuint32_t rbox[2] = {64, Cfg::TILE_M};
    if ((rc = encode_tiled(&tmR, residual ? residual : x, 2, dims, strides, rbox, CU_TENSOR_MAP_SWIZZLE_128B)))
      return rc;
    if ((rc = encode_tiled(&tmO, out, 2, dims, strides, rbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  {
    // packed filter [C][10*C]: tap (r,s) at K columns (3r+s)*C .. ; the trailing CxC identity is not used here
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(10 * C), static_cast<cuuint64_t>(C)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(10 * C) * 2};
    cuuint32_t box[2] = {64, Cfg::BH};
    if ((rc = encode_tiled(&tmW, wp, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  sblk::FlatConv2Params p;
  p.m_total = static_cast<int>(rows);
  p.num_tiles = (p.m_total + 255) / 256;
  p.H = H; p.W = W; p.relu = relu; p.has_res = residual ? 1 : 0;
  p.bias = bias;
  p.reverse = reverse ? 1 : 0;
  const int pairs = p.num_tiles < sms / 2 ? p.num_tiles : sms / 2;
  return launch(sblk::flatconv2_kernel<CB>, dim3(2 * pairs), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, stream, true,
                "flatconv2_kernel", tmX, tmW, tmR, tmO, p);
}
}  // extern "C++"

int sblk_flatconv3x3_fwd(const void* x, const void* wp, const float* bias, const void* residual, void* out, int F,
                         int H, int W, int C, int relu, void* stream) {
  return sblk_flatconv3x3_dir_fwd(x, wp, bias, residual, out, F, H, W, C, relu, 0, stream);
}

int sblk_flatconv3x3_dir_fwd(const void* x, const void* wp, const float* bias, const void* residual, void* out, int F,
                             int H, int W, int C, int relu, int reverse, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !wp || !bias || !out) return fail(-1, "sblk_flatconv3x3_fwd: null pointer");
  if (C != 64 && C != 128)
    return fail(-1, "sblk_flatconv3x3_fwd: only 64 -> 64 and 128 -> 128 channels are implemented (got %d)", C);
  if (F <= 0 || H <= 0 || W <= 0 || W + 2 > 31)
    return fail(-1, "sblk_flatconv3x3_fwd: bad shape F=%d H=%d W=%d (W <= 29)", F, H, W);
  if (!aligned16(x) || !aligned16(wp) || !aligned16(out) || (residual && !aligned16(residual)) || !aligned16(bias))
    return fail(-1, "sblk_flatconv3x3_fwd: pointers must be 16-byte aligned");
  const long long rows = sblk_flat_rows(F, H, W);
  if (rows > 0x7fffffffLL - 1024) return fail(-1, "sblk_flatconv3x3_fwd: problem too large");
  if (C == 128) return launch_flatconv2<2>(x, wp, bias, residual, out, rows, H, W, relu, sms, static_cast<cudaStream_t>(stream), reverse);
  return launch_flatconv2<1>(x, wp, bias, residual, out, rows, H, W, relu, sms, static_cast<cudaStream_t>(stream), reverse);
}

// K-extension of a conv (sblk_conv2d_igemm_ext_fwd): a 1x1 / pad 0 / stride `stride` conv of a second tensor x2
// [F,H2,W2,Cin2] with filter w2 [Cout][Cin2], accumulated into the same output tile
struct ConvExt {
  const void* x2;
  const void* w2;
  int H2, W2, Cin2, stride, row_pitch, frame_pitch;
};

static int conv2d_igemm_impl(const void* x, const void* wp, const float* bias, const void* residual, void* out, int F,
                             int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int relu,
                             int in_row_pitch, int in_frame_pitch, const void* wp_ds, const float* bias_ds,
                             void* out_ds, int flat_out, void* stream, const ConvExt* ext = nullptr);

int sblk_conv2d_igemm_fwd(const void* x, const void* wp, const float* bias, const void* residual, void* out, int F,
                          int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int relu,
                          int in_row_pitch, int in_frame_pitch, void* stream) {
  return conv2d_igemm_impl(x, wp, bias, residual, out, F, H, W, Cin, Cout, R, S, stride, pad, relu, in_row_pitch,
                           in_frame_pitch, nullptr, nullptr, nullptr, 0, stream);
}

// im2col view of a bf16 [F,h,w,c] tensor (pitches in pixels, 0 = dense NHWC) for an r x s / pad pd / stride st conv
static int encode_im2col_map(CUtensorMap* tm, const void* ptr, int F, int c, int w, int h, int row_pitch_px,
                             int frame_pitch_px, int r, int s_, int pd, int st) {
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(c), static_cast<cuuint64_t>(w), static_cast<cuuint64_t>(h),
                        static_cast<cuuint64_t>(F)};
  const cuuint64_t row_pitch = row_pitch_px > 0 ? row_pitch_px : w;
  const cuuint64_t frame_pitch = frame_pitch_px > 0 ? frame_pitch_px : static_cast<cuuint64_t>(h) * w;
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(c) * 2, row_pitch * c * 2, frame_pitch * c * 2};
  int lower[2] = {-pd, -pd};
  int upper[2] = {pd - (s_ - 1), pd - (r - 1)};
  cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(st), static_cast<cuuint32_t>(st), 1};
  CUresult cr = g_encode_im2col(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, lower,
                                upper, 64, 128, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return fail(-10, "cuTensorMapEncodeIm2col failed with CUresult %d", static_cast<int>(cr));
  const unsigned long long tensor_bytes = static_cast<unsigned long long>(F) * frame_pitch * c * 2ull;
  if (g_driver_version <= 13010 && tensor_bytes < 131072ull)   // see conv2d_igemm_impl
    reinterpret_cast<unsigned long long*>(tm)[1] &= ~(1ull << 21);
  return 0;
}

int sblk_conv_block_flag_words(int F, int H, int W, int stride) {
  if (F <= 0 || H <= 0 || W <= 0 || (stride != 1 && stride != 2)) return -1;
  const int P = (H + 2 - 3) / stride + 1, Q = (W + 2 - 3) / stride + 1;
  const int pq = P * Q;
  if (pq > 256) return -1;
  const long long M = static_cast<long long>(F) * pq;
  const int rpt = (256 / pq) * pq;
  return static_cast<int>(2 * ((M + rpt - 1) / rpt));
}

int sblk_conv_block_fwd(const void* x, const void* w1, const float* bias1, const void* w2, const float* bias2,
                        const void* w_ds, void* y1_ws, void* flags_ws, void* out, int F, int H, int W, int Cin, int Cout,
                        int stride, int in_row_pitch, int in_frame_pitch, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !w1 || !bias1 || !w2 || !bias2 || !y1_ws || !out) return fail(-1, "sblk_conv_block_fwd: null pointer");
  if (F <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cin % 64 != 0) return fail(-1, "sblk_conv_block_fwd: bad shape F=%d H=%d W=%d Cin=%d", F, H, W, Cin);
  if (Cout != 256 && Cout != 512) return fail(-1, "sblk_conv_block_fwd: Cout=%d (256 or 512: ResNet layer 3 / layer 4)", Cout);
  if (stride != 1 && stride != 2) return fail(-1, "sblk_conv_block_fwd: stride %d not implemented", stride);
  if ((w_ds != nullptr) != (stride == 2 || Cin != Cout))
    return fail(-1, "sblk_conv_block_fwd: a downsample filter is needed exactly when the block changes shape (stride %d, %d -> %d)", stride, Cin, Cout);
  if (Cout > 256 && !flags_ws) return fail(-1, "sblk_conv_block_fwd: Cout=%d needs the flag workspace (sblk_conv_block_flag_words zeroed uint32)", Cout);
  if (!aligned16(x) || !aligned16(w1) || !aligned16(w2) || (w_ds && !aligned16(w_ds)) || !aligned16(y1_ws) || !aligned16(out) ||
      !aligned16(bias1) || !aligned16(bias2) || (flags_ws && (reinterpret_cast<uintptr_t>(flags_ws) & 3u)))
    return fail(-1, "sblk_conv_block_fwd: pointers must be 16-byte aligned");
  const int P = (H + 2 - 3) / stride + 1, Q = (W + 2 - 3) / stride + 1;
  const int pq = P * Q;
  if (pq > 256) return fail(-1, "sblk_conv_block_fwd: %dx%d output maps do not fit a 256-row pair tile", P, Q);
  const long long M64 = static_cast<long long>(F) * pq;
  if (M64 > 0x7fffffffLL - 256) return fail(-1, "sblk_conv_block_fwd: problem too large");
  sblk::BlockConvParams p;
  p.M = static_cast<int>(M64); p.P = P; p.Q = Q;
  p.N = Cout; p.n_tiles = Cout / 256;
  p.rows_per_tile = (256 / pq) * pq;
  p.num_tiles = (p.M + p.rows_per_tile - 1) / p.rows_per_tile;
  const int units = p.num_tiles * p.n_tiles;
  const int pairs = units < sms / 2 ? units : sms / 2;
  if (pairs < 1 || (units + pairs - 1) / pairs > sblk::BLK_MAX_TILES)
    return fail(-2, "sblk_conv_block_fwd: %d work units on %d CTA pairs: more than %d tiles per pair (launch the convs one by one)",
                units, pairs, sblk::BLK_MAX_TILES);
  p.c1_cblocks = Cin / 64; p.c1_stride = stride; p.c2_cblocks = Cout / 64;
  p.ext_cblocks = w_ds ? Cin / 64 : 0; p.ext_stride = stride;
  p.bias1 = bias1; p.bias2 = bias2;
  p.residual = w_ds ? nullptr : static_cast<const __nv_bfloat16*>(x);
  if (!w_ds && (in_row_pitch > 0 || in_frame_pitch > 0))
    return fail(-1, "sblk_conv_block_fwd: the identity residual needs a dense NHWC block input");
  p.y1 = static_cast<__nv_bfloat16*>(y1_ws); p.out = static_cast<__nv_bfloat16*>(out);
  p.flags = static_cast<unsigned int*>(flags_ws);
  CUtensorMap tmA1, tmB1, tmA2, tmB2, tmA3, tmB3;
  if ((rc = encode_im2col_map(&tmA1, x, F, Cin, W, H, in_row_pitch, in_frame_pitch, 3, 3, 1, stride))) return rc;
  if ((rc = encode_im2col_map(&tmA2, y1_ws, F, Cout, Q, P, 0, 0, 3, 3, 1, 1))) return rc;
  tmA3 = tmA1;
  if (w_ds && (rc = encode_im2col_map(&tmA3, x, F, Cin, W, H, in_row_pitch, in_frame_pitch, 1, 1, 0, stride))) return rc;
  cuuint32_t box[2] = {64, 128};
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(9 * Cin), static_cast<cuuint64_t>(Cout)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(9 * Cin) * 2};
    if ((rc = encode_tiled(&tmB1, w1, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(9 * Cout), static_cast<cuuint64_t>(Cout)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(9 * Cout) * 2};
    if ((rc = encode_tiled(&tmB2, w2, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  tmB3 = tmB2;
  if (w_ds) {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(Cin), static_cast<cuuint64_t>(Cout)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(Cin) * 2};
    if ((rc = encode_tiled(&tmB3, w_ds, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  return launch(sblk::igemm2_block_kernel, dim3(2 * pairs), dim3(sblk::Igemm2Cfg<256>::THREADS),
                sblk::Igemm2Cfg<256>::SMEM_BYTES, static_cast<cudaStream_t>(stream), true, "igemm2_block_kernel", tmA1, tmB1,
                tmA2, tmB2, tmA3, tmB3, p);
}

int sblk_conv2d_igemm_ext_fwd(const void* x, const void* wp, const float* bias, const void* residual, void* out, int F,
                              int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int relu,
                              int in_row_pitch, int in_frame_pitch, const void* x2, const void* w2, int H2, int W2,
                              int Cin2, int stride2, int x2_row_pitch, int x2_frame_pitch, void* stream) {
  if (!x2 || !w2) return fail(-1, "sblk_conv2d_igemm_ext_fwd: null pointer");
  if (!aligned16(x2) || !aligned16(w2)) return fail(-1, "sblk_conv2d_igemm_ext_fwd: pointers must be 16-byte aligned");
  if (Cin2 <= 0 || Cin2 % 64 != 0) return fail(-1, "sblk_conv2d_igemm_ext_fwd: Cin2=%d must be a positive multiple of 64", Cin2);
  if (stride2 != 1 && stride2 != 2) return fail(-1, "sblk_conv2d_igemm_ext_fwd: stride2 %d not implemented", stride2);
  if (H2 <= 0 || W2 <= 0) return fail(-1, "sblk_conv2d_igemm_ext_fwd: bad shape H2=%d W2=%d", H2, W2);
  const ConvExt ext{x2, w2, H2, W2, Cin2, stride2, x2_row_pitch, x2_frame_pitch};
  return conv2d_igemm_impl(x, wp, bias, residual, out, F, H, W, Cin, Cout, R, S, stride, pad, relu, in_row_pitch,
                           in_frame_pitch, nullptr, nullptr, nullptr, 0, stream, &ext);
}

int sblk_conv2d_dual_igemm_fwd(const void* x, const void* wp, const float* bias, const void* wp_ds,
                               const float* bias_ds, void* out, void* out_ds, int F, int H, int W, int Cin, int Cout,
                               int stride, int relu, int in_row_pitch, int in_frame_pitch, int flat_out, void* stream) {
  if (!wp_ds || !bias_ds || !out_ds || !bias) return fail(-1, "sblk_conv2d_dual_igemm_fwd: null pointer");
  if (!aligned16(wp_ds) || !aligned16(bias_ds) || !aligned16(out_ds))
    return fail(-1, "sblk_conv2d_dual_igemm_fwd: pointers must be 16-byte aligned");
  if (Cout % 128 != 0) return fail(-1, "sblk_conv2d_dual_igemm_fwd: Cout=%d must be a multiple of 128", Cout);
  return conv2d_igemm_impl(x, wp, bias, nullptr, out, F, H, W, Cin, Cout, 3, 3, stride, 1, relu, in_row_pitch,
                           in_frame_pitch, wp_ds, bias_ds, out_ds, flat_out, stream);
}

static int conv2d_igemm_impl(const void* x, const void* wp, const float* bias, const void* residual, void* out, int F,
                             int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int relu,
                             int in_row_pitch, int in_frame_pitch, const void* wp_ds, const float* bias_ds,
                             void* out_ds, int flat_out, void* stream, const ConvExt* ext) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !wp || !out) return fail(-1, "sblk_conv2d_igemm_fwd: null pointer");
  if (F <= 0 || H <= 0 || W <= 0) return fail(-1, "sblk_conv2d_igemm_fwd: bad shape F=%d H=%d W=%d", F, H, W);
  if (Cin % 64 != 0 || Cout % 64 != 0 || Cin <= 0 || Cout <= 0)
    return fail(-1, "sblk_conv2d_igemm_fwd: Cin=%d and Cout=%d must be positive multiples of 64", Cin, Cout);
  if (!((R == 3 && S == 3 && pad == 1) || (R == 1 && S == 1 && pad == 0)))
    return fail(-1, "sblk_conv2d_igemm_fwd: only 3x3/pad1 and 1x1/pad0 filters are implemented (got %dx%d pad %d)", R,
                S, pad);
  if (stride != 1 && stride != 2) return fail(-1, "sblk_conv2d_igemm_fwd: stride %d not implemented", stride);
  if (!aligned16(x) || !aligned16(wp) || !aligned16(out) || (residual && !aligned16(residual)) ||
      (bias && !aligned16(bias)))
    return fail(-1, "sblk_conv2d_igemm_fwd: pointers must be 16-byte aligned");
  const int P = (H + 2 * pad - R) / stride + 1;
  const int Q = (W + 2 * pad - S) / stride + 1;
  const long long M64 = static_cast<long long>(F) * P * Q;
  if (M64 > 0x7fffffffLL - 256) return fail(-1, "sblk_conv2d_igemm_fwd: problem too large");
  const int M = static_cast<int>(M64);
  const int Ktot = R * S * Cin;

  CUtensorMap tmA, tmB, tmA2, tmB2;
  // im2col view of a bf16 [F,h,w,c] tensor (pitches in pixels, 0 = dense NHWC) for an r x s / pad pd / stride st conv
  auto encode_im2col = [&](CUtensorMap* tm, const void* ptr, int c, int w, int h, int row_pitch_px, int frame_pitch_px,
                           int r, int s_, int pd, int st) -> int {
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(c), static_cast<cuuint64_t>(w), static_cast<cuuint64_t>(h),
                          static_cast<cuuint64_t>(F)};
    const cuuint64_t row_pitch = row_pitch_px > 0 ? row_pitch_px : w;
    const cuuint64_t frame_pitch = frame_pitch_px > 0 ? frame_pitch_px : static_cast<cuuint64_t>(h) * w;
    cuuint64_t strides[3] = {static_cast<cuuint64_t>(c) * 2, row_pitch * c * 2, frame_pitch * c * 2};
    int lower[2] = {-pd, -pd};
    int upper[2] = {pd - (s_ - 1), pd - (r - 1)};
    cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(st), static_cast<cuuint32_t>(st), 1};
    CUresult cr = g_encode_im2col(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides,
                                  lower, upper, 64 /*channelsPerPixel*/, 128 /*pixelsPerColumn*/, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return fail(-10, "cuTensorMapEncodeIm2col failed with CUresult %d", static_cast<int>(cr));
    // Driver <= 13.1 sets a descriptor bit that breaks im2col loads of tensors smaller than 128 KiB;
    // clear it as NVIDIA's own conv kernels do.
    const unsigned long long tensor_bytes = static_cast<unsigned long long>(F) * frame_pitch * c * 2ull;
    if (g_driver_version <= 13010 && tensor_bytes < 131072ull)
      reinterpret_cast<unsigned long long*>(tm)[1] &= ~(1ull << 21);
    return 0;
  };
  // input pixels may sit in a pitched (e.g. zero-haloed flat) layout
  if ((rc = encode_im2col(&tmA, x, Cin, W, H, in_row_pitch, in_frame_pitch, R, S, pad, stride))) return rc;
  tmA2 = tmA;
  if (ext) {
    if (wp_ds) return fail(-1, "sblk_conv2d_igemm_ext_fwd: the K-extension and the dual head are exclusive");
    if ((ext->H2 - 1) / ext->stride + 1 != P || (ext->W2 - 1) / ext->stride + 1 != Q)
      return fail(-1, "sblk_conv2d_igemm_ext_fwd: the extension's output grid %dx%d does not match the conv's %dx%d",
                  (ext->H2 - 1) / ext->stride + 1, (ext->W2 - 1) / ext->stride + 1, P, Q);
    if (Cout % 128 != 0)
      return fail(-1, "sblk_conv2d_igemm_ext_fwd: needs the CTA-pair kernel (Cout %% 128 == 0)");
    if ((rc = encode_im2col(&tmA2, ext->x2, ext->Cin2, ext->W2, ext->H2, ext->row_pitch, ext->frame_pitch, 1, 1, 0,
                            ext->stride)))
      return rc;
  }
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(Ktot), static_cast<cuuint64_t>(Cout)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(Ktot) * 2};
    const int m_tiles = (M + 127) / 128;
    // CTA-pair kernel (sblk_igemm2.cuh) for every conv with Cout >= 128: half the B bytes per SM
    int bn2 = Cout % 128 == 0 ? ((wp_ds || Cout % 256 != 0) ? 128 : 256) : 0;
    if (bn2 == 256) {
      // small problems (the 8-clip shard of BASELINE configs[2]: 24 pair tiles of 256 x 256 at layer 4 on 74 CTA pairs):
      // 256 x 128 tiles when they still run as one wave — twice the CTAs, half the k-loop time each.  A tile's time is
      // ~ its width, so the choice minimises waves x width; ties keep the wider tile (fewer operand bytes per FLOP).
      // Bit-identical either way: every output element accumulates its K range in the same order.
      const long long pairs_avail = sms / 2 > 0 ? sms / 2 : 1;
      const long long t256 = static_cast<long long>((M + 255) / 256) * (Cout / 256);
      const long long time256 = ((t256 + pairs_avail - 1) / pairs_avail) * 2;
      const long long time128 = (2 * t256 + pairs_avail - 1) / pairs_avail;
      if (time128 < time256) bn2 = 128;
    }
    const int bn = bn2 ? bn2 : pick_block_n(m_tiles, Cout, sms);
    if (flat_out && !bn2) return fail(-1, "sblk_conv2d_dual_igemm_fwd: flat_out needs the CTA-pair kernel (Cout %% 128 == 0)");
    cuuint32_t box[2] = {64, static_cast<cuuint32_t>(bn2 ? bn2 / 2 : bn)};
    if ((rc = encode_tiled(&tmB, wp, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
    sblk::IgemmParams p;
    p.splits = 1; p.split_stride = 0; p.flat_out = flat_out; p.fp16 = 0;
    p.bias2 = bias_ds;
    p.out2_bf16 = static_cast<__nv_bfloat16*>(out_ds);
    if (wp_ds) {
      // fused 1x1 downsample branch: its [Cout][Cin] filter rides along with the centre-tap k-blocks
      cuuint64_t dims2[2] = {static_cast<cuuint64_t>(Cin), static_cast<cuuint64_t>(Cout)};
      cuuint64_t strides2[1] = {static_cast<cuuint64_t>(Cin) * 2};
      if ((rc = encode_tiled(&tmB2, wp_ds, 2, dims2, strides2, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
      p.M = M; p.N = Cout; p.taps_r = R; p.taps_s = S; p.cblocks = Cin / 64; p.P = P; p.Q = Q;
      p.stride = stride; p.pad = pad; p.relu = relu; p.ldo = Cout;
      p.bias = bias; p.residual = nullptr;
      p.out_bf16 = static_cast<__nv_bfloat16*>(out); p.out_f32 = nullptr;
      const int tiles2 = ((M + 255) / 256) * (Cout / 128);
      const int pairs = tiles2 < sms / 2 ? tiles2 : sms / 2;
      return launch(sblk::igemm2_kernel<128, true, true>, dim3(2 * pairs), dim3(sblk::Igemm2Cfg<128, true>::THREADS),
                    sblk::Igemm2Cfg<128, true>::SMEM_BYTES, static_cast<cudaStream_t>(stream), true,
                    "igemm2_kernel<128,dual>", tmA, tmB, tmB2, tmA2, p);
    }
    p.M = M; p.N = Cout; p.taps_r = R; p.taps_s = S; p.cblocks = Cin / 64; p.P = P; p.Q = Q;
    p.stride = stride; p.pad = pad; p.relu = relu; p.ldo = Cout;
    p.bias = bias;
    p.residual = static_cast<const __nv_bfloat16*>(residual);
    p.out_bf16 = static_cast<__nv_bfloat16*>(out);
    p.out_f32 = nullptr;
    tmB2 = tmB;
    if (ext) {
      // the extension's filter [Cout][Cin2] streams through the same B ring (same box) behind the conv's own k-blocks
      cuuint64_t dims2[2] = {static_cast<cuuint64_t>(ext->Cin2), static_cast<cuuint64_t>(Cout)};
      cuuint64_t strides2[1] = {static_cast<cuuint64_t>(ext->Cin2) * 2};
      if ((rc = encode_tiled(&tmB2, ext->w2, 2, dims2, strides2, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
      p.ext_cblocks = ext->Cin2 / 64;
      p.ext_stride = ext->stride;
    }
    if (bn2) {
      const int tiles2 = ((M + 255) / 256) * (Cout / bn2);
      const int pairs = tiles2 < sms / 2 ? tiles2 : sms / 2;
      if (bn2 == 256) {
        return launch(sblk::igemm2_kernel<256, true>, dim3(2 * pairs), dim3(sblk::Igemm2Cfg<256>::THREADS),
                      sblk::Igemm2Cfg<256>::SMEM_BYTES, static_cast<cudaStream_t>(stream), true, "igemm2_kernel<256>",
                      tmA, tmB, tmB2, tmA2, p);
      }
      return launch(sblk::igemm2_kernel<128, true>, dim3(2 * pairs), dim3(sblk::Igemm2Cfg<128>::THREADS), sblk::Igemm2Cfg<128>::SMEM_BYTES,
                    static_cast<cudaStream_t>(stream), true, "igemm2_kernel<128>", tmA, tmB, tmB2, tmA2, p);
    }
    return launch_igemm<true>(bn, tmA, tmB, p, sms, static_cast<cudaStream_t>(stream));
  }
}

// Linear layers: the BLOCK_N that minimises the operand bytes one CTA has to pull through its L2 port,
// rounds * (128 + BLOCK_N) (the path is latency / port bound at the BASELINE token count, not tensor bound).
static int pick_block_n_linear(int m_tiles, int N, int splits, int num_sms) {
  const int cand[3] = {256, 128, 64};
  int best = 0;
  long long best_cost = 0;
  for (int i = 0; i < 3; ++i) {
    const int bn = cand[i];
    if (N % bn != 0) continue;
    const long long tiles = static_cast<long long>(m_tiles) * (N / bn) * splits;
    const long long cost = ((tiles + num_sms - 1) / num_sms) * (128 + bn);
    if (best == 0 || cost < best_cost) { best = bn; best_cost = cost; }
  }
  return best;
}

static int gemm_impl(const void* a, const void* w, const float* bias, const void* residual, void* out_bf16,
                     float* out_f32, int M, int N, int K, int relu, int splits, void* stream, const char* who,
                     int fp16 = SBLK_ENC_FP16 ? 1 : 0) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!a || !w || (!out_bf16 && !out_f32)) return fail(-1, "%s: null pointer", who);
  if (M <= 0 || N <= 0 || K <= 0 || N % 64 != 0 || K % 64 != 0)
    return fail(-1, "%s: M=%d N=%d K=%d unsupported (N and K must be multiples of 64)", who, M, N, K);
  if (splits < 1 || (K / 64) % splits != 0)
    return fail(-1, "%s: splits=%d must divide the %d K-blocks of 64", who, splits, K / 64);
  if (splits > 1 && (out_bf16 || residual || relu || !out_f32))
    return fail(-1, "%s: split-K writes raw fp32 partials only (no bf16 output, residual or ReLU)", who);
  if (!aligned16(a) || !aligned16(w) || (out_bf16 && !aligned16(out_bf16)) || (out_f32 && !aligned16(out_f32)) ||
      (residual && !aligned16(residual)) || (bias && !aligned16(bias)))
    return fail(-1, "%s: pointers must be 16-byte aligned", who);
  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(M)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
    cuuint32_t box[2] = {64, 128};
    if ((rc = encode_tiled(&tmA, a, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  const int m_tiles = (M + 127) / 128;
  const int bn = pick_block_n_linear(m_tiles, N, splits, sms);
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(N)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
    cuuint32_t box[2] = {64, static_cast<cuuint32_t>(bn)};
    if ((rc = encode_tiled(&tmB, w, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  sblk::IgemmParams p;
  p.bias2 = nullptr; p.out2_bf16 = nullptr;
  p.M = M; p.N = N; p.taps_r = 1; p.taps_s = 1; p.cblocks = K / 64; p.P = 1; p.Q = 1;
  p.stride = 1; p.pad = 0; p.relu = relu; p.ldo = N;
  p.bias = bias;
  p.residual = static_cast<const __nv_bfloat16*>(residual);
  p.out_bf16 = static_cast<__nv_bfloat16*>(out_bf16);
  p.out_f32 = out_f32;
  p.splits = splits; p.flat_out = 0; p.fp16 = fp16;
  p.split_stride = static_cast<long long>(M) * N;
  return launch_igemm<false>(bn, tmA, tmB, p, sms, static_cast<cudaStream_t>(stream));
}

int sblk_gemm_fwd(const void* a, const void* w, const float* bias, const void* residual, void* out_bf16,
                  float* out_f32, int M, int N, int K, int relu, void* stream) {
  return gemm_impl(a, w, bias, residual, out_bf16, out_f32, M, N, K, relu, 1, stream, "sblk_gemm_fwd");
}

int sblk_gemm_splitk_plan(int M, int N, int K) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc < 0 ? rc : -rc;
  if (M <= 0 || N <= 0 || K <= 0 || N % 64 != 0 || K % 64 != 0) return fail(-1, "sblk_gemm_splitk_plan: bad shape");
  const int bn = N % 128 == 0 ? 128 : 64;
  const long long base = static_cast<long long>((M + 127) / 128) * (N / bn);
  int splits = 1;
  while (splits < 8 && base * (splits * 2) <= sms && (K / 64) % (splits * 2) == 0 && K / 64 / (splits * 2) >= 2)
    splits *= 2;
  return splits;
}

int sblk_gemm_splitk_fwd(const void* a, const void* w, const float* bias, float* out_partials, int M, int N, int K,
                         int splits, void* stream) {
  return gemm_impl(a, w, bias, nullptr, nullptr, out_partials, M, N, K, 0, splits, stream, "sblk_gemm_splitk_fwd");
}

int sblk_avgpool_scale_fwd(const void* x, const float* scale, float* out_f32, void* out_bf16, int F, int HW, int C,
                           int out16_enc, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || (!out_f32 && !out_bf16)) return fail(-1, "sblk_avgpool_fwd: null pointer");
  if (F <= 0 || HW <= 0 || C <= 0 || (C & 1)) return fail(-1, "sblk_avgpool_fwd: bad shape F=%d HW=%d C=%d", F, HW, C);
  if ((reinterpret_cast<uintptr_t>(x) & 3u) || (scale && (reinterpret_cast<uintptr_t>(scale) & 7u)) ||
      (out_f32 && (reinterpret_cast<uintptr_t>(out_f32) & 7u)) || (reinterpret_cast<uintptr_t>(out_bf16) & 3u))
    return fail(-1, "sblk_avgpool_fwd: misaligned pointer");
  if (C % 8 == 0 && aligned16(x) && (!scale || aligned16(scale)) && (!out_f32 || aligned16(out_f32)) &&
      (!out_bf16 || aligned16(out_bf16))) {
    const long long items8 = static_cast<long long>(F) * (C / 8);
    return launch(sblk::avgpool8_kernel, dim3(elementwise_grid(items8, 256, sms)), dim3(256), 0,
                  static_cast<cudaStream_t>(stream), true, "avgpool8_kernel", static_cast<const uint4*>(x), scale,
                  out_f32, out_bf16, F, HW, C / 8, (out16_enc && SBLK_ENC_FP16) ? 1 : 0);
  }
  const long long items = static_cast<long long>(F) * (C / 2);
  return launch(sblk::avgpool_kernel, dim3(elementwise_grid(items, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "avgpool_kernel", static_cast<const __nv_bfloat16*>(x), scale,
                out_f32, static_cast<__nv_bfloat16*>(out_bf16), F, HW, C, (out16_enc && SBLK_ENC_FP16) ? 1 : 0);
}

int sblk_avgpool_fwd(const void* x, float* out_f32, void* out_bf16, int F, int HW, int C, void* stream) {
  return sblk_avgpool_scale_fwd(x, nullptr, out_f32, out_bf16, F, HW, C, 0, stream);
}

int sblk_sum_layernorm_fwd(const float* x_parts, int nparts, const float* bias, const float* residual,
                           const float* gamma, const float* beta, const float* pe, const int* lengths,
                           float* out_f32, void* out_bf16, int M, int T, int D, float eps, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x_parts || !gamma || !beta || (!out_f32 && !out_bf16)) return fail(-1, "sblk_sum_layernorm_fwd: null pointer");
  if (D != 512) return fail(-1, "sblk_sum_layernorm_fwd: d_model=%d not implemented (only 512)", D);
  if (M <= 0 || T <= 0 || M % T != 0 || nparts < 1)
    return fail(-1, "sblk_sum_layernorm_fwd: bad shape M=%d T=%d nparts=%d", M, T, nparts);
  if (!aligned16(x_parts) || !aligned16(gamma) || !aligned16(beta) || (residual && !aligned16(residual)) ||
      (bias && !aligned16(bias)) || (pe && !aligned16(pe)) || (out_f32 && !aligned16(out_f32)) ||
      (out_bf16 && !aligned16(out_bf16)))
    return fail(-1, "sblk_sum_layernorm_fwd: pointers must be 16-byte aligned");
  sblk::LnParams p;
  p.x = x_parts; p.nparts = nparts; p.part_stride = static_cast<long long>(M) * D; p.bias = bias;
  p.residual = residual; p.gamma = gamma; p.beta = beta; p.pe = pe; p.lengths = lengths;
  p.out_f32 = out_f32; p.out_bf16 = static_cast<sblk::enc16_t*>(out_bf16); p.M = M; p.T = T; p.eps = eps;
  // one warp per row; 4 rows per CTA so that the BASELINE 928 tokens spread over all SMs
  const int rows_per_block = 4;
  int grid = (M + rows_per_block - 1) / rows_per_block;
  if (grid > sms * 16) grid = sms * 16;
  return launch(sblk::add_layernorm512_kernel, dim3(grid), dim3(32 * rows_per_block), 0,
                static_cast<cudaStream_t>(stream), true, "add_layernorm512_kernel", p);
}

int sblk_add_layernorm_fwd(const float* x, const float* residual, const float* gamma, const float* beta,
                           const float* pe, const int* lengths, float* out_f32, void* out_bf16, int M, int T, int D,
                           float eps, void* stream) {
  return sblk_sum_layernorm_fwd(x, 1, nullptr, residual, gamma, beta, pe, lengths, out_f32, out_bf16, M, T, D, eps,
                                stream);
}

int sblk_attention_fwd(const void* qkv, void* out, float* probs, const int* lengths, int N, int T, int H, int d_k,
                       float scale, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!qkv || !out) return fail(-1, "sblk_attention_fwd: null pointer");
  if (d_k != 64) return fail(-1, "sblk_attention_fwd: d_k=%d not implemented (only 64)", d_k);
  if (N <= 0 || T <= 0 || H <= 0) return fail(-1, "sblk_attention_fwd: bad shape N=%d T=%d H=%d", N, T, H);
  if (T > 128) return fail(-1, "sblk_attention_fwd: T=%d > 128 not implemented", T);
  if (!aligned16(qkv)) return fail(-1, "sblk_attention_fwd: qkv must be 16-byte aligned");
  sblk::AttnParams p;
  p.qkv = static_cast<const sblk::enc16_t*>(qkv);
  p.out = static_cast<sblk::enc16_t*>(out);
  p.probs = probs; p.lengths = lengths; p.N = N; p.T = T; p.H = H; p.scale = scale;
  const int pairs = N * H;
  const dim3 grid((pairs + sblk::ATTN_WARPS - 1) / sblk::ATTN_WARPS), block(sblk::ATTN_WARPS * 32);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (T <= 32)
    return launch(sblk::attention_kernel<4>, grid, block, sblk::ATTN_WARPS * 3 * 32 * 128, s, true,
                  "attention_kernel<4>", p);
  if (T <= 64)
    return launch(sblk::attention_kernel<8>, grid, block, sblk::ATTN_WARPS * 3 * 64 * 128, s, true,
                  "attention_kernel<8>", p);
  return launch(sblk::attention_kernel<16>, grid, block, sblk::ATTN_WARPS * 3 * 128 * 128, s, true,
                "attention_kernel<16>", p);
}

int sblk_gemm_ln_fwd(const void* a, const void* w, const float* bias, const float* residual, const float* gamma,
                     const float* beta, const float* pe, const int* lengths, float* out_f32, void* out_bf16, int M,
                     int N, int K, int T, float eps, void* stream) {
  using namespace sblk::gln;
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!a || !w || !gamma || !beta || (!out_f32 && !out_bf16)) return fail(-1, "sblk_gemm_ln_fwd: null pointer");
  if (N != D) return fail(-1, "sblk_gemm_ln_fwd: N=%d not implemented (LayerNorm width must be 512)", N);
  if (M <= 0 || K <= 0 || K % 64 != 0 || T <= 0 || M % T != 0)
    return fail(-1, "sblk_gemm_ln_fwd: bad shape M=%d K=%d T=%d (K %% 64 == 0, M %% T == 0)", M, K, T);
  if (!aligned16(a) || !aligned16(w) || !aligned16(gamma) || !aligned16(beta) || (bias && !aligned16(bias)) ||
      (residual && !aligned16(residual)) || (pe && !aligned16(pe)) || (out_f32 && !aligned16(out_f32)) ||
      (out_bf16 && !aligned16(out_bf16)))
    return fail(-1, "sblk_gemm_ln_fwd: pointers must be 16-byte aligned");
  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(M)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
    cuuint32_t box[2] = {64, BLOCK_M};
    if ((rc = encode_tiled(&tmA, a, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(N)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
    cuuint32_t box[2] = {64, BLOCK_N};
    if ((rc = encode_tiled(&tmB, w, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  sblk::GemmLnParams p;
  p.M = M; p.K = K; p.T = T; p.bias = bias; p.residual = residual; p.gamma = gamma; p.beta = beta; p.pe = pe;
  p.lengths = lengths; p.out_f32 = out_f32; p.out_bf16 = static_cast<sblk::enc16_t*>(out_bf16); p.eps = eps;
  const int m_tiles = (M + BLOCK_M - 1) / BLOCK_M;
  return launch(sblk::gemm_ln512_kernel, dim3(CLUSTER * m_tiles), dim3(THREADS), SMEM_BYTES,
                static_cast<cudaStream_t>(stream), true, "gemm_ln512_kernel", tmA, tmB, p);
}

int sblk_qkv_group_clips(int T) {
  if (T <= 0 || T > 128) return -1;
  const int tp = T <= 32 ? 32 : T <= 64 ? 64 : 128;
  int g = 128 / T;
  const int cap = (sblk::qa::QKV_ROWS - tp) / T + 1;   // key padding of the group's last clip stays inside the tile
  if (g > cap) g = cap;
  return g < 1 ? 1 : g;
}

int sblk_qkv_attention_fwd(const void* x, const void* w_heads, const float* bias_heads, const int* lengths, void* out,
                           int N, int T, int H, int d_k, int K, float scale, void* stream) {
  using namespace sblk::qa;
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !w_heads || !bias_heads || !out) return fail(-1, "sblk_qkv_attention_fwd: null pointer");
  if (d_k != 64) return fail(-1, "sblk_qkv_attention_fwd: d_k=%d not implemented (only 64)", d_k);
  if (N <= 0 || T <= 0 || H <= 0 || K <= 0 || K % 64 != 0)
    return fail(-1, "sblk_qkv_attention_fwd: bad shape N=%d T=%d H=%d K=%d", N, T, H, K);
  if (T > 128) return fail(-1, "sblk_qkv_attention_fwd: T=%d > 128 not implemented", T);
  if (!aligned16(x) || !aligned16(w_heads) || !aligned16(bias_heads) || !aligned16(out))
    return fail(-1, "sblk_qkv_attention_fwd: pointers must be 16-byte aligned");
  const long long M = static_cast<long long>(N) * T;
  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(M)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
    cuuint32_t box[2] = {64, BLOCK_M};
    if ((rc = encode_tiled(&tmA, x, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(H) * BLOCK_N};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
    cuuint32_t box[2] = {64, BLOCK_N};
    if ((rc = encode_tiled(&tmB, w_heads, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  sblk::QkvAttnParams p;
  p.N = N; p.T = T; p.H = H; p.G = sblk_qkv_group_clips(T); p.K = K; p.bias = bias_heads; p.lengths = lengths;
  p.out = static_cast<sblk::enc16_t*>(out); p.scale = scale;
  const dim3 grid((N + p.G - 1) / p.G, H), block(THREADS);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (T <= 32) return launch(sblk::qkv_attention_kernel<4>, grid, block, SMEM_BYTES, s, true, "qkv_attention_kernel<4>", tmA, tmB, p);
  if (T <= 64) return launch(sblk::qkv_attention_kernel<8>, grid, block, SMEM_BYTES, s, true, "qkv_attention_kernel<8>", tmA, tmB, p);
  return launch(sblk::qkv_attention_kernel<16>, grid, block, SMEM_BYTES, s, true, "qkv_attention_kernel<16>", tmA, tmB, p);
}

// ---- whole-encoder-stack kernel -------------------------------------------------------------------------------
extern "C++" {
template <int CL, int NT, bool MC>
static int launch_encoder_stack(const CUtensorMap* tm, const sblk::EncStackParams& p, int groups, cudaStream_t stream) {
  using Cfg = sblk::EncCfg<CL>;
  auto kernel = sblk::encoder_stack_kernel<CL, NT, MC>;
  static std::atomic<int> prepared[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (prepared[dev & 63].load(std::memory_order_acquire) == 0) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(encoder_stack smem)");
    if (CL > 8) {
      e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(NonPortableClusterSizeAllowed)");
    }
    prepared[dev & 63].store(1, std::memory_order_release);
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(groups * CL);
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  int nattr = 1;
  if (g_pdl != 0) {
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    nattr = 2;
  }
  cfg.attrs = attr;
  cfg.numAttrs = nattr;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], tm[6], tm[7], tm[8], p);
  if (e != cudaSuccess) return cuda_fail(e, "encoder_stack_kernel");
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return 0;
}

template <int CL, bool MC>
static int launch_encoder_stack_nt(int T, const CUtensorMap* tm, const sblk::EncStackParams& p, int groups,
                                   cudaStream_t stream) {
  if (T <= 32) return launch_encoder_stack<CL, 4, MC>(tm, p, groups, stream);
  if (T <= 64) return launch_encoder_stack<CL, 8, MC>(tm, p, groups, stream);
  return launch_encoder_stack<CL, 16, MC>(tm, p, groups, stream);
}
}  // extern "C++"

long long sblk_encoder_stack_workspace_bytes(int N, int T, int d_inner) {
  if (N <= 0 || T <= 0 || d_inner <= 0) return -1;
  const long long M = static_cast<long long>(N) * T;
  return M * (512 + 512 + d_inner) * 2;   // x16 | att16 | h16, bf16
}

int sblk_encoder_stack_fwd(const sblk_encoder_stack_args* a, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (a == nullptr) return fail(-1, "sblk_encoder_stack_fwd: null argument block");
  const int N = a->N, T = a->T, L = a->n_layers, d_in = a->d_in, d_inner = a->d_inner;
  if (a->n_head != 8 || a->d_k != 64 || a->d_model != 512)
    return fail(-1, "sblk_encoder_stack_fwd: only n_head=8, d_k=d_v=64, d_model=512 are implemented (got %d, %d, %d)",
                a->n_head, a->d_k, a->d_model);
  if (N <= 0 || T <= 0 || T > 128 || L <= 0 || d_in <= 0 || d_in % 128 != 0 || d_inner <= 0 || d_inner % 1024 != 0)
    return fail(-1, "sblk_encoder_stack_fwd: bad shape N=%d T=%d layers=%d d_in=%d d_inner=%d (T <= 128, d_in %% 128 "
                "== 0, d_inner %% 1024 == 0)", N, T, L, d_in, d_inner);
  const void* ptrs[] = {a->x_in, a->w_in, a->b_in, a->ln_in_gamma, a->ln_in_beta, a->pe, a->w_heads, a->b_heads,
                        a->w_fc, a->b_fc, a->ln1_gamma, a->ln1_beta, a->w_1, a->b_1, a->w_2, a->b_2, a->ln2_gamma,
                        a->ln2_beta, a->out, a->workspace};
  for (const void* q : ptrs) {
    if (q == nullptr) return fail(-1, "sblk_encoder_stack_fwd: null pointer");
    if (!aligned16(q)) return fail(-1, "sblk_encoder_stack_fwd: pointers must be 16-byte aligned");
  }
  // Cluster size: 16 CTAs per clip group stream the least weight bytes per SM, but only 7 clusters of 16 are ever
  // co-resident on a B200 (measured: GPC granularity), so batches with more groups use clusters of 8 (all 8 groups
  // of the BASELINE batch in one wave).  args.cluster_size / args.no_multicast select the variants explicitly.
  const int G = sblk_qkv_group_clips(T);
  const int groups = (N + G - 1) / G;
  const int gpc = a->groups_per_cluster == 2 ? 2 : 1;   // clip groups interleaved per cluster
  const int clusters = (groups + gpc - 1) / gpc;
  int cl = a->cluster_size != 0 ? a->cluster_size : (clusters <= 7 ? 16 : 8);
  const bool mc = a->no_multicast == 0;
  if (cl != 8 && cl != 16) return fail(-1, "sblk_encoder_stack_fwd: cluster_size must be 0 (automatic), 8 or 16");
  if (d_inner % (64 * cl) != 0 || d_inner / cl > (cl == 16 ? 192 : 256))
    return fail(-1, "sblk_encoder_stack_fwd: d_inner=%d not supported by the fused stack (d_inner %% %d == 0, "
                "d_inner / %d <= %d)", d_inner, 64 * cl, cl, cl == 16 ? 192 : 256);
  const long long M = static_cast<long long>(N) * T;
  sblk::enc16_t* ws = static_cast<sblk::enc16_t*>(a->workspace);
  sblk::EncStackParams p;
  p.N = N; p.T = T; p.G = G; p.L = L; p.M = static_cast<int>(M); p.d_in = d_in; p.d_inner = d_inner;
  p.b_in = a->b_in; p.g_in = a->ln_in_gamma; p.be_in = a->ln_in_beta; p.pe = a->pe;
  p.b_heads = a->b_heads; p.b_fc = a->b_fc; p.g1 = a->ln1_gamma; p.be1 = a->ln1_beta;
  p.b_w1 = a->b_1; p.b_w2 = a->b_2; p.g2 = a->ln2_gamma; p.be2 = a->ln2_beta;
  p.lengths = a->lengths; p.out = a->out;
  p.x16 = ws; p.att16 = ws + M * 512; p.h16 = ws + M * 1024;
  p.scale = a->scale; p.eps = a->eps;
  p.dbg = static_cast<unsigned long long*>(a->debug_stamps);
  p.resident = static_cast<unsigned int*>(a->resident_counter);
  p.gpc = gpc;

  CUtensorMap tm[9];
  const cuuint32_t a_rows = mc ? static_cast<cuuint32_t>(128 / cl) : 128u;
  auto enc = [&](CUtensorMap* t, const void* ptr, long long rows, int cols, cuuint32_t box_rows) -> int {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
    cuuint32_t box[2] = {64, box_rows};
    return encode_tiled(t, ptr, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
  };
  const cuuint32_t ns = static_cast<cuuint32_t>(512 / cl), nw = static_cast<cuuint32_t>(d_inner / cl);
  if ((rc = enc(&tm[0], a->x_in, M, d_in, a_rows))) return rc;
  if ((rc = enc(&tm[1], p.x16, M, 512, a_rows))) return rc;
  if ((rc = enc(&tm[2], p.att16, M, 512, a_rows))) return rc;
  if ((rc = enc(&tm[3], p.h16, M, d_inner, a_rows))) return rc;
  if ((rc = enc(&tm[4], a->w_in, 512, d_in, ns))) return rc;
  if ((rc = enc(&tm[5], a->w_heads, static_cast<long long>(L) * 1536, 512, 192))) return rc;
  if ((rc = enc(&tm[6], a->w_fc, static_cast<long long>(L) * 512, 512, ns))) return rc;
  if ((rc = enc(&tm[7], a->w_1, static_cast<long long>(L) * d_inner, 512, nw))) return rc;
  if ((rc = enc(&tm[8], a->w_2, static_cast<long long>(L) * 512, d_inner, ns))) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (cl == 16) {
    return mc ? launch_encoder_stack_nt<16, true>(T, tm, p, clusters, s)
              : launch_encoder_stack_nt<16, false>(T, tm, p, clusters, s);
  }
  return mc ? launch_encoder_stack_nt<8, true>(T, tm, p, clusters, s)
            : launch_encoder_stack_nt<8, false>(T, tm, p, clusters, s);
}


// =====================================================================================================================
// Training path (forward with batch statistics + backward): see include/sblk.h "training" section, sblk_train.cuh
// =====================================================================================================================
int sblk_gemm_fmt_fwd(const void* a, const void* w, const float* bias, const void* residual, void* out_16,
                      float* out_f32, int M, int N, int K, int relu, int splits, int fp16, void* stream) {
  return gemm_impl(a, w, bias, residual, out_16, out_f32, M, N, K, relu, splits, stream, "sblk_gemm_fmt_fwd",
                   fp16 ? 1 : 0);
}

int sblk_transpose16(const void* in, void* out, long long R, int C, long long ld_in, long long ld_out, int convert,
                     void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!in || !out) return fail(-1, "sblk_transpose16: null pointer");
  if (R <= 0 || C <= 0 || ld_in < C || ld_out < R) return fail(-1, "sblk_transpose16: bad shape R=%lld C=%d ld_in=%lld ld_out=%lld", R, C, ld_in, ld_out);
  if ((C & 7) || (ld_in & 7) || (ld_out & 7) || !aligned16(in) || !aligned16(out))
    return fail(-1, "sblk_transpose16: C, ld_in, ld_out must be multiples of 8 and the bases 16-byte aligned");
  const long long tiles = ((ld_out + 63) / 64) * ((C + 63) / 64);
  const long long cap = static_cast<long long>(sms) * 8;
  return launch(sblk::transpose16_kernel, dim3(static_cast<unsigned>(tiles < cap ? tiles : cap)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "transpose16_kernel", static_cast<const uint16_t*>(in),
                static_cast<uint16_t*>(out), R, C, ld_in, ld_out, convert);
}

int sblk_im2col_t(const void* x, void* out, int F, int H, int W, int C, int R, int S, int stride, int pad,
                  long long ld_out, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !out) return fail(-1, "sblk_im2col_t: null pointer");
  if (F <= 0 || H <= 0 || W <= 0 || C <= 0 || C % 64 != 0 || R <= 0 || S <= 0 || stride <= 0 || pad < 0)
    return fail(-1, "sblk_im2col_t: bad shape (C %% 64 == 0)");
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  const long long M = static_cast<long long>(F) * P * Q;
  if (ld_out < M) return fail(-1, "sblk_im2col_t: ld_out=%lld < M=%lld", ld_out, M);
  if ((ld_out & 7) || !aligned16(x) || !aligned16(out)) return fail(-1, "sblk_im2col_t: ld_out must be a multiple of 8 and the bases 16-byte aligned");
  const long long tiles = ((ld_out + 63) / 64) * (C / 64) * R * S;
  const long long cap = static_cast<long long>(sms) * 8;
  return launch(sblk::im2col_t_kernel, dim3(static_cast<unsigned>(tiles < cap ? tiles : cap)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "im2col_t_kernel", static_cast<const uint16_t*>(x),
                static_cast<uint16_t*>(out), F, H, W, C, P, Q, R, S, stride, pad, ld_out);
}

int sblk_stem_im2col(const float* x, void* out, int N, int T, int transposed, long long ld_out, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !out) return fail(-1, "sblk_stem_im2col: null pointer");
  const long long M = static_cast<long long>(N) * T * 44 * 44;
  if (N <= 0 || T <= 0) return fail(-1, "sblk_stem_im2col: bad shape");
  if (transposed && (ld_out < M || (ld_out & 1))) return fail(-1, "sblk_stem_im2col: ld_out must be even and >= M");
  if (!aligned16(out)) return fail(-1, "sblk_stem_im2col: output must be 16-byte aligned");
  const dim3 grid = transposed ? dim3(256, static_cast<unsigned>((ld_out + 1935) / 1936))
                               : dim3(static_cast<unsigned>(static_cast<long long>(N) * T * 44));
  if (transposed && grid.y > 65535u) return fail(-1, "sblk_stem_im2col: too many frames for one launch (%u)", grid.y);
  return launch(sblk::stem_im2col_kernel, grid, dim3(256), 0, static_cast<cudaStream_t>(stream), false,
                "stem_im2col_kernel", x, static_cast<uint16_t*>(out), N, T, transposed, ld_out);
}

int sblk_stem_im2col_u8(const void* x_u8, const void* lut_bf16, const int* crop_yx, int crop_y0, int crop_x0,
                        const int* flip, void* out, int N, int T_in, int T_out, int H0, int W0, int transposed,
                        long long ld_out, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x_u8 || !lut_bf16 || !out) return fail(-1, "sblk_stem_im2col_u8: null pointer");
  if (N <= 0 || T_in <= 0 || T_out < T_in || H0 < 88 || W0 < 88)
    return fail(-1, "sblk_stem_im2col_u8: bad shape N=%d T_in=%d T_out=%d H0=%d W0=%d (T_out >= T_in, frames >= 88x88)",
                N, T_in, T_out, H0, W0);
  if (!crop_yx && (crop_y0 < 0 || crop_x0 < 0 || crop_y0 + 88 > H0 || crop_x0 + 88 > W0))
    return fail(-1, "sblk_stem_im2col_u8: crop offset (%d, %d) leaves the %dx%d frame", crop_y0, crop_x0, H0, W0);
  const long long M = static_cast<long long>(N) * T_out * 44 * 44;
  if (transposed && (ld_out < M || (ld_out & 1))) return fail(-1, "sblk_stem_im2col_u8: ld_out must be even and >= M");
  if (!aligned16(out)) return fail(-1, "sblk_stem_im2col_u8: output must be 16-byte aligned");
  const long long rows = static_cast<long long>(N) * T_out * 44;
  if (!transposed && rows > 0x7fffffffLL) return fail(-1, "sblk_stem_im2col_u8: too many frames for one launch (%lld rows)", rows);
  // transposed: one block per (temporal tap, 1936-column frame slot), the sixth tap group writes the zero rows 245..255
  const dim3 grid = transposed ? dim3(6, static_cast<unsigned>((ld_out + 1935) / 1936)) : dim3(static_cast<unsigned>(rows));
  if (transposed && grid.y > 65535u) return fail(-1, "sblk_stem_im2col_u8: too many frames for one launch (%u)", grid.y);
  sblk::StemU8Src s;
  s.x = static_cast<const uint8_t*>(x_u8);
  s.lut = static_cast<const uint16_t*>(lut_bf16);
  s.crop_yx = crop_yx;
  s.flip = flip;
  s.crop_y0 = crop_y0; s.crop_x0 = crop_x0;
  s.N = N; s.T_in = T_in; s.T = T_out; s.H0 = H0; s.W0 = W0;
  return launch(sblk::stem_im2col_u8_kernel, grid, dim3(256), 0, static_cast<cudaStream_t>(stream), false,
                "stem_im2col_u8_kernel", s, static_cast<uint16_t*>(out), transposed, ld_out);
}

static const int kColReduceBlocks = 592;
long long sblk_colreduce_workspace_floats(int C) { return C > 0 ? static_cast<long long>(kColReduceBlocks) * 2 * C : -1; }

int sblk_colreduce(int mode, const void* a, const void* b, const void* c, const float* mean, const float* rstd,
                   long long M, int C, int fp16, float* workspace, float* out_2C, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!a || !workspace || !out_2C) return fail(-1, "sblk_colreduce: null pointer");
  if (mode != 0 && mode != 1 && mode != 2 && mode != 4) return fail(-1, "sblk_colreduce: unknown mode %d", mode);
  if (mode == 1 && (!c || !mean || !rstd)) return fail(-1, "sblk_colreduce: mode 1 needs x, mean, rstd");
  if (M <= 0 || C <= 0 || C % 8 != 0) return fail(-1, "sblk_colreduce: bad shape M=%lld C=%d (C %% 8 == 0)", M, C);
  const int cols8 = C / 8;
  const int cpb = cols8 < 64 ? cols8 : 64;
  if (256 % cpb != 0 || cols8 % cpb != 0) return fail(-1, "sblk_colreduce: C=%d not supported (C/8 must divide 256 or be a multiple of 64)", C);
  if (!aligned16(a) || (b && !aligned16(b)) || (c && !aligned16(c))) return fail(-1, "sblk_colreduce: pointers must be 16-byte aligned");
  const int rif = 256 / cpb;
  long long grid = (M + rif - 1) / rif;
  const long long cap = sms * 4 < kColReduceBlocks ? sms * 4 : kColReduceBlocks;
  if (grid > cap) grid = cap;
  sblk::ColReduceParams p;
  p.a = a; p.b = b; p.c = c; p.mean = mean; p.rstd = rstd; p.lengths = nullptr; p.part = workspace; p.M = M; p.C = C;
  p.mode = mode; p.fp16 = fp16; p.T = 1; p.eps = 0.0f;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if ((rc = launch(sblk::colreduce_kernel, dim3(static_cast<unsigned>(grid)), dim3(256), 256 * 16 * sizeof(float), s, false,
                   "colreduce_kernel", p)))
    return rc;
  return launch(sblk::colreduce_finish_kernel, dim3((2 * C + 31) / 32), dim3(256), 0, s, false,
                "colreduce_finish_kernel", static_cast<const float*>(workspace), out_2C, static_cast<int>(grid), 2 * C);
}

int sblk_bn_finalize(const float* sums_2C, float* mean, float* rstd, float* running_mean, float* running_var, int C,
                     float count, float eps, float momentum, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!sums_2C || !mean || !rstd || C <= 0 || count <= 0.0f) return fail(-1, "sblk_bn_finalize: bad arguments");
  if ((running_mean == nullptr) != (running_var == nullptr)) return fail(-1, "sblk_bn_finalize: running_mean / running_var must come together");
  return launch(sblk::bn_finalize_kernel, dim3((C + 127) / 128), dim3(128), 0, static_cast<cudaStream_t>(stream), false,
                "bn_finalize_kernel", sums_2C, mean, rstd, running_mean, running_var, C, count, eps, momentum);
}

int sblk_bn_apply_fwd(const void* x, const void* residual, const float* mean, const float* rstd, const float* gamma,
                      const float* beta, void* out, long long M, int C, int relu, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !mean || !rstd || !gamma || !beta || !out) return fail(-1, "sblk_bn_apply_fwd: null pointer");
  if (M <= 0 || C <= 0 || C % 8 != 0) return fail(-1, "sblk_bn_apply_fwd: bad shape M=%lld C=%d (C %% 8 == 0)", M, C);
  if (256 % (C / 8) != 0) return fail(-1, "sblk_bn_apply_fwd: C=%d not supported (C / 8 must divide 256: per-thread constant channels)", C);
  if (!aligned16(x) || !aligned16(out) || (residual && !aligned16(residual))) return fail(-1, "sblk_bn_apply_fwd: pointers must be 16-byte aligned");
  const long long total8 = M * (C / 8);
  return launch(sblk::bn_apply_kernel, dim3(elementwise_grid(total8, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "bn_apply_kernel", static_cast<const uint4*>(x),
                static_cast<const uint4*>(residual), mean, rstd, gamma, beta, static_cast<uint4*>(out), total8, C, relu);
}

int sblk_bn_bwd(const void* dy, const void* out_act, const void* x, const float* mean, const float* rstd,
                const float* gamma, const float* sums_2C, void* dx, void* dres, long long M, int C, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!dy || !x || !mean || !rstd || !gamma || !sums_2C || !dx) return fail(-1, "sblk_bn_bwd: null pointer");
  if (M <= 0 || C <= 0 || C % 8 != 0) return fail(-1, "sblk_bn_bwd: bad shape M=%lld C=%d (C %% 8 == 0)", M, C);
  if (256 % (C / 8) != 0) return fail(-1, "sblk_bn_bwd: C=%d not supported (C / 8 must divide 256: per-thread constant channels)", C);
  if (!aligned16(dy) || !aligned16(x) || !aligned16(dx) || (out_act && !aligned16(out_act)) || (dres && !aligned16(dres)))
    return fail(-1, "sblk_bn_bwd: pointers must be 16-byte aligned");
  const long long total8 = M * (C / 8);
  return launch(sblk::bn_bwd_apply_kernel, dim3(elementwise_grid(total8, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "bn_bwd_apply_kernel", static_cast<const uint4*>(dy),
                static_cast<const uint4*>(out_act), static_cast<const uint4*>(x), mean, rstd, gamma, sums_2C,
                static_cast<uint4*>(dx), static_cast<uint4*>(dres), total8, C, 1.0f / static_cast<float>(M));
}

int sblk_maxpool3x3s2_fwd(const void* x, void* out, int F, int H, int W, int C, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !out || F <= 0 || H <= 0 || W <= 0 || C <= 0 || (C & 1)) return fail(-1, "sblk_maxpool3x3s2_fwd: bad arguments");
  const int P = (H - 1) / 2 + 1, Q = (W - 1) / 2 + 1;
  const long long total = static_cast<long long>(F) * P * Q * (C / 2);
  return launch(sblk::maxpool3x3s2_fwd_kernel, dim3(elementwise_grid(total, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "maxpool3x3s2_fwd_kernel", static_cast<const uint32_t*>(x),
                static_cast<uint32_t*>(out), F, H, W, C / 2, P, Q);
}

int sblk_maxpool3x3s2_bwd(const void* x, const void* pooled, const void* dy, void* dx, int F, int H, int W, int C,
                          void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!x || !pooled || !dy || !dx || F <= 0 || H <= 0 || W <= 0 || C <= 0 || (C & 7)) return fail(-1, "sblk_maxpool3x3s2_bwd: bad arguments (C %% 8 == 0)");
  if (!aligned16(x) || !aligned16(pooled) || !aligned16(dy) || !aligned16(dx)) return fail(-1, "sblk_maxpool3x3s2_bwd: pointers must be 16-byte aligned");
  const int P = (H - 1) / 2 + 1, Q = (W - 1) / 2 + 1;
  const long long total = static_cast<long long>(F) * H * W * (C / 8);
  return launch(sblk::maxpool3x3s2_bwd_kernel, dim3(elementwise_grid(total, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "maxpool3x3s2_bwd_kernel", static_cast<const uint4*>(x),
                static_cast<const uint4*>(pooled), static_cast<const uint4*>(dy), static_cast<uint4*>(dx), F, H, W, C / 8, P, Q);
}

int sblk_avgpool_bwd(const float* dfeat, void* dx, long long F, int HW, int C, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!dfeat || !dx || F <= 0 || HW <= 0 || C <= 0 || (C & 1)) return fail(-1, "sblk_avgpool_bwd: bad arguments");
  const long long total = F * HW * (C / 2);
  return launch(sblk::avgpool_bwd_kernel, dim3(elementwise_grid(total, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "avgpool_bwd_kernel", reinterpret_cast<const float2*>(dfeat),
                static_cast<uint32_t*>(dx), F, HW, C / 2);
}

int sblk_zero_stuff2(const void* dy, void* out, int F, int H, int W, int C, int P, int Q, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!dy || !out || F <= 0 || H <= 0 || W <= 0 || C <= 0 || C % 8 != 0 || P <= 0 || Q <= 0)
    return fail(-1, "sblk_zero_stuff2: bad arguments (C %% 8 == 0)");
  if (2 * (P - 1) >= H || 2 * (Q - 1) >= W) return fail(-1, "sblk_zero_stuff2: P x Q does not fit H x W at stride 2");
  if (!aligned16(dy) || !aligned16(out)) return fail(-1, "sblk_zero_stuff2: pointers must be 16-byte aligned");
  const long long total = static_cast<long long>(F) * H * W * (C / 8);
  return launch(sblk::zero_stuff2_kernel, dim3(elementwise_grid(total, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "zero_stuff2_kernel", static_cast<const uint4*>(dy),
                static_cast<uint4*>(out), F, H, W, C / 8, P, Q);
}

int sblk_relu_bwd(void* dh_bf16, const void* h_enc16, long long n, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!dh_bf16 || !h_enc16 || n <= 0 || (n & 1)) return fail(-1, "sblk_relu_bwd: bad arguments");
  return launch(sblk::relu_bwd_kernel, dim3(elementwise_grid(n / 2, 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "relu_bwd_kernel", static_cast<uint32_t*>(dh_bf16),
                static_cast<const uint32_t*>(h_enc16), n / 2, SBLK_ENC_FP16 ? 1 : 0);
}

long long sblk_ln_bwd_workspace_floats(void) { return static_cast<long long>(kColReduceBlocks) * 1024; }

int sblk_ln_bwd(const float* dy, const float* z, const float* gamma, const int* lengths, float* dz_f32, void* dz_bf16,
                float* dgamma_dbeta_1024, float* workspace, int M, int T, float eps, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!dy || !z || !gamma || !dgamma_dbeta_1024 || !workspace || (!dz_f32 && !dz_bf16)) return fail(-1, "sblk_ln_bwd: null pointer");
  if (M <= 0 || T <= 0 || M % T != 0) return fail(-1, "sblk_ln_bwd: bad shape M=%d T=%d", M, T);
  if (!aligned16(dy) || !aligned16(z) || !aligned16(gamma) || (dz_f32 && !aligned16(dz_f32)) || (dz_bf16 && !aligned16(dz_bf16)))
    return fail(-1, "sblk_ln_bwd: pointers must be 16-byte aligned");
  sblk::LnBwdParams p;
  p.dy = dy; p.z = z; p.gamma = gamma; p.lengths = lengths; p.dz_f32 = dz_f32; p.dz_bf16 = static_cast<uint16_t*>(dz_bf16);
  p.part = workspace; p.M = M; p.T = T; p.eps = eps;
  int grid = (M + 7) / 8;
  const int cap = sms * 2 < kColReduceBlocks ? sms * 2 : kColReduceBlocks;
  if (grid > cap) grid = cap;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if ((rc = launch(sblk::ln_bwd_kernel, dim3(grid), dim3(256), 0, s, false, "ln_bwd_kernel", p))) return rc;
  return launch(sblk::colreduce_finish_kernel, dim3(1024 / 32), dim3(256), 0, s, false, "colreduce_finish_kernel",
                static_cast<const float*>(workspace), dgamma_dbeta_1024, grid, 1024);
}

static int attn_train_impl(bool bwd, const void* qkv, const float* drop, float* probs, void* out, const void* dout,
                           void* dqkv, const int* lengths, int N, int T, int H, float scale, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!qkv || !probs || (!bwd && !out) || (bwd && (!dout || !dqkv))) return fail(-1, "sblk_attention_train: null pointer");
  if (N <= 0 || T <= 0 || T > 64 || H <= 0) return fail(-1, "sblk_attention_train: bad shape N=%d T=%d H=%d (training attention: T <= 64)", N, T, H);
  sblk::AttnTrainParams p;
  p.qkv = static_cast<const uint16_t*>(qkv); p.drop = drop; p.probs = probs; p.out = static_cast<uint16_t*>(out);
  p.dout = static_cast<const uint16_t*>(dout); p.dqkv = static_cast<uint16_t*>(dqkv); p.lengths = lengths;
  p.N = N; p.T = T; p.H = H; p.scale = scale; p.fp16 = SBLK_ENC_FP16 ? 1 : 0;
  const size_t fl = static_cast<size_t>(3) * T * 65 + static_cast<size_t>(T) * (T + 1) +
                    (bwd ? static_cast<size_t>(T) * 65 + static_cast<size_t>(T) * (T + 1) : 0);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bwd)
    return launch(sblk::attn_train_kernel<true>, dim3(N * H), dim3(256), fl * sizeof(float), s, false,
                  "attn_train_kernel<bwd>", p);
  return launch(sblk::attn_train_kernel<false>, dim3(N * H), dim3(256), fl * sizeof(float), s, false,
                "attn_train_kernel<fwd>", p);
}

int sblk_attention_train_fwd(const void* qkv, const float* drop, float* probs, void* out, const int* lengths, int N,
                             int T, int H, float scale, void* stream) {
  return attn_train_impl(false, qkv, drop, probs, out, nullptr, nullptr, lengths, N, T, H, scale, stream);
}

int sblk_attention_train_bwd(const void* qkv, const float* drop, const float* probs, const void* dout, void* dqkv,
                             const int* lengths, int N, int T, int H, float scale, void* stream) {
  return attn_train_impl(true, qkv, drop, const_cast<float*>(probs), nullptr, dout, dqkv, lengths, N, T, H, scale, stream);
}

static int xattn_train_impl(bool bwd, const char* name, sblk::XAttnTrainParams& p, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!p.q || !p.k || !p.v || !p.probs || (!bwd && !p.out) || (bwd && (!p.dout || !p.dq || !p.dk || !p.dv)))
    return fail(-1, "%s: null pointer", name);
  if (p.N <= 0 || p.H <= 0 || p.Lq <= 0 || p.Lq > 64 || p.Lk <= 0 || p.Lk > 64)
    return fail(-1, "%s: bad shape N=%d H=%d Lq=%d Lk=%d (training attention: Lq <= 64, Lk <= 64)", name, p.N, p.H, p.Lq, p.Lk);
  const int hd = p.H * 64;
  if (p.ldq < hd || p.ldk < hd || p.ldv < hd || (!bwd && p.ldo < hd) ||
      (bwd && (p.lddo < hd || p.lddq < hd || p.lddk < hd || p.lddv < hd)))
    return fail(-1, "%s: row pitches must cover H*64 features", name);
  p.causal = p.causal ? 1 : 0;
  p.fp16 = SBLK_ENC_FP16 ? 1 : 0;
  const size_t Lq = p.Lq, Lk = p.Lk;
  const size_t fl = (Lq + 2 * Lk) * 65 + Lq * (Lk + 1) + (bwd ? Lq * 65 + Lq * (Lk + 1) : 0);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bwd)
    return launch(sblk::xattn_train_kernel<true>, dim3(p.N * p.H), dim3(256), fl * sizeof(float), s, false,
                  "xattn_train_kernel<bwd>", p);
  return launch(sblk::xattn_train_kernel<false>, dim3(p.N * p.H), dim3(256), fl * sizeof(float), s, false,
                "xattn_train_kernel<fwd>", p);
}

int sblk_xattention_train_fwd(const void* q, const void* k, const void* v, const float* drop, float* probs, void* out,
                              const int* klens, int ldq, int ldk, int ldv, int ldo, int N, int Lq, int Lk, int H,
                              int causal, float scale, void* stream) {
  sblk::XAttnTrainParams p = {};
  p.q = static_cast<const uint16_t*>(q); p.k = static_cast<const uint16_t*>(k); p.v = static_cast<const uint16_t*>(v);
  p.drop = drop; p.probs = probs; p.out = static_cast<uint16_t*>(out); p.klens = klens;
  p.ldq = ldq; p.ldk = ldk; p.ldv = ldv; p.ldo = ldo;
  p.N = N; p.Lq = Lq; p.Lk = Lk; p.H = H; p.causal = causal; p.scale = scale;
  return xattn_train_impl(false, "sblk_xattention_train_fwd", p, stream);
}

int sblk_xattention_train_bwd(const void* q, const void* k, const void* v, const float* drop, const float* probs,
                              const void* dout, void* dq, void* dk, void* dv, const int* klens, int ldq, int ldk,
                              int ldv, int lddo, int lddq, int lddk, int lddv, int N, int Lq, int Lk, int H, int causal,
                              float scale, void* stream) {
  sblk::XAttnTrainParams p = {};
  p.q = static_cast<const uint16_t*>(q); p.k = static_cast<const uint16_t*>(k); p.v = static_cast<const uint16_t*>(v);
  p.drop = drop; p.probs = const_cast<float*>(probs); p.dout = static_cast<const uint16_t*>(dout);
  p.dq = static_cast<uint16_t*>(dq); p.dk = static_cast<uint16_t*>(dk); p.dv = static_cast<uint16_t*>(dv);
  p.klens = klens; p.ldq = ldq; p.ldk = ldk; p.ldv = ldv; p.lddo = lddo; p.lddq = lddq; p.lddk = lddk; p.lddv = lddv;
  p.N = N; p.Lq = Lq; p.Lk = Lk; p.H = H; p.causal = causal; p.scale = scale;
  return xattn_train_impl(true, "sblk_xattention_train_bwd", p, stream);
}


// =====================================================================================================================
// SBL bidirectional decoder glue (row f.1): see include/sblk.h "decoder" section, sblk_decoder.cuh
// =====================================================================================================================
int sblk_xattention_fwd(const void* q, const void* k, const void* v, void* out, const int* klens, int ldq, int ldk,
                        int ldv, int ldo, int N, int Lq, int Lk, int H, int causal, float scale, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!q || !k || !v || !out) return fail(-1, "sblk_xattention_fwd: null pointer");
  if (N <= 0 || H <= 0 || Lq <= 0 || Lq > 32 || Lk <= 0 || Lk > 128)
    return fail(-1, "sblk_xattention_fwd: bad shape N=%d H=%d Lq=%d Lk=%d (Lq <= 32, Lk <= 128)", N, H, Lq, Lk);
  if (ldq < H * 64 || ldk < H * 64 || ldv < H * 64 || ldo < H * 64) return fail(-1, "sblk_xattention_fwd: row pitches must cover H*64 features");
  sblk::XAttnParams p;
  p.q = static_cast<const uint16_t*>(q); p.k = static_cast<const uint16_t*>(k); p.v = static_cast<const uint16_t*>(v);
  p.out = static_cast<uint16_t*>(out); p.klens = klens; p.ldq = ldq; p.ldk = ldk; p.ldv = ldv; p.ldo = ldo;
  p.N = N; p.Lq = Lq; p.Lk = Lk; p.H = H; p.causal = causal ? 1 : 0; p.scale = scale; p.fp16 = SBLK_ENC_FP16 ? 1 : 0;
  const size_t fl = static_cast<size_t>(Lq + 2 * Lk) * 65 + static_cast<size_t>(Lq) * (Lk + 1);
  return launch(sblk::xattention_kernel, dim3(N * H), dim3(128), fl * sizeof(float), static_cast<cudaStream_t>(stream),
                true, "xattention_kernel", p);
}

int sblk_embed_pe_fwd(const void* tokens_i64, int ld_tokens, const float* emb, const float* pe, float* out_f32,
                      void* out_16, int rows, int L, int D, int vocab, float scale, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!tokens_i64 || !emb || !pe || !out_f32) return fail(-1, "sblk_embed_pe_fwd: null pointer");
  if (rows <= 0 || L <= 0 || rows % L != 0 || D <= 0 || D % 4 != 0 || vocab <= 0 || ld_tokens < L) return fail(-1, "sblk_embed_pe_fwd: bad shape");
  if (!aligned16(emb) || !aligned16(pe) || !aligned16(out_f32) || (out_16 && (reinterpret_cast<uintptr_t>(out_16) & 7u)))
    return fail(-1, "sblk_embed_pe_fwd: misaligned pointer");
  return launch(sblk::embed_pe_kernel, dim3(elementwise_grid(static_cast<long long>(rows) * (D / 4), 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "embed_pe_kernel", static_cast<const long long*>(tokens_i64), ld_tokens, emb,
                pe, out_f32, static_cast<uint16_t*>(out_16), rows, L, D, vocab, scale, SBLK_ENC_FP16 ? 1 : 0);
}

int sblk_bidir_mix_fwd(const float* l2r, const float* r2l, float* l2r_out, float* r2l_out, void* l2r_16, void* r2l_16,
                       int N, int L, int D, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!l2r || !r2l || !l2r_out || !r2l_out || !l2r_16 || !r2l_16) return fail(-1, "sblk_bidir_mix_fwd: null pointer");
  if (N <= 0 || L <= 0 || D <= 0 || D % 4 != 0) return fail(-1, "sblk_bidir_mix_fwd: bad shape");
  if (l2r == l2r_out || r2l == r2l_out || l2r == r2l_out || r2l == l2r_out) return fail(-1, "sblk_bidir_mix_fwd: outputs must not alias inputs");
  if (!aligned16(l2r) || !aligned16(r2l) || !aligned16(l2r_out) || !aligned16(r2l_out)) return fail(-1, "sblk_bidir_mix_fwd: pointers must be 16-byte aligned");
  // the enc16 copies are stored four elements (one uint2) at a time
  if ((reinterpret_cast<uintptr_t>(l2r_16) & 7u) || (reinterpret_cast<uintptr_t>(r2l_16) & 7u))
    return fail(-1, "sblk_bidir_mix_fwd: 16-bit outputs must be 8-byte aligned");
  return launch(sblk::bidir_mix_kernel, dim3(elementwise_grid(static_cast<long long>(N) * L * (D / 4), 256, sms)), dim3(256), 0,
                static_cast<cudaStream_t>(stream), false, "bidir_mix_kernel", l2r, r2l, l2r_out, r2l_out,
                static_cast<uint16_t*>(l2r_16), static_cast<uint16_t*>(r2l_16), N, L, D, SBLK_ENC_FP16 ? 1 : 0);
}

int sblk_bidir_mix_bwd(const float* g_l2r, const float* g_r2l, float* d_l2r, float* d_r2l, int N, int L, int D,
                       void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!g_l2r || !g_r2l || !d_l2r || !d_r2l) return fail(-1, "sblk_bidir_mix_bwd: null pointer");
  if (N <= 0 || L <= 0 || D <= 0 || D % 4 != 0) return fail(-1, "sblk_bidir_mix_bwd: bad shape N=%d L=%d D=%d", N, L, D);
  if (g_l2r == d_l2r || g_l2r == d_r2l || g_r2l == d_l2r || g_r2l == d_r2l || d_l2r == d_r2l)
    return fail(-1, "sblk_bidir_mix_bwd: outputs must not alias inputs or each other");
  if (!aligned16(g_l2r) || !aligned16(g_r2l) || !aligned16(d_l2r) || !aligned16(d_r2l))
    return fail(-1, "sblk_bidir_mix_bwd: pointers must be 16-byte aligned");
  return launch(sblk::bidir_mix_bwd_kernel, dim3(elementwise_grid(static_cast<long long>(N) * L * (D / 4), 256, sms)),
                dim3(256), 0, static_cast<cudaStream_t>(stream), false, "bidir_mix_bwd_kernel", g_l2r, g_r2l, d_l2r, d_r2l,
                N, L, D);
}

int sblk_embed_bwd(const void* tokens_i64, int ld_tokens, const float* dx, float* demb, int rows, int L, int D,
                   int vocab, float scale, void* stream) {
  int sms, rc;
  if ((rc = ensure_init(&sms))) return rc;
  if (!tokens_i64 || !dx || !demb) return fail(-1, "sblk_embed_bwd: null pointer");
  if (rows <= 0 || L <= 0 || rows % L != 0 || D <= 0 || D % 4 != 0 || vocab <= 0 || ld_tokens < L)
    return fail(-1, "sblk_embed_bwd: bad shape rows=%d L=%d D=%d vocab=%d ld_tokens=%d", rows, L, D, vocab, ld_tokens);
  if (!aligned16(dx) || !aligned16(demb)) return fail(-1, "sblk_embed_bwd: pointers must be 16-byte aligned");
  return launch(sblk::embed_bwd_kernel, dim3(vocab, (D / 4 + 31) / 32), dim3(256), 0, static_cast<cudaStream_t>(stream),
                false, "embed_bwd_kernel", static_cast<const long long*>(tokens_i64), ld_tokens, dx, demb, rows, L, D, vocab,
                scale);
}

}  // extern "C"

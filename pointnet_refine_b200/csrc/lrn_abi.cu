// C ABI of the B200-native LineRefineNet forward hot path (see include/lrn_b200.h).
// Host side only orchestrates: it builds TMA tensor maps, carves the caller's workspace and
// enqueues kernels on the caller's stream.  It never allocates device memory and never syncs.
#include "../../include/lrn_b200.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <utility>
#include <vector>

#include "gemm_common.cuh"
#include "gemm_pair_sm100.cuh"
#include "chain_pair_sm100.cuh"
#include "ctx_attn_sm100.cuh"
#include "scene_kernels.cuh"
#include "query_kernels.cuh"
#include "query_small.cuh"
#include "pointwise.cuh"

namespace {

using namespace lrn;

thread_local char g_err[512] = "";

int fail(int status, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return status;
}

#define LRN_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess) return fail(LRN_ERR_CUDA, "%s -> %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

// Returns the status of a call of this library (helper, launch) from the enclosing function unless it is LRN_OK.
#define LRN_TRY(expr)                       \
  do {                                      \
    if (const int st_ = (expr)) return st_; \
  } while (0)

// Declares `dev` (current device ordinal, SM count); off compute capability 10.0 the enclosing call returns
// LRN_ERR_UNSUPPORTED_ARCH.
#define LRN_DEVICE(dev) \
  DeviceInfo dev;       \
  LRN_TRY(device_info(&dev))

// Every kernel of this library is enqueued by launch(); lrn_launch_count() reports how many.
std::atomic<uint64_t> g_launches{0};

template <typename... P, typename... A>
int launch(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, A&&... args) {
  kernel<<<grid, block, smem, s>>>(std::forward<A>(args)...);
  LRN_CUDA(cudaGetLastError());
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return LRN_OK;
}

// launch() with programmatic stream serialization: the kernel may start once the previous kernel of the stream has
// executed griddepcontrol.launch_dependents in every CTA (or completed), and must itself call griddepcontrol.wait
// before it touches memory the previous kernel reads or writes.  With programmatic=false: an ordinary launch.
template <typename... P, typename... A>
int launch_programmatic(bool programmatic, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                        A&&... args) {
  if (!programmatic) return launch(kernel, grid, block, smem, s, std::forward<A>(args)...);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  LRN_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return LRN_OK;
}

// True when any of the pointers is not `align`-byte aligned (align is a power of two; NULL is aligned).
template <typename... T>
bool misaligned(uintptr_t align, T*... p) {
  return ((reinterpret_cast<uintptr_t>(p) & (align - 1)) | ...) != 0;
}

constexpr int kCat = 2048;          // operand row: feat1..feat5 (1984) + gate hidden (64)
constexpr int kFusionK = 1984;
constexpr int kGateK = 64;
constexpr int64_t kDefaultChunkRows = 148 * 128 * 16;  // 303,104 points per wave: 16 tiles of 256 points per CTA pair
                                                        // (measured: 75,776 -> 303,104 points per wave is +3.8 %, flat beyond)
const int kChan[6] = {4, 64, 128, 256, 512, 1024};
const int kCatOff[6] = {0, 0, 64, 192, 448, 960};  // column of feat_k inside the operand row

size_t elem_size(int precision) { return precision == LRN_PREC_BF16 ? 2 : 4; }
// fp32x3 tier: every tensor-core operand row is stored twice as wide, [hi | lo] TF32 halves of the fp32 value
int op_mul(int precision) { return precision == LRN_PREC_FP32X3 ? 2 : 1; }
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------ packed weight blob
struct PackedLayout {
  size_t w1, b1, wg1, bg1;  // fp32: (64,4) (64) (64) (64)
  size_t w[6];              // operand type: w[2..5] = conv2..conv5 (Cout, Cin)
  size_t wfg;               // (1024, 2048): [fusion folded | gate layer 2]
  size_t wp;                // (256, 1024) context_proj
  size_t b[6];              // fp32 biases conv2..conv5
  size_t bf, bg, bp;        // fp32 (1024) (1024) (256)
  size_t total;
};

PackedLayout packed_layout(int precision) {
  PackedLayout L{};
  const size_t es = elem_size(precision);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  L.w1 = take(64 * 4 * 4);
  L.b1 = take(64 * 4);
  L.wg1 = take(64 * 4);
  L.bg1 = take(64 * 4);
  const size_t wm = size_t(op_mul(precision));
  for (int k = 2; k <= 5; ++k) L.w[k] = take(size_t(kChan[k]) * kChan[k - 1] * es * wm);
  L.wfg = take(size_t(1024) * kCat * es * wm);
  L.wp = take(size_t(256) * 1024 * es * wm);
  for (int k = 2; k <= 5; ++k) L.b[k] = take(size_t(kChan[k]) * 4);
  L.bf = take(1024 * 4);
  L.bg = take(1024 * 4);
  L.bp = take(256 * 4);
  L.total = off;
  return L;
}

// ------------------------------------------------------------------ device / driver helpers
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* out) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    LRN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (!p || q != cudaDriverEntryPointSuccess) return fail(LRN_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  *out = fn;
  return LRN_OK;
}

// Every tensor map of the library: `rank` dimensions (innermost first), byte strides of dimensions 1.., box in elements,
// dense element strides, 128B swizzle, 256-byte L2 promotion, no out-of-bounds fill value (zeros).
int encode_tmap(CUtensorMap* m, CUtensorMapDataType dtype, cuuint32_t rank, const void* base, const cuuint64_t* dims,
                const cuuint64_t* strides, const cuuint32_t* box) {
  EncodeTiledFn enc;
  LRN_TRY(get_encode_fn(&enc));
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, dtype, rank, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LRN_ERR_CUDA, "cuTensorMapEncodeTiled%s failed (%d)", rank == 4 ? " (4-D)" : "", int(r));
  return LRN_OK;
}

// K-major 2-D operand: `rows` x `cols` elements, row pitch `ld` elements; box = 128 bytes x box_rows, 128B swizzle.
int make_tmap(CUtensorMap* m, int precision, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  const size_t es = elem_size(precision);
  if (misaligned(16, base) || (ld * es) % 16) return fail(LRN_ERR_MISALIGNED, "tensor map base/pitch");
  const cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  const cuuint64_t strides[1] = {cuuint64_t(ld * es)};
  const cuuint32_t box[2] = {cuuint32_t(128 / es), cuuint32_t(box_rows)};
  return encode_tmap(m, precision != LRN_PREC_BF16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                     base, dims, strides, box);
}

// Tiled operand matrix (bf16): [row tile of 128][column block of 64][128 rows][128 bytes] - every [128 x 64] box that the
// kernels move is one contiguous 16 KB block in global memory (a row-major matrix scatters it as 128 pieces of 128 bytes
// at the row pitch, which caps the write bandwidth of the chain kernel at about half of a streaming copy).
int make_tmap_tiled(CUtensorMap* m, const void* base, int64_t rows, int64_t cols) {
  if (misaligned(1024, base) || cols % 64) return fail(LRN_ERR_MISALIGNED, "tiled tensor map base / columns");
  const cuuint64_t nb = cuuint64_t(cols / 64), nt = cuuint64_t((rows + 127) / 128);
  const cuuint64_t dims[4] = {64, 128, nb, nt};
  const cuuint64_t strides[3] = {128, 16384, nb * 16384};
  const cuuint32_t box[4] = {64, 128, 1, 1};
  return encode_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box);
}

// MN-major sibling of make_tmap: matrix stored (K rows, C cols) row-major, box = 64 cols x 64 rows
int make_tmap_mn(CUtensorMap* m, const void* base, int64_t k_rows, int64_t cols, int64_t ld) {
  if (misaligned(16, base) || (ld * 2) % 16) return fail(LRN_ERR_MISALIGNED, "tensor map base/pitch");
  const cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(k_rows)};
  const cuuint64_t strides[1] = {cuuint64_t(ld * 2)};
  const cuuint32_t box[2] = {64, 64};
  return encode_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box);
}

struct DeviceInfo {
  int device = -1;
  int sms = 0;
  int cc = 0;
};

int device_info(DeviceInfo* out) {
  static thread_local DeviceInfo cache;
  int dev = 0;
  LRN_CUDA(cudaGetDevice(&dev));
  if (cache.device != dev) {
    int major = 0, minor = 0, sms = 0;
    LRN_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    LRN_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
    LRN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cache.device = dev;
    cache.sms = sms;
    cache.cc = major * 10 + minor;
  }
  *out = cache;
  if (cache.cc != 100)
    return fail(LRN_ERR_UNSUPPORTED_ARCH, "device compute capability %d.%d is not 10.0 (sm_100a only, no fallback)",
                cache.cc / 10, cache.cc % 10);
  return LRN_OK;
}

// ------------------------------------------------------------------ GEMM launch
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: `done` remembers (one bit per device ordinal) where a
// kernel has been configured, so a process that drives several GPUs configures every one of them.
template <typename Kern>
int configure_smem(Kern kern, int bytes, std::atomic<uint64_t>& done) {
  int dev = 0;
  LRN_CUDA(cudaGetDevice(&dev));
  const uint64_t bit = uint64_t(1) << (dev & 63);
  if (!(done.load(std::memory_order_acquire) & bit)) {
    LRN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done.fetch_or(bit, std::memory_order_release);
  }
  return LRN_OK;
}

template <int BN, bool TF32, int EPI, int STAGES, bool GENERAL = true, bool STAGED = false, bool MN = false>
int launch_pair_t(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout, const GemmParams& p, int sms,
                  cudaStream_t stream) {
  using L = PairSmem<BN, STAGES, EPI == EPI_FUSION, STAGED>;
  auto kern = gemm_pair_kernel<BN, TF32, EPI, STAGES, GENERAL, STAGED, MN>;
  static std::atomic<uint64_t> configured{0};  // per instantiation
  LRN_TRY(configure_smem(kern, L::kDynamic, configured));
  const int tiles = p.m_tiles * p.n_tiles * std::max(p.k_splits, 1);
  if (tiles <= 0) return LRN_OK;
  const int grid = 2 * std::min(tiles, sms / 2);  // one CTA pair (cluster of 2) per work-item slot
  // the bf16 fusion kernel always follows the chain kernel of its wave (see lrn_encoder_forward)
  return launch_programmatic(EPI == EPI_FUSION && !TF32, kern, grid, kPairThreads, L::kDynamic, stream, ta, tb, tout, p);
}

// How one GEMM is tiled over CTA pairs (cta_group::2, 256-row tiles).
struct GemmPlan {
  int bn;          // output channels per tile
  int b_box_rows;  // weight rows per TMA box (= rows one CTA stages)
  int m_rows;      // points per tile
};

GemmPlan plan_gemm(int64_t N, int epi) {
  GemmPlan g{};
  g.bn = (epi == EPI_FUSION || N % 256 == 0) ? 256 : 128;
  g.b_box_rows = g.bn / 2;
  g.m_rows = 2 * BM;
  return g;
}

// `tout`: tensor map of the bf16 output (box 64 x 128, 128B swizzle) or nullptr -> direct stores.
int launch_gemm(int precision, const GemmPlan& g, int epi, const CUtensorMap& ta, const CUtensorMap& tb,
                const GemmParams& p, int sms, cudaStream_t stream, const CUtensorMap* tout = nullptr) {
  const bool tf32 = precision != LRN_PREC_BF16;
  if (epi == EPI_ACT && !tf32 && !p.out_f32 && tout) {  // bf16 output: staged TMA stores
    return g.bn == 128 ? launch_pair_t<128, false, EPI_ACT, 6, true, true>(ta, tb, *tout, p, sms, stream)
                       : launch_pair_t<256, false, EPI_ACT, 4, true, true>(ta, tb, *tout, p, sms, stream);
  }
  if (epi == EPI_FUSION) {
    // fast variant: no argmax and every warp's 32 points are valid and inside one segment
    const bool fast = !(p.flags & FUSE_ARGMAX) && p.npts % 32 == 0 && p.M % 32 == 0 && p.row0 % 32 == 0;
    if (fast)
      return tf32 ? launch_pair_t<256, true, EPI_FUSION, 5, false>(ta, tb, ta, p, sms, stream)
                  : launch_pair_t<256, false, EPI_FUSION, 5, false>(ta, tb, ta, p, sms, stream);
    return tf32 ? launch_pair_t<256, true, EPI_FUSION, 5, true>(ta, tb, ta, p, sms, stream)
                : launch_pair_t<256, false, EPI_FUSION, 5, true>(ta, tb, ta, p, sms, stream);
  }
  if (g.bn == 128)
    return tf32 ? launch_pair_t<128, true, EPI_ACT, 8>(ta, tb, ta, p, sms, stream)
                : launch_pair_t<128, false, EPI_ACT, 8>(ta, tb, ta, p, sms, stream);
  return tf32 ? launch_pair_t<256, true, EPI_ACT, 6>(ta, tb, ta, p, sms, stream)
              : launch_pair_t<256, false, EPI_ACT, 6>(ta, tb, ta, p, sms, stream);
}

int fold_one(int precision, const float* w, const float* b, const float* g, const float* beta, const float* mean,
             const float* var, float eps, int cout, int cin, void* out_w, int64_t ld, int col0, float* out_b,
             cudaStream_t stream, bool operand = true, int64_t lo_off = 0) {
  const long long total = static_cast<long long>(cout) * cin;
  const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, 4096));
  if (precision != LRN_PREC_BF16)
    return launch(fold_linear_kernel<float>, grid, 256, 0, stream, w, b, g, beta, mean, var, eps, cout, cin,
                  static_cast<float*>(out_w), ld, col0, out_b, operand ? 1 : 0,
                  precision == LRN_PREC_FP32X3 && operand ? lo_off : 0);
  return launch(fold_linear_kernel<__nv_bfloat16>, grid, 256, 0, stream, w, b, g, beta, mean, var, eps, cout, cin,
                static_cast<__nv_bfloat16*>(out_w), ld, col0, out_b, 0, 0);
}

// ------------------------------------------------------------------ optional per-stage timing
struct StageProfile {
  bool on = false;
  std::vector<cudaEvent_t> ev;   // begin/end pairs
  std::vector<int> stage;        // stage id of each pair
  std::vector<cudaEvent_t> pool; // recycled events
};
StageProfile g_prof;

struct StageTimer {  // RAII: brackets the kernels of one stage with events when profiling is on
  cudaStream_t s;
  cudaEvent_t e1 = nullptr;
  StageTimer(int stage, cudaStream_t stream) : s(stream) {
    if (!g_prof.on) return;
    cudaEvent_t e[2];
    for (auto& x : e) {
      if (!g_prof.pool.empty()) { x = g_prof.pool.back(); g_prof.pool.pop_back(); }
      else if (cudaEventCreate(&x) != cudaSuccess) return;
    }
    cudaEventRecord(e[0], s);
    g_prof.ev.push_back(e[0]);
    g_prof.ev.push_back(e[1]);
    g_prof.stage.push_back(stage);
    e1 = e[1];
  }
  ~StageTimer() { if (e1) cudaEventRecord(e1, s); }
};

long long* g_dbg = nullptr;  // lrn_debug_timeline: device buffer for clock64() stamps of the fusion kernel

bool bad_precision(int p) { return p != LRN_PREC_BF16 && p != LRN_PREC_TF32 && p != LRN_PREC_FP32X3; }

struct WorkspaceLayout {
  int64_t chunk;
  size_t cat, fused_pm, keys, total;
};

WorkspaceLayout workspace_layout(int64_t B, int64_t N, int precision, int flags, int64_t chunk_rows) {
  WorkspaceLayout W{};
  const size_t es = elem_size(precision);
  const int64_t P = B * N;
  int64_t chunk = chunk_rows > 0 ? chunk_rows : kDefaultChunkRows;
  chunk = std::min<int64_t>(align_up(size_t(std::max<int64_t>(chunk, 128)), 128), align_up(size_t(P), 128));
  W.chunk = chunk;
  size_t off = 0;
  W.cat = off;
  off = align_up(off + size_t(chunk) * kCat * es * op_mul(precision), 1024);
  W.fused_pm = off;
  if (flags & LRN_OUT_MEMORY) off = align_up(off + size_t(chunk) * 1024 * es * op_mul(precision), 1024);
  W.keys = off;
  if (flags & LRN_OUT_ARGMAX) off = align_up(off + size_t(B) * 1024 * 8, 1024);
  W.total = off;
  return W;
}

}  // namespace

// ======================================================================== exported C ABI
extern "C" {

int lrn_abi_version(void) { return LRN_ABI_VERSION; }

const char* lrn_status_string(int status) {
  switch (status) {
    case LRN_OK: return "ok";
    case LRN_ERR_BAD_SHAPE: return "bad shape";
    case LRN_ERR_MISALIGNED: return "misaligned pointer";
    case LRN_ERR_UNSUPPORTED_ARCH: return "unsupported architecture (sm_100a only)";
    case LRN_ERR_CUDA: return "CUDA error";
    case LRN_ERR_WORKSPACE: return "workspace too small";
    case LRN_ERR_BAD_ARG: return "bad argument";
  }
  return "unknown status";
}

const char* lrn_last_error(void) { return g_err; }

size_t lrn_launch_count(void) { return size_t(g_launches.load(std::memory_order_relaxed)); }

int lrn_device_check(void) {
  DeviceInfo d;
  return device_info(&d);
}

size_t lrn_encoder_packed_bytes(int precision) {
  if (bad_precision(precision)) return 0;
  return packed_layout(precision).total;
}

int lrn_encoder_fold(const lrn_encoder_params* pr, int precision, void* packed, size_t packed_bytes,
                     lrn_stream_t stream) {
  if (!pr || !packed || bad_precision(precision)) return fail(LRN_ERR_BAD_ARG, "null params/packed or bad precision");
  LRN_DEVICE(dev);
  const PackedLayout L = packed_layout(precision);
  if (packed_bytes < L.total) return fail(LRN_ERR_WORKSPACE, "packed buffer %zu < %zu", packed_bytes, L.total);
  if (misaligned(1024, packed)) return fail(LRN_ERR_MISALIGNED, "packed buffer must be 1024-byte aligned");
  for (int k = 0; k < 5; ++k)
    if (!pr->conv_w[k] || !pr->conv_b[k] || !pr->bn_w[k] || !pr->bn_b[k] || !pr->bn_mean[k] || !pr->bn_var[k])
      return fail(LRN_ERR_BAD_ARG, "null conv/bn parameter %d", k + 1);
  if (!pr->fusion_w || !pr->fusion_b || !pr->fusion_bn_w || !pr->fusion_bn_b || !pr->fusion_bn_mean ||
      !pr->fusion_bn_var || !pr->gate0_w || !pr->gate0_b || !pr->gate2_w || !pr->gate2_b)
    return fail(LRN_ERR_BAD_ARG, "null fusion/gate parameter");
  uint8_t* base = static_cast<uint8_t*>(packed);
  const int wm = op_mul(precision);
  // conv1 stays fp32 (FMA kernel); gate layer 1 is copied as is
  LRN_TRY(fold_one(LRN_PREC_TF32, pr->conv_w[0], pr->conv_b[0], pr->bn_w[0], pr->bn_b[0], pr->bn_mean[0], pr->bn_var[0],
                   pr->bn_eps, 64, 4, base + L.w1, 4, 0, reinterpret_cast<float*>(base + L.b1), stream, /*operand=*/false));
  LRN_CUDA(cudaMemcpyAsync(base + L.wg1, pr->gate0_w, 64 * 4, cudaMemcpyDeviceToDevice, stream));
  LRN_CUDA(cudaMemcpyAsync(base + L.bg1, pr->gate0_b, 64 * 4, cudaMemcpyDeviceToDevice, stream));
  for (int k = 2; k <= 5; ++k)
    LRN_TRY(fold_one(precision, pr->conv_w[k - 1], pr->conv_b[k - 1], pr->bn_w[k - 1], pr->bn_b[k - 1], pr->bn_mean[k - 1],
                     pr->bn_var[k - 1], pr->bn_eps, kChan[k], kChan[k - 1], base + L.w[k], kChan[k - 1] * wm, 0,
                     reinterpret_cast<float*>(base + L.b[k]), stream, true, kChan[k - 1]));
  LRN_TRY(fold_one(precision, pr->fusion_w, pr->fusion_b, pr->fusion_bn_w, pr->fusion_bn_b, pr->fusion_bn_mean,
                   pr->fusion_bn_var, pr->bn_eps, 1024, kFusionK, base + L.wfg, kCat * wm, 0,
                   reinterpret_cast<float*>(base + L.bf), stream, true, kCat));
  LRN_TRY(fold_one(precision, pr->gate2_w, pr->gate2_b, nullptr, nullptr, nullptr, nullptr, 0.f, 1024, kGateK,
                   base + L.wfg, kCat * wm, kFusionK, reinterpret_cast<float*>(base + L.bg), stream, true, kCat));
  if (pr->proj_w && pr->proj_b)
    LRN_TRY(fold_one(precision, pr->proj_w, pr->proj_b, nullptr, nullptr, nullptr, nullptr, 0.f, 256, 1024, base + L.wp,
                     1024 * wm, 0, reinterpret_cast<float*>(base + L.bp), stream, true, 1024));
  return LRN_OK;
}

size_t lrn_encoder_workspace_bytes(int64_t B, int64_t N, int precision, int flags, int64_t chunk_rows) {
  if (B <= 0 || N <= 0 || bad_precision(precision)) return 0;
  return workspace_layout(B, N, precision, flags, chunk_rows).total;
}

int lrn_encoder_forward(const void* packed, int precision, const float* context, int64_t B, int64_t N, int flags,
                        float* global_feat, float* fused, int64_t* argmax, void* memory, int64_t chunk_rows,
                        void* workspace, size_t workspace_bytes, lrn_stream_t stream) {
  if (bad_precision(precision)) return fail(LRN_ERR_BAD_ARG, "bad precision %d", precision);
  if ((flags & LRN_OUT_MEMORY_BF16) && (precision != LRN_PREC_BF16 || !(flags & LRN_OUT_MEMORY)))
    return fail(LRN_ERR_BAD_ARG, "LRN_OUT_MEMORY_BF16 needs LRN_OUT_MEMORY and the bf16 tier");
  if (B <= 0 || N <= 0) return fail(LRN_ERR_BAD_SHAPE, "empty input B=%lld N=%lld", (long long)B, (long long)N);
  if (B * N >= (int64_t(1) << 31) - 128) return fail(LRN_ERR_BAD_SHAPE, "B*N = %lld must be < 2^31", (long long)(B * N));
  if (!packed || !context || !workspace) return fail(LRN_ERR_BAD_ARG, "null packed/context/workspace");
  if (!(flags & (LRN_OUT_POOL | LRN_OUT_ARGMAX | LRN_OUT_FUSED | LRN_OUT_MEMORY)))
    return fail(LRN_ERR_BAD_ARG, "no output requested");
  if ((flags & (LRN_OUT_POOL | LRN_OUT_ARGMAX)) && !global_feat) return fail(LRN_ERR_BAD_ARG, "global_feat is null");
  if ((flags & LRN_OUT_ARGMAX) && !argmax) return fail(LRN_ERR_BAD_ARG, "argmax is null");
  if ((flags & LRN_OUT_FUSED) && !fused) return fail(LRN_ERR_BAD_ARG, "fused is null");
  if ((flags & LRN_OUT_MEMORY) && !memory) return fail(LRN_ERR_BAD_ARG, "memory is null");
  if (misaligned(16, context, memory, global_feat) || misaligned(1024, workspace, packed))
    return fail(LRN_ERR_MISALIGNED, "context/memory/global_feat need 16-byte, packed/workspace 1024-byte alignment");
  LRN_DEVICE(dev);

  const bool tf32 = precision != LRN_PREC_BF16;      // fp32 operands on the kind::tf32 tensor-core path
  const bool x3 = precision == LRN_PREC_FP32X3;      // ... as hi / lo halves, three passes per k-block (fp32-class products)
  const int wm = op_mul(precision), kpass = x3 ? 3 : 1;
  const size_t es = elem_size(precision);
  const int bk = int(128 / es);
  const PackedLayout L = packed_layout(precision);
  const WorkspaceLayout W = workspace_layout(B, N, precision, flags, chunk_rows);
  if (workspace_bytes < W.total) return fail(LRN_ERR_WORKSPACE, "workspace %zu < %zu", workspace_bytes, W.total);
  const uint8_t* pk = static_cast<const uint8_t*>(packed);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  void* cat = ws + W.cat;
  void* fused_pm = ws + W.fused_pm;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + W.keys);
  const int64_t P = B * N;

  if (flags & (LRN_OUT_POOL | LRN_OUT_ARGMAX)) LRN_CUDA(cudaMemsetAsync(global_feat, 0, size_t(B) * 2048 * 4, stream));
  if (flags & LRN_OUT_ARGMAX) LRN_CUDA(cudaMemsetAsync(keys, 0, size_t(B) * 1024 * 8, stream));

  // weight tensor maps (B operands)
  CUtensorMap tw[6], twfg, twp;
  GemmPlan plan[6];
  for (int k = 2; k <= 5; ++k) {
    plan[k] = plan_gemm(kChan[k], EPI_ACT);
    LRN_TRY(make_tmap(&tw[k], precision, pk + L.w[k], kChan[k], kChan[k - 1] * wm, kChan[k - 1] * wm, plan[k].b_box_rows));
  }
  const GemmPlan plan_f = plan_gemm(1024, EPI_FUSION), plan_p = plan_gemm(256, EPI_ACT);
  CUtensorMap tw_chain[4];
  if (!tf32) {
    for (int k = 2; k <= 5; ++k) {
      // TMA box = the weight rows ONE CTA of the pair stages per k-block: N / 2 (conv2 and conv5 run as N = 128 MMAs)
      LRN_TRY(make_tmap(&tw_chain[k - 2], precision, pk + L.w[k], kChan[k], kChan[k - 1], kChan[k - 1],
                        (k == 2 || k == 5) ? 64 : 128));
    }
  }
  LRN_TRY(make_tmap(&twfg, precision, pk + L.wfg, 1024, kCat * wm, kCat * wm, plan_f.b_box_rows));
  if (flags & LRN_OUT_MEMORY) LRN_TRY(make_tmap(&twp, precision, pk + L.wp, 256, 1024 * wm, 1024 * wm, plan_p.b_box_rows));

  EmbedWeights ew{reinterpret_cast<const float*>(pk + L.w1), reinterpret_cast<const float*>(pk + L.b1),
                  reinterpret_cast<const float*>(pk + L.wg1), reinterpret_cast<const float*>(pk + L.bg1)};

  for (int64_t r0 = 0; r0 < P; r0 += W.chunk) {
    const int64_t rows = std::min<int64_t>(W.chunk, P - r0);
    auto m_tiles_of = [&](const GemmPlan& g) { return int((rows + g.m_rows - 1) / g.m_rows); };
    CUtensorMap ta, tpm;
    LRN_TRY(make_tmap(&ta, precision, cat, rows, kCat * wm, kCat * wm, BM));

    // bf16 tier: conv1..conv5 + gate layer 1 as ONE fused kernel (activations stay on the SM, the operand matrix is kept
    // in the tiled layout); the tf32 tier runs one kernel per layer on row-major operand rows.
    const bool fused_chain = !tf32;
    const bool tiled = fused_chain;
    if (tiled) LRN_TRY(make_tmap_tiled(&ta, cat, rows, kCat));
    if (fused_chain) {
      static std::atomic<uint64_t> configured{0};
      LRN_TRY(configure_smem(chain_pair_kernel, ChainSmem::kDynamic, configured));
      ChainParams cp{};
      cp.M = int(rows);
      cp.num_tiles = int((rows + 2 * BM - 1) / (2 * BM));
      cp.ctx = reinterpret_cast<const float4*>(context) + r0;
      cp.w1 = ew.w1; cp.b1 = ew.b1; cp.wg1 = ew.wg1; cp.bg1 = ew.bg1;
      cp.b2 = reinterpret_cast<const float*>(pk + L.b[2]);
      cp.b3 = reinterpret_cast<const float*>(pk + L.b[3]);
      cp.b4 = reinterpret_cast<const float*>(pk + L.b[4]);
      cp.b5 = reinterpret_cast<const float*>(pk + L.b[5]);
      cp.cat = cat;
#ifdef LRN_TIMELINE
      static const int dbg_layer = [] { const char* e = getenv("LRN_DBG_LAYER"); return e ? atoi(e) : 0; }();
      cp.dbg = dbg_layer == 4 ? g_dbg : nullptr;
#endif
      StageTimer timer(LRN_STAGE_CONV5, stream);  // reported as stage "conv5"; the other chain stages then read 0
      const int grid = 2 * std::min(cp.num_tiles, dev.sms / 2);
#ifdef LRN_TIMELINE   // tools/l2_ring_probe.py: fusion kernel alone on whatever the operand buffer holds
      const char* skip_chain = getenv("LRN_DBG_SKIP_CHAIN");
      if (!(skip_chain && atoi(skip_chain)))
#endif
      // Waves run back to back with programmatic dependent launch: each chain and fusion kernel starts on the SMs the
      // kernel before it leaves, and sets up, loads weights (chain: also the first tile's points, conv1 / gate layer 1
      // and conv2) before griddepcontrol.wait.  The hazards that wait covers, all on the single operand buffer `cat`:
      //   chain(w) stores into cat  after  fusion(w - 1) has read it        (write after read; the first store waits)
      //   fusion(w) loads cat       after  chain(w) has written it          (read after write; every A load waits)
      //   fusion(w) pooling atomics after  the global_feat memset above     (chain(w) waited, so fusion(w - 1) is done)
      // A second operand buffer would not let chain(w) start sooner: its CTA needs the SM that fusion(w - 1)'s CTA holds.
      // The first chain kernel of a call is an ordinary launch: it follows the memsets and whatever the caller enqueued.
      // (With LRN_OUT_MEMORY the projection, an ordinary launch, sits between fusion(w - 1) and chain(w).)
      LRN_TRY(launch_programmatic(r0 > 0, chain_pair_kernel, grid, kPairThreads, ChainSmem::kDynamic, stream, tw_chain[0],
                                  tw_chain[1], tw_chain[2], tw_chain[3], ta, cp));
    } else {  // layer 1 (+ gate layer 1): raw points -> operand columns
      StageTimer timer(LRN_STAGE_EMBED, stream);
      const int grid = int(std::min<int64_t>((rows + 15) / 16, int64_t(dev.sms) * 16));
      if (tf32)
        LRN_TRY(launch(point_embed_kernel<true>, grid, 256, 0, stream, reinterpret_cast<const float4*>(context) + r0, rows, ew, cat,
                       kCat * wm, x3 ? kCat : 0));
      else
        LRN_TRY(launch(point_embed_kernel<false>, grid, 256, 0, stream, reinterpret_cast<const float4*>(context) + r0, rows, ew,
                       cat, kCat, 0));
    }
    for (int k = fused_chain ? 6 : 2; k <= 5; ++k) {  // tf32 tier: conv2..conv5, each writes its own column block of the operand row
      GemmParams p{};
      p.M = int(rows);
      p.m_tiles = m_tiles_of(plan[k]);
      p.n_tiles = kChan[k] / plan[k].bn;
      p.kb_main = kpass * (kChan[k - 1] / bk);
      p.kb_gate = 0;
      p.split3 = x3 ? 1 : 0;
      p.a_lo_off = kCat;
      p.b_lo_off = kChan[k - 1];
      p.out_lo_off = kCat;
      p.a_col0 = kCatOff[k - 1];
      p.bias = reinterpret_cast<const float*>(pk + L.b[k]);
      p.out = static_cast<uint8_t*>(cat) + size_t(kCatOff[k]) * es;
      p.ldo = kCat * wm;
      p.out_f32 = tf32 ? 1 : 0;
      p.relu = 1;
      p.round_tf32 = tf32 ? 1 : 0;
      p.out_col0 = kCatOff[k];  // staged TMA stores go through the operand-row tensor map itself
#ifdef LRN_TIMELINE
      static const int dbg_layer = [] { const char* e = getenv("LRN_DBG_LAYER"); return e ? atoi(e) : 0; }();
      p.dbg = (k == dbg_layer) ? g_dbg : nullptr;
#endif
      StageTimer timer(LRN_STAGE_CONV2 + (k - 2), stream);
      LRN_TRY(launch_gemm(precision, plan[k], EPI_ACT, ta, tw[k], p, dev.sms, stream, &ta));
    }
    {  // fusion + gate + pooling
      GemmParams p{};
      p.M = int(rows);
      p.m_tiles = m_tiles_of(plan_f);
      p.n_tiles = 1024 / plan_f.bn;
      p.kb_main = kpass * (kFusionK / bk);
      p.kb_gate = kpass * (kGateK / bk);
      p.split3 = x3 ? 1 : 0;
      p.exact_gate = x3 ? 1 : 0;
      p.a_lo_off = kCat;
      p.b_lo_off = kCat;
      p.a_col0 = 0;
      p.a_tiled = tiled ? 1 : 0;
      p.bias_f = reinterpret_cast<const float*>(pk + L.bf);
      p.bias_g = reinterpret_cast<const float*>(pk + L.bg);
      p.row0 = r0;
      p.npts = int(N);
      p.inv_npts = 1.0f / float(N);
      p.flags = ((flags & LRN_OUT_ARGMAX) ? (FUSE_ARGMAX | FUSE_POOL) : (flags & LRN_OUT_POOL) ? FUSE_POOL : 0) |
                ((flags & LRN_OUT_FUSED) ? FUSE_STORE_CN : 0) | ((flags & LRN_OUT_MEMORY) ? FUSE_STORE_PM : 0);
      p.global_feat = global_feat;
      p.pool_key = keys;
      p.fused_cn = fused;
      p.fused_pm = fused_pm;
#ifdef LRN_TIMELINE
      p.dbg = getenv("LRN_DBG_LAYER") ? nullptr : g_dbg;
      if (const char* ring = getenv("LRN_DBG_RING")) p.a_ring = atoi(ring);
#endif
      StageTimer timer(LRN_STAGE_FUSION, stream);
      LRN_TRY(launch_gemm(precision, plan_f, EPI_FUSION, ta, twfg, p, dev.sms, stream));
    }
    if (flags & LRN_OUT_MEMORY) {  // memory = fused * Wp^T + bp
      LRN_TRY(make_tmap(&tpm, precision, fused_pm, rows, 1024 * wm, 1024 * wm, BM));
      GemmParams p{};
      p.M = int(rows);
      p.m_tiles = m_tiles_of(plan_p);
      p.n_tiles = 256 / plan_p.bn;
      p.kb_main = kpass * (1024 / bk);
      p.split3 = x3 ? 1 : 0;
      p.a_lo_off = 1024;
      p.b_lo_off = 1024;
      p.a_col0 = 0;
      p.bias = reinterpret_cast<const float*>(pk + L.bp);
      p.relu = 0;
      CUtensorMap tmem_out;
      const bool mem_bf16 = flags & LRN_OUT_MEMORY_BF16;
      if (mem_bf16) {  // bf16 rows of pitch 512: [memory | 256 columns left to the caller], TMA-store epilogue
        p.out = reinterpret_cast<uint16_t*>(memory) + r0 * 512;
        p.ldo = 512;
        p.out_f32 = 0;
        LRN_TRY(make_tmap(&tmem_out, precision, p.out, rows, 256, 512, BM));
      } else {
        p.out = reinterpret_cast<float*>(memory) + r0 * 256;
        p.ldo = 256;
        p.out_f32 = 1;
      }
      StageTimer timer(LRN_STAGE_PROJ, stream);
      LRN_TRY(launch_gemm(precision, plan_p, EPI_ACT, tpm, twp, p, dev.sms, stream, mem_bf16 ? &tmem_out : nullptr));
    }
  }
  if (flags & LRN_OUT_ARGMAX) {
    const int grid = int(std::min<int64_t>((B * 1024 + 255) / 256, 2048));
    LRN_TRY(launch(argmax_finalize_kernel, grid, 256, 0, stream, keys, B, global_feat, reinterpret_cast<long long*>(argmax)));
  }
  return LRN_OK;
}

int lrn_gemm_tn(const void* At, int64_t lda, const void* Bt, int64_t ldb, float* out, int64_t ldo, int64_t M, int64_t N,
                int64_t K, lrn_stream_t stream) {
  if (!At || !Bt || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (M <= 0 || N <= 0 || K <= 0 || N % 128 || M % 64) return fail(LRN_ERR_BAD_SHAPE, "M=%lld N=%lld K=%lld", (long long)M, (long long)N, (long long)K);
  LRN_DEVICE(dev);
  const int bn = (N % 256 == 0) ? 256 : 128;
  CUtensorMap ta, tb;
  LRN_TRY(make_tmap_mn(&ta, At, K, M, lda));
  LRN_TRY(make_tmap_mn(&tb, Bt, K, N, ldb));
  GemmParams p{};
  p.M = int(M);
  p.m_tiles = int((M + 2 * BM - 1) / (2 * BM));
  p.n_tiles = int(N / bn);
  p.kb_main = int((K + 63) / 64);  // rows beyond K are zero-filled by TMA
  p.out = out;
  p.ldo = ldo;
  p.out_f32 = 1;
  const int out_tiles = p.m_tiles * p.n_tiles, slots = dev.sms / 2;
  if (out_tiles < slots && p.kb_main >= 64) {  // split K over the idle CTA pairs (fp32 atomic accumulation)
    // The kernel is persistent (one CTA pair per slot walks the work items): pick the split count whose item count fills
    // whole rounds of the `slots` pairs best - e.g. 32 output tiles: 9 splits = 288 items = 3.9 rounds of 74, where
    // "about two items per pair" (5 splits = 160 items = 2.2 rounds) left a third of the last round empty.
    int want = 1;
    double best = 0.0;
    const int max_split = std::min(p.kb_main / 16, 6 * slots / out_tiles + 1);
    for (int sp = 2; sp <= max_split; ++sp) {
      const int items = out_tiles * sp, rounds = (items + slots - 1) / slots;
      const double eff = double(items) / (double(rounds) * slots);
      if (eff > best + 0.02) {  // prefer fewer splits (fewer atomic passes over the output) unless clearly better
        best = eff;
        want = sp;
      }
    }
    if (want > 1) {
      p.kb_per_split = (p.kb_main + want - 1) / want;
      p.k_splits = (p.kb_main + p.kb_per_split - 1) / p.kb_per_split;
      LRN_CUDA(cudaMemset2DAsync(out, size_t(ldo) * 4, 0, size_t(N) * 4, size_t(M), stream));
    }
  }
  return bn == 256 ? launch_pair_t<256, false, EPI_ACT, 6, true, false, true>(ta, tb, ta, p, dev.sms, stream)
                   : launch_pair_t<128, false, EPI_ACT, 8, true, false, true>(ta, tb, ta, p, dev.sms, stream);
}

int lrn_ctx_attention_splits(int B, int N) {
  if (B <= 0 || N <= 0) return 0;
  DeviceInfo dev;
  if (device_info(&dev)) return 0;
  const int total = (N + kAttnStep - 1) / kAttnStep, slots = dev.sms / 2;
  int splits = std::max(1, std::min((slots + B - 1) / B, total));
  const int per = (total + splits - 1) / splits;
  return (total + per - 1) / per;
}

int lrn_ctx_attention(const void* qfold, const void* kp, int64_t ld_kp, const void* mem, int64_t ld_mem, int B, int N,
                      int splits, void* out, int out_bf16, float* lse, lrn_stream_t stream) {
  if (!qfold || !kp || !mem || !out || !lse) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (B <= 0 || N <= 0 || int64_t(B) * N >= (int64_t(1) << 31) - 256) return fail(LRN_ERR_BAD_SHAPE, "B=%d N=%d", B, N);
  if (ld_kp < 256 || ld_mem < 256) return fail(LRN_ERR_BAD_ARG, "row pitch below 256");
  const int total = (N + kAttnStep - 1) / kAttnStep;
  if (splits < 1 || splits > total) return fail(LRN_ERR_BAD_ARG, "splits=%d (1..%d)", splits, total);
  const int per = (total + splits - 1) / splits;
  if ((splits - 1) * per >= total) return fail(LRN_ERR_BAD_ARG, "splits=%d leaves an empty split (use lrn_ctx_attention_splits)", splits);
  LRN_DEVICE(dev);
  CUtensorMap tq, tk, tv;
  LRN_TRY(make_tmap(&tq, LRN_PREC_BF16, qfold, int64_t(B) * 256, 256, 256, 128));
  LRN_TRY(make_tmap(&tk, LRN_PREC_BF16, kp, int64_t(B) * N, 256, ld_kp, 64));
  LRN_TRY(make_tmap_mn(&tv, mem, int64_t(B) * N, 256, ld_mem));
  AttnParams p{};
  p.items = B * splits;
  p.N = N;
  p.splits = splits;
  p.steps_per_split = per;
  p.out = out;
  p.out_bf16 = out_bf16 ? 1 : 0;
  p.lse = lse;
  static std::atomic<uint64_t> configured{0};
  LRN_TRY(configure_smem(ctx_attn_kernel, int(AttnSmem::kDynamic), configured));
  const int clusters = std::min(B * splits, dev.sms / 2);  // persistent: one cluster per SM pair walks the items
  return launch(ctx_attn_kernel, 2 * clusters, kAttnThreads, AttnSmem::kDynamic, stream, tq, tk, tv, p);
}

int lrn_pos_hidden(const float* w1, const float* b1, const float* context, int64_t P, void* out, int64_t ld_out,
                   lrn_stream_t stream) {
  if (!w1 || !b1 || !context || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (P <= 0) return fail(LRN_ERR_BAD_SHAPE, "P=%lld", (long long)P);
  if (misaligned(16, context, out) || ld_out < 256 || (ld_out * 2) % 16)
    return fail(LRN_ERR_MISALIGNED, "context / out need 16-byte alignment, ld_out >= 256 and a multiple of 8");
  LRN_DEVICE(dev);
  const int grid = int(std::min<int64_t>((P + 7) / 8, int64_t(dev.sms) * 8));
  return launch(pos_hidden_kernel, grid, 256, 0, stream, reinterpret_cast<const float4*>(context), P, w1, b1,
                reinterpret_cast<uint16_t*>(out), ld_out);
}

int lrn_pos_hidden_backward(const float* context, int64_t P, const void* hidden, int64_t ld_hidden, const void* d_hidden,
                            int64_t ld_d, float* d_w1, float* d_b1, lrn_stream_t stream) {
  if (!context || !hidden || !d_hidden || !d_w1 || !d_b1) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (P <= 0) return fail(LRN_ERR_BAD_SHAPE, "P=%lld", (long long)P);
  if (misaligned(16, context, hidden, d_hidden) || ld_hidden % 8 || ld_d % 8 || ld_hidden < 256 || ld_d < 256)
    return fail(LRN_ERR_MISALIGNED, "16-byte alignment, row pitches >= 256 and multiples of 8");
  LRN_DEVICE(dev);
  LRN_CUDA(cudaMemsetAsync(d_w1, 0, 256 * 3 * 4, stream));
  LRN_CUDA(cudaMemsetAsync(d_b1, 0, 256 * 4, stream));
  const int grid = int(std::min<int64_t>((P + 7) / 8, int64_t(dev.sms) * 4));
  return launch(pos_hidden_bwd_kernel, grid, 256, 0, stream, reinterpret_cast<const float4*>(context), P,
                reinterpret_cast<const uint16_t*>(hidden), ld_hidden, reinterpret_cast<const uint16_t*>(d_hidden), ld_d, d_w1, d_b1);
}

// ---------------------------------------------------------------- scene preprocessing (section 8f row 3)
namespace {
struct SceneLayout {
  size_t aabb, dense_f, count, fill, imin, imax, offset, cand, keys, first, cursor, order, total;
};
// the line grouping by scene (first (K+1), cursor (K), order (L) ints) follows the per-line arrays
SceneLayout scene_layout(int L, int64_t capacity, int K) {
  SceneLayout w{};
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  w.aabb = take(size_t(L) * scene::kBoxFloats * 4);
  w.dense_f = take(size_t(L) * scene::kDense * 3 * 4);
  w.count = take(size_t(L) * 4);
  w.fill = take(size_t(L) * 4);
  w.imin = take(size_t(L) * 4);
  w.imax = take(size_t(L) * 4);
  w.offset = take(size_t(L + 1) * 8);
  w.cand = take(size_t(capacity) * 4);
  w.keys = take(size_t(capacity) * 8);
  w.first = take(size_t(K + 1) * 4);
  w.cursor = take(size_t(K) * 4);
  w.order = take(size_t(L) * 4);
  w.total = off;
  return w;
}
int scene_cap(int N) {
  int c = 2;
  while (c < 2 * N) c <<= 1;
  return c;
}
}  // namespace

int lrn_scene_resample(const double* vertices, const int64_t* offsets, int L, int max_vertices, double* line32, double* dense200,
                       double* centers, float* noisy_centered, lrn_stream_t stream) {
  if (!vertices || !offsets || !line32 || !dense200 || !centers || !noisy_centered) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (L <= 0 || max_vertices < 0 || max_vertices > scene::kMaxVertices)
    return fail(LRN_ERR_BAD_SHAPE, "L=%d, longest polyline %d vertices (limit %d)", L, max_vertices, scene::kMaxVertices);
  LRN_DEVICE(dev);
  return launch(scene::resample_kernel, L, 256, 0, stream, vertices, reinterpret_cast<const long long*>(offsets), L, line32,
                dense200, centers, noisy_centered);
}

size_t lrn_scenes_workspace_bytes(int L, int K, int64_t capacity) {
  if (L <= 0 || K <= 0 || capacity <= 0) return 0;
  return scene_layout(L, capacity, K).total;
}

// group / prep / count / scan / fill / keys / select
int lrn_scenes_segments(const float* points, const int64_t* scene_offsets, int K, int64_t S_total, const float* sorted_points,
                        const int32_t* perm, const int32_t* line_scene, const double* dense200, const double* line32,
                        const double* centers, const uint64_t* seeds, const uint32_t* line_ids, int L, int N, double crop_radius,
                        double decay_scale, double coord_extent, int64_t capacity, float* context, int64_t* indices, int32_t* counts,
                        int64_t* status, void* workspace, size_t workspace_bytes, lrn_stream_t stream) {
  if (!points || !scene_offsets || !line_scene || !dense200 || !line32 || !centers || !seeds || !line_ids || !context || !indices ||
      !counts || !status || !workspace)
    return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (S_total <= 0 || S_total >= (int64_t(1) << 31) || K <= 0 || K > 65535 || L <= 0 || L > 65535 || N <= 0 || N > 4096 ||
      capacity <= 0)
    return fail(LRN_ERR_BAD_SHAPE, "S_total=%lld K=%d L=%d N=%d capacity=%lld (S_total < 2^31, K <= 65535, L <= 65535, N <= 4096)",
                (long long)S_total, K, L, N, (long long)capacity);
  if (!(crop_radius > 0) || !(decay_scale > 0) || !(coord_extent >= 0) ||
      (crop_radius + 2.0) / decay_scale > 25.0)
    return fail(LRN_ERR_BAD_ARG, "crop_radius=%g decay_scale=%g: (radius + 2) / decay must stay <= 25 (weights must not underflow)",
                crop_radius, decay_scale);
  if (misaligned(16, points, context) || misaligned(256, workspace))
    return fail(LRN_ERR_MISALIGNED, "points / context need 16-byte, workspace 256-byte alignment");
  const SceneLayout w = scene_layout(L, capacity, K);
  if (workspace_bytes < w.total) return fail(LRN_ERR_WORKSPACE, "workspace %zu < %zu bytes", workspace_bytes, w.total);
  LRN_DEVICE(dev);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  float* aabb = reinterpret_cast<float*>(ws + w.aabb);
  float* dense_f = reinterpret_cast<float*>(ws + w.dense_f);
  int* count = reinterpret_cast<int*>(ws + w.count);
  int* fill = reinterpret_cast<int*>(ws + w.fill);
  int* imin = reinterpret_cast<int*>(ws + w.imin);
  int* imax = reinterpret_cast<int*>(ws + w.imax);
  long long* offset = reinterpret_cast<long long*>(ws + w.offset);
  uint32_t* cand = reinterpret_cast<uint32_t*>(ws + w.cand);
  uint64_t* keys = reinterpret_cast<uint64_t*>(ws + w.keys);
  int* first = reinterpret_cast<int*>(ws + w.first);
  int* order = reinterpret_cast<int*>(ws + w.order);
  long long* stat = reinterpret_cast<long long*>(status);
  // fp32 pre-filter: decides `distance < radius` outside a band of +-eps, the band is evaluated in double
  const double eps = 1e-3 + 4e-6 * coord_extent;
  const double rlo = std::max(crop_radius - eps, 0.0), rhi = crop_radius + eps;
  const float r2_lo = float(rlo * rlo * (1.0 - 1e-6)), r2_hi = float(rhi * rhi * (1.0 + 1e-6));
  const float4* pts = reinterpret_cast<const float4*>(points);
  if ((sorted_points != nullptr) != (perm != nullptr)) return fail(LRN_ERR_BAD_ARG, "sorted_points and perm come together");
  if (misaligned(16, sorted_points)) return fail(LRN_ERR_MISALIGNED, "sorted_points needs 16-byte alignment");
  const float4* crop_pts = sorted_points ? reinterpret_cast<const float4*>(sorted_points) : pts;
  const long long* scene_off = reinterpret_cast<const long long*>(scene_offsets);
  const scene::Lines src{scene_off, line_scene, seeds, line_ids, K};
  const scene::Groups grp{scene_off, first, order, K};
  LRN_TRY(launch(scene::group_kernel, 1, 1024, 0, stream, line_scene, L, K, first, reinterpret_cast<int*>(ws + w.cursor), order));
  LRN_TRY(launch(scene::prep_kernel, L, 128, 0, stream, dense200, L, float(rhi * (1.0 + 1e-6)), aabb, dense_f, count, fill, imin,
                 imax));
  const int grid = int((S_total + 255) / 256);
  auto crop = [&](auto kernel) {
    return launch(kernel, grid, 256, 0, stream, crop_pts, S_total, aabb, dense_f, dense200, crop_radius, r2_lo, r2_hi, count, imin,
                  imax, fill, offset, capacity, perm, cand, grp);
  };
  LRN_TRY(crop(scene::tube_crop_kernel<false>));
  LRN_TRY(launch(scene::scan_kernel, 1, 1024, 0, stream, count, L, capacity, offset, stat));
  LRN_TRY(crop(scene::tube_crop_kernel<true>));
  LRN_TRY(launch(scene::sample_keys_kernel, dim3(32, L), 256, 0, stream, pts, line32, count, offset, imin, imax, N, decay_scale,
                 src, stat, cand, keys));
  const int cap = scene_cap(N);
  const size_t smem = size_t(cap) * 12;
  // the opt-in above 48 KB is per device and the size depends on N: set it on every call (a host-side attribute write)
  LRN_CUDA(cudaFuncSetAttribute(scene::select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  return launch(scene::select_kernel, L, 256, smem, stream, pts, centers, count, offset, N, cap, src, stat, cand, keys, context,
                reinterpret_cast<long long*>(indices), counts);
}

int lrn_debug_timeline(long long* device_buffer) {
#ifdef LRN_TIMELINE
  g_dbg = device_buffer;
  return LRN_OK;
#else
  (void)device_buffer;
  return fail(LRN_ERR_BAD_ARG, "this library was built without -DLRN_TIMELINE (tools/timeline.py builds the tuning variant)");
#endif
}

int lrn_profile_enable(int on) {
  g_prof.on = on != 0;
  return LRN_OK;
}

int lrn_profile_read(float* ms_per_stage, int64_t* launches_per_stage) {
  if (!ms_per_stage || !launches_per_stage) return fail(LRN_ERR_BAD_ARG, "null output");
  for (int i = 0; i < LRN_STAGE_COUNT; ++i) { ms_per_stage[i] = 0.f; launches_per_stage[i] = 0; }
  for (size_t i = 0; i < g_prof.stage.size(); ++i) {
    cudaEvent_t a = g_prof.ev[2 * i], b = g_prof.ev[2 * i + 1];
    LRN_CUDA(cudaEventSynchronize(b));
    float ms = 0.f;
    LRN_CUDA(cudaEventElapsedTime(&ms, a, b));
    ms_per_stage[g_prof.stage[i]] += ms;
    launches_per_stage[g_prof.stage[i]] += 1;
    g_prof.pool.push_back(a);
    g_prof.pool.push_back(b);
  }
  g_prof.ev.clear();
  g_prof.stage.clear();
  return LRN_OK;
}

int lrn_point_embed(const void* packed, int precision, const float* context, int64_t rows, void* operand_rows, int tiled,
                    lrn_stream_t stream) {
  if ((precision != LRN_PREC_BF16 && precision != LRN_PREC_TF32) || !packed || !context || !operand_rows || rows <= 0)
    return fail(LRN_ERR_BAD_ARG, "bad argument");
  if (tiled && precision != LRN_PREC_BF16) return fail(LRN_ERR_BAD_ARG, "the tiled operand layout is the bf16 tier's");
  LRN_DEVICE(dev);
  const PackedLayout L = packed_layout(precision);
  const uint8_t* pk = static_cast<const uint8_t*>(packed);
  EmbedWeights ew{reinterpret_cast<const float*>(pk + L.w1), reinterpret_cast<const float*>(pk + L.b1),
                  reinterpret_cast<const float*>(pk + L.wg1), reinterpret_cast<const float*>(pk + L.bg1)};
  const int grid = int(std::min<int64_t>((rows + 15) / 16, int64_t(dev.sms) * 16));
  if (precision == LRN_PREC_TF32)
    return launch(point_embed_kernel<true>, grid, 256, 0, stream, reinterpret_cast<const float4*>(context), rows, ew, operand_rows,
                  kCat, 0);
  return launch(point_embed_kernel<false>, grid, 256, 0, stream, reinterpret_cast<const float4*>(context), rows, ew, operand_rows,
                tiled ? 0 : kCat, 0);
}

int lrn_head_forward(const float* w1, const float* b1, const float* w2, const float* b2, const float* tgt,
                     int64_t rows, float* current, const float* noisy, float* cum_out, lrn_stream_t stream) {
  if (!w1 || !b1 || !w2 || !b2 || !tgt || !current || !noisy || !cum_out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (rows <= 0 || rows > (int64_t(1) << 31)) return fail(LRN_ERR_BAD_SHAPE, "rows=%lld", (long long)rows);
  if (misaligned(16, tgt, w1)) return fail(LRN_ERR_MISALIGNED, "tgt/w1 need 16-byte alignment");
  LRN_DEVICE(dev);
  const int grid = int((rows + kHeadRows - 1) / kHeadRows);
  return launch(head_kernel, grid, 128, 0, stream, w1, b1, w2, b2, tgt, rows, current, noisy, cum_out);
}

int lrn_gemm_bias_act(int precision, const void* A, int64_t lda, const void* Wt, int64_t ldw, const float* bias,
                      void* out, int64_t ldo, int out_f32, int relu, int64_t M, int64_t N, int64_t K,
                      lrn_stream_t stream) {
  if ((precision != LRN_PREC_BF16 && precision != LRN_PREC_TF32) || !A || !Wt || !out) return fail(LRN_ERR_BAD_ARG, "null pointer or bad precision");
  const size_t es = elem_size(precision);
  const int bk = int(128 / es);
  if (M <= 0 || N <= 0 || K <= 0 || K % bk || N % 128 || M >= (int64_t(1) << 31))
    return fail(LRN_ERR_BAD_SHAPE, "M=%lld N=%lld K=%lld", (long long)M, (long long)N, (long long)K);
  LRN_DEVICE(dev);
  GemmPlan g = plan_gemm(N, EPI_ACT);
  if (g.bn == 256 && ((M + g.m_rows - 1) / g.m_rows) * (N / 256) < dev.sms / 2) {
    g.bn = 128;  // few tiles (the decoder's query side: a few thousand rows): 128-column tiles give the idle CTA pairs work
    g.b_box_rows = 64;
  }
  CUtensorMap ta, tb;
  LRN_TRY(make_tmap(&ta, precision, A, M, K, lda, BM));
  LRN_TRY(make_tmap(&tb, precision, Wt, N, K, ldw, g.b_box_rows));
  GemmParams p{};
  p.M = int(M);
  p.m_tiles = int((M + g.m_rows - 1) / g.m_rows);
  p.n_tiles = int(N / g.bn);
  p.kb_main = int(K / bk);
  p.bias = bias;
  p.out = out;
  p.ldo = ldo;
  p.out_f32 = out_f32;
  p.relu = relu;
  // Weight gradients: few output tiles, K = all points.  Split K over the idle CTA pairs; the splits add their
  // partial products atomically into the zeroed fp32 output.
  const int out_tiles = p.m_tiles * p.n_tiles, slots = dev.sms / 2;
  if (out_f32 && !relu && precision == LRN_PREC_BF16 && out_tiles < slots && p.kb_main >= 64) {
    const int want = std::min((2 * slots + out_tiles - 1) / out_tiles, p.kb_main / 16);
    if (want > 1) {
      p.kb_per_split = (p.kb_main + want - 1) / want;
      p.k_splits = (p.kb_main + p.kb_per_split - 1) / p.kb_per_split;
      LRN_CUDA(cudaMemset2DAsync(out, size_t(ldo) * 4, 0, size_t(N) * 4, size_t(M), stream));
    }
  }
  CUtensorMap tout;
  const bool staged_ok = precision == LRN_PREC_BF16 && !out_f32 && !misaligned(16, out) && (ldo * 2) % 16 == 0;
  if (staged_ok) LRN_TRY(make_tmap(&tout, precision, out, M, N, ldo, BM));
  return launch_gemm(precision, g, EPI_ACT, ta, tb, p, dev.sms, stream, staged_ok ? &tout : nullptr);
}

}  // extern "C"

// =====================================================================================================
// Train-mode path: batch-statistic BatchNorm forward + hand-written backward of the context encoder
// (reference: MultiScalePointNetEncoder.forward in model.train(), src/model.py:39-55, driven by the training
// loops train.py:56-72 / train_dist.py:168-189).  bf16 tensor-core operands, fp32 master weights and gradients.
// Every GEMM (forward, dgrad, wgrad) is the tcgen05 pair kernel; csrc/train_kernels.cuh holds the glue.
// =====================================================================================================
#include "train_kernels.cuh"
#include "train_attn.cuh"

namespace {

const int kUOff[6] = {0, 64, 192, 448, 960, 1984};  // column of U_k (pre-BN) inside the (P, 3008) buffer; [5] = fusion
const int kUW[6] = {64, 128, 256, 512, 1024, 1024};
constexpr int kULd = 3008;
constexpr int kStatLd = 3008;

struct TrainWs {
  int64_t P, Pp;
  // activations saved by the forward
  size_t X, U, Z;
  // statistics (fp32, kStatLd each): sum, sumsq, mean, rstd, scale, shift, S1, S2; Sz (1024)
  size_t stats;
  // bf16 weights: W2..W5, Wf (1024 x 2048), Wg2 (1024 x 64), and transposed copies for the dgrads
  size_t w[6], wf, wg2, wt[6], wft, wg2t, wpack_end;
  // backward temporaries
  size_t dA, dB, dU, dZ, dHp, gW;
  size_t total;
};

TrainWs train_layout(int64_t B, int64_t N) {
  TrainWs W{};
  W.P = B * N;
  W.Pp = (W.P + 255) / 256 * 256;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  W.X = take(size_t(W.Pp) * kCat * 2);
  W.U = take(size_t(W.Pp) * kULd * 2);
  W.Z = take(size_t(W.Pp) * 1024 * 2);
  W.stats = take(size_t(8 * kStatLd + 1024) * 4);
  const size_t wstart = off;
  for (int k = 2; k <= 5; ++k) W.w[k] = take(size_t(kChan[k]) * kChan[k - 1] * 2);
  W.wf = take(size_t(1024) * kCat * 2);
  W.wg2 = take(size_t(1024) * 64 * 2);
  for (int k = 2; k <= 5; ++k) W.wt[k] = take(size_t(std::max(kChan[k - 1], 128)) * kChan[k] * 2);
  W.wft = take(size_t(kCat) * 1024 * 2);
  W.wg2t = take(size_t(128) * 1024 * 2);
  W.wpack_end = off;
  (void)wstart;
  W.dA = take(size_t(W.Pp) * kCat * 2);
  W.dB = take(size_t(W.Pp) * 512 * 2);
  W.dU = take(size_t(W.Pp) * 1024 * 2);
  W.dZ = take(size_t(W.Pp) * 1024 * 2);
  W.dHp = take(size_t(W.Pp) * 128 * 2);
  W.gW = take(size_t(1024) * kCat * 4);
  W.total = off;
  return W;
}

// out (M x N) = [relu](A (M x K) * Wt (N x K)^T + bias), bf16 operands, bf16 or fp32 output
int run_gemm_bf16(const void* A, int64_t lda, int64_t M, int64_t K, const void* Wt, int64_t ldw, int64_t N,
                  const float* bias, void* out, int64_t ldo, int out_f32, int relu, cudaStream_t s) {
  return lrn_gemm_bias_act(LRN_PREC_BF16, A, lda, Wt, ldw, bias, out, ldo, out_f32, relu, M, N, K,
                           reinterpret_cast<lrn_stream_t>(s));
}

int pack_w(const float* src, int rows, int cols, void* dst, int64_t ld, bool transpose, cudaStream_t s) {
  const long long total = static_cast<long long>(rows) * cols;
  return launch(pack_bf16_kernel, int(std::min<long long>((total + 255) / 256, 2048)), 256, 0, s, src, rows, cols,
                static_cast<__nv_bfloat16*>(dst), ld, transpose ? 1 : 0);
}

// Streaming kernels over a (rows x C) bf16 matrix: grid = (column blocks of 64 channels, row slabs), blocks loop over the rows.
// The grid is sized to what is resident: the blocks of these streaming kernels loop over the rows, so a grid of
// exactly (SMs x resident blocks per SM) leaves no partial last wave (1200 blocks at 2 per SM were 4.05 waves).
template <typename Kernel>
dim3 stream_grid(Kernel kernel, int C, int64_t rows, int sms) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 2;
  const int64_t slabs = std::max<int64_t>(1, std::min<int64_t>((rows + 31) / 32, int64_t(sms) * per_sm / (C / 64)));
  return dim3(C / 64, unsigned(slabs));
}

int elem_grid(long long total) { return int(std::min<long long>((total + 255) / 256, 148 * 32)); }

}  // namespace

extern "C" {

size_t lrn_train_workspace_bytes(int64_t B, int64_t N) {
  if (B <= 0 || N <= 0) return 0;
  return train_layout(B, N).total;
}

int lrn_encoder_train_forward(const lrn_encoder_params* pr, const lrn_bn_running* running, float momentum,
                              const float* context, int64_t B, int64_t N, void* fused, int fused_point_major,
                              float* global_feat, int64_t* argmax, void* workspace, size_t workspace_bytes,
                              lrn_stream_t stream) {
  if (!pr || !context || !fused || !workspace) return fail(LRN_ERR_BAD_ARG, "null argument");
  if ((global_feat != nullptr) != (argmax != nullptr) || (global_feat && fused_point_major))
    return fail(LRN_ERR_BAD_ARG, "global_feat and argmax come together and need the (B,1024,N) fused layout");
  if (B <= 0 || N <= 0 || B * N >= (int64_t(1) << 31) - 256) return fail(LRN_ERR_BAD_SHAPE, "B=%lld N=%lld", (long long)B, (long long)N);
  LRN_DEVICE(dev);
  const TrainWs W = train_layout(B, N);
  if (workspace_bytes < W.total) return fail(LRN_ERR_WORKSPACE, "workspace %zu < %zu", workspace_bytes, W.total);
  if (misaligned(1024, workspace)) return fail(LRN_ERR_MISALIGNED, "workspace must be 1024-byte aligned");
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  auto* X = reinterpret_cast<__nv_bfloat16*>(ws + W.X);
  auto* U = reinterpret_cast<__nv_bfloat16*>(ws + W.U);
  auto* Z = reinterpret_cast<__nv_bfloat16*>(ws + W.Z);
  float* stats = reinterpret_cast<float*>(ws + W.stats);
  float *sum = stats, *sumsq = stats + kStatLd, *mean = stats + 2 * kStatLd, *rstd = stats + 3 * kStatLd,
        *scale = stats + 4 * kStatLd, *shift = stats + 5 * kStatLd;
  const int64_t P = W.P;

  LRN_CUDA(cudaMemsetAsync(stats, 0, size_t(2 * kStatLd) * 4, stream));
  LRN_CUDA(cudaMemsetAsync(ws + W.w[2], 0, W.wpack_end - W.w[2], stream));
  for (int k = 2; k <= 5; ++k) {  // bf16 copies of the (unfolded) weights, and transposed for the dgrads
    LRN_TRY(pack_w(pr->conv_w[k - 1], kChan[k], kChan[k - 1], ws + W.w[k], kChan[k - 1], false, stream));
    LRN_TRY(pack_w(pr->conv_w[k - 1], kChan[k], kChan[k - 1], ws + W.wt[k], kChan[k], true, stream));
  }
  LRN_TRY(pack_w(pr->fusion_w, 1024, kFusionK, ws + W.wf, kCat, false, stream));
  LRN_TRY(pack_w(pr->fusion_w, 1024, kFusionK, ws + W.wft, 1024, true, stream));
  LRN_TRY(pack_w(pr->gate2_w, 1024, 64, ws + W.wg2, 64, false, stream));
  LRN_TRY(pack_w(pr->gate2_w, 1024, 64, ws + W.wg2t, 1024, true, stream));

  LRN_TRY(launch(train_embed_kernel, int(std::min<int64_t>((P + 15) / 16, int64_t(dev.sms) * 16)), 256, 0, stream,
                 reinterpret_cast<const float4*>(context), P, pr->conv_w[0], pr->conv_b[0], pr->gate0_w, pr->gate0_b, U, kULd, X,
                 kCat));

  for (int i = 0; i < 6; ++i) {  // i = 0..4: conv1..conv5, i = 5: fusion
    const int C = kUW[i], uo = kUOff[i];
    const float* gamma = i < 5 ? pr->bn_w[i] : pr->fusion_bn_w;
    const float* beta = i < 5 ? pr->bn_b[i] : pr->fusion_bn_b;
    LRN_TRY(launch(col_stats_kernel, stream_grid(col_stats_kernel, C, P, dev.sms), 256, 0, stream, U + uo, kULd, P, sum + uo,
                   sumsq + uo, 1));
    LRN_TRY(launch(bn_finalize_kernel, (C + 127) / 128, 128, 0, stream, sum + uo, sumsq + uo, U + uo, P, C, gamma, beta, pr->bn_eps,
                   momentum, running ? running->mean[i] : nullptr, running ? running->var[i] : nullptr, mean + uo, rstd + uo,
                   scale + uo, shift + uo));
    if (i == 5) break;
    LRN_TRY(launch(bn_relu_apply_kernel, stream_grid(bn_relu_apply_kernel, C, P, dev.sms), 256, 0, stream, U + uo, kULd, P, C,
                   scale + uo, shift + uo, X + kCatOff[i + 1], kCat));
    if (i < 4) {  // next layer's pre-activation: U_{k+1} = X_k W_{k+1}^T + b_{k+1}
      const int k = i + 2;
      LRN_TRY(run_gemm_bf16(X + kCatOff[i + 1], kCat, P, kChan[k - 1], ws + W.w[k], kChan[k - 1], kChan[k], pr->conv_b[k - 1],
                            U + kUOff[i + 1], kULd, 0, 0, stream));
    } else {  // fusion conv over the whole operand row, and gate layer 2 over the gate hidden block
      LRN_TRY(run_gemm_bf16(X, kCat, P, kFusionK, ws + W.wf, kCat, 1024, pr->fusion_b, U + kUOff[5], kULd, 0, 0, stream));
      LRN_TRY(run_gemm_bf16(X + kFusionK, kCat, P, kGateK, ws + W.wg2, kGateK, 1024, pr->gate2_b, Z, 1024, 0, 0, stream));
    }
  }
  if (fused_point_major)
    return launch(fusion_gate_fwd_pm_kernel, stream_grid(fusion_gate_fwd_pm_kernel, 1024, P, dev.sms), 256, 0, stream, U + kUOff[5],
                  kULd, Z, 1024, P, scale + kUOff[5], shift + kUOff[5], static_cast<__nv_bfloat16*>(fused));
  LRN_TRY(launch(fusion_gate_fwd_kernel, dim3(unsigned((P + 31) / 32), 32), 256, 0, stream, U + kUOff[5], kULd, Z, 1024, P, int(N),
                 scale + kUOff[5], shift + kUOff[5], static_cast<float*>(fused)));
  if (global_feat)
    LRN_TRY(launch(pool_rows_kernel, int(std::min<int64_t>((B * 1024 + 7) / 8, int64_t(dev.sms) * 16)), 256, 0, stream,
                   static_cast<const float*>(fused), B * 1024, int(N), global_feat, reinterpret_cast<long long*>(argmax)));
  return LRN_OK;
}

int lrn_encoder_train_backward(const lrn_encoder_params* pr, const float* context, int64_t B, int64_t N,
                               const void* d_fused, int fused_point_major, const float* d_global_feat,
                               const int64_t* argmax, const lrn_encoder_grads* g, void* workspace, size_t workspace_bytes,
                               lrn_stream_t stream) {
  if (!pr || !context || !g || !workspace) return fail(LRN_ERR_BAD_ARG, "null argument");
  if (!d_fused && !d_global_feat) return fail(LRN_ERR_BAD_ARG, "no output gradient (d_fused and d_global_feat are null)");
  if (d_global_feat && (!argmax || fused_point_major))
    return fail(LRN_ERR_BAD_ARG, "d_global_feat needs the forward's argmax and the (B,1024,N) fused layout");
  LRN_DEVICE(dev);
  const TrainWs W = train_layout(B, N);
  if (workspace_bytes < W.total) return fail(LRN_ERR_WORKSPACE, "workspace %zu < %zu", workspace_bytes, W.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  auto* X = reinterpret_cast<__nv_bfloat16*>(ws + W.X);
  auto* U = reinterpret_cast<__nv_bfloat16*>(ws + W.U);
  auto* Z = reinterpret_cast<__nv_bfloat16*>(ws + W.Z);
  auto* dA = reinterpret_cast<__nv_bfloat16*>(ws + W.dA);
  auto* dB = reinterpret_cast<__nv_bfloat16*>(ws + W.dB);
  auto* dU = reinterpret_cast<__nv_bfloat16*>(ws + W.dU);
  auto* dZ = reinterpret_cast<__nv_bfloat16*>(ws + W.dZ);
  auto* dHp = reinterpret_cast<__nv_bfloat16*>(ws + W.dHp);
  float* gW = reinterpret_cast<float*>(ws + W.gW);
  float* stats = reinterpret_cast<float*>(ws + W.stats);
  float *mean = stats + 2 * kStatLd, *rstd = stats + 3 * kStatLd, *scale = stats + 4 * kStatLd, *shift = stats + 5 * kStatLd,
        *S1 = stats + 6 * kStatLd, *S2 = stats + 7 * kStatLd, *Sz = stats + 8 * kStatLd;
  const int64_t P = W.P;
  auto d2d = [&](float* dst, const float* src, int n) { return cudaMemcpyAsync(dst, src, size_t(n) * 4, cudaMemcpyDeviceToDevice, stream); };
  auto copy_sub = [&](const float* src, int64_t ld, int c0, int rows, int cols, float* dst) {
    return launch(copy_submatrix_kernel, elem_grid(static_cast<long long>(rows) * cols), 256, 0, stream, src, ld, c0, rows, cols, dst);
  };

  LRN_CUDA(cudaMemsetAsync(S1, 0, size_t(2 * kStatLd + 1024) * 4, stream));
  LRN_CUDA(cudaMemsetAsync(g->conv_w[0], 0, 64 * 4 * 4, stream));
  LRN_CUDA(cudaMemsetAsync(g->conv_b[0], 0, 64 * 4, stream));
  LRN_CUDA(cudaMemsetAsync(g->gate0_w, 0, 64 * 4, stream));
  LRN_CUDA(cudaMemsetAsync(g->gate0_b, 0, 64 * 4, stream));
  for (int k = 1; k < 5; ++k) LRN_CUDA(cudaMemsetAsync(g->conv_b[k], 0, size_t(kChan[k + 1]) * 4, stream));
  LRN_CUDA(cudaMemsetAsync(g->fusion_b, 0, 1024 * 4, stream));

  // ---- fused output: gate, ReLU, fusion BatchNorm
  {
    const int uo = kUOff[5];
    if (fused_point_major) {   // dY, dZ and the column sums S1 / S2 (BatchNorm backward) and Sz (gate bias) in one pass
      LRN_TRY(launch(fusion_gate_bwd_pm_kernel, stream_grid(fusion_gate_bwd_pm_kernel, 1024, P, dev.sms), 256, 0, stream,
                     static_cast<const __nv_bfloat16*>(d_fused), U + uo, kULd, Z, 1024, P, scale + uo, shift + uo, mean + uo,
                     rstd + uo, dU, dZ, 1024, S1 + uo, S2 + uo, Sz));
    } else {
      LRN_TRY(launch(fusion_gate_bwd_kernel, dim3(unsigned((P + 31) / 32), 32), 256, 0, stream, static_cast<const float*>(d_fused),
                     d_global_feat, reinterpret_cast<const long long*>(argmax), U + uo, kULd, Z, 1024, P, int(N), scale + uo,
                     shift + uo, dU, dZ, 1024));
      LRN_TRY(launch(col_stats_kernel, stream_grid(col_stats_kernel, 1024, P, dev.sms), 256, 0, stream, dZ, 1024, P, Sz, nullptr,
                     0));  // d(gate layer 2 bias)
      LRN_TRY(launch(bn_bwd_reduce_kernel, stream_grid(bn_bwd_reduce_kernel, 1024, P, dev.sms), 256, 0, stream, dU, 1024, nullptr, 0,
                     nullptr, nullptr, U + uo, kULd, P, mean + uo, rstd + uo, S1 + uo, S2 + uo));
    }
    LRN_CUDA(d2d(g->gate2_b, Sz, 1024));
    LRN_CUDA(d2d(g->fusion_bn_b, S1 + uo, 1024));
    LRN_CUDA(d2d(g->fusion_bn_w, S2 + uo, 1024));
    LRN_TRY(launch(bn_bwd_apply_kernel, stream_grid(bn_bwd_apply_kernel, 1024, P, dev.sms), 256, 0, stream, dU, 1024, nullptr, 0,
                   nullptr, nullptr, U + uo, kULd, P, 1024, mean + uo, rstd + uo, pr->fusion_bn_w, S1 + uo, S2 + uo, dU, 1024));
    // d(fusion conv bias) = sum_p dU is exactly zero: dU is the output of a batch-statistic BatchNorm backward, whose
    // columns sum to zero over the batch (the bias only shifts the batch mean).  It stays at the memset above instead of
    // the bf16 rounding noise a column sum of dU would give; same for conv2..conv5 below.
    // d(operand row) = dUf Wf  (columns >= 1984 of the padded transposed weight are zero)
    LRN_TRY(run_gemm_bf16(dU, 1024, P, 1024, ws + W.wft, 1024, kCat, nullptr, dA, kCat, 0, 0, stream));
    // dWf = dUf^T X   (K = points; MN-major operands straight from the point-major buffers)
    LRN_TRY(lrn_gemm_tn(dU, 1024, X, kCat, gW, kCat, 1024, kCat, P, stream));
    LRN_TRY(copy_sub(gW, kCat, 0, 1024, kFusionK, g->fusion_w));
    // gate layer 2: dH = dZ Wg2, dWg2 = dZ^T H
    LRN_TRY(run_gemm_bf16(dZ, 1024, P, 1024, ws + W.wg2t, 1024, 128, nullptr, dHp, 128, 0, 0, stream));
    LRN_TRY(lrn_gemm_tn(dZ, 1024, X + 1920, kCat, gW, 128, 1024, 128, P, stream));
    LRN_TRY(copy_sub(gW, 128, 64, 1024, 64, g->gate2_w));
  }
  // ---- chain, back to front: layer k consumes d(feat_k) = fusion dgrad slice (+ dgrad of layer k + 1)
  for (int k = 5; k >= 1; --k) {
    const int i = k - 1, C = kChan[k], uo = kUOff[i], xo = kCatOff[k];
    const __nv_bfloat16* d2 = k < 5 ? dB : nullptr;
    LRN_TRY(launch(bn_bwd_reduce_kernel, stream_grid(bn_bwd_reduce_kernel, C, P, dev.sms), 256, 0, stream, dA + xo, kCat, d2, 512,
                   scale + uo, shift + uo, U + uo, kULd, P, mean + uo, rstd + uo, S1 + uo, S2 + uo));
    LRN_CUDA(d2d(g->bn_b[i], S1 + uo, C));
    LRN_CUDA(d2d(g->bn_w[i], S2 + uo, C));
    LRN_TRY(launch(bn_bwd_apply_kernel, stream_grid(bn_bwd_apply_kernel, C, P, dev.sms), 256, 0, stream, dA + xo, kCat, d2, 512,
                   scale + uo, shift + uo, U + uo, kULd, P, C, mean + uo, rstd + uo, pr->bn_w[i], S1 + uo, S2 + uo, dU, 1024));
    if (k == 1) break;
    const int cin = kChan[k - 1], cin_p = std::max(cin, 128);
    // dW_k = dU_k^T X_{k-1}
    LRN_TRY(lrn_gemm_tn(dU, 1024, X + kCatOff[k - 1], kCat, gW, cin_p, C, cin_p, P, stream));
    LRN_TRY(copy_sub(gW, cin_p, 0, C, cin, g->conv_w[i]));
    // d(feat_{k-1}) += dU_k W_k
    LRN_TRY(run_gemm_bf16(dU, 1024, P, C, ws + W.wt[k], C, cin_p, nullptr, dB, 512, 0, 0, stream));
  }
  // ---- conv1 and gate layer 1 (fp32 reductions over the points)
  LRN_TRY(launch(conv1_gate1_bwd_kernel, int(std::min<int64_t>((P + 2047) / 2048, 1024)), 256, 0, stream,
                 reinterpret_cast<const float4*>(context), P, dU, 1024, dHp, 128, X + kFusionK, kCat, g->conv_w[0], g->conv_b[0],
                 g->gate0_w, g->gate0_b));
  LRN_CUDA(cudaMemsetAsync(g->conv_b[0], 0, 64 * 4, stream));  // in front of bn1: exactly zero as well (see fusion_b above)
  return LRN_OK;
}

int lrn_adam_step_capturable(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int64_t* step_state, lrn_stream_t stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq || !step_state) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (n <= 0) return fail(LRN_ERR_BAD_SHAPE, "n=%lld", (long long)n);
  LRN_DEVICE(dev);
  const int grid = int(std::min<int64_t>((n + 255) / 256, int64_t(dev.sms) * 16));
  LRN_TRY(launch(adam_bump_step_kernel, 1, 1, 0, stream, reinterpret_cast<long long*>(step_state)));
  return launch(adam_step_dev_kernel, grid, 256, 0, stream, params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                weight_decay, reinterpret_cast<const long long*>(step_state));
}

int lrn_l1_deep_supervision(const float* pred, const float* target, int L, int64_t n, float* loss, float* dpred,
                            lrn_stream_t stream) {
  if (!pred || !target || !loss) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (L <= 0 || n <= 0) return fail(LRN_ERR_BAD_SHAPE, "L=%d n=%lld", L, (long long)n);
  LRN_DEVICE(dev);
  LRN_CUDA(cudaMemsetAsync(loss, 0, 4, stream));
  const int grid = int(std::min<int64_t>((int64_t(L) * n + 255) / 256, int64_t(dev.sms) * 4));
  return launch(l1_deep_supervision_kernel, grid, 256, 0, stream, pred, target, L, n, loss, dpred);
}

int lrn_add_layernorm(const float* x, const float* y, const float* gamma, const float* beta, float eps, float* out,
                      float* stats, int64_t rows, int64_t cols, lrn_stream_t stream) {
  if (!x || !gamma || !beta || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (rows <= 0 || cols != 256) return fail(LRN_ERR_BAD_SHAPE, "rows=%lld cols=%lld (d_model = 256)", (long long)rows, (long long)cols);
  if (misaligned(16, x, y, out, gamma, beta)) return fail(LRN_ERR_MISALIGNED, "16-byte alignment");
  LRN_DEVICE(dev);
  const int grid = int(std::min<int64_t>((rows + 7) / 8, int64_t(dev.sms) * 8));
  return launch(add_layernorm256_kernel, grid, 256, 0, stream, x, y, gamma, beta, eps, out, stats, rows);
}

int lrn_add_layernorm_backward(const float* dy, const float* x, const float* y, const float* stats, const float* gamma, float* dz,
                               float* dgamma, float* dbeta, int64_t rows, int64_t cols, lrn_stream_t stream) {
  if (!dy || !x || !stats || !gamma || !dz || !dgamma || !dbeta) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (rows <= 0 || cols != 256) return fail(LRN_ERR_BAD_SHAPE, "rows=%lld cols=%lld (d_model = 256)", (long long)rows, (long long)cols);
  if (misaligned(16, x, y, dy, dz, gamma)) return fail(LRN_ERR_MISALIGNED, "16-byte alignment");
  LRN_DEVICE(dev);
  LRN_CUDA(cudaMemsetAsync(dgamma, 0, 256 * 4, stream));
  LRN_CUDA(cudaMemsetAsync(dbeta, 0, 256 * 4, stream));
  const int grid = int(std::min<int64_t>((rows + 7) / 8, int64_t(dev.sms) * 4));
  return launch(add_layernorm256_bwd_kernel, grid, 256, 0, stream, dy, x, y, stats, gamma, dz, dgamma, dbeta, rows);
}

int lrn_self_attention32(const float* qk, const float* v, float* out, int B, lrn_stream_t stream) {
  if (!qk || !v || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (B <= 0) return fail(LRN_ERR_BAD_SHAPE, "B=%d", B);
  LRN_DEVICE(dev);
  static std::atomic<uint64_t> configured{0};
  LRN_TRY(configure_smem(self_attn32_kernel, int(kSelfAttnSmem), configured));
  return launch(self_attn32_kernel, std::min(B, dev.sms * 2), 256, kSelfAttnSmem, stream, qk, v, out, B);
}

int lrn_head_update(const float* hidden, const float* w2, const float* b2, int64_t rows, float* current, const float* noisy,
                    float* cum, lrn_stream_t stream) {
  if (!hidden || !w2 || !b2 || !current || !noisy || !cum) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (rows <= 0) return fail(LRN_ERR_BAD_SHAPE, "rows=%lld", (long long)rows);
  if (misaligned(16, hidden, w2)) return fail(LRN_ERR_MISALIGNED, "hidden / w2 need 16-byte alignment");
  LRN_DEVICE(dev);
  const int grid = int(std::min<int64_t>((rows + 7) / 8, int64_t(dev.sms) * 8));
  return launch(head_update_kernel, grid, 256, 0, stream, hidden, w2, b2, rows, current, noisy, cum);
}

int lrn_rows_linear(const float* x, int64_t ldx, const float* x2, int64_t ldx2, const float* mlp3_w1, const float* mlp3_b1,
                    const float* w, const float* bias, void* out, int64_t ldo, int out_bf16, int relu, int64_t M, int64_t N,
                    int64_t K, lrn_stream_t stream) {
  if (!x || !w || !out || (mlp3_w1 && (!mlp3_b1 || x2))) return fail(LRN_ERR_BAD_ARG, "null pointer or both x2 and mlp3_w1 given");
  if (M <= 0 || M > (int64_t(1) << 24) || N <= 0 || N % 8 || K <= 0 || K % 32 || K > (1 << 20))
    return fail(LRN_ERR_BAD_SHAPE, "M=%lld N=%lld K=%lld (N %% 8 == 0, K %% 32 == 0)", (long long)M, (long long)N, (long long)K);
  if (misaligned(16, w)) return fail(LRN_ERR_MISALIGNED, "w needs 16-byte alignment");
  LRN_DEVICE(dev);
  RowsLinearArgs a{};
  a.x = x; a.x2 = x2; a.w1 = mlp3_w1; a.b1 = mlp3_b1; a.w = w; a.bias = bias; a.out = out;
  a.ldx = ldx; a.ldx2 = ldx2; a.ldo = ldo;
  a.M = int(M); a.N = int(N); a.K = int(K);
  a.relu = relu ? 1 : 0;
  a.out_bf16 = out_bf16 ? 1 : 0;
  const unsigned row_tiles = unsigned((M + 31) / 32);
  if (row_tiles > 65535) return fail(LRN_ERR_BAD_SHAPE, "M=%lld: more than 65535 row tiles", (long long)M);
  const bool nb4 = (N / 8) * row_tiles < unsigned(dev.sms);  // few blocks: halve the columns per block
  const dim3 grid(unsigned(N / (nb4 ? 4 : 8)), row_tiles);
  if (nb4) {
    if (mlp3_w1) return launch(rows_linear_kernel<ROWS_IN_MLP3, 4>, grid, 256, 0, stream, a);
    if (x2) return launch(rows_linear_kernel<ROWS_IN_SUM, 4>, grid, 256, 0, stream, a);
    return launch(rows_linear_kernel<ROWS_IN_PLAIN, 4>, grid, 256, 0, stream, a);
  }
  if (mlp3_w1) return launch(rows_linear_kernel<ROWS_IN_MLP3, 8>, grid, 256, 0, stream, a);
  if (x2) return launch(rows_linear_kernel<ROWS_IN_SUM, 8>, grid, 256, 0, stream, a);
  return launch(rows_linear_kernel<ROWS_IN_PLAIN, 8>, grid, 256, 0, stream, a);
}

int lrn_query_pos_hidden(const float* w1, const float* b1, const float* coords, int64_t ld, int64_t rows, float* out,
                         int round_tf32, lrn_stream_t stream) {
  if (!w1 || !b1 || !coords || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (rows <= 0 || ld < 3) return fail(LRN_ERR_BAD_SHAPE, "rows=%lld ld=%lld", (long long)rows, (long long)ld);
  if (misaligned(16, out)) return fail(LRN_ERR_MISALIGNED, "out needs 16-byte alignment");
  LRN_DEVICE(dev);
  const int grid = int(std::min<int64_t>((rows + 7) / 8, int64_t(dev.sms) * 8));
  return launch(query_pos_hidden_kernel, grid, 256, 0, stream, coords, ld, rows, w1, b1, out, round_tf32 ? 1 : 0);
}

int lrn_add(const float* a, const float* b, float* out, int64_t n, int round_tf32, lrn_stream_t stream) {
  if (!a || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (n <= 0 || n % 4) return fail(LRN_ERR_BAD_SHAPE, "n=%lld (a positive multiple of 4)", (long long)n);
  if (misaligned(16, a, b, out)) return fail(LRN_ERR_MISALIGNED, "16-byte alignment");
  LRN_DEVICE(dev);
  const int grid = int(std::min<int64_t>((n / 4 + 255) / 256, int64_t(dev.sms) * 8));
  return launch(add_kernel, grid, 256, 0, stream, reinterpret_cast<const float4*>(a), reinterpret_cast<const float4*>(b),
                reinterpret_cast<float4*>(out), n / 4, round_tf32 ? 1 : 0);
}

int lrn_cross_attention32(const float* q, const float* k, const float* v, int64_t ld_kv, int B, int N, float* out,
                          lrn_stream_t stream) {
  if (!q || !k || !v || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (B <= 0 || N <= 0 || ld_kv < 256 || int64_t(B) * 8 >= (int64_t(1) << 31)) return fail(LRN_ERR_BAD_SHAPE, "B=%d N=%d ld=%lld", B, N, (long long)ld_kv);
  if (misaligned(16, q)) return fail(LRN_ERR_MISALIGNED, "q needs 16-byte alignment");
  LRN_DEVICE(dev);
  static std::atomic<uint64_t> configured{0};
  LRN_TRY(configure_smem(cross_attn32_kernel, int(kCrossAttnSmem), configured));
  return launch(cross_attn32_kernel, B * 8, 256, kCrossAttnSmem, stream, q, k, v, ld_kv, N, out);
}

int lrn_ctx_attention_merge(const float* part, const float* lse, int B, int splits, void* out, int out_bf16, lrn_stream_t stream) {
  if (!part || !lse || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (B <= 0 || splits <= 0 || int64_t(B) * 256 >= (int64_t(1) << 31)) return fail(LRN_ERR_BAD_SHAPE, "B=%d splits=%d", B, splits);
  if (misaligned(16, part, out)) return fail(LRN_ERR_MISALIGNED, "16-byte alignment");
  LRN_DEVICE(dev);
  const int rows = B * 256;
  const int grid = std::min((rows + 7) / 8, dev.sms * 8);
  return launch(ctx_merge_kernel, grid, 256, 0, stream, part, lse, rows, splits, out, out_bf16 ? 1 : 0);
}

static int train_attn_args(TrainAttnParams* p, const float* q, const void* k, int64_t ld_k, const void* v, int64_t ld_v, int B, int N,
                           float* out, float* lse, float p_drop, uint64_t seed, const uint64_t* seed_state) {
  if (!q || !k || !v || !out || !lse) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (B <= 0 || N <= 0 || ld_k < 32 || ld_k % 8 || ld_v < 32 || ld_v % 8 || int64_t(B) * 8 >= (int64_t(1) << 31))
    return fail(LRN_ERR_BAD_SHAPE, "B=%d N=%d ld_k=%lld ld_v=%lld", B, N, (long long)ld_k, (long long)ld_v);
  if (!(p_drop >= 0.f && p_drop < 1.f)) return fail(LRN_ERR_BAD_ARG, "dropout probability %f", p_drop);
  if (misaligned(16, q, k, v, out)) return fail(LRN_ERR_MISALIGNED, "16-byte alignment");
  p->q = q;
  p->k = static_cast<const __nv_bfloat16*>(k);
  p->v = static_cast<const __nv_bfloat16*>(v);
  p->ld = ld_k;
  p->ldv = ld_v;
  p->B = B;
  p->N = N;
  p->out = out;
  p->lse = lse;
  p->p_drop = p_drop;
  p->seed = seed;
  p->seed_state = reinterpret_cast<const unsigned long long*>(seed_state);
  return LRN_OK;
}

int lrn_train_attention_forward(const float* q, const void* k, int64_t ld_k, const void* v, int64_t ld_v, int B, int N, float* out,
                                float* lse, float p_drop, uint64_t seed, const uint64_t* seed_state, lrn_stream_t stream) {
  TrainAttnParams p{};
  LRN_TRY(train_attn_args(&p, q, k, ld_k, v, ld_v, B, N, out, lse, p_drop, seed, seed_state));
  LRN_DEVICE(dev);
  return launch(train_attn_fwd_kernel, B * 8, 128, kTaFwdSmem, stream, p);
}

int lrn_train_attention_backward(const float* q, const void* k, int64_t ld_k, const void* v, int64_t ld_v, int B, int N,
                                 const float* out, const float* lse, const float* dout, float* dq, void* dk, int64_t ld_dk, void* dv,
                                 int64_t ld_dv, float p_drop, uint64_t seed, const uint64_t* seed_state, lrn_stream_t stream) {
  TrainAttnParams p{};
  LRN_TRY(train_attn_args(&p, q, k, ld_k, v, ld_v, B, N, const_cast<float*>(out), const_cast<float*>(lse), p_drop, seed, seed_state));
  if (!dout || !dq || !dk || !dv) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (ld_dk < 32 || ld_dk % 2 || ld_dv < 32 || ld_dv % 2 || misaligned(16, dout, dq) || misaligned(4, dk, dv))
    return fail(LRN_ERR_MISALIGNED, "dout / dq need 16-byte, dk / dv 4-byte alignment; gradient row pitches even and >= 32");
  p.dout = dout;
  p.dq = dq;
  p.dk = static_cast<__nv_bfloat16*>(dk);
  p.dv = static_cast<__nv_bfloat16*>(dv);
  p.ldg = ld_dk;
  p.ldgv = ld_dv;
  LRN_DEVICE(dev);
  return launch(train_attn_bwd_kernel, B * 8, 128, kTaBwdSmem, stream, p);
}

int lrn_col_sum_bf16(const void* A, int64_t ld, int64_t rows, int64_t cols, float* out, lrn_stream_t stream) {
  if (!A || !out) return fail(LRN_ERR_BAD_ARG, "null pointer");
  if (rows <= 0 || cols <= 0 || cols % 64 || ld < cols || ld % 8) return fail(LRN_ERR_BAD_SHAPE, "rows=%lld cols=%lld ld=%lld (cols %% 64 == 0, ld %% 8 == 0)", (long long)rows, (long long)cols, (long long)ld);
  if (misaligned(16, A)) return fail(LRN_ERR_MISALIGNED, "A needs 16-byte alignment");
  LRN_DEVICE(dev);
  LRN_CUDA(cudaMemsetAsync(out, 0, size_t(cols) * 4, stream));
  return launch(col_stats_kernel, stream_grid(col_stats_kernel, int(cols), rows, dev.sms), 256, 0, stream,
                reinterpret_cast<const __nv_bfloat16*>(A), ld, rows, out, nullptr, 0);
}

}  // extern "C"

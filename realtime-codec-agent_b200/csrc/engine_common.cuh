// Shared internals of the engine: the handle, error macros, workspace arena and the TMA
// descriptor cache.  Included by engine.cu and by the kernel launchers (attn_sm100.cuh, vq_sm100.cuh).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <climits>
#include <map>
#include <set>
#include <string>
#include <tuple>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/magicodec_b200.h"
#include "ptx_sm100.cuh"

typedef __nv_bfloat16 bf16;

namespace mc_internal {

inline thread_local std::string g_create_error;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(p);
    }
  }
  return fn;
}

struct Tensor {
  const void* p = nullptr;
  int64_t numel = 0;
};

}  // namespace mc_internal
using mc_internal::Tensor;

struct mc_handle {
  mc_spec spec{};
  int device = 0;
  int num_sms = 148;
  bool finalized = false;
  std::unordered_map<std::string, Tensor> tensors;
  std::string err;
  int64_t launches = 0;
  uint32_t tensor_gen = 0;    // bumped by mc_set_tensor
  int attn_impl = 0, vq_impl = 0;
  int gemm_pair = 1;  // use the cta_group::2 GEMM where the shape allows
  bool fast_epilogue = true;  // mode-specialised, software-pipelined epilogues in the CTA-pair GEMM
  bool attn_p_tmem = true;    // attention: P through tensor memory (v4) instead of shared memory (v3)
  // GEMMs of <= 256 rows with K split over a thread-block cluster (gemm_splitk_sm100.cuh): 0 never, 1 inside streaming
  // sessions (the latency path; stateless mc_encode / mc_decode stay batch-invariant), 2 always
  int split_k = 1;
  bool in_session = false;
  int debug_repeat = 1;
  int fuse_norm = 1;          // RMSNorms in the epilogues of the GEMMs around them: 0 never, 1 few-rows path, 2 / 3 also offline
  bool l2_prefetch = true;    // split-K GEMMs pull the next GEMM's weights into L2 while they run
  bool pdl = true;            // programmatic dependent launch between consecutive kernels of a pass
  bool shared_stem = true;  // overlapping hop-aligned windows share one pass of the conv stack (exact)
  bool exact_cut = true;    // dead-output elimination cuts windows at the exact row, not at multiples of 16 frames (exact)
  // optional per-class device timing (bench.py's roofline): event pairs around each launch
  struct ProfRec { cudaEvent_t a, b; int cls; double flops; double bytes; };
  bool profiling = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> event_pool;
  // kernels whose dynamic-smem limit has been raised on THIS handle's device (the attribute is per device)
  std::set<const void*> smem_configured;
  // workspace arena
  uint8_t* arena = nullptr;
  size_t arena_cap = 0;
  size_t arena_off = 0;
  // TMA descriptor cache
  std::map<std::tuple<const void*, uint64_t, uint64_t, uint64_t, uint32_t, uint32_t>, CUtensorMap> maps;

  int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err = buf;
    return code;
  }
  const Tensor* find(const std::string& name) const {
    auto it = tensors.find(name);
    return it == tensors.end() ? nullptr : &it->second;
  }
  template <typename T>
  const T* ptr(const std::string& name) const {
    return reinterpret_cast<const T*>(tensors.at(name).p);
  }
};

#define MC_CUDA(h, expr)                                                                         \
  do {                                                                                           \
    cudaError_t e__ = (expr);                                                                    \
    if (e__ != cudaSuccess)                                                                      \
      return (h)->fail(MC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define MC_TRY(expr)          \
  do {                        \
    int rc__ = (expr);        \
    if (rc__ != MC_OK) return rc__; \
  } while (0)
// Kernel classes for mc_profile_*: 0 GEMM (tcgen05), 1 attention, 2 VQ search, 3 HBM-bound elementwise
struct McProfScope {
  mc_handle* h; cudaStream_t st; bool on;
  mc_handle::ProfRec rec;
  static cudaEvent_t get_event(mc_handle* h) {
    if (!h->event_pool.empty()) { cudaEvent_t e = h->event_pool.back(); h->event_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
  McProfScope(mc_handle* h_, int cls, double flops, double bytes, cudaStream_t s) : h(h_), st(s), on(h_->profiling) {
    if (!on) return;
    rec.a = get_event(h); rec.b = get_event(h); rec.cls = cls; rec.flops = flops; rec.bytes = bytes;
    cudaEventRecord(rec.a, st);
  }
  ~McProfScope() {
    if (!on) return;
    cudaEventRecord(rec.b, st);
    h->prof.push_back(rec);
  }
};

// cudaFuncAttributeMaxDynamicSharedMemorySize once per (handle, kernel)
template <typename K>
inline int mc_allow_smem(mc_handle* h, K kernel, int bytes) {
  const void* key = reinterpret_cast<const void*>(kernel);
  if (h->smem_configured.count(key)) return MC_OK;
  MC_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  h->smem_configured.insert(key);
  return MC_OK;
}

// Kernel launch with (optionally) the programmatic-stream-serialization attribute; the kernels call pdl_wait()
// before touching anything a predecessor may have written.
template <typename... P, typename... A>
inline void mc_launch(mc_handle* h, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = h->pdl ? 1 : 0;
  (void)cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...);   // errors surface through MC_LAUNCH_CHECK
}

#define MC_LAUNCH_CHECK(h, what)                                                                  \
  do {                                                                                            \
    cudaError_t e__ = cudaGetLastError();                                                         \
    if (e__ != cudaSuccess) return (h)->fail(MC_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e__)); \
    (h)->launches++;                                                                              \
  } while (0)

namespace mc_internal {

// ------------------------------------------------------------------ arena
inline int arena_reserve(mc_handle* h, size_t bytes, cudaStream_t stream) {
  if (bytes <= h->arena_cap) return MC_OK;
  MC_CUDA(h, cudaStreamSynchronize(stream));
  if (h->arena) MC_CUDA(h, cudaFree(h->arena));
  h->arena = nullptr;
  h->arena_cap = 0;
  h->maps.clear();
  const size_t cap = bytes + bytes / 8 + (1u << 20);
  cudaError_t e = cudaMalloc(&h->arena, cap);
  if (e != cudaSuccess) return h->fail(MC_ERR_NOMEM, "workspace cudaMalloc(%zu) failed: %s", cap, cudaGetErrorString(e));
  h->arena_cap = cap;
  return MC_OK;
}
struct Carver {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t at = off;
    off += (bytes + 1023) & ~size_t(1023);
    return at;
  }
};

// ------------------------------------------------------------ TMA helpers
// 2-D tiled, 128B-swizzled tensor map over a row-major [dim1, dim0] array of `esize`-byte elements
// with `row_stride_bytes` between rows (esize 2 = bf16, 4 = fp32).
inline int get_map_2d(mc_handle* h, const void* base, int esize, uint64_t dim0, uint64_t dim1, uint64_t row_stride_bytes,
                      uint32_t box0, uint32_t box1, const CUtensorMap** out, int swizzle_bytes = 128) {
  auto key = std::make_tuple(base, dim0, dim1, row_stride_bytes, (uint32_t)(box0 | (esize << 16) | (swizzle_bytes << 20)), box1);
  auto it = h->maps.find(key);
  if (it != h->maps.end()) {
    *out = &it->second;
    return MC_OK;
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return h->fail(MC_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || row_stride_bytes % 16 != 0 || box0 * esize > (uint32_t)swizzle_bytes)
    return h->fail(MC_ERR_ARG, "TMA operand misaligned (base %p, row stride %llu B, box %u x %d B)", base,
                   (unsigned long long)row_stride_bytes, box0, esize);
  CUtensorMap m;
  cuuint64_t gdim[2] = {dim0, dim1};
  cuuint64_t gstride[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box0, box1};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = enc(&m, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   const_cast<void*>(base), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return h->fail(MC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) dims %llu x %llu box %u x %u esize %d", (int)r,
                   (unsigned long long)dim0, (unsigned long long)dim1, box0, box1, esize);
  auto ins = h->maps.emplace(key, m);
  *out = &ins.first->second;
  return MC_OK;
}
inline int get_map_2d_bf16(mc_handle* h, const void* base, uint64_t dim0, uint64_t dim1, uint32_t box0, uint32_t box1,
                           const CUtensorMap** out, int swizzle_bytes = 128) {
  return get_map_2d(h, base, 2, dim0, dim1, dim0 * 2, box0, box1, out, swizzle_bytes);
}
}  // namespace mc_internal

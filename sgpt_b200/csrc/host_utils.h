// Host-side helpers: error plumbing for the C ABI and TMA tensor-map construction (driver entry point resolved
// at run time through the CUDA runtime, so the library never links libcuda directly).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sgpt {

// thread-local last-error message, returned by sgpt_last_error()
void set_error(const char* fmt, ...);
const char* get_error();

#define SGPT_CHECK_CUDA(expr)                                                               \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      ::sgpt::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return SGPT_ERR_CUDA;                                                                 \
    }                                                                                       \
  } while (0)

#define SGPT_REQUIRE(cond, ...)        \
  do {                                 \
    if (!(cond)) {                     \
      ::sgpt::set_error(__VA_ARGS__);  \
      return SGPT_ERR_INVALID;         \
    }                                  \
  } while (0)

// 2-D bf16 row-major tensor [rows, cols] with row pitch `ld` elements; box = [box_rows, box_cols] with the
// 128-byte swizzle (box_cols must be 64 bf16 = 128 B).  Returns 0 on success.
int make_tma_2d_bf16(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows, uint32_t box_cols);
// Same for fp32 elements (box_cols = 32 floats = 128 B).
int make_tma_2d_f32(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    uint32_t box_cols);
// 1-byte elements (int8 corpus shards and queries)
int make_tma_2d_u8(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                   uint32_t box_cols);

int sm_count();  // multiprocessors of the CURRENT device (cached per device)

// "Do this once per device": kernel attributes such as cudaFuncAttributeMaxDynamicSharedMemorySize are per device, so a
// process that drives several GPUs (one Encoder / CorpusShard per device) must opt in on each of them.
//   static PerDeviceOnce once;  if (once.first()) cudaFuncSetAttribute(...);
struct PerDeviceOnce {
  bool first();            // true exactly once per CUDA device (current device), thread-safe
  unsigned char done_[64] = {};
};

// Programmatic dependent launch is on unless SGPT_PDL=0 is set in the environment (A/B measurements).
bool pdl_enabled();

// Launch with the programmatic-stream-serialization attribute (common.cuh: pdl_wait / pdl_launch_dependents).
template <class... KArgs, class... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace sgpt

// ---------------------------------------------------------------------------------------------------------------
// Launch accounting (always on) and optional per-category CUDA-event timing (sgpt_profile_*).
// ---------------------------------------------------------------------------------------------------------------
namespace sgpt {
enum LaunchCat { kCatEmbed = 0, kCatLayerNorm, kCatGemm, kCatAttention, kCatPool, kCatScores, kCatTopk, kCatMisc, kNumCats };

struct LaunchScope {
  LaunchScope(int cat, cudaStream_t stream);
  ~LaunchScope();
  int cat_;
  cudaStream_t stream_;
  int slot_;
};
}  // namespace sgpt

#include "host_utils.h"

#include <stdlib.h>

#include <cudaTypedefs.h>
#include <stdarg.h>
#include <stdio.h>

#include "../../include/sgpt_b200.h"

namespace sgpt {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

static PFN_cuTensorMapEncodeTiled_v12000 resolve_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

static int make_tma_2d(CUtensorMap* map, CUtensorMapDataType dt, uint64_t esz, const void* base, uint64_t rows,
                       uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols);

int make_tma_2d_bf16(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows, uint32_t box_cols) {
  return make_tma_2d(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, ld, box_rows, box_cols);
}
int make_tma_2d_f32(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    uint32_t box_cols) {
  return make_tma_2d(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, rows, cols, ld, box_rows, box_cols);
}
int make_tma_2d_u8(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                   uint32_t box_cols) {
  return make_tma_2d(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, base, rows, cols, ld, box_rows, box_cols);
}

static int make_tma_2d(CUtensorMap* map, CUtensorMapDataType dt, uint64_t esz, const void* base, uint64_t rows,
                       uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
  auto fn = resolve_encode();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
    return SGPT_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld * esz) % 16 != 0) {
    set_error("TMA operand must be 16-byte aligned with a 16-byte-multiple row pitch (base=%p ld=%llu)", base,
              (unsigned long long)ld);
    return SGPT_ERR_INVALID;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld * esz};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = fn(map, dt, 2, const_cast<void*>(base), gdim, gstride, box, estride,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu ld=%llu box=%ux%u)", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
    return SGPT_ERR_CUDA;
  }
  return SGPT_OK;
}

bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("SGPT_PDL");
    return !(e != nullptr && e[0] == '0');
  }();
  return on;
}

int sm_count() {
  static int n[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (n[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n[dev] = v;  // benign race: every thread writes the same value
  }
  return n[dev];
}

bool PerDeviceOnce::first() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;  // unknown device: just do it again
  return __atomic_exchange_n(&done_[dev], static_cast<unsigned char>(1), __ATOMIC_ACQ_REL) == 0;
}

}  // namespace sgpt

extern "C" const char* sgpt_last_error(void) { return sgpt::get_error(); }

// ---------------------------------------------------------------------------------------------------------------
// launch accounting / profiling
// ---------------------------------------------------------------------------------------------------------------
#include <atomic>
#include <mutex>
#include <vector>

namespace sgpt {

static std::atomic<long long> g_launches[kNumCats];
static std::atomic<bool> g_prof_on{false};
static std::mutex g_prof_mu;
struct ProfRec { cudaEvent_t a, b; int cat; };
static std::vector<ProfRec> g_recs;       // recorded scopes since the last read
static std::vector<ProfRec> g_free;       // recycled event pairs

LaunchScope::LaunchScope(int cat, cudaStream_t stream) : cat_(cat), stream_(stream), slot_(-1) {
  g_launches[cat].fetch_add(1, std::memory_order_relaxed);
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  ProfRec r;
  if (!g_free.empty()) {
    r = g_free.back();
    g_free.pop_back();
  } else {
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  }
  r.cat = cat;
  cudaEventRecord(r.a, stream);
  g_recs.push_back(r);
  slot_ = static_cast<int>(g_recs.size()) - 1;
}

LaunchScope::~LaunchScope() {
  if (slot_ < 0) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (slot_ < static_cast<int>(g_recs.size())) cudaEventRecord(g_recs[slot_].b, stream_);
}

}  // namespace sgpt

extern "C" int sgpt_profile_enable(int on) {
  sgpt::g_prof_on.store(on != 0);
  return SGPT_OK;
}

extern "C" int sgpt_profile_read(double* ms_by_cat, int64_t* timed_launches_by_cat, int64_t* total_launches_by_cat) {
  using namespace sgpt;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int c = 0; c < kNumCats; ++c) {
    if (ms_by_cat) ms_by_cat[c] = 0.0;
    if (timed_launches_by_cat) timed_launches_by_cat[c] = 0;
    if (total_launches_by_cat) total_launches_by_cat[c] = g_launches[c].load();
  }
  for (auto& r : g_recs) {
    if (cudaEventSynchronize(r.b) == cudaSuccess) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
        if (ms_by_cat) ms_by_cat[r.cat] += ms;
        if (timed_launches_by_cat) timed_launches_by_cat[r.cat] += 1;
      }
    }
    g_free.push_back(r);
  }
  g_recs.clear();
  cudaGetLastError();
  return SGPT_OK;
}

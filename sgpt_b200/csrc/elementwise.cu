// HBM-bound row kernels of the encoder: token(+position) embedding gather (F1), LayerNorm (F2/F7), and the
// position-weighted masked pooling with ln_f fused in (P1/P2).  All reductions accumulate in fp32; all global
// accesses are 16-byte vectorised and coalesced along d.
#include <math.h>
#include <stdlib.h>

#include "../../include/sgpt_b200.h"
#include "common.cuh"
#include "host_utils.h"

namespace sgpt {

// Four consecutive elements of a residual-stream row: the stream is fp32 (default) or bf16 (SGPT_RESID_BF16=1, the storage
// the reference's own bf16 checkpoints use: HF keeps hidden_states in the model dtype).  idx4 counts groups of 4 elements.
__device__ __forceinline__ float4 ld_row4(const void* x, size_t idx4, int is_bf16) {
  if (is_bf16) {
    const uint2 u = reinterpret_cast<const uint2*>(x)[idx4];
    return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
  }
  return reinterpret_cast<const float4*>(x)[idx4];
}

// ---------------------------------------------------------------------------------------------------------------
// F1: resid[t, :] = wte[ids[t], :] (+ wpe[pos[t], :])        one warp-wide 16-B vector per thread-iteration
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embed_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ pos,
                                                    const uint4* __restrict__ wte, const uint4* __restrict__ wpe,
                                                    float4* __restrict__ resid, int T, int d8, int vocab,
                                                    int max_pos, int out_bf16) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  // d8 = d / 8: number of 16-B bf16 vectors per row.  Grid-stride over (token, vector).
  const long long total = static_cast<long long>(T) * d8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int t = static_cast<int>(i / d8);
    const int v = static_cast<int>(i - static_cast<long long>(t) * d8);
    int id = __ldg(ids + t);
    id = min(max(id, 0), vocab - 1);
    uint4 e = __ldg(wte + static_cast<size_t>(id) * d8 + v);
    float f[8] = {bf16_lo(e.x), bf16_hi(e.x), bf16_lo(e.y), bf16_hi(e.y),
                  bf16_lo(e.z), bf16_hi(e.z), bf16_lo(e.w), bf16_hi(e.w)};
    if (wpe != nullptr) {
      int p = __ldg(pos + t);
      p = min(max(p, 0), max_pos - 1);
      uint4 q = __ldg(wpe + static_cast<size_t>(p) * d8 + v);
      f[0] += bf16_lo(q.x); f[1] += bf16_hi(q.x); f[2] += bf16_lo(q.y); f[3] += bf16_hi(q.y);
      f[4] += bf16_lo(q.z); f[5] += bf16_hi(q.z); f[6] += bf16_lo(q.w); f[7] += bf16_hi(q.w);
    }
    if (out_bf16) {
      reinterpret_cast<uint4*>(resid)[static_cast<size_t>(t) * d8 + v] =
          make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
    } else {
      float4* dst = resid + (static_cast<size_t>(t) * d8 + v) * 2;
      dst[0] = make_float4(f[0], f[1], f[2], f[3]);
      dst[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// F2/F7: LayerNorm, fp32 in, bf16 out.  TPR threads cooperate on one row; each holds V float4 (row in registers,
// exact two-pass mean/variance like torch's CPU kernel).
// ---------------------------------------------------------------------------------------------------------------
template <int TPR>
__device__ __forceinline__ float group_sum(float v, float* scratch /* [rows_per_cta][TPR/32] */, int row_in_cta,
                                           int lane_in_row) {
  v = warp_sum(v);
  if (TPR == 32) return v;
  constexpr int W = TPR / 32;
  __syncthreads();  // protect scratch reuse between consecutive reductions
  if ((lane_in_row & 31) == 0) scratch[row_in_cta * W + (lane_in_row >> 5)] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < W; ++i) s += scratch[row_in_cta * W + i];
  return s;
}

__device__ __forceinline__ void ln_store(uint2* y, size_t idx, float o0, float o1, float o2, float o3) {
  y[idx] = make_uint2(pack_bf16(o0, o1), pack_bf16(o2, o3));
}
__device__ __forceinline__ void ln_store(float4* y, size_t idx, float o0, float o1, float o2, float o3) {
  y[idx] = make_float4(o0, o1, o2, o3);
}

template <int TPR, int V, class OutT>
__device__ __forceinline__ void layernorm_body(const void* x, int x_bf16, const float4* __restrict__ g,
                                               const float4* __restrict__ b, OutT* y, int T, int d4, float eps,
                                               const int32_t* __restrict__ src_rows = nullptr) {
  constexpr int ROWS = 256 / TPR;
  __shared__ float scratch[ROWS * (TPR / 32) + 1];
  const int row_in_cta = threadIdx.x / TPR;
  const int l = threadIdx.x % TPR;
  const int row = blockIdx.x * ROWS + row_in_cta;
  const bool active = row < T;
  // gather variant: output row `row` is the LayerNorm of input row src_rows[row]
  const int src = (src_rows != nullptr && active) ? __ldg(src_rows + row) : row;
  float4 v[V];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = l + i * TPR;
    v[i] = (active && c < d4) ? ld_row4(x, static_cast<size_t>(src) * d4 + c, x_bf16) : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float inv_d = 1.0f / static_cast<float>(d4 * 4);
  const float mean = group_sum<TPR>(s, scratch, row_in_cta, l) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = l + i * TPR;
    if (c < d4) {
      const float a = v[i].x - mean, bb = v[i].y - mean, cc = v[i].z - mean, dd = v[i].w - mean;
      q += (a * a + bb * bb) + (cc * cc + dd * dd);
    }
  }
  const float var = group_sum<TPR>(q, scratch, row_in_cta, l) * inv_d;
  const float rstd = rsqrtf(var + eps);
  if (!active) return;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = l + i * TPR;
    if (c < d4) {
      const float4 gg = __ldg(g + c), bb = __ldg(b + c);
      const float o0 = (v[i].x - mean) * rstd * gg.x + bb.x;
      const float o1 = (v[i].y - mean) * rstd * gg.y + bb.y;
      const float o2 = (v[i].z - mean) * rstd * gg.z + bb.z;
      const float o3 = (v[i].w - mean) * rstd * gg.w + bb.w;
      ln_store(y, static_cast<size_t>(row) * d4 + c, o0, o1, o2, o3);
    }
  }
}

template <int TPR, int V>
__global__ void __launch_bounds__(256) layernorm_kernel(const void* x, const float4* __restrict__ g,
                                                        const float4* __restrict__ b, uint2* y, int T,
                                                        int d4, float eps, int x_bf16) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  layernorm_body<TPR, V>(x, x_bf16, g, b, y, T, d4, eps);  // (bf16 in: y may alias x — a thread rewrites only what it read)
}

// bf16 residual stream -> bf16 normalised row with 16-byte accesses (8 elements per load / store; the generic kernel above
// would read a bf16 row with 8-byte loads and write with 8-byte stores: measured 1.2x SLOWER than its fp32-input form
// although it moves a third fewer bytes).  May run in place (a thread rewrites only the chunks it read).
template <int TPR, int V8, int MINB = 1>
__global__ void __launch_bounds__(256, MINB) layernorm_bf16_kernel(const uint4* x, const float4* __restrict__ g,
                                                             const float4* __restrict__ b, uint4* y, int T, int d8,
                                                             float eps) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  constexpr int ROWS = 256 / TPR;
  __shared__ float scratch[ROWS * (TPR / 32) + 1];
  const int row_in_cta = threadIdx.x / TPR;
  const int l = threadIdx.x % TPR;
  const int row = blockIdx.x * ROWS + row_in_cta;
  const bool active = row < T;
  float v[V8][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V8; ++i) {
    const int c = l + i * TPR;
    uint4 u = make_uint4(0u, 0u, 0u, 0u);
    if (active && c < d8) u = x[static_cast<size_t>(row) * d8 + c];
    v[i][0] = bf16_lo(u.x); v[i][1] = bf16_hi(u.x); v[i][2] = bf16_lo(u.y); v[i][3] = bf16_hi(u.y);
    v[i][4] = bf16_lo(u.z); v[i][5] = bf16_hi(u.z); v[i][6] = bf16_lo(u.w); v[i][7] = bf16_hi(u.w);
    s += ((v[i][0] + v[i][1]) + (v[i][2] + v[i][3])) + ((v[i][4] + v[i][5]) + (v[i][6] + v[i][7]));
  }
  const float inv_d = 1.0f / static_cast<float>(d8 * 8);
  const float mean = group_sum<TPR>(s, scratch, row_in_cta, l) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V8; ++i) {
    if (l + i * TPR < d8) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float a = v[i][e] - mean;
        q = fmaf(a, a, q);
      }
    }
  }
  const float var = group_sum<TPR>(q, scratch, row_in_cta, l) * inv_d;
  const float rstd = rsqrtf(var + eps);
  if (!active) return;
#pragma unroll
  for (int i = 0; i < V8; ++i) {
    const int c = l + i * TPR;
    if (c < d8) {
      const float4 g0 = __ldg(g + 2 * c), g1 = __ldg(g + 2 * c + 1), b0 = __ldg(b + 2 * c), b1 = __ldg(b + 2 * c + 1);
      const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = (v[i][e] - mean) * rstd * gg[e] + bb[e];
      y[static_cast<size_t>(row) * d8 + c] =
          make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
    }
  }
}

// Persistent form of the kernel above (the default for d <= 768 and 1024 < d <= 4096).  tools/ln_bench.cu measured what
// the one-row-per-group kernel spends its time on: with the gamma / beta loads removed it runs at the speed of a plain copy
// (d 768: 18.6 us against 26.7 us per 32768-row pass; d 2048: 25.5 / 39.0; d 4096: 28.9 / 45.1) — every row re-reads
// 8 bytes of gamma / beta per element through the L1 against 2 bytes of x.  Here a thread group keeps its gamma / beta
// chunks in registers and walks over rows (grid = MINB CTAs per SM), with the next row's loads issued as soon as the
// current row is unpacked: 22.4 / 28.6 / 32.8 us.  May run in place (a group rewrites only rows it has already read, and
// the row it prefetches is a different one).
template <int TPR, bool kWholeCta>
__device__ __forceinline__ float group_sum_once(float v, float* scratch /* [ROWS][TPR/32] of one parity */, int row_in_cta,
                                                int lane_in_row) {
  v = warp_sum(v);
  if (TPR == 32) return v;
  constexpr int W = TPR / 32;
  if ((lane_in_row & 31) == 0) scratch[row_in_cta * W + (lane_in_row >> 5)] = v;
  // one barrier per reduction: the two reductions of a row use two scratch parities, and a group can only come back to
  // a parity after every thread of the group has passed the barrier of the other one
  if (kWholeCta) __syncthreads();
  else asm volatile("bar.sync %0, %1;" ::"r"(row_in_cta + 1), "r"(TPR) : "memory");
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < W; ++i) s += scratch[row_in_cta * W + i];
  return s;
}

template <int TPR, int V8, int MINB>
__global__ void __launch_bounds__(256, MINB) layernorm_bf16_persist_kernel(const uint4* x, const float4* __restrict__ g,
                                                                           const float4* __restrict__ b, uint4* y, int T,
                                                                           int d8, float eps) {
  constexpr int ROWS = 256 / TPR;
  constexpr int W = TPR / 32;
  __shared__ float scratch[2][ROWS * W + 1];
  const int rg = threadIdx.x / TPR;
  const int l = threadIdx.x % TPR;
  // weights: never written by a preceding kernel, so they are fetched before the programmatic-dependency wait
  float gg[V8][8], bb[V8][8];
#pragma unroll
  for (int i = 0; i < V8; ++i) {
    const int c = l + i * TPR;
    float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0, b0 = g0, b1 = g0;
    if (c < d8) {
      g0 = __ldg(g + 2 * c); g1 = __ldg(g + 2 * c + 1); b0 = __ldg(b + 2 * c); b1 = __ldg(b + 2 * c + 1);
    }
    gg[i][0] = g0.x; gg[i][1] = g0.y; gg[i][2] = g0.z; gg[i][3] = g0.w;
    gg[i][4] = g1.x; gg[i][5] = g1.y; gg[i][6] = g1.z; gg[i][7] = g1.w;
    bb[i][0] = b0.x; bb[i][1] = b0.y; bb[i][2] = b0.z; bb[i][3] = b0.w;
    bb[i][4] = b1.x; bb[i][5] = b1.y; bb[i][6] = b1.z; bb[i][7] = b1.w;
  }
  pdl_sync();  // programmatic dependent launch: the residual stream is read only below this line
  const int stride = gridDim.x * ROWS;
  const int cta_row0 = blockIdx.x * ROWS;
  const int n_iter = cta_row0 < T ? (T - cta_row0 + stride - 1) / stride : 0;  // CTA-uniform (the barriers need that)
  const float inv_d = 1.0f / static_cast<float>(d8 * 8);
  uint4 buf[V8];
  auto load_row = [&](int row) {
#pragma unroll
    for (int i = 0; i < V8; ++i) {
      const int c = l + i * TPR;
      buf[i] = make_uint4(0u, 0u, 0u, 0u);
      if (row < T && c < d8) buf[i] = x[static_cast<size_t>(row) * d8 + c];
    }
  };
  int row = cta_row0 + rg;
  load_row(row);
  for (int it = 0; it < n_iter; ++it, row += stride) {
    float v[V8][8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < V8; ++i) {
      const uint4 u = buf[i];
      v[i][0] = bf16_lo(u.x); v[i][1] = bf16_hi(u.x); v[i][2] = bf16_lo(u.y); v[i][3] = bf16_hi(u.y);
      v[i][4] = bf16_lo(u.z); v[i][5] = bf16_hi(u.z); v[i][6] = bf16_lo(u.w); v[i][7] = bf16_hi(u.w);
      s += ((v[i][0] + v[i][1]) + (v[i][2] + v[i][3])) + ((v[i][4] + v[i][5]) + (v[i][6] + v[i][7]));
    }
    load_row(row + stride);  // the raw registers are free: the next row's loads overlap this row's arithmetic
    const float mean = group_sum_once<TPR, TPR == 256>(s, scratch[0], rg, l) * inv_d;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < V8; ++i) {
      if (l + i * TPR < d8) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float a = v[i][e] - mean;
          q = fmaf(a, a, q);
        }
      }
    }
    const float var = group_sum_once<TPR, TPR == 256>(q, scratch[1], rg, l) * inv_d;
    const float rstd = rsqrtf(var + eps);
    if (row < T) {
#pragma unroll
      for (int i = 0; i < V8; ++i) {
        const int c = l + i * TPR;
        if (c < d8) {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = (v[i][e] - mean) * rstd * gg[i][e] + bb[i][e];
          y[static_cast<size_t>(row) * d8 + c] =
              make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
        }
      }
    }
  }
}

// bf16 -> bf16 LayerNorm with the rows staged through shared memory by bulk async copies (UBLKCP): a CTA owns 8 * NS
// consecutive rows and issues the copies of ALL its stages (8 rows = one contiguous 8 * d * 2-byte chunk each) before it
// touches the first one, so every SM has ~190 KB of reads in flight regardless of register pressure.  One warp per row:
// sum, centred sum of squares and the normalised output are three sweeps over the row IN SHARED MEMORY (16-byte, conflict-
// free), the output leaves with 16-byte global stores.  The register-resident kernels above are latency x occupancy
// bound at 3.4 TB/s (32 rows in flight per SM).  May run in place (a stage is read completely before its rows are written;
// stages of different CTAs are disjoint).
template <int NS>
__global__ void __launch_bounds__(256) layernorm_bf16_bulk_kernel(const uint4* x, const float4* __restrict__ g,
                                                                  const float4* __restrict__ b, uint4* y, int T, int d8,
                                                                  float eps) {
  extern __shared__ uint8_t ln_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ln_smem_raw) + 127) & ~uintptr_t(127));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);          // NS barriers (128 bytes reserved)
  uint4* rows = reinterpret_cast<uint4*>(smem + 128);          // [NS][8][d8]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row_base = blockIdx.x * 8 * NS;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  pdl_sync();  // programmatic dependent launch: the residual stream is read only below this line
  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      const int r0 = row_base + 8 * s;
      if (r0 >= T) break;
      const int nr = min(8, T - r0);
      const uint32_t bytes = static_cast<uint32_t>(nr) * static_cast<uint32_t>(d8) * 16u;
      mbar_expect_tx(&bars[s], bytes);
      bulk_load_1d(rows + static_cast<size_t>(s) * 8 * d8, x + static_cast<size_t>(r0) * d8, bytes, &bars[s]);
    }
  }
  const float inv_d = 1.0f / static_cast<float>(d8 * 8);
#pragma unroll 1
  for (int s = 0; s < NS; ++s) {
    const int row = row_base + 8 * s + warp;
    if (row_base + 8 * s >= T) break;  // CTA-uniform
    mbar_wait(&bars[s], 0);
    if (row >= T) continue;            // warp-uniform
    const uint4* r = rows + (static_cast<size_t>(s) * 8 + warp) * d8;
    float sum = 0.f;
    for (int c = lane; c < d8; c += 32) {
      const uint4 u = r[c];
      sum += ((bf16_lo(u.x) + bf16_hi(u.x)) + (bf16_lo(u.y) + bf16_hi(u.y))) +
             ((bf16_lo(u.z) + bf16_hi(u.z)) + (bf16_lo(u.w) + bf16_hi(u.w)));
    }
    const float mean = warp_sum(sum) * inv_d;
    float q = 0.f;
    for (int c = lane; c < d8; c += 32) {
      const uint4 u = r[c];
      const float e[8] = {bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y), bf16_lo(u.z), bf16_hi(u.z), bf16_lo(u.w), bf16_hi(u.w)};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float a = e[i] - mean;
        q = fmaf(a, a, q);
      }
    }
    const float rstd = rsqrtf(warp_sum(q) * inv_d + eps);
    uint4* yo = y + static_cast<size_t>(row) * d8;
    for (int c = lane; c < d8; c += 32) {
      const uint4 u = r[c];
      const float e[8] = {bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y), bf16_lo(u.z), bf16_hi(u.z), bf16_lo(u.w), bf16_hi(u.w)};
      const float4 g0 = __ldg(g + 2 * c), g1 = __ldg(g + 2 * c + 1), b0 = __ldg(b + 2 * c), b1 = __ldg(b + 2 * c + 1);
      const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = (e[i] - mean) * rstd * gg[i] + bb[i];
      yo[c] = make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
    }
  }
}

template <int NS>
static int launch_layernorm_bulk(const uint4* x, const float4* g, const float4* b, uint4* y, int T, int d8, float eps,
                                 cudaStream_t stream) {
  const size_t smem = 128 + 128 + static_cast<size_t>(NS) * 8 * d8 * 16;
  auto kern = layernorm_bf16_bulk_kernel<NS>;
  static PerDeviceOnce attr_once;
  if (attr_once.first()) SGPT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  SGPT_CHECK_CUDA(launch_kernel(kern, dim3((T + 8 * NS - 1) / (8 * NS)), dim3(256), smem, stream, x, g, b, y, T, d8, eps));
  return SGPT_OK;
}

// LayerNorm of a gathered subset of rows: y[m,:] = LN(x[rows[m],:]) (the LM-head input of the cross-encoder scorer)
template <int TPR, int V>
__global__ void __launch_bounds__(256) layernorm_gather_kernel(const void* __restrict__ x,
                                                               const float4* __restrict__ g,
                                                               const float4* __restrict__ b, uint2* __restrict__ y,
                                                               int M, int d4, float eps,
                                                               const int32_t* __restrict__ rows, int x_bf16) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  layernorm_body<TPR, V>(x, x_bf16, g, b, y, M, d4, eps, rows);
}

// fp32 output, may run in place (each thread rewrites exactly the elements it read)
template <int TPR, int V>
__global__ void __launch_bounds__(256) layernorm_f32_kernel(const float4* x, const float4* __restrict__ g,
                                                            const float4* __restrict__ b, float4* y, int T, int d4,
                                                            float eps) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  layernorm_body<TPR, V>(x, 0, g, b, y, T, d4, eps);
}

// Row statistics only (mean, rstd) -> stats[2*t], used by the pooling kernel to apply ln_f on the fly.
template <int TPR, int V>
__global__ void __launch_bounds__(256) row_stats_kernel(const void* __restrict__ x, float2* __restrict__ stats,
                                                        int T, int d4, float eps, int x_bf16) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  constexpr int ROWS = 256 / TPR;
  __shared__ float scratch[ROWS * (TPR / 32) + 1];
  const int row_in_cta = threadIdx.x / TPR;
  const int l = threadIdx.x % TPR;
  const int row = blockIdx.x * ROWS + row_in_cta;
  const bool active = row < T;
  float4 v[V];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = l + i * TPR;
    v[i] = (active && c < d4) ? ld_row4(x, static_cast<size_t>(row) * d4 + c, x_bf16) : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float inv_d = 1.0f / static_cast<float>(d4 * 4);
  const float mean = group_sum<TPR>(s, scratch, row_in_cta, l) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = l + i * TPR;
    if (c < d4) {
      const float a = v[i].x - mean, bb = v[i].y - mean, cc = v[i].z - mean, dd = v[i].w - mean;
      q += (a * a + bb * bb) + (cc * cc + dd * dd);
    }
  }
  const float var = group_sum<TPR>(q, scratch, row_in_cta, l) * inv_d;
  if (active && l == 0) stats[row] = make_float2(mean, rsqrtf(var + eps));
}

// Residual stream -> what the LayerNorm-folded GEMMs consume: xb = bf16(resid) and, per row and 128-column group, the
// partial sums (sum x, sum x^2) (common.cuh ln_row_from_partials).  16 lanes per (row, group): each lane one 32-byte
// vector of 8 floats — 512-byte contiguous reads, 256-byte contiguous writes; used once per forward (after the token
// embedding); inside the blocks the out-proj / c_proj epilogues produce both themselves.
__global__ void __launch_bounds__(256) resid_stats_kernel(const float4* __restrict__ x, uint4* __restrict__ xb,
                                                          float2* __restrict__ stats, int T, int d, int P) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  const long long total = static_cast<long long>(T) * P;
  const int sub = threadIdx.x & 15;
  for (long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 4; i < ((total + 15) & ~15ll);
       i += (static_cast<long long>(gridDim.x) * blockDim.x) >> 4) {
    const bool live = i < total;
    const int t = live ? static_cast<int>(i / P) : 0;
    const int g = live ? static_cast<int>(i - static_cast<long long>(t) * P) : 0;
    const int col = g * 128 + sub * 8;
    float s1 = 0.f, s2 = 0.f;
    if (live && col < d) {
      const float4* src = x + (static_cast<size_t>(t) * d + col) / 4;
      const float4 a = src[0], b = src[1];
      s1 = ((a.x + a.y) + (a.z + a.w)) + ((b.x + b.y) + (b.z + b.w));
      s2 = ((a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w)) + ((b.x * b.x + b.y * b.y) + (b.z * b.z + b.w * b.w));
      xb[(static_cast<size_t>(t) * d + col) / 8] =
          make_uint4(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w), pack_bf16(b.x, b.y), pack_bf16(b.z, b.w));
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (live && sub == 0) stats[i] = make_float2(s1, s2);
  }
}

// Fold a LayerNorm into the linear layer that consumes it (gemm.cuh OpTmaLnBiasActBF16), once per model:
//   w_out[n, k] = bf16(w[n, k] * gamma[k]);  colsum[n] = sum_k float(w_out[n, k]);  bias_out[n] = bias[n] + sum_k beta[k] w[n, k]
// One warp per output row n.
__global__ void __launch_bounds__(256) fold_layernorm_kernel(const __nv_bfloat16* __restrict__ w,
                                                             const float* __restrict__ gamma,
                                                             const float* __restrict__ beta,
                                                             const float* __restrict__ bias,
                                                             __nv_bfloat16* __restrict__ w_out,
                                                             float* __restrict__ colsum, float* __restrict__ bias_out,
                                                             int N, int K) {
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (n >= N) return;
  const int lane = threadIdx.x & 31;
  float cs = 0.f, bs = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float wv = __bfloat162float(w[static_cast<size_t>(n) * K + k]);
    const __nv_bfloat16 f = __float2bfloat16_rn(wv * gamma[k]);
    w_out[static_cast<size_t>(n) * K + k] = f;
    cs += __bfloat162float(f);
    bs = fmaf(beta[k], wv, bs);
  }
  cs = warp_sum(cs);
  bs = warp_sum(bs);
  if (lane == 0) {
    colsum[n] = cs;
    bias_out[n] = bs + (bias != nullptr ? bias[n] : 0.f);
  }
}

// Choose (threads-per-row, float4-per-thread) so the row lives in registers: d <= 1024 -> one warp per row.
#define SGPT_ROW_DISPATCH(KERNEL, d4, T, stream, ...)                                               \
  do {                                                                                              \
    if (d4 <= 32 * 8) {                                                                             \
      const int rows = 8;                                                                           \
      SGPT_CHECK_CUDA(launch_kernel(KERNEL<32, 8>, dim3((T + rows - 1) / rows), dim3(256), 0, stream, __VA_ARGS__)); \
    } else if (d4 <= 128 * 8) {                                                                     \
      const int rows = 2;                                                                           \
      SGPT_CHECK_CUDA(launch_kernel(KERNEL<128, 8>, dim3((T + rows - 1) / rows), dim3(256), 0, stream, __VA_ARGS__)); \
    } else if (d4 <= 256 * 16) {                                                                    \
      SGPT_CHECK_CUDA(launch_kernel(KERNEL<256, 16>, dim3(T), dim3(256), 0, stream, __VA_ARGS__));  \
    } else {                                                                                        \
      set_error("hidden size %d too large for the row kernels", d4 * 4);                            \
      return SGPT_ERR_UNSUPPORTED;                                                                  \
    }                                                                                               \
  } while (0)

// ---------------------------------------------------------------------------------------------------------------
// P1/P2: out[b, :] = sum_t w_t * LN(x_t) / sum_t w_t   over the tokens of sequence b.
//   grid = (B, d / 128); 128 threads = 4 warps; each warp strides over the tokens of the sequence, each lane owns one
//   float4 column group (coalesced 512-B row segments); fp32 accumulators; cross-warp combine through smem.
//   With ln_f:  sum_t w_t ((x_t - mu_t) r_t g + b) = g * sum_t w_t r_t (x_t - mu_t) + b * W.
//   w_t = pos_t + 1 (weightedmean), pw[pos_t] (learnt WeightedMeanPooling), 1 (mean) or [t is last] (lasttoken).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) pool_kernel(const void* __restrict__ x, const int32_t* __restrict__ pos,
                                                   const float* __restrict__ pw, int n_pw,
                                                   const int32_t* __restrict__ cu, const float2* __restrict__ stats,
                                                   const float4* __restrict__ g, const float4* __restrict__ bta,
                                                   float4* __restrict__ out, float* __restrict__ sumsq, int d4,
                                                   int mode, int clamp_den, int accumulate, float out_scale,
                                                   int n_partials, float eps, int x_bf16) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  __shared__ float4 part[4][32];
  __shared__ float wpart[4];
  const int b = blockIdx.x;
  const int col = blockIdx.y * 32 + (threadIdx.x & 31);
  const int warp = threadIdx.x >> 5;
  const int t0 = __ldg(cu + b), t1 = __ldg(cu + b + 1);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float wsum = 0.f;
  const bool col_ok = col < d4;
  for (int t = t0 + warp; t < t1; t += 4) {
    float w;
    if (mode == SGPT_POOL_WEIGHTEDMEAN) {
      // fixed weights i+1 (BDR:259-265), or the learnt table of ST/models/WeightedMeanPooling.py:29 indexed by position
      const int p = __ldg(pos + t);
      w = pw != nullptr ? __ldg(pw + min(p, n_pw - 1)) : static_cast<float>(p + 1);
    }
    else if (mode == SGPT_POOL_LASTTOKEN) w = (t == t1 - 1) ? 1.f : 0.f;
    else w = 1.f;
    wsum += w;
    if (w != 0.f && col_ok) {
      float4 v = ld_row4(x, static_cast<size_t>(t) * d4 + col, x_bf16);
      if (stats != nullptr) {
        // n_partials == 0: stats[t] = (mean, rstd) from row_stats_kernel; > 0: the partial sums left by the kernel that
        // wrote the residual stream (no separate pass over it)
        float2 s;
        if (n_partials > 0) {
          const LnRow lr = ln_row_from_partials(stats, n_partials, 0.25f / static_cast<float>(d4), eps, t, t + 1);
          s = make_float2(lr.rm / lr.r, lr.r);
        } else {
          s = __ldg(stats + t);
        }
        const float wr = w * s.y;
        acc.x += wr * (v.x - s.x); acc.y += wr * (v.y - s.x); acc.z += wr * (v.z - s.x); acc.w += wr * (v.w - s.x);
      } else {
        acc.x += w * v.x; acc.y += w * v.y; acc.z += w * v.z; acc.w += w * v.w;
      }
    }
  }
  part[warp][threadIdx.x & 31] = acc;
  if ((threadIdx.x & 31) == 0) wpart[warp] = wsum;
  __syncthreads();
  if (warp == 0) {
    float4 a = part[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < 4; ++i) {
      const float4 p = part[i][threadIdx.x];
      a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
    }
    float W = (wpart[0] + wpart[1]) + (wpart[2] + wpart[3]);
    float den = W;
    if (clamp_den) den = fmaxf(den, 1e-9f);
    float4 o;
    if (stats != nullptr && col_ok) {
      const float4 gg = __ldg(g + col), bb = __ldg(bta + col);
      o.x = (gg.x * a.x + bb.x * W) / den; o.y = (gg.y * a.y + bb.y * W) / den;
      o.z = (gg.z * a.z + bb.z * W) / den; o.w = (gg.w * a.w + bb.w * W) / den;
    } else {
      o.x = a.x / den; o.y = a.y / den; o.z = a.z / den; o.w = a.w / den;
    }
    // all-layer modes (meanmean / lasttokenmean): out = [out +] out_scale * pooled(this hidden state)
    o.x *= out_scale; o.y *= out_scale; o.z *= out_scale; o.w *= out_scale;
    if (accumulate && col_ok) {
      const float4 prev = out[static_cast<size_t>(b) * d4 + col];
      o.x += prev.x; o.y += prev.y; o.z += prev.z; o.w += prev.w;
    }
    if (col_ok) out[static_cast<size_t>(b) * d4 + col] = o;
    if (sumsq != nullptr) {
      float ss = col_ok ? (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w) : 0.f;
      ss = warp_sum(ss);
      if (threadIdx.x == 0) atomicAdd(sumsq + b, ss);
    }
  }
}

// F7 + P1 (+ P2) in ONE pass over the residual stream for rows of at most 1024 elements: one CTA per sequence, one warp per
// token row.  A warp loads the row (registers), takes its mean / variance with shuffles (exact two-pass), and adds
// w_t r_t (x_t - mu_t) to per-lane accumulators of the columns it owns; the eight warps' accumulators meet in shared
// memory, gamma / beta / the weight sum are applied once, and the L2 normalisation (the CTA holds the whole output row)
// needs no second kernel.  (The two-kernel form — row statistics, then pooling — reads the stream twice.)
__global__ void __launch_bounds__(256) pool_lnf_fused_kernel(const void* __restrict__ x, int x_bf16,
                                                             const int32_t* __restrict__ pos, const float* __restrict__ pw,
                                                             int n_pw, const int32_t* __restrict__ cu,
                                                             const float4* __restrict__ g, const float4* __restrict__ bta,
                                                             float4* __restrict__ out, int d4, float eps, int mode,
                                                             int clamp_den, int normalize, int accumulate, float out_scale) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  __shared__ float4 part[8][256];
  __shared__ float wpart[8];
  __shared__ float s_ss[8];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t0 = __ldg(cu + b), t1 = __ldg(cu + b + 1);
  float4 acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  float wsum = 0.f;
  const float inv_d = 0.25f / static_cast<float>(d4);
  // two token rows per iteration: both rows' loads are in flight before the first reduction
  for (int tb = t0 + warp; tb < t1; tb += 16) {
    float w[2];
    float4 v[2][8];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int t = tb + 8 * r;
      w[r] = 0.f;
      if (t < t1) {
        if (mode == SGPT_POOL_WEIGHTEDMEAN) {
          const int p = __ldg(pos + t);
          w[r] = pw != nullptr ? __ldg(pw + min(p, n_pw - 1)) : static_cast<float>(p + 1);
        } else if (mode == SGPT_POOL_LASTTOKEN) {
          w[r] = (t == t1 - 1) ? 1.f : 0.f;
        } else {
          w[r] = 1.f;
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = lane + 32 * i;
        v[r][i] = (w[r] != 0.f && c < d4) ? ld_row4(x, static_cast<size_t>(t) * d4 + c, x_bf16) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      wsum += w[r];
      if (w[r] == 0.f) continue;  // warp-uniform
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s += (v[r][i].x + v[r][i].y) + (v[r][i].z + v[r][i].w);
      const float mean = warp_sum(s) * inv_d;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (lane + 32 * i < d4) {
          const float a0 = v[r][i].x - mean, a1 = v[r][i].y - mean, a2 = v[r][i].z - mean, a3 = v[r][i].w - mean;
          q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
        }
      }
      const float wr = w[r] * rsqrtf(warp_sum(q) * inv_d + eps);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (lane + 32 * i < d4) {
          acc[i].x += wr * (v[r][i].x - mean); acc[i].y += wr * (v[r][i].y - mean);
          acc[i].z += wr * (v[r][i].z - mean); acc[i].w += wr * (v[r][i].w - mean);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (lane + 32 * i < d4) part[warp][lane + 32 * i] = acc[i];
  if (lane == 0) wpart[warp] = wsum;
  __syncthreads();
  float W = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) W += wpart[i];
  float den = W;
  if (clamp_den) den = fmaxf(den, 1e-9f);
  float ss = 0.f;
  float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
  const int col = threadIdx.x;  // one float4 column group per thread (d4 <= 256)
  if (col < d4) {
    float4 a = part[0][col];
#pragma unroll
    for (int i = 1; i < 8; ++i) {
      const float4 p = part[i][col];
      a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
    }
    const float4 gg = __ldg(g + col), bb = __ldg(bta + col);
    o.x = (gg.x * a.x + bb.x * W) / den; o.y = (gg.y * a.y + bb.y * W) / den;
    o.z = (gg.z * a.z + bb.z * W) / den; o.w = (gg.w * a.w + bb.w * W) / den;
    o.x *= out_scale; o.y *= out_scale; o.z *= out_scale; o.w *= out_scale;
    if (accumulate) {
      const float4 prev = out[static_cast<size_t>(b) * d4 + col];
      o.x += prev.x; o.y += prev.y; o.z += prev.z; o.w += prev.w;
    }
    ss = (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w);
  }
  if (normalize) {
    ss = warp_sum(ss);
    if (lane == 0) s_ss[warp] = ss;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += s_ss[i];
    const float inv = 1.0f / fmaxf(sqrtf(tot), 1e-12f);
    o.x *= inv; o.y *= inv; o.z *= inv; o.w *= inv;
  }
  if (col < d4) out[static_cast<size_t>(b) * d4 + col] = o;
}

// P2: x[b,:] /= max(sqrt(sumsq[b]), 1e-12)      (F.normalize(p=2, dim=1))
__global__ void __launch_bounds__(256) l2_scale_rows_kernel(float4* __restrict__ x, const float* __restrict__ sumsq,
                                                            int B, int d4) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  const long long total = static_cast<long long>(B) * d4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / d4);
    const float inv = 1.0f / fmaxf(sqrtf(__ldg(sumsq + b)), 1e-12f);
    float4 v = x[i];
    v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
    x[i] = v;
  }
}

// Stand-alone P2 for embeddings that went through a head after pooling: one warp per row, any d.
__global__ void __launch_bounds__(256) l2_normalize_rows_kernel(float* __restrict__ x, int B, int d) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= B) return;
  const int lane = threadIdx.x & 31;
  float* r = x + static_cast<size_t>(row) * d;
  float s = 0.f;
  for (int c = lane; c < d; c += 32) s = fmaf(r[c], r[c], s);
  s = warp_sum(s);
  const float inv = 1.0f / fmaxf(sqrtf(s), 1e-12f);
  for (int c = lane; c < d; c += 32) r[c] *= inv;
}

// ---------------------------------------------------------------------------------------------------------------
// Shard maintenance: fp32 -> bf16 rows, and 1 / max(||row||, 1e-12) of the *stored* bf16 rows.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) f32_to_bf16_kernel(const float4* __restrict__ x, uint2* __restrict__ y,
                                                          long long n4) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = x[i];
    y[i] = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
  }
}

__global__ void __launch_bounds__(256) bf16_to_f32_kernel(const uint2* __restrict__ x, float4* __restrict__ y, long long n4) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint2 u = x[i];
    y[i] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
  }
}

// one warp per row; D % 8 == 0
__global__ void __launch_bounds__(256) row_inv_norm_kernel(const uint4* __restrict__ x, float* __restrict__ inv,
                                                           long long n, int d8) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  const long long row = blockIdx.x * 8ll + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int c = lane; c < d8; c += 32) {
    const uint4 e = __ldg(x + row * d8 + c);
    const float f0 = bf16_lo(e.x), f1 = bf16_hi(e.x), f2 = bf16_lo(e.y), f3 = bf16_hi(e.y);
    const float f4 = bf16_lo(e.z), f5 = bf16_hi(e.z), f6 = bf16_lo(e.w), f7 = bf16_hi(e.w);
    s += ((f0 * f0 + f1 * f1) + (f2 * f2 + f3 * f3)) + ((f4 * f4 + f5 * f5) + (f6 * f6 + f7 * f7));
  }
  s = warp_sum(s);
  if (lane == 0) inv[row] = 1.0f / fmaxf(sqrtf(s), 1e-12f);
}

// Symmetric per-row int8 quantization of int8 corpus shards and their queries (include/sgpt_b200.h
// sgpt_quantize_rows_i8 states the arithmetic; the CPU oracle in tests/int8_oracle.py reproduces it bit for bit, which is
// why every step is an explicitly IEEE-rounded intrinsic).  One warp per row, 16 elements per lane step (4 x 16-byte fp32
// loads or 2 x 16-byte bf16 loads, one 16-byte store).  The row is read twice — the maximum first, then the quantization —
// and the second read is served by the L2 that the first one filled.  D % 16 == 0.
template <bool kBF16>
__device__ __forceinline__ void load_row16(const void* x, long long i16, float (&v)[16]) {
  if constexpr (kBF16) {
    const uint4* p = static_cast<const uint4*>(x) + i16 * 2;
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    const uint32_t u[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[2 * j] = bf16_lo(u[j]);
      v[2 * j + 1] = bf16_hi(u[j]);
    }
  } else {
    const float4* p = static_cast<const float4*>(x) + i16 * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 f = __ldg(p + j);
      v[4 * j] = f.x;
      v[4 * j + 1] = f.y;
      v[4 * j + 2] = f.z;
      v[4 * j + 3] = f.w;
    }
  }
}

template <bool kBF16>
__global__ void __launch_bounds__(256) quantize_rows_i8_kernel(const void* __restrict__ x, uint4* __restrict__ out,
                                                               float* __restrict__ scale, float* __restrict__ inv,
                                                               long long n, int d16) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  const long long row = blockIdx.x * 8ll + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  float a = 0.f;
  for (int c = lane; c < d16; c += 32) {
    float v[16];
    load_row16<kBF16>(x, row * d16 + c, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) a = fmaxf(a, fabsf(v[i]));
  }
  a = warp_max(a);
  const float s = __fdiv_rn(a, 127.0f);
  int n2 = 0;
  for (int c = lane; c < d16; c += 32) {
    float v[16];
    load_row16<kBF16>(x, row * d16 + c, v);
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      // s == 0 only for an all-zero row (or one whose maximum underflows): every code is 0 then
      const int q = s > 0.f ? static_cast<int>(fminf(fmaxf(rintf(__fdiv_rn(v[i], s)), -127.f), 127.f)) : 0;
      n2 += q * q;
      w[i >> 2] |= (static_cast<uint32_t>(q) & 0xffu) << (8 * (i & 3));
    }
    out[row * d16 + c] = make_uint4(w[0], w[1], w[2], w[3]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);  // exact: n2 <= 127^2 x 65536 < 2^31
  if (lane == 0) {
    scale[row] = s;
    inv[row] = __fdiv_rn(1.0f, fmaxf(__fsqrt_rn(__int2float_rn(n2)), 1e-12f));
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Sentence-embedding head: y[b,o] = act(sum_k x[b,k] * w[o,k] + bias[o]) in fp32 (ST/models/Dense.py:40-43 applied to
// the pooled embedding).  B x in x out is tiny (<= a few hundred MFLOP), so this is a plain smem-tiled SIMT kernel kept
// in fp32 end to end: 32 x 32 output tile per CTA, 256 threads x (2 x 2) outputs, K in steps of 32, fixed summation
// order (deterministic).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dense_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                    const float* __restrict__ bias, float* __restrict__ y, int B,
                                                    int K, int N, int act) {
  pdl_sync();  // programmatic dependent launch: see common.cuh
  __shared__ float xs[32][33];
  __shared__ float ws[32][33];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int o0 = blockIdx.x * 32, b0 = blockIdx.y * 32;
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = threadIdx.x + i * 256;  // 0..1023
      const int r = e >> 5, c = e & 31;
      const int k = k0 + c;
      xs[r][c] = (b0 + r < B && k < K) ? x[static_cast<size_t>(b0 + r) * K + k] : 0.f;
      ws[r][c] = (o0 + r < N && k < K) ? __ldg(w + static_cast<size_t>(o0 + r) * K + k) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int c = 0; c < 32; ++c) {
      const float x0 = xs[ty][c], x1 = xs[ty + 16][c];
      const float w0 = ws[tx][c], w1 = ws[tx + 16][c];
      acc[0][0] = fmaf(x0, w0, acc[0][0]); acc[0][1] = fmaf(x0, w1, acc[0][1]);
      acc[1][0] = fmaf(x1, w0, acc[1][0]); acc[1][1] = fmaf(x1, w1, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int b = b0 + ty + 16 * i, o = o0 + tx + 16 * j;
      if (b < B && o < N) {
        float v = acc[i][j] + (bias != nullptr ? __ldg(bias + o) : 0.f);
        if (act == SGPT_ACT_TANH) v = tanhf(v);
        else if (act == SGPT_ACT_RELU) v = fmaxf(v, 0.f);
        else if (act == SGPT_ACT_SIGMOID) v = 1.0f / (1.0f + expf(-v));
        y[static_cast<size_t>(b) * N + o] = v;
      }
    }
}

static inline int grid_for(long long work_items, int threads) {
  long long blocks = (work_items + threads - 1) / threads;
  const long long cap = static_cast<long long>(sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace sgpt

using namespace sgpt;

extern "C" int sgpt_embed_tokens(const int32_t* ids, const int32_t* pos, const void* wte, const void* wpe,
                                 float* resid, int T, int d, int vocab, int max_pos, sgpt_stream_t stream_) {
  return sgpt_embed_tokens_ex(ids, pos, wte, wpe, resid, T, d, vocab, max_pos, 0, stream_);
}

extern "C" int sgpt_embed_tokens_ex(const int32_t* ids, const int32_t* pos, const void* wte, const void* wpe,
                                    void* resid, int T, int d, int vocab, int max_pos, int resid_bf16,
                                    sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(T >= 0 && d > 0 && d % 8 == 0, "sgpt_embed_tokens: d=%d must be a positive multiple of 8", d);
  SGPT_REQUIRE(wpe == nullptr || pos != nullptr, "sgpt_embed_tokens: pos required when wpe is given");
  if (T == 0) return SGPT_OK;
  const int d8 = d / 8;
  LaunchScope _ls(kCatEmbed, stream);
  SGPT_CHECK_CUDA(launch_kernel(embed_kernel, dim3(grid_for(static_cast<long long>(T) * d8, 256)), dim3(256), 0, stream,
                                ids, pos, static_cast<const uint4*>(wte), static_cast<const uint4*>(wpe),
                                reinterpret_cast<float4*>(resid), T, d8, vocab, max_pos, resid_bf16));
  return SGPT_OK;
}

extern "C" int sgpt_layernorm(const float* x, const float* gamma, const float* beta, void* y, int T, int d,
                              float eps, sgpt_stream_t stream_) {
  return sgpt_layernorm_ex(x, 0, gamma, beta, y, T, d, eps, stream_);
}

extern "C" int sgpt_layernorm_ex(const void* x, int x_bf16, const float* gamma, const float* beta, void* y, int T, int d,
                                 float eps, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(T >= 0 && d > 0 && d % 4 == 0, "sgpt_layernorm: d=%d must be a positive multiple of 4", d);
  if (T == 0) return SGPT_OK;
  const int d4 = d / 4;
  LaunchScope _ls(kCatLayerNorm, stream);
  if (x_bf16 && d % 8 == 0 && d <= 8192) {
    const int d8 = d / 8;
    const uint4* xi = static_cast<const uint4*>(x);
    const float4 *gi = reinterpret_cast<const float4*>(gamma), *bi = reinterpret_cast<const float4*>(beta);
    uint4* yo = static_cast<uint4*>(y);
    // SGPT_LN_BULK=1: rows staged through shared memory by bulk async copies — measured SLOWER (0.98 vs 0.79 ms per 125M
    // step in the same call; 1.3B 2.4 -> 2.4, bloom 3.4 -> 4.2 ms), off by default
    static const bool bulk = [] { const char* e = getenv("SGPT_LN_BULK"); return e != nullptr && e[0] == '1'; }();
    if (bulk) {
      // stages of 8 rows; as many per CTA as ~48 KB hold (d 768: 4, d 2048: 1, d 4096: 1)
      const size_t stage = static_cast<size_t>(8) * d8 * 16;
      if (4 * stage <= 56 * 1024) return launch_layernorm_bulk<4>(xi, gi, bi, yo, T, d8, eps, stream);
      if (2 * stage <= 56 * 1024) return launch_layernorm_bulk<2>(xi, gi, bi, yo, T, d8, eps, stream);
      return launch_layernorm_bulk<1>(xi, gi, bi, yo, T, d8, eps, stream);
    }
    // Persistent groups with gamma / beta in registers (see layernorm_bf16_persist_kernel); SGPT_LN_PERSIST=0 selects the
    // one-row-per-group kernels.  Widths without a persistent instance (768 < d <= 1024, d > 4096) use those as well.
    static const bool persist = [] { const char* e = getenv("SGPT_LN_PERSIST"); return !(e != nullptr && e[0] == '0'); }();
    const int sms = sm_count();
    auto grid_for_rows = [&](int rows_per_cta, int ctas_per_sm) {
      const int need = (T + rows_per_cta - 1) / rows_per_cta;
      return dim3(static_cast<unsigned>(need < sms * ctas_per_sm ? need : sms * ctas_per_sm));
    };
    if (persist && d8 <= 32 * 3)
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_persist_kernel<32, 3, 2>, grid_for_rows(8, 2), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    else if (persist && d8 > 32 * 4 && d8 <= 128 * 2)
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_persist_kernel<128, 2, 3>, grid_for_rows(2, 3), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    else if (persist && d8 > 128 * 2 && d8 <= 256 * 2)
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_persist_kernel<256, 2, 3>, grid_for_rows(1, 3), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    else if (d8 <= 32 * 3)
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_kernel<32, 3, 6>, dim3((T + 7) / 8), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    else if (d8 <= 32 * 4)
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_kernel<32, 4>, dim3((T + 7) / 8), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    else if (d8 <= 128 * 4)
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_kernel<128, 4>, dim3((T + 1) / 2), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    else
      SGPT_CHECK_CUDA(launch_kernel(layernorm_bf16_kernel<256, 4>, dim3(T), dim3(256), 0, stream, xi, gi, bi, yo, T, d8, eps));
    return SGPT_OK;
  }
  SGPT_ROW_DISPATCH(layernorm_kernel, d4, T, stream, x,
                    reinterpret_cast<const float4*>(gamma), reinterpret_cast<const float4*>(beta),
                    static_cast<uint2*>(y), T, d4, eps, x_bf16);
  SGPT_CHECK_CUDA(cudaGetLastError());
  return SGPT_OK;
}

extern "C" int sgpt_layernorm_gather(const float* x, const int32_t* row_idx, const float* gamma, const float* beta, void* y,
                                     int M, int d, float eps, sgpt_stream_t stream_) {
  return sgpt_layernorm_gather_ex(x, 0, row_idx, gamma, beta, y, M, d, eps, stream_);
}

extern "C" int sgpt_layernorm_gather_ex(const void* x, int x_bf16, const int32_t* row_idx, const float* gamma,
                                        const float* beta, void* y, int M, int d, float eps, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(M >= 0 && d > 0 && d % 4 == 0, "sgpt_layernorm_gather: d=%d must be a positive multiple of 4", d);
  SGPT_REQUIRE(row_idx != nullptr, "sgpt_layernorm_gather: rows required");  // (`rows` is a local of the macro below)
  if (M == 0) return SGPT_OK;
  const int d4 = d / 4;
  LaunchScope _ls(kCatLayerNorm, stream);
  SGPT_ROW_DISPATCH(layernorm_gather_kernel, d4, M, stream, x,
                    reinterpret_cast<const float4*>(gamma), reinterpret_cast<const float4*>(beta),
                    static_cast<uint2*>(y), M, d4, eps, row_idx, x_bf16);
  SGPT_CHECK_CUDA(cudaGetLastError());
  return SGPT_OK;
}

extern "C" int sgpt_layernorm_f32_inplace(float* x, const float* gamma, const float* beta, int T, int d, float eps,
                                          sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(T >= 0 && d > 0 && d % 4 == 0, "sgpt_layernorm_f32_inplace: d=%d must be a positive multiple of 4", d);
  if (T == 0) return SGPT_OK;
  const int d4 = d / 4;
  LaunchScope _ls(kCatLayerNorm, stream);
  SGPT_ROW_DISPATCH(layernorm_f32_kernel, d4, T, stream, reinterpret_cast<const float4*>(x),
                    reinterpret_cast<const float4*>(gamma), reinterpret_cast<const float4*>(beta),
                    reinterpret_cast<float4*>(x), T, d4, eps);
  SGPT_CHECK_CUDA(cudaGetLastError());
  return SGPT_OK;
}

// shared launcher: `stats` is either (mean, rstd) per row (n_partials == 0) or the [T, n_partials] partial sums
static int pool_launch(const void* x, int x_bf16, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                       const float* beta, float eps, const float* pos_weights, int n_pos_weights, float* out,
                       const float2* stats, int n_partials, float* sumsq, int B, int d, int mode, int clamp_denominator,
                       int normalize, int accumulate, float out_scale, cudaStream_t stream) {
  const int d4 = d / 4;
  if (normalize) SGPT_CHECK_CUDA(cudaMemsetAsync(sumsq, 0, sizeof(float) * B, stream));
  dim3 grid(B, (d4 + 31) / 32);
  SGPT_CHECK_CUDA(launch_kernel(pool_kernel, grid, dim3(128), 0, stream, x, pos,
                                pos_weights, n_pos_weights, cu_seqlens, stats, reinterpret_cast<const float4*>(gamma),
                                reinterpret_cast<const float4*>(beta), reinterpret_cast<float4*>(out),
                                normalize ? sumsq : nullptr, d4, mode, clamp_denominator, accumulate, out_scale,
                                n_partials, eps, x_bf16));
  if (normalize) {
    SGPT_CHECK_CUDA(launch_kernel(l2_scale_rows_kernel, dim3(grid_for(static_cast<long long>(B) * d4, 256)), dim3(256),
                                  0, stream, reinterpret_cast<float4*>(out), sumsq, B, d4));
  }
  return SGPT_OK;
}

static int pool_check(const int32_t* pos, const float* gamma, const float* beta, const float* pos_weights,
                      int n_pos_weights, int d, int mode) {
  SGPT_REQUIRE(d > 0 && d % 4 == 0, "sgpt_pool: d=%d must be a positive multiple of 4", d);
  SGPT_REQUIRE(mode >= SGPT_POOL_MEAN && mode <= SGPT_POOL_LASTTOKEN,
               "sgpt_pool: mode %d is not a single-hidden-state pooling mode", mode);
  SGPT_REQUIRE(mode != SGPT_POOL_WEIGHTEDMEAN || pos != nullptr, "sgpt_pool: weightedmean needs pos");
  SGPT_REQUIRE(pos_weights == nullptr || (mode == SGPT_POOL_WEIGHTEDMEAN && n_pos_weights > 0),
               "sgpt_pool: a position-weight table needs mode WEIGHTEDMEAN and n_pos_weights > 0");
  SGPT_REQUIRE((gamma == nullptr) == (beta == nullptr), "sgpt_pool: gamma and beta must be given together");
  return SGPT_OK;
}

extern "C" int sgpt_pool_ex(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                            const float* beta, float eps, const float* pos_weights, int n_pos_weights, float* out,
                            float* row_stats_ws, int B, int T, int d, int mode, int clamp_denominator, int normalize,
                            int accumulate, float out_scale, sgpt_stream_t stream_) {
  return sgpt_pool_ex2(x, 0, pos, cu_seqlens, gamma, beta, eps, pos_weights, n_pos_weights, out, row_stats_ws, B, T, d, mode,
                       clamp_denominator, normalize, accumulate, out_scale, stream_);
}

extern "C" int sgpt_pool_ex2(const void* x, int x_bf16, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                             const float* beta, float eps, const float* pos_weights, int n_pos_weights, float* out,
                             float* row_stats_ws, int B, int T, int d, int mode, int clamp_denominator, int normalize,
                             int accumulate, float out_scale, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = pool_check(pos, gamma, beta, pos_weights, n_pos_weights, d, mode);
  if (rc != SGPT_OK) return rc;
  SGPT_REQUIRE(gamma == nullptr || row_stats_ws != nullptr, "sgpt_pool: ln_f fusion needs row_stats_ws");
  SGPT_REQUIRE(!normalize || row_stats_ws != nullptr, "sgpt_pool: normalize needs row_stats_ws (>= 2*T + B floats)");
  if (B == 0) return SGPT_OK;
  LaunchScope _ls(kCatPool, stream);
  const int d4 = d / 4;
  if (gamma != nullptr && d4 <= 256) {
    // ln_f + pooling (+ normalisation) in one pass over the residual stream
    SGPT_CHECK_CUDA(launch_kernel(pool_lnf_fused_kernel, dim3(B), dim3(256), 0, stream, x, x_bf16, pos, pos_weights,
                                  n_pos_weights, cu_seqlens, reinterpret_cast<const float4*>(gamma),
                                  reinterpret_cast<const float4*>(beta), reinterpret_cast<float4*>(out), d4, eps, mode,
                                  clamp_denominator, normalize, accumulate, out_scale));
    return SGPT_OK;
  }
  const float2* stats = nullptr;
  if (gamma != nullptr && T > 0) {
    SGPT_ROW_DISPATCH(row_stats_kernel, d4, T, stream, x,
                      reinterpret_cast<float2*>(row_stats_ws), T, d4, eps, x_bf16);
    SGPT_CHECK_CUDA(cudaGetLastError());
    stats = reinterpret_cast<const float2*>(row_stats_ws);
  }
  return pool_launch(x, x_bf16, pos, cu_seqlens, gamma, beta, eps, pos_weights, n_pos_weights, out, stats, 0,
                     normalize ? row_stats_ws + 2 * static_cast<size_t>(T) : nullptr, B, d, mode, clamp_denominator,
                     normalize, accumulate, out_scale, stream);
}

// ln_f + pooling from the partial row sums the residual-producing kernels left behind (one pass over the residual
// stream instead of two): partial_stats float2[T, n_partials], sumsq_ws float[B] (only with normalize).
extern "C" int sgpt_pool_partials(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                                  const float* beta, float eps, const float* pos_weights, int n_pos_weights, float* out,
                                  const float* partial_stats, int n_partials, float* sumsq_ws, int B, int T, int d,
                                  int mode, int clamp_denominator, int normalize, int accumulate, float out_scale,
                                  sgpt_stream_t stream_) {
  (void)T;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = pool_check(pos, gamma, beta, pos_weights, n_pos_weights, d, mode);
  if (rc != SGPT_OK) return rc;
  SGPT_REQUIRE(gamma != nullptr && partial_stats != nullptr && n_partials > 0,
               "sgpt_pool_partials: gamma/beta and the partial row sums are required");
  SGPT_REQUIRE(!normalize || sumsq_ws != nullptr, "sgpt_pool_partials: normalize needs sumsq_ws");
  if (B == 0) return SGPT_OK;
  LaunchScope _ls(kCatPool, stream);
  return pool_launch(x, 0, pos, cu_seqlens, gamma, beta, eps, pos_weights, n_pos_weights, out,
                     reinterpret_cast<const float2*>(partial_stats), n_partials, sumsq_ws, B, d, mode, clamp_denominator,
                     normalize, accumulate, out_scale, stream);
}

extern "C" int sgpt_resid_stats(const float* resid, void* xb, float* stats, int T, int d, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(T >= 0 && d > 0 && d % 8 == 0, "sgpt_resid_stats: d=%d must be a positive multiple of 8", d);
  if (T == 0) return SGPT_OK;
  const int P = (d + 127) / 128;
  LaunchScope _ls(kCatLayerNorm, stream);
  SGPT_CHECK_CUDA(launch_kernel(resid_stats_kernel, dim3(grid_for(static_cast<long long>(T) * P * 16, 256)), dim3(256), 0,
                                stream, reinterpret_cast<const float4*>(resid), static_cast<uint4*>(xb),
                                reinterpret_cast<float2*>(stats), T, d, P));
  return SGPT_OK;
}

extern "C" int sgpt_fold_layernorm(const void* w, const float* gamma, const float* beta, const float* bias, void* w_out,
                                   float* colsum_out, float* bias_out, int N, int K, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(N > 0 && K > 0 && w != nullptr && gamma != nullptr && beta != nullptr && w_out != nullptr &&
                   colsum_out != nullptr && bias_out != nullptr, "sgpt_fold_layernorm: bad arguments");
  LaunchScope _ls(kCatMisc, stream);
  fold_layernorm_kernel<<<(N + 7) / 8, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(w), gamma, beta, bias,
                                                         static_cast<__nv_bfloat16*>(w_out), colsum_out, bias_out, N, K);
  SGPT_CHECK_CUDA(cudaGetLastError());
  return SGPT_OK;
}

extern "C" int sgpt_pool_accumulate(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                                    const float* beta, float eps, float* out, float* row_stats_ws, int B, int T, int d,
                                    int mode, int clamp_denominator, int normalize, int accumulate, float out_scale,
                                    sgpt_stream_t stream_) {
  return sgpt_pool_ex(x, pos, cu_seqlens, gamma, beta, eps, nullptr, 0, out, row_stats_ws, B, T, d, mode,
                      clamp_denominator, normalize, accumulate, out_scale, stream_);
}

extern "C" int sgpt_pool(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                         const float* beta, float eps, float* out, float* row_stats_ws, int B, int T, int d, int mode,
                         int clamp_denominator, int normalize, sgpt_stream_t stream_) {
  return sgpt_pool_ex(x, pos, cu_seqlens, gamma, beta, eps, nullptr, 0, out, row_stats_ws, B, T, d, mode,
                      clamp_denominator, normalize, /*accumulate=*/0, /*out_scale=*/1.0f, stream_);
}

extern "C" int sgpt_normalize_rows(float* x, int B, int d, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(B >= 0 && d > 0, "sgpt_normalize_rows: bad sizes");
  if (B == 0) return SGPT_OK;
  LaunchScope _ls(kCatPool, stream);
  SGPT_CHECK_CUDA(launch_kernel(l2_normalize_rows_kernel, dim3((B + 7) / 8), dim3(256), 0, stream, x, B, d));
  return SGPT_OK;
}

extern "C" int sgpt_dense(const float* x, const float* w, const float* bias, float* y, int B, int in_features,
                          int out_features, int activation, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(B >= 0 && in_features > 0 && out_features > 0, "sgpt_dense: bad sizes");
  SGPT_REQUIRE(activation >= SGPT_ACT_IDENTITY && activation <= SGPT_ACT_SIGMOID, "sgpt_dense: unknown activation %d",
               activation);
  SGPT_REQUIRE(x != y, "sgpt_dense: x and y must not alias");
  if (B == 0) return SGPT_OK;
  LaunchScope _ls(kCatPool, stream);
  dim3 grid((out_features + 31) / 32, (B + 31) / 32);
  SGPT_CHECK_CUDA(launch_kernel(dense_kernel, grid, dim3(256), 0, stream, x, w, bias, y, B, in_features, out_features,
                                activation));
  return SGPT_OK;
}

extern "C" int sgpt_row_inv_norms(const void* x, float* inv_norm, int64_t n, int D, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(D > 0 && D % 8 == 0, "sgpt_row_inv_norms: D=%d must be a positive multiple of 8", D);
  if (n == 0) return SGPT_OK;
  const long long blocks = (n + 7) / 8;
  SGPT_REQUIRE(blocks < (1ll << 31), "sgpt_row_inv_norms: too many rows");
  LaunchScope _ls(kCatMisc, stream);
  SGPT_CHECK_CUDA(launch_kernel(row_inv_norm_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, stream,
                                static_cast<const uint4*>(x), inv_norm, n, D / 8));
  return SGPT_OK;
}

extern "C" int sgpt_bf16_to_f32(const void* x, float* y, int64_t count, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(count >= 0 && count % 4 == 0, "sgpt_bf16_to_f32: count must be a multiple of 4");
  if (count == 0) return SGPT_OK;
  LaunchScope _ls(kCatMisc, stream);
  SGPT_CHECK_CUDA(launch_kernel(bf16_to_f32_kernel, dim3(grid_for(count / 4, 256)), dim3(256), 0, stream,
                                static_cast<const uint2*>(x), reinterpret_cast<float4*>(y), count / 4));
  return SGPT_OK;
}

extern "C" int sgpt_f32_to_bf16(const float* x, void* y, int64_t count, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(count >= 0 && count % 4 == 0, "sgpt_f32_to_bf16: count must be a multiple of 4");
  if (count == 0) return SGPT_OK;
  LaunchScope _ls(kCatMisc, stream);
  SGPT_CHECK_CUDA(launch_kernel(f32_to_bf16_kernel, dim3(grid_for(count / 4, 256)), dim3(256), 0, stream,
                                reinterpret_cast<const float4*>(x), static_cast<uint2*>(y), count / 4));
  return SGPT_OK;
}

extern "C" int sgpt_quantize_rows_i8(const void* x, int x_is_bf16, int64_t n, int D, int8_t* out, float* scale,
                                     float* inv_norm, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(n >= 0 && D > 0 && D % 16 == 0 && D <= 65536,
               "sgpt_quantize_rows_i8: D=%d must be a positive multiple of 16 and <= 65536 (n=%lld)", D, (long long)n);
  SGPT_REQUIRE(n == 0 || (x != nullptr && out != nullptr && scale != nullptr && inv_norm != nullptr),
               "sgpt_quantize_rows_i8: null argument");
  if (n == 0) return SGPT_OK;
  const long long blocks = (n + 7) / 8;
  SGPT_REQUIRE(blocks < (1ll << 31), "sgpt_quantize_rows_i8: too many rows");
  LaunchScope _ls(kCatMisc, stream);
  auto kern = x_is_bf16 ? quantize_rows_i8_kernel<true> : quantize_rows_i8_kernel<false>;
  SGPT_CHECK_CUDA(launch_kernel(kern, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, stream, x,
                                reinterpret_cast<uint4*>(out), scale, inv_norm, static_cast<long long>(n), D / 16));
  return SGPT_OK;
}

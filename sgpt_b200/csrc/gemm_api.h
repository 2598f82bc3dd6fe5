// Internal (C++) entry points of gemm.cu used by search.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sgpt {

constexpr int kSimBN = 256;  // corpus rows per similarity tile (N-tile width of the query x corpus GEMM)

// Geometry of the candidate lists the filter GEMM writes for a launch over `tiles` corpus tiles: every (CTA, column
// half) is a group with a private list of `L` entries per query (worst case: every score of every visited tile).
struct FilterGeometry {
  int groups;  // 2 x CTAs (nq <= 128) or 2 x CTA pairs (128 < nq <= 256) of the launch
  int L;       // entries per (query, group) list
};
FilterGeometry filter_geometry(long long tiles, int nq);

// Similarity GEMM whose epilogue appends every score >= tau[q] (tau == nullptr: every score) as (score bits, local doc
// index) to the list cand[q * stride_q + (group0 + g) * L + ...] — scores >= tau_hi[q] at its front, the others at its
// back (tau_hi == nullptr: all at the front) — and writes counts / counts_back[(group0 + g) * nq + q] for the groups g of
// this launch (filter_geometry of the visited tile count).  tile_mode/tile_stride select the corpus tiles visited
// (gemm.cuh TileMap).  nq <= 256 (above 128: CTA pairs, M = 256).  elem: SGPT_ELEM_BF16 or SGPT_ELEM_I8 (Q and C both
// of that type; int8 launches take the s32 accumulator through the same scaling).
int launch_filter_candidates(const void* Q, const void* C, const float* q_scale, const float* c_scale,
                             const float* tau, const float* tau_hi, uint2* cand, int* counts, int* counts_back,
                             long long stride_q, int L, int group0, int nq, int n, int D, int elem, int tile_mode,
                             int tile_stride, cudaStream_t stream);

// The same GEMM over every tile_stride-th corpus tile in sample mode: pool[q * stride_p + g * Lp + ...] receives the
// maximum score of every 4 consecutive documents the group visited (filter_geometry(sampled tiles).L / 4 floats per list,
// unused slots = 0xffffffff).  Input of launch_tau_select (topk.cuh).
int launch_sample_maxima(const void* Q, const void* C, const float* q_scale, const float* c_scale, float* pool,
                         long long stride_p, int Lp, int nq, int n, int D, int elem, int tile_stride,
                         cudaStream_t stream);

// sgpt_scores for either element type: scores[q, j] = fixnan(acc * q_scale[q] * c_scale[j]) as fp32 [nq, lds].
int launch_scores(const void* Q, const void* C, const float* q_scale, const float* c_scale, float* scores, int64_t lds,
                  int nq, int64_t n, int D, int elem, cudaStream_t stream);

}  // namespace sgpt

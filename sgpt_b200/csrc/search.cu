// S1+S2 for one corpus shard without materialising the [nq, n] score matrix.
//
// Two passes of the same tcgen05 similarity GEMM:
//   pass A  scans a strided SAMPLE of the corpus tiles (every s-th 256-document tile, at most one tile per SM, so the pass
//           is a single round) and keeps, per query, the maximum score of every 4 consecutive documents (gemm.cuh
//           EpiFilterRows, sample mode).  tau[q] = the k-th largest of those maxima (tau_select_kernel: ten block-wide
//           counting steps over register-resident keys) is a valid lower bound of the final k-th best score, because each
//           maximum is the score of a distinct real document.
//           A second, higher threshold tau_hi[q] = the k_hi-th largest maximum, k_hi = 2.5 k x (sample fraction), is the
//           level above which ~2.5 k documents of the WHOLE shard are expected.
//   pass B  scans ALL tiles — the sampled ones again: 1/s <= 1/8 of the shard, cheaper than carrying the sample's winners
//           along as a seed list through a full selection — and its epilogue keeps only scores >= tau[q] (expected
//           ~1.1 k s survivors per query), those >= tau_hi[q] at the front of the thread's list and the others at its back;
//           the score matrix never reaches HBM.
//   final   exact selection + sort -> top-k.  It reads the FRONT parts only (~2.5 k entries per query instead of ~30 k) and
//           touches the back parts only for a query whose front parts hold fewer than k entries (tau_hi is a statistical
//           estimate; tau is the guarantee), so the result is exact either way.
// Candidates live in per-(query, group) lists, one group per (CTA, tile half) of the GEMM (gemm.cuh EpiFilterRows): no
// atomics, and every list is sized for the worst case (every score admitted), so no overflow path exists; only the
// touched prefix of each list ever generates memory traffic.  Small shards take the direct path (dense scores + select).
#include "../../include/sgpt_b200.h"
#include "gemm_api.h"
#include "host_utils.h"
#include "topk.cuh"

#include <stdlib.h>
#include <string.h>

using namespace sgpt;

namespace {

inline int64_t padded_cols(int64_t n) { return (n + 3) & ~int64_t(3); }
inline int64_t align256(int64_t x) { return (x + 255) & ~int64_t(255); }

struct Plan {
  bool two_pass;
  int stride;          // tile stride of the sample
  int Lp;              // sampled maxima per (query, group)
  int64_t stride_p;    // sampled maxima per query (= groups of pass A x Lp)
  FilterGeometry gb;   // pass-B candidate lists
  int64_t stride_b;    // candidate entries per query block
  int k_hi;            // rank (among the sampled maxima) of the upper threshold
};

Plan make_plan(int nq, int64_t n, int k) {
  Plan p{};
  const int64_t n_tiles = (n + kSimBN - 1) / kSimBN;
  const int sms = sm_count();
  // the sample: every `stride`-th tile, at most one per SM (one round) and at most an eighth of the shard (it is scanned
  // twice); a sampled tile yields kSimBN / 4 maxima per query and the sample must hold 2 k of them
  // (more than 128 queries are scanned by CTA pairs, M = 256: the same ~one tile per SM then means two per pair)
  p.stride = static_cast<int>((n_tiles + sms - 1) / sms);
  if (p.stride < 8) p.stride = 8;
  const int64_t sampled_tiles = (n_tiles + p.stride - 1) / p.stride;
  const FilterGeometry ga = filter_geometry(sampled_tiles, nq);  // L = kSimBN / 2 per tile a CTA (pair) visits
  p.Lp = ga.L / 4;
  p.stride_p = static_cast<int64_t>(ga.groups) * p.Lp;
  // (below two tiles per SM the dense score matrix is small and two launches beat four)
  p.two_pass = nq <= 256 && n_tiles >= 2ll * sms && sampled_tiles * (kSimBN / 4) >= 2ll * k &&
               p.stride_p <= kMaxTauSample && (p.Lp % 8) == 0;
  if (!p.two_pass) return p;
  p.gb = filter_geometry(n_tiles, nq);
  p.stride_b = static_cast<int64_t>(p.gb.groups) * p.gb.L;
  // upper threshold: ~2.5 k documents of the whole shard expected above it (relative sd 1 / sqrt(k_hi): with k_hi >= 24
  // the front lists hold k entries in all but a negligible share of the queries; the others take the back lists too)
  const double frac = static_cast<double>(sampled_tiles) / static_cast<double>(n_tiles);
  int64_t k_hi = static_cast<int64_t>(2.5 * k * frac + 0.5);
  if (k_hi < 24) k_hi = 24;
  if (const char* e = getenv("SGPT_SEARCH_K_HI")) {  // tests: 1 forces the back-list path, k disables the split
    const long v = atol(e);
    if (v >= 1) k_hi = v;
  }
  if (k_hi > k) k_hi = k;
  p.k_hi = static_cast<int>(k_hi);
  return p;
}

}  // namespace

// queries per scan of the two-pass path: 256 = one M-tile per CTA of a pair (gemm.cu launch_filter_gemm); batches of up
// to 128 queries run on independent CTAs.  The dense path (small shards) takes the same blocks.
constexpr int kQueryBlock = 256;

static int64_t plan_bytes(int nq, int64_t n, int k) {
  const Plan p = make_plan(nq, n, k);
  if (!p.two_pass) return static_cast<int64_t>(nq) * padded_cols(n) * 4 + 256;
  return align256(static_cast<int64_t>(nq) * p.stride_p * 4) + align256(static_cast<int64_t>(nq) * p.stride_b * 8) +
         2 * align256(static_cast<int64_t>(p.gb.groups) * nq * 4) + 3 * align256(nq * 4) + 256;
}

extern "C" int64_t sgpt_search_workspace_bytes(int nq, int64_t n, int k) {
  if (nq <= 128) return plan_bytes(nq, n, k);
  // larger batches are processed in blocks of kQueryBlock that reuse the workspace; the last block may hold <= 128 queries
  // and then takes the single-CTA plan, whose lists are laid out differently
  const int64_t a = plan_bytes(nq < kQueryBlock ? nq : kQueryBlock, n, k), b = plan_bytes(128, n, k);
  return a > b ? a : b;
}

// One shard, all query blocks.  `fin` carries the packed destinations of the final selection (TopkExtra::dst/flag:
// this rank's buffer and/or peer gather buffers); out_scores / out_ids may be null when only those are wanted.
// Checks of the element type shared by the _ex entry points; they run before any CUDA call.
static int check_elem(const char* who, int elem, int D) {
  SGPT_REQUIRE(elem == SGPT_ELEM_BF16 || elem == SGPT_ELEM_I8, "%s: unknown element type %d", who, elem);
  // int8 rows: the TMA row pitch (D bytes) must be a multiple of 16, and |acc| <= 127^2 D must fit in int32
  SGPT_REQUIRE(elem != SGPT_ELEM_I8 || (D > 0 && D % 16 == 0 && D <= 65536),
               "%s: int8 rows need D a positive multiple of 16 and <= 65536 (D=%d)", who, D);
  return SGPT_OK;
}

// (elem: SGPT_ELEM_BF16 / SGPT_ELEM_I8, checked by the callers; plan and workspace do not depend on it)
static int search_impl(const void* Q, const void* Cm, const float* q_scale, const float* c_scale, int nq, int64_t n, int D,
                       int k, int64_t id_base, float* out_scores, int64_t* out_ids, void* ws, int64_t ws_bytes,
                       const TopkExtra& fin, int elem, cudaStream_t stream) {
  SGPT_REQUIRE(nq >= 0 && n >= 0 && k > 0, "sgpt_search: bad sizes nq=%d n=%lld k=%d", nq, (long long)n, k);
  SGPT_REQUIRE(n < (1ll << 31), "sgpt_search: shard too large for one launch (n=%lld)", (long long)n);
  SGPT_REQUIRE(D > 0 && D % 8 == 0, "sgpt_search: D=%d must be a positive multiple of 8", D);
  SGPT_REQUIRE(ws != nullptr && ws_bytes >= sgpt_search_workspace_bytes(nq, n, k),
               "sgpt_search: workspace too small (%lld < %lld bytes)", (long long)ws_bytes,
               (long long)sgpt_search_workspace_bytes(nq, n, k));
  if (nq == 0) return SGPT_OK;
  if (nq > kQueryBlock) {
    for (int q0 = 0; q0 < nq; q0 += kQueryBlock) {
      const int nb = (nq - q0 < kQueryBlock) ? nq - q0 : kQueryBlock;
      TopkExtra f = fin;
      for (int p = 0; p < f.n_dst; ++p) {  // rows of this block inside each destination
        f.dst[p] += static_cast<size_t>(q0) * k;
        if (f.flag[p] != nullptr) f.flag[p] += q0;
      }
      const size_t row_bytes = static_cast<size_t>(D) * (elem == SGPT_ELEM_I8 ? 1 : 2);
      int rc = search_impl(static_cast<const uint8_t*>(Q) + static_cast<size_t>(q0) * row_bytes, Cm,
                           q_scale ? q_scale + q0 : nullptr, c_scale, nb, n, D, k, id_base,
                           out_scores ? out_scores + static_cast<size_t>(q0) * k : nullptr,
                           out_ids ? out_ids + static_cast<size_t>(q0) * k : nullptr, ws, ws_bytes, f, elem, stream);
      if (rc != SGPT_OK) return rc;
    }
    return SGPT_OK;
  }
  const Plan p = make_plan(nq, n, k);
  if (!p.two_pass) {
    float* scores = static_cast<float*>(ws);
    const int64_t lds = padded_cols(n);
    int rc = launch_scores(Q, Cm, q_scale, c_scale, scores, lds, nq, n, D, elem, stream);
    if (rc != SGPT_OK) return rc;
    TopkSrc src{};
    src.scores = scores;
    src.id_base = id_base;
    src.G = 1;
    src.nq = nq;
    src.L = n;
    src.stride_q = lds;
    return launch_topk_select(src, nq, k, out_scores, out_ids, stream, fin);
  }

  uint8_t* w = static_cast<uint8_t*>(ws);
  float* pool = reinterpret_cast<float*>(w);
  w += align256(static_cast<int64_t>(nq) * p.stride_p * 4);
  uint2* cand = reinterpret_cast<uint2*>(w);
  w += align256(static_cast<int64_t>(nq) * p.stride_b * 8);
  int* cnt = reinterpret_cast<int*>(w);  // every group of the pass-B launch writes its own counts (groups = 2 x its CTAs)
  w += align256(static_cast<int64_t>(p.gb.groups) * nq * 4);
  int* cnt_back = reinterpret_cast<int*>(w);
  w += align256(static_cast<int64_t>(p.gb.groups) * nq * 4);
  float* tau = reinterpret_cast<float*>(w);
  w += align256(nq * 4);
  float* tau_hi = reinterpret_cast<float*>(w);
  w += align256(nq * 4);
  int* need_generic = reinterpret_cast<int*>(w);

  // pass A: block maxima of the sampled tiles -> admission thresholds
  int rc = launch_sample_maxima(Q, Cm, q_scale, c_scale, pool, p.stride_p, p.Lp, nq, static_cast<int>(n), D, elem,
                                p.stride, stream);
  if (rc != SGPT_OK) return rc;
  rc = launch_tau_select(pool, p.stride_p, static_cast<int>(p.stride_p), nq, k, p.k_hi, tau, tau_hi, stream);
  if (rc != SGPT_OK) return rc;
  // pass B: the whole shard, admission threshold tau[q], front / back split at tau_hi[q]
  rc = launch_filter_candidates(Q, Cm, q_scale, c_scale, tau, tau_hi, cand, cnt, cnt_back, p.stride_b, p.gb.L, 0, nq,
                                static_cast<int>(n), D, elem, /*tile_mode=*/0, 1, stream);
  if (rc != SGPT_OK) return rc;
  // final exact selection over the candidates
  TopkSrc src{};
  src.packed = cand;
  src.counts = cnt;
  src.counts_back = cnt_back;
  src.id_base = id_base;
  src.G = p.gb.groups;
  src.nq = nq;
  src.L = p.gb.L;
  src.stride_g = p.gb.L;
  src.stride_q = p.stride_b;
  // normal case (front parts hold k .. 4096 entries): packed, sorted, done; the generic kernel answers the other queries
  bool front = false;
  rc = launch_front_select(src, nq, k, out_scores, out_ids, stream, fin, need_generic, &front);
  if (rc != SGPT_OK) return rc;
  if (front) src.run_flag = need_generic;
  return launch_topk_select(src, nq, k, out_scores, out_ids, stream, fin);
}

extern "C" int sgpt_search_ex(const void* Q, const void* Cm, const float* q_scale, const float* c_scale, int nq,
                              int64_t n, int D, int k, int64_t id_base, float* out_scores, int64_t* out_ids, void* ws,
                              int64_t ws_bytes, int elem, sgpt_stream_t stream_) {
  if (int rc = check_elem("sgpt_search", elem, D)) return rc;
  SGPT_REQUIRE(nq == 0 || (out_scores != nullptr && out_ids != nullptr), "sgpt_search: null output");
  return search_impl(Q, Cm, q_scale, c_scale, nq, n, D, k, id_base, out_scores, out_ids, ws, ws_bytes, TopkExtra(), elem,
                     static_cast<cudaStream_t>(stream_));
}

extern "C" int sgpt_search(const void* Q, const void* Cm, const float* q_scale, const float* c_scale, int nq,
                           int64_t n, int D, int k, int64_t id_base, float* out_scores, int64_t* out_ids, void* ws,
                           int64_t ws_bytes, sgpt_stream_t stream_) {
  return sgpt_search_ex(Q, Cm, q_scale, c_scale, nq, n, D, k, id_base, out_scores, out_ids, ws, ws_bytes, SGPT_ELEM_BF16,
                        stream_);
}

extern "C" int sgpt_search_packed_ex(const void* Q, const void* Cm, const float* q_scale, const float* c_scale, int nq,
                                     int64_t n, int D, int k, int64_t id_base, uint64_t* out_packed, void* ws,
                                     int64_t ws_bytes, int elem, sgpt_stream_t stream_) {
  if (int rc = check_elem("sgpt_search_packed", elem, D)) return rc;
  SGPT_REQUIRE(nq == 0 || out_packed != nullptr, "sgpt_search_packed: null output");
  SGPT_REQUIRE(id_base >= 0 && id_base + n < (1ll << 31), "sgpt_search_packed: global ids must fit 31 bits (id_base=%lld n=%lld)",
               (long long)id_base, (long long)n);
  TopkExtra fin{};
  fin.dst[0] = reinterpret_cast<uint2*>(out_packed);
  fin.n_dst = 1;
  fin.dst_slot = 0;
  fin.dst_nq = nq;
  return search_impl(Q, Cm, q_scale, c_scale, nq, n, D, k, id_base, nullptr, nullptr, ws, ws_bytes, fin, elem,
                     static_cast<cudaStream_t>(stream_));
}

extern "C" int sgpt_search_packed(const void* Q, const void* Cm, const float* q_scale, const float* c_scale, int nq,
                                  int64_t n, int D, int k, int64_t id_base, uint64_t* out_packed, void* ws,
                                  int64_t ws_bytes, sgpt_stream_t stream_) {
  return sgpt_search_packed_ex(Q, Cm, q_scale, c_scale, nq, n, D, k, id_base, out_packed, ws, ws_bytes, SGPT_ELEM_BF16,
                               stream_);
}

// ---------------------------------------------------------------------------------------------------------------
// Row-sharded corpus across the GPUs of one box (SURVEY.md §8e): per-shard top-k -> all ranks -> merge, WITHOUT a
// collective library call.  Every rank owns a gather buffer [2 parities][world][nq_cap][k] of packed (score, id) entries
// plus per-query arrival counters, allocated with cudaMalloc and exported through CUDA IPC; every rank maps all peers'
// buffers.  The final selection kernel of a search writes its sorted winners straight into slot `rank` of EVERY rank's
// buffer (16-byte stores over NVLink for the peers) and then bumps that rank's counter for the query with a
// system-scope release; the merge kernel's CTA for query q acquires counter[q] == world x (uses of this parity) and merges
// the `world` lists (same kernel as the chunk merge XS:121-132).  No barrier, no host synchronisation; the two parities
// make the buffers safe to reuse: rank A can start search s+2 only after its merge s+1, which needed rank B's push s+1,
// which B's stream orders after B's merge s — the last reader of the parity search s+2 overwrites.
// ---------------------------------------------------------------------------------------------------------------
struct sgpt_gather {
  int rank = 0, world = 1, nq_cap = 0, k = 0;
  uint8_t* local = nullptr;
  uint8_t* peers[kMaxPeers] = {};
  bool opened[kMaxPeers] = {};
  size_t parity_bytes = 0, flags_off = 0, total = 0;
  unsigned long long uses[2] = {0, 0}, calls = 0;
};

extern "C" int sgpt_gather_create(int rank, int world, int nq_cap, int k, sgpt_gather_t* out, void* handle_out) {
  SGPT_REQUIRE(out != nullptr && handle_out != nullptr, "sgpt_gather_create: null argument");
  *out = nullptr;
  SGPT_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "sgpt_gather_create: rank %d / world %d (max %d)",
               rank, world, kMaxPeers);
  SGPT_REQUIRE(nq_cap > 0 && k > 0 && k <= 4096, "sgpt_gather_create: bad nq_cap=%d k=%d", nq_cap, k);
  static_assert(sizeof(cudaIpcMemHandle_t) == SGPT_IPC_HANDLE_BYTES, "IPC handle size");
  sgpt_gather* g = new sgpt_gather();
  g->rank = rank; g->world = world; g->nq_cap = nq_cap; g->k = k;
  g->parity_bytes = static_cast<size_t>(align256(static_cast<int64_t>(world) * nq_cap * k * 8));
  g->flags_off = 2 * g->parity_bytes;
  g->total = g->flags_off + 2 * static_cast<size_t>(align256(static_cast<int64_t>(nq_cap) * 4));
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&g->local), g->total);
  if (e == cudaSuccess) e = cudaMemset(g->local, 0, g->total);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, g->local);
  if (e != cudaSuccess) {
    set_error("sgpt_gather_create: %s", cudaGetErrorString(e));
    cudaFree(g->local);
    delete g;
    return SGPT_ERR_CUDA;
  }
  memcpy(handle_out, &h, sizeof(h));
  g->peers[rank] = g->local;
  *out = g;
  return SGPT_OK;
}

extern "C" int sgpt_gather_connect(sgpt_gather_t g, const void* all_handles) {
  SGPT_REQUIRE(g != nullptr && all_handles != nullptr, "sgpt_gather_connect: null argument");
  for (int r = 0; r < g->world; ++r) {
    if (r == g->rank || g->opened[r]) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const uint8_t*>(all_handles) + static_cast<size_t>(r) * sizeof(h), sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("sgpt_gather_connect: cannot map the gather buffer of rank %d: %s", r, cudaGetErrorString(e));
      return SGPT_ERR_CUDA;
    }
    g->peers[r] = static_cast<uint8_t*>(p);
    g->opened[r] = true;
  }
  return SGPT_OK;
}

extern "C" void sgpt_gather_destroy(sgpt_gather_t g) {
  if (!g) return;
  for (int r = 0; r < g->world; ++r)
    if (g->opened[r]) cudaIpcCloseMemHandle(g->peers[r]);
  cudaFree(g->local);
  delete g;
}

extern "C" int sgpt_search_gather_ex(sgpt_gather_t g, const void* Q, const void* Cm, const float* q_scale,
                                     const float* c_scale, int nq, int64_t n, int D, int k, int64_t id_base,
                                     const int64_t* exclude_ids, float* out_scores, int64_t* out_ids, void* ws,
                                     int64_t ws_bytes, int elem, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (int rc = check_elem("sgpt_search_gather", elem, D)) return rc;
  SGPT_REQUIRE(g != nullptr, "sgpt_search_gather: null gather context");
  SGPT_REQUIRE(nq >= 0 && nq <= g->nq_cap && k == g->k, "sgpt_search_gather: nq=%d k=%d do not fit the context (nq<=%d, k=%d)",
               nq, k, g->nq_cap, g->k);
  SGPT_REQUIRE(id_base >= 0 && id_base + n < (1ll << 31), "sgpt_search_gather: global ids must fit 31 bits");
  SGPT_REQUIRE(nq == 0 || (out_scores != nullptr && out_ids != nullptr), "sgpt_search_gather: null output");
  for (int r = 0; r < g->world; ++r)
    SGPT_REQUIRE(g->peers[r] != nullptr, "sgpt_search_gather: rank %d is not connected (sgpt_gather_connect)", r);
  if (nq == 0) return SGPT_OK;  // every rank passes the same nq: nobody pushes, nobody waits
  const int par = static_cast<int>(g->calls & 1ull);
  const unsigned int target = static_cast<unsigned int>((g->uses[par] + 1ull) * static_cast<unsigned long long>(g->world));
  TopkExtra fin{};
  fin.n_dst = g->world;
  fin.dst_slot = g->rank;
  fin.dst_nq = g->nq_cap;
  const size_t flag_off = g->flags_off + static_cast<size_t>(par) * static_cast<size_t>(align256(static_cast<int64_t>(g->nq_cap) * 4));
  for (int r = 0; r < g->world; ++r) {
    fin.dst[r] = reinterpret_cast<uint2*>(g->peers[r] + static_cast<size_t>(par) * g->parity_bytes);
    fin.flag[r] = reinterpret_cast<unsigned int*>(g->peers[r] + flag_off);
  }
  int rc = search_impl(Q, Cm, q_scale, c_scale, nq, n, D, k, id_base, nullptr, nullptr, ws, ws_bytes, fin, elem, stream);
  // the counters of this parity are consumed whether or not the merge below is launched
  g->uses[par] += 1;
  g->calls += 1;
  if (rc != SGPT_OK) return rc;
  TopkSrc src{};
  src.packed = reinterpret_cast<const uint2*>(g->local + static_cast<size_t>(par) * g->parity_bytes);
  src.packed_global = 1;
  src.lists_sorted = 1;  // written by the final selection kernels of the ranks
  src.exclude = reinterpret_cast<const long long*>(exclude_ids);
  src.G = g->world;
  src.nq = nq;
  src.L = k;
  src.stride_g = static_cast<long long>(g->nq_cap) * k;
  src.stride_q = k;
  src.wait_flag = reinterpret_cast<const unsigned int*>(g->local + flag_off);
  src.wait_target = target;
  return launch_topk_select(src, nq, k, out_scores, out_ids, stream);
}

extern "C" int sgpt_search_gather(sgpt_gather_t g, const void* Q, const void* Cm, const float* q_scale,
                                  const float* c_scale, int nq, int64_t n, int D, int k, int64_t id_base,
                                  const int64_t* exclude_ids, float* out_scores, int64_t* out_ids, void* ws,
                                  int64_t ws_bytes, sgpt_stream_t stream_) {
  return sgpt_search_gather_ex(g, Q, Cm, q_scale, c_scale, nq, n, D, k, id_base, exclude_ids, out_scores, out_ids, ws,
                               ws_bytes, SGPT_ELEM_BF16, stream_);
}

extern "C" int sgpt_topk_merge_packed(const uint64_t* in_packed, int G, int nq, int k, float* out_scores,
                                      int64_t* out_ids, const int64_t* exclude_ids, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(G >= 1 && nq >= 0 && in_packed != nullptr, "sgpt_topk_merge_packed: bad arguments G=%d nq=%d", G, nq);
  if (nq == 0) return SGPT_OK;
  TopkSrc src{};
  src.packed = reinterpret_cast<const uint2*>(in_packed);
  src.packed_global = 1;
  src.lists_sorted = 1;  // contract of the entry point (include/sgpt_b200.h)
  src.exclude = reinterpret_cast<const long long*>(exclude_ids);
  src.G = G;
  src.nq = nq;
  src.L = k;
  src.stride_g = static_cast<long long>(nq) * k;
  src.stride_q = k;
  return launch_topk_select(src, nq, k, out_scores, out_ids, stream);
}

// Host launchers for the tcgen05 GEMM (gemm.cuh): nn.Linear with fused epilogues (F3/F5/F6), the query x corpus
// similarity (S1) and its threshold-filter variant used by the fused search (search.cu).
#include "gemm.cuh"

#include <stdlib.h>

#include <type_traits>

#include "../../include/sgpt_b200.h"
#include "gemm_api.h"
#include "host_utils.h"

namespace sgpt {

template <int BN, class Epi, int CL = 1, int kOperand = kOperandBF16>
static int launch_gemm(const void* a, int64_t lda, const void* b, int64_t ldb, int M, int N, int K,
                       const typename Epi::Params& ep, cudaStream_t stream, int cat = kCatGemm,
                       TileMap tmap = TileMap()) {
  using Cfg = GemmCfg<BN, CL, EpiStaging<Epi>::value>;
  constexpr int kBK = OperandTraits<kOperand>::kBK;  // one 128-byte row segment: 64 bf16 or 128 int8
  auto make_map = kOperand == kOperandS8 ? make_tma_2d_u8 : make_tma_2d_bf16;
  CUtensorMap ta, tb;
  int rc = make_map(&ta, a, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), kGemmBM, kBK);
  if (rc != SGPT_OK) return rc;
  // in a CTA pair each CTA holds half of the B tile; with two pairs per cluster (CL = 4) it fetches a quarter and
  // receives the other quarter of its half by multicast from the CTA of its parity in the other pair
  rc = make_map(&tb, b, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), BN / CL, kBK);
  if (rc != SGPT_OK) return rc;
  auto kern = gemm_bf16_tn_kernel<BN, Epi, CL, kOperand>;
  static PerDeviceOnce attr_once;
  if (attr_once.first()) {
    SGPT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  }
  const int m_tiles = ((M + kGemmBM - 1) / kGemmBM + CL - 1) / CL;
  const int n_tiles = tmap.count((N + BN - 1) / BN);
  // work units (one per cluster iteration): tile groups x K slices
  const long long tiles = static_cast<long long>(m_tiles) * n_tiles * tmap.ksplit;
  if (tiles == 0) return SGPT_OK;
  long long clusters = sm_count() / CL;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(128 + 32 * Epi::kEpiWarps);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (CL == 4) {
    // 4-CTA clusters cannot use every SM (GPCs whose SM count is not a multiple of 4): ask how many fit at once
    static int max_clusters[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && max_clusters[dev] == 0) {
      cudaLaunchConfig_t q = cfg;
      q.gridDim = dim3(static_cast<unsigned>(clusters * CL));
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = CL;
      qa[0].val.clusterDim.y = 1;
      qa[0].val.clusterDim.z = 1;
      q.attrs = qa;
      q.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, kern, &q) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        n = static_cast<int>(clusters);
      }
      max_clusters[dev] = n;
    }
    if (dev >= 0 && dev < 64 && max_clusters[dev] > 0 && max_clusters[dev] < clusters) clusters = max_clusters[dev];
  }
  if (tiles < clusters) clusters = tiles;
  cfg.gridDim = dim3(static_cast<unsigned>(clusters * CL));
  if (CL > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = CL;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  LaunchScope _ls(cat, stream);
  SGPT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, M, N, K, ep, tmap));
  return SGPT_OK;
}

// SGPT_GEMM_CL4=1 enables the 4-CTA (two pairs, multicast weights) clusters.  Measured on B200 (profiles/
// r02_gemm_epilogues_cl4_vs_cl2.jsonl): correct, but 3-8 % SLOWER than plain pairs on every encoder shape — the mainloop
// is not bound by the L2 -> SM stream the multicast relieves but by the per-SM shared-memory fill, which is unchanged —
// so it stays off by default.
static bool cl4_enabled() {
  static const bool v = [] {
    const char* e = getenv("SGPT_GEMM_CL4");
    return e != nullptr && e[0] == '1';
  }();
  return v;
}

// nn.Linear dispatch: tile width by wave efficiency; CTA pairs (cta_group::2, M = 256) whenever there are at least two
// M-tiles — a third less L2->SM and smem traffic per FLOP than independent CTAs; two pairs per cluster sharing the weight
// tile by multicast (another quarter less L2->SM traffic) when there are at least four M-tiles and 256-wide tiles.
// Tile rasterisation (gemm.cuh TileMap::band): banded M-fastest order once the weight matrix no longer fits in the L2
// next to the activations.  SGPT_GEMM_BAND=<g> forces a band height (0 = N fastest) for A/B measurements; read per call.
static int pick_band(int M, int N, int K) {
  if (const char* e = getenv("SGPT_GEMM_BAND")) return atoi(e);
  const long long w_bytes = 2ll * N * K;
  const int m_groups = (M + 2 * kGemmBM - 1) / (2 * kGemmBM);
  return (w_bytes >= (64ll << 20) && m_groups >= 16) ? 8 : 0;
}

// The 16-warp early-release epilogue (gemm.cuh EpiTma16) for CTA pairs on 256-wide tiles: ON unless SGPT_GEMM_EPI16=0 (read
// per call: the GPU tests compare both forms in one process).  Same box, alternating runs of bench.py: 38.70 k embeddings/s
// with 8 epilogue warps, 39.73 / 39.76 k with 16 (GEMM time per step 5.50 -> 5.22 / 5.35 ms).
static bool epi16_enabled() {
  const char* e = getenv("SGPT_GEMM_EPI16");
  return !(e != nullptr && e[0] == '0');
}

template <class Epi>
static int launch_linear(const void* x, int64_t ldx, const void* w, int64_t ldw, int M, int N, int K,
                         const typename Epi::Params& p, int bn, cudaStream_t stream, int ksplit = 1) {
  const bool pair = M > kGemmBM;
  TileMap tm;
  tm.ksplit = ksplit;
  tm.band = pick_band(M, N, K);
  using Epi16 = typename Epi16Of<Epi>::type;
  if constexpr (!std::is_same<Epi16, Epi>::value) {
    // (the opt-in 4-CTA-cluster experiment keeps its own 8-warp form)
    if (bn == 256 && pair && epi16_enabled() && !cl4_enabled())
      return launch_gemm<256, Epi16, 2>(x, ldx, w, ldw, M, N, K, p, stream, kCatGemm, tm);
  }
  if (bn == 256) {
    if (M >= 4 * kGemmBM && cl4_enabled() && ksplit == 1)
      return launch_gemm<256, Epi, 4>(x, ldx, w, ldw, M, N, K, p, stream);
    return pair ? launch_gemm<256, Epi, 2>(x, ldx, w, ldw, M, N, K, p, stream, kCatGemm, tm)
                : launch_gemm<256, Epi, 1>(x, ldx, w, ldw, M, N, K, p, stream, kCatGemm, tm);
  }
  return pair ? launch_gemm<128, Epi, 2>(x, ldx, w, ldw, M, N, K, p, stream, kCatGemm, tm)
              : launch_gemm<128, Epi, 1>(x, ldx, w, ldw, M, N, K, p, stream, kCatGemm, tm);
}

// Split-K for the reduce-add (residual) epilogues: OFF unless SGPT_GEMM_SPLITK=2/3/4 asks for it (experiments, tests).
// The idea: these GEMMs have few, long tiles (N = d_model) — 384 tile groups on 74 CTA pairs (125M c_proj) run as 6 rounds
// of which the last is 19 % full — and S K-slices per tile give S x as many units of 1/S the length, so the tail shrinks
// to a fraction of a slice.  Measured on B200 (tools/bench_splitk.py, isolated launches, us, unsplit / 2 / 3 / 4 slices):
// 125M c_proj 117 / 115 / 121 / 117, 1.3B c_proj 328 / 339 / 379 / 403, 5.8B c_proj 874 / 907 / 953 / 1175 — the second
// reduce-add per output element costs what the shorter tail saves.  And it is not free semantically: with S > 1 the order
// in which the slices' partial sums reach the bf16 residual stream varies from run to run, so the encoder is no longer
// bit-reproducible (tests/test_gpu_full_depth.py caught it).  A slice is at least 16 k-blocks (1024 of K).
static int pick_ksplit(int M, int N, int K, int bn) {
  const char* env = getenv("SGPT_GEMM_SPLITK");  // read per call: the GPU tests flip it in-process
  const int forced = env != nullptr ? atoi(env) : -1;
  const int num_kb = (K + kGemmBK - 1) / kGemmBK;
  if (forced >= 2) return (forced <= 4 && num_kb / forced >= 16) ? forced : 1;
  (void)M; (void)N; (void)bn;
  return 1;
}

// Tile-width heuristic: BN=256 halves the smem bytes the tensor core must read per FLOP, but with few tiles the
// last wave is emptier; take the width with the better wave efficiency, preferring 256 on ties.
static int pick_bn(int M, int N) {
  if (N <= 128) return 128;
  const int sms = sm_count();
  auto eff = [&](int bn) {
    const long long tiles = static_cast<long long>((M + kGemmBM - 1) / kGemmBM) * ((N + bn - 1) / bn);
    const long long waves = (tiles + sms - 1) / sms;
    const double useful = static_cast<double>(M) * N;
    return useful / (static_cast<double>(waves) * sms * kGemmBM * bn);
  };
  return (eff(256) * 1.25 >= eff(128)) ? 256 : 128;
}

FilterGeometry filter_geometry(long long tiles, int nq) {
  // queries above one M-tile are scanned by CTA pairs (M = 256): one group per (pair, column half)
  const long long units = nq > kGemmBM ? sm_count() / 2 : sm_count();
  const long long ctas = tiles < units ? (tiles > 0 ? tiles : 1) : units;
  const long long per_cta = (tiles + ctas - 1) / ctas;
  FilterGeometry g;
  g.groups = static_cast<int>(2 * ctas);
  g.L = static_cast<int>(per_cta * (kSimBN / 2));
  return g;
}

// nq <= 128: independent CTAs (M = 128).  128 < nq <= 256: CTA pairs running tcgen05.mma.cta_group::2 with M = 256 — each CTA
// holds 128 of the queries and HALF of every corpus tile, so a scan moves half the corpus bytes per query through each SM
// and the kernel turns from HBM-bound into tensor-bound (2 x the queries per pass over the shard).  elem selects bf16 or
// int8 operands (kind::f16 / kind::i8; the epilogue then converts the s32 accumulator).
template <class P>
static int launch_filter_gemm(const void* Q, const void* C, int nq, int n, int D, int elem, const P& p,
                              cudaStream_t stream, TileMap tm) {
  if (elem == SGPT_ELEM_I8) {
    if (nq > kGemmBM)
      return launch_gemm<kSimBN, EpiFilterRowsS8, 2, kOperandS8>(Q, D, C, D, nq, n, D, p, stream, kCatScores, tm);
    return launch_gemm<kSimBN, EpiFilterRowsS8, 1, kOperandS8>(Q, D, C, D, nq, n, D, p, stream, kCatScores, tm);
  }
  if (nq > kGemmBM) return launch_gemm<kSimBN, EpiFilterRows, 2>(Q, D, C, D, nq, n, D, p, stream, kCatScores, tm);
  return launch_gemm<kSimBN, EpiFilterRows, 1>(Q, D, C, D, nq, n, D, p, stream, kCatScores, tm);
}

int launch_filter_candidates(const void* Q, const void* C, const float* q_scale, const float* c_scale,
                             const float* tau, const float* tau_hi, uint2* cand, int* counts, int* counts_back,
                             long long stride_q, int L, int group0, int nq, int n, int D, int elem, int tile_mode,
                             int tile_stride, cudaStream_t stream) {
  SGPT_REQUIRE(nq <= 2 * kGemmBM, "filter GEMM: at most %d queries per launch (got %d)", 2 * kGemmBM, nq);
  TileMap tm;
  tm.mode = tile_mode;
  tm.stride = tile_stride;
  const FilterGeometry g = filter_geometry(tm.count((n + kSimBN - 1) / kSimBN), nq);
  SGPT_REQUIRE(L >= g.L && (L % 2) == 0 && (stride_q % 2) == 0, "filter GEMM: candidate lists too small (L=%d < %d)", L,
               g.L);
  EpiFilterRows::Params p{q_scale, c_scale, tau, tau_hi, cand, counts, counts_back, stride_q, L, group0, nq, nullptr, 0, 0,
                          nq > kGemmBM ? 1 : 0};
  return launch_filter_gemm(Q, C, nq, n, D, elem, p, stream, tm);
}

int launch_sample_maxima(const void* Q, const void* C, const float* q_scale, const float* c_scale, float* pool,
                         long long stride_p, int Lp, int nq, int n, int D, int elem, int tile_stride,
                         cudaStream_t stream) {
  SGPT_REQUIRE(nq <= 2 * kGemmBM, "sample GEMM: at most %d queries per launch (got %d)", 2 * kGemmBM, nq);
  TileMap tm;
  tm.mode = 1;
  tm.stride = tile_stride;
  const FilterGeometry g = filter_geometry(tm.count((n + kSimBN - 1) / kSimBN), nq);
  SGPT_REQUIRE(Lp >= g.L / 4 && (Lp % 8) == 0 && (stride_p % 8) == 0 && stride_p >= static_cast<long long>(g.groups) * Lp,
               "sample GEMM: maxima lists too small (Lp=%d < %d)", Lp, g.L / 4);
  EpiFilterRows::Params p{q_scale, c_scale, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, nq, pool, stride_p, Lp,
                          nq > kGemmBM ? 1 : 0};
  return launch_filter_gemm(Q, C, nq, n, D, elem, p, stream, tm);
}

int launch_scores(const void* Q, const void* C, const float* q_scale, const float* c_scale, float* scores, int64_t lds,
                  int nq, int64_t n, int D, int elem, cudaStream_t stream) {
  SGPT_REQUIRE(nq >= 0 && n >= 0 && D > 0 && D % 8 == 0, "sgpt_scores: bad sizes nq=%d n=%lld D=%d", nq,
               (long long)n, D);
  SGPT_REQUIRE(n < (1ll << 31), "sgpt_scores: shard too large for one launch (n=%lld)", (long long)n);
  SGPT_REQUIRE(lds >= n, "sgpt_scores: lds < n");
  if (nq == 0 || n == 0) return SGPT_OK;
  EpiScoresF32::Params p{scores, q_scale, c_scale, static_cast<long long>(lds)};
  // lanes = queries (A operand), columns = corpus rows (B operand, streamed once from HBM)
  if (elem == SGPT_ELEM_I8)
    return launch_gemm<kSimBN, EpiScoresF32S8, 1, kOperandS8>(Q, D, C, D, nq, static_cast<int>(n), D, p, stream,
                                                              kCatScores);
  return launch_gemm<kSimBN, EpiScoresF32>(Q, D, C, D, nq, static_cast<int>(n), D, p, stream, kCatScores);
}

}  // namespace sgpt

using namespace sgpt;

extern "C" int sgpt_profile_gemm_clock(double* sm_cycles, double* nanoseconds) {
  SGPT_REQUIRE(sm_cycles != nullptr && nanoseconds != nullptr, "sgpt_profile_gemm_clock: null output");
  unsigned long long h[2] = {0, 0}, zero[2] = {0, 0};
  SGPT_CHECK_CUDA(cudaDeviceSynchronize());
  SGPT_CHECK_CUDA(cudaMemcpyFromSymbol(h, g_gemm_clock, sizeof(h)));
  SGPT_CHECK_CUDA(cudaMemcpyToSymbol(g_gemm_clock, zero, sizeof(zero)));
  *sm_cycles = static_cast<double>(h[0]);
  *nanoseconds = static_cast<double>(h[1]);
  return SGPT_OK;
}

extern "C" int sgpt_linear(const void* x, int64_t ldx, const void* w, int64_t ldw, const float* bias, void* out,
                           int64_t ldo, const float* resid, int M, int N, int K, int epilogue,
                           sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(M >= 0 && N > 0 && K > 0, "sgpt_linear: bad sizes M=%d N=%d K=%d", M, N, K);
  SGPT_REQUIRE(K % 8 == 0 && ldx % 8 == 0 && ldw % 8 == 0, "sgpt_linear: K, ldx, ldw must be multiples of 8");
  SGPT_REQUIRE(ldx >= K && ldw >= K && ldo >= N, "sgpt_linear: row pitch smaller than the row");
  if (M == 0) return SGPT_OK;
  int bn = pick_bn(M, N);
  if (const char* e = getenv("SGPT_GEMM_BN")) {  // experiments: force the tile width (128 / 256)
    const int v = atoi(e);
    if (v == 128 || (v == 256 && N > 128)) bn = v;
  }
  switch (epilogue) {
    case SGPT_EPI_BF16:
    case SGPT_EPI_GELU_BF16: {
      SGPT_REQUIRE(ldo % 8 == 0, "sgpt_linear: ldo must be a multiple of 8 for bf16 output");
      // output boxes of 32 rows x 64 bf16 (one 128-byte row segment per row), written by the epilogue through TMA
      CUtensorMap om;
      int rc = make_tma_2d_bf16(&om, out, static_cast<uint64_t>(M), static_cast<uint64_t>(N),
                                static_cast<uint64_t>(ldo), 32, 64);
      if (rc != SGPT_OK) return rc;
      if (epilogue == SGPT_EPI_BF16) {
        EpiBiasActBF16<false>::Params p{om, bias, out, static_cast<int>(ldo)};
        return launch_linear<EpiBiasActBF16<false>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
      }
      EpiBiasActBF16<true>::Params p{om, bias, out, static_cast<int>(ldo)};
      return launch_linear<EpiBiasActBF16<true>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
    }
    case SGPT_EPI_RESID_F32: {
      SGPT_REQUIRE(resid != nullptr, "sgpt_linear: SGPT_EPI_RESID_F32 needs resid");
      SGPT_REQUIRE(ldo % 4 == 0, "sgpt_linear: ldo must be a multiple of 4 for fp32 output");
      if (resid != static_cast<const float*>(out)) {
        // not in place: seed the output with the residual, the epilogue then adds acc + bias into it
        SGPT_CHECK_CUDA(cudaMemcpy2DAsync(out, static_cast<size_t>(ldo) * 4, resid, static_cast<size_t>(ldo) * 4,
                                          static_cast<size_t>(N) * 4, static_cast<size_t>(M),
                                          cudaMemcpyDeviceToDevice, stream));
      }
      CUtensorMap om;
      int rc = make_tma_2d_f32(&om, out, static_cast<uint64_t>(M), static_cast<uint64_t>(N),
                               static_cast<uint64_t>(ldo), 32, 32);
      if (rc != SGPT_OK) return rc;
      EpiResidualF32::Params p{om, bias, out, static_cast<int>(ldo)};
      return launch_linear<EpiResidualF32>(x, ldx, w, ldw, M, N, K, p, bn, stream, pick_ksplit(M, N, K, bn));
    }
    case SGPT_EPI_RESID_BF16: {
      SGPT_REQUIRE(resid != nullptr && static_cast<const void*>(resid) == out,
                   "sgpt_linear: SGPT_EPI_RESID_BF16 updates the bf16 residual stream in place (resid must alias out)");
      SGPT_REQUIRE(ldo % 8 == 0, "sgpt_linear: ldo must be a multiple of 8 for bf16 output");
      CUtensorMap om;
      int rc = make_tma_2d_bf16(&om, out, static_cast<uint64_t>(M), static_cast<uint64_t>(N),
                                static_cast<uint64_t>(ldo), 32, 64);
      if (rc != SGPT_OK) return rc;
      EpiResidualBF16::Params p{om, bias, out, static_cast<int>(ldo)};
      return launch_linear<EpiResidualBF16>(x, ldx, w, ldw, M, N, K, p, bn, stream, pick_ksplit(M, N, K, bn));
    }
    case 102:
    case 103:
    case 104:
    case 105: {  // profiling aids: bf16 epilogue without the TMA store (102) / without the smem-reuse wait (103)
      CUtensorMap om;
      int rc = make_tma_2d_bf16(&om, out, static_cast<uint64_t>(M), static_cast<uint64_t>(N),
                                static_cast<uint64_t>(ldo), 32, 64);
      if (rc != SGPT_OK) return rc;
      OpTmaBiasActBF16<false>::Params p{om, bias, out, static_cast<int>(ldo)};
      if (epilogue == 102) return launch_linear<EpiTma<OpTmaBiasActBF16<false>, 1>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
      if (epilogue == 105) return launch_linear<EpiTma<OpTmaBiasActBF16<false>, 4>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
      if (epilogue == 104) return launch_linear<EpiTma<OpTmaBiasActBF16<false>, 3>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
      return launch_linear<EpiTma<OpTmaBiasActBF16<false>, 2>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
    }
    case 100: {  // profiling aid: mainloop only
      EpiDebugNull<false>::Params p{0};
      return launch_linear<EpiDebugNull<false>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
    }
    case 101: {  // profiling aid: mainloop + TMEM loads
      EpiDebugNull<true>::Params p{0};
      return launch_linear<EpiDebugNull<true>>(x, ldx, w, ldw, M, N, K, p, bn, stream);
    }
    default:
      set_error("sgpt_linear: unknown epilogue %d", epilogue);
      return SGPT_ERR_INVALID;
  }
}

extern "C" int sgpt_linear_qkv_rotary(const void* x, int64_t ldx, const void* w_qkv, void* qkv, const int32_t* pos,
                                      const float* cos_sin, int M, int d_model, int head_dim, int rotary_dim,
                                      int max_pos, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(M >= 0 && d_model > 0 && d_model % 8 == 0 && ldx % 8 == 0 && ldx >= d_model,
               "sgpt_linear_qkv_rotary: bad sizes M=%d d=%d ldx=%lld", M, d_model, (long long)ldx);
  SGPT_REQUIRE(head_dim > 0 && d_model % head_dim == 0 && head_dim % 8 == 0, "sgpt_linear_qkv_rotary: bad head_dim %d",
               head_dim);
  SGPT_REQUIRE(rotary_dim >= 0 && rotary_dim <= head_dim && rotary_dim % 8 == 0,
               "sgpt_linear_qkv_rotary: rotary_dim %d must be a multiple of 8 and <= head_dim", rotary_dim);
  SGPT_REQUIRE(pos != nullptr && cos_sin != nullptr && max_pos > 0, "sgpt_linear_qkv_rotary: pos / cos_sin missing");
  if (M == 0) return SGPT_OK;
  const int N = 3 * d_model;
  CUtensorMap om;
  int rc = make_tma_2d_bf16(&om, qkv, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(N), 32,
                            64);
  if (rc != SGPT_OK) return rc;
  EpiRotaryBF16::Params p{om, pos, reinterpret_cast<const float2*>(cos_sin), M, d_model, head_dim, rotary_dim, max_pos,
                          qkv, N};
  return launch_linear<EpiRotaryBF16>(x, ldx, w_qkv, d_model, M, N, d_model, p, pick_bn(M, N), stream);
}

// F2+F3 / F2+F6 with the LayerNorm folded into the GEMM (gemm.cuh OpTmaLnBiasActBF16): x_bf16 is the bf16 copy of the
// residual stream, w the gamma-folded weight, bias / colsum the folded vectors, row_stats the partial sums.
extern "C" int sgpt_linear_lnfold(const void* x_bf16, int64_t ldx, const void* w_folded, int64_t ldw,
                                  const float* bias_folded, const float* colsum, const float* row_stats, int n_groups,
                                  float eps, void* out, int64_t ldo, int M, int N, int K, int gelu,
                                  sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(M >= 0 && N > 0 && K > 0, "sgpt_linear_lnfold: bad sizes M=%d N=%d K=%d", M, N, K);
  SGPT_REQUIRE(K % 8 == 0 && ldx % 8 == 0 && ldw % 8 == 0 && ldo % 8 == 0, "sgpt_linear_lnfold: K, ldx, ldw, ldo must be multiples of 8");
  SGPT_REQUIRE(ldx >= K && ldw >= K && ldo >= N, "sgpt_linear_lnfold: row pitch smaller than the row");
  SGPT_REQUIRE(bias_folded != nullptr && colsum != nullptr && row_stats != nullptr && n_groups > 0,
               "sgpt_linear_lnfold: folded bias / column sums / row statistics are required");
  SGPT_REQUIRE(N % 4 == 0, "sgpt_linear_lnfold: N must be a multiple of 4");
  if (M == 0) return SGPT_OK;
  CUtensorMap om;
  int rc = make_tma_2d_bf16(&om, out, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldo), 32, 64);
  if (rc != SGPT_OK) return rc;
  const int bn = pick_bn(M, N);
  const float inv_d = 1.0f / static_cast<float>(K);
  if (gelu) {
    EpiLnBiasActBF16<true>::Params p{om, bias_folded, colsum, reinterpret_cast<const float2*>(row_stats), n_groups, inv_d, eps,
                                     out, static_cast<int>(ldo)};
    return launch_linear<EpiLnBiasActBF16<true>>(x_bf16, ldx, w_folded, ldw, M, N, K, p, bn, stream);
  }
  EpiLnBiasActBF16<false>::Params p{om, bias_folded, colsum, reinterpret_cast<const float2*>(row_stats), n_groups, inv_d, eps,
                                    out, static_cast<int>(ldo)};
  return launch_linear<EpiLnBiasActBF16<false>>(x_bf16, ldx, w_folded, ldw, M, N, K, p, bn, stream);
}

extern "C" int sgpt_linear_qkv_rotary_lnfold(const void* x_bf16, int64_t ldx, const void* w_folded,
                                             const float* bias_folded, const float* colsum, const float* row_stats,
                                             int n_groups, float eps, void* qkv, const int32_t* pos,
                                             const float* cos_sin, int M, int d_model, int head_dim, int rotary_dim,
                                             int max_pos, sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(M >= 0 && d_model > 0 && d_model % 8 == 0 && ldx % 8 == 0 && ldx >= d_model,
               "sgpt_linear_qkv_rotary_lnfold: bad sizes M=%d d=%d ldx=%lld", M, d_model, (long long)ldx);
  SGPT_REQUIRE(head_dim > 0 && d_model % head_dim == 0 && head_dim % 8 == 0, "sgpt_linear_qkv_rotary_lnfold: bad head_dim %d",
               head_dim);
  SGPT_REQUIRE(rotary_dim >= 0 && rotary_dim <= head_dim && rotary_dim % 8 == 0,
               "sgpt_linear_qkv_rotary_lnfold: rotary_dim %d must be a multiple of 8 and <= head_dim", rotary_dim);
  SGPT_REQUIRE(pos != nullptr && cos_sin != nullptr && max_pos > 0, "sgpt_linear_qkv_rotary_lnfold: pos / cos_sin missing");
  SGPT_REQUIRE(bias_folded != nullptr && colsum != nullptr && row_stats != nullptr && n_groups > 0,
               "sgpt_linear_qkv_rotary_lnfold: folded bias / column sums / row statistics are required");
  if (M == 0) return SGPT_OK;
  const int N = 3 * d_model;
  CUtensorMap om;
  int rc = make_tma_2d_bf16(&om, qkv, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(N), 32, 64);
  if (rc != SGPT_OK) return rc;
  EpiLnRotaryBF16::Params p{{om, pos, reinterpret_cast<const float2*>(cos_sin), M, d_model, head_dim, rotary_dim, max_pos, qkv, N},
                            bias_folded, colsum, reinterpret_cast<const float2*>(row_stats), n_groups,
                            1.0f / static_cast<float>(d_model), eps, qkv, N};
  return launch_linear<EpiLnRotaryBF16>(x_bf16, ldx, w_folded, d_model, M, N, d_model, p, pick_bn(M, N), stream);
}

// F5 / F6b with the statistics of the NEXT LayerNorm (gemm.cuh EpiResidLn): resid += x w^T + bias in place, plus the
// bf16 copy and the per-(row, 128-column group) partial sums of the new residual.
extern "C" int sgpt_linear_resid_ln(const void* x, int64_t ldx, const void* w, int64_t ldw, const float* bias,
                                    float* resid, void* xb_out, float* stats_out, int M, int N, int K,
                                    sgpt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGPT_REQUIRE(M >= 0 && N > 0 && K > 0, "sgpt_linear_resid_ln: bad sizes M=%d N=%d K=%d", M, N, K);
  SGPT_REQUIRE(K % 8 == 0 && ldx % 8 == 0 && ldw % 8 == 0 && ldx >= K && ldw >= K, "sgpt_linear_resid_ln: bad pitches");
  SGPT_REQUIRE(N % 64 == 0, "sgpt_linear_resid_ln: N=%d must be a multiple of 64", N);
  SGPT_REQUIRE(resid != nullptr && xb_out != nullptr && stats_out != nullptr, "sgpt_linear_resid_ln: null output");
  if (M == 0) return SGPT_OK;
  EpiResidLn::Params p;
  int rc = make_tma_2d_f32(&p.resid_map, resid, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(N), 32, 32);
  if (rc != SGPT_OK) return rc;
  rc = make_tma_2d_bf16(&p.xb_map, xb_out, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(N), 32, 64);
  if (rc != SGPT_OK) return rc;
  p.bias = bias;
  p.stats = reinterpret_cast<float2*>(stats_out);
  p.P = (N + 127) / 128;
  {
    static const int l2pf = [] { const char* e = getenv("SGPT_RESID_L2_PREFETCH"); return (e != nullptr && e[0] == '0') ? 0 : 1; }();
    p.l2_prefetch = l2pf;
  }
  // always 256-wide tiles: each epilogue warp then owns exactly one 128-column statistics group
  if (M >= 4 * kGemmBM && cl4_enabled()) return launch_gemm<256, EpiResidLn, 4>(x, ldx, w, ldw, M, N, K, p, stream);
  return M > kGemmBM ? launch_gemm<256, EpiResidLn, 2>(x, ldx, w, ldw, M, N, K, p, stream)
                     : launch_gemm<256, EpiResidLn, 1>(x, ldx, w, ldw, M, N, K, p, stream);
}

extern "C" int sgpt_scores(const void* Q, const void* C, const float* q_scale, const float* c_scale, float* scores,
                           int64_t lds, int nq, int64_t n, int D, sgpt_stream_t stream_) {
  return launch_scores(Q, C, q_scale, c_scale, scores, lds, nq, n, D, SGPT_ELEM_BF16, static_cast<cudaStream_t>(stream_));
}

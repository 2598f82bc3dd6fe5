// Persistent, warp-specialised tcgen05 GEMM for sm_100a:  C[M,N] = A[M,K] * B[N,K]^T  (bf16 in, fp32 accumulate; the
// similarity scans of int8 corpus shards: int8 in, s32 accumulate, see kOperandS8).
//
//   A : activations / queries, row-major [M,K]  -> K-major UMMA operand A (TMEM lane = row of A)
//   B : nn.Linear weight [out,in] / corpus shard [n,D], row-major [N,K] -> K-major UMMA operand B
//
// Roles (E epilogue warps + 4 control warps = 256 or 384 threads, 1 CTA per SM):
//   warps 0..E-1  epilogue       (E = 8 for the TMA epilogues: two warps per TMEM lane quarter, each half the columns)
//   warp  E       TMA producer   (one lane; kStages-deep smem ring of {A 128x64, B BNx64} bf16 tiles, SWIZZLE_128B)
//   warp  E+1     MMA issuer     (one lane; tcgen05.mma M=128, N=BN, K=16; 2 TMEM accumulator stages)
//   warp  E+2     TMEM allocator
//
// The accumulator is double-buffered in TMEM so tile i's epilogue overlaps tile i+1's MMAs; smem stages and TMEM
// stages are handed over with mbarriers only (no __syncthreads in the main loop).
//
// Epilogue data paths.  tcgen05.ld hands thread r of a warp row r of the tile (32 consecutive columns per load); a
// direct global store from that layout would touch 32 different rows per instruction.  Two families:
//   EpiTma<Op>    (nn.Linear outputs)  thread = row: bias/activation in registers, the 128-byte row segment is written
//                 to a per-warp smem box in the SWIZZLE_128B layout and one elected lane hands the [32 x 128 B] box to
//                 the TMA engine — a plain tensor store (bf16 outputs) or an fp32 reduce-add into the residual stream
//                 (`resid += acc + bias`, performed by the L2; no residual load in the SM at all).  Two boxes per warp
//                 are double-buffered with cp.async.bulk.wait_group.read; M/N tails are clipped by the tensor map.
//   EpiStaged<Op> (similarity scores / threshold filter)  smem transpose so that lane = column pair and each warp
//                 instruction touches one contiguous row segment; needed where the work is per-(query row) with
//                 warp-wide ballots.
#pragma once
#include "common.cuh"

namespace sgpt {

constexpr int kGemmBM = 128;
constexpr int kGemmBK = 64;

// Operand kind of the persistent GEMM.  A k-block is one 128-byte SWIZZLE_128B row either way: 64 bf16 (kind::f16,
// K = 16 per MMA, fp32 accumulator) or 128 int8 (kind::i8, K = 32 per MMA, s32 accumulator); stage sizes, smem
// descriptors and their advance are the same.  Epilogues of int8 launches convert the s32 accumulator with acc_to_f32.
constexpr int kOperandBF16 = 0;
constexpr int kOperandS8 = 1;
template <int kOperand>
struct OperandTraits {
  static constexpr int kBK = kGemmBK;  // elements per k-block
};
template <>
struct OperandTraits<kOperandS8> {
  static constexpr int kBK = 2 * kGemmBK;
};
template <bool kS8>
__device__ __forceinline__ float acc_to_f32(uint32_t v) {
  if constexpr (kS8) return __int2float_rn(static_cast<int>(v));
  else return __uint_as_float(v);
}
constexpr int kGemmThreads = 256;
constexpr int kStageBytesPerWarp = 8192;  // per epilogue warp: 2 TMA boxes of 32 x 128 B, or one 32 x 64 fp32 slab

template <int BN, int CL = 1, int kStagingOverride = 0>
struct GemmCfg {
  static constexpr int kABytes = kGemmBM * kGemmBK * 2;
  static constexpr int kBBytes = (BN / (CL >= 2 ? 2 : 1)) * kGemmBK * 2;  // a CTA pair splits the B tile between its two CTAs
  static constexpr int kStageBytes = kABytes + kBBytes;    // 48 / 32 KB (single CTA, BN 256 / 128); 32 / 24 KB (pair)
  static constexpr int kBarrierBytes = 512;
  // epilogue staging: 4 KB boxes, one per epilogue warp behind the 48 KB stages, two (double-buffered) otherwise; an
  // epilogue that needs more (EpiResidLn: residual load boxes) states its own total
  static constexpr int kStagingBytes =
      kStagingOverride > 0 ? kStagingOverride : ((kStageBytes == 49152) ? 4 * kStageBytesPerWarp : 8 * kStageBytesPerWarp);
  static constexpr int kStagesFit = (232448 - 1024 - kStagingBytes - kBarrierBytes) / kStageBytes;
  static constexpr int kStagesDefault = (kStageBytes == 49152) ? 4 : (kStageBytes == 32768) ? 5 : 6;
  static constexpr int kStages = kStagesFit < kStagesDefault ? kStagesFit : kStagesDefault;
  static_assert(kStages >= 2, "not enough shared memory for a double-buffered mainloop");
  static constexpr int kTmemCols = 2 * BN;  // 256 or 512 (power of two)
  // smem: [<=1024 align slack][stages * (A|B)][epilogue staging][barriers + tmem holder (+ epilogue barriers)]
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + kStagingBytes + kBarrierBytes;
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
};

template <class Epi, class = void>
struct EpiHasPrefetch { static constexpr bool value = false; };
template <class Epi>
struct EpiHasPrefetch<Epi, decltype((void)&Epi::prefetch_next)> { static constexpr bool value = true; };

// Epilogue states with a `ks` member are told which K slice of a split-K launch the current work unit covers
template <class State, class = void>
struct StateHasKs { static constexpr bool value = false; };
template <class State>
struct StateHasKs<State, decltype((void)State::ks)> { static constexpr bool value = true; };

// Epilogues with a kEarlyRelease member split their tile work into load() — the warp's accumulator columns into registers
// — and store(); the kernel hands the TMEM accumulator stage back to the MMA issuer between the two.
template <class Epi, class = void>
struct EpiEarlyRelease { static constexpr bool value = false; };
template <class Epi>
struct EpiEarlyRelease<Epi, decltype((void)Epi::kEarlyRelease)> { static constexpr bool value = true; };

// Epilogues may state a total staging size (kStagingBytes member); 0 / absent = the default rule of GemmCfg.
template <class Epi, class = void>
struct EpiStaging { static constexpr int value = 0; };
template <class Epi>
struct EpiStaging<Epi, decltype((void)Epi::kStagingBytes)> { static constexpr int value = Epi::kStagingBytes; };

// [0] SM cycles, [1] nanoseconds spent inside GEMM kernels (sgpt_profile_gemm_clock); one thread per launch adds to it
__device__ unsigned long long g_gemm_clock[2];
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Optional selection of N-tiles: the similarity search scans a strided sample of corpus tiles first (to establish
// per-query thresholds) and the remaining tiles afterwards.
//   mode 0: all tiles;  mode 1: tiles 0, s, 2s, ...;  mode 2: every tile that is NOT a multiple of s   (s >= 2)
struct TileMap {
  int mode = 0;
  int stride = 1;
  // split-K (reduce-add epilogues only): every output tile is computed as `ksplit` work units over disjoint K ranges,
  // each adding its partial sum into the output; unit index = tile * ksplit + k-slice
  int ksplit = 1;
  // Rasterisation of the output tiles over the persistent CTAs.  band <= 1: N fastest (consecutive work units share the
  // activation rows and sweep the whole weight matrix: right while the weights stay in L2).  band = g: M-tile groups are
  // taken in bands of g, and inside a band the M index runs fastest — the ~74 CTA pairs working at the same time then cover
  // g M-groups x ~74/g N-tiles and fetch g + 74/g operand tiles instead of 1-2 + 64: for weight matrices larger than the
  // L2 (GPT-J / BLOOM-7B c_fc: 134 MB streamed once per ~1.2 M-groups = 5 TB/s of HBM reads with N fastest) the operand
  // traffic per wave drops ~4x.
  int band = 0;
  __host__ __device__ void coords(int tile, int m_tiles, int n_tiles, int& mg, int& nt) const {
    if (band <= 1) {
      mg = tile / n_tiles;
      nt = tile - mg * n_tiles;
      return;
    }
    const int per_band = band * n_tiles;
    const int b = tile / per_band, r = tile - b * per_band;
    const int rest = m_tiles - b * band;
    const int h = rest < band ? rest : band;  // height of this band (the last one may be lower)
    nt = r / h;
    mg = b * band + (r - nt * h);
  }
  __host__ __device__ int count(int n_tiles) const {
    if (mode == 0) return n_tiles;
    const int sampled = (n_tiles + stride - 1) / stride;
    return mode == 1 ? sampled : n_tiles - sampled;
  }
  __host__ __device__ int map(int j) const {
    if (mode == 0) return j;
    if (mode == 1) return j * stride;
    return j + j / (stride - 1) + 1;
  }
};

// CL = 1: independent CTAs, tcgen05.mma.cta_group::1, one 128 x BN tile per CTA iteration.
// CL = 2: CTA pairs (2-CTA clusters = the two SMs of a TPC) executing tcgen05.mma.cta_group::2 with M = 256: CTA r of
//   the pair owns rows [128 r, 128 r + 128) of the 256 x BN tile (its A rows in its smem, its accumulator rows in its
//   TMEM) and holds B rows [BN/2 r, BN/2 r + BN/2) — half of the weight tile — in its smem.  Only the leader (rank 0)
//   issues MMAs; both CTAs run a TMA producer (signalling the LEADER's full barrier) and the epilogue of their rows.
//   Per SM this removes a third of the smem writes (TMA) and operand reads (MMA) of the single-CTA kernel — measured:
//   with cta_group::1 the mainloop alone ran at the tensor peak but every byte the epilogue moved through smem
//   (st.shared + TMA-store reads) slowed it down (75 -> 103 us on the 32768 x 2304 x 768 QKV GEMM).
//   Barrier protocol: full[s] (leader, 1 arrive + 2 x stage bytes) <- both producers' TMA; empty[s] (each CTA, count 1)
//   <- leader's tcgen05.commit multicast; tmem_full[a] (each CTA) <- commit multicast; tmem_empty[a] (leader, count
//   2 x epilogue warps) <- both CTAs' epilogue warps (remote arrive from the peer).
// CL = 4: TWO CTA pairs (ranks {0,1} and {2,3}) on the same N-tile and adjacent 256-row M-groups.  At K = 768 the
//   CL = 2 mainloop is bound by the L2 -> SM operand stream (64 B/clk/SM at the tensor peak against the ~43 B/clk/SM the
//   L2 delivers: ncu l1tex__m_xbar2l1tex_read_bytes 12.9 TB/s), not by the tensor pipe.  Both pairs need the SAME weight
//   tile, so every CTA fetches only a QUARTER of it (BN/4 rows) and multicasts it into its own smem and into the smem of
//   the CTA of the same parity in the other pair: per k-block the four CTAs read 64 KB of A + 32 KB of B from L2 instead
//   of 64 + 64 (-25 %).  Each pair still runs its own cta_group::2 MMA from its own leader; a smem stage is written by
//   CTAs of BOTH pairs, so empty[s] counts one commit from each pair's leader (multicast to all four CTAs).
// kOperand: kOperandBF16 (the name's case) or kOperandS8 (int8 x int8 -> s32; the similarity scans of int8 shards).
template <int BN, class Epi, int CL = 1, int kOperand = kOperandBF16>
__global__ void __launch_bounds__(128 + 32 * Epi::kEpiWarps, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, int M,
                    int N, int K, const __grid_constant__ typename Epi::Params ep, TileMap tmap) {
  using Cfg = GemmCfg<BN, CL, EpiStaging<Epi>::value>;
  constexpr int kStages = Cfg::kStages;
  static_assert(CL == 1 || CL == 2 || CL == 4, "cluster size");
  constexpr bool kPair = CL >= 2;
  constexpr bool kS8 = kOperand == kOperandS8;
  constexpr int kBK = OperandTraits<kOperand>::kBK;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_tiles = smem;
  float* stage_base = reinterpret_cast<float*>(smem + kStages * Cfg::kStageBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes + Cfg::kStagingBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  uint64_t* epi_bars = tmem_empty_bar + 3;  // 2 mbarriers per epilogue warp (EpiResidLn's residual loads)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // Warp roles.  The epilogue warps take the LOW warp ids and the TMA producer / MMA issuer the HIGH ones: the SM's
  // issue arbiter favours higher warp ids among ready warps, and the two single-thread control warps must never be
  // starved of issue slots by epilogue arithmetic sharing their scheduler (measured: with the control warps at ids
  // 0/1 the epilogue's issue time added directly to the MMA time of every tile).
  constexpr int kWarpProducer = Epi::kEpiWarps, kWarpMma = Epi::kEpiWarps + 1, kWarpTmem = Epi::kEpiWarps + 2;

  const uint32_t crank = kPair ? cluster_ctarank() : 0u;  // position inside the cluster = M-tile of the group
  const uint32_t prank = crank & 1u;                       // rank inside the CTA pair; leader = crank & ~1
  const int cid = blockIdx.x / CL, ncl = gridDim.x / CL;      // cluster index / number of clusters
  const int m_tiles = ((M + kGemmBM - 1) / kGemmBM + CL - 1) / CL;  // M-tile groups (CL tiles each)
  const int n_tiles = tmap.count((N + BN - 1) / BN);                // N-tiles this launch visits
  const int ksplit = tmap.ksplit;
  const int num_tiles = m_tiles * n_tiles * ksplit;  // work units
  const int num_kb = (K + kBK - 1) / kBK;
  const int kb_per = (num_kb + ksplit - 1) / ksplit;  // k-blocks per slice (the host keeps every slice non-empty)

  if (warp == kWarpProducer && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == kWarpMma && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], CL == 4 ? 2 : 1);  // CL = 4: both pairs must have consumed the stage
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full_bar[i], 1);
      mbar_init(&tmem_empty_bar[i], (kPair ? 2 : 1) * Epi::kEpiWarps);  // one arrive per epilogue warp (of both CTAs of a pair)
    }
    fence_mbar_init();
  }
  if (warp == kWarpTmem) {
    if (kPair) {
      tmem_alloc_pair(tmem_holder, Cfg::kTmemCols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_holder, Cfg::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (kPair) cluster_sync_all();  // peer barriers / TMEM must exist before any remote arrive, commit or pair MMA
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  pdl_sync();  // everything above overlapped the previous kernel's tail; global memory is touched only below
  const bool clock_probe = (blockIdx.x == 0 && threadIdx.x == 0);
  const long long probe_c0 = clock_probe ? clock64() : 0;
  const uint64_t probe_t0 = clock_probe ? global_timer_ns() : 0;

  if (warp == kWarpProducer) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = cid; unit < num_tiles; unit += ncl) {
        const int tile = unit / ksplit, ks = unit - tile * ksplit;
        int mg, nt;
        tmap.coords(tile, m_tiles, n_tiles, mg, nt);
        const int m0 = (mg * CL + static_cast<int>(crank)) * kGemmBM;
        const int n0 = tmap.map(nt) * BN;
        const int kb_end = min(num_kb, (ks + 1) * kb_per);
        for (int kb = ks * kb_per; kb < kb_end; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem_tiles + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + Cfg::kABytes;
          if (kPair) {
            // my A rows and my half of the B tile land in MY smem; the bytes are accounted on the pair leader's barrier
            const uint32_t leader_full = mapa_shared(smem_u32(&full_bar[stage]), crank & ~1u);
            if (prank == 0) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
            tma_load_2d_pair(sa, &tma_a, leader_full, kb * kBK, m0);
            if (CL == 2) {
              tma_load_2d_pair(sb, &tma_b, leader_full, kb * kBK, n0 + static_cast<int>(prank) * (BN / 2));
            } else {
              // quarter (crank >> 1) of my pair-rank's half of the weight tile, multicast to the CTA of my parity in both
              // pairs (same smem offset there); each destination accounts the bytes on ITS pair leader's full barrier
              const int quarter = static_cast<int>(crank >> 1);
              tma_load_2d_pair_multicast(sb + quarter * (BN / 4) * 128, &tma_b, leader_full,
                                         kb * kBK, n0 + static_cast<int>(prank) * (BN / 2) + quarter * (BN / 4),
                                         static_cast<uint16_t>(0x5u << prank));
            }
          } else {
            mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
            tma_load_2d(sa, &tma_a, &full_bar[stage], kb * kBK, m0);
            tma_load_2d(sb, &tma_b, &full_bar[stage], kb * kBK, n0);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpMma) {
    // ===================== MMA issuer =====================
    if (lane == 0 && prank == 0) {
      constexpr uint32_t idesc =
          kS8 ? make_idesc_s8(kGemmBM * (kPair ? 2 : 1), BN) : make_idesc_bf16(kGemmBM * (kPair ? 2 : 1), BN, false);
      // commit masks: my pair's two CTAs; the smem stages of a 4-CTA cluster are shared by both pairs
      const uint16_t pair_mask = static_cast<uint16_t>(0x3u << (crank & ~1u));
      const uint16_t stage_mask = (CL == 4) ? static_cast<uint16_t>(0xF) : pair_mask;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int unit = cid; unit < num_tiles; unit += ncl) {
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        const int ks = unit % ksplit;
        const int kb_begin = ks * kb_per, kb_end = min(num_kb, kb_begin + kb_per);
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem_tiles + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + Cfg::kABytes;
          const uint64_t da = make_smem_desc_sw128(sa, 16, 1024);
          const uint64_t db = make_smem_desc_sw128(sb, 16, 1024);
#pragma unroll
          for (int k = 0; k < kGemmBK / 16; ++k) {
            // advance 16 bf16 = 32 B along K inside the 128-B swizzle row: +2 in the (addr >> 4) field (int8: 32 values,
            // the same 32 B)
            if constexpr (kS8) {
              if (kPair) umma_s8_ss_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, ((kb - kb_begin) | k) != 0);
              else umma_s8_ss(tmem_d, da + 2 * k, db + 2 * k, idesc, ((kb - kb_begin) | k) != 0);
            } else {
              if (kPair) umma_bf16_ss_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, ((kb - kb_begin) | k) != 0);
              else umma_bf16_ss(tmem_d, da + 2 * k, db + 2 * k, idesc, ((kb - kb_begin) | k) != 0);
            }
          }
          // frees this smem stage (in both CTAs of a pair) once the MMAs above have read it
          if (kPair) umma_commit_pair(&empty_bar[stage], stage_mask);
          else umma_commit(&empty_bar[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        // accumulator complete -> epilogue (of both CTAs)
        if (kPair) umma_commit_pair(&tmem_full_bar[acc], pair_mask);
        else umma_commit(&tmem_full_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp < Epi::kEpiWarps) {
    // ===================== epilogue =====================
    // A warp may only touch TMEM lanes 32*(warp%4)..+31.  With 8 epilogue warps two warps share a lane quarter and
    // split the tile's columns (half 0 / half 1): twice the warps to hide TMEM-load, bias-load and smem latencies.
    const int ew = warp & 3;              // TMEM lane quarter (hardware: warp id % 4) == 32-row slab of the tile
    const int half = warp >> 2;           // column half handled by this warp (always 0 with 4 epilogue warps)
    constexpr int kColsPerWarp = BN / (Epi::kEpiWarps / 4);
    constexpr int kSlabBytes = Cfg::kStagingBytes / Epi::kEpiWarps;
    float* stage_slab = stage_base + warp * (kSlabBytes / 4);
    const uint32_t leader_tmem_empty0 = kPair ? mapa_shared(smem_u32(&tmem_empty_bar[0]), crank & ~1u) : 0u;
    typename Epi::State st;
    Epi::init(st, ep, ew * 32 + lane, epi_bars + 2 * warp);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = cid; unit < num_tiles; unit += ncl) {
      const int tile = unit / ksplit;
      if constexpr (StateHasKs<typename Epi::State>::value) st.ks = static_cast<uint32_t>(unit - tile * ksplit);
      int mg, ntile;
      tmap.coords(tile, m_tiles, n_tiles, mg, ntile);
      const int m0 = (mg * CL + static_cast<int>(crank)) * kGemmBM + ew * 32;  // this warp's 32-row slab
      const int n0 = tmap.map(ntile) * BN + half * kColsPerWarp;
      // work that does not depend on the accumulator (EpiResidLn: the first residual loads, and an L2 prefetch of the
      // residual boxes of the tile after this one) overlaps the mainloop
      if constexpr (EpiHasPrefetch<Epi>::value) {
        const int nt = (unit + ncl) / ksplit;  // (split-K is never combined with a prefetching epilogue)
        if (unit + ncl < num_tiles) {
          int mg2, nt2;
          tmap.coords(nt, m_tiles, n_tiles, mg2, nt2);
          Epi::prefetch_next(ep, (mg2 * CL + static_cast<int>(crank)) * kGemmBM + ew * 32,
                             tmap.map(nt2) * BN + half * kColsPerWarp, lane, M, N);
        }
      }
      Epi::template pre_tile<kColsPerWarp, kSlabBytes>(st, ep, m0, n0, lane, stage_slab, M, N);
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t trow = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BN + half * kColsPerWarp;
      if constexpr (EpiEarlyRelease<Epi>::value) {
        // the accumulator stage goes back to the MMA issuer as soon as this warp's columns are in registers: the stage is
        // held for one TMEM load, not for the arithmetic, the shared-memory stores, the proxy fence and the TMA hand-over
        Epi::template load<kColsPerWarp, kSlabBytes>(st, trow);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kPair) mbar_arrive_cluster(leader_tmem_empty0 + acc * 8);
          else mbar_arrive(&tmem_empty_bar[acc]);
        }
        Epi::template store<kColsPerWarp, kSlabBytes>(st, ep, m0, n0, lane, stage_slab, M, N);
      } else {
        Epi::template tile<kColsPerWarp, kSlabBytes>(st, ep, m0, n0, lane, trow, stage_slab, M, N);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kPair) mbar_arrive_cluster(leader_tmem_empty0 + acc * 8);
          else mbar_arrive(&tmem_empty_bar[acc]);
        }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    Epi::finish(st, ep, static_cast<int>(crank) * kGemmBM + ew * 32 + lane);  // row inside the CL x 128-row tile group
    if (clock_probe) {
      atomicAdd(&g_gemm_clock[0], static_cast<unsigned long long>(clock64() - probe_c0));
      atomicAdd(&g_gemm_clock[1], static_cast<unsigned long long>(global_timer_ns() - probe_t0));
    }
  }

  tc_fence_before();
  if (kPair) cluster_sync_all();  // the peers may still multicast-arrive on this CTA's barriers until they are done too
  else __syncthreads();
  if (warp == kWarpTmem) {
    tc_fence_after();
    if (kPair) tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
    else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// TMA epilogue driver: TMEM -> registers (thread = row) -> Op (bias / activation) -> swizzled smem box -> TMA
// ---------------------------------------------------------------------------------------------------------------
template <class Row>
struct EpiTmaState {
  uint32_t it;  // boxes issued so far by this warp (selects the double buffer)
  uint32_t ks;  // K slice of the current work unit (split-K launches; 0 otherwise): only slice 0 adds the bias
  Row row;      // per-row constants of the CURRENT tile (LayerNorm mean / rstd), fetched in pre_tile: the loads overlap
                // the wait for the accumulator instead of sitting at the head of the epilogue's critical path
};

// Ops whose result is ADDED to the output (TMA reduce-add) can run split-K: they declare kSplitK and take a flag that
// tells whether this K slice contributes the bias.
template <class Op, class = void>
struct OpSplitK { static constexpr bool value = false; };
template <class Op>
struct OpSplitK<Op, decltype((void)Op::kSplitK)> { static constexpr bool value = true; };

template <class Op, int kDebug = 0>  // kDebug: 1 = skip the TMA store (timing experiment), 2 = skip the smem-reuse wait
struct EpiTma {
  using Params = typename Op::Params;
  using State = EpiTmaState<typename Op::Row>;
  static constexpr int kEpiWarps = 8;                 // 2 warps per TMEM lane quarter; each owns ONE 4 KB smem box
  static constexpr int kCols = 128 / Op::kElemBytes;  // columns per 128-byte row segment: 64 (bf16) or 32 (fp32)
  static __device__ __forceinline__ void init(State& st, const Params&, int, uint64_t*) { st.it = 0; st.ks = 0; }
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void pre_tile(State& st, const Params& p, int m0, int, int lane, float*, int M, int) {
    if (m0 < M) st.row = Op::row_init(p, m0 + lane, M);
  }
  static __device__ __forceinline__ void finish(State&, const Params&, int lane_row) {
    if ((lane_row & 31) == 0) bulk_wait_group<0>();  // all stores of this warp have fully completed
  }

  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void tile(State& st, const Params& p, int m0, int n0, int lane, uint32_t trow,
                                              float* slab, int M, int N) {
    if (m0 >= M) return;  // whole 32-row slab out of range (warp-uniform)
    const uint32_t sbase = smem_u32(slab);
    const typename Op::Row rc = st.row;  // per-row constants (thread = row), fetched in pre_tile
#pragma unroll 1
    for (int c = 0; c < BN; c += kCols) {
      const int n = n0 + c;
      if (n >= N) break;  // warp-uniform
      // kBoxes smem boxes per warp, used round-robin: a box may be rewritten once the TMA store issued kBoxes
      // iterations ago has finished READING it (the stores themselves complete asynchronously)
      constexpr int kBoxes = kSlabBytes / 4096;
      static_assert(kBoxes == 1 || kBoxes == 2, "one or two 4 KB boxes per epilogue warp");
      const uint32_t box = sbase + (kBoxes == 2 ? (st.it & 1u) * 4096u : 0u);
      if (st.it >= kBoxes && kDebug == 0) {
        if (lane == 0) bulk_wait_group_read<kBoxes - 1>();
        __syncwarp();
      }
      uint32_t v[kCols];
      tmem_ld_32x32(trow + c, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
      if (kCols == 64) tmem_ld_32x32(trow + c + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[kCols - 32]));
      tmem_ld_wait();
      // 8 chunks of 16 bytes; chunk j of row r lives at position j ^ (r & 7) of the row (SWIZZLE_128B)
      // All 8 chunks are computed before any of them is stored: the bias / rotary-table loads inside Op::chunk are then
      // independent ordinary loads the compiler batches up front (one exposed latency per box instead of one per chunk;
      // the volatile smem stores would otherwise fence them apart).
      const uint32_t row_addr = box + lane * 128u;
      uint32_t o[8][4];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if constexpr (OpSplitK<Op>::value)
          Op::chunk(p, rc, &v[j * (kCols / 8)], n + j * (kCols / 8), N, m0 + lane, o[j], st.ks == 0);
        else
          Op::chunk(p, rc, &v[j * (kCols / 8)], n + j * (kCols / 8), N, m0 + lane, o[j]);
      }
      if (kDebug == 4) {  // experiment: straight 16-byte global stores from the thread = row layout (no smem, no TMA)
        if (m0 + lane < M) {
          uint4* g = reinterpret_cast<uint4*>(static_cast<uint8_t*>(p.out_ptr) +
                                              (static_cast<size_t>(m0 + lane) * p.ldc + n) * Op::kElemBytes);
#pragma unroll
          for (int j = 0; j < 8; ++j) g[j] = make_uint4(o[j][0], o[j][1], o[j][2], o[j][3]);
        }
        ++st.it;
        continue;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) sts_v4(row_addr + ((j ^ (lane & 7)) << 4), o[j][0], o[j][1], o[j][2], o[j][3]);
      if (kDebug != 3) fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && kDebug != 1 && kDebug != 3) {
        Op::issue(p, reinterpret_cast<const void*>(__cvta_shared_to_generic(box)), n, m0);
        bulk_commit_group();
      }
      ++st.it;
    }
  }
};

// ---------------------------------------------------------------------------------------------------------------
// Default for CTA pairs on 256-wide tiles since the end of round 2 (SGPT_GEMM_EPI16=0 restores 8 warps): 16 epilogue warps — four per TMEM lane quarter, 64 accumulator
// columns (= one 128-byte bf16 box) each — that release the accumulator stage EARLY (kernel: load -> arrive -> store).
// Why: with 8 warps a warp walks through four boxes per tile in series (smem box free -> tcgen05.ld -> arithmetic -> 8 x
// st.shared -> fence.proxy.async -> TMA) and keeps the TMEM stage until the last one; at K = 768 that chain is about as
// long as the 6144-clock mainloop of the next tile, so the MMA issuer waits for a free accumulator (ncu: tensor pipe 41-55 %
// active, issue slots 15-35 % busy).  Here the stage is held for ONE TMEM load.  640 threads -> at most 96 registers per
// thread: the 64 accumulator values stay in registers and the box is computed and stored in two halves of four chunks.
// ---------------------------------------------------------------------------------------------------------------
template <class Op>
struct EpiTma16 {
  using Params = typename Op::Params;
  struct State {
    uint32_t it;
    uint32_t ks;
    typename Op::Row row;
    uint32_t v[64];  // this warp's accumulator columns of the current tile (thread = row)
  };
  static constexpr int kEpiWarps = 16;
  static constexpr bool kEarlyRelease = true;
  static constexpr int kCols = 128 / Op::kElemBytes;  // columns per 128-byte row segment: 64 (bf16) or 32 (fp32)
  static __device__ __forceinline__ void init(State& st, const Params&, int, uint64_t*) { st.it = 0; st.ks = 0; }
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void pre_tile(State& st, const Params& p, int m0, int, int lane, float*, int M, int) {
    if (m0 < M) st.row = Op::row_init(p, m0 + lane, M);
  }
  static __device__ __forceinline__ void finish(State&, const Params&, int lane_row) {
    if ((lane_row & 31) == 0) bulk_wait_group<0>();
  }
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void load(State& st, uint32_t trow) {
    static_assert(BN == 64, "EpiTma16: 64 accumulator columns per warp (256-wide tiles)");
    tmem_ld_32x32(trow, *reinterpret_cast<uint32_t(*)[32]>(&st.v[0]));
    tmem_ld_32x32(trow + 32, *reinterpret_cast<uint32_t(*)[32]>(&st.v[32]));
    tmem_ld_wait();
  }
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void store(State& st, const Params& p, int m0, int n0, int lane, float* slab, int M,
                                               int N) {
    static_assert(kSlabBytes == 4096, "EpiTma16: one 4 KB box per warp");
    if (m0 >= M) return;  // whole 32-row slab out of range (warp-uniform)
    const uint32_t box = smem_u32(slab);
    const uint32_t row_addr = box + lane * 128u;
    const typename Op::Row rc = st.row;
#pragma unroll
    for (int c = 0; c < BN; c += kCols) {  // one box (bf16 outputs) or two (fp32)
      const int n = n0 + c;
      if (n >= N) break;  // warp-uniform
      if (st.it >= 1) {   // the TMA store of this warp's previous box must have finished READING the box
        if (lane == 0) bulk_wait_group_read<0>();
        __syncwarp();
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t o[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int jj = 4 * h + j;
          if constexpr (OpSplitK<Op>::value)
            Op::chunk(p, rc, &st.v[c + jj * (kCols / 8)], n + jj * (kCols / 8), N, m0 + lane, o[j], st.ks == 0);
          else
            Op::chunk(p, rc, &st.v[c + jj * (kCols / 8)], n + jj * (kCols / 8), N, m0 + lane, o[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int jj = 4 * h + j;
          sts_v4(row_addr + ((jj ^ (lane & 7)) << 4), o[j][0], o[j][1], o[j][2], o[j][3]);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        Op::issue(p, reinterpret_cast<const void*>(__cvta_shared_to_generic(box)), n, m0);
        bulk_commit_group();
      }
      ++st.it;
    }
  }
};

// The 16-warp form of an epilogue, for the three ops it has been validated and measured with (bit-identical outputs,
// tests/test_gpu_raster.py; whole-model parity; +2.7 % embeddings/s on SGPT-125M, profiles/r02_gemm_epilogue_16_warps_ab.jsonl):
// bias (+ gelu_new) -> bf16 and the bf16 residual reduce-add.  Every other epilogue (GPT-J rotary, fp32 residual, the
// LayerNorm-fold family, the search filter) maps to itself.  (The ops are declared below.)
template <class Epi>
struct Epi16Of { using type = Epi; };

// bias index helper: columns beyond N are clipped by the tensor map, their bias is read from the last valid entry
__device__ __forceinline__ float bias_at(const float* bias, int col, int N) {
  return bias ? __ldg(bias + (col < N ? col : N - 1)) : 0.f;
}

// out_bf16[m, n] = act(acc + bias[n])          act = identity | gelu_new
template <bool kGelu>
struct OpTmaBiasActBF16 {
  static constexpr int kElemBytes = 2;
  struct Params {
    CUtensorMap out_map;  // bf16 [M, N], box 32 rows x 64 cols, SWIZZLE_128B
    const float* bias;    // may be null
    void* out_ptr;        // same tensor as out_map (direct-store variant)
    int ldc;
  };
  struct Row {};
  static __device__ __forceinline__ Row row_init(const Params&, int, int) { return Row(); }
  // 8 consecutive columns starting at `col` -> 16 bytes
  static __device__ __forceinline__ void chunk(const Params& p, const Row&, const uint32_t* acc, int col, int N,
                                               int /*row*/, uint32_t (&o)[4]) {
    float x[8];
    if (p.bias && col + 8 <= N) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col) + 1);
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(acc[i]) + bb[i];
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(acc[i]) + bias_at(p.bias, col + i, N);
    }
    if (kGelu) {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = gelu_new(x[i]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = pack_bf16(x[2 * i], x[2 * i + 1]);
  }
  static __device__ __forceinline__ void issue(const Params& p, const void* box, int n, int m0) {
    tma_store_2d(&p.out_map, box, n, m0);
  }
};

// GPT-J fused q/k/v projection: out_bf16[m, n] = rotary(acc) for the first `rotary_dim` dims of every q and k head
// (HF:gptj/modeling_gptj.py:55-67, 196-207: interleaved pairs (x[2i], x[2i+1]) -> (x[2i] c - x[2i+1] s, x[2i+1] c + x[2i] s)
// with angle pos[m] * 10000^(-2i/rotary_dim)); v columns and the non-rotary dims pass through.  No bias (:98-101).
struct OpTmaRotaryBF16 {
  static constexpr int kElemBytes = 2;
  struct Params {
    CUtensorMap out_map;     // bf16 [M, 3d]
    const int32_t* pos;      // [M] position of each token row
    const float2* table;     // [max_pos, rotary_dim/2] (cos, sin)
    int M, d_model, head_dim, rotary_dim, max_pos;
    void* out_ptr;
    int ldc;
  };
  struct Row {};
  static __device__ __forceinline__ Row row_init(const Params&, int, int) { return Row(); }
  static __device__ __forceinline__ void chunk(const Params& p, const Row&, const uint32_t* acc, int col, int N, int row,
                                               uint32_t (&o)[4]) {
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(acc[i]);
    const int in_head = col % p.head_dim;  // 8-column chunks never straddle heads (head_dim % 8 == 0)
    if (col < 2 * p.d_model && in_head < p.rotary_dim) {
      int ps = __ldg(p.pos + (row < p.M ? row : p.M - 1));
      ps = min(max(ps, 0), p.max_pos - 1);
      const float4* t4 = reinterpret_cast<const float4*>(p.table + static_cast<size_t>(ps) * (p.rotary_dim >> 1) +
                                                         (in_head >> 1));
      const float4 a = __ldg(t4), b = __ldg(t4 + 1);  // (c0,s0,c1,s1), (c2,s2,c3,s3)
      const float cs[4] = {a.x, a.z, b.x, b.z}, sn[4] = {a.y, a.w, b.y, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float e = x[2 * i], od = x[2 * i + 1];
        x[2 * i] = e * cs[i] - od * sn[i];
        x[2 * i + 1] = od * cs[i] + e * sn[i];
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = pack_bf16(x[2 * i], x[2 * i + 1]);
  }
  static __device__ __forceinline__ void issue(const Params& p, const void* box, int n, int m0) {
    tma_store_2d(&p.out_map, box, n, m0);
  }
};

// resid_f32[m, n] += acc + bias[n]      (fp32 residual stream updated in place by a TMA reduce-add)
struct OpTmaResidAddF32 {
  static constexpr int kElemBytes = 4;
  struct Params {
    CUtensorMap out_map;  // fp32 [M, N], box 32 rows x 32 cols, SWIZZLE_128B
    const float* bias;    // may be null
    void* out_ptr;
    int ldc;
  };
  struct Row {};
  static __device__ __forceinline__ Row row_init(const Params&, int, int) { return Row(); }
  // 4 consecutive columns -> 16 bytes
  static constexpr bool kSplitK = true;
  static __device__ __forceinline__ void chunk(const Params& p, const Row&, const uint32_t* acc, int col, int N,
                                               int /*row*/, uint32_t (&o)[4], bool add_bias) {
    const float* bias = add_bias ? p.bias : nullptr;
    if (bias && col + 4 <= N) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(bias + col));
      o[0] = __float_as_uint(__uint_as_float(acc[0]) + b.x);
      o[1] = __float_as_uint(__uint_as_float(acc[1]) + b.y);
      o[2] = __float_as_uint(__uint_as_float(acc[2]) + b.z);
      o[3] = __float_as_uint(__uint_as_float(acc[3]) + b.w);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = __float_as_uint(__uint_as_float(acc[i]) + bias_at(bias, col + i, N));
    }
  }
  static __device__ __forceinline__ void issue(const Params& p, const void* box, int n, int m0) {
    tma_reduce_add_2d(&p.out_map, box, n, m0);
  }
};

// resid_bf16[m, n] += acc + bias[n]     (bf16 residual stream, SGPT_RESID_BF16=1: the add is a bf16 TMA reduce-add
// performed by the L2 — half the epilogue's shared-memory and HBM traffic of the fp32 stream)
struct OpTmaResidAddBF16 {
  static constexpr int kElemBytes = 2;
  struct Params {
    CUtensorMap out_map;  // bf16 [M, N], box 32 rows x 64 cols, SWIZZLE_128B
    const float* bias;    // may be null
    void* out_ptr;
    int ldc;
  };
  struct Row {};
  static __device__ __forceinline__ Row row_init(const Params&, int, int) { return Row(); }
  static constexpr bool kSplitK = true;
  static __device__ __forceinline__ void chunk(const Params& p, const Row&, const uint32_t* acc, int col, int N,
                                               int /*row*/, uint32_t (&o)[4], bool add_bias) {
    const float* bias = add_bias ? p.bias : nullptr;
    float x[8];
    if (bias && col + 8 <= N) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col) + 1);
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(acc[i]) + bb[i];
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(acc[i]) + bias_at(bias, col + i, N);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = pack_bf16(x[2 * i], x[2 * i + 1]);
  }
  static __device__ __forceinline__ void issue(const Params& p, const void* box, int n, int m0) {
    tma_reduce_add_2d(&p.out_map, box, n, m0);
  }
};

// ---- LayerNorm folded into the consumer GEMM -------------------------------------------------------------------------
// y = LN(x) W^T + b  with  LN(x) = (x - mu) r (*) gamma + beta   is evaluated as
//     y[t, n] = r_t * (xb W'^T)[t, n] - r_t mu_t * c[n] + b'[n],
// W' = bf16(W (*) gamma) (gamma folded into the weight columns when the model is created), c[n] = sum_k W'[n, k] (fp32, of
// the ROUNDED folded weights so that the mean term cancels exactly against the GEMM), b'[n] = b[n] + sum_k beta_k W[n, k],
// xb = bf16 copy of the fp32 residual stream (written by the kernel that produced the residual), and (mu_t, r_t) from
// the row's partial sums (ln_row_from_partials).  The separate LayerNorm pass over the residual stream (read 4 B + write
// 2 B per element, twice per block) disappears; the GEMM reads the same number of bytes as before.
// out_bf16[m, n] = act(r_m * acc - rm_m * colsum[n] + bias[n])
template <bool kGelu>
struct OpTmaLnBiasActBF16 {
  static constexpr int kElemBytes = 2;
  struct Params {
    CUtensorMap out_map;   // bf16 [M, N], box 32 rows x 64 cols, SWIZZLE_128B
    const float* bias;     // b'  [N]
    const float* colsum;   // c   [N]
    const float2* stats;   // [M, P] partial (sum x, sum x^2)
    int P;
    float inv_d, eps;
    void* out_ptr;
    int ldc;
  };
  using Row = LnRow;
  static __device__ __forceinline__ Row row_init(const Params& p, int row, int M) {
    return ln_row_from_partials(p.stats, p.P, p.inv_d, p.eps, row, M);
  }
  static __device__ __forceinline__ void chunk(const Params& p, const Row& rc, const uint32_t* acc, int col, int N,
                                               int /*row*/, uint32_t (&o)[4]) {
    float x[8];
    if (col + 8 <= N) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col) + 1);
      const float4 c0 = __ldg(reinterpret_cast<const float4*>(p.colsum + col));
      const float4 c1 = __ldg(reinterpret_cast<const float4*>(p.colsum + col) + 1);
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      const float cc[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = fmaf(rc.r, __uint_as_float(acc[i]), fmaf(-rc.rm, cc[i], bb[i]));
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        x[i] = fmaf(rc.r, __uint_as_float(acc[i]), fmaf(-rc.rm, bias_at(p.colsum, col + i, N), bias_at(p.bias, col + i, N)));
    }
    if (kGelu) {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = gelu_new(x[i]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = pack_bf16(x[2 * i], x[2 * i + 1]);
  }
  static __device__ __forceinline__ void issue(const Params& p, const void* box, int n, int m0) {
    tma_store_2d(&p.out_map, box, n, m0);
  }
};

// GPT-J q/k/v projection with ln_1 folded in (as above, no activation) followed by the rotary embedding of OpTmaRotaryBF16.
struct OpTmaLnRotaryBF16 {
  static constexpr int kElemBytes = 2;
  struct Params {
    OpTmaRotaryBF16::Params rot;
    const float* bias;     // b' [3d]
    const float* colsum;   // c  [3d]
    const float2* stats;
    int P;
    float inv_d, eps;
    void* out_ptr;  // (direct-store debug variant of the driver only)
    int ldc;
  };
  using Row = LnRow;
  static __device__ __forceinline__ Row row_init(const Params& p, int row, int M) {
    return ln_row_from_partials(p.stats, p.P, p.inv_d, p.eps, row, M);
  }
  static __device__ __forceinline__ void chunk(const Params& p, const Row& rc, const uint32_t* acc, int col, int N, int row,
                                               uint32_t (&o)[4]) {
    uint32_t y[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      y[i] = __float_as_uint(fmaf(rc.r, __uint_as_float(acc[i]),
                                  fmaf(-rc.rm, bias_at(p.colsum, col + i, N), bias_at(p.bias, col + i, N))));
    OpTmaRotaryBF16::chunk(p.rot, OpTmaRotaryBF16::Row(), y, col, N, row, o);
  }
  static __device__ __forceinline__ void issue(const Params& p, const void* box, int n, int m0) {
    tma_store_2d(&p.rot.out_map, box, n, m0);
  }
};

// ---- residual epilogue that also feeds the NEXT LayerNorm --------------------------------------------------------------
// resid_f32[m, n] = resid_f32[m, n] + acc + bias[n]  (out-proj / c_proj), and in the same pass
//     xb_bf16[m, n] = bf16(new residual)                       (A operand of the next QKV / c_fc GEMM)
//     stats[m, n / 128] = (sum, sum of squares) of the new residual over this warp's 128 columns
// The old residual is fetched by TMA into a per-warp smem box (two boxes in flight: the first two loads of a tile are
// issued BEFORE the accumulator is waited for, the rest chase the stores), updated in place by the row-owning threads
// and written back with a TMA store; the bf16 copy leaves through a second box.  8 epilogue warps; BN = 256 only (each
// warp then owns exactly one 128-column statistics group).  N % 64 == 0.
struct EpiResidLn {
  struct Params {
    CUtensorMap resid_map;  // fp32 [M, N], box 32 rows x 32 cols, SWIZZLE_128B (load and store)
    CUtensorMap xb_map;     // bf16 [M, N], box 32 rows x 64 cols, SWIZZLE_128B
    const float* bias;      // may be null
    float2* stats;          // [M, P]
    int P;
    int l2_prefetch;        // prefetch the NEXT tile's residual boxes into L2 one tile ahead (hides the HBM latency)
  };
  struct State {
    uint32_t it;     // residual boxes processed so far by this warp (selects the load buffer and its barrier phase)
    uint64_t* bars;  // two mbarriers of this warp
  };
  static constexpr int kEpiWarps = 8;
  static constexpr int kStagingBytes = 8 * 12288;  // per warp: two fp32 load/store boxes + one bf16 store box
  static __device__ __forceinline__ void init(State& st, const Params&, int lane_row, uint64_t* bars) {
    st.it = 0;
    st.bars = bars;
    if ((lane_row & 31) == 0) {
      mbar_init(&bars[0], 1);
      mbar_init(&bars[1], 1);
      fence_mbar_init();
    }
    __syncwarp();
  }
  static __device__ __forceinline__ void finish(State&, const Params&, int lane_row) {
    if ((lane_row & 31) == 0) bulk_wait_group<0>();
  }
  // called right before pre_tile of the current tile with the coordinates of the tile AFTER it
  static __device__ __forceinline__ void prefetch_next(const Params& p, int m0, int n0, int lane, int M, int N) {
    if (!p.l2_prefetch || m0 >= M || lane != 0) return;
    const int nb = boxes(n0, N, 128);
    for (int j = 0; j < nb; ++j) tma_prefetch_l2_2d(&p.resid_map, n0 + 32 * j, m0);
  }
  static __device__ __forceinline__ int boxes(int n0, int N, int cols) {
    if (n0 >= N) return 0;
    const int left = (N - n0) >> 5;
    return left < (cols >> 5) ? left : (cols >> 5);
  }

  template <int COLS, int kSlabBytes>
  static __device__ __forceinline__ void pre_tile(State& st, const Params& p, int m0, int n0, int lane, float* slab,
                                                  int M, int N) {
    static_assert(COLS == 128 && kSlabBytes == 12288, "EpiResidLn: 128 columns and 12 KB of staging per warp");
    if (m0 >= M) return;
    const int nb = boxes(n0, N, COLS);
    if (nb <= 0) return;
    if (lane == 0) {
      bulk_wait_group_read<0>();  // the previous tile's stores have finished reading all three boxes
      const uint32_t sbase = smem_u32(slab);
      for (int j = 0; j < 2 && j < nb; ++j) {
        const uint32_t b = (st.it + j) & 1u;
        mbar_expect_tx(&st.bars[b], 4096);
        tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(sbase + b * 4096u)), &p.resid_map, &st.bars[b],
                    n0 + 32 * j, m0);
      }
    }
    __syncwarp();
  }

  template <int COLS, int kSlabBytes>
  static __device__ __forceinline__ void tile(State& st, const Params& p, int m0, int n0, int lane, uint32_t trow,
                                              float* slab, int M, int N) {
    if (m0 >= M) return;
    const int nb = boxes(n0, N, COLS);
    if (nb <= 0) return;
    const uint32_t sbase = smem_u32(slab);
    const uint32_t hbox = sbase + 8192u;
    const uint32_t hrow = hbox + lane * 128u;
    float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
    for (int c = 0; c < nb; ++c) {
      const uint32_t b = st.it & 1u, ph = (st.it >> 1) & 1u;
      const uint32_t fb = sbase + b * 4096u;
      const int n = n0 + 32 * c;
      uint32_t v[32];
      tmem_ld_32x32(trow + 32 * c, v);
      mbar_wait(&st.bars[b], ph);  // old residual box has landed
      tmem_ld_wait();
      const uint32_t row_addr = fb + lane * 128u;
      uint32_t h[16];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t a = row_addr + ((j ^ (lane & 7)) << 4);
        const float4 old = lds_v4(a);
        float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias != nullptr) bz = __ldg(reinterpret_cast<const float4*>(p.bias + n) + j);
        const float x0 = old.x + (__uint_as_float(v[4 * j]) + bz.x), x1 = old.y + (__uint_as_float(v[4 * j + 1]) + bz.y);
        const float x2 = old.z + (__uint_as_float(v[4 * j + 2]) + bz.z), x3 = old.w + (__uint_as_float(v[4 * j + 3]) + bz.w);
        sts_v4(a, __float_as_uint(x0), __float_as_uint(x1), __float_as_uint(x2), __float_as_uint(x3));
        s1 += (x0 + x1) + (x2 + x3);
        s2 += (x0 * x0 + x1 * x1) + (x2 * x2 + x3 * x3);
        h[2 * j] = pack_bf16(x0, x1);
        h[2 * j + 1] = pack_bf16(x2, x3);
      }
      // bf16 copy: these 32 columns are chunks 4 (c & 1) .. + 3 of the row's 128-byte segment in the 64-column box
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4)
        sts_v4(hrow + (((((c & 1) << 2) + q4) ^ (lane & 7)) << 4), h[4 * q4], h[4 * q4 + 1], h[4 * q4 + 2], h[4 * q4 + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&p.resid_map, reinterpret_cast<const void*>(__cvta_shared_to_generic(fb)), n, m0);
        if (c & 1) tma_store_2d(&p.xb_map, reinterpret_cast<const void*>(__cvta_shared_to_generic(hbox)), n - 32, m0);
        bulk_commit_group();
        if (c + 2 < nb) {
          bulk_wait_group_read<0>();  // this box (and the bf16 box) may be overwritten now
          mbar_expect_tx(&st.bars[b], 4096);
          tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(fb)), &p.resid_map, &st.bars[b], n + 64, m0);
        }
      }
      __syncwarp();
      ++st.it;
    }
    if (m0 + lane < M) p.stats[static_cast<size_t>(m0 + lane) * p.P + (n0 >> 7)] = make_float2(s1, s2);
  }
};

// ---------------------------------------------------------------------------------------------------------------
// Staged epilogue driver: TMEM -> registers (thread = row) -> smem slab -> (lane = column pair) -> Op::rows()
// The slab is [32 rows][32 column pairs] of float2 without padding; pair p of row r is stored at p ^ (r & 15), which
// makes both the row-wise writes and the column-wise reads bank-conflict free for 8-byte accesses.
// ---------------------------------------------------------------------------------------------------------------
struct EpiNoState {};

template <class Op>
struct EpiStaged {
  using Params = typename Op::Params;
  using State = EpiNoState;
  static constexpr int kEpiWarps = 4;
  static __device__ __forceinline__ void init(State&, const Params&, int, uint64_t*) {}
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void pre_tile(State&, const Params&, int, int, int, float*, int, int) {}
  static __device__ __forceinline__ void finish(State&, const Params&, int) {}

  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void tile(State&, const Params& p, int m0, int n0, int lane, uint32_t trow,
                                              float* slab_ptr, int M, int N) {
    const int rows = min(32, M - m0);  // warp-uniform; <= 0 when the whole slab is out of range
    const uint32_t slab = smem_u32(slab_ptr);
#pragma unroll 1
    for (int c = 0; c < BN; c += 64) {
      const int n = n0 + c;
      if (n >= N) break;  // warp-uniform
      uint32_t v0[32], v1[32];
      tmem_ld_32x32(trow + c, v0);
      if (n + 32 < N) {
        tmem_ld_32x32(trow + c + 32, v1);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v1[i] = 0u;
      }
      tmem_ld_wait();
      __syncwarp();  // the previous slab's readers are done
      const uint32_t wrow = slab + lane * 256u;
      const uint32_t sw = lane & 15;
#pragma unroll
      for (int i = 0; i < 16; ++i) sts_v2(wrow + ((i ^ sw) << 3), v0[2 * i], v0[2 * i + 1]);
#pragma unroll
      for (int i = 0; i < 16; ++i) sts_v2(wrow + (((16 + i) ^ sw) << 3), v1[2 * i], v1[2 * i + 1]);
      __syncwarp();
      if (rows > 0) Op::rows(p, slab, m0, rows, n + 2 * lane, N, lane);
    }
  }
};

// columns (2*lane, 2*lane+1) of staged row r
__device__ __forceinline__ float2 slab_read(uint32_t slab, int r, int lane) {
  return lds_v2(slab + r * 256u + ((lane ^ (r & 15)) << 3));
}

// scores_f32[q, doc] = fixnan(acc * row_scale[q] * col_scale[doc])       (cos_sim / dot_score, NaN -> -1)
// (kS8: the staged accumulator holds s32 values of an int8 launch, converted to fp32 before the scaling)
struct ScoresF32Params {
  float* out;
  const float* row_scale;  // per query  (1/||q|| for cos_sim; null = 1)
  const float* col_scale;  // per doc    (1/||d|| for cos_sim; null = 1)
  long long ldc;
};
template <bool kS8 = false>
struct OpScoresF32T {
  using Params = ScoresF32Params;
  static __device__ __forceinline__ void rows(const Params& p, uint32_t slab, int m0, int rows, int col, int N,
                                              int lane) {
    const bool ok0 = col < N, ok1 = col + 1 < N;
    float c0 = 1.f, c1 = 1.f;
    if (p.col_scale) {
      if (ok0) c0 = __ldg(p.col_scale + col);
      if (ok1) c1 = __ldg(p.col_scale + col + 1);
    }
    const bool vec = ok1 && ((p.ldc & 1) == 0);
    float* dst = p.out + static_cast<size_t>(m0) * p.ldc + col;
    float my_rs = 1.f;  // lane r keeps row m0 + r's scale; broadcast per row with a shuffle
    if (p.row_scale && lane < rows) my_rs = __ldg(p.row_scale + m0 + lane);
    int r = 0;
    for (; r + 8 <= rows; r += 8) {
      float2 a[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) a[u] = slab_read(slab, r + u, lane);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float rs = __shfl_sync(0xffffffffu, my_rs, r + u);
        float x = acc_to_f32<kS8>(__float_as_uint(a[u].x)) * rs * c0, y = acc_to_f32<kS8>(__float_as_uint(a[u].y)) * rs * c1;
        x = (x != x) ? -1.f : x;
        y = (y != y) ? -1.f : y;
        if (vec) *reinterpret_cast<float2*>(dst) = make_float2(x, y);
        else {
          if (ok0) dst[0] = x;
          if (ok1) dst[1] = y;
        }
        dst += p.ldc;
      }
    }
    for (; r < rows; ++r) {
      const float rs = __shfl_sync(0xffffffffu, my_rs, r);
      const float2 a = slab_read(slab, r, lane);
      float x = acc_to_f32<kS8>(__float_as_uint(a.x)) * rs * c0, y = acc_to_f32<kS8>(__float_as_uint(a.y)) * rs * c1;
      x = (x != x) ? -1.f : x;
      y = (y != y) ? -1.f : y;
      if (vec) *reinterpret_cast<float2*>(dst) = make_float2(x, y);
      else {
        if (ok0) dst[0] = x;
        if (ok1) dst[1] = y;
      }
      dst += p.ldc;
    }
  }
};
using OpScoresF32 = OpScoresF32T<false>;

// Threshold filter of the fused search (search.cu): score = fixnan(acc * row_scale[q] * col_scale[doc]); every score
// >= tau[q] is appended as a packed (score bits, local doc index) pair to a candidate list; the score matrix itself is
// never written to HBM.
//
// In the accumulator's native layout thread r of a warp owns query row r, i.e. ONE admission threshold: the compare
// needs no transpose, no shuffles and no ballots.  Each (CTA, column-half) pair is a GROUP with a PRIVATE list per query
// (cand[q][group][L]); the thread keeps its list length in a register across all tiles of the persistent kernel and
// writes it out once at the end, so there are NO atomics at all.  (The first version reserved space in one list per
// query with an atomicAdd per 32-document chunk: ~17 k same-address atomics per counter per search serialised in the
// L2 and, not the HBM stream, set the kernel's duration.)  L is sized for the worst case (every score of every tile the
// CTA visits admitted), so there is no overflow path; only the touched prefix of each list generates memory traffic.
// 8 epilogue warps (two per TMEM lane quarter, half the tile's documents each); no shared memory.
//
// Sample mode (Params::pool != nullptr; pass A of the search): nothing is filtered; the thread writes the MAXIMUM of
// every 4 consecutive documents' scores (32 floats per query and tile half) to pool[q][group][Lp].  Each maximum is the
// score of a distinct real document, so the k-th largest of a query's maxima is a valid lower bound of its final k-th
// best score — at a quarter of the entries (and no document indices) the full sample would need.  Slots this thread never
// fills are written as 0xffffffff (maps to the invalid key 0 of the selection kernels).
struct FilterRowsParams {
  const float* row_scale;  // [M] or null
  const float* col_scale;  // [N] or null
  const float* tau;        // [M] per-query admission threshold; null -> admit everything
  const float* tau_hi;     // [M] upper threshold (>= tau) or null: scores >= tau_hi are appended at the FRONT of the list,
                           // scores in [tau, tau_hi) at its BACK (filled downwards from slot L - 1); null -> all front
  uint2* cand;             // [M][groups][L]
  int* counts;             // [groups][M] front entries
  int* counts_back;        // [groups][M] back entries (only with tau_hi)
  long long stride_q;      // entries between consecutive queries' list blocks
  int L;                   // entries per (query, group) list
  int group0;              // first group index this launch writes
  int nq;
  float* pool;             // sample mode: [M][groups][Lp] block maxima (cand / counts / tau unused)
  long long stride_p;      // floats between consecutive queries' blocks of `pool`
  int Lp;                  // floats per (query, group): 32 x tiles per CTA
  int pair;                // 1: launched as CTA pairs (cta_group::2, M = 256 queries per scan)
};
template <bool kS8>  // kS8: s32 accumulator of an int8 launch
struct EpiFilterRowsT {
  using Params = FilterRowsParams;
  struct State {
    int cnt;    // front entries (sample mode: maxima written)
    int cnt_b;  // back entries
    // per-tile constants fetched in pre_tile, i.e. BEFORE the wait for the accumulator: lane l holds the inverse norms of
    // documents n0 + 4 l .. + 3 of this warp's 128-document half tile (broadcast by shuffles below), the query's scale and
    // its admission threshold.  (Fetched inside the chunk loop, the norms cost one exposed HBM round trip per 32 documents
    // — 4 B per document that nobody else has touched — while the TMA stream saturates the memory system: ~4 serial
    // misses per tile per warp against a tile time of 9 us.)
    float4 cs;
    float rs, tau, tau_hi;
  };
  static constexpr int kEpiWarps = 8;
  // one group per (cluster, column half): with CTA pairs (Params::pair = 1: up to 256 queries per scan, rank r of the pair
  // owns queries 128 r .. 128 r + 127 and all 256 documents of the tile) both CTAs of a pair write the SAME group's lists —
  // of different queries
  static __device__ __forceinline__ int group_of(const Params& p) {
    return p.group0 + static_cast<int>(blockIdx.x >> p.pair) * 2 + static_cast<int>(threadIdx.x >> 7);
  }
  static __device__ __forceinline__ void init(State& st, const Params&, int, uint64_t*) { st.cnt = 0; st.cnt_b = 0; }
  template <int COLS, int kSlabBytes>
  static __device__ __forceinline__ void pre_tile(State& st, const Params& p, int m0, int n0, int lane, float*, int M, int N) {
    static_assert(COLS == 128, "one float4 of document scales per lane covers the warp's half tile");
    const int q = m0 + lane;
    const bool qok = q < M;
    st.rs = (qok && p.row_scale) ? __ldg(p.row_scale + q) : 1.f;
    st.tau = !qok ? INFINITY : (p.tau != nullptr ? __ldg(p.tau + q) : -INFINITY);  // +inf: rows beyond nq admit nothing
    st.tau_hi = (qok && p.tau_hi != nullptr) ? fmaxf(__ldg(p.tau_hi + q), st.tau) : st.tau;
    st.cs = make_float4(1.f, 1.f, 1.f, 1.f);
    if (p.col_scale != nullptr && m0 < M) {
      const int c = n0 + 4 * lane;
      if (c + 4 <= N) {
        st.cs = __ldg(reinterpret_cast<const float4*>(p.col_scale + c));
      } else if (N > 0) {
        st.cs.x = __ldg(p.col_scale + min(c, N - 1));
        st.cs.y = __ldg(p.col_scale + min(c + 1, N - 1));
        st.cs.z = __ldg(p.col_scale + min(c + 2, N - 1));
        st.cs.w = __ldg(p.col_scale + min(c + 3, N - 1));
      }
    }
  }
  static __device__ __forceinline__ void finish(State& st, const Params& p, int lane_row) {
    if (lane_row >= p.nq) return;
    if (p.pool != nullptr) {
      uint32_t* d = reinterpret_cast<uint32_t*>(p.pool + static_cast<long long>(lane_row) * p.stride_p +
                                               static_cast<long long>(group_of(p)) * p.Lp);
      for (int i = st.cnt; i < p.Lp; ++i) d[i] = 0xffffffffu;  // CTAs that visited fewer tiles than the longest
    } else {
      p.counts[static_cast<long long>(group_of(p)) * p.nq + lane_row] = st.cnt;  // cnt + cnt_b <= L by construction
      if (p.counts_back != nullptr) p.counts_back[static_cast<long long>(group_of(p)) * p.nq + lane_row] = st.cnt_b;
    }
  }

  template <int COLS, int kSlabBytes>
  static __device__ __forceinline__ void tile(State& st, const Params& p, int m0, int n0, int lane, uint32_t trow,
                                              float*, int M, int N) {
    if (m0 >= M) return;  // warp-uniform
    const int q = m0 + lane;
    const bool qok = q < M;
    const float rs = st.rs;
    const bool pooled = (p.pool != nullptr);
    const float tau = st.tau, tau_hi = st.tau_hi;
    const bool nan_path = __any_sync(0xffffffffu, !pooled && tau <= -1.0f) != 0;  // warp-uniform
    const float csv[4] = {st.cs.x, st.cs.y, st.cs.z, st.cs.w};
    uint2* dst = p.cand + static_cast<long long>(qok ? q : 0) * p.stride_q + static_cast<long long>(group_of(p)) * p.L;
    int cnt = st.cnt, cnt_b = st.cnt_b;
#pragma unroll 1
    for (int c = 0; c < COLS; c += 32) {
      const int n = n0 + c;
      if (n >= N) break;  // warp-uniform
      uint32_t v[32];
      tmem_ld_32x32(trow + c, v);
      const bool full = (n + 32 <= N);
      // scale of column c + i: component i % 4 of lane (c + i) / 4 (all lanes take part: the loop is warp-uniform)
      float cs[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) cs[i] = __shfl_sync(0xffffffffu, csv[i & 3], (c >> 2) + (i >> 2));
      tmem_ld_wait();
      // XS:99 maps a NaN score to -1.  While tau > -1 (always, except for degenerate corpora) a NaN fails `x >= tau` exactly
      // as its image -1 would, and in sample mode fmaxf drops it (a smaller maximum keeps tau a valid lower bound): the
      // explicit mapping (two instructions per score) is only executed when some row of the warp could admit a -1.
      float x[32];
      if (nan_path) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float s = acc_to_f32<kS8>(v[i]) * rs * cs[i];
          x[i] = (s != s) ? -1.f : s;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) x[i] = acc_to_f32<kS8>(v[i]) * rs * cs[i];
      }
      if (pooled) {
        // sample pass: maxima of 4 consecutive documents, two 16-byte stores (cnt is a multiple of 8, the lists 32-byte
        // aligned); documents beyond the shard never win
        float m[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float mx = -INFINITY;
#pragma unroll
          for (int u = 0; u < 4; ++u) mx = (full || n + 4 * j + u < N) ? fmaxf(mx, x[4 * j + u]) : mx;
          m[j] = mx;
        }
        if (qok && cnt + 8 <= p.Lp) {
          float4* d4 = reinterpret_cast<float4*>(p.pool + static_cast<long long>(q) * p.stride_p +
                                                 static_cast<long long>(group_of(p)) * p.Lp + cnt);
          d4[0] = make_float4(m[0], m[1], m[2], m[3]);
          d4[1] = make_float4(m[4], m[5], m[6], m[7]);
        }
        cnt += 8;
      } else {
        // Branch-free admission: one predicated 8-byte store per score, the two list lengths advance by predicates.  (With
        // a branch per score — taken by SOME lane for ~60 % of the scores at a 3 % admission rate — the 32 convergence
        // regions per chunk were the longest dependent chain of the epilogue.)  cnt + cnt_b never exceeds L: L is every
        // score of every tile this CTA visits (checked by the launcher).
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const bool pass = (full || n + i < N) && x[i] >= tau;  // tau = +inf for rows beyond the query count
          const bool hi = x[i] >= tau_hi;
          const uint32_t slot = static_cast<uint32_t>(hi ? cnt : (p.L - 1 - cnt_b));  // unsigned: one IMAD.WIDE.U32 per address
          // (a predicated store in PTX: as plain C++ the compiler wraps the store and its address arithmetic in a branch)
          asm volatile(
              "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.global.v2.u32 [%1], {%2, %3};\n\t}\n" ::"r"(
                  static_cast<uint32_t>(pass)),
              "l"(dst + slot), "r"(__float_as_uint(x[i])), "r"(static_cast<uint32_t>(n + i))
              : "memory");
          cnt += (pass && hi) ? 1 : 0;
          cnt_b += (pass && !hi) ? 1 : 0;
        }
      }
    }
    st.cnt = cnt;
    st.cnt_b = cnt_b;
  }
};
using EpiFilterRows = EpiFilterRowsT<false>;
using EpiFilterRowsS8 = EpiFilterRowsT<true>;
using EpiFilterCandidates = EpiFilterRows;


template <bool kGelu>
struct Epi16Of<EpiTma<OpTmaBiasActBF16<kGelu>, 0>> { using type = EpiTma16<OpTmaBiasActBF16<kGelu>>; };
template <>
struct Epi16Of<EpiTma<OpTmaResidAddBF16, 0>> { using type = EpiTma16<OpTmaResidAddBF16>; };

template <bool kGelu>
using EpiBiasActBF16 = EpiTma<OpTmaBiasActBF16<kGelu>>;
using EpiResidualF32 = EpiTma<OpTmaResidAddF32>;
using EpiResidualBF16 = EpiTma<OpTmaResidAddBF16>;
using EpiRotaryBF16 = EpiTma<OpTmaRotaryBF16>;
template <bool kGelu>
using EpiLnBiasActBF16 = EpiTma<OpTmaLnBiasActBF16<kGelu>>;
using EpiLnRotaryBF16 = EpiTma<OpTmaLnRotaryBF16>;

// Bring-up / profiling aids (sgpt_linear epilogue codes 100, 101): no epilogue work at all, or TMEM loads only.
template <bool kLoad>
struct EpiDebugNull {
  struct Params { int dummy; };
  using State = EpiNoState;
  static constexpr int kEpiWarps = 4;
  static __device__ __forceinline__ void init(State&, const Params&, int, uint64_t*) {}
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void pre_tile(State&, const Params&, int, int, int, float*, int, int) {}
  static __device__ __forceinline__ void finish(State&, const Params&, int) {}
  template <int BN, int kSlabBytes>
  static __device__ __forceinline__ void tile(State&, const Params&, int, int, int, uint32_t trow, float*, int, int) {
    if (kLoad) {
      uint32_t acc = 0;
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        uint32_t v[32];
        tmem_ld_32x32(trow + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) acc ^= v[i];
      }
      if (acc == 0x12345678u) printf("~");  // keep the loads alive
    }
  }
};
using EpiScoresF32 = EpiStaged<OpScoresF32>;
using EpiScoresF32S8 = EpiStaged<OpScoresF32T<true>>;

}  // namespace sgpt

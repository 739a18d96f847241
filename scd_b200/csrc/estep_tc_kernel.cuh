// k-means E-step on the tcgen05 tensor cores (SURVEY 8a rows a1 + a2).
//
//   dist[n, k] = ||x_n||^2 - 2 x_n . c_k + ||c_k||^2      labels[n] = argmin_k (ties -> lowest k, NaN wins)
//   replaces  pairwise_distance (local_utils/faster_mix_k_means_pytorch.py:177-212) + torch.min (:59 / :106)
//
// The reference computes sum_d (x - c)^2 directly in fp32.  A single bf16 pass of the x.c contraction
// cannot keep its 1e-4 / argmin-margin parity once the centroids are fp32 means (BASELINE.md section 5),
// so the contraction is issued as three bf16 MMAs with fp32 accumulation:
//     x.c ~= x_hi.c_hi + x_hi.c_lo + x_lo.c_hi        (x_hi = bf16(x), x_lo = bf16(x - x_hi); same for c)
// which measures 3.8e-7 max abs error on unit-norm data (the fp32 direct form: 2.6e-7).
//
// X stays fp32 in HBM and is read exactly ONCE per E-step: TMA brings 128 x 32 fp32 tiles into a ring,
// four converter warps (thread = row) split them into the hi / lo bf16 A operand and accumulate ||x||^2 on
// the way.  Where the converted operand goes is the template parameter:
//   kTmemA = true  (n_tile <= 160, i.e. K <= 160): into TENSOR MEMORY (tcgen05.st, thread = row = TMEM lane, one 32-bit
//       column = two consecutive k), in the columns the double-buffered accumulators leave free, and the MMAs take A
//       from TMEM.  Per 32-wide k-block this removes 16 KB of converter stores and 24 KB of MMA operand reads from
//       shared memory - the round-1 kernel moved 107 KB per k-block through shared memory (~840 cycles at 128 B/clk
//       against ~340 cycles of tensor work) and sat at 0.5 of the HBM roofline, shared-memory-bandwidth bound
//       (profiles/r1_estep_cycle_counters.txt) - and the 48 KB of the old A ring become three more X stages in flight.
//   kTmemA = false (wider centroid tiles, no free TMEM columns): K-major operand tiles in shared memory (SWIZZLE_64B
//       layout written by hand, fence.proxy.async, mbarrier hand-off to the MMA warp).
// The centroid hi / lo planes (+ ||c||^2) are prepared per iteration by a tiny kernel and streamed from L2.  Accumulators live in TMEM (2 x 256 columns, double buffered); the
// epilogue warps (thread = row) fold  ||c||^2 - 2 acc  into a running argmin, so [N, K] never exists.
// HBM-bound while 3 * K <~ 500 (K = 100 / 120 / 200); tensor-bound for K = 1000 (SURVEY 8d).
//
// Warp roles (608 threads, 1 CTA / SM, persistent over 128-row tiles):
//   0, 3 X TMA producers (alternate k-blocks) | 1, 16, 17 MMA issuers (k-blocks round-robin, named-barrier token) |
//   2 (also the TMEM allocator), 18 centroid TMA producers (alternate k-blocks; hi + lo planes as one 3-D box) |
//   4-11 converters (two sets of four warps that take alternate k-blocks, so every scheduler has two conversions in
//   flight) | 12-15 epilogue
#pragma once
#include "ptx.cuh"
#include <cuda_bf16.h>
#include <utility>

namespace scd {

constexpr int kEsBM = 128;              // rows per tile
constexpr int kEsBK = 32;               // k per stage
constexpr int kEsMaxXStages = 12;       // fp32 X ring: as deep as shared memory allows (host picks EsParams::x_stages)
constexpr int kEsAStages = 3;           // converted hi/lo ring in shared memory (kTmemA = false)
constexpr int kEsMaxAStages = 8;        // ... in tensor memory (kTmemA = true): 32 columns per stage, up to 4 above each accumulator
constexpr int kEsBStages = 3;           // centroid hi/lo ring, kTmemA = false
constexpr int kEsMaxBStages = 6;        // ... kTmemA = true (narrow centroid tiles: six stages still leave >= 6 X stages)
__host__ __device__ constexpr int es_b_stages(bool tmem_a) { return tmem_a ? kEsMaxBStages : kEsBStages; }
constexpr int kEsXBytes = kEsBM * kEsBK * 4;          // 16384
constexpr int kEsAPlane = kEsBM * kEsBK * 2;          // 8192 (one of hi / lo)
constexpr int kEsConvSets = 2;          // converter warp sets (4 warps each), alternating k-blocks; a third set (736 threads,
                                        // 80 registers) measured no faster: the converters then wait for X (HBM)
constexpr int kEsIssuers = 3;           // MMA issuer warps (1, 16, 17), k-blocks round-robin
constexpr int kEsFirstExtraIssuer = 4 + 4 * kEsConvSets + 4;       // warps 16, 17
constexpr int kEsSecondCProducer = kEsFirstExtraIssuer + kEsIssuers - 1;   // warp 18
constexpr int kEsThreads = 32 * (kEsSecondCProducer + 1);          // 608: one scheduler holds five warps, so still 96 registers
constexpr int kEsMaxK = 1024;

// Dynamic shared memory: [X ring: x_stages x 16 KB][A ring: 3 x (hi, lo) x 8 KB, kTmemA = false only][B ring: 3 x (hi, lo) x b_plane]
// [tail: barriers, TMEM pointer, ||c||^2, ||x||^2 ring].  The E-step is HBM-latency bound (ncu, round 1: the
// converters wait on x_full), so whatever the centroid ring does not need goes to X stages in flight.
struct EsTail {
  static constexpr int x_full = 0;                                              // [12]
  static constexpr int x_empty = x_full + 8 * kEsMaxXStages;
  static constexpr int a_full = x_empty + 8 * kEsMaxXStages;                    // [8]
  static constexpr int a_empty = a_full + 8 * kEsMaxAStages;
  static constexpr int b_full = a_empty + 8 * kEsMaxAStages;                    // [6]
  static constexpr int b_empty = b_full + 8 * kEsMaxBStages;
  static constexpr int t_full = b_empty + 8 * kEsMaxBStages;                    // [2]
  static constexpr int t_empty = t_full + 16;
  static constexpr int drain = t_empty + 16;                                    // every issuer's last commit has landed
  static constexpr int tmem_ptr = drain + 16;
  static constexpr int cnorm = tmem_ptr + 16;                                   // [kEsMaxK] floats
  static constexpr int xnorm = cnorm + 4 * kEsMaxK;                             // [4 tiles][sets][128] floats
  static constexpr int total = xnorm + 4 * 4 * kEsConvSets * kEsBM;
};
constexpr int kEsSmemLimit = 232448;    // 227 KB opt-in maximum per CTA

struct EsParams {
  long long n_rows;
  int n_clusters;          // K
  int n_tile;              // UMMA N (multiple of 16, <= 256)
  int n_ntiles;            // ceil(K / 256) (1 for K <= 256)
  int num_kb;              // ceil(D / 32)
  int n_row_tiles;
  int x_stages;            // depth of the fp32 X ring (2 .. kEsMaxXStages), EVEN: a stage must belong to one producer /
                           // converter-set pair (see scd_estep)
  int b_plane;             // bytes of one centroid plane stage: n_tile * 64 (n_tile % 16 == 0, so a multiple of 1024)
  int a_stages;            // depth of the converted-operand ring: kEsAStages = 3 (shared memory) or 6 (TMEM) - a multiple of
                           // the issuer count; never more than 2 * num_kb, so the 4-deep ||x||^2 ring cannot be overrun
  const float* cnorm;      // [K]
  long long* labels;       // [N]
  float* mindist;          // nullable [N]
  double* inertia;         // nullable
  long long* prof;         // nullable: [CTAs][16] cycle counters (scd_debug_set_name_profile), debugging aid
};

// host + device: byte offsets of the rings for a given plan
struct EsLayout {
  int x_off, a_off, b_off, tail_off, total;
  __host__ __device__ EsLayout(int x_stages, int b_plane, bool tmem_a) {
    x_off = 0;
    a_off = x_off + x_stages * kEsXBytes;
    b_off = a_off + (tmem_a ? 0 : kEsAStages * 2 * kEsAPlane);
    tail_off = b_off + es_b_stages(tmem_a) * 2 * b_plane;
    total = tail_off + EsTail::total;
  }
};

// ---- The E-step's centroid operands: bf16 hi / lo planes [K, D] and ||c||^2 [K].  centroid_split_kernel,
// finalize_centers_kernel and finalize_centers_peer_kernel write them, and SCD_ESTEP_PLANES_READY needs all three to give
// the same bits: each uses es_store_split, and sums ||c_k||^2 in one block of kEsCentroidThreads threads (thread t
// accumulates d = t, t + kEsCentroidThreads, .. with fmaf, then block_sum_to_thread0).
constexpr int kEsCentroidThreads = 256;

__device__ __forceinline__ void es_store_split(float c, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t i) {
  const __nv_bfloat16 h = __float2bfloat16_rn(c);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(c - __bfloat162float(h));
}

// block-wide sums of per-thread floats in a fixed order: __shfl_down tree in each warp, then thread 0 adds the warps in
// order; the totals are left in thread 0's arguments only.  Each value gets its own shared array (block_sum_slot): one
// [n][32] array instead made ptxas schedule the finalize kernels differently.  At most one call per kernel: the slots are
// static and there is no barrier after thread 0 reads them, so a second call could overwrite them under that read.
template <int I> __device__ __forceinline__ float* block_sum_slot() { __shared__ float sh[32]; return sh; }
template <int... I, typename... F>
__device__ __forceinline__ void block_sum_to_thread0(std::integer_sequence<int, I...>, F&... v) {
  for (int off = 16; off > 0; off >>= 1) ((v += __shfl_down_sync(0xffffffffu, v, off)), ...);
  if ((threadIdx.x & 31) == 0) ((block_sum_slot<I>()[threadIdx.x >> 5] = v), ...);
  __syncthreads();
  if (threadIdx.x == 0) {
    ((v = 0.f), ...);
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) ((v += block_sum_slot<I>()[w]), ...);
  }
}
template <typename... F>
__device__ __forceinline__ void block_sum_to_thread0(F&... v) {
  block_sum_to_thread0(std::make_integer_sequence<int, sizeof...(F)>{}, v...);
}

// fp32 centroids -> the operands above
__global__ void centroid_split_kernel(const float* __restrict__ C, int K, int D, __nv_bfloat16* __restrict__ hi,
                                      __nv_bfloat16* __restrict__ lo, float* __restrict__ cnorm) {
  const int k = blockIdx.x;
  float part = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float c = C[(long long)k * D + d];
    es_store_split(c, hi, lo, (long long)k * D + d);
    part = fmaf(c, c, part);
  }
  block_sum_to_thread0(part);
  if (threadIdx.x == 0) cnorm[k] = part;
}

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ float fmin_nan(float a, float b) {        // NaN if either input is NaN
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

__device__ __forceinline__ bool es_better(float cand, float cur) {
  return (cand < cur) || (cand != cand && cur == cur);      // torch.min: strict '<', a NaN beats any number
}

// TMEM column of A stage s (kTmemA): stages alternate between the free columns above accumulator 0 and accumulator 1;
// hi plane = 16 columns (32 k), lo plane = the next 16
__device__ __forceinline__ uint32_t es_a_col(int s, int n_tile) { return (uint32_t)((s & 1) * 256 + n_tile + (s >> 1) * 32); }

template <bool kTmemA>
__global__ void __launch_bounds__(kEsThreads, 1)
estep_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_c, const EsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sbase = ptx::smem_u32(smem);
  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31;
  const int nkb = p.num_kb;
  const EsLayout L(p.x_stages, p.b_plane, kTmemA);
  const int kEsXStages = p.x_stages;
  const int n_as = p.a_stages;
  constexpr uint32_t kNB = (uint32_t)es_b_stages(kTmemA);      // centroid ring depth

  auto bar = [&](int base, int i) { return sbase + L.tail_off + base + 8 * i; };
  const bool prof = p.prof != nullptr;
  long long* const pf = prof ? p.prof + (size_t)blockIdx.x * 16 : nullptr;
  auto twait = [&](uint32_t b, uint32_t parity, int tag, long long& acc) {
    if (!prof) { ptx::mbar_wait(b, parity, tag); return; }
    const long long c0 = clock64();
    ptx::mbar_wait(b, parity, tag);
    acc += clock64() - c0;
  };

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_c);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kEsXStages; ++s) { ptx::mbar_init(bar(EsTail::x_full, s), 1); ptx::mbar_init(bar(EsTail::x_empty, s), 4); }
    for (int s = 0; s < n_as; ++s) { ptx::mbar_init(bar(EsTail::a_full, s), 4); ptx::mbar_init(bar(EsTail::a_empty, s), 1); }
    for (int s = 0; s < kNB; ++s) { ptx::mbar_init(bar(EsTail::b_full, s), 1); ptx::mbar_init(bar(EsTail::b_empty, s), 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(bar(EsTail::t_full, b), 1); ptx::mbar_init(bar(EsTail::t_empty, b), 4); }
    ptx::mbar_init(bar(EsTail::drain, 0), kEsIssuers);
    ptx::fence_mbar_init_cluster();
  }
  if (warp == 2) {
    ptx::tmem_alloc<1>(sbase + L.tail_off + EsTail::tmem_ptr, 512);
    ptx::tmem_relinquish<1>();
  }
  {
    float* cn = reinterpret_cast<float*>(smem + L.tail_off + EsTail::cnorm);
    for (int k = threadIdx.x; k < p.n_clusters; k += blockDim.x) cn[k] = p.cnorm[k];
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + L.tail_off + EsTail::tmem_ptr);

  if (warp == 0 || warp == 3) {
    // =================================================== X TMA producers (warp 0: even k-blocks, warp 3: odd)
    // One warp gets one tensor box out of L2/HBM every ~400-550 cycles whatever its size, several warps issue
    // independently (tools/tma_feed_bench.cu): with a single producer thread issuing X + hi + lo (72 boxes per row
    // tile) this kernel sat at 0.51 of the HBM roofline, issue-bound.  Ring slots and parities derive from the
    // running k-block index g, exactly as in the converters.
    if (lane == 0) {
      const uint32_t me = warp == 0 ? 0u : 1u;
      uint32_t g = 0;
      long long w_xe = 0; const long long t0 = prof ? clock64() : 0;
      for (int rt = blockIdx.x; rt < p.n_row_tiles; rt += gridDim.x) {
        for (int nt = 0; nt < p.n_ntiles; ++nt) {
          for (int kb = 0; kb < nkb; ++kb, ++g) {
            if ((g & 1u) != me) continue;
            const uint32_t xs = g % kEsXStages, xph = (g / kEsXStages) & 1u;
            twait(bar(EsTail::x_empty, xs), xph ^ 1, 700 + xs, w_xe);
            ptx::mbar_arrive_expect_tx(bar(EsTail::x_full, xs), kEsXBytes);
            ptx::tma_load_2d<1>(sbase + L.x_off + xs * kEsXBytes, &map_x, bar(EsTail::x_full, xs), kb * kEsBK, rt * kEsBM,
                                p.n_ntiles > 1 ? ptx::kEvictNormal : ptx::kEvictFirst);
          }
        }
      }
      if (prof && warp == 0) { pf[0] = clock64() - t0; pf[1] = w_xe; }
    }
  } else if (warp == 2 || warp == kEsSecondCProducer) {
    // =================================================== centroid TMA producers: hi + lo planes in ONE 3-D box
    // (warp 2: even k-blocks, warp 18: odd - one warp gets one box out of L2 every ~500-600 cycles, which is the
    // whole k-block budget once the MMAs run at the tensor pipe's rate)
    if (lane == 0) {
      const uint32_t me = warp == 2 ? 0u : 1u;
      const uint32_t b_bytes = 2u * (uint32_t)p.n_tile * kEsBK * 2u;
      uint32_t g = 0;
      long long w_be = 0;
      for (int rt = blockIdx.x; rt < p.n_row_tiles; rt += gridDim.x) {
        for (int nt = 0; nt < p.n_ntiles; ++nt) {
          for (int kb = 0; kb < nkb; ++kb, ++g) {
            if ((g & 1u) != me) continue;
            const uint32_t bs = g % kNB, bph = (g / kNB) & 1u;
            twait(bar(EsTail::b_empty, bs), bph ^ 1, 710 + bs, w_be);
            ptx::mbar_arrive_expect_tx(bar(EsTail::b_full, bs), b_bytes);
            ptx::tma_load_3d(sbase + L.b_off + bs * 2 * p.b_plane, &map_c, bar(EsTail::b_full, bs), kb * kEsBK, nt * 256, 0,
                             ptx::kEvictLast);
          }
        }
      }
      if (prof && warp == 2) pf[2] = w_be;
    }
  } else if (warp == 1 || (warp >= kEsFirstExtraIssuer && warp < kEsFirstExtraIssuer + kEsIssuers - 1)) {
    // =================================================== MMA issuers (warps 1, 16, 17), k-blocks round-robin
    // tools/mma_rate_bench.cu: the pipe runs a 128 x N x 16 MMA in N/2 cycles only when the next one is already queued;
    // an issuer that recomputes its descriptors between MMAs pays a ~96-cycle floor per MMA (N = 112: 56 ideal), because
    // tcgen05.mma keeps the uniform registers of its descriptors busy until it has run.  With ONE issuing thread this
    // kernel spent ~150 cycles per MMA, ~900 per k-block against a 710-cycle HBM budget (profiles/r1_estep_cycle_
    // counters.txt; moving A into TMEM did not change that).  So, as in the naming kernel, three warps take the k-blocks
    // round-robin: each prepares its six MMAs' operands and does its barrier waits while the other two warps' MMAs run,
    // waits for a named-barrier token (ids 1..3), fires its MMAs back to back and hands the token on before committing.
    // The token keeps the issue order = the pipe's execution order, so the last k-block's commit covers the whole tile.
    // Issuer `me` owns k-blocks g = me, me + 3, ...: the centroid and A rings are 3 or 6 deep, so its stages are always
    // `me` (or alternate me, me + 3) and every descriptor is LOOP INVARIANT: computed once, selected by the unroll index.
    static_assert(kEsBStages == kEsIssuers && kEsMaxBStages == 2 * kEsIssuers, "an issuer's centroid stages must be fixed");
    static_assert(kEsConvSets == 2, "X producers and converter sets pair up by the parity of g (even X ring, see scd_estep)");
    constexpr int kASets = kTmemA ? 2 : 1;                       // A stages per issuer (a_stages = 3 * kASets)
    constexpr int kBSets = (int)kNB / kEsIssuers;                // centroid stages per issuer
    constexpr int kSets = kASets > kBSets ? kASets : kBSets;     // k-blocks per unrolled issuer step
    const uint32_t me = warp == 1 ? 0u : warp - kEsFirstExtraIssuer + 1u;
    const uint32_t idesc = ptx::make_idesc_bf16_f32(kEsBM, (uint32_t)p.n_tile);
    uint64_t dbh[kBSets][2], dbl[kBSets][2], dah[kASets][2], dal[kASets][2];
    uint32_t ath[kASets][2], atl[kASets][2];
#pragma unroll
    for (int kk = 0; kk < kEsBK / 16; ++kk) {
      const uint32_t ko = kk * 32;                               // 16 bf16 = 32 bytes inside the 64-byte swizzle atom
#pragma unroll
      for (int u = 0; u < kBSets; ++u) {
        const uint32_t b_hi = sbase + L.b_off + (me + 3u * u) * 2 * p.b_plane;
        dbh[u][kk] = ptx::make_kmajor_desc(b_hi + ko, 64);
        dbl[u][kk] = ptx::make_kmajor_desc(b_hi + p.b_plane + ko, 64);
      }
#pragma unroll
      for (int u = 0; u < kASets; ++u) {
        const int as = (int)me + 3 * u;
        if constexpr (kTmemA) {
          ath[u][kk] = tmem_base + es_a_col(as, p.n_tile) + kk * 8;       // hi: columns +0..15, lo: +16..31
          atl[u][kk] = ath[u][kk] + 16;
          dah[u][kk] = dal[u][kk] = 0;
        } else {
          const uint32_t a_hi = sbase + L.a_off + as * 2 * kEsAPlane;
          dah[u][kk] = ptx::make_kmajor_desc(a_hi + ko, 64);
          dal[u][kk] = ptx::make_kmajor_desc(a_hi + kEsAPlane + ko, 64);
          ath[u][kk] = atl[u][kk] = 0;
        }
      }
    }
    const uint32_t my_tiles = blockIdx.x < (uint32_t)p.n_row_tiles ? ((uint32_t)p.n_row_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0u;
    const uint32_t g_total = my_tiles * (uint32_t)p.n_ntiles * (uint32_t)nkb;
    const bool iprof = prof && me == 0;
    long long w_te = 0, w_af = 0, w_bf = 0, w_tok = 0; const long long t0 = iprof ? clock64() : 0;
    uint32_t kb = me % (uint32_t)nkb, tile_no = me / (uint32_t)nkb;      // of k-block g, advanced by 3 per step
    for (uint32_t g0 = me; g0 < g_total; g0 += kEsIssuers * kSets) {
#pragma unroll
      for (int u = 0; u < kSets; ++u) {
        const uint32_t g = g0 + kEsIssuers * u;
        if (g >= g_total) break;
        const int ua = u % kASets, ub = u % kBSets;                  // compile-time after unrolling
        const uint32_t as = me + 3u * (uint32_t)ua, bs = me + 3u * (uint32_t)ub;
        const uint32_t aph = (g / (uint32_t)(kEsIssuers * kASets)) & 1u, bph = (g / kNB) & 1u;
        const uint32_t buf = tile_no & 1u;
        const uint32_t d_tmem = tmem_base + buf * 256;
        if (kb == 0) {
          if (iprof) twait(bar(EsTail::t_empty, buf), ((tile_no >> 1) & 1u) ^ 1u, 720 + buf, w_te);
          else ptx::mbar_wait(bar(EsTail::t_empty, buf), ((tile_no >> 1) & 1u) ^ 1u, 720 + buf);
        }
        if (iprof) { twait(bar(EsTail::a_full, as), aph, 730 + as, w_af); twait(bar(EsTail::b_full, bs), bph, 740 + bs, w_bf); }
        else { ptx::mbar_wait(bar(EsTail::a_full, as), aph, 730 + as); ptx::mbar_wait(bar(EsTail::b_full, bs), bph, 740 + bs); }
        ptx::tc_fence_after_sync();
        if (g > 0) {                                                   // token: the previous issuer has issued k-block g - 1
          const long long c0 = iprof ? clock64() : 0;
          ptx::named_bar_sync(1 + me, 64);
          if (iprof) w_tok += clock64() - c0;
        }
        const bool elected = ptx::elect_one();
        if (elected) {
#pragma unroll
          for (int kk = 0; kk < kEsBK / 16; ++kk) {
            if constexpr (kTmemA) {
              ptx::umma_bf16_ts<1>(d_tmem, ath[ua][kk], dbh[ub][kk], idesc, (kb | (uint32_t)kk) != 0 ? 1u : 0u);
              ptx::umma_bf16_ts<1>(d_tmem, ath[ua][kk], dbl[ub][kk], idesc, 1u);
              ptx::umma_bf16_ts<1>(d_tmem, atl[ua][kk], dbh[ub][kk], idesc, 1u);
            } else {
              ptx::umma_bf16<1>(d_tmem, dah[ua][kk], dbh[ub][kk], idesc, (kb | (uint32_t)kk) != 0 ? 1u : 0u);
              ptx::umma_bf16<1>(d_tmem, dah[ua][kk], dbl[ub][kk], idesc, 1u);
              ptx::umma_bf16<1>(d_tmem, dal[ua][kk], dbh[ub][kk], idesc, 1u);
            }
          }
        }
        __syncwarp();
        if (g + 1 < g_total) ptx::named_bar_arrive(1 + (me + 1) % kEsIssuers, 64);      // hand the token over ...
        if (elected) {                                                                  // ... then commit
          ptx::umma_commit<1>(bar(EsTail::a_empty, as), 0);
          ptx::umma_commit<1>(bar(EsTail::b_empty, bs), 0);
          if (kb == (uint32_t)nkb - 1) ptx::umma_commit<1>(bar(EsTail::t_full, buf), 0);
        }
        __syncwarp();
        kb += kEsIssuers;
        while (kb >= (uint32_t)nkb) { kb -= (uint32_t)nkb; ++tile_no; }
      }
    }
    // No tcgen05.commit of this CTA may still be in flight when it exits (its mbarrier arrive would land in shared
    // memory that no longer belongs to it): commits of one thread complete in order, so one more per issuer on a
    // drain barrier, awaited by all issuers, covers the a_empty / b_empty commits nobody waits for at the end.
    if (ptx::elect_one()) ptx::umma_commit<1>(bar(EsTail::drain, 0), 0);
    __syncwarp();
    ptx::mbar_wait(bar(EsTail::drain, 0), 0, 790);
    if (iprof && lane == 0) { pf[3] = clock64() - t0; pf[4] = w_te; pf[5] = w_af; pf[6] = w_bf; pf[11] = tile_no; pf[12] = w_tok; }
  } else if (warp >= 4 && warp < 4 + 4 * kEsConvSets) {
    // =================================================== converters: fp32 tile -> bf16 hi / lo operand tiles
    // Set `cset` handles the k-blocks whose running index g (over the whole kernel) is congruent to cset.
    const int cset = (int)(warp - 4) >> 2;
    const int row = (int)((warp - 4) & 3) * 32 + (int)lane;
    const uint32_t x_row = (uint32_t)row * 128u, x_sw = (uint32_t)(row & 7);
    const uint32_t a_row = (uint32_t)row * 64u, a_sw = (uint32_t)((row >> 1) & 3);
    const uint32_t a_lane = (((warp & 3u) * 32u) << 16);       // this warp's TMEM lane quadrant (row = quadrant * 32 + lane)
    float* xnorm_s = reinterpret_cast<float*>(smem + L.tail_off + EsTail::xnorm);
    uint32_t g = 0;                       // running k-block index: ring slots and parities derive from it
    uint32_t my_tile = 0;                 // row tiles this CTA has converted: ||x||^2 slot = my_tile & 3
    long long w_xf = 0, w_ae = 0; const long long t0c = prof ? clock64() : 0;
    int pend_as = -1;                     // kTmemA: A stage whose tcgen05.st are in flight and not yet published
    auto publish_pending = [&]() {
      ptx::tmem_st_wait();
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar(EsTail::a_full, (uint32_t)pend_as));
      pend_as = -1;
    };
    // ring slots / parities of this set's k-blocks advance incrementally (g steps by kEsConvSets): the runtime
    // divisions by x_stages / a_stages cost ~40 dependent instructions per k-block (ncu source view)
    uint32_t xs = (uint32_t)cset % (uint32_t)kEsXStages, xph = ((uint32_t)cset / (uint32_t)kEsXStages) & 1u;
    uint32_t as = (uint32_t)cset % (uint32_t)n_as, aph = ((uint32_t)cset / (uint32_t)n_as) & 1u;
    for (int rt = blockIdx.x; rt < p.n_row_tiles; rt += gridDim.x, ++my_tile) {
      for (int nt = 0; nt < p.n_ntiles; ++nt, g += (uint32_t)nkb) {
        float2 norm2 = make_float2(0.f, 0.f);
        // g = running index of this tile's k-block 0; this set owns the k-blocks with (g + kb) % kEsConvSets == cset
        for (int kb = (int)(((uint32_t)cset + kEsConvSets - g % kEsConvSets) % kEsConvSets); kb < nkb; kb += kEsConvSets) {
          // the previous k-block's TMEM stores are published only once this k-block's X tile is in registers (their
          // latency hides behind the wait and the loads) - unless that tile is not there yet
          if (pend_as >= 0 && !__all_sync(0xffffffffu, ptx::mbar_test_wait(bar(EsTail::x_full, xs), xph))) publish_pending();
          twait(bar(EsTail::x_full, xs), xph, 750 + xs, w_xf);
          const uint8_t* xt = smem + L.x_off + xs * kEsXBytes + x_row;
          float4 f[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = *reinterpret_cast<const float4*>(xt + ((((uint32_t)j) ^ x_sw) << 4));
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(bar(EsTail::x_empty, xs));      // the fp32 stage is in registers
          if (pend_as >= 0) publish_pending();
          uint4 hi[4], lo[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float2 v[4] = {make_float2(f[2 * c].x, f[2 * c].y), make_float2(f[2 * c].z, f[2 * c].w),
                                 make_float2(f[2 * c + 1].x, f[2 * c + 1].y), make_float2(f[2 * c + 1].z, f[2 * c + 1].w)};
            uint32_t h[4], l[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const __nv_bfloat162 hh = __floats2bfloat162_rn(v[q].x, v[q].y);
              h[q] = *reinterpret_cast<const uint32_t*>(&hh);
              // residual x - x_hi (exact in fp32) and ||x||^2, two lanes per instruction (fma.rn.f32x2)
              const float2 hf = make_float2(__uint_as_float(h[q] << 16), __uint_as_float(h[q] & 0xffff0000u));
              const float2 r = __ffma2_rn(hf, make_float2(-1.f, -1.f), v[q]);
              const __nv_bfloat162 ll = __floats2bfloat162_rn(r.x, r.y);
              l[q] = *reinterpret_cast<const uint32_t*>(&ll);
              norm2 = __ffma2_rn(v[q], v[q], norm2);
            }
            hi[c] = make_uint4(h[0], h[1], h[2], h[3]);
            lo[c] = make_uint4(l[0], l[1], l[2], l[3]);
          }
          twait(bar(EsTail::a_empty, as), aph ^ 1, 760 + as, w_ae);
          // this set's last k-block of the tile: publish its share of ||x||^2 before the a_full arrive
          if (nt == 0 && kb + kEsConvSets >= nkb) xnorm_s[((my_tile & 3u) * kEsConvSets + cset) * kEsBM + row] = norm2.x + norm2.y;
          if constexpr (kTmemA) {
            ptx::tc_fence_after_sync();                                   // the MMAs that read this stage have completed
            const uint32_t a_t = tmem_base + a_lane + es_a_col((int)as, p.n_tile);
            ptx::tmem_st_32x16(a_t, reinterpret_cast<const uint32_t*>(hi));
            ptx::tmem_st_32x16(a_t + 16, reinterpret_cast<const uint32_t*>(lo));
            pend_as = (int)as;                                            // wait::st + a_full arrive: publish_pending()
          } else {
            uint8_t* at = smem + L.a_off + as * 2 * kEsAPlane + a_row;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint32_t off = (((uint32_t)c) ^ a_sw) << 4;
              *reinterpret_cast<uint4*>(at + off) = hi[c];
              *reinterpret_cast<uint4*>(at + kEsAPlane + off) = lo[c];
            }
            fence_proxy_async_smem();                                     // generic-proxy writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(bar(EsTail::a_full, as));
          }
          xs += kEsConvSets; while (xs >= (uint32_t)kEsXStages) { xs -= (uint32_t)kEsXStages; xph ^= 1u; }
          as += kEsConvSets; while (as >= (uint32_t)n_as) { as -= (uint32_t)n_as; aph ^= 1u; }
        }
      }
    }
    if (pend_as >= 0) publish_pending();
    if (prof && warp == 4 && lane == 0) { pf[7] = clock64() - t0c; pf[8] = w_xf; pf[9] = w_ae; }
  } else if (warp >= 4 + 4 * kEsConvSets && warp < 4 + 4 * kEsConvSets + 4) {
    // =================================================== epilogue: running argmin per row
    const uint32_t quad = warp & 3u;
    const int row_in_tile = (int)quad * 32 + (int)lane;
    const uint32_t lane_addr = (quad * 32u) << 16;
    const float* cn = reinterpret_cast<const float*>(smem + L.tail_off + EsTail::cnorm);
    const float* xnorm_s = reinterpret_cast<const float*>(smem + L.tail_off + EsTail::xnorm);
    uint32_t tile_no = 0, my_tile = 0;
    double inertia_local = 0.0;
    long long w_tf = 0;
    // the converters run at most 2 accumulator tiles + a_stages <= 2 * num_kb operand stages (two tiles) ahead of
    // this warp, so the 4-deep ||x||^2 ring (slot = row tiles done & 3) is never overwritten before it is read
    for (int rt = blockIdx.x; rt < p.n_row_tiles; rt += gridDim.x, ++my_tile) {
      float best = INFINITY; int best_k = -1;
      float xn = 0.f;
      for (int nt = 0; nt < p.n_ntiles; ++nt, ++tile_no) {
        const uint32_t buf = tile_no & 1u;
        twait(bar(EsTail::t_full, buf), (tile_no >> 1) & 1u, 770 + buf, w_tf);
        ptx::tc_fence_after_sync();
        if (nt == 0) {
#pragma unroll
          for (int cs = 0; cs < kEsConvSets; ++cs) xn += xnorm_s[((my_tile & 3u) * kEsConvSets + cs) * kEsBM + row_in_tile];
        }
        const uint32_t taddr = tmem_base + lane_addr + buf * 256;
        const int k0 = nt * 256;
        const int n_here = min(p.n_clusters - k0, 256);
#pragma unroll 1
        for (int c = 0; c * 32 < n_here; ++c) {
          uint32_t r[32];
          // Never read accumulator columns the MMA did not write (n_tile is a multiple of 16, so a ragged last chunk
          // is exactly 16 columns): reading never-written tensor memory made about one launch in 10^4 die with an
          // "unspecified launch failure" - only for tile widths with n_tile % 32 == 16 whose upper columns nothing
          // ever writes (K = 161 / 200; randomised stress tools/estep_stress2.py, profiles/r1q_estep_stress.txt).
          if (c * 32 + 32 <= p.n_tile) {
            ptx::tmem_ld_32x32(taddr + c * 32, r);
          } else {
#pragma unroll
            for (int j = 16; j < 32; ++j) r[j] = 0u;
            ptx::tmem_ld_32x16(taddr + c * 32, r);
          }
          ptx::tmem_ld_wait(r);
          const int kbase = k0 + c * 32;
          const int n_valid = min(n_here - c * 32, 32);    // <= 16 in the ragged chunk: columns past it are masked below
          float d[32];
          const float4* cn4 = reinterpret_cast<const float4*>(cn + kbase);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 c4 = cn4[j4];
            d[4 * j4 + 0] = fmaf(-2.f, __uint_as_float(r[4 * j4 + 0]), c4.x);
            d[4 * j4 + 1] = fmaf(-2.f, __uint_as_float(r[4 * j4 + 1]), c4.y);
            d[4 * j4 + 2] = fmaf(-2.f, __uint_as_float(r[4 * j4 + 2]), c4.z);
            d[4 * j4 + 3] = fmaf(-2.f, __uint_as_float(r[4 * j4 + 3]), c4.w);
          }
          if (n_valid < 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) d[j] = j < n_valid ? d[j] : INFINITY;
          }
          // chunk minimum with NaN propagation (min.NaN): the 32-element scan below runs only for the chunks that
          // improve the row's best (about two per tile) - the per-element running argmin cost 28 instructions per
          // element and made this warp role the slowest of the kernel (ncu source view, 3600 instructions per tile)
          float m8[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) m8[q] = fmin_nan(fmin_nan(d[4 * q], d[4 * q + 1]), fmin_nan(d[4 * q + 2], d[4 * q + 3]));
          const float m = fmin_nan(fmin_nan(fmin_nan(m8[0], m8[1]), fmin_nan(m8[2], m8[3])), fmin_nan(fmin_nan(m8[4], m8[5]), fmin_nan(m8[6], m8[7])));
          if (m == m) {                               // no NaN in the chunk: new best iff strictly smaller (ties keep the lower k)
            if (best_k < 0 || m < best) {
              int idx = 31;
#pragma unroll
              for (int j = 30; j >= 0; --j) idx = d[j] == m ? j : idx;      // first column holding the minimum
              best = m; best_k = kbase + idx;
            }
          } else if (best_k < 0 || best == best) {    // a NaN distance beats any number (torch.min): exact ascending scan
#pragma unroll 1
            for (int j = 0; j < n_valid; ++j) {
              float dj = d[0];
#pragma unroll
              for (int t = 1; t < 32; ++t) dj = t == j ? d[t] : dj;
              if (best_k < 0 || es_better(dj, best)) { best = dj; best_k = kbase + j; }
            }
          }
        }
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar(EsTail::t_empty, buf));
      }
      const long long row = (long long)rt * kEsBM + row_in_tile;
      if (row < p.n_rows) {
        float d = xn + best;
        d = d < 0.f ? 0.f : d;                    // the direct form is never negative; keeps NaN
        p.labels[row] = best_k;
        if (p.mindist) p.mindist[row] = d;
        inertia_local += (double)d;
      }
    }
    if (prof && warp == 4 + 4 * kEsConvSets && lane == 0) pf[10] = w_tf;
    if (p.inertia) {
      for (int off = 16; off > 0; off >>= 1) inertia_local += __shfl_down_sync(0xffffffffu, inertia_local, off);
      if (lane == 0) atomicAdd(p.inertia, inertia_local);
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc<1>(tmem_base, 512);
}

}  // namespace scd

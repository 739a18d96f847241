// Image x vocabulary scoring with a fused per-row top-k epilogue (SURVEY 8a rows a8 / a11).
//
//   scores[n, v] = sum_d X[n, d] * Wt[v, d]          X: [N, 768] bf16 row-major (K-major A)
//                                                    Wt: [V, 768] bf16 row-major (K-major B), the
//                                                    one-off transpose of the reference's [D, V]
//   replaces  main_unsup.py:519-529 / main_ptsup.py:538-543 (GEMM -> [1024, V] logits in HBM ->
//   softmax -> topk twice) and main_unsup.py:610-614 (k = 1 over the K selected columns).
//
// The N x V score matrix never exists: a CTA pair (cta_group::2, 256 x 224 x 16 tcgen05.mma) keeps its 256 image
// rows stationary for a whole vocabulary sweep, streams the vocabulary through a TMA ring, accumulates each
// 256 x 224 tile in TMEM (double buffered) and eight epilogue warps read the tile back with tcgen05.ld - one
// thread per image row.
//
// Operand placement is what the measurements forced (profiles/r1_name_cycle_counters.txt, r1_tma_feed.txt): a
// vocabulary box needs ~600 cycles from L2 plus ~400 cycles of barrier round trips, so the ring must hold >= 3
// k-blocks ahead of the tensor pipe; with all 192 KB of stationary rows in shared memory only 32 KB (2 k-blocks) were
// left and the issuer spent 40 % of its time waiting for B (65 % tensor-active).  Now the first TWO 64-wide
// k-blocks of the rows live in TENSOR MEMORY as the A operand (tcgen05.mma with A from TMEM; loader warps write them
// with tcgen05.st, thread = row = TMEM lane), the other ten stay in shared memory (SWIZZLE_128B), and the 32 KB
// that frees plus the old ring hold a 9-deep ring of 112-row x 32-k vocabulary boxes (7 KB per CTA, SWIZZLE_64B):
// the two MMAs kk = 0, 1 of a k-block read one stage, kk = 2, 3 the next, so a stage is free again after two MMAs.
// Wider tiles (224 instead of 192) amortise the fixed per-MMA issue cost over more columns - the tile sweep
// (96 -> 192 -> 240 -> 224) measured 224 x 2 TMEM k-blocks fastest (2.76 ms on C2).
// TMEM: accumulators at columns [0,224) and [256,480), A k-blocks at [224,256) and [480,512).
//
// The epilogue is a two-level selection: per 32-column chunk only the chunk maximum is computed (31 FMNMX) and
// compared with the row's k-th best chunk maximum; the rare chunk that beats it is parked (32 floats) in an
// L2-resident scratch slot.  The true top-k of a row lies inside its k chunks with the largest maxima, so one
// exact scan of those k parked chunks at the end of the vocabulary sweep finishes the row.  (The unsupervised
// driver's softmax additionally keeps a running max / sum-exp.)  Only [N, k] leaves the SM.
//
// Warp roles (640 threads = 5 warpgroups; setmaxnreg moves registers from the control warps to the epilogue):
//   WG0 (warps 0..3)   0, 2 = vocabulary (B) TMA producers (2 also allocates TMEM); 1, 3 = MMA issuers
//   WG1, WG2 (4..11)   epilogue (TMEM lane quadrant = warp & 3; warps 4..7 take columns 0..127 of every accumulator
//                      tile, warps 8..11 columns 128..223)
//   WG3 (12..15)       loaders of the TMEM-resident A k-blocks (global -> registers -> tcgen05.st); 12 is also the
//                      TMA producer of the shared-memory A k-blocks
//   WG4 (16..19)       16 = third MMA issuer (leader CTA only, k-blocks round-robin, a token keeps the issue order),
//                      17 = third B producer, 18 and 19 idle
#pragma once
#include "ptx.cuh"
#include <cuda_bf16.h>

namespace scd {

constexpr int kNameMaxD = 768;         // widest embedding the stationary A operand holds (any D <= 768, D % 8 == 0)
constexpr int kBlockM = 128;           // rows per CTA (256 per pair)
constexpr int kTileN = 224;            // vocabulary entries per accumulator tile (112 loaded per CTA)
constexpr int kAKBlock = 64;           // k per A / B block  (128 B rows, SWIZZLE_128B)
constexpr int kNumAKBlocks = kNameMaxD / kAKBlock;   // 12 (capacity; the live count is NameParams::num_kb)
constexpr int kTmemAKBlocks = 2;       // A k-blocks 0, 1 live in tensor memory (32 columns above each accumulator)
constexpr int kSmemAKBlocks = kNumAKBlocks - kTmemAKBlocks;   // 8 in shared memory
constexpr int kBStageK = 32;           // k per vocabulary stage: half a k-block (64 B rows, SWIZZLE_64B)
constexpr int kBStages = 9;            // one stage = one 32-k half of a k-block (7 KB) of one vocabulary tile
constexpr int kBProducers = 3;         // warps 0, 2 and 17 issue stages round-robin (one warp keeps only one box in
                                       // flight, ~500-600 cycles each: tools/tma_feed_bench.cu); kBStages must be a
                                       // multiple of it, so that every stage always has the same producer (DESIGN 3.2)
constexpr int kABlockBytes = kBlockM * kAKBlock * 2;     // 16384
constexpr int kBStageBytes = (kTileN / 2) * kBStageK * 2;   // 7168 per CTA
constexpr int kNumIssuers = 3;          // MMA issuer warps 1, 3 and 16, round-robin over k-blocks
constexpr int kNameThreads = 640;
// per-thread registers after setmaxnreg (launched at 65536 / 640 -> 96): the other warpgroups give up what the
// epilogue's four 32-column loads in flight need, 2 x (96 - 48) + (96 - 48) = 2 x (168 - 96).  The smallest counts
// at which ptxas compiles every role of name_topk_kernel<1>, <5> and <8> without spilling.
constexpr int kCtrlRegs = 48;           // WG0, WG4: producers and issuers
constexpr int kLoaderRegs = 48;         // WG3: one 32-register row buffer per thread
constexpr int kEpiRegs = 168;           // WG1, WG2
static_assert((2 * kCtrlRegs + kLoaderRegs + 2 * kEpiRegs) * 128 <= kNameThreads * 96, "setmaxnreg budget exceeds the launch allocation");
static_assert(kBStages % kBProducers == 0 && kAKBlock == 2 * kBStageK, "vocabulary ring plan");
constexpr int kEpiHalves = 2;           // column halves of a tile, one epilogue warp set each
constexpr int kHalfCols = 128;          // epilogue warps 4..7 take columns [0,128), warps 8..11 columns [128,224)
constexpr int kTmemCols = 512;
constexpr int kAccStride = 256;         // accumulator buffer b starts at column b * 256

// TMEM column of the kk-th 16-wide k-step of TMEM-resident A k-block kb: the 32 columns above accumulator buffer kb
__host__ __device__ constexpr int a_tmem_col(int kb, int kk) { return kTileN + kb * kAccStride + kk * 8; }
static_assert(kTileN + 32 <= kAccStride && kTmemAKBlocks == 2, "TMEM column plan");

struct NameSmem {
  // offsets inside dynamic shared memory (base aligned to 1024)
  static constexpr int a_off = 0;
  static constexpr int b_off = kSmemAKBlocks * kABlockBytes;                // 163840
  static constexpr int bar_off = b_off + kBStages * kBStageBytes;           // 228352
  // barriers (8 B each)
  static constexpr int full_bar = bar_off;                                  // [kBStages]
  static constexpr int empty_bar = full_bar + 8 * kBStages;                 // [kBStages]
  static constexpr int a_full_bar = empty_bar + 8 * kBStages;               // [12]
  static constexpr int a_empty_bar = a_full_bar + 8 * kNumAKBlocks;         // [12]
  static constexpr int tmem_full_bar = a_empty_bar + 8 * kNumAKBlocks;      // [2]
  static constexpr int tmem_empty_bar = tmem_full_bar + 16;                 // [2]
  static constexpr int tmem_ptr = tmem_empty_bar + 16;
  static constexpr int issue_seq = tmem_ptr + 16;                           // k-blocks issued so far (the issuers' token)
  static constexpr int total = issue_seq + 16;
};
static_assert(NameSmem::total + 1024 <= 232448, "exceeds 227 KB of shared memory");

struct NameParams {
  long long n_rows;        // N
  long long v_total;       // V (this rank's vocabulary slice length)
  // work partition: the (row block, vocabulary tile) space, row-block major, is cut into one contiguous range of
  // tiles per CTA pair (NameWork); a range covers the end of one row block, whole row blocks, and the start of another.
  // Each piece of a row block is a work item; its result goes to partial-list slot `piece ordinal within the row block`.
  long long work_total;    // n_row_blocks * tiles_total
  int tiles_total;         // ceil(V / kTileN)
  int n_row_blocks;        // ceil(N / 256)
  int num_kb;              // ceil(D / 64) live A k-blocks (TMA zero-fills the ragged end of D)
  int want_softmax;
  float scale_log2e;       // scale * log2(e) for the running sum-exp
  // partial results, one slot per (piece of the row block, column half): [n_slots * 2][N][KT] / [n_slots * 2][N]
  // (the merge derives the number of pieces of a row block from the same NameWork arithmetic)
  float* part_val;
  int* part_idx;
  float* part_max;
  float* part_sum;
  float* scratch;          // [gridDim.x][2 halves][4 warps][KT slots][8][32 lanes] float4: parked chunks, lane-interleaved
  long long* prof;         // nullable: [pairs][16] cycle counters (scd_debug_set_name_profile), debugging aid
  const __nv_bfloat16* x;  // [N, d] row-major: the loader warps read the TMEM-resident k-blocks straight from global memory
  int d;
};

// Linear partition of the work: tile index l = row_block * T + tile; pair q of P owns [bound(q), bound(q + 1)).
// Loads differ by at most one tile between pairs, and a pair starts at most (range / T + 2) work items - at N = 8 ranks
// (63 row blocks on 74 pairs) that is two items of ~40 tiles instead of six of 14, each of which paid the item
// start-up and the final exact scan (DESIGN 3.1).
struct NameWork {
  long long W;   // work_total
  int T;         // tiles per row block
  int P;         // pairs
  __host__ __device__ long long bound(int q) const { return (W * q) / P; }
  __host__ __device__ int owner(long long l) const {       // the pair whose range holds tile l (0 <= l < W)
    int q = (int)(((l + 1) * P + W - 1) / W) - 1;          // largest q with bound(q) <= l
    while (q + 1 < P && bound(q + 1) <= l) ++q;
    while (q > 0 && bound(q) > l) --q;
    return q;
  }
  // pieces a row block is cut into (1 when one pair sweeps it whole)
  __host__ __device__ int pieces(int rb) const { return owner((long long)(rb + 1) * T - 1) - owner((long long)rb * T) + 1; }
};

struct NameItem { int rb, t0, nt, part; };

// the work item of pair q that starts at tile l of its range [.., hi)   (work_total < 2^31, checked by the host)
__host__ __device__ inline NameItem name_item_at(const NameWork& w, int q, int l, int hi) {
  NameItem it;
  it.rb = l / w.T;
  it.t0 = l - it.rb * w.T;
  it.nt = hi - l < w.T - it.t0 ? hi - l : w.T - it.t0;
  it.part = it.t0 == 0 ? 0 : q - w.owner((long long)it.rb * w.T);
  return it;
}

// One sorted top-KT list in registers, ordered by (value descending, column ascending) - the order
// torch.topk(..., largest=True, sorted=True) yields when ties resolve to the lower index.  Columns may
// be pushed in any order.
template <int KT>
struct TopK {
  float v[KT];
  int i[KT];
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int j = 0; j < KT; ++j) { v[j] = -INFINITY; i[j] = -1; }
  }
  static __device__ __forceinline__ bool before(float xa, int ia, float xb, int ib) {
    return xa > xb || (xa == xb && (ib < 0 || ia < ib));
  }
  __device__ __forceinline__ void push(float x, int col) {
    if (x > -INFINITY && before(x, col, v[KT - 1], i[KT - 1])) {
      v[KT - 1] = x; i[KT - 1] = col;
#pragma unroll
      for (int j = KT - 1; j > 0; --j) {
        if (before(v[j], i[j], v[j - 1], i[j - 1])) {
          float tv = v[j]; v[j] = v[j - 1]; v[j - 1] = tv;
          int ti = i[j]; i[j] = i[j - 1]; i[j - 1] = ti;
        }
      }
    }
  }
};

// The KT chunks (32 consecutive columns) with the largest chunk maxima seen so far, sorted by (maximum
// descending, first column ascending) - an order that does not depend on the sequence in which chunks are
// visited.  slot[] says which scratch slot holds the chunk's 32 values, col[] its first column.
template <int KT>
struct ChunkTop {
  float m[KT];
  int slot[KT];
  int col[KT];
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int j = 0; j < KT; ++j) { m[j] = -INFINITY; slot[j] = j; col[j] = -1; }
  }
  __device__ __forceinline__ bool admits(float cmax, int colbase) const {
    return cmax > m[KT - 1] || (cmax == m[KT - 1] && colbase < col[KT - 1]);
  }
  // the caller has already parked the chunk in slot[KT-1]
  __device__ __forceinline__ void insert_last(float cmax, int colbase) {
    m[KT - 1] = cmax; col[KT - 1] = colbase;
#pragma unroll
    for (int j = KT - 1; j > 0; --j) {
      if (m[j] > m[j - 1] || (m[j] == m[j - 1] && col[j] < col[j - 1])) {
        float tm = m[j]; m[j] = m[j - 1]; m[j - 1] = tm;
        int ts = slot[j]; slot[j] = slot[j - 1]; slot[j - 1] = ts;
        int tc = col[j]; col[j] = col[j - 1]; col[j - 1] = tc;
      }
    }
  }
};

template <int KT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kNameThreads, 1)
name_topk_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                 const NameParams p) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need a 1024-aligned base; both CTAs of the pair compute the same offset
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sbase = ptx::smem_u32(smem);
  // the shuffle makes the warp index provably warp-uniform for ptxas: role loops then run on the uniform datapath
  // (descriptor arithmetic in UIADD3 instead of vector math + R2UR in front of every tcgen05.mma)
  const uint32_t warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t cta_rank = ptx::cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int pair = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;
  const NameWork work{p.work_total, p.tiles_total, n_pairs};
  const int l_lo = (int)work.bound(pair), l_hi = (int)work.bound(pair + 1);      // this pair's range of tiles

  const int nkb = p.num_kb;
  const int nkb_tmem = min(nkb, kTmemAKBlocks);
  auto full_bar = [&](int s) { return sbase + NameSmem::full_bar + 8 * s; };
  auto empty_bar = [&](int s) { return sbase + NameSmem::empty_bar + 8 * s; };
  auto a_full_bar = [&](int kb) { return sbase + NameSmem::a_full_bar + 8 * kb; };
  auto a_empty_bar = [&](int kb) { return sbase + NameSmem::a_empty_bar + 8 * kb; };
  auto tmem_full_bar = [&](int b) { return sbase + NameSmem::tmem_full_bar + 8 * b; };
  auto tmem_empty_bar = [&](int b) { return sbase + NameSmem::tmem_empty_bar + 8 * b; };

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kBStages; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
    for (int kb = 0; kb < kNumAKBlocks; ++kb) {
      // TMEM-resident k-blocks: the four loader warps of both CTAs arrive; shared-memory k-blocks: one expect_tx
      ptx::mbar_init(a_full_bar(kb), kb < kTmemAKBlocks ? 8 : 1);
      ptx::mbar_init(a_empty_bar(kb), 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tmem_full_bar(b), 1);
      ptx::mbar_init(tmem_empty_bar(b), 16);     // 8 epilogue warps x 2 CTAs arrive on the leader's copy
    }
    *reinterpret_cast<volatile uint32_t*>(smem + NameSmem::issue_seq) = 0u;
    ptx::fence_mbar_init_cluster();
  }
  if (warp == 2) {
    ptx::tmem_alloc<2>(sbase + NameSmem::tmem_ptr, kTmemCols);
    ptx::tmem_relinquish<2>();
  }
  ptx::tc_fence_before_sync();
  ptx::cluster_sync_all();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + NameSmem::tmem_ptr);

  // Staggered sweep: pair q starts its walk over an item's tiles at a different offset and wraps around, so
  // at any moment the 74 pairs read 74 different vocabulary tiles (spread over all L2 slices) instead of
  // all hammering the same lines.  The result does not depend on the visiting order (explicit tie rules).
  auto item_tile = [&](const NameItem& it, int t) {
    const int start = (int)(((long long)pair * it.nt) / n_pairs);
    int tt = t + start;
    if (tt >= it.nt) tt -= it.nt;
    return it.t0 + tt;
  };

  // Registers by role (setmaxnreg acts on whole warpgroups): the epilogue keeps a tile's four 32-column loads in
  // flight (128 registers of scores); producers and issuers live on uniform registers, a loader on one 32-register
  // row buffer.  Each role's code is dominated by its own setmaxnreg, so ptxas allocates it within that budget.
  // Every branch ends in its own copy of the teardown: no code is shared after the roles split, which is what lets
  // ptxas compile each role at its own register count.
  // Teardown: nobody may free TMEM / exit while the peer can still touch this CTA's memory.
  auto teardown = [&]() {
    ptx::tc_fence_before_sync();
    ptx::cluster_sync_all();
    if (warp == 2) ptx::tmem_dealloc<2>(tmem_base, kTmemCols);
  };
  const uint32_t wg = warp >> 2;
  if (wg == 0 || wg == 4) {
    ptx::setmaxnreg_dec<kCtrlRegs>();
    if (warp == 0 || warp == 2 || warp == 17) {
      // ======================================================= vocabulary (B) TMA producers
      // Stage g (a running count of 32-k halves of k-blocks over the whole kernel) belongs to producer g % 3.  Whole
      // warp runs the loop (warp-uniform control flow keeps addresses in uniform registers); one elected lane issues.
      // A half that lies wholly beyond D (ragged last k-block) is still loaded: TMA fills it with zeros.
      const uint32_t me = warp == 0 ? 0u : (warp == 2 ? 1u : 2u);
      uint32_t g = 0;
      const bool prof = p.prof != nullptr;
      long long pf_t0 = prof ? clock64() : 0, pf_e = 0;
      for (int l = l_lo; l < l_hi;) {
        const NameItem it = name_item_at(work, pair, l, l_hi);
        l += it.nt;
        const int nt = it.nt;
        for (int t = 0; t < nt; ++t) {
          const int v0 = item_tile(it, t) * kTileN + (int)cta_rank * (kTileN / 2);
          for (int kb = 0; kb < nkb; ++kb) {
            for (int hh = 0; hh < 2; ++hh, ++g) {
              if ((g % kBProducers) != me) continue;
              const int stage = (int)(g % kBStages);
              const uint32_t phase = (g / kBStages) & 1u;
              { const long long c0 = prof ? clock64() : 0;
                ptx::mbar_wait_nocall(empty_bar(stage), phase ^ 1, 200 + stage);
                if (prof) pf_e += clock64() - c0; }
              if (ptx::elect_one()) {
                if (leader) ptx::mbar_arrive_expect_tx(full_bar(stage), 2 * kBStageBytes);
                ptx::tma_load_2d<2>(sbase + NameSmem::b_off + stage * kBStageBytes, &map_w,
                                    full_bar(stage) & ptx::kPeerBitMask, kb * kAKBlock + hh * kBStageK, v0, ptx::kEvictLast);
              }
              __syncwarp();
            }
          }
        }
      }
      if (prof && lane == 0) {
        long long* o = p.prof + (size_t)pair * 32;
        const int base = (leader ? 0 : 16) + (me == 0 ? 6 : (me == 1 ? 12 : 14));   // leader: 6,7 / 12,13 / 14,15; peer: +16
        o[base] = clock64() - pf_t0; o[base + 1] = pf_e;
      }
    } else if (warp == 1 || warp == 3 || warp == 16) {
      // ======================================================= MMA issuers (leader CTA; one elected lane of each issues)
      // What the measurements say about issuing (tools/mma_rate_bench.cu, profiles/r1_mma_rate_*.txt): the tensor pipe
      // runs an MMA in exactly N/2 cycles when the next one is already queued, the queue is only a couple of MMAs deep,
      // and a tcgen05.mma keeps the uniform registers of its descriptors busy until it has run - so an issuer that
      // prepares the next k-block's descriptors after its own MMAs does so behind an idle pipe (+43 cycles per MMA).
      // Two warps therefore take alternate k-blocks (running count g): each has its own uniform registers, computes
      // its descriptors and does its barrier waits while the other warp's four MMAs run, then waits for a named-barrier
      // token (ids 1 / 2) and fires its four MMAs back to back.  The token keeps the issue order, which is also the
      // execution order of the pipe, so the last k-block's commit covers the whole tile.
      if (leader) {
        const uint32_t me = warp == 1 ? 0u : (warp == 3 ? 1u : 2u);
        const uint32_t idesc = ptx::make_idesc_bf16_f32(2 * kBlockM, kTileN);
        uint32_t g = 0, tile_no = 0;
        int my_item_no = 0;
        const long long g_total = (long long)(l_hi - l_lo) * nkb;
        const bool prof = p.prof != nullptr && me == 0;
        long long pf_t0 = prof ? clock64() : 0, pf_te = 0, pf_a = 0, pf_b = 0, pf_tok = 0;
        const uint64_t pf_ns0 = prof ? ptx::globaltimer_stable_ns() : 0;          // wall time of the same span: clock rate
        long long* const trace = (p.prof != nullptr && pair == 0 && me < 2) ? p.prof + (size_t)n_pairs * 32 + me * 384 : nullptr;
        int n_ev = 0;
        for (int l = l_lo; l < l_hi; ++my_item_no) {
          const NameItem it = name_item_at(work, pair, l, l_hi);
          l += it.nt;
          const int nt = it.nt;
          for (int t = 0; t < nt; ++t, ++tile_no) {
            const uint32_t buf = tile_no & 1u;
            const uint32_t d_tmem = tmem_base + buf * kAccStride;
            for (int kb = 0; kb < nkb; ++kb, ++g) {
              if ((g % kNumIssuers) != me) continue;
              // k-block g reads vocabulary stages 2g (MMAs kk = 0, 1) and 2g + 1 (kk = 2, 3)
              const int stage0 = (int)((2 * g) % kBStages), stage1 = (int)((2 * g + 1) % kBStages);
              const uint32_t phase0 = ((2 * g) / kBStages) & 1u, phase1 = ((2 * g + 1) / kBStages) & 1u;
              // operands of the four MMAs, ready in registers before the token arrives
              const bool a_in_tmem = kb < kTmemAKBlocks;
              const uint32_t b_addr0 = sbase + NameSmem::b_off + stage0 * kBStageBytes;
              const uint32_t b_addr1 = sbase + NameSmem::b_off + stage1 * kBStageBytes;
              const uint32_t a_addr = sbase + NameSmem::a_off + (a_in_tmem ? 0 : kb - kTmemAKBlocks) * kABlockBytes;
              uint64_t bd[4], ad[4];
              uint32_t at[4];
  #pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                bd[kk] = ptx::make_kmajor_desc((kk < 2 ? b_addr0 : b_addr1) + (kk & 1) * 32, 64);
                ad[kk] = ptx::make_kmajor_desc(a_addr + kk * 32, 128);
                at[kk] = tmem_base + a_tmem_col(a_in_tmem ? kb : 0, kk);
                asm volatile("" : "+l"(bd[kk]), "+l"(ad[kk]), "+r"(at[kk]));
              }
              // Accumulator buffer free / rows of the item loaded?  Waited for ahead of the token - except when a tile has fewer
              // k-blocks than there are issuers (D <= 128).  A parity wait is only sound if the waiter cannot be more than one
              // phase away from the one it asks for.  With one k-block per tile an issuer sits three tiles ahead of the one it
              // issued last: the release it needs (tile - 2) can still have the previous release (tile - 4) pending, the wait
              // returned at once, the MMAs overwrote a buffer the epilogue was reading, and the pair deadlocked (round 1).
              // With two k-blocks per tile and the ONE-TILE work items the linear partition of round 2 produces at range ends,
              // an issuer meets k-block kb of an item only every third item: its early wait on a_full(kb) could alias with the
              // fill before last and the MMAs read rows that were still being written (tools/naming_stress.py: 46 wrong
              // indices in one launch of 19000 x 5000 x 128 out of ~10^4).  After the token every earlier k-block has been
              // issued by a warp that waited for its own fill / release, so the barrier is at most one phase behind.
              const bool te_after_token = nkb < kNumIssuers;
              if (kb == 0 && !te_after_token) { const long long c0 = prof ? clock64() : 0;
                ptx::mbar_wait_nocall(tmem_empty_bar(buf), ((tile_no >> 1) & 1u) ^ 1u, 300 + buf);
                if (prof) pf_te += clock64() - c0; }
              if (t == 0 && !te_after_token) { const long long c0 = prof ? clock64() : 0;
                ptx::mbar_wait_nocall(a_full_bar(kb), my_item_no & 1, 400 + kb);
                if (prof) pf_a += clock64() - c0; }
              // both stages in one probe (their barrier round trips overlap).  Neither can complete a later phase
              // meanwhile: their next fills wait for the releases this k-block's MMAs commit.
              { const long long c0 = prof ? clock64() : 0;
                ptx::mbar_wait2_nocall(full_bar(stage0), phase0, full_bar(stage1), phase1, 500 + stage0);
                if (prof) pf_b += clock64() - c0; }
              ptx::tc_fence_after_sync();
              const long long tr0 = trace ? clock64() : 0;
              // token: the previous issuer has issued k-block g - 1
              if (g > 0) { const long long c0 = prof ? clock64() : 0;
                ptx::named_bar_sync(1 + me, 64);
                if (prof) pf_tok += clock64() - c0; }
              if (te_after_token) {          // same reasoning for the rows of the item: with one k-block per tile the
                if (kb == 0) ptx::mbar_wait_nocall(tmem_empty_bar(buf), ((tile_no >> 1) & 1u) ^ 1u, 310 + buf);    // issuers
                if (t == 0) ptx::mbar_wait_nocall(a_full_bar(kb), my_item_no & 1, 410 + kb);    // take turns on a_full(0) too
                ptx::tc_fence_after_sync();
              }
              const long long tr1 = trace ? clock64() : 0;
              if (p.prof != nullptr && pair == 0 && t == 0 && kb == 0 && lane == 0 && my_item_no < 64)
                p.prof[(size_t)n_pairs * 32 + 4 * 384 + my_item_no * 6 + 0] = clock64();            // first k-block of the item issued
              const bool elected = ptx::elect_one();
              // the first stage is released as soon as its two MMAs have run, the second after the k-block's last MMA
              if (elected) {
                if (a_in_tmem) {
  #pragma unroll
                  for (int kk = 0; kk < 4; ++kk) {
                    ptx::umma_bf16_ts<2>(d_tmem, at[kk], bd[kk], idesc, (kb | kk) != 0 ? 1u : 0u);
                    if (kk == 1) ptx::umma_commit<2>(empty_bar(stage0), 0b11);
                  }
                } else {
  #pragma unroll
                  for (int kk = 0; kk < 4; ++kk) {
                    ptx::umma_bf16<2>(d_tmem, ad[kk], bd[kk], idesc, 1u);
                    if (kk == 1) ptx::umma_commit<2>(empty_bar(stage0), 0b11);
                  }
                }
              }
              __syncwarp();
              if ((long long)g + 1 < g_total) ptx::named_bar_arrive(1 + (me + 1) % kNumIssuers, 64);     // hand the token over ...
              if (elected) {                                                                            // ... then commit
                ptx::umma_commit<2>(empty_bar(stage1), 0b11);
                if (t == nt - 1) ptx::umma_commit<2>(a_empty_bar(kb), 0b11);
                if (kb == nkb - 1) ptx::umma_commit<2>(tmem_full_bar(buf), 0b11);
              }
              __syncwarp();
              if (trace && lane == 0 && n_ev < 128) { trace[3 * n_ev] = tr0; trace[3 * n_ev + 1] = tr1; trace[3 * n_ev + 2] = clock64(); ++n_ev; }
            }
          }
        }
        if (prof && lane == 0) {
          long long* o = p.prof + (size_t)pair * 32;
          o[0] = clock64() - pf_t0; o[1] = pf_te; o[2] = pf_a; o[3] = pf_b; o[4] = pf_tok; o[5] = tile_no;
          o[17] = (long long)(ptx::globaltimer_stable_ns() - pf_ns0);
        }
      }
    }                                    // warps 18, 19: no role
    teardown();
  } else if (wg == 3) {
    ptx::setmaxnreg_dec<kLoaderRegs>();
    // ======================================================= loaders of the TMEM-resident A k-blocks
    // thread = image row = TMEM lane; one k-block = 64 bf16 = 32 packed columns.  Global loads of a k-block are in
    // flight before the wait for its columns to be released by the previous item's last tile.
    const uint32_t quad = warp & 3u;
    const uint32_t lane_addr = (quad * 32u) << 16;
    int my_item_no = 0;
    for (int l = l_lo; l < l_hi; ++my_item_no) {
      const NameItem it = name_item_at(work, pair, l, l_hi);
      l += it.nt;
      const long long row = (long long)it.rb * 2 * kBlockM + cta_rank * kBlockM + quad * 32 + lane;
      const uint4* src = reinterpret_cast<const uint4*>(p.x + (size_t)(row < p.n_rows ? row : 0) * p.d);
      for (int kb = 0; kb < nkb_tmem; ++kb) {
        uint32_t r[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          uint4 v = make_uint4(0u, 0u, 0u, 0u);
          if (row < p.n_rows && kb * kAKBlock + q * 8 < p.d) v = __ldg(src + kb * 8 + q);
          r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
        }
        ptx::mbar_wait_nocall(a_empty_bar(kb), (my_item_no & 1) ^ 1, 150 + kb);
        ptx::tc_fence_after_sync();
        ptx::tmem_st_32x32(tmem_base + lane_addr + a_tmem_col(kb, 0), r);
        ptx::tmem_st_wait();
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_remote(a_full_bar(kb) & ptx::kPeerBitMask);
      }
      // warp 12 is also the TMA producer of the shared-memory A k-blocks: k-block kb >= kTmemAKBlocks of the NEXT item
      // is loaded as soon as the last tile of the current item has consumed it (a_empty, committed by the MMA issuer)
      if (warp == 12) {
        const int row0 = it.rb * 2 * kBlockM + (int)cta_rank * kBlockM;
        for (int kb = kTmemAKBlocks; kb < nkb; ++kb) {
          ptx::mbar_wait_nocall(a_empty_bar(kb), (my_item_no & 1) ^ 1, 100 + kb);
          if (ptx::elect_one()) {
            if (leader) ptx::mbar_arrive_expect_tx(a_full_bar(kb), 2 * kABlockBytes);
            ptx::tma_load_2d<2>(sbase + NameSmem::a_off + (kb - kTmemAKBlocks) * kABlockBytes, &map_x,
                                a_full_bar(kb) & ptx::kPeerBitMask, kb * kAKBlock, row0, ptx::kEvictFirst);
          }
          __syncwarp();
        }
        if (p.prof != nullptr && pair == 0 && leader && lane == 0 && my_item_no < 64)
          p.prof[(size_t)n_pairs * 32 + 4 * 384 + my_item_no * 6 + 5] = clock64();                // the item's rows are on their way
      }
    }
    teardown();
  } else {
    ptx::setmaxnreg_inc<kEpiRegs>();
    // ======================================================= epilogue: one thread per image row
    const uint32_t quad = warp & 3u;                 // TMEM lane quadrant this warp may read
    const uint32_t half = (warp - 4u) >> 2;          // column half of every tile this warp scans
    const uint32_t lane_addr = (quad * 32u) << 16;
    uint32_t tile_no = 0;
    ChunkTop<KT> ctop;
    // parked chunks of this warp's 32 rows: [KT slots][8 float4][32 lanes] - lane-interleaved, so a warp reading one
    // slot of all its rows touches 4 lines per instruction (the per-thread layout of round 1 touched 32: the exact scan
    // was bound by the load/store unit, ~20 k cycles per work item)
    float4* const my_scratch = reinterpret_cast<float4*>(p.scratch) +
                               ((((size_t)blockIdx.x * kEpiHalves + half) * 4 + quad) * KT * 8) * 32 + lane;
    const bool prof = p.prof != nullptr && warp == 4 && leader;
    long long pf_t0 = prof ? clock64() : 0, pf_w = 0, pf_fin = 0;
    long long* const trace = (prof && pair == 0) ? p.prof + (size_t)n_pairs * 32 + 2 * 384 : nullptr;
    int n_ev = 0;
    int epi_item_no = 0;
    for (int l = l_lo; l < l_hi; ++epi_item_no) {
      const NameItem it = name_item_at(work, pair, l, l_hi);
      l += it.nt;
      const int nt = it.nt;
      const long long row = (long long)it.rb * 2 * kBlockM + cta_rank * kBlockM + quad * 32 + lane;
      long long* const itrace = (prof && pair == 0 && lane == 0 && epi_item_no < 64) ? p.prof + (size_t)n_pairs * 32 + 4 * 384 + epi_item_no * 6 : nullptr;
      ctop.reset();
      float run_max = -INFINITY, run_sum = 0.f;

      // one 32-column chunk of this row: chunk maximum -> filter -> (rarely) park the chunk
      auto process = [&](uint32_t (&r)[32], int colbase, int n_valid_here) {
        if (n_valid_here <= 0) return;
        if (n_valid_here < 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j) if (j >= n_valid_here) r[j] = 0xff800000u;   // -inf
        }
        float m8[8];
#pragma unroll
        for (int g = 0; g < 8; ++g)
          m8[g] = fmaxf(fmaxf(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1])),
                        fmaxf(__uint_as_float(r[4 * g + 2]), __uint_as_float(r[4 * g + 3])));
        const float cmax = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
        if (p.want_softmax) {
          if (cmax > run_max) { run_sum *= exp2f((run_max - cmax) * p.scale_log2e); run_max = cmax; }
          float acc = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) acc += exp2f((__uint_as_float(r[j]) - run_max) * p.scale_log2e);
          run_sum += acc;
        }
        if (ctop.admits(cmax, colbase)) {
          float4* dst = my_scratch + ctop.slot[KT - 1] * (8 * 32);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            dst[q * 32] = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                                 __uint_as_float(r[4 * q + 3]));
          ctop.insert_last(cmax, colbase);
        }
      };

      for (int t = 0; t < nt; ++t, ++tile_no) {
        const uint32_t buf = tile_no & 1u;
        const int col0 = item_tile(it, t) * kTileN + (int)half * kHalfCols;
        const int half_cols = half == 0 ? kHalfCols : kTileN - kHalfCols;
        const int n_valid = (int)min((long long)half_cols, p.v_total - col0);      // may be <= 0 on the last tile
        { const long long c0 = prof ? clock64() : 0;
          ptx::mbar_wait_nocall(tmem_full_bar(buf), (tile_no >> 1) & 1u, 600 + buf);
          if (prof) pf_w += clock64() - c0; }
        ptx::tc_fence_after_sync();
        if (itrace && t == 0) itrace[1] = clock64();                                            // first tile of the item seen
        const long long tr0 = trace ? clock64() : 0;
        const uint32_t taddr = tmem_base + lane_addr + buf * kAccStride + half * kHalfCols;
        // four 32-column chunks in the first half, three in the second (96 columns).  Its fourth chunk would be the
        // TMEM-resident A columns: never read tensor memory that may not have been written (for D <= 64 the second
        // A k-block does not exist) - see the E-step epilogue for what that costs.
        // Every load of the warp's share is in flight before the one wait, and the buffer goes back to the MMA issuer
        // before any chunk is processed: it is free again one TMEM load latency after the tile completed.
        uint32_t c0[32], c1[32], c2[32], c3[32];
        ptx::tmem_ld_32x32(taddr, c0);
        ptx::tmem_ld_32x32(taddr + 32, c1);
        ptx::tmem_ld_32x32(taddr + 64, c2);
        if (half == 0) ptx::tmem_ld_32x32(taddr + 96, c3);
        ptx::tmem_ld_wait(c0);
        ptx::tmem_ld_keep(c1);
        ptx::tmem_ld_keep(c2);
        if (half == 0) ptx::tmem_ld_keep(c3);
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_remote(tmem_empty_bar(buf) & ptx::kPeerBitMask);
        const long long tr1 = trace ? clock64() : 0;
        process(c0, col0, n_valid);
        process(c1, col0 + 32, n_valid - 32);
        process(c2, col0 + 64, n_valid - 64);
        if (half == 0) process(c3, col0 + 96, n_valid - 96);
        if (trace && lane == 0 && n_ev < 128) { trace[3 * n_ev] = tr0; trace[3 * n_ev + 1] = tr1; trace[3 * n_ev + 2] = clock64(); ++n_ev; }
      }

      // Exact top-k of the row from its (at most KT) parked chunks.  Every parked chunk contributes its own maximum, so
      // the k-th best element is at least T = the smallest parked maximum; only elements >= T can be in the top-k
      // and on real score distributions there are k .. k + 3 of them among the KT * 32 parked values.
      //  1. one pass over the parked chunks (next chunk's loads in flight behind the current one's compares) builds a
      //     32-bit survivor mask per chunk - no value is kept, no local memory is touched;
      //  2. the first KT + 4 survivors (normally all of them) are re-read from the scratch slots with independent loads -
      //     one L2 round trip - and pushed; a lock-step loop drains what is left (flat score distributions only).
      // Round 2 start: the drain loop did one DEPENDENT L2 load per extra survivor of the warp's worst lane, ~22 k cycles
      // per item (profiles/r2b_name_item_timeline.txt) of which ~11 k hide behind the two tiles the issuers can run
      // ahead into the double-buffered accumulators.  (Round 1 appended survivors to per-thread candidate lists in
      // local memory: divergent st.local, ~28 k cycles per item with the tensor pipe idle for ~18 k of them - 4 % of a
      // whole-vocabulary sweep but 20-37 % of the short items a small row shard is cut into, DESIGN 7.1.)
      const long long pf_c1 = prof ? clock64() : 0;
      if (itrace) itrace[2] = pf_c1;                                                            // last tile processed
      TopK<KT> top;
      top.reset();
      {
        const float keep_from = ctop.m[KT - 1];
        // first column of the chunk parked in PHYSICAL slot e (-1: empty); the scan walks the slots in physical order -
        // every lane reads the same slot, and the order of the pushes does not matter (explicit tie rules)
        int scol[KT];
#pragma unroll
        for (int e = 0; e < KT; ++e) {
          scol[e] = -1;
#pragma unroll
          for (int f = 0; f < KT; ++f) if (ctop.slot[f] == e) scol[e] = ctop.col[f];
        }
        uint32_t mask[KT];
        float4 xa[8], xb[8];
        auto load_chunk = [&](int e, float4 (&x)[8]) {
          const float4* src = my_scratch + e * (8 * 32);
#pragma unroll
          for (int q = 0; q < 8; ++q) x[q] = src[q * 32];
        };
        auto survivors = [&](const float4 (&x)[8], int col) {
          uint32_t m = 0u;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float xv[4] = {x[q].x, x[q].y, x[q].z, x[q].w};
#pragma unroll
            for (int w = 0; w < 4; ++w)
              if (xv[w] >= keep_from && xv[w] > -INFINITY) m |= 1u << (4 * q + w);
          }
          return col >= 0 ? m : 0u;              // an empty slot holds stale values
        };
        load_chunk(0, xa);
#pragma unroll
        for (int e = 0; e < KT; ++e) {
          if (e + 1 < KT) { if (e & 1) load_chunk(e + 1, xa); else load_chunk(e + 1, xb); }
          mask[e] = (e & 1) ? survivors(xb, scol[e]) : survivors(xa, scol[e]);
        }
        // every survivor of the row in ONE round trip: kGather independent scalar re-reads (lowest slot, lowest
        // column first), then the pushes.  kGather = KT + 4 covers what real score distributions leave (k .. k + 3).
        const float* const my_scalars = reinterpret_cast<const float*>(my_scratch);
        auto parked = [&](int slot, int j) { return my_scalars[((slot * 8 + (j >> 2)) * 32) * 4 + (j & 3)]; };
        constexpr int kGather = KT + 4;
        float gv[kGather];
        int gc[kGather];
#pragma unroll
        for (int s2 = 0; s2 < kGather; ++s2) {
          uint32_t m = 0u;
          int slot_sel = 0, col_sel = 0;
#pragma unroll
          for (int e = KT - 1; e >= 0; --e)
            if (mask[e] != 0u) { m = mask[e]; slot_sel = e; col_sel = scol[e]; }
          const bool live = m != 0u;
          const int j = live ? __ffs((int)m) - 1 : 0;
          gv[s2] = live ? parked(slot_sel, j) : -INFINITY;
          gc[s2] = live ? col_sel + j : -1;
          bool cleared = false;
#pragma unroll
          for (int e = 0; e < KT; ++e)
            if (!cleared && mask[e] != 0u) { mask[e] &= mask[e] - 1u; cleared = true; }
        }
#pragma unroll
        for (int s2 = 0; s2 < kGather; ++s2) top.push(gv[s2], gc[s2]);
        // the rest (ties at the threshold / flat score distributions; normally nothing): lock-step, lowest slot first
        uint32_t left = 0u;
#pragma unroll
        for (int e = 0; e < KT; ++e) left |= mask[e];
#pragma unroll 1
        while (__any_sync(0xffffffffu, left != 0u)) {
          uint32_t m = 0u;
          int slot_sel = 0, col_sel = 0;
#pragma unroll
          for (int e = KT - 1; e >= 0; --e)
            if (mask[e] != 0u) { m = mask[e]; slot_sel = e; col_sel = scol[e]; }
          const bool live = m != 0u;
          const int j = live ? __ffs((int)m) - 1 : 0;
          const float v = live ? parked(slot_sel, j) : -INFINITY;
          top.push(v, live ? col_sel + j : -1);
          bool cleared = false;
          left = 0u;
#pragma unroll
          for (int e = 0; e < KT; ++e) {
            if (!cleared && mask[e] != 0u) { mask[e] &= mask[e] - 1u; cleared = true; }
            left |= mask[e];
          }
        }
      }
      if (itrace) itrace[3] = clock64();                                                        // exact scan done
      if (row < p.n_rows) {
        const long long slot = (long long)(it.part * kEpiHalves + (int)half) * p.n_rows + row;
#pragma unroll
        for (int j = 0; j < KT; ++j) { p.part_val[slot * KT + j] = top.v[j]; p.part_idx[slot * KT + j] = top.i[j]; }
        p.part_max[slot] = run_max;
        p.part_sum[slot] = run_sum;
      }
      if (prof) pf_fin += clock64() - pf_c1;
      if (itrace) itrace[4] = clock64();
    }
    if (prof && lane == 0) {
      long long* o = p.prof + (size_t)pair * 32;
      o[8] = clock64() - pf_t0; o[9] = pf_w; o[10] = pf_fin;
    }
    teardown();
  }
}

// Merge `parts` partial top-k lists per row (vocabulary chunks of one GPU: IdxT=int, raw accumulators;
// or the all-gathered lists of several vocabulary shards: IdxT=long long, PRESCALED values) into the
// final sorted top-k: value descending, ties -> lower index.  Also finishes the optional softmax:
//   p_j = exp(scale * (v_j - M)) / sum_parts s_p * exp(scale * (m_p - M)).
template <typename IdxT, bool PRESCALED, int KMAX, bool FULL>   // KMAX >= max(kt_in, k_out), FULL: k_out == KMAX - the lists live in
                                                                 // registers and every subscript is a compile-time constant
__global__ void topk_merge_kernel(const float* __restrict__ part_val, const IdxT* __restrict__ part_idx,
                                  const float* __restrict__ part_max, const float* __restrict__ part_sum,
                                  int parts, long long n_rows, int kt_in, int k_out, float scale, int want_softmax,
                                  long long idx_offset, float* __restrict__ out_val, long long* __restrict__ out_idx,
                                  float* __restrict__ out_max, float* __restrict__ out_sum, const NameWork work) {
  const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  // lists of one launch of name_topk_kernel: a row block has pieces(rb) pieces x 2 column halves (work.P > 0);
  // all-gathered vocabulary shards: `parts` lists for every row
  if (work.P > 0) parts = work.pieces((int)(row / (2 * kBlockM))) * kEpiHalves;
  float bv[KMAX]; long long bi[KMAX];                    // (value descending, index ascending); entries >= k_out stay empty
#pragma unroll
  for (int j = 0; j < KMAX; ++j) { bv[j] = -INFINITY; bi[j] = -1; }
  auto before = [](float xa, long long ia, float xb, long long ib) { return ib < 0 || xa > xb || (xa == xb && ia < ib); };
  float M = -INFINITY;
  for (int q = 0; q < parts; ++q) {
    const long long slot = (long long)q * n_rows + row;
    // the whole list of part q is loaded at once (independent loads).  Round 2a's version indexed its lists with runtime
    // subscripts: they lived in local memory and the shifting loop was 55 % of the kernel's instructions (31 us at C2).
    float xv[KMAX]; long long xi[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
      xv[j] = j < kt_in ? part_val[slot * kt_in + j] : -INFINITY;
      xi[j] = j < kt_in ? (long long)part_idx[slot * kt_in + j] : -1;
    }
    if (xi[0] < 0) continue;                             // this row has nothing in part q
    if (part_max) M = fmaxf(M, part_max[slot]);
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
      if (xi[j] < 0) continue;
      float lv = bv[KMAX - 1]; long long li = bi[KMAX - 1];      // the last element currently kept (position k_out - 1)
      if (!FULL) {
#pragma unroll
        for (int t = 0; t < KMAX; ++t) if (t == k_out - 1) { lv = bv[t]; li = bi[t]; }
      }
      if (!before(xv[j], xi[j], lv, li)) continue;
      if (FULL) { bv[KMAX - 1] = xv[j]; bi[KMAX - 1] = xi[j]; }
      else {
#pragma unroll
        for (int t = 0; t < KMAX; ++t) if (t == k_out - 1) { bv[t] = xv[j]; bi[t] = xi[j]; }
      }
#pragma unroll
      for (int t = KMAX - 1; t > 0; --t) {
        if ((FULL || t < k_out) && before(bv[t], bi[t], bv[t - 1], bi[t - 1])) {
          const float tv = bv[t]; bv[t] = bv[t - 1]; bv[t - 1] = tv;
          const long long ti = bi[t]; bi[t] = bi[t - 1]; bi[t - 1] = ti;
        }
      }
    }
  }
  float S = 0.f;
  if (part_max) {
    for (int q = 0; q < parts; ++q) {
      const long long slot = (long long)q * n_rows + row;
      if ((long long)part_idx[slot * kt_in] < 0) continue;
      const float m = part_max[slot];
      if (m > -INFINITY) S += part_sum[slot] * expf(scale * (m - M));
    }
    if (out_max) { out_max[row] = M; out_sum[row] = S; }
  }
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    if (j >= k_out) continue;
    float val = PRESCALED ? bv[j] : bv[j] * scale;
    if (want_softmax) val = (PRESCALED ? expf(bv[j] - scale * M) : expf(scale * (bv[j] - M))) / S;
    out_val[row * k_out + j] = val;
    out_idx[row * k_out + j] = bi[j] < 0 ? -1 : bi[j] + idx_offset;
  }
}

}  // namespace scd

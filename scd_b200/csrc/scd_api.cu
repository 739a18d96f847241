// C ABI of scd_b200 (see include/scd_b200.h): argument checking, workspace carving, tensor-map
// construction and kernel launches.  No allocation, no synchronisation.
#include "../../include/scd_b200.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>

#include "estep_tc_kernel.cuh"
#include "kmeans_kernel.cuh"
#include "naming_kernel.cuh"
#include "vote_kernel.cuh"
#include "eval_kernel.cuh"
#include "peer_kernel.cuh"

namespace {

thread_local std::string g_last_error;
long long* g_name_prof = nullptr;      // scd_debug_set_name_profile

int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return 1;
}

#define SCD_CUDA(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) return fail("%s failed: %s", #expr, cudaGetErrorString(_e));    \
  } while (0)

#define SCD_LAUNCH_CHECK(name)                                                             \
  do {                                                                                     \
    cudaError_t _e = cudaGetLastError();                                                   \
    if (_e != cudaSuccess) return fail("launch of %s failed: %s", name, cudaGetErrorString(_e)); \
  } while (0)

inline cudaStream_t as_stream(scd_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Per-device caches: function attributes and SM counts belong to a device, and although the intended deployment is one
// process per GPU, a host process may switch devices between calls.
constexpr int kMaxDevices = 64;

int current_device_slot() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 0;
  return dev;
}

int device_sm_count() {
  static int cached[kMaxDevices] = {};
  const int dev = current_device_slot();
  if (cached[dev]) return cached[dev];
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  cached[dev] = n;
  return n;
}

// Raises Kernel's dynamic shared-memory limit on the current device to `bytes` unless it is set that high already.
template <auto Kernel>
int allow_dynamic_smem(int bytes) {
  static int set[kMaxDevices] = {};
  const int dev = current_device_slot();
  if (bytes > set[dev]) {
    SCD_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    set[dev] = bytes;
  }
  return 0;
}

// ---------------------------------------------------------------- tensor maps
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 2-D row-major [rows, cols] tensor (bf16 or fp32), box = [box_rows, box_cols], inner (cols) swizzled
int make_map_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows, uint32_t box_cols,
                CUtensorMapSwizzle swz, bool is_f32 = false) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail("cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * (is_f32 ? 4u : 2u)};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base),
                  dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu)", (int)r,
                                     (unsigned long long)rows, (unsigned long long)cols);
  return 0;
}

// two bf16 planes [2][rows, cols] `plane_bytes` apart as one 3-D tensor, box = [2][box_rows][box_cols], SWIZZLE_64B
int make_map_planes(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t plane_bytes, uint32_t box_rows,
                    uint32_t box_cols) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail("cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {cols, rows, 2};
  cuuint64_t strides[2] = {cols * 2u, plane_bytes};
  cuuint32_t box[3] = {box_cols, box_rows, 2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (planes) failed with CUresult %d (rows=%llu cols=%llu)", (int)r,
                                     (unsigned long long)rows, (unsigned long long)cols);
  return 0;
}

// ---------------------------------------------------------------- naming plan
struct NamePlan {
  int kt;                 // compiled list length (1, 5 or 8)
  int n_row_blocks;
  int tiles_total;
  int n_pairs;
  int n_slots;            // most pieces any row block is cut into (partial-list slots per row and column half)
  long long work_total;   // n_row_blocks * tiles_total
  size_t off_val, off_idx, off_max, off_sum, off_scratch, bytes;
};

// top-k list length the scoring and merge kernels are compiled for, k in 1..8
inline int list_len(int k) { return k == 1 ? 1 : (k <= 5 ? 5 : 8); }

bool plan_naming(int64_t N, int64_t V, int k, NamePlan* pl) {
  if (k < 1 || k > 8) return false;
  pl->kt = list_len(k);
  pl->n_row_blocks = (int)((N + 2 * scd::kBlockM - 1) / (2 * scd::kBlockM));
  pl->tiles_total = (int)((V + scd::kTileN - 1) / scd::kTileN);
  pl->work_total = (long long)pl->n_row_blocks * pl->tiles_total;
  if (pl->work_total >= (1ll << 31)) return false;
  const int pairs_hw = std::max(1, device_sm_count() / 2);
  // The (row block, tile) space is cut into one contiguous range per CTA pair (scd::NameWork): every pair gets the same
  // number of tiles (+-1) whatever N is, and starts as few work items as possible.  (Round 1 gave whole row blocks to
  // whole waves and cut only the tail wave along the vocabulary: at 63 row blocks on 74 pairs that made six 14-tile
  // items per pair, each paying the item start-up and the final exact scan.)
  pl->n_pairs = (int)std::max<long long>(1, std::min<long long>(pairs_hw, pl->work_total));
  const scd::NameWork w{pl->work_total, pl->tiles_total, pl->n_pairs};
  int slots = 1;
  if (pl->work_total % pl->n_pairs != 0 || (pl->work_total / pl->n_pairs) % pl->tiles_total != 0) {
    // a pair boundary falls inside some row block: bound the pieces by ceil(T / smallest range) + 1, then tighten by
    // walking the boundaries (n_pairs of them)
    slots = 0;
    int cur_rb = -1, cur = 0;
    for (int q = 0; q < pl->n_pairs; ++q) {
      const long long lo = w.bound(q), hi = w.bound(q + 1);
      if (lo >= hi) continue;
      const int rb_first = (int)(lo / pl->tiles_total), rb_last = (int)((hi - 1) / pl->tiles_total);
      if (rb_first == cur_rb) ++cur; else { cur_rb = rb_first; cur = 1; }
      slots = std::max(slots, cur);
      if (rb_last != rb_first) { cur_rb = rb_last; cur = 1; }
    }
    slots = std::max(slots, 1);
  }
  pl->n_slots = slots;
  size_t o = 0;
  const size_t lists = (size_t)pl->n_slots * scd::kEpiHalves * (size_t)N;      // one partial list per (piece, column half)
  pl->off_val = o; o = align_up(o + lists * pl->kt * sizeof(float), 256);
  pl->off_idx = o; o = align_up(o + lists * pl->kt * sizeof(int), 256);
  pl->off_max = o; o = align_up(o + lists * sizeof(float), 256);
  pl->off_sum = o; o = align_up(o + lists * sizeof(float), 256);
  pl->off_scratch = o; o = align_up(o + (size_t)2 * pairs_hw * scd::kEpiHalves * scd::kBlockM * pl->kt * 32 * sizeof(float), 256);
  pl->bytes = std::max<size_t>(o, 256);
  return true;
}

template <int KT>
int launch_name_topk(const CUtensorMap& mx, const CUtensorMap& mw, const scd::NameParams& p, int n_pairs, cudaStream_t st) {
  const int smem = scd::NameSmem::total + 1024;
  if (int e = allow_dynamic_smem<scd::name_topk_kernel<KT>>(smem)) return e;
  scd::name_topk_kernel<KT><<<2 * n_pairs, scd::kNameThreads, smem, st>>>(mx, mw, p);
  SCD_LAUNCH_CHECK("name_topk_kernel");
  return 0;
}

// topk_merge_kernel for lists of `kmax` = list_len(k) entries; FULL (every subscript a compile-time constant) when k == kmax
template <typename IdxT, bool PRESCALED, typename... Args>
void launch_topk_merge(int kmax, int k, int64_t n_rows, cudaStream_t st, const Args&... args) {
  auto kernel = scd::topk_merge_kernel<IdxT, PRESCALED, 1, true>;
  if (kmax == 5) kernel = k == 5 ? scd::topk_merge_kernel<IdxT, PRESCALED, 5, true> : scd::topk_merge_kernel<IdxT, PRESCALED, 5, false>;
  else if (kmax == 8) kernel = k == 8 ? scd::topk_merge_kernel<IdxT, PRESCALED, 8, true> : scd::topk_merge_kernel<IdxT, PRESCALED, 8, false>;
  kernel<<<(unsigned)((n_rows + 127) / 128), 128, 0, st>>>(args...);
}

// ---- counting sort of rows by label: workspace carving shared by the M-step and the vote
// ints: offsets[K+1] | cursor[K] | acc[K] | ticket[1] | order[N]
struct SortWs {
  int* offsets; int* cursor; int* acc; unsigned* ticket; int* order;
  SortWs(void* ws, int K) {
    offsets = reinterpret_cast<int*>(ws);
    cursor = offsets + K + 1;
    acc = cursor + K;
    ticket = reinterpret_cast<unsigned*>(acc + K);
    order = acc + K + 1;
  }
  static size_t ints(int64_t N, int K) { return 3 * (size_t)K + 2 + (size_t)std::max<int64_t>(N, 0); }
};
constexpr int kMaxSortK = 11264;          // 44 KB of shared-memory counters (+ the static scan scratch stays under 48 KB)

// ---- E-step workspace carving shared by scd_estep and the finalize entry points that leave the next E-step's operands
// bf16 hi plane [K, D] | bf16 lo plane [K, D] | ||c||^2 [K], each 256-byte aligned; a null workspace carves null pointers
struct EsWs {
  __nv_bfloat16* chi = nullptr; __nv_bfloat16* clo = nullptr; float* cnorm = nullptr;
  size_t plane;                           // bytes from one plane to the next
  EsWs(void* ws, int K, int D) : plane(plane_bytes(K, D)) {
    if (!ws) return;
    uint8_t* w8 = reinterpret_cast<uint8_t*>(ws);
    chi = reinterpret_cast<__nv_bfloat16*>(w8);
    clo = reinterpret_cast<__nv_bfloat16*>(w8 + plane);
    cnorm = reinterpret_cast<float*>(w8 + 2 * plane);
  }
  static size_t plane_bytes(int K, int D) { return align_up((size_t)K * D * 2, 256); }
  static size_t bytes(int K, int D) { return plane_bytes(K, D) * 2 + align_up((size_t)K * sizeof(float), 256) + 256; }
};

template <typename LabT>
int sort_rows_by_label(const LabT* labels, long long stride, int64_t N, int K, int32_t* counts_out, const SortWs& w,
                              float* zero_me, size_t n_zero_floats, cudaStream_t st) {
  SCD_CUDA(cudaMemsetAsync(w.acc, 0, sizeof(int) * ((size_t)K + 1), st));          // accumulator + ticket
  const int blocks = (int)std::max<long long>(1, std::min<long long>((N + scd::kSortThreads - 1) / scd::kSortThreads, device_sm_count() * 4));
  scd::label_hist_scan_kernel<LabT><<<blocks, scd::kSortThreads, sizeof(int) * (size_t)K, st>>>(
      labels, stride, N, K, w.acc, w.ticket, counts_out, w.offsets, w.cursor, reinterpret_cast<float4*>(zero_me),
      (long long)(n_zero_floats / 4));
  SCD_LAUNCH_CHECK("label_hist_scan_kernel");
  if (N > 0) {
    const int sblocks = (int)((N + scd::kScatterRows - 1) / scd::kScatterRows);
    scd::label_scatter_kernel<LabT><<<sblocks, scd::kSortThreads, sizeof(int) * (size_t)K, st>>>(labels, stride, N, K, w.cursor, w.order);
    SCD_LAUNCH_CHECK("label_scatter_kernel");
  }
  return 0;
}

template <typename IdxT, bool SEG = false>
int launch_vote(const IdxT* topk_idx, long long idx_stride, int k_used, int64_t N, const int* order, const int* offsets, int K,
                       const int64_t* excluded, int n_excluded, int M, int64_t* out_names, int32_t* out_counts,
                       int32_t* out_distinct, int32_t* overflow, void* spill, size_t spill_bytes, cudaStream_t st,
                       const int* seg_offsets = nullptr, int seg_world = 0, long long seg_per = 0, int32_t* out_rows = nullptr) {
  if (spill && spill_bytes < scd::vote_spill_bytes(N, k_used)) return fail("vote: spill buffer too small (%zu < %zu)", spill_bytes, scd::vote_spill_bytes(N, k_used));
  SCD_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int), st));
  if (int e = allow_dynamic_smem<scd::vote_kernel<IdxT, SEG>>(scd::kVoteSmemBytes)) return e;
  scd::vote_kernel<IdxT, SEG><<<K, scd::kVoteThreads, scd::kVoteSmemBytes, st>>>(
      topk_idx, idx_stride, k_used, order, offsets, K, reinterpret_cast<const long long*>(excluded), n_excluded, M,
      reinterpret_cast<long long*>(out_names), out_counts, out_distinct, overflow, reinterpret_cast<int*>(spill),
      seg_offsets, seg_world, seg_per, out_rows);
  SCD_LAUNCH_CHECK("vote_kernel");
  return 0;
}

// the checks every vote entry point makes; `who` names the entry point in the error message
int check_vote_args(const char* who, int64_t N, int K, int k_total, int k_used, int M, const int64_t* excluded, int n_excluded,
                    const int64_t* out_names, const int32_t* out_counts, const int32_t* out_distinct, const int32_t* overflow) {
  if (N < 0 || K <= 0 || k_total <= 0 || k_used <= 0 || k_used > k_total || M <= 0) return fail("%s: bad arguments", who);
  if (N * (int64_t)k_used >= (1ll << 31)) return fail("%s: N * k_used exceeds the 31-bit position range", who);
  if (K > kMaxSortK) return fail("%s: K=%d too large", who, K);
  if (!out_names || !out_counts || !out_distinct || !overflow) return fail("%s: null pointer", who);
  if (n_excluded > 0 && !excluded) return fail("%s: excluded list is null", who);
  return 0;
}

int make_peer_ptrs(scd::PeerPtrs* pp, void* const* bufs, void* const* flags, int world, int rank, const char* who) {
  if (world < 2 || world > scd::kPeerMaxWorld || rank < 0 || rank >= world) return fail("%s: bad world / rank (%d / %d)", who, world, rank);
  if (!bufs) return fail("%s: null peer buffer table", who);
  for (int r = 0; r < scd::kPeerMaxWorld; ++r) {
    pp->buf[r] = r < world ? bufs[r] : nullptr;
    pp->flags[r] = (r < world && flags) ? reinterpret_cast<unsigned*>(flags[r]) : nullptr;
    if (r < world && (!pp->buf[r] || (flags && !pp->flags[r]))) return fail("%s: null peer pointer for rank %d", who, r);
  }
  pp->world = world;
  pp->rank = rank;
  return 0;
}

}  // namespace

extern "C" {

int scd_version(void) { return 200; }

void scd_debug_set_name_profile(void* dev_buf_pairs_x16_i64) { g_name_prof = reinterpret_cast<long long*>(dev_buf_pairs_x16_i64); }

const char* scd_last_error(void) { return g_last_error.c_str(); }

// ============================================================================ k-means
int scd_pairwise_distance(const float* X, int64_t N, int D, const float* C, int K, float* out, int32_t* cost_x1000,
                          scd_stream_t stream) {
  if (N < 0 || D <= 0 || K <= 0) return fail("scd_pairwise_distance: bad shape N=%lld D=%d K=%d", (long long)N, D, K);
  if (N == 0) return 0;
  if (!X || !C || (!out && !cost_x1000)) return fail("scd_pairwise_distance: null pointer");
  dim3 grid((unsigned)((N + scd::kDistBM - 1) / scd::kDistBM), (unsigned)((K + scd::kDistBN - 1) / scd::kDistBN));
  scd::sqdist_kernel<false><<<grid, scd::kDistThreads, 0, as_stream(stream)>>>(X, N, D, C, K, out, cost_x1000, nullptr, nullptr, nullptr);
  SCD_LAUNCH_CHECK("sqdist_kernel<full>");
  return 0;
}

int scd_estep_uses_tensor_cores(int64_t N, int D, int K) {
  return D % 8 == 0 && D > scd::kEsBK * (scd::kEsConvSets - 1) && K > 0 && K <= scd::kEsMaxK && N < (1ll << 31) ? 1 : 0;
}

size_t scd_estep_workspace_bytes(int K, int D) {
  if (K <= 0 || D <= 0) return 256;
  return EsWs::bytes(K, D);
}

int scd_estep(const float* X, int64_t N, int D, const float* C, int K, int64_t* labels, float* mindist, double* inertia_acc,
              int flags, void* ws, size_t ws_bytes, scd_stream_t stream) {
  if (N < 0 || D <= 0 || K <= 0) return fail("scd_estep: bad shape N=%lld D=%d K=%d", (long long)N, D, K);
  if (N == 0) return 0;
  if (!X || !C || !labels) return fail("scd_estep: null pointer");
  const bool exact = (flags & SCD_ESTEP_EXACT) != 0;
  cudaStream_t st = as_stream(stream);
  // TMA needs 16-byte row pitches: fp32 X (D % 4) and the bf16 centroid planes (D % 8); every converter
  // warp set must own at least one k-block per tile (it publishes its share of ||x||^2 there)
  const bool tc_ok = !exact && scd_estep_uses_tensor_cores(N, D, K) && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && ws &&
                     ws_bytes >= scd_estep_workspace_bytes(K, D);
  if (!tc_ok) {
    dim3 grid((unsigned)((N + scd::kDistBM - 1) / scd::kDistBM));
    scd::sqdist_kernel<true><<<grid, scd::kDistThreads, 0, st>>>(X, N, D, C, K, nullptr, nullptr,
                                                                 reinterpret_cast<long long*>(labels), mindist, inertia_acc);
    SCD_LAUNCH_CHECK("sqdist_kernel<fused argmin>");
    return 0;
  }
  const EsWs w(ws, K, D);
  if (!(flags & SCD_ESTEP_PLANES_READY)) {      // scd_finalize_centers(estep_ws = ws) already left the planes of C there
    scd::centroid_split_kernel<<<K, scd::kEsCentroidThreads, 0, st>>>(C, K, D, w.chi, w.clo, w.cnorm);
    SCD_LAUNCH_CHECK("centroid_split_kernel");
  }

  scd::EsParams p;
  p.n_rows = N;
  p.n_clusters = K;
  p.n_ntiles = (K + 255) / 256;
  p.n_tile = p.n_ntiles > 1 ? 256 : ((K + 15) / 16) * 16;
  p.num_kb = (D + scd::kEsBK - 1) / scd::kEsBK;
  p.n_row_tiles = (int)((N + scd::kEsBM - 1) / scd::kEsBM);
  p.cnorm = w.cnorm;
  p.labels = reinterpret_cast<long long*>(labels);
  p.mindist = mindist;
  p.inertia = inertia_acc;
  p.prof = g_name_prof;
  CUtensorMap mx, mc;
  if (int e = make_map_2d(&mx, X, (uint64_t)N, (uint64_t)D, scd::kEsBM, scd::kEsBK, CU_TENSOR_MAP_SWIZZLE_128B, true)) return e;
  // hi and lo planes as one 3-D tensor [2][K][D]: a single box brings both k-slabs of a stage
  if (int e = make_map_planes(&mc, w.chi, (uint64_t)K, (uint64_t)D, w.plane, (uint32_t)p.n_tile, scd::kEsBK)) return e;
  // shared-memory plan: the centroid ring takes what n_tile needs, the rest goes to fp32 X stages in flight
  p.b_plane = p.n_tile * scd::kEsBK * 2;          // n_tile % 16 == 0 -> a multiple of 1024 (swizzle-atom aligned)
  // converted-operand ring: six stages in the TMEM columns the two accumulators leave free (32 columns per stage, three
  // above each accumulator) when they exist, else three stages in shared memory
  const bool tmem_a = p.n_ntiles == 1 && p.n_tile + 3 * 32 <= 256 && p.num_kb >= 3;
  p.a_stages = tmem_a ? 6 : scd::kEsAStages;
  {
    const int fixed = scd::EsLayout(0, p.b_plane, tmem_a).total + 1024;
    p.x_stages = std::max(2, std::min(scd::kEsMaxXStages, (scd::kEsSmemLimit - fixed) / scd::kEsXBytes));
    // EVEN, always: k-block g is loaded by X producer (g & 1) and read by converter set (g & 1).  With an even ring a
    // stage belongs to one producer / set pair and its x_full phases are consumed in order.  With an odd ring the two
    // sets alternate on every stage, and a set that runs one ring revolution ahead of the other sees the parity of
    // the phase before last as "its" phase (parity aliasing): it reads a stale tile, releases the stage early, and the
    // producers then double-arrive on x_full - about one launch in 10^3..10^4 died with "unspecified launch failure"
    // for K = 200 / 208 / 224 (five stages) until this was found with tools/estep_stress2.py.
    p.x_stages &= ~1;
  }
  const int smem = scd::EsLayout(p.x_stages, p.b_plane, tmem_a).total + 1024;
  if (smem > scd::kEsSmemLimit) return fail("scd_estep: shared-memory plan does not fit (%d bytes)", smem);
  if (int e = tmem_a ? allow_dynamic_smem<scd::estep_tc_kernel<true>>(smem) : allow_dynamic_smem<scd::estep_tc_kernel<false>>(smem)) return e;
  const int grid = std::min(device_sm_count(), p.n_row_tiles);
  if (tmem_a) scd::estep_tc_kernel<true><<<grid, scd::kEsThreads, smem, st>>>(mx, mc, p);
  else scd::estep_tc_kernel<false><<<grid, scd::kEsThreads, smem, st>>>(mx, mc, p);
  SCD_LAUNCH_CHECK("estep_tc_kernel");
  return 0;
}

// ---------------------------------------------------------------------------- k-means++ seeding (a5)
size_t scd_kpp_workspace_bytes(int64_t N) {
  const size_t nb = (size_t)((std::max<int64_t>(N, 1) + scd::kKppRowsPerBlock - 1) / scd::kKppRowsPerBlock);
  return align_up(nb * sizeof(double), 256) + 256;
}

int scd_kpp_update(const float* X, int64_t N, int D, const int64_t* pick, const float* center, int first, float* d2,
                   float* center_out, void* ws, size_t ws_bytes, scd_stream_t stream) {
  if (N <= 0 || D <= 0) return fail("scd_kpp_update: bad shape N=%lld D=%d", (long long)N, D);
  if (!X || (!pick && !center) || !d2 || !ws) return fail("scd_kpp_update: null pointer");
  if (ws_bytes < scd_kpp_workspace_bytes(N)) return fail("scd_kpp_update: workspace too small");
  const int nb = (int)((N + scd::kKppRowsPerBlock - 1) / scd::kKppRowsPerBlock);
  scd::kpp_update_kernel<<<nb, 256, 0, as_stream(stream)>>>(X, N, D, reinterpret_cast<const long long*>(pick), center, first, d2,
                                                            reinterpret_cast<double*>(ws), center_out);
  SCD_LAUNCH_CHECK("kpp_update_kernel");
  return 0;
}

int scd_kpp_select(const float* d2, int64_t N, int sums_valid, double r, int64_t* pick, int32_t* no_hit, void* ws, size_t ws_bytes,
                   scd_stream_t stream) {
  if (N <= 0) return fail("scd_kpp_select: bad shape N=%lld", (long long)N);
  if (!d2 || !pick || !no_hit || !ws) return fail("scd_kpp_select: null pointer");
  if (ws_bytes < scd_kpp_workspace_bytes(N)) return fail("scd_kpp_select: workspace too small");
  const int nb = (int)((N + scd::kKppRowsPerBlock - 1) / scd::kKppRowsPerBlock);
  cudaStream_t st = as_stream(stream);
  if (!sums_valid) {
    scd::kpp_block_sums_kernel<<<nb, 256, 0, st>>>(d2, N, reinterpret_cast<double*>(ws));
    SCD_LAUNCH_CHECK("kpp_block_sums_kernel");
  }
  scd::kpp_select_kernel<<<1, 1024, 0, st>>>(d2, N, reinterpret_cast<const double*>(ws), nb, r, reinterpret_cast<long long*>(pick), no_hit);
  SCD_LAUNCH_CHECK("kpp_select_kernel");
  return 0;
}

int scd_labelled_inertia(const float* L, const int64_t* labels, int64_t n, int D, const float* C, int K, double* acc,
                         scd_stream_t stream) {
  if (n < 0 || D <= 0 || K <= 0) return fail("scd_labelled_inertia: bad shape");
  if (n == 0) return 0;
  if (!L || !labels || !C || !acc) return fail("scd_labelled_inertia: null pointer");
  const long long threads = n * 32;
  scd::gather_sqdist_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, as_stream(stream)>>>(
      L, reinterpret_cast<const long long*>(labels), n, D, C, K, acc);
  SCD_LAUNCH_CHECK("gather_sqdist_kernel");
  return 0;
}

size_t scd_mstep_workspace_bytes(int64_t N, int K) { return align_up(SortWs::ints(N, std::max(K, 0)) * sizeof(int), 256) + 256; }

int scd_label_histogram(const int64_t* labels, int64_t N, int K, int32_t* counts, scd_stream_t stream) {
  if (N < 0 || K <= 0) return fail("scd_label_histogram: bad shape N=%lld K=%d", (long long)N, K);
  if (K > kMaxSortK) return fail("scd_label_histogram: K=%d too large for the shared-memory histogram", K);
  if (!counts || (N > 0 && !labels)) return fail("scd_label_histogram: null pointer");
  cudaStream_t st = as_stream(stream);
  SCD_CUDA(cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)K, st));
  if (N > 0) {
    const int blocks = (int)std::min<long long>((N + 255) / 256, device_sm_count() * 8);
    scd::label_hist_kernel<<<blocks, 256, sizeof(int) * (size_t)K, st>>>(reinterpret_cast<const long long*>(labels), N, K, counts);
    SCD_LAUNCH_CHECK("label_hist_kernel");
  }
  return 0;
}

int scd_mstep_sums(const float* X, const int64_t* labels, int64_t N, int D, int K, float* sums, int32_t* counts, void* ws,
                   size_t ws_bytes, scd_stream_t stream) {
  if (N < 0 || D <= 0 || K <= 0) return fail("scd_mstep_sums: bad shape N=%lld D=%d K=%d", (long long)N, D, K);
  if (N >= (1ll << 31)) return fail("scd_mstep_sums: N=%lld exceeds the int32 row-index range", (long long)N);
  const bool vec_ok = D % 4 == 0 && D <= 128 * scd::kSegMaxVec + 124 && (reinterpret_cast<uintptr_t>(X) & 15) == 0;
  if (K > kMaxSortK) return fail("scd_mstep_sums: K=%d too large for the shared-memory histogram", K);
  if (!sums || !counts || !ws) return fail("scd_mstep_sums: null pointer");
  if (ws_bytes < scd_mstep_workspace_bytes(N, K)) return fail("scd_mstep_sums: workspace too small (%zu < %zu)", ws_bytes, scd_mstep_workspace_bytes(N, K));
  cudaStream_t st = as_stream(stream);
  const SortWs w(ws, K);
  const size_t n_sums = (size_t)K * D;
  const bool zero_in_kernel = n_sums % 4 == 0 && (reinterpret_cast<uintptr_t>(sums) & 15) == 0;
  if (!zero_in_kernel) SCD_CUDA(cudaMemsetAsync(sums, 0, sizeof(float) * n_sums, st));
  if (int e = sort_rows_by_label<long long>(reinterpret_cast<const long long*>(labels), 1, N, K, counts, w, zero_in_kernel ? sums : nullptr,
                                            zero_in_kernel ? n_sums : 0, st)) return e;
  const int* order = w.order;
  const int* offsets = w.offsets;
  if (N > 0 && vec_ok) {
    const long long warps = (N + scd::kSegRows - 1) / scd::kSegRows;
    const long long blocks = (warps * 32 + 255) / 256;
    const int nvec = D >> 7;
    if (nvec <= 2) scd::segment_sum_kernel<2><<<(unsigned)blocks, 256, 0, st>>>(X, order, offsets, K, D, sums);
    else if (nvec <= 4) scd::segment_sum_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(X, order, offsets, K, D, sums);
    else if (nvec <= 6) scd::segment_sum_kernel<6><<<(unsigned)blocks, 256, 0, st>>>(X, order, offsets, K, D, sums);
    else scd::segment_sum_kernel<8><<<(unsigned)blocks, 256, 0, st>>>(X, order, offsets, K, D, sums);
    SCD_LAUNCH_CHECK("segment_sum_kernel");
  } else if (N > 0) {
    dim3 grid((unsigned)K, (unsigned)((D + 127) / 128));
    scd::segment_sum_generic_kernel<<<grid, 128, 0, st>>>(X, order, offsets, K, D, sums);
    SCD_LAUNCH_CHECK("segment_sum_generic_kernel");
  }
  return 0;
}

int scd_pack_counts_inertia(const int32_t* counts, const double* inertia, int K, float* out, scd_stream_t stream) {
  if (K <= 0 || !counts || !out) return fail("scd_pack_counts_inertia: bad arguments");
  scd::pack_counts_inertia_kernel<<<(K + 1 + 255) / 256, 256, 0, as_stream(stream)>>>(counts, inertia, K, out);
  SCD_LAUNCH_CHECK("pack_counts_inertia_kernel");
  return 0;
}

int scd_finalize_centers(const float* sums, const int32_t* counts, const float* counts_f, const float* C_old, float* C_new,
                         float* shift, int K, int D, void* ws, size_t ws_bytes, void* estep_ws, size_t estep_ws_bytes,
                         scd_stream_t stream) {
  if (K <= 0 || D <= 0) return fail("scd_finalize_centers: bad shape");
  if (!sums || (!counts && !counts_f) || !C_new) return fail("scd_finalize_centers: null pointer");
  if (shift && (!C_old || !ws)) return fail("scd_finalize_centers: shift needs C_old and K floats of workspace");
  if (ws && ws_bytes < sizeof(float) * (size_t)K) return fail("scd_finalize_centers: workspace too small (K floats)");
  if (estep_ws && estep_ws_bytes < scd_estep_workspace_bytes(K, D)) return fail("scd_finalize_centers: estep workspace too small");
  cudaStream_t st = as_stream(stream);
  float* norms = (ws && C_old) ? reinterpret_cast<float*>(ws) : nullptr;
  const EsWs es(estep_ws, K, D);
  scd::finalize_centers_kernel<<<K, scd::kEsCentroidThreads, 0, st>>>(sums, counts_f, counts, C_old, C_new, norms, K, D, es.chi, es.clo,
                                                                      es.cnorm);
  SCD_LAUNCH_CHECK("finalize_centers_kernel");
  if (shift) {
    scd::sum_small_kernel<<<1, 1024, 0, st>>>(norms, K, shift);
    SCD_LAUNCH_CHECK("sum_small_kernel");
  }
  return 0;
}

// ============================================================================ naming
int scd_vocab_prepare(const void* W, int w_is_bf16, int D, int64_t V, int64_t ldw, scd_bf16_t* Wt, scd_stream_t stream) {
  if (D <= 0 || V < 0 || ldw < V) return fail("scd_vocab_prepare: bad shape D=%d V=%lld ldw=%lld", D, (long long)V, (long long)ldw);
  if (V == 0) return 0;
  if (!W || !Wt) return fail("scd_vocab_prepare: null pointer");
  dim3 grid((unsigned)((V + 31) / 32), (unsigned)((D + 31) / 32)), block(32, 8);
  if (w_is_bf16)
    scd::transpose_to_bf16_kernel<__nv_bfloat16><<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(W), D, V, ldw,
                                                                                         reinterpret_cast<__nv_bfloat16*>(Wt));
  else
    scd::transpose_to_bf16_kernel<float><<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const float*>(W), D, V, ldw,
                                                                                 reinterpret_cast<__nv_bfloat16*>(Wt));
  SCD_LAUNCH_CHECK("transpose_to_bf16_kernel");
  return 0;
}

int scd_cast_bf16(const float* in, int64_t n, scd_bf16_t* out, scd_stream_t stream) {
  if (n < 0) return fail("scd_cast_bf16: bad size");
  if (n == 0) return 0;
  if (!in || !out) return fail("scd_cast_bf16: null pointer");
  const int blocks = (int)std::min<long long>((n + 255) / 256, device_sm_count() * 16);
  scd::cast_f32_to_bf16_kernel<<<blocks, 256, 0, as_stream(stream)>>>(in, n, reinterpret_cast<__nv_bfloat16*>(out));
  SCD_LAUNCH_CHECK("cast_f32_to_bf16_kernel");
  return 0;
}

int scd_gather_rows_bf16(const scd_bf16_t* Wt, const int64_t* sel, int n_sel, int D, int64_t V, scd_bf16_t* out, scd_stream_t stream) {
  if (n_sel < 0 || D <= 0) return fail("scd_gather_rows_bf16: bad shape");
  if (n_sel == 0) return 0;
  if (!Wt || !sel || !out) return fail("scd_gather_rows_bf16: null pointer");
  scd::gather_rows_bf16_kernel<<<n_sel, 128, 0, as_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(Wt),
                                                                    reinterpret_cast<const long long*>(sel), n_sel, D, V,
                                                                    reinterpret_cast<__nv_bfloat16*>(out));
  SCD_LAUNCH_CHECK("gather_rows_bf16_kernel");
  return 0;
}

size_t scd_name_topk_workspace_bytes(int64_t N, int64_t V, int k) {
  NamePlan pl;
  if (N <= 0 || V <= 0 || !plan_naming(N, V, k, &pl)) return 256;
  return pl.bytes;
}

int scd_name_topk_plan(int64_t N, int64_t V, int k, int32_t* out6) {
  NamePlan pl;
  if (!out6 || N <= 0 || V <= 0 || !plan_naming(N, V, k, &pl)) return fail("scd_name_topk_plan: bad arguments");
  const scd::NameWork w{pl.work_total, pl.tiles_total, pl.n_pairs};
  int most_items = 0;                       // work items the busiest pair starts
  for (int q = 0; q < pl.n_pairs; ++q) {
    int items = 0;
    for (int l = (int)w.bound(q), hi = (int)w.bound(q + 1); l < hi; ++items) l += scd::name_item_at(w, q, l, hi).nt;
    most_items = std::max(most_items, items);
  }
  int most_pieces = 0;                      // what the merge kernel derives per row block must agree with the slot count
  for (int rb = 0; rb < pl.n_row_blocks; ++rb) most_pieces = std::max(most_pieces, w.pieces(rb));
  if (most_pieces != pl.n_slots) return fail("scd_name_topk_plan: internal error, %d pieces vs %d slots", most_pieces, pl.n_slots);
  out6[0] = pl.n_row_blocks; out6[1] = pl.tiles_total; out6[2] = pl.n_pairs; out6[3] = pl.n_slots;
  out6[4] = (int)(pl.work_total / pl.n_pairs);          // tiles of the least loaded pair (the busiest has at most one more)
  out6[5] = most_items;
  return 0;
}

int scd_name_topk_plan_pair(int64_t N, int64_t V, int k, int pair, int32_t* out, int max_items) {
  NamePlan pl;
  if (N <= 0 || V <= 0 || !plan_naming(N, V, k, &pl) || pair < 0 || pair >= pl.n_pairs || (max_items > 0 && !out)) {
    fail("scd_name_topk_plan_pair: bad arguments");
    return -1;
  }
  const scd::NameWork w{pl.work_total, pl.tiles_total, pl.n_pairs};
  int items = 0;
  for (int l = (int)w.bound(pair), hi = (int)w.bound(pair + 1); l < hi; ++items) {
    const scd::NameItem it = scd::name_item_at(w, pair, l, hi);
    if (items < max_items) { out[4 * items] = it.rb; out[4 * items + 1] = it.t0; out[4 * items + 2] = it.nt; out[4 * items + 3] = it.part; }
    l += it.nt;
  }
  return items;
}

int scd_name_topk(const scd_bf16_t* X, int64_t N, int D, const scd_bf16_t* Wt, int64_t V, float scale, int k, int want_softmax,
                  int64_t idx_offset, float* vals, int64_t* idx, float* row_max, float* row_sumexp, void* ws, size_t ws_bytes,
                  scd_stream_t stream) {
  if (N < 0 || V <= 0 || D <= 0) return fail("scd_name_topk: bad shape N=%lld V=%lld D=%d", (long long)N, (long long)V, D);
  if (D > scd::kNameMaxD || D % 8 != 0) return fail("scd_name_topk: D=%d unsupported (need D <= %d and D %% 8 == 0)", D, scd::kNameMaxD);
  if (k < 1 || k > 8) return fail("scd_name_topk: k=%d unsupported (1..8)", k);
  if (V >= (1ll << 31) || N >= (1ll << 31)) return fail("scd_name_topk: N or V exceeds the int32 tile-coordinate range");
  if (!(scale > 0.f)) return fail("scd_name_topk: scale must be positive");
  if (N == 0) return 0;
  if (!X || !Wt || !vals || !idx || !ws) return fail("scd_name_topk: null pointer");
  if (((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(Wt)) & 15) != 0) return fail("scd_name_topk: X and Wt must be 16-byte aligned");
  NamePlan pl;
  if (!plan_naming(N, V, k, &pl)) return fail("scd_name_topk: planning failed");
  if (ws_bytes < pl.bytes) return fail("scd_name_topk: workspace too small (%zu < %zu)", ws_bytes, pl.bytes);
  cudaStream_t st = as_stream(stream);

  CUtensorMap mx, mw;
  if (int e = make_map_2d(&mx, X, (uint64_t)N, (uint64_t)D, scd::kBlockM, scd::kAKBlock, CU_TENSOR_MAP_SWIZZLE_128B)) return e;
  // vocabulary stages are 32-k halves of a k-block: 64-byte rows
  if (int e = make_map_2d(&mw, Wt, (uint64_t)V, (uint64_t)D, scd::kTileN / 2, scd::kBStageK, CU_TENSOR_MAP_SWIZZLE_64B)) return e;

  uint8_t* w8 = reinterpret_cast<uint8_t*>(ws);
  scd::NameParams p;
  p.n_rows = N;
  p.v_total = V;
  p.work_total = pl.work_total;
  p.tiles_total = pl.tiles_total;
  p.n_row_blocks = pl.n_row_blocks;
  p.num_kb = (D + scd::kAKBlock - 1) / scd::kAKBlock;
  p.want_softmax = (want_softmax || row_max || row_sumexp) ? 1 : 0;     // running max / sum-exp needed
  p.scale_log2e = scale * 1.4426950408889634f;
  p.part_val = reinterpret_cast<float*>(w8 + pl.off_val);
  p.part_idx = reinterpret_cast<int*>(w8 + pl.off_idx);
  p.part_max = reinterpret_cast<float*>(w8 + pl.off_max);
  p.part_sum = reinterpret_cast<float*>(w8 + pl.off_sum);
  p.scratch = reinterpret_cast<float*>(w8 + pl.off_scratch);
  p.prof = g_name_prof;
  p.x = reinterpret_cast<const __nv_bfloat16*>(X);
  p.d = D;
  int e = 0;
  if (pl.kt == 1) e = launch_name_topk<1>(mx, mw, p, pl.n_pairs, st);
  else if (pl.kt == 5) e = launch_name_topk<5>(mx, mw, p, pl.n_pairs, st);
  else e = launch_name_topk<8>(mx, mw, p, pl.n_pairs, st);
  if (e) return e;

  const bool stats = want_softmax || row_max || row_sumexp;
  launch_topk_merge<int, false>(pl.kt, k, N, st, p.part_val, p.part_idx, stats ? p.part_max : nullptr, stats ? p.part_sum : nullptr,
                                pl.n_slots * scd::kEpiHalves, N, pl.kt, k, scale, want_softmax ? 1 : 0, idx_offset, vals,
                                reinterpret_cast<long long*>(idx), row_max, row_sumexp,
                                scd::NameWork{pl.work_total, pl.tiles_total, pl.n_pairs});
  SCD_LAUNCH_CHECK("topk_merge_kernel");
  return 0;
}

int scd_topk_merge(const float* part_vals, const int64_t* part_idx, const float* part_max, const float* part_sum, int parts,
                   int64_t N, int k, float scale, int want_softmax, float* vals, int64_t* idx, scd_stream_t stream) {
  if (parts < 1 || N < 0 || k < 1 || k > 8) return fail("scd_topk_merge: bad arguments parts=%d N=%lld k=%d", parts, (long long)N, k);
  if (N == 0) return 0;
  if (!part_vals || !part_idx || !vals || !idx) return fail("scd_topk_merge: null pointer");
  if (want_softmax && (!part_max || !part_sum)) return fail("scd_topk_merge: softmax needs per-part row_max / row_sumexp");
  launch_topk_merge<long long, true>(list_len(k), k, N, as_stream(stream), part_vals, reinterpret_cast<const long long*>(part_idx),
                                     want_softmax ? part_max : nullptr, want_softmax ? part_sum : nullptr, parts, N, k, k, scale,
                                     want_softmax ? 1 : 0, 0, vals, reinterpret_cast<long long*>(idx), nullptr, nullptr,
                                     scd::NameWork{0, 1, 0});
  SCD_LAUNCH_CHECK("topk_merge_kernel<shards>");
  return 0;
}

// workspace layout (ints): counts[K] | the sort workspace (offsets[K+1] | cursor[K] | acc[K] | ticket | order[N])
size_t scd_vote_workspace_bytes(int64_t N, int K) {
  return align_up(((size_t)std::max(K, 0) + SortWs::ints(N, std::max(K, 0))) * sizeof(int), 256) + 256;
}

size_t scd_vote_spill_bytes(int64_t N, int k_used) { return scd::vote_spill_bytes(std::max<int64_t>(N, 0), std::max(k_used, 1)); }

int scd_vote(const int64_t* topk_idx, int k_total, int k_used, const int64_t* cluster_of_row, int64_t N, int K,
             const int64_t* excluded, int n_excluded, int M, int64_t* out_names, int32_t* out_counts, int32_t* out_distinct,
             int32_t* out_rows, int32_t* overflow, void* ws, size_t ws_bytes, void* spill, size_t spill_bytes, scd_stream_t stream) {
  if (int e = check_vote_args("scd_vote", N, K, k_total, k_used, M, excluded, n_excluded, out_names, out_counts, out_distinct,
                              overflow)) return e;
  if (!topk_idx || !cluster_of_row || !out_rows || !ws) return fail("scd_vote: null pointer");
  if (ws_bytes < scd_vote_workspace_bytes(N, K)) return fail("scd_vote: workspace too small");
  cudaStream_t st = as_stream(stream);
  int* counts = reinterpret_cast<int*>(ws);
  const SortWs w(counts + K, K);
  if (int e = sort_rows_by_label<long long>(reinterpret_cast<const long long*>(cluster_of_row), 1, N, K, out_rows, w, nullptr, 0, st)) return e;
  return launch_vote<long long>(reinterpret_cast<const long long*>(topk_idx), k_total, k_used, N, w.order, w.offsets, K, excluded, n_excluded,
                                M, out_names, out_counts, out_distinct, overflow, spill, spill_bytes, st);
}

int scd_vote_presorted(const int64_t* topk_idx, int k_total, int k_used, const void* mstep_ws, int64_t N, int K,
                       const int64_t* excluded, int n_excluded, int M, int64_t* out_names, int32_t* out_counts,
                       int32_t* out_distinct, int32_t* overflow, void* spill, size_t spill_bytes, scd_stream_t stream) {
  if (int e = check_vote_args("scd_vote_presorted", N, K, k_total, k_used, M, excluded, n_excluded, out_names, out_counts, out_distinct,
                              overflow)) return e;
  if (!topk_idx || !mstep_ws) return fail("scd_vote_presorted: null pointer");
  const SortWs w(const_cast<void*>(mstep_ws), K);         // as written by scd_mstep_sums
  return launch_vote<long long>(reinterpret_cast<const long long*>(topk_idx), k_total, k_used, N, w.order, w.offsets, K, excluded, n_excluded,
                                M, out_names, out_counts, out_distinct, overflow, spill, spill_bytes, as_stream(stream));
}

int scd_pack_vote_records(const int64_t* labels, const int64_t* topk_idx, int k_total, int k_used, int64_t n, int32_t* rec,
                          scd_stream_t stream) {
  if (n < 0 || k_total <= 0 || k_used <= 0 || k_used > k_total) return fail("scd_pack_vote_records: bad arguments");
  if (n == 0) return 0;
  if (!labels || !topk_idx || !rec) return fail("scd_pack_vote_records: null pointer");
  if (k_used > 8) return fail("scd_pack_vote_records: k_used=%d unsupported (<= 8)", k_used);
  const int blocks = (int)std::min<long long>((n + 255) / 256, device_sm_count() * 8);
  scd::pack_vote_records_kernel<<<blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(labels),
                                                                       reinterpret_cast<const long long*>(topk_idx), k_total, k_used, n, rec);
  SCD_LAUNCH_CHECK("pack_vote_records_kernel");
  return 0;
}

int scd_vote_records(const int32_t* rec, int k_used, int64_t N, int K, const int64_t* excluded, int n_excluded, int M,
                     int64_t* out_names, int32_t* out_counts, int32_t* out_distinct, int32_t* out_rows, int32_t* overflow,
                     void* ws, size_t ws_bytes, void* spill, size_t spill_bytes, scd_stream_t stream) {
  if (int e = check_vote_args("scd_vote_records", N, K, k_used, k_used, M, excluded, n_excluded, out_names, out_counts, out_distinct,
                              overflow)) return e;
  if (!rec || !out_rows || !ws) return fail("scd_vote_records: null pointer");
  if (ws_bytes < scd_vote_workspace_bytes(N, K)) return fail("scd_vote_records: workspace too small");
  cudaStream_t st = as_stream(stream);
  int* counts = reinterpret_cast<int*>(ws);
  const SortWs w(counts + K, K);
  const long long stride = 1 + k_used;
  if (int e = sort_rows_by_label<int>(rec, stride, N, K, out_rows, w, nullptr, 0, st)) return e;
  return launch_vote<int>(rec + 1, stride, k_used, N, w.order, w.offsets, K, excluded, n_excluded, M, out_names, out_counts, out_distinct,
                          overflow, spill, spill_bytes, st);
}

// ============================================================================ peer-memory exchange (SURVEY 8e)
size_t scd_peer_flag_bytes(void) { return sizeof(unsigned) * scd::kPeerFlagWords; }

size_t scd_peer_mstep_bytes(int K, int D) { return K > 0 && D > 0 ? sizeof(float) * scd::peer_mstep_words(K, D) : 0; }

int scd_peer_barrier(void* const* peer_flags, int world, int rank, int channel, scd_stream_t stream) {
  scd::PeerPtrs pp;
  if (channel < 0 || channel >= scd::kPeerChannels) return fail("scd_peer_barrier: bad channel %d", channel);
  if (int e = make_peer_ptrs(&pp, peer_flags, peer_flags, world, rank, "scd_peer_barrier")) return e;
  scd::peer_barrier_kernel<<<1, 32, 0, as_stream(stream)>>>(pp, channel);
  SCD_LAUNCH_CHECK("peer_barrier_kernel");
  return 0;
}

int scd_finalize_centers_peer(void* const* peer_bufs, void* const* peer_flags, int world, int rank, int channel,
                              size_t buf_byte_offset, const float* C_old, float* C_new, float* move_norms, float* counts_out,
                              double* inertia_out, int K, int D, void* estep_ws, size_t estep_ws_bytes, scd_stream_t stream) {
  if (K <= 0 || D <= 0) return fail("scd_finalize_centers_peer: bad shape");
  if (channel < 0 || channel >= scd::kPeerChannels) return fail("scd_finalize_centers_peer: bad channel %d", channel);
  if (!C_new || !peer_flags) return fail("scd_finalize_centers_peer: null pointer");
  if (buf_byte_offset % 16 != 0) return fail("scd_finalize_centers_peer: buffer offset must be a multiple of 16 bytes");
  if (move_norms && !C_old) return fail("scd_finalize_centers_peer: move norms need C_old");
  if (estep_ws && estep_ws_bytes < scd_estep_workspace_bytes(K, D)) return fail("scd_finalize_centers_peer: estep workspace too small");
  scd::PeerPtrs pp;
  if (int e = make_peer_ptrs(&pp, peer_bufs, peer_flags, world, rank, "scd_finalize_centers_peer")) return e;
  const EsWs es(estep_ws, K, D);
  scd::finalize_centers_peer_kernel<<<K, scd::kEsCentroidThreads, 0, as_stream(stream)>>>(
      pp, channel, buf_byte_offset / sizeof(float), C_old, C_new, move_norms, counts_out, inertia_out, K, D, es.chi, es.clo, es.cnorm);
  SCD_LAUNCH_CHECK("finalize_centers_peer_kernel");
  return 0;
}

int scd_pack_vote_records_peer(void* const* peer_bufs, int world, int rank, size_t buf_byte_offset, const int64_t* labels,
                               const int64_t* topk_idx, int k_total, int k_used, int64_t n, int64_t row_offset, scd_stream_t stream) {
  if (n < 0 || row_offset < 0 || k_total <= 0 || k_used <= 0 || k_used > k_total) return fail("scd_pack_vote_records_peer: bad arguments");
  if (buf_byte_offset % 4 != 0) return fail("scd_pack_vote_records_peer: buffer offset must be a multiple of 4 bytes");
  scd::PeerPtrs pp;
  if (int e = make_peer_ptrs(&pp, peer_bufs, nullptr, world, rank, "scd_pack_vote_records_peer")) return e;
  if (n == 0) return 0;
  if (!labels || !topk_idx) return fail("scd_pack_vote_records_peer: null pointer");
  if (k_used > 8) return fail("scd_pack_vote_records_peer: k_used=%d unsupported (<= 8)", k_used);
  const int blocks = (int)std::min<long long>((n + scd::kPackRows - 1) / scd::kPackRows, device_sm_count() * 8);
  scd::pack_vote_records_peer_kernel<<<blocks, 256, 0, as_stream(stream)>>>(pp, buf_byte_offset, reinterpret_cast<const long long*>(labels),
                                                                            reinterpret_cast<const long long*>(topk_idx), k_total, k_used, n, row_offset);
  SCD_LAUNCH_CHECK("pack_vote_records_peer_kernel");
  return 0;
}

int scd_pack_sorted_records_peer(void* const* peer_bufs, int world, int rank, size_t rec_byte_offset, size_t off_byte_offset,
                                 const int64_t* topk_idx, int k_total, int k_used, int64_t n, int64_t row_offset, const void* mstep_ws,
                                 int K, scd_stream_t stream) {
  if (n < 0 || row_offset < 0 || k_total <= 0 || k_used <= 0 || k_used > k_total || k_used > 8 || K <= 0)
    return fail("scd_pack_sorted_records_peer: bad arguments");
  if (rec_byte_offset % 4 != 0 || off_byte_offset % 4 != 0) return fail("scd_pack_sorted_records_peer: offsets must be multiples of 4 bytes");
  if (!mstep_ws || (n > 0 && !topk_idx)) return fail("scd_pack_sorted_records_peer: null pointer");
  scd::PeerPtrs pp;
  if (int e = make_peer_ptrs(&pp, peer_bufs, nullptr, world, rank, "scd_pack_sorted_records_peer")) return e;
  const SortWs w(const_cast<void*>(mstep_ws), K);           // as written by scd_mstep_sums on this rank's labels
  const int blocks = (int)std::max<long long>(1, std::min<long long>((n + scd::kPackRows - 1) / scd::kPackRows, device_sm_count() * 8));
  scd::pack_sorted_records_peer_kernel<<<blocks, 256, 0, as_stream(stream)>>>(pp, rec_byte_offset, off_byte_offset,
      reinterpret_cast<const long long*>(topk_idx), k_total, k_used, n, row_offset, w.order, w.offsets, K);
  SCD_LAUNCH_CHECK("pack_sorted_records_peer_kernel");
  return 0;
}

int scd_vote_segments(const int32_t* rec, int k_used, int64_t n_total, int64_t per, int world, const int32_t* seg_offsets, int K,
                      const int64_t* excluded, int n_excluded, int M, int64_t* out_names, int32_t* out_counts,
                      int32_t* out_distinct, int32_t* out_rows, int32_t* overflow, void* spill, size_t spill_bytes,
                      scd_stream_t stream) {
  if (per < 0 || world < 1 || world > scd::kVoteMaxSeg || n_total > per * world) return fail("scd_vote_segments: bad arguments");
  if (int e = check_vote_args("scd_vote_segments", n_total, K, k_used, k_used, M, excluded, n_excluded, out_names, out_counts,
                              out_distinct, overflow)) return e;
  if (!rec || !seg_offsets || !out_rows) return fail("scd_vote_segments: null pointer");
  return launch_vote<int, true>(rec, 1 + k_used, k_used, n_total, nullptr, nullptr, K, excluded, n_excluded, M, out_names, out_counts,
                                out_distinct, overflow, spill, spill_bytes, as_stream(stream), seg_offsets, world, per, out_rows);
}

int scd_contingency(const void* y_pred, int pred_is_f64, const void* y_true, int true_is_f64, int64_t N, int D,
                    const uint8_t* mask, int64_t* w, int64_t* first_row, int64_t* col_masked, int32_t* bad, scd_stream_t stream) {
  if (N < 0 || D <= 0 || D > 46340) return fail("scd_contingency: bad shape N=%lld D=%d", (long long)N, D);
  if (!w || !bad || (N > 0 && (!y_pred || !y_true)) || (mask && !col_masked)) return fail("scd_contingency: null pointer");
  cudaStream_t st = as_stream(stream);
  const long long cells = (long long)D * D;
  SCD_CUDA(cudaMemsetAsync(w, 0, sizeof(int64_t) * (size_t)cells, st));
  if (col_masked) SCD_CUDA(cudaMemsetAsync(col_masked, 0, sizeof(int64_t) * (size_t)D, st));
  if (first_row) {
    scd::fill_u64_kernel<<<(D + 255) / 256, 256, 0, st>>>(reinterpret_cast<unsigned long long*>(first_row), D, (unsigned long long)N);
    SCD_LAUNCH_CHECK("fill_u64_kernel");
  }
  if (N == 0) return 0;
  const int use_smem = cells <= scd::kContSmemCells ? 1 : 0;
  const size_t smem = use_smem ? sizeof(int) * (size_t)cells : 0;
  const int blocks = (int)std::min<long long>((N + 255) / 256, (long long)device_sm_count() * (use_smem ? 2 : 8));
  auto* wp = reinterpret_cast<unsigned long long*>(w);
  auto* fp = reinterpret_cast<unsigned long long*>(first_row);
  auto* cm = reinterpret_cast<unsigned long long*>(col_masked);
  if (!pred_is_f64 && !true_is_f64)
    scd::contingency_kernel<long long, long long><<<blocks, 256, smem, st>>>(static_cast<const long long*>(y_pred), static_cast<const long long*>(y_true), N, D, mask, wp, fp, cm, bad, use_smem);
  else if (!pred_is_f64 && true_is_f64)
    scd::contingency_kernel<long long, double><<<blocks, 256, smem, st>>>(static_cast<const long long*>(y_pred), static_cast<const double*>(y_true), N, D, mask, wp, fp, cm, bad, use_smem);
  else if (pred_is_f64 && !true_is_f64)
    scd::contingency_kernel<double, long long><<<blocks, 256, smem, st>>>(static_cast<const double*>(y_pred), static_cast<const long long*>(y_true), N, D, mask, wp, fp, cm, bad, use_smem);
  else
    scd::contingency_kernel<double, double><<<blocks, 256, smem, st>>>(static_cast<const double*>(y_pred), static_cast<const double*>(y_true), N, D, mask, wp, fp, cm, bad, use_smem);
  SCD_LAUNCH_CHECK("contingency_kernel");
  return 0;
}

}  // extern "C"

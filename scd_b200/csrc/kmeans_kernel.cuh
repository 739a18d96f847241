// k-means E-step / M-step kernels (SURVEY 8a rows a1-a4), fp32.
//
//   a1  pairwise_distance  local_utils/faster_mix_k_means_pytorch.py:177-212   dis[n,k] = sum_d (x-c)^2  (direct form)
//   a2  E-step             :58-60 / :105-111    row min + argmin (ties -> lowest index, NaN wins) + inertia
//   a3  M-step             :61-64 / :113-116    centers[j] = mean(X[labels == j]);  empty cluster -> NaN row
//   a4  convergence        :71 / :123           shift = sum_k || c_k - c_k_old ||_2
//
// Layout in HBM: X [N, D] fp32 row-major, centroids [K, D] fp32 row-major, labels [N] int64 (the
// reference's dtype), per-cluster sums [K, D] fp32 + counts [K] int32 (split from the divide so an
// NCCL all-reduce can sit between when rows are sharded across GPUs).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <math.h>
#include "estep_tc_kernel.cuh"

namespace scd {

// --------------------------------------------------------------------------------------------
// Direct-form squared distance tile kernel.  Block = 256 threads, 128 rows x 64 centroids per
// tile step, 16-wide d-chunks staged through shared memory (transposed, so the inner loop reads
// float4 along rows / centroids), 8 x 4 accumulators per thread.
//   FUSED = false : write the full [N, K] matrix (the pairwise_distance() drop-in; optional
//                   int32 cost matrix round(1000 * sqrt(d)) for the size-constrained variant,
//                   local_utils/sskm_constrained.py:116 + :324)
//   FUSED = true  : keep a running (min, argmin) per row over all centroid tiles, write labels /
//                   mindist and add the block's inertia (fp64) - the [N, K] matrix never exists.
// --------------------------------------------------------------------------------------------
constexpr int kDistBM = 128, kDistBN = 64, kDistBK = 16, kDistThreads = 256;

__device__ __forceinline__ bool dist_better(float cand, float cur) {
  // torch.min semantics: strict '<' keeps the lowest index among ties; a NaN beats any number.
  return (cand < cur) || (cand != cand && cur == cur);
}

template <bool FUSED>
__global__ void __launch_bounds__(kDistThreads)
sqdist_kernel(const float* __restrict__ X, long long N, int D, const float* __restrict__ C, int K,
              float* __restrict__ out, int* __restrict__ cost_x1000,
              long long* __restrict__ labels, float* __restrict__ mindist, double* __restrict__ inertia) {
  __shared__ __align__(16) float Xs[kDistBK][kDistBM + 4];
  __shared__ __align__(16) float Cs[kDistBK][kDistBN + 4];
  __shared__ float red_val[kDistBM][17];
  __shared__ int red_idx[kDistBM][17];

  const int tid = threadIdx.x;
  const int tr = tid >> 4;          // 0..15 -> rows tr*8 .. tr*8+7
  const int tc = tid & 15;          // 0..15 -> cols tc*4 .. tc*4+3
  const long long row0 = (long long)blockIdx.x * kDistBM;

  float best[8];
  int best_k[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { best[i] = INFINITY; best_k[i] = 0; }
  bool have[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) have[i] = false;

  const int kt_begin = FUSED ? 0 : blockIdx.y;
  const int kt_end = FUSED ? (K + kDistBN - 1) / kDistBN : blockIdx.y + 1;

  for (int kt = kt_begin; kt < kt_end; ++kt) {
    const int col0 = kt * kDistBN;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int d0 = 0; d0 < D; d0 += kDistBK) {
      // stage X tile: 128 rows x 16 d  (2048 floats, 8 per thread), coalesced along d
      {
        const int r = tid >> 1;              // 0..127
        const int dd = (tid & 1) * 8;        // 0 or 8
        const long long gr = row0 + r;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int d = d0 + dd + q;
          Xs[dd + q][r] = (gr < N && d < D) ? X[gr * D + d] : 0.f;
        }
      }
      // stage C tile: 64 centroids x 16 d (1024 floats, 4 per thread)
      {
        const int c = tid >> 2;              // 0..63
        const int dd = (tid & 3) * 4;
        const int gc = col0 + c;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int d = d0 + dd + q;
          Cs[dd + q][c] = (gc < K && d < D) ? C[(long long)gc * D + d] : 0.f;
        }
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < kDistBK; ++kk) {
        const float4 xa = *reinterpret_cast<const float4*>(&Xs[kk][tr * 8]);
        const float4 xb = *reinterpret_cast<const float4*>(&Xs[kk][tr * 8 + 4]);
        const float4 cv = *reinterpret_cast<const float4*>(&Cs[kk][tc * 4]);
        const float xr[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
        const float cr[4] = {cv.x, cv.y, cv.z, cv.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float diff = xr[i] - cr[j];
            acc[i][j] = fmaf(diff, diff, acc[i][j]);
          }
      }
      __syncthreads();
    }

    if constexpr (!FUSED) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long gr = row0 + tr * 8 + i;
        if (gr >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int gc = col0 + tc * 4 + j;
          if (gc < K) {
            if (out) out[gr * K + gc] = acc[i][j];
            if (cost_x1000) {
              // sskm_constrained.py:324: np.around(costs * 1000).astype(int32) on the float64 promotion of the fp32
              // sqrt - the product is rounded in fp64 (an fp32 product can cross a .5 boundary); NaN (distance to an
              // empty cluster's NaN centroid) becomes INT_MIN like NumPy's cast on x86
              const float r = sqrtf(acc[i][j]);
              cost_x1000[gr * K + gc] = r != r ? (int)0x80000000 : __double2int_rn((double)r * 1000.0);
            }
          }
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int gc = col0 + tc * 4 + j;
          if (gc < K && (!have[i] || dist_better(acc[i][j], best[i]))) { best[i] = acc[i][j]; best_k[i] = gc; have[i] = true; }
        }
    }
  }

  if constexpr (FUSED) {
    // reduce the 16 column-group candidates of each row (ascending centroid index inside a thread
    // and across tc, so scanning tc upward with the same predicate keeps torch.min's tie rule)
#pragma unroll
    for (int i = 0; i < 8; ++i) { red_val[tr * 8 + i][tc] = best[i]; red_idx[tr * 8 + i][tc] = have[i] ? best_k[i] : -1; }
    __syncthreads();
    double local = 0.0;
    if (tid < kDistBM) {
      const long long gr = row0 + tid;
      float bv = 0.f; int bk = -1;
      for (int c = 0; c < 16; ++c) {
        const int k = red_idx[tid][c];
        if (k < 0) continue;
        const float v = red_val[tid][c];
        // candidates are not globally index-ordered across tc (each thread saw every tile), so
        // compare on (value, index) explicitly
        if (bk < 0 || dist_better(v, bv) || (v == bv && k < bk) || (v != v && bv != bv && k < bk)) { bv = v; bk = k; }
      }
      if (gr < N) {
        labels[gr] = bk;
        if (mindist) mindist[gr] = bv;
        local = (double)bv;
      }
    }
    // block inertia: warp shuffle then one fp64 atomic per warp
    for (int off = 16; off > 0; off >>= 1) local += __shfl_down_sync(0xffffffffu, local, off);
    if ((tid & 31) == 0 && tid < kDistBM && inertia) atomicAdd(inertia, local);
  }
}

// --------------------------------------------------------------------------------------------
// M-step, part 1: counting sort of row ids by label, two launches.
//   label_hist_scan_kernel  per-block shared-memory histogram -> global accumulator; the LAST block to finish (ticket)
//                           turns the accumulated counts into counts_out / offsets / cursor (exclusive scan) and
//                           leaves accumulator and ticket zeroed for the next call.  Also zeroes `zero_me` (the
//                           [K, D] sums the segment sum accumulates into) so no separate memset node is needed.
//   label_scatter_kernel    a block ranks its 1024 rows per label in shared memory and reserves ONE range per
//                           (block, label) in the global cursor: N / 1024 * min(K, 1024) global atomics instead of N
//                           (round 1: 29 us for 127 k rows on 100 cursors, the contended L2 atomics serialise).
// Labels are read through (pointer, element stride): int64 label vectors (stride 1) or the label column of the
// packed int32 vote records [N][1 + k] of the multi-GPU path.  Labels outside [0, K) (e.g. the reference's -1
// "unassigned") are ignored.  The order of the rows inside a cluster is not deterministic (atomics); the vote does
// not depend on it (first positions are row ids), the fp32 segment sums do in their last bits (DESIGN 4).
// --------------------------------------------------------------------------------------------
// plain label histogram (scd_label_histogram: the size check of the constrained E-step)
__global__ void label_hist_kernel(const long long* __restrict__ labels, long long N, int K, int* __restrict__ counts) {
  extern __shared__ int sh_hist[];
  for (int k = threadIdx.x; k < K; k += blockDim.x) sh_hist[k] = 0;
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
    const long long l = labels[i];
    if (l >= 0 && l < K) atomicAdd(&sh_hist[(int)l], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) if (sh_hist[k]) atomicAdd(&counts[k], sh_hist[k]);
}

constexpr int kSortThreads = 256;
constexpr int kScatterRowsPerThread = 4;
constexpr int kScatterRows = kSortThreads * kScatterRowsPerThread;      // rows per block of the scatter

template <typename LabT>
__global__ void __launch_bounds__(kSortThreads)
label_hist_scan_kernel(const LabT* __restrict__ labels, long long stride, long long N, int K, int* __restrict__ acc /* [K] zero on entry */,
                       unsigned* __restrict__ ticket /* zero on entry */, int* __restrict__ counts_out /* nullable */,
                       int* __restrict__ offsets, int* __restrict__ cursor, float4* __restrict__ zero_me, long long n_zero4) {
  extern __shared__ int sh_hist[];
  __shared__ bool is_last;
  __shared__ int sh_part[kSortThreads];
  for (int k = threadIdx.x; k < K; k += blockDim.x) sh_hist[k] = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_zero4; i += (long long)gridDim.x * blockDim.x)
    zero_me[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
    const long long l = (long long)labels[i * stride];
    if (l >= 0 && l < K) atomicAdd(&sh_hist[(int)l], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) if (sh_hist[k]) atomicAdd(&acc[k], sh_hist[k]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // exclusive scan over K counts: thread t owns the contiguous slice [t * per, (t + 1) * per)
  const int per = (K + kSortThreads - 1) / kSortThreads;
  const int k0 = min(threadIdx.x * per, K), k1 = min(k0 + per, K);
  int local = 0;
  for (int k = k0; k < k1; ++k) local += __ldcg(&acc[k]);
  sh_part[threadIdx.x] = local;
  __syncthreads();
  for (int off = 1; off < kSortThreads; off <<= 1) {
    const int t = (int)threadIdx.x >= off ? sh_part[threadIdx.x - off] : 0;
    __syncthreads();
    sh_part[threadIdx.x] += t;
    __syncthreads();
  }
  int run = sh_part[threadIdx.x] - local;
  for (int k = k0; k < k1; ++k) {
    const int c = __ldcg(&acc[k]);
    offsets[k] = run; cursor[k] = run;
    if (counts_out) counts_out[k] = c;
    acc[k] = 0;
    run += c;
  }
  if (threadIdx.x == kSortThreads - 1) { offsets[K] = sh_part[kSortThreads - 1]; *ticket = 0u; }
}

template <typename LabT>
__global__ void __launch_bounds__(kSortThreads)
label_scatter_kernel(const LabT* __restrict__ labels, long long stride, long long N, int K, int* __restrict__ cursor,
                     int* __restrict__ order) {
  extern __shared__ int sh_cnt[];          // [K] rows of this block per label, then the block's base per label
  for (int k = threadIdx.x; k < K; k += blockDim.x) sh_cnt[k] = 0;
  __syncthreads();
  const long long row0 = (long long)blockIdx.x * kScatterRows;
  int lab[kScatterRowsPerThread], rank[kScatterRowsPerThread];
#pragma unroll
  for (int q = 0; q < kScatterRowsPerThread; ++q) {
    const long long i = row0 + q * kSortThreads + threadIdx.x;
    lab[q] = -1;
    if (i < N) {
      const long long l = (long long)labels[i * stride];
      if (l >= 0 && l < K) { lab[q] = (int)l; rank[q] = atomicAdd(&sh_cnt[(int)l], 1); }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const int c = sh_cnt[k];
    if (c) sh_cnt[k] = atomicAdd(&cursor[k], c);
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kScatterRowsPerThread; ++q)
    if (lab[q] >= 0) order[sh_cnt[lab[q]] + rank[q]] = (int)(row0 + q * kSortThreads + threadIdx.x);
}

// --------------------------------------------------------------------------------------------
// M-step, part 2: segmented sum over the label-sorted row order.  One warp owns kSegRows
// consecutive sorted positions; lane l keeps D/128 float4 accumulators (columns j*128 + 4l..4l+3,
// so every row read is one coalesced 512 B request per j); when the cluster id changes, or at the
// end of the chunk, the warp flushes with vector reductions (red.global.add.v4.f32) into sums[k].
// Atomics per (cluster, column) ~ rows_in_cluster / kSegRows instead of rows_in_cluster.
// --------------------------------------------------------------------------------------------
constexpr int kSegRows = 32;       // one row id per lane: the chunk's order[] entries arrive in one coalesced load
constexpr int kSegMaxVec = 8;      // supports D <= 1024 (D % 4 == 0)

__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <int NV>     // register capacity in float4 per lane (NV * 128 >= D rounded down to 128); 2 / 4 / 6 / 8
__global__ void __launch_bounds__(256)
segment_sum_kernel(const float* __restrict__ X, const int* __restrict__ order, const int* __restrict__ offsets,
                   int K, int D, float* __restrict__ sums) {
  const int total = offsets[K];
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int p0 = warp_global * kSegRows;
  if (p0 >= total) return;
  const int p1 = min(p0 + kSegRows, total);
  const int nvec = D >> 7;                       // float4 per lane for the 128-column-aligned part
  const int tail = D - (nvec << 7);              // < 128 remaining columns (multiple of 4)
  const int my_row = (p0 + lane < p1) ? order[p0 + lane] : 0;
  // cluster of the first position: binary search in offsets
  int lo = 0, hi = K;
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (offsets[mid] <= p0) lo = mid; else hi = mid; }
  int k = lo;
  while (k < K - 1 && offsets[k + 1] <= p0) ++k;   // skip empty clusters
  float4 acc[NV], cur[NV], nxt[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 acc_tail = make_float4(0.f, 0.f, 0.f, 0.f), cur_tail = acc_tail, nxt_tail = acc_tail;
  const bool tail_lane = (lane * 4) < tail;

  auto flush = [&](int kk) {
    float* dst = sums + (long long)kk * D;
#pragma unroll
    for (int j = 0; j < NV; ++j)
      if (j < nvec) { red_add_v4(dst + j * 128 + lane * 4, acc[j]); acc[j] = make_float4(0.f, 0.f, 0.f, 0.f); }
    if (tail_lane) { red_add_v4(dst + nvec * 128 + lane * 4, acc_tail); acc_tail = make_float4(0.f, 0.f, 0.f, 0.f); }
  };
  auto load_row = [&](int p, float4 (&dst)[NV], float4& dst_tail) {
    const float* src = X + (long long)__shfl_sync(0xffffffffu, my_row, p - p0) * D;
#pragma unroll
    for (int j = 0; j < NV; ++j)
      if (j < nvec) dst[j] = __ldg(reinterpret_cast<const float4*>(src + j * 128 + lane * 4));
    if (tail_lane) dst_tail = __ldg(reinterpret_cast<const float4*>(src + nvec * 128 + lane * 4));
  };

  int seg_end = offsets[k + 1];
  load_row(p0, cur, cur_tail);
  for (int p = p0; p < p1; ++p) {
    if (p + 1 < p1) load_row(p + 1, nxt, nxt_tail);          // next row in flight while this one is added
    while (p >= seg_end) { flush(k); ++k; seg_end = offsets[k + 1]; }
#pragma unroll
    for (int j = 0; j < NV; ++j)
      if (j < nvec) { acc[j].x += cur[j].x; acc[j].y += cur[j].y; acc[j].z += cur[j].z; acc[j].w += cur[j].w; cur[j] = nxt[j]; }
    if (tail_lane) { acc_tail.x += cur_tail.x; acc_tail.y += cur_tail.y; acc_tail.z += cur_tail.z; acc_tail.w += cur_tail.w; cur_tail = nxt_tail; }
  }
  flush(k);
}

// Shape-generic variant (any D, any alignment): one thread per (cluster, column), fixed summation order.
// Used when D is not a multiple of 4 or X is not 16-byte aligned (e.g. the reference's 2-D blobs demo).
__global__ void segment_sum_generic_kernel(const float* __restrict__ X, const int* __restrict__ order,
                                           const int* __restrict__ offsets, int K, int D, float* __restrict__ sums) {
  const int k = blockIdx.x;
  const int d = blockIdx.y * blockDim.x + threadIdx.x;
  if (d >= D) return;
  float acc = 0.f;
  for (int p = offsets[k]; p < offsets[k + 1]; ++p) acc += X[(long long)order[p] * D + d];
  sums[(long long)k * D + d] = acc;
}

// centers = sums / counts (0/0 -> NaN, as torch's mean over zero rows), per-cluster move norm; optionally also the
// next E-step's operands of the new centres (estep_tc_kernel.cuh), so the iteration loop needs no split launch.
__global__ void finalize_centers_kernel(const float* __restrict__ sums, const float* __restrict__ counts_f, const int* __restrict__ counts_i,
                                        const float* __restrict__ c_old, float* __restrict__ c_new, float* __restrict__ move_norm,
                                        int K, int D, __nv_bfloat16* __restrict__ plane_hi, __nv_bfloat16* __restrict__ plane_lo,
                                        float* __restrict__ cnorm) {
  const int k = blockIdx.x;
  const float cnt = counts_i ? (float)counts_i[k] : counts_f[k];
  float part = 0.f, npart = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float c = sums[(long long)k * D + d] / cnt;
    c_new[(long long)k * D + d] = c;
    if (c_old) { const float df = c - c_old[(long long)k * D + d]; part += df * df; }
    if (plane_hi) {
      es_store_split(c, plane_hi, plane_lo, (long long)k * D + d);
      npart = fmaf(c, c, npart);
    }
  }
  block_sum_to_thread0(part, npart);
  if (threadIdx.x == 0) {
    if (move_norm) move_norm[k] = sqrtf(part);
    if (cnorm) cnorm[k] = npart;
  }
}

// tail of the packed all-reduce buffer [K*D sums | K counts | inertia], all fp32 (counts < 2^24 are exact)
__global__ void pack_counts_inertia_kernel(const int* __restrict__ counts, const double* __restrict__ inertia, int K,
                                           float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K) out[i] = (float)counts[i];
  else if (i == K) out[K] = inertia ? (float)*inertia : 0.f;
}

// shift = sum_k move_norm[k], one block, fixed order (deterministic)
__global__ void sum_small_kernel(const float* __restrict__ v, int n, float* __restrict__ out) {
  __shared__ float sh[1024];
  float t = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) t += v[i];
  sh[threadIdx.x] = t;
  __syncthreads();
  for (int off = blockDim.x >> 1; off > 0; off >>= 1) {
    if (threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = sh[0];
}

// a4 labelled inertia, ref :108-109: sum_i || L_i - C[label_i] ||^2  (one warp per row, fp64 atomic per block)
__global__ void __launch_bounds__(256)
gather_sqdist_kernel(const float* __restrict__ L, const long long* __restrict__ labels, long long n, int D,
                     const float* __restrict__ C, int K, double* __restrict__ acc) {
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  float part = 0.f;
  if (row < n) {
    const long long l = labels[row];
    if (l >= 0 && l < K) {
      for (int d = lane; d < D; d += 32) { const float df = L[row * D + d] - C[l * D + d]; part = fmaf(df, df, part); }
    }
  }
  for (int off = 16; off > 0; off >>= 1) part += __shfl_down_sync(0xffffffffu, part, off);
  __shared__ double sh[8];
  if (lane == 0) sh[threadIdx.x >> 5] = (double)part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[w];
    atomicAdd(acc, t);
  }
}

// --------------------------------------------------------------------------------------------
// a5 k-means++ seeding, faster_mix_k_means_pytorch.py:20-36 (gcd copy :82-110).  The reference recomputes the full
// N x c distance matrix for every added centre; here a running min-distance vector d2[N] is updated against the newest
// centre only (kpp_update_kernel: one pass over X per centre, block sums of d2 in fp64) and the draw is resolved on the
// device (kpp_select_kernel): prob = d2 / sum(d2), first index with cumsum(prob) >= r  <=>  first index whose prefix
// sum of d2 reaches r * sum(d2) (fp64 prefix sums; the reference's fp32 cumsum is only accurate to a few rows' worth of
// probability mass at N ~ 1e5, so the picked row can differ within that margin - DESIGN 4).  The picked row index
// never visits the host: the next update reads it from device memory.
// --------------------------------------------------------------------------------------------
constexpr int kKppRowsPerBlock = 64;     // 8 warps x 8 rows

// d2[i] = min(d2[i], ||X_i - c||^2) with c = `center` when given (row-sharded seeding: the picked row lives on another
// rank and arrives by broadcast), else X[*pick]  (first == 1: no min, plain assignment);  also centers_out[:] = c.
// *pick < 0 (no candidate was found by the select step) leaves d2 untouched and only refreshes the block sums.
__global__ void __launch_bounds__(256)
kpp_update_kernel(const float* __restrict__ X, long long N, int D, const long long* __restrict__ pick, const float* __restrict__ center,
                  int first, float* __restrict__ d2, double* __restrict__ block_sums, float* __restrict__ center_out) {
  const long long src = center ? 0 : *pick;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* c = center ? center : X + (src >= 0 ? src : 0) * D;
  if (blockIdx.x == 0 && center_out && src >= 0)
    for (int d = threadIdx.x; d < D; d += blockDim.x) center_out[d] = c[d];
  double local = 0.0;
  for (int r = 0; r < kKppRowsPerBlock / 8; ++r) {
    const long long row = (long long)blockIdx.x * kKppRowsPerBlock + warp * (kKppRowsPerBlock / 8) + r;
    if (row >= N) break;
    float part = 0.f;
    if (src >= 0) {
      const float* x = X + row * D;
      for (int d = lane; d < D; d += 32) { const float df = x[d] - c[d]; part = fmaf(df, df, part); }
      for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    }
    if (lane == 0) {
      float v = d2[row];
      if (src >= 0) { v = first ? part : fminf(v, part); d2[row] = v; }
      local += (double)v;
    }
  }
  __shared__ double sh[8];
  if (lane == 0) sh[warp] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[w];
    block_sums[blockIdx.x] = t;
  }
}

// block sums of an existing d2 vector (seeding from several pre-centres: d2 comes from the E-step's mindist)
__global__ void __launch_bounds__(256)
kpp_block_sums_kernel(const float* __restrict__ d2, long long N, double* __restrict__ block_sums) {
  const long long base = (long long)blockIdx.x * kKppRowsPerBlock;
  double v = 0.0;
  if (threadIdx.x < kKppRowsPerBlock && base + threadIdx.x < N) v = (double)d2[base + threadIdx.x];
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  __shared__ double sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) block_sums[blockIdx.x] = sh[0] + sh[1];
}

// one block: total = sum(block_sums); target = r * total; first row whose inclusive prefix sum of d2 >= target.
// *pick is left unchanged when no row qualifies (r beyond the last cumulative value, or total is 0 / NaN) and
// *no_hit gets bit 0 (sticky; bit 1 as well when there is no previous pick to fall back on) - the gcd copy reuses the previous index (:104-107), the local copy raises IndexError (:34).
__global__ void __launch_bounds__(1024)
kpp_select_kernel(const float* __restrict__ d2, long long N, const double* __restrict__ block_sums, int n_blocks, double r,
                  long long* __restrict__ pick, int* __restrict__ no_hit) {
  __shared__ double sh[1024];
  __shared__ double s_total;
  __shared__ int s_block;
  __shared__ double s_before;
  // total, in a fixed order
  double t = 0.0;
  for (int b = threadIdx.x; b < n_blocks; b += blockDim.x) t += block_sums[b];
  sh[threadIdx.x] = t;
  __syncthreads();
  for (int off = 512; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) { s_total = sh[0]; s_block = -1; s_before = 0.0; }
  __syncthreads();
  const double total = s_total;
  const double target = r * total;
  if (!(total > 0.0)) {                       // 0 / 0 probabilities are NaN in the reference: nothing compares >= r
    if (threadIdx.x == 0) atomicOr(no_hit, 1 | (*pick < 0 ? 2 : 0));
    return;
  }
  // first block whose inclusive prefix reaches the target: thread 0 walks the (few thousand) block sums
  if (threadIdx.x == 0) {
    double run = 0.0;
    for (int b = 0; b < n_blocks; ++b) {
      const double nxt = run + block_sums[b];
      if (nxt >= target) { s_block = b; s_before = run; break; }
      run = nxt;
    }
  }
  __syncthreads();
  if (s_block < 0) {
    if (threadIdx.x == 0) atomicOr(no_hit, 1 | (*pick < 0 ? 2 : 0));
    return;
  }
  if (threadIdx.x == 0) {
    const long long base = (long long)s_block * kKppRowsPerBlock;
    double run = s_before;
    long long found = -1;
    for (int i = 0; i < kKppRowsPerBlock && base + i < N; ++i) {
      run += (double)d2[base + i];
      if (run >= target) { found = base + i; break; }
    }
    if (found < 0) found = min(base + kKppRowsPerBlock, N) - 1;      // rounding between the two summation orders
    *pick = found;
  }
}

}  // namespace scd

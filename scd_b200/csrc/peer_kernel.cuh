// Exchange steps of the sharded path over NVLink peer memory (SURVEY 8e), fused with the kernels that follow them.
//
// One process per GPU; every rank maps the others' exchange buffers into its own address space (torch symmetric
// memory: cuMem allocations exported / imported once per fit, scd_b200/peer.py).  Two exchanges exist on the path:
//
//   * k-means M-step (faster_mix_k_means_pytorch.py:61-64 over sharded rows): every rank's segment sum leaves
//     [K*D sums | K counts | inertia] in ITS buffer; finalize_centers_peer_kernel is the all-reduce AND the divide: after
//     a flag barrier it reads the G buffers with peer loads, adds them in rank order (bitwise the same centres on every
//     rank) and writes centres, move norms and the next E-step's operands.  No pack kernel, no NCCL launch, no second
//     pass over the reduced buffer.
//   * vote (main_unsup.py:575-577 over sharded rows): pack_vote_records_peer_kernel stores the rank's
//     [label, name_0 .. name_(k-1)] int32 records straight into every rank's gathered array (the all-gather is the
//     store); peer_barrier_kernel orders it against the vote.
//
// Flags: each rank owns a pad of 32-bit words, written remotely by its peers.  Channel c:
//     arrive[c][r]  (r = 0 .. G-1)   epoch rank r has reached on channel c   (written by rank r, read locally)
//     epoch[c], ticket[c]            local bookkeeping (only this rank touches them)
// A barrier = store (my epoch + 1) into arrive[c][me] of every peer, then wait until all G local arrive words have
// reached it.  Epochs live on the device, so a captured CUDA graph replays correctly.  Every wait is bounded by wall
// clock and traps with a message instead of hanging the GPU (a rank that died, or ranks launching different sequences).
#pragma once
#include "ptx.cuh"
#include "estep_tc_kernel.cuh"
#include <cuda_bf16.h>

namespace scd {

constexpr int kPeerMaxWorld = 16;
constexpr int kPeerChannels = 8;
constexpr int kPeerChannelWords = 32;            // arrive[16] | epoch | ticket | pad
constexpr int kPeerFlagWords = kPeerChannels * kPeerChannelWords;

struct PeerPtrs {                                 // by value in the kernel parameters
  void* buf[kPeerMaxWorld];                       // rank r's exchange buffer, mapped here
  unsigned* flags[kPeerMaxWorld];                 // rank r's flag pad, mapped here
  int world, rank;
};

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer_f4(const float* p) {       // never served from a stale L1 line
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_peer_f1(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_peer_i1(const int* p) {
  int v;
  asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double ld_peer_d1(const double* p) {
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

__device__ __noinline__ void peer_timeout_trap(int channel, int from_rank, unsigned have, unsigned want) {
  printf("[scd_b200] peer barrier timed out: block %d channel %d waiting for rank %d (flag %u, want %u)\n", (int)blockIdx.x,
         channel, from_rank, have, want);
  __trap();
}

// the epoch this launch has to reach on `channel` (every block of the launch reads the same value: it only moves when the
// launch's last block calls peer_finish)
__device__ __forceinline__ unsigned peer_target(const PeerPtrs& pp, int channel) {
  return *reinterpret_cast<volatile unsigned*>(pp.flags[pp.rank] + channel * kPeerChannelWords + kPeerMaxWorld) + 1u;
}
// threads [0, world) of ONE block of the launch: everything this rank wrote before (earlier kernels of the stream, or this
// block after a __syncthreads) becomes visible to a peer that sees the flag
__device__ __forceinline__ void peer_signal(const PeerPtrs& pp, int channel, unsigned target) {
  if ((int)threadIdx.x < pp.world) {
    __threadfence_system();
    st_release_sys(pp.flags[threadIdx.x] + channel * kPeerChannelWords + pp.rank, target);
  }
}
// threads [0, world) of every block that is going to read peer data; ends with a block barrier
__device__ __forceinline__ void peer_wait(const PeerPtrs& pp, int channel, unsigned target) {
  if ((int)threadIdx.x < pp.world) {
    const unsigned* f = pp.flags[pp.rank] + channel * kPeerChannelWords + threadIdx.x;
    unsigned v = ld_acquire_sys(f);
    if ((int)(v - target) < 0) {
      ptx::WaitClock clk;
      while ((int)((v = ld_acquire_sys(f)) - target) < 0) {
        if (clk.expired()) peer_timeout_trap(channel, (int)threadIdx.x, v, target);
        __nanosleep(20);
      }
    }
  }
  __syncthreads();
}
// last block of the launch publishes the new epoch (ticket counts the blocks that are done with the channel)
__device__ __forceinline__ void peer_finish(const PeerPtrs& pp, int channel, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned* base = pp.flags[pp.rank] + channel * kPeerChannelWords + kPeerMaxWorld;
    __threadfence();
    if (atomicAdd(base + 1, 1u) == gridDim.x * gridDim.y - 1u) {
      base[1] = 0u;
      *reinterpret_cast<volatile unsigned*>(base) = target;
      __threadfence();
    }
  }
}

// plain barrier between two kernels of the stream (one block)
__global__ void peer_barrier_kernel(const PeerPtrs pp, int channel) {
  const unsigned target = peer_target(pp, channel);
  peer_signal(pp, channel, target);
  peer_wait(pp, channel, target);
  peer_finish(pp, channel, target);
}

// ---------------------------------------------------------------------------------------------
// All-reduce + divide of the row-sharded M-step.  Exchange buffer of a rank (fp32 words unless noted):
//     [K*D sums | K counts (int32) | pad to 8 B | inertia (fp64)]          (peer_mstep_words)
// One block per cluster, as finalize_centers_kernel; block 0 also leaves the summed inertia in *inertia_out.
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline size_t peer_mstep_inertia_word(int K, int D) { return (((size_t)K * D + K + 1) / 2) * 2; }
__host__ __device__ inline size_t peer_mstep_words(int K, int D) { return peer_mstep_inertia_word(K, D) + 2; }

__global__ void __launch_bounds__(kEsCentroidThreads)
finalize_centers_peer_kernel(const PeerPtrs pp, int channel, size_t buf_word_offset, const float* __restrict__ c_old,
                             float* __restrict__ c_new, float* __restrict__ move_norm, float* __restrict__ counts_out,
                             double* __restrict__ inertia_out, int K, int D, __nv_bfloat16* __restrict__ plane_hi,
                             __nv_bfloat16* __restrict__ plane_lo, float* __restrict__ cnorm) {
  const unsigned target = peer_target(pp, channel);
  if (blockIdx.x == 0) peer_signal(pp, channel, target);
  peer_wait(pp, channel, target);

  const int k = blockIdx.x;
  const int G = pp.world;
  // Every peer load of the block is issued before the first one is consumed: a load over NVLink takes ~2 us, and the first
  // version's `for r: s += load(r)` paid that G times in a row (47 us for the reduce + divide at 8 ranks, 11 us at one).
  __shared__ int sh_cnt[kPeerMaxWorld];
  __shared__ double sh_inertia[kPeerMaxWorld];
  if ((int)threadIdx.x < G)
    sh_cnt[threadIdx.x] = ld_peer_i1(reinterpret_cast<const int*>(reinterpret_cast<const float*>(pp.buf[threadIdx.x]) + buf_word_offset + (size_t)K * D) + k);
  if (k == 0 && inertia_out && threadIdx.x >= 32 && (int)threadIdx.x < 32 + G)
    sh_inertia[threadIdx.x - 32] = ld_peer_d1(reinterpret_cast<const double*>(reinterpret_cast<const float*>(pp.buf[threadIdx.x - 32]) +
                                                                                 buf_word_offset + peer_mstep_inertia_word(K, D)));
  float part = 0.f, npart = 0.f;
  const bool vec = (D & 3) == 0;
  float cnt = 0.f;
  bool have_cnt = false;
  for (int d4 = threadIdx.x * 4; d4 < D || !have_cnt; d4 += blockDim.x * 4) {
    float4 v[kPeerMaxWorld];
    const int nd = min(4, D - d4);
    if (d4 < D) {
#pragma unroll
      for (int r = 0; r < kPeerMaxWorld; ++r) {          // fixed rank order below: identical bits on every rank
        if (r >= G) continue;
        const float* src = reinterpret_cast<const float*>(pp.buf[r]) + buf_word_offset + (size_t)k * D + d4;
        if (vec) v[r] = ld_peer_f4(src);
        else { v[r] = make_float4(0.f, 0.f, 0.f, 0.f); v[r].x = ld_peer_f1(src); if (nd > 1) v[r].y = ld_peer_f1(src + 1); if (nd > 2) v[r].z = ld_peer_f1(src + 2); if (nd > 3) v[r].w = ld_peer_f1(src + 3); }
      }
    }
    if (!have_cnt) {                                     // first trip: the counts (and the inertia) have landed in shared memory
      __syncthreads();
      int cnt_i = 0;
      for (int r = 0; r < G; ++r) cnt_i += sh_cnt[r];
      cnt = (float)cnt_i;
      have_cnt = true;
      if (threadIdx.x == 0 && counts_out) counts_out[k] = cnt;
      if (k == 0 && threadIdx.x == 0 && inertia_out) {
        double t = 0.0;
        for (int r = 0; r < G; ++r) t += sh_inertia[r];
        *inertia_out = t;
      }
    }
    if (d4 >= D) break;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int r = 0; r < kPeerMaxWorld; ++r) {
      if (r >= G) continue;
      s[0] += v[r].x; s[1] += v[r].y; s[2] += v[r].z; s[3] += v[r].w;
    }
    for (int q = 0; q < nd; ++q) {
      const int d = d4 + q;
      const float c = s[q] / cnt;                      // 0 / 0 -> NaN row, as torch's mean over zero rows
      c_new[(size_t)k * D + d] = c;
      if (c_old) { const float df = c - c_old[(size_t)k * D + d]; part += df * df; }
      if (plane_hi) es_store_split(c, plane_hi, plane_lo, (size_t)k * D + d);
    }
  }
  // ||c||^2 must be summed in the operands' order (estep_tc_kernel.cuh), not in the 4-wide one above: a second, cheap pass
  // over the row this block has just written
  __syncthreads();
  if (plane_hi)
    for (int d = threadIdx.x; d < D; d += blockDim.x) { const float c = c_new[(size_t)k * D + d]; npart = fmaf(c, c, npart); }
  block_sum_to_thread0(part, npart);
  if (threadIdx.x == 0) {
    if (move_norm) move_norm[k] = sqrtf(part);
    if (cnorm) cnorm[k] = npart;
  }
  peer_finish(pp, channel, target);
}

// ---------------------------------------------------------------------------------------------
// The all-gather of the vote records IS the store: rec[g] = [label, name_0 .. name_(k-1)] (int32) of global row
// g = row_offset + i goes to every rank's gathered array.
// ---------------------------------------------------------------------------------------------
// A block packs kPackRows records into shared memory (coalesced reads of labels / indices), then streams the packed bytes
// to every rank with 8-byte stores that are contiguous across the block (a record is (1 + k) * 4 bytes: 8-byte aligned
// whenever k is odd, as with k = 5; otherwise 4-byte stores).  The first version stored word by word from one thread per row:
// 48 scattered 4-byte remote stores per row at 8 ranks - 320-640 us for C5's 160 k rows per rank.
constexpr int kPackRows = 256;

__global__ void __launch_bounds__(256)
pack_vote_records_peer_kernel(const PeerPtrs pp, size_t buf_byte_offset, const long long* __restrict__ labels,
                              const long long* __restrict__ idx, int k_total, int k_used, long long n, long long row_offset) {
  __shared__ __align__(16) int rec[kPackRows * 9];            // k_used <= 8
  const int w = 1 + k_used;
  for (long long r0 = (long long)blockIdx.x * kPackRows; r0 < n; r0 += (long long)gridDim.x * kPackRows) {
    const int rows = (int)min((long long)kPackRows, n - r0);
    __syncthreads();                                          // the previous tile has left shared memory
    for (int t = threadIdx.x; t < rows * w; t += blockDim.x) {
      const int i = t / w, j = t - i * w;
      rec[t] = j == 0 ? (int)labels[r0 + i] : (int)idx[(r0 + i) * k_total + (j - 1)];
    }
    __syncthreads();
    const long long first_word = (row_offset + r0) * w;       // word offset of the tile in the gathered array
    const int words = rows * w;
    const bool wide = ((first_word | words) & 1) == 0 && (buf_byte_offset & 7) == 0;
    for (int r = 0; r < pp.world; ++r) {
      int* dst = reinterpret_cast<int*>(reinterpret_cast<char*>(pp.buf[r]) + buf_byte_offset) + first_word;
      if (wide) {
        for (int t = threadIdx.x; t < words / 2; t += blockDim.x)
          reinterpret_cast<int2*>(dst)[t] = reinterpret_cast<const int2*>(rec)[t];
      } else {
        for (int t = threadIdx.x; t < words; t += blockDim.x) dst[t] = rec[t];
      }
    }
  }
}

// The same exchange WITHOUT the second sort: the rank's records go out in the label-sorted order its M-step has just produced
// (`order` / `offsets` of scd_mstep_sums), record = [global row id, names], together with the rank's offsets table - every rank
// then votes by walking the `world` sorted runs of each cluster (vote_kernel<SEG>), no histogram / scan / scatter of the
// gathered records.
__global__ void __launch_bounds__(256)
pack_sorted_records_peer_kernel(const PeerPtrs pp, size_t rec_byte_offset, size_t off_byte_offset, const long long* __restrict__ idx,
                                int k_total, int k_used, long long n, long long row_offset, const int* __restrict__ order,
                                const int* __restrict__ offsets, int K) {
  __shared__ __align__(16) int rec[kPackRows * 9];
  const int w = 1 + k_used;
  if (blockIdx.x == 0) {                                    // this rank's offsets -> row `rank` of every rank's table
    for (int r = 0; r < pp.world; ++r) {
      int* dst = reinterpret_cast<int*>(reinterpret_cast<char*>(pp.buf[r]) + off_byte_offset) + (size_t)pp.rank * (K + 1);
      for (int t = threadIdx.x; t <= K; t += blockDim.x) dst[t] = offsets[t];
    }
  }
  for (long long p0 = (long long)blockIdx.x * kPackRows; p0 < n; p0 += (long long)gridDim.x * kPackRows) {
    const int rows = (int)min((long long)kPackRows, n - p0);
    __syncthreads();
    for (int i = threadIdx.x; i < rows; i += blockDim.x) {
      const int row = order[p0 + i];
      rec[i * w] = (int)(row_offset + row);
      for (int j = 0; j < k_used; ++j) rec[i * w + 1 + j] = (int)idx[(long long)row * k_total + j];
    }
    __syncthreads();
    const long long first_word = (row_offset + p0) * w;
    const int words = rows * w;
    const bool wide = ((first_word | words) & 1) == 0 && (rec_byte_offset & 7) == 0;
    for (int r = 0; r < pp.world; ++r) {
      int* dst = reinterpret_cast<int*>(reinterpret_cast<char*>(pp.buf[r]) + rec_byte_offset) + first_word;
      if (wide) {
        for (int t = threadIdx.x; t < words / 2; t += blockDim.x) reinterpret_cast<int2*>(dst)[t] = reinterpret_cast<const int2*>(rec)[t];
      } else {
        for (int t = threadIdx.x; t < words; t += blockDim.x) dst[t] = rec[t];
      }
    }
  }
}

}  // namespace scd

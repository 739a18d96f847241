// How many clusters of the scoring kernel (name_topk_kernel<5>: 640 threads, one CTA per SM, its real dynamic shared
// memory) the device can hold at once, for cluster sizes 1 .. 8.  The kernel is a persistent grid of one CTA per SM, so
// a cluster shape pays only if max-active-clusters x size still covers every SM; otherwise the clusters that do not fit
// run as a second wave (DESIGN 7, item 1: sharing vocabulary stages between two CTA pairs needs 4-CTA clusters).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o cluster_residency tools/cluster_residency.cu -lcuda
//   ./cluster_residency
// The kernel is compiled here without its compile-time __cluster_dims__(2, 1, 1), so that the launch configuration can
// ask for any cluster size; registers, threads and shared memory are those of the library's kernel.
#include <cuda_runtime.h>
#include <cstdio>
#undef __cluster_dims__
#define __cluster_dims__(...)
#include "../scd_b200/csrc/naming_kernel.cuh"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

int main() {
  int dev = 0, sms = 0, clk_khz = 0;
  CK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CK(cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, dev));
  const auto kernel = scd::name_topk_kernel<5>;
  const int smem = scd::NameSmem::total + 1024;              // as launch_name_topk
  CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, kernel));
  printf("device %d: %s, %d SMs, max SM clock %d MHz, %zu B shared memory per SM\n", dev, prop.name, sms, clk_khz / 1000,
         prop.sharedMemPerMultiprocessor);
  printf("name_topk_kernel<5>: %d threads, %d registers/thread, %d B dynamic + %zu B static shared memory\n",
         scd::kNameThreads, fa.numRegs, smem, fa.sharedSizeBytes);
  int blocks_per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kernel, scd::kNameThreads, smem));
  printf("CTAs per SM: %d\n", blocks_per_sm);
  for (int cs = 1; cs <= 8; ++cs) {
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = cs; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cs * (sms / cs), 1, 1);
    cfg.blockDim = dim3(scd::kNameThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int clusters = 0;
    const cudaError_t e = cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg);
    if (e != cudaSuccess) { printf("cluster size %d: %s\n", cs, cudaGetErrorString(e)); cudaGetLastError(); continue; }
    printf("cluster size %d: %d active clusters = %d of %d SMs (%d idle)\n", cs, clusters, clusters * cs, sms,
           sms - clusters * cs);
  }
  return 0;
}

// obs_compression_probe.cu -- device half of tools/obs_compression_probe.py: does an observation block write faster
// into compressible memory?  Loaded through ctypes; the script builds it into a temporary directory with
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fPIC -o probe.so obs_compression_probe.cu -lcuda
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

// dst[t * n16 + j] = pat[j] for every tile t: a pattern of n16 16-byte units tiled ntiles times.  Each thread loads
// its pattern unit once and writes it into tiles blockIdx.y, blockIdx.y + gridDim.y, ... (coalesced per tile).
template <bool CS>
__global__ void tile_write(uint4* __restrict__ dst, const uint4* __restrict__ pat, size_t n16, int ntiles) {
  const size_t j = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (j >= n16) return;
  const uint4 v = __ldg(pat + j);
  for (int t = blockIdx.y; t < ntiles; t += gridDim.y) {
    if (CS) __stcs(dst + (size_t)t * n16 + j, v);
    else dst[(size_t)t * n16 + j] = v;
  }
}

// Launches `reps` tile writes on the default stream and returns their total time in ms (CUDA events), or -1.
extern "C" float probe_tile_write(void* dst, const void* pat, size_t pat_bytes, int ntiles, int cs, int reps) {
  const size_t n16 = pat_bytes / 16;
  const dim3 block(256), grid((unsigned)((n16 + 255) / 256), 8);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  cudaEventRecord(a);
  for (int r = 0; r < reps; ++r) {
    if (cs) tile_write<true><<<grid, block>>>((uint4*)dst, (const uint4*)pat, n16, ntiles);
    else tile_write<false><<<grid, block>>>((uint4*)dst, (const uint4*)pat, n16, ntiles);
  }
  cudaEventRecord(b);
  float ms = -1.0f;
  if (cudaEventSynchronize(b) == cudaSuccess) cudaEventElapsedTime(&ms, a, b);
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  return cudaGetLastError() == cudaSuccess ? ms : -1.0f;
}

// What the driver reports for a compressible allocation of `bytes` on `device`: out[0] the device attribute
// CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, out[1] the allocation granularity asked with the compression
// flag, out[2] the compressionType cuMemGetAllocationPropertiesFromHandle reads back (-1 if not asked), out[3] the
// CUresult of the first failing call (0 = none).  The allocation is released again.
extern "C" void probe_compression_props(int device, size_t bytes, long long out[4]) {
  out[0] = out[1] = 0; out[2] = -1; out[3] = 0;
  cudaSetDevice(device);
  cudaFree(0);                                   // primary context
  int supported = 0;
  CUresult r = cuDeviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device);
  if (r != CUDA_SUCCESS) { out[3] = r; return; }
  out[0] = supported;
  CUmemAllocationProp prop;
  memset(&prop, 0, sizeof prop);
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = device;
  prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
  size_t gran = 0;
  r = cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED);
  if (r != CUDA_SUCCESS) { out[3] = r; return; }
  out[1] = (long long)gran;
  CUmemGenericAllocationHandle h;
  r = cuMemCreate(&h, (bytes + gran - 1) / gran * gran, &prop, 0);
  if (r != CUDA_SUCCESS) { out[3] = r; return; }
  CUmemAllocationProp got;
  memset(&got, 0, sizeof got);
  r = cuMemGetAllocationPropertiesFromHandle(&got, h);
  if (r != CUDA_SUCCESS) out[3] = r;
  else out[2] = got.allocFlags.compressionType;
  cuMemRelease(h);
}

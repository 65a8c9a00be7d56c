// Test-only helper of tests/test_poison_gpu.py (built there with nvcc into a temporary directory, loaded with
// ctypes; never part of libsrst.so): fills the shared memory of every SM with a 32-bit pattern, and probes whether
// that pattern is still there when the next kernel starts.
//
// A CTA that asks for the opt-in maximum of dynamic shared memory occupies (nearly) all of an SM's shared memory, so
// 2 x SM-count such CTAs cover every SM.  Whether the contents survive into the next kernel's CTAs is not something
// CUDA guarantees; the probe measures it, and the tests skip when it does not hold.
#include <cuda_runtime.h>

namespace {

__global__ void smem_fill_kernel(unsigned value, unsigned words) {
  extern __shared__ unsigned s_fill[];
  for (unsigned i = threadIdx.x; i < words; i += blockDim.x) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(s_fill + i);
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(value) : "memory");  // a store the compiler must keep
  }
}

// Reads the whole window without writing it; counts[blockIdx.x] = words equal to `value`.
__global__ void smem_probe_kernel(unsigned value, unsigned words, unsigned* counts) {
  extern __shared__ unsigned s_probe[];
  unsigned n = 0;
  for (unsigned i = threadIdx.x; i < words; i += blockDim.x) {
    unsigned v;
    const unsigned a = (unsigned)__cvta_generic_to_shared(s_probe + i);
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    n += (v == value);
  }
  atomicAdd(counts + blockIdx.x, n);
}

int max_dyn_smem(int* bytes, int* sms) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(bytes, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
  return (int)e;
}

}  // namespace

extern "C" {

// Number of CTAs smem_poison_fill / smem_poison_probe launch (2 x SM count); 0 on error.
int smem_poison_blocks(void) {
  int bytes = 0, sms = 0;
  return max_dyn_smem(&bytes, &sms) ? 0 : 2 * sms;
}

// Words of shared memory each CTA covers.
int smem_poison_words(void) {
  int bytes = 0, sms = 0;
  return max_dyn_smem(&bytes, &sms) ? 0 : bytes / 4;
}

int smem_poison_fill(unsigned value, void* stream) {
  int bytes = 0, sms = 0;
  int e = max_dyn_smem(&bytes, &sms);
  if (e) return e;
  if ((e = (int)cudaFuncSetAttribute(smem_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes))) return e;
  smem_fill_kernel<<<2 * sms, 1024, bytes, (cudaStream_t)stream>>>(value, (unsigned)bytes / 4);
  return (int)cudaGetLastError();
}

// counts: device array of smem_poison_blocks() zeroed unsigned ints.
int smem_poison_probe(unsigned value, unsigned* counts, void* stream) {
  int bytes = 0, sms = 0;
  int e = max_dyn_smem(&bytes, &sms);
  if (e) return e;
  if ((e = (int)cudaFuncSetAttribute(smem_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes))) return e;
  smem_probe_kernel<<<2 * sms, 1024, bytes, (cudaStream_t)stream>>>(value, (unsigned)bytes / 4, counts);
  return (int)cudaGetLastError();
}

}  // extern "C"

// gather_ceiling.cu -- the ceiling for n-tuple lookups: random 4-byte reads from a float table, nothing else.
// Thread t makes `lookups` reads at hashed uniform indices into a table of 2^log2_entries floats, sums them and writes one
// float (so the reads cannot be dropped).  Built by tools/ntuple_bench.py into a temporary directory and called via ctypes:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -shared -Xcompiler -fPIC -o libgather_ceiling.so tools/gather_ceiling.cu
#include <cuda_runtime.h>
#include <stdint.h>

__global__ void __launch_bounds__(256) gather_kernel(const float *__restrict__ table, uint32_t mask, int lookups, float *out, int64_t threads)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= threads) return;
    uint32_t h = (uint32_t)t * 0x9E3779B1u + 0x7F4A7C15u;
    float acc = 0.0f;
#pragma unroll 8
    for (int j = 0; j < lookups; ++j) {
        h ^= h >> 15;
        h *= 0x2C1B3C6Du;
        h ^= h >> 12;
        acc += __ldg(table + (h & mask));
    }
    out[t] = acc;
}

extern "C" int gather_ceiling(const float *table, int log2_entries, int lookups, float *out, int64_t threads, void *stream)
{
    const int64_t grid = (threads + 255) / 256;
    gather_kernel<<<(unsigned)grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(table, (1u << log2_entries) - 1u, lookups, out, threads);
    return (int)cudaGetLastError();
}

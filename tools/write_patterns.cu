// write_patterns.cu -- which write pattern reaches the pure-write ceiling of HBM (torch fill_: 7.5 TB/s on this B200)?
// The fused step kernel writes 1 KiB of one-hot per game; its tile writer saturates at 6.67 TB/s.  These kernels write the
// same 16 GiB with different shapes of "who writes what when":
//   grid_stride  : thread t of the whole grid writes 16 B at t*16, then strides by the grid (what an elementwise fill does)
//   tile<T,KB>   : block b owns the contiguous tile [b*KB KiB, (b+1)*KB KiB) and writes it with T threads, 16 B per thread
//                  per pass (what the step kernel's plain-store writer does: KB = T)
//   tile_tma     : the same tile through shared memory + cp.async.bulk (what the shipped writer does)
//   persistent   : G resident blocks; block b writes chunk b, b+G, b+2G ... of CH KiB each (a compact moving write front)
// `--compressible` instead times the shipped writer's shape on two 16 GiB outputs, plain cudaMalloc memory and memory
// allocated with cuMemCreate(compressionType = CU_MEM_ALLOCATION_COMP_GENERIC), both holding the fp32 one-hot of
// seeded steady-state-like boards (see compressible_probe below).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o /tmp/write_patterns tools/write_patterns.cu -lcuda && /tmp/write_patterns
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#define CK(x)                                                                                 \
    do {                                                                                      \
        cudaError_t e_ = (x);                                                                 \
        if (e_ != cudaSuccess) {                                                              \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
            exit(1);                                                                          \
        }                                                                                     \
    } while (0)

__global__ void grid_stride(uint4 *out, size_t n16)
{
    const uint4 v = make_uint4(0x3f800000u, 0, 0, 0x3f800000u);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) out[i] = v;
}

template <int T>
__global__ void __launch_bounds__(T) tile(uint4 *out, size_t n16, int tile16)  // tile16 = 16-byte pieces per block
{
    const uint4 v = make_uint4(0x3f800000u, 0, 0, 0x3f800000u);
    uint4 *base = out + (size_t)blockIdx.x * tile16;
    for (int i = threadIdx.x; i < tile16; i += T) base[i] = v;
}

template <int T>
__global__ void __launch_bounds__(T) tile_tma(uint4 *out, size_t n16, int tile16, int chunk16)
{
    extern __shared__ __align__(128) uint4 stage[];  // [2][chunk16]
    const uint4 v = make_uint4(0x3f800000u, 0, 0, 0x3f800000u);
    char *base = reinterpret_cast<char *>(out + (size_t)blockIdx.x * tile16);
    int buf = 0;
    for (int c0 = 0; c0 < tile16; c0 += chunk16, buf ^= 1) {
        uint4 *dst = stage + buf * chunk16;
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncthreads();
        for (int i = threadIdx.x; i < chunk16; i += T) dst[i] = v;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(base + (size_t)c0 * 16), "r"(src),
                         "r"((uint32_t)chunk16 * 16u)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
}

template <int T>
__global__ void __launch_bounds__(T) persistent(uint4 *out, size_t n16, int chunk16)
{
    const uint4 v = make_uint4(0x3f800000u, 0, 0, 0x3f800000u);
    const size_t chunks = n16 / chunk16;
    for (size_t c = blockIdx.x; c < chunks; c += gridDim.x) {
        uint4 *base = out + c * chunk16;
        for (int i = threadIdx.x; i < chunk16; i += T) base[i] = v;
    }
}

// tile_tma + what the step kernel does besides the tile: per thread a 16 B + 3 x 4 B read at the start (board, mask, step,
// score) and/or the narrow side writes (board 16 B, mask/reward/score/step 4 B, two 1-byte flags)
// read_mask: the reads wrap inside (read_mask + 1) games (small = L2-resident inputs); prefetch_ahead: blocks ahead whose
// inputs this block pulls into L2 (0 = none)
template <int T, bool kReads, bool kSideWrites>
__global__ void __launch_bounds__(T) tile_tma_mixed(uint4 *out, size_t n16, int tile16, int chunk16, const uint4 *rd16, const uint32_t *rd4,
                                                    uint4 *wr16, uint32_t *wr4, uint8_t *wr1, size_t games, size_t read_mask = ~(size_t)0,
                                                    int prefetch_ahead = 0)
{
    extern __shared__ __align__(128) uint4 stage[];
    const size_t g = (size_t)blockIdx.x * T + threadIdx.x;
    uint4 v = make_uint4(0x3f800000u, 0, 0, 0x3f800000u);
    if (kReads) {
        const size_t r = g & read_mask;
        const uint4 b = rd16[r];
        v.y = b.x ^ b.y ^ b.z ^ b.w ^ rd4[r] ^ rd4[games + r] ^ rd4[2 * games + r];
        if (prefetch_ahead) {
            const size_t p = g + (size_t)prefetch_ahead * T;
            if (p < games) {
                if ((threadIdx.x & 1) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(rd16 + p));  // one per 32-byte sector
                if ((threadIdx.x & 7) == 0) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rd4 + p));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rd4 + games + p));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rd4 + 2 * games + p));
                }
            }
        }
    }
    if (kSideWrites) {
        wr16[g] = v;
        wr4[g] = v.y, wr4[games + g] = v.x, wr4[2 * games + g] = v.y, wr4[3 * games + g] = v.x;
        wr1[g] = 0, wr1[games + g] = 1;
    }
    char *base = reinterpret_cast<char *>(out + (size_t)blockIdx.x * tile16);
    int buf = 0;
    for (int c0 = 0; c0 < tile16; c0 += chunk16, buf ^= 1) {
        uint4 *dst = stage + buf * chunk16;
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncthreads();
        for (int i = threadIdx.x; i < chunk16; i += T) dst[i] = v;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(base + (size_t)c0 * 16), "r"(src),
                         "r"((uint32_t)chunk16 * 16u)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
}

// the same with every block owning `tiles` consecutive tiles and loading the inputs of tile k+1 (into registers) before it
// writes tile k: the read latency never stands between two tiles
template <int T>
__global__ void __launch_bounds__(T) tile_tma_pipelined(uint4 *out, size_t n16, int tile16, int chunk16, const uint4 *rd16, const uint32_t *rd4,
                                                         size_t games, int tiles)
{
    extern __shared__ __align__(128) uint4 stage[];
    size_t g = ((size_t)blockIdx.x * tiles) * T + threadIdx.x;
    uint4 b = rd16[g];
    uint32_t x0 = rd4[g], x1 = rd4[games + g], x2 = rd4[2 * games + g];
    int buf = 0;
    for (int t = 0; t < tiles; ++t) {
        uint4 v = make_uint4(0x3f800000u, b.x ^ b.y ^ b.z ^ b.w ^ x0 ^ x1 ^ x2, 0, 0x3f800000u);
        char *base = reinterpret_cast<char *>(out + ((size_t)blockIdx.x * tiles + t) * tile16);
        if (t + 1 < tiles) {  // next tile's inputs: in flight while this tile is written
            g += T;
            b = rd16[g];
            x0 = rd4[g], x1 = rd4[games + g], x2 = rd4[2 * games + g];
        }
        for (int c0 = 0; c0 < tile16; c0 += chunk16, buf ^= 1) {
            uint4 *dst = stage + buf * chunk16;
            if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            __syncthreads();
            for (int i = threadIdx.x; i < chunk16; i += T) dst[i] = v;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (threadIdx.x == 0) {
                const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(base + (size_t)c0 * 16), "r"(src),
                             "r"((uint32_t)chunk16 * 16u)
                             : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
}

// read-side variations: mode 0 = 16-byte read only, 1 = three 4-byte reads only, 2 = all reads with ld.global.cg (L2 only),
// 3 = all reads, result not used by the tile (consumed by a never-taken store after the tile), 4 = all reads via ld.global.nc
template <int T, int kMode>
__global__ void __launch_bounds__(T) tile_tma_reads(uint4 *out, size_t n16, int tile16, int chunk16, const uint4 *rd16, const uint32_t *rd4,
                                                     size_t games, uint32_t *sink)
{
    extern __shared__ __align__(128) uint4 stage[];
    const size_t g = (size_t)blockIdx.x * T + threadIdx.x;
    uint4 v = make_uint4(0x3f800000u, 0, 0, 0x3f800000u);
    uint32_t acc = 0;
    if (kMode == 0) { const uint4 b = rd16[g]; acc = b.x ^ b.y ^ b.z ^ b.w; }
    if (kMode == 1) acc = rd4[g] ^ rd4[games + g] ^ rd4[2 * games + g];
    if (kMode == 2) { const uint4 b = __ldcg(rd16 + g); acc = b.x ^ b.y ^ b.z ^ b.w ^ __ldcg(rd4 + g) ^ __ldcg(rd4 + games + g) ^ __ldcg(rd4 + 2 * games + g); }
    if (kMode == 3 || kMode == 4) { const uint4 b = __ldg(rd16 + g); acc = b.x ^ b.y ^ b.z ^ b.w ^ __ldg(rd4 + g) ^ __ldg(rd4 + games + g) ^ __ldg(rd4 + 2 * games + g); }
    if (kMode != 3) v.y = acc;
    char *base = reinterpret_cast<char *>(out + (size_t)blockIdx.x * tile16);
    int buf = 0;
    for (int c0 = 0; c0 < tile16; c0 += chunk16, buf ^= 1) {
        uint4 *dst = stage + buf * chunk16;
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncthreads();
        for (int i = threadIdx.x; i < chunk16; i += T) dst[i] = v;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(base + (size_t)c0 * 16), "r"(src),
                         "r"((uint32_t)chunk16 * 16u)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
    if (kMode == 3 && acc == 0x12345678u) sink[0] = acc;
}

// the block's inputs fetched by the TMA engine as four bulk copies (12 KiB + 3 x 3 KiB) into shared memory instead of
// ~100 warp-level loads: does the memory system treat few large read requests more kindly inside a write stream?
template <int T>
__global__ void __launch_bounds__(T) tile_tma_bulkreads(uint4 *out, size_t n16, int tile16, int chunk16, const uint4 *rd16, const uint32_t *rd4,
                                                         size_t games)
{
    extern __shared__ __align__(128) uint4 stage[];  // [2][chunk16] staging, then the inputs
    __shared__ __align__(8) unsigned long long bar;
    uint4 *in16 = stage + 2 * chunk16;
    uint32_t *in4 = reinterpret_cast<uint32_t *>(in16 + T);
    const size_t g0 = (size_t)blockIdx.x * T;
    const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t total = T * 16 + 3 * T * 4;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(total) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(in16)),
                     "l"(rd16 + g0), "r"((uint32_t)(T * 16)), "r"(bar_a)
                     : "memory");
        for (int k = 0; k < 3; ++k)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             (uint32_t)__cvta_generic_to_shared(in4 + k * T)),
                         "l"(rd4 + k * games + g0), "r"((uint32_t)(T * 4)), "r"(bar_a)
                         : "memory");
    }
    {
        uint32_t done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(bar_a) : "memory");
    }
    const uint4 b = in16[threadIdx.x];
    uint4 v = make_uint4(0x3f800000u, b.x ^ b.y ^ b.z ^ b.w ^ in4[threadIdx.x] ^ in4[T + threadIdx.x] ^ in4[2 * T + threadIdx.x], 0, 0x3f800000u);
    char *base = reinterpret_cast<char *>(out + (size_t)blockIdx.x * tile16);
    int buf = 0;
    for (int c0 = 0; c0 < tile16; c0 += chunk16, buf ^= 1) {
        uint4 *dst = stage + buf * chunk16;
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncthreads();
        for (int i = threadIdx.x; i < chunk16; i += T) dst[i] = v;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(base + (size_t)c0 * 16), "r"(src),
                         "r"((uint32_t)chunk16 * 16u)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
}

template <class F>
static float timed(F launch, int reps = 6)
{
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    launch();
    float best = 1e9f;
    for (int r = 0; r < reps; ++r) {
        CK(cudaEventRecord(e0));
        launch();
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        best = ms < best ? ms : best;
    }
    CK(cudaGetLastError());
    return best;
}

// ---- --compressible: plain against compressible output memory, realistic one-hot data ----------------------------

#define CKD(x)                                                                                   \
    do {                                                                                         \
        CUresult r_ = (x);                                                                       \
        if (r_ != CUDA_SUCCESS) {                                                                \
            const char *s_ = "?";                                                                \
            cuGetErrorString(r_, &s_);                                                           \
            fprintf(stderr, "%s:%d %s: %s (%d)\n", __FILE__, __LINE__, #x, s_, (int)r_);         \
            exit(1);                                                                             \
        }                                                                                        \
    } while (0)

__host__ __device__ inline uint64_t splitmix64(uint64_t x)
{
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

// A board like the step kernel sees at steady state, one byte per cell, from a fixed seed: each cell empty with
// probability 1/2, else exponent 1 + (trailing ones of a random word), capped at 11 (1/2, 1/4, ... of the tiles).
__device__ inline uint4 synth_board(uint64_t g)
{
    uint32_t w[4];
    for (int q = 0; q < 4; ++q) {
        w[q] = 0;
        for (int b = 0; b < 4; ++b) {
            const uint64_t h = splitmix64(0x2048c0ffee000000ull ^ (g * 16 + q * 4 + b));
            const uint32_t e = (h & 1) ? 0u : 1u + min(10u, (uint32_t)__ffsll((long long)~(h >> 1)) - 1u);
            w[q] |= e << (8 * b);
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

__global__ void fill_inputs(uint4 *rd16, uint32_t *rd4, size_t games)
{
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < games; g += (size_t)gridDim.x * blockDim.x) {
        rd16[g] = synth_board(g);
        rd4[g] = 0xffffu, rd4[games + g] = (uint32_t)g, rd4[2 * games + g] = 0x3f800000u;  // mask, step, score
    }
}

// The shipped fp32 writer (write_onehot_tile_tma in vecgame_kernels.cu): out[g][k][c] = (board[g][c] == k), block b owns
// games [b*T, (b+1)*T), 48 KiB chunks staged in shared memory and stored by cp.async.bulk, double-buffered.
// kReads: the board comes from memory with the step's three 4-byte reads beside it (else synth_board in registers);
// kSideWrites: the step's narrow side writes (board 16 B, mask/reward/score/step 4 B, two 1-byte flags).
template <int T, bool kReads, bool kSideWrites>
__global__ void __launch_bounds__(T) onehot_tma(uint4 *out, int chunk16, const uint4 *rd16, const uint32_t *rd4, uint4 *wr16,
                                                uint32_t *wr4, uint8_t *wr1, size_t games)
{
    extern __shared__ __align__(128) uint4 stage[];  // [2][chunk16]
    __shared__ uint4 sboards[T];
    const size_t g = (size_t)blockIdx.x * T + threadIdx.x;
    uint4 b;
    uint32_t x = 0;
    if (kReads) {
        b = rd16[g];
        x = rd4[g] ^ rd4[games + g] ^ rd4[2 * games + g];
    } else {
        b = synth_board(g);
    }
    if (kSideWrites) {
        wr16[g] = b;
        wr4[g] = x, wr4[games + g] = b.x, wr4[2 * games + g] = x, wr4[3 * games + g] = b.y;
        wr1[g] = 0, wr1[games + g] = 1;
    }
    sboards[threadIdx.x] = b;
    __syncthreads();
    char *base = reinterpret_cast<char *>(out + (size_t)blockIdx.x * T * 64);
    int buf = 0;
    for (int c0 = 0; c0 < T * 64; c0 += chunk16, buf ^= 1) {
        uint4 *dst = stage + buf * chunk16;
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncthreads();
        for (int i = threadIdx.x; i < chunk16; i += T) {
            const int q = c0 + i, piece = q & 63;
            const uint32_t k = (uint32_t)piece >> 2;
            const uint32_t word = reinterpret_cast<const uint32_t *>(sboards + (q >> 6))[piece & 3];
            uint4 v;
            v.x = ((word & 0xff) == k) ? 0x3f800000u : 0u;
            v.y = (((word >> 8) & 0xff) == k) ? 0x3f800000u : 0u;
            v.z = (((word >> 16) & 0xff) == k) ? 0x3f800000u : 0u;
            v.w = ((word >> 24) == k) ? 0x3f800000u : 0u;
            dst[i] = v;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(dst);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(base + (size_t)c0 * 16), "r"(src),
                         "r"((uint32_t)chunk16 * 16u)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
}

// sum of word * (index + 1) and the number of 1.0f words over the buffer: equal for equal contents
__global__ void checksum(const uint32_t *p, size_t n, unsigned long long *acc)
{
    unsigned long long s = 0, ones = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        s += (unsigned long long)p[i] * (i + 1);
        ones += p[i] == 0x3f800000u;
    }
    atomicAdd(acc, s);
    atomicAdd(acc + 1, ones);
}

struct Compressible {
    CUdeviceptr ptr = 0;
    size_t size = 0, granted = 0;
    std::vector<CUmemGenericAllocationHandle> handles;
};

// reserve `bytes` (rounded up to the granularity), back it with `chunks` equal cuMemCreate allocations asking for generic
// compression, and count the bytes whose allocation the driver granted it (read back, not assumed)
static Compressible alloc_compressible(int dev, size_t bytes, int chunks)
{
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = dev;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    CKD(cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    Compressible c;
    const size_t chunk = (bytes / chunks + gran - 1) / gran * gran;
    c.size = chunk * chunks;
    CKD(cuMemAddressReserve(&c.ptr, c.size, gran, 0, 0));
    for (int i = 0; i < chunks; ++i) {
        CUmemGenericAllocationHandle h;
        CKD(cuMemCreate(&h, chunk, &prop, 0));
        CUmemAllocationProp got = {};
        CKD(cuMemGetAllocationPropertiesFromHandle(&got, h));
        if (got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC) c.granted += chunk;
        CKD(cuMemMap(c.ptr + (size_t)i * chunk, chunk, 0, h, 0));
        c.handles.push_back(h);
    }
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    CKD(cuMemSetAccess(c.ptr, c.size, &acc, 1));
    return c;
}

static void free_compressible(Compressible &c)
{
    CK(cudaDeviceSynchronize());
    CKD(cuMemUnmap(c.ptr, c.size));
    for (auto h : c.handles) CKD(cuMemRelease(h));
    CKD(cuMemAddressFree(c.ptr, c.size));
    c = Compressible();
}

static int compressible_probe(int reps)
{
    const size_t bytes = (size_t)16 << 30, n16 = bytes / 16, games = n16 / 64;  // 2^24 games x 1 KiB
    CK(cudaSetDevice(0));
    CK(cudaFree(0));  // the primary context, which the driver calls below use
    CUdevice dev;
    CKD(cuDeviceGet(&dev, 0));
    char name[256];
    CKD(cuDeviceGetName(name, sizeof name, dev));
    int supported = 0;
    CKD(cuDeviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
    int drv = 0;
    CKD(cuDriverGetVersion(&drv));
    printf("device: %s, driver API %d, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = %d\n", name, drv, supported);
    {
        CUmemAllocationProp prop = {};
        prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
        prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        prop.location.id = 0;
        size_t gmin = 0, grec = 0, pmin = 0;
        CKD(cuMemGetAllocationGranularity(&pmin, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM));
        prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
        CKD(cuMemGetAllocationGranularity(&gmin, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM));
        CKD(cuMemGetAllocationGranularity(&grec, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
        printf("granularity: plain minimum %zu B; compressible minimum %zu B, recommended %zu B\n", pmin, gmin, grec);
    }
    if (!supported) {
        printf("no generic compression on this device: nothing to compare\n");
        return 0;
    }
    Compressible comp = alloc_compressible(0, bytes, 1);
    printf("one %zu-byte allocation: %zu bytes granted compression\n", comp.size, comp.granted);
    if (comp.granted < comp.size) {
        free_compressible(comp);
        for (int chunks : {8, 64}) {
            comp = alloc_compressible(0, bytes, chunks);
            printf("%d chunks of %zu bytes: %zu bytes granted compression\n", chunks, comp.size / chunks, comp.granted);
            if (comp.granted == comp.size) break;
            free_compressible(comp);
        }
    }
    uint4 *plain;
    CK(cudaMalloc(&plain, bytes));
    uint4 *bufs[2] = {plain, reinterpret_cast<uint4 *>(comp.ptr)};
    const char *bufname[2] = {"plain", "compressible"};

    uint4 *rd16, *wr16;
    uint32_t *rd4, *wr4;
    uint8_t *wr1;
    CK(cudaMalloc(&rd16, games * 16));
    CK(cudaMalloc(&wr16, games * 16));
    CK(cudaMalloc(&rd4, games * 12));
    CK(cudaMalloc(&wr4, games * 16));
    CK(cudaMalloc(&wr1, games * 2));
    fill_inputs<<<4096, 256>>>(rd16, rd4, games);
    CK(cudaGetLastError());
    const unsigned grid = (unsigned)(games / 768);
    const int smem = 2 * 49152, chunk16 = 3072;
    CK(cudaFuncSetAttribute(onehot_tma<768, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CK(cudaFuncSetAttribute(onehot_tma<768, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    unsigned long long *acc;
    CK(cudaMalloc(&acc, 2 * 2 * sizeof(unsigned long long)));

    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    auto ab = [&](const char *what, auto launch) {  // warm both, then alternate plain / compressible, median of `reps` each
        std::vector<float> t[2];
        for (int i = 0; i < 2; ++i) launch(bufs[i]);
        for (int r = 0; r < reps; ++r)
            for (int i = 0; i < 2; ++i) {
                CK(cudaEventRecord(e0));
                launch(bufs[i]);
                CK(cudaEventRecord(e1));
                CK(cudaEventSynchronize(e1));
                float ms;
                CK(cudaEventElapsedTime(&ms, e0, e1));
                t[i].push_back(ms);
            }
        CK(cudaGetLastError());
        float med[2];
        for (int i = 0; i < 2; ++i) {
            std::sort(t[i].begin(), t[i].end());
            med[i] = t[i][t[i].size() / 2];
            printf("%-46s %-12s median %7.3f ms (min %7.3f, max %7.3f) over %d, %6.0f GB/s of output\n", what, bufname[i], med[i],
                   t[i].front(), t[i].back(), reps, bytes / med[i] / 1e6);
        }
        printf("%-46s compressible / plain time %.3f\n", what, med[1] / med[0]);
    };
    auto sums = [&](const char *what) {
        unsigned long long h[4];
        CK(cudaMemset(acc, 0, 4 * sizeof(unsigned long long)));
        for (int i = 0; i < 2; ++i) checksum<<<4096, 256>>>(reinterpret_cast<const uint32_t *>(bufs[i]), bytes / 4, acc + 2 * i);
        CK(cudaMemcpy(h, acc, sizeof h, cudaMemcpyDeviceToHost));
        printf("checksum after %s: plain %016llx / %llu ones, compressible %016llx / %llu ones: %s\n", what, h[0], h[1], h[2], h[3],
               (h[0] == h[2] && h[1] == h[3]) ? "equal" : "DIFFERENT");
        return h[0] == h[2] && h[1] == h[3];
    };

    ab("cudaMemset 0", [&](uint4 *o) { CK(cudaMemsetAsync(o, 0, bytes)); });
    bool same = sums("cudaMemset 0");
    ab("tile_tma 768, one-hot of synthetic boards", [&](uint4 *o) {
        onehot_tma<768, false, false><<<grid, 768, smem>>>(o, chunk16, rd16, rd4, wr16, wr4, wr1, games);
    });
    same = sums("tile_tma 768") && same;
    ab("tile_tma 768 + reads + side writes (step mix)", [&](uint4 *o) {
        onehot_tma<768, true, true><<<grid, 768, smem>>>(o, chunk16, rd16, rd4, wr16, wr4, wr1, games);
    });
    same = sums("tile_tma 768 + reads + side writes") && same;

    CK(cudaFree(plain));
    CK(cudaFree(rd16));
    CK(cudaFree(wr16));
    CK(cudaFree(rd4));
    CK(cudaFree(wr4));
    CK(cudaFree(wr1));
    CK(cudaFree(acc));
    free_compressible(comp);
    return same ? 0 : 1;
}

int main(int argc, char **argv)
{
    if (argc > 1 && !strcmp(argv[1], "--compressible")) return compressible_probe(argc > 2 ? atoi(argv[2]) : 15);
    const size_t bytes = (size_t)16 << 30, n16 = bytes / 16;
    uint4 *out;
    CK(cudaMalloc(&out, bytes));
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    auto report = [&](const char *name, float ms) { printf("%-58s %8.3f ms  %7.0f GB/s\n", name, ms, bytes / ms / 1e6); };

    report("cudaMemset", timed([&] { CK(cudaMemsetAsync(out, 0, bytes)); }));
    report("grid_stride, 256 thr, grid = 148*8", timed([&] { grid_stride<<<sms * 8, 256>>>(out, n16); }));
    report("grid_stride, 256 thr, grid = n16/256/4 (4 stores/thread)", timed([&] { grid_stride<<<(unsigned)(n16 / 256 / 4), 256>>>(out, n16); }));
    report("grid_stride, 256 thr, grid = n16/256 (1 store/thread)", timed([&] { grid_stride<<<(unsigned)(n16 / 256), 256>>>(out, n16); }));
    for (int kb : {16, 64, 256, 768}) {
        char name[96];
        const int tile16 = kb * 64;
        snprintf(name, sizeof name, "tile, 256 thr, %d KiB per block", kb);
        report(name, timed([&] { tile<256><<<(unsigned)(n16 / tile16), 256>>>(out, n16, tile16); }));
    }
    report("tile, 768 thr, 768 KiB per block", timed([&] { tile<768><<<(unsigned)(n16 / (768 * 64)), 768>>>(out, n16, 768 * 64); }));
    report("tile, 1024 thr, 1024 KiB per block", timed([&] { tile<1024><<<(unsigned)(n16 / (1024 * 64)), 1024>>>(out, n16, 1024 * 64); }));
    CK(cudaFuncSetAttribute(tile_tma<768>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
    report("tile_tma, 768 thr, 768 KiB per block, 2 x 48 KiB chunks", timed([&] { tile_tma<768><<<(unsigned)(n16 / (768 * 64)), 768, 2 * 49152>>>(out, n16, 768 * 64, 3072); }));
    CK(cudaFuncSetAttribute(tile_tma<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 16384));
    report("tile_tma, 256 thr, 256 KiB per block, 2 x 16 KiB chunks", timed([&] { tile_tma<256><<<(unsigned)(n16 / (256 * 64)), 256, 2 * 16384>>>(out, n16, 256 * 64, 1024); }));
    report("tile_tma, 256 thr, 64 KiB per block, 2 x 16 KiB chunks", timed([&] { tile_tma<256><<<(unsigned)(n16 / (64 * 64)), 256, 2 * 16384>>>(out, n16, 64 * 64, 1024); }));
    {
        const size_t games = n16 / 64;  // 1 KiB of tile per "game"
        uint4 *rd16, *wr16;
        uint32_t *rd4, *wr4;
        uint8_t *wr1;
        CK(cudaMalloc(&rd16, games * 16));
        CK(cudaMalloc(&wr16, games * 16));
        CK(cudaMalloc(&rd4, games * 12));
        CK(cudaMalloc(&wr4, games * 16));
        CK(cudaMalloc(&wr1, games * 2));
        CK(cudaMemset(rd16, 1, games * 16));
        CK(cudaMemset(rd4, 1, games * 12));
        const unsigned grid = (unsigned)(games / 768);
        CK(cudaFuncSetAttribute(tile_tma_mixed<768, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        CK(cudaFuncSetAttribute(tile_tma_mixed<768, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        CK(cudaFuncSetAttribute(tile_tma_mixed<768, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        report("tile_tma 768 + 28 B/game reads", timed([&] { tile_tma_mixed<768, true, false><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games); }));
        report("tile_tma 768 + reads from a 1 Mi-game window (28 MB, re-read every 160 us)", timed([&] { tile_tma_mixed<768, true, false><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games, (1u << 20) - 1, 0); }));
        report("tile_tma 768 + reads from a 64 Ki-game window (1.8 MB, re-read every 10 us)", timed([&] { tile_tma_mixed<768, true, false><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games, (1u << 16) - 1, 0); }));
        report("tile_tma 768 + reads from a 4 Ki-game window (115 KB, always in L2)", timed([&] { tile_tma_mixed<768, true, false><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games, (1u << 12) - 1, 0); }));
        for (int ahead : {296, 600, 1200, 2400})
        {
            char name[96];
            snprintf(name, sizeof name, "tile_tma 768 + reads, L2 prefetch %d blocks ahead", ahead);
            report(name, timed([&] { tile_tma_mixed<768, true, false><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games, ~(size_t)0, ahead); }));
        }
        CK(cudaFuncSetAttribute(tile_tma_reads<768, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        CK(cudaFuncSetAttribute(tile_tma_reads<768, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        CK(cudaFuncSetAttribute(tile_tma_reads<768, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        CK(cudaFuncSetAttribute(tile_tma_reads<768, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        CK(cudaFuncSetAttribute(tile_tma_reads<768, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        report("tile_tma 768 + the 16-byte read only", timed([&] { tile_tma_reads<768, 0><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, games, wr4); }));
        report("tile_tma 768 + the three 4-byte reads only", timed([&] { tile_tma_reads<768, 1><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, games, wr4); }));
        report("tile_tma 768 + reads via ld.global.cg", timed([&] { tile_tma_reads<768, 2><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, games, wr4); }));
        report("tile_tma 768 + reads (nc) not feeding the tile", timed([&] { tile_tma_reads<768, 3><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, games, wr4); }));
        report("tile_tma 768 + reads via ld.global.nc", timed([&] { tile_tma_reads<768, 4><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, games, wr4); }));
        CK(cudaFuncSetAttribute(tile_tma_bulkreads<768>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152 + 768 * 28));
        report("tile_tma 768 + the reads as four TMA bulk loads per block", timed([&] { tile_tma_bulkreads<768><<<grid, 768, 2 * 49152 + 768 * 28>>>(out, n16, 768 * 64, 3072, rd16, rd4, games); }));
        CK(cudaFuncSetAttribute(tile_tma_pipelined<768>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 49152));
        for (int tiles : {1, 2, 37, 74})
        {
            char name[96];
            snprintf(name, sizeof name, "tile_tma_pipelined 768 + reads, %d tiles per block", tiles);
            report(name, timed([&] { tile_tma_pipelined<768><<<grid / tiles, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, games, tiles); }));
        }
        CK(cudaFuncSetAttribute(tile_tma_mixed<384, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 24576));
        report("tile_tma 384 thr (4 blocks/SM, 2 x 24 KiB) + reads", timed([&] { tile_tma_mixed<384, true, false><<<(unsigned)(games / 384), 384, 2 * 24576>>>(out, n16, 384 * 64, 1536, rd16, rd4, wr16, wr4, wr1, games); }));
        report("tile_tma 768 + 34 B/game narrow side writes", timed([&] { tile_tma_mixed<768, false, true><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games); }));
        report("tile_tma 768 + reads + side writes", timed([&] { tile_tma_mixed<768, true, true><<<grid, 768, 2 * 49152>>>(out, n16, 768 * 64, 3072, rd16, rd4, wr16, wr4, wr1, games); }));
    }
    for (int kb : {64}) {
        for (int per_sm : {2}) {
            char name[96];
            snprintf(name, sizeof name, "persistent, 256 thr, %d blocks/SM, %d KiB chunks", per_sm, kb);
            report(name, timed([&] { persistent<256><<<sms * per_sm, 256>>>(out, n16, kb * 64); }));
        }
    }
    report("persistent, 1024 thr, 2 blocks/SM, 64 KiB chunks", timed([&] { persistent<1024><<<sms * 2, 1024>>>(out, n16, 64 * 64); }));
    return 0;
}

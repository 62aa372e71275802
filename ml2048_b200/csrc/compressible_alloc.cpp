// ml2048_alloc_compressible / ml2048_free_compressible: device memory the L2 may store compressed before it goes to HBM.
//
// The fp32 one-hot observation is 15/16 zeros and is written in full every step; in memory allocated with
// cuMemCreate(allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC) the L2 compresses such lines, so the step writes
// fewer DRAM bytes for the same values.  The driver functions are resolved at run time through the runtime's entry-point
// query (no -lcuda), so the library still loads where there is no driver; every failure is a return code.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>

#include <string.h>

#include "../../include/ml2048_b200.h"

namespace {

struct Driver {
    PFN_cuDeviceGetAttribute_v2000 device_get_attribute;
    PFN_cuMemGetAllocationGranularity_v10020 granularity;
    PFN_cuMemAddressReserve_v10020 address_reserve;
    PFN_cuMemAddressFree_v10020 address_free;
    PFN_cuMemCreate_v10020 create;
    PFN_cuMemRelease_v10020 release;
    PFN_cuMemMap_v10020 map;
    PFN_cuMemUnmap_v10020 unmap;
    PFN_cuMemSetAccess_v10020 set_access;
    PFN_cuMemGetAllocationPropertiesFromHandle_v10020 properties;
};

bool resolve(const char *name, unsigned version, void **fn)
{
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    return cudaGetDriverEntryPointByVersion(name, fn, version, cudaEnableDefault, &q) == cudaSuccess &&
           q == cudaDriverEntryPointSuccess && *fn;
}

// null when the driver (or one of the functions) is missing
const Driver *driver()
{
    static Driver d;
    static const bool ok = resolve("cuDeviceGetAttribute", 2000, (void **)&d.device_get_attribute) &&
                           resolve("cuMemGetAllocationGranularity", 10020, (void **)&d.granularity) &&
                           resolve("cuMemAddressReserve", 10020, (void **)&d.address_reserve) &&
                           resolve("cuMemAddressFree", 10020, (void **)&d.address_free) &&
                           resolve("cuMemCreate", 10020, (void **)&d.create) &&
                           resolve("cuMemRelease", 10020, (void **)&d.release) &&
                           resolve("cuMemMap", 10020, (void **)&d.map) &&
                           resolve("cuMemUnmap", 10020, (void **)&d.unmap) &&
                           resolve("cuMemSetAccess", 10020, (void **)&d.set_access) &&
                           resolve("cuMemGetAllocationPropertiesFromHandle", 10020, (void **)&d.properties);
    return ok ? &d : nullptr;
}

// unmap, release and unreserve whatever of `c` exists (a partly built mapping too); `c` is cleared
void teardown(const Driver &d, ml2048_compressible *c)
{
    const uint64_t chunk = c->chunks ? c->size / (uint64_t)c->chunks : 0;
    for (int i = 0; i < c->chunks; ++i) {
        if (!c->handles[i]) continue;
        if (c->ptr) d.unmap((CUdeviceptr)(c->ptr + (uint64_t)i * chunk), chunk);  // fails harmlessly on a chunk never mapped
        d.release((CUmemGenericAllocationHandle)c->handles[i]);
    }
    if (c->ptr) d.address_free((CUdeviceptr)c->ptr, c->size);
    memset(c, 0, sizeof *c);
}

// [ptr, ptr + chunks * chunk) backed by `chunks` allocations, each asking for generic compression and checked separately
int build(const Driver &d, const CUmemAllocationProp &prop, uint64_t chunk, int chunks, uint64_t gran, ml2048_compressible *c)
{
    memset(c, 0, sizeof *c);
    c->device = prop.location.id;
    c->chunks = chunks;
    c->size = chunk * (uint64_t)chunks;
    CUdeviceptr va = 0;
    CUresult r = d.address_reserve(&va, c->size, gran, 0, 0);
    if (r != CUDA_SUCCESS) return (int)r;
    c->ptr = (uint64_t)va;
    for (int i = 0; i < chunks; ++i) {
        CUmemGenericAllocationHandle h = 0;
        if ((r = d.create(&h, chunk, &prop, 0)) != CUDA_SUCCESS) break;
        c->handles[i] = (uint64_t)h;
        CUmemAllocationProp got;
        memset(&got, 0, sizeof got);
        if ((r = d.properties(&got, h)) != CUDA_SUCCESS) break;
        if (got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC) c->granted += chunk;
        if ((r = d.map(va + (CUdeviceptr)((uint64_t)i * chunk), chunk, 0, h, 0)) != CUDA_SUCCESS) break;
    }
    if (r == CUDA_SUCCESS) {
        CUmemAccessDesc acc;
        memset(&acc, 0, sizeof acc);
        acc.location = prop.location;
        acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        r = d.set_access(va, c->size, &acc, 1);
    }
    if (r != CUDA_SUCCESS) teardown(d, c);
    return (int)r;
}

}  // namespace

int ml2048_alloc_compressible(int32_t device, int64_t bytes, ml2048_compressible *out)
{
    if (!out) return ML2048_E_NULL;
    memset(out, 0, sizeof *out);
    if (bytes <= 0) return ML2048_E_SIZE;
    const Driver *d = driver();
    int count = 0;
    if (!d || cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return ML2048_E_UNSUPPORTED;
    int supported = 0;
    if (d->device_get_attribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, (CUdevice)device) != CUDA_SUCCESS ||
        !supported)
        return ML2048_E_UNSUPPORTED;
    // the driver calls act on the current context: make it the device's primary context, as the runtime does
    int prev = 0;
    if (cudaGetDevice(&prev) != cudaSuccess) return ML2048_E_UNSUPPORTED;
    if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess) {
        cudaSetDevice(prev);
        return ML2048_E_UNSUPPORTED;
    }
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof prop);
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    int rc = (int)d->granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED);
    if (rc == 0 && gran == 0) rc = ML2048_E_UNSUPPORTED;
    // one allocation; where the driver does not grant it compression, the same range from 8, then 64 equal allocations
    // (none smaller than the granularity); the last attempt stays mapped whatever it was granted
    for (int chunks = 1; rc == 0;) {
        const uint64_t per = ((uint64_t)bytes + (uint64_t)chunks - 1) / (uint64_t)chunks;
        rc = build(*d, prop, (per + gran - 1) / gran * gran, chunks, gran, out);
        const int next = chunks * 8;
        if (rc != 0 || out->granted == out->size || next > ML2048_COMPRESSIBLE_MAX_CHUNKS || (uint64_t)bytes / (uint64_t)next < gran)
            break;
        teardown(*d, out);
        chunks = next;
    }
    cudaSetDevice(prev);
    return rc;
}

int ml2048_free_compressible(ml2048_compressible *c)
{
    if (!c) return ML2048_E_NULL;
    if (!c->ptr) return 0;
    const Driver *d = driver();
    if (!d) return ML2048_E_UNSUPPORTED;
    int prev = 0;
    if (cudaGetDevice(&prev) != cudaSuccess) return ML2048_E_UNSUPPORTED;
    // work still queued on any stream may write the range: it must finish before the pages go
    int rc = (int)cudaSetDevice(c->device);
    if (rc == 0) rc = (int)cudaDeviceSynchronize();
    if (rc == 0) teardown(*d, c);
    cudaSetDevice(prev);
    return rc;
}

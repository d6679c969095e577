// Compressible device memory for observation buffers (include/marl_sat_b200.h, "observation memory").
//
// The observations are int32 words of -1 / 0 / 1 and dominate the DRAM writes of a rollout step.  Memory created
// with CU_MEM_ALLOCATION_COMP_GENERIC is compressed by the L2 on its way to DRAM and expanded on the way back, so
// kernels, copies and torch ops see the same bytes while DRAM moves fewer.  Such memory only comes from the
// driver's virtual-memory API (cuMemCreate + cuMemMap); the driver functions are resolved through the runtime's
// entry-point query so that the library keeps linking against the runtime alone.
#include <cuda.h>
#include <cuda_runtime.h>

#include <map>
#include <mutex>

#include "../../include/marl_sat_b200.h"

namespace {

struct Driver {
    decltype(&cuDeviceGet) deviceGet = nullptr;
    decltype(&cuDeviceGetAttribute) deviceGetAttribute = nullptr;
    decltype(&cuMemGetAllocationGranularity) granularity = nullptr;
    decltype(&cuMemCreate) create = nullptr;
    decltype(&cuMemGetAllocationPropertiesFromHandle) properties = nullptr;
    decltype(&cuMemRelease) release = nullptr;
    decltype(&cuMemAddressReserve) reserve = nullptr;
    decltype(&cuMemAddressFree) addressFree = nullptr;
    decltype(&cuMemMap) map = nullptr;
    decltype(&cuMemUnmap) unmap = nullptr;
    decltype(&cuMemSetAccess) setAccess = nullptr;
    bool ok = false;
};

template <class F>
bool resolve(const char* name, F& fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess || !p)
        return false;
    fn = reinterpret_cast<F>(p);
    return true;
}

const Driver& driver() {
    static const Driver d = [] {
        Driver r;
        r.ok = resolve("cuDeviceGet", r.deviceGet) && resolve("cuDeviceGetAttribute", r.deviceGetAttribute) &&
               resolve("cuMemGetAllocationGranularity", r.granularity) && resolve("cuMemCreate", r.create) &&
               resolve("cuMemGetAllocationPropertiesFromHandle", r.properties) &&
               resolve("cuMemRelease", r.release) && resolve("cuMemAddressReserve", r.reserve) &&
               resolve("cuMemAddressFree", r.addressFree) && resolve("cuMemMap", r.map) &&
               resolve("cuMemUnmap", r.unmap) && resolve("cuMemSetAccess", r.setAccess);
        return r;
    }();
    return d;
}

CUmemAllocationProp compressible_prop(int device) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    return prop;
}

struct Mapping {
    CUmemGenericAllocationHandle handle;
    size_t bytes;
};

std::mutex g_mu;
std::map<CUdeviceptr, Mapping> g_maps;          // every live mapping of msat_obs_alloc
std::map<int, int> g_granted;                   // device -> 1 compressible, 0 not; filled by the first query
std::map<int, bool> g_denied;                   // device -> an allocation came back uncompressed

// One granule created with the compressible property: the driver reports whether it honoured it.
int probe(int device, int* granted) {
    const Driver& d = driver();
    *granted = 0;
    if (!d.ok) return MSAT_OK;
    CUdevice dev;
    int supported = 0;
    if (d.deviceGet(&dev, device) != CUDA_SUCCESS) return MSAT_EINVAL;
    CUresult r = d.deviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev);
    if (r != CUDA_SUCCESS) return (int)r;
    if (!supported) return MSAT_OK;
    CUmemAllocationProp prop = compressible_prop(device), got = {};
    size_t gran = 0;
    if ((r = d.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM)) != CUDA_SUCCESS) return (int)r;
    CUmemGenericAllocationHandle h;
    if ((r = d.create(&h, gran, &prop, 0)) != CUDA_SUCCESS) return (int)r;
    r = d.properties(&got, h);
    d.release(h);
    if (r != CUDA_SUCCESS) return (int)r;
    *granted = got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
    return MSAT_OK;
}

}  // namespace

extern "C" {

int msat_obs_compression(int device, int* granted) {
    if (!granted || device < 0) return MSAT_EINVAL;
    std::lock_guard<std::mutex> lock(g_mu);
    auto it = g_granted.find(device);
    if (it == g_granted.end()) {
        int g = 0;
        int rc = probe(device, &g);
        if (rc != MSAT_OK) return rc;
        it = g_granted.emplace(device, g).first;
    }
    *granted = it->second && !g_denied[device];
    return MSAT_OK;
}

void* msat_obs_alloc(size_t size, int device, void*) {
    const Driver& d = driver();
    if (!d.ok || size == 0) return nullptr;
    CUmemAllocationProp prop = compressible_prop(device), got = {};
    size_t gran = 0;
    if (d.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS) return nullptr;
    const size_t bytes = (size + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h;
    if (d.create(&h, bytes, &prop, 0) != CUDA_SUCCESS) return nullptr;
    CUdeviceptr p = 0;
    CUmemAccessDesc access = {};
    access.location = prop.location;
    access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (d.properties(&got, h) != CUDA_SUCCESS || d.reserve(&p, bytes, gran, 0, 0) != CUDA_SUCCESS) {
        d.release(h);
        return nullptr;
    }
    if (d.map(p, bytes, 0, h, 0) != CUDA_SUCCESS) {
        d.addressFree(p, bytes);
        d.release(h);
        return nullptr;
    }
    if (d.setAccess(p, bytes, &access, 1) != CUDA_SUCCESS) {
        d.unmap(p, bytes);
        d.addressFree(p, bytes);
        d.release(h);
        return nullptr;
    }
    std::lock_guard<std::mutex> lock(g_mu);
    // the memory is usable either way; an uncompressed grant only turns msat_obs_compression off for the device
    if (got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) g_denied[device] = true;
    g_maps[p] = Mapping{h, bytes};
    return reinterpret_cast<void*>(p);
}

void msat_obs_free(void* ptr, size_t, int device, void*) {
    Mapping m;
    {
        std::lock_guard<std::mutex> lock(g_mu);
        auto it = g_maps.find(reinterpret_cast<CUdeviceptr>(ptr));
        if (it == g_maps.end()) return;
        m = it->second;
        g_maps.erase(it);
    }
    // cudaFree waits for the device before it returns memory; unmapping must not overtake queued work either
    int cur = -1;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != device) cudaSetDevice(device);
    cudaDeviceSynchronize();
    if (cur >= 0 && cur != device) cudaSetDevice(cur);
    const Driver& d = driver();
    const CUdeviceptr p = reinterpret_cast<CUdeviceptr>(ptr);
    d.unmap(p, m.bytes);
    d.release(m.handle);
    d.addressFree(p, m.bytes);
}

}  // extern "C"

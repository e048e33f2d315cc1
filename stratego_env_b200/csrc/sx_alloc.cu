// sx_alloc.cu -- device allocations of the library (sx_device_alloc / sx_device_free, include/stratego_b200.h).
//
// The engine's outputs are an almost constant image (the background of DESIGN.md section 3.1 plus a few hundred
// state-dependent bytes per game), and the fused kernel is bound by the DRAM write stream.  Memory created with
// CU_MEM_ALLOCATION_COMP_GENERIC is compressed by the memory system between L2 and DRAM, transparently to kernels,
// copy engines and torch, so such output buffers cost fewer DRAM bytes per step (DESIGN.md section 3.1).
// Driver entry points come through cudaGetDriverEntryPointByVersion: the library does not link libcuda.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <string>
#include <type_traits>
#include <map>

#include "../../include/stratego_b200.h"
#include "sx_host.h"

namespace {

struct Driver {
    bool ok = false;
    decltype(&::cuDeviceGet) DeviceGet;
    decltype(&::cuDeviceGetAttribute) DeviceGetAttribute;
    decltype(&::cuMemGetAllocationGranularity) MemGetAllocationGranularity;
    decltype(&::cuMemCreate) MemCreate;
    decltype(&::cuMemGetAllocationPropertiesFromHandle) MemGetAllocationPropertiesFromHandle;
    decltype(&::cuMemRelease) MemRelease;
    decltype(&::cuMemAddressReserve) MemAddressReserve;
    decltype(&::cuMemAddressFree) MemAddressFree;
    decltype(&::cuMemMap) MemMap;
    decltype(&::cuMemUnmap) MemUnmap;
    decltype(&::cuMemSetAccess) MemSetAccess;
};

const Driver &driver()
{
    static Driver d;
    static std::once_flag once;
    std::call_once(once, [] {
        bool ok = true;
        auto get = [&](const char *name, auto &fn) {
            cudaDriverEntryPointQueryResult q;
            void *p = nullptr;
            if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
                q != cudaDriverEntryPointSuccess || !p)
                ok = false;
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
        };
        get("cuDeviceGet", d.DeviceGet);
        get("cuDeviceGetAttribute", d.DeviceGetAttribute);
        get("cuMemGetAllocationGranularity", d.MemGetAllocationGranularity);
        get("cuMemCreate", d.MemCreate);
        get("cuMemGetAllocationPropertiesFromHandle", d.MemGetAllocationPropertiesFromHandle);
        get("cuMemRelease", d.MemRelease);
        get("cuMemAddressReserve", d.MemAddressReserve);
        get("cuMemAddressFree", d.MemAddressFree);
        get("cuMemMap", d.MemMap);
        get("cuMemUnmap", d.MemUnmap);
        get("cuMemSetAccess", d.MemSetAccess);
        cudaGetLastError();  // a missing entry point must not stay behind as the runtime's last error
        d.ok = ok;
    });
    return d;
}

struct Allocation {
    int device;
    uint64_t bytes;   // what the caller asked for
    uint64_t mapped;  // 0: cudaMalloc; else the size of the compressible mapping
};

std::mutex g_mutex;
std::map<uintptr_t, Allocation> g_allocations;  // by base address, so that an address inside can be looked up

// a compressible mapping of at least `bytes` on `device` (the current device); nullptr when the device or the driver
// does not grant generic compression
void *map_compressible(int device, uint64_t bytes, uint64_t *mapped)
{
    const Driver &drv = driver();
    if (!drv.ok) return nullptr;
    CUdevice dev;
    int supported = 0;
    if (drv.DeviceGet(&dev, device) != CUDA_SUCCESS ||
        drv.DeviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev) != CUDA_SUCCESS ||
        !supported)
        return nullptr;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if (drv.MemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM) != CUDA_SUCCESS || gran == 0)
        return nullptr;
    const uint64_t size = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle handle;
    if (drv.MemCreate(&handle, size, &prop, 0) != CUDA_SUCCESS) return nullptr;
    // the driver may hand back plain memory: only a granted compression type counts
    CUmemAllocationProp got = {};
    if (drv.MemGetAllocationPropertiesFromHandle(&got, handle) != CUDA_SUCCESS ||
        got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) {
        drv.MemRelease(handle);
        return nullptr;
    }
    CUdeviceptr va = 0;
    if (drv.MemAddressReserve(&va, size, gran, 0, 0) != CUDA_SUCCESS) {
        drv.MemRelease(handle);
        return nullptr;
    }
    CUmemAccessDesc access = {};
    access.location = prop.location;
    access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (drv.MemMap(va, size, 0, handle, 0) != CUDA_SUCCESS) {
        drv.MemAddressFree(va, size);
        drv.MemRelease(handle);
        return nullptr;
    }
    drv.MemRelease(handle);  // the mapping keeps the physical memory until it is unmapped
    if (drv.MemSetAccess(va, size, &access, 1) != CUDA_SUCCESS) {
        drv.MemUnmap(va, size);
        drv.MemAddressFree(va, size);
        return nullptr;
    }
    *mapped = size;
    return reinterpret_cast<void *>(va);
}

// runs `fn` with `device` current and puts the caller's device back
template <class F>
cudaError_t on_device(int device, F fn)
{
    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (prev != device && (e = cudaSetDevice(device)) != cudaSuccess) return e;
    e = fn();
    if (prev != device) {
        const cudaError_t r = cudaSetDevice(prev);
        if (e == cudaSuccess) e = r;
    }
    return e;
}

}  // namespace

extern "C" int sx_device_alloc(int32_t device, uint64_t bytes, uint32_t flags, void **ptr, uint32_t *granted_flags)
{
    if (!ptr) return sx_set_error("sx_device_alloc: null ptr");
    *ptr = nullptr;
    if (granted_flags) *granted_flags = 0;
    if (flags & ~uint32_t(SX_ALLOC_COMPRESSIBLE))
        return sx_set_error("sx_device_alloc: unknown flags " + std::to_string(flags));
    int n_devices = 0;
    if (cudaGetDeviceCount(&n_devices) != cudaSuccess) n_devices = 0;
    cudaGetLastError();
    if (device < 0 || device >= n_devices) return sx_set_error("sx_device_alloc: no CUDA device " + std::to_string(device));
    if (bytes == 0) bytes = 1;
    void *p = nullptr;
    uint64_t mapped = 0;
    const cudaError_t e = on_device(device, [&] {
        if (flags & SX_ALLOC_COMPRESSIBLE) p = map_compressible(device, bytes, &mapped);
        return p ? cudaSuccess : cudaMalloc(&p, bytes);
    });
    if (e != cudaSuccess) {
        cudaGetLastError();
        return sx_set_error(std::string("sx_device_alloc: ") + cudaGetErrorString(e));
    }
    {
        std::lock_guard<std::mutex> lock(g_mutex);
        g_allocations[reinterpret_cast<uintptr_t>(p)] = Allocation{device, bytes, mapped};
    }
    *ptr = p;
    if (granted_flags) *granted_flags = mapped ? SX_ALLOC_COMPRESSIBLE : 0;
    return 0;
}

extern "C" int sx_device_free(void *ptr)
{
    if (!ptr) return 0;
    Allocation a;
    {
        std::lock_guard<std::mutex> lock(g_mutex);
        auto it = g_allocations.find(reinterpret_cast<uintptr_t>(ptr));
        if (it == g_allocations.end()) return sx_set_error("sx_device_free: pointer was not allocated by sx_device_alloc (or was freed already)");
        a = it->second;
        g_allocations.erase(it);
    }
    const cudaError_t e = on_device(a.device, [&] {
        if (!a.mapped) return cudaFree(ptr);
        // unmapping does not wait for work in flight the way cudaFree does: finish it first (buffers are freed rarely)
        cudaError_t r = cudaDeviceSynchronize();
        const Driver &drv = driver();
        const CUdeviceptr va = reinterpret_cast<CUdeviceptr>(ptr);
        if (drv.MemUnmap(va, a.mapped) != CUDA_SUCCESS || drv.MemAddressFree(va, a.mapped) != CUDA_SUCCESS)
            if (r == cudaSuccess) r = cudaErrorInvalidValue;
        return r;
    });
    if (e != cudaSuccess) {
        cudaGetLastError();
        return sx_set_error(std::string("sx_device_free: ") + cudaGetErrorString(e));
    }
    return 0;
}

extern "C" int sx_device_alloc_info(const void *ptr, uint64_t *bytes, uint32_t *granted_flags, int64_t *live_allocations)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    if (live_allocations) *live_allocations = int64_t(g_allocations.size());
    if (!ptr) return 0;
    auto it = g_allocations.find(reinterpret_cast<uintptr_t>(ptr));
    if (it == g_allocations.end()) return sx_set_error("sx_device_alloc_info: pointer was not allocated by sx_device_alloc");
    if (bytes) *bytes = it->second.bytes;
    if (granted_flags) *granted_flags = it->second.mapped ? SX_ALLOC_COMPRESSIBLE : 0;
    return 0;
}

bool sx_in_compressible_allocation(const void *p)
{
    if (!p) return false;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    std::lock_guard<std::mutex> lock(g_mutex);
    auto it = g_allocations.upper_bound(a);
    if (it == g_allocations.begin()) return false;
    --it;
    return it->second.mapped && a - it->first < it->second.bytes;
}

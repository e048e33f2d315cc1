// Compressible-memory probe (development aid): does the B200's generic data compression make the engine's output
// stream cheaper?  Allocates one plain (cudaMalloc) and one compressible (cuMemCreate with
// CU_MEM_ALLOCATION_COMP_GENERIC) output buffer of 262 144 Barrage games (PO observation + mask, 8.0 GB each) and
// times the engine's output pattern into both, alternating, with the engine's launch shape (148 blocks x 8 warps,
// one game per warp, TMA bulk copies of a block-shared image, 4-byte head/tail mask words):
//   zeros      every byte 0
//   background the exact Barrage background image (67 floats per cell: 39 x 0.0, 2 x 0.5, 24 x -1.0, 2 x 0.0) +
//              an all-zero mask row
//   bg+sparse  the same, then after the copy completes 50 scattered 4-byte observation stores and 15 mask byte
//              stores per game (what the fused kernel does)
//   random     an incompressible image (a hash per word), to see what compressible memory costs when it cannot help
// Driver entry points come through cudaGetDriverEntryPointByVersion; nothing links libcuda.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o probe_compress tools/probes/probe_compress.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)
#define DK(x) do { CUresult r = (x); if (r != CUDA_SUCCESS) { printf("%s: CUresult %d\n", #x, int(r)); exit(1); } } while (0)

#define DRV(name) static decltype(&::name) p_##name;
DRV(cuDeviceGetAttribute) DRV(cuMemGetAllocationGranularity) DRV(cuMemCreate) DRV(cuMemAddressReserve) DRV(cuMemMap)
DRV(cuMemSetAccess) DRV(cuMemRetainAllocationHandle) DRV(cuMemGetAllocationPropertiesFromHandle) DRV(cuMemRelease)
DRV(cuMemUnmap) DRV(cuMemAddressFree)
static void load_driver() {
    cudaDriverEntryPointQueryResult q;
#define LOAD(name) CK(cudaGetDriverEntryPointByVersion(#name, reinterpret_cast<void **>(&p_##name), 12000, cudaEnableDefault, &q)); if (q != cudaDriverEntryPointSuccess) { printf("no %s\n", #name); exit(1); }
    LOAD(cuDeviceGetAttribute) LOAD(cuMemGetAllocationGranularity) LOAD(cuMemCreate) LOAD(cuMemAddressReserve)
    LOAD(cuMemMap) LOAD(cuMemSetAccess) LOAD(cuMemRetainAllocationHandle) LOAD(cuMemGetAllocationPropertiesFromHandle)
    LOAD(cuMemRelease) LOAD(cuMemUnmap) LOAD(cuMemAddressFree)
}

static CUmemAllocationProp device_prop(int dev, bool compressible) {
    CUmemAllocationProp p = {};
    p.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    p.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    p.location.id = dev;
    if (compressible) p.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    return p;
}

// compressible allocation; prints what the driver granted
static uint8_t *alloc_compressible(int dev, size_t bytes, size_t *mapped) {
    CUmemAllocationProp prop = device_prop(dev, true);
    size_t gran = 0;
    DK(p_cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM));
    size_t rec = 0;
    DK(p_cuMemGetAllocationGranularity(&rec, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    bytes = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h;
    DK(p_cuMemCreate(&h, bytes, &prop, 0));
    CUdeviceptr va;
    DK(p_cuMemAddressReserve(&va, bytes, gran, 0, 0));
    DK(p_cuMemMap(va, bytes, 0, h, 0));
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    DK(p_cuMemSetAccess(va, bytes, &acc, 1));
    CUmemGenericAllocationHandle h2;
    DK(p_cuMemRetainAllocationHandle(&h2, reinterpret_cast<void *>(va)));
    CUmemAllocationProp got = {};
    DK(p_cuMemGetAllocationPropertiesFromHandle(&got, h2));
    DK(p_cuMemRelease(h2));
    DK(p_cuMemRelease(h));  // the mapping keeps the memory
    printf("compressible allocation: granularity min %zu B, recommended %zu B; %zu B mapped; compressionType granted = %d (%s)\n",
           gran, rec, bytes, int(got.allocFlags.compressionType),
           got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC ? "GENERIC" : "none: plain memory");
    *mapped = bytes;
    return reinterpret_cast<uint8_t *>(va);
}

__device__ __forceinline__ uint32_t hash32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

// image: 0 zeros, 1 Barrage background, 2 random words (mask row zeros in every case but 2)
__global__ void k_fill_image(uint8_t *img, int obs_bytes, int mask_bytes, int image) {
    uint32_t *w = reinterpret_cast<uint32_t *>(img);
    for (int i = threadIdx.x; i < (obs_bytes + mask_bytes + 32) / 4; i += blockDim.x) {
        uint32_t v = 0;
        if (image == 1 && i < obs_bytes / 4) {
            const int ch = i % 67;
            v = (ch == 39 || ch == 40) ? __float_as_uint(0.5f) : (ch >= 41 && ch < 65) ? __float_as_uint(-1.0f) : 0u;
        }
        if (image == 2) v = hash32(uint32_t(i) * 2654435761u + 12345u);
        w[i] = v;
    }
}

// the engine's per-game output: TMA bulk copy of the block's image (obs 16-byte aligned; mask body 16-byte aligned,
// 4-byte head / tail words), wait for completion, then `sparse` scattered stores per game
__global__ void __launch_bounds__(512) k_emit(uint8_t *obs, uint8_t *mask, const uint8_t *image, size_t n_envs,
                                              int obs_bytes, int mask_bytes, int sparse, uint32_t seed) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const int img_bytes = obs_bytes + mask_bytes + 32;
    for (int i = threadIdx.x * 4; i < img_bytes; i += blockDim.x * 4) *reinterpret_cast<uint32_t *>(smem + i) = *reinterpret_cast<const uint32_t *>(image + i);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    const int mask_off = (obs_bytes + 15) & ~15;
    const uint32_t s_obs = (uint32_t)__cvta_generic_to_shared(smem), s_mask = s_obs + mask_off;
    for (size_t e = blockIdx.x * (size_t)wpb + warp; e < n_envs; e += (size_t)gridDim.x * wpb) {
        uint8_t *go = obs + e * obs_bytes, *gm = mask + e * mask_bytes;
        const int head = int((16 - (reinterpret_cast<uintptr_t>(gm) & 15)) & 15), body = (mask_bytes - head) & ~15, tail = mask_bytes - head - body;
        if (lane < (head >> 2)) reinterpret_cast<uint32_t *>(gm)[lane] = 0;
        if (lane >= 8 && lane - 8 < (tail >> 2)) *reinterpret_cast<uint32_t *>(gm + head + body + ((lane - 8) << 2)) = 0;
        if (lane == 0) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gm + head), "r"(s_mask + 16), "r"(body) : "memory");
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(go), "r"(s_obs), "r"(obs_bytes) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            __nanosleep(0);
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
        __syncwarp();
        if (sparse) {
            // 50 observation words (one-hot style 1.0 in channels 0..38 of random cells) + 15 mask bytes
            const uint32_t r = hash32(seed ^ uint32_t(e) * 0x9e3779b9u ^ uint32_t(lane) * 0x85ebca6bu);
            const uint32_t r2 = hash32(r + 0x68e31da4u);
            const int cells = obs_bytes / (67 * 4);
            if (lane < 25) {
                reinterpret_cast<float *>(go)[(r % cells) * 67 + (r >> 16) % 39] = 1.0f;
                reinterpret_cast<float *>(go)[(r2 % cells) * 67 + (r2 >> 16) % 39] = 1.0f;
            }
            if (lane < 15) gm[r2 % mask_bytes] = 1;
        }
    }
}

int main() {
    const int dev = 0;
    CK(cudaSetDevice(dev));
    CK(cudaFree(0));
    load_driver();
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    printf("device: %s, %d SMs\n", prop.name, prop.multiProcessorCount);
    fflush(stdout);
    if (system("nvidia-smi -i 0 --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem --format=csv") != 0) printf("nvidia-smi query failed\n");
    int vmm = 0, comp = 0;
    DK(p_cuDeviceGetAttribute(&vmm, CU_DEVICE_ATTRIBUTE_VIRTUAL_MEMORY_MANAGEMENT_SUPPORTED, dev));
    DK(p_cuDeviceGetAttribute(&comp, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
    printf("VIRTUAL_MEMORY_MANAGEMENT_SUPPORTED = %d, GENERIC_COMPRESSION_SUPPORTED = %d\n", vmm, comp);
    if (!comp) { printf("no generic compression on this device\n"); return 0; }

    const int ob = 26800, mb = 3700;
    const size_t n_envs = 262144, obs_total = n_envs * ob, bytes = obs_total + n_envs * mb;
    uint8_t *plain, *compr, *image;
    CK(cudaMalloc(&plain, bytes));
    size_t mapped = 0;
    compr = alloc_compressible(dev, bytes, &mapped);
    CK(cudaMalloc(&image, ob + mb + 64));
    CK(cudaFuncSetAttribute(k_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int warps = 8, launches = 20, rounds = 6;
    const char *names[4] = {"zeros", "background", "bg+sparse", "random"};
    for (int pat = 0; pat < 4; ++pat) {
        const int img = pat == 0 ? 0 : pat == 3 ? 2 : 1, sparse = pat == 2;
        k_fill_image<<<1, 256>>>(image, ob, mb, img);
        CK(cudaDeviceSynchronize());
        std::vector<double> t[2];
        for (int r = 0; r < rounds; ++r)
            for (int which = 0; which < 2; ++which) {
                uint8_t *base = which ? compr : plain;
                auto go = [&](int i) { k_emit<<<148, warps * 32, 48 * 1024>>>(base, base + obs_total, image, n_envs, ob, mb, sparse, 1234u + i); };
                go(0); go(1);
                CK(cudaDeviceSynchronize());
                cudaEventRecord(e0);
                for (int i = 0; i < launches; ++i) go(i);
                cudaEventRecord(e1);
                CK(cudaEventSynchronize(e1));
                CK(cudaGetLastError());
                float ms; cudaEventElapsedTime(&ms, e0, e1);
                t[which].push_back(ms / launches);
            }
        for (int which = 0; which < 2; ++which) {
            std::vector<double> v = t[which];
            std::sort(v.begin(), v.end());
            const double med = 0.5 * (v[rounds / 2 - 1] + v[rounds / 2]);
            printf("%-11s %-12s median %.4f ms  min %.4f  max %.4f  spread %.2f %%  %6.0f GB/s algorithmic  rounds:", names[pat],
                   which ? "compressible" : "plain", med, v.front(), v.back(), 100.0 * (v.back() - v.front()) / med, bytes / med / 1e6);
            for (double x : t[which]) printf(" %.4f", x);
            printf("\n");
        }
        fflush(stdout);
    }
    // the output of the last launch must be the same bytes in both buffers (compression is transparent)
    {
        std::vector<uint8_t> a(1 << 20), b(1 << 20);
        bool same = true;
        for (size_t off : {size_t(0), bytes / 2, bytes - (1 << 20)}) {
            CK(cudaMemcpy(a.data(), plain + off, a.size(), cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(b.data(), compr + off, b.size(), cudaMemcpyDeviceToHost));
            same = same && a == b;
        }
        printf("plain and compressible contents equal at three 1 MB windows: %s\n", same ? "yes" : "NO");
    }
    CK(cudaDeviceSynchronize());
    DK(p_cuMemUnmap(reinterpret_cast<CUdeviceptr>(compr), mapped));
    DK(p_cuMemAddressFree(reinterpret_cast<CUdeviceptr>(compr), mapped));
    CK(cudaFree(plain));
    CK(cudaFree(image));
    return 0;
}

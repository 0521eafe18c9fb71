// probe_compressible.cu — does Blackwell's generic L2 compression cut the DRAM bytes of k_step's Float32 observation stores?
//
// Allocates 2^20 x 800 B (the Float32 two-frame observation of 2^20 envs) twice: with cudaMalloc, and with cuMemCreate +
// CU_MEM_ALLOCATION_COMP_GENERIC (mapped with cuMemAddressReserve / cuMemMap / cuMemSetAccess).  Into each it writes, with
// k_step's store shape (one 16-byte store per thread, a warp covering 512 contiguous bytes, a CTA of 256 threads covering its
// 256 envs' 204,800 contiguous bytes), three contents:
//   obs    the observation byte pattern: (10,10,2,N) Float32 boards, 36 wall cells of -1, one food cell of 2, a few snake
//          cells of 1, zeros elsewhere (32 distinct envs, built per CTA in shared memory: no DRAM reads)
//   random random bits (the control: it cannot compress, so it must take the same time on both allocations)
//   zeros  all zero
// and times 200 launches of each (CUDA events around every launch; median and min/max), plus cudaMemset of the same size.
// Driver entry points come from cudaGetDriverEntryPoint: no -lcuda.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o probe_compressible probe_compressible.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#define CK(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e__ = (x);                                                                  \
        if (e__ != cudaSuccess) {                                                               \
            fprintf(stderr, "%s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e__)); \
            exit(1);                                                                            \
        }                                                                                       \
    } while (0)
#define CD(x)                                                                      \
    do {                                                                           \
        CUresult r__ = (x);                                                        \
        if (r__ != CUDA_SUCCESS) {                                                 \
            fprintf(stderr, "%s:%d %s -> CUresult %d\n", __FILE__, __LINE__, #x, (int)r__); \
            exit(1);                                                               \
        }                                                                          \
    } while (0)

constexpr long long N_ENVS = 1ll << 20;
constexpr size_t BYTES = (size_t)N_ENVS * 800;
constexpr int TPB = 256;
constexpr int REPS = 200;

__device__ __forceinline__ uint32_t mix(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
// value of cell k (0..99, k = r + 10c) of frame f of env e
__device__ __forceinline__ float obs_cell(uint32_t e, int f, int k) {
    const int r = k % 10, c = k / 10;
    if (r == 0 || r == 9 || c == 0 || c == 9) return -1.0f;
    const uint32_t h = mix(e * 2u + (uint32_t)f + 0x9e3779b9u);
    const int ir = r - 1, ic = c - 1;
    if (ir == (int)(h & 7u) && ic == (int)((h >> 3) & 7u)) return 2.0f;          // food
    const uint32_t hr = (h >> 6) & 7u, hc = (h >> 9) & 7u, len = 2u + ((h >> 12) & 3u);
    // a short snake lying along row hr from column hc
    return (ir == (int)hr && ic >= (int)hc && ic < (int)(hc + len)) ? 1.0f : 0.0f;
}

constexpr int VARIANTS = 32;   // distinct env observations the obs pattern cycles through (a shared-memory table: no reads)

template <int MODE>   // 0 = obs pattern, 1 = random, 2 = zeros
__global__ void __launch_bounds__(TPB) k_store(float4 *out, uint32_t salt) {
    __shared__ float4 s_obs[VARIANTS * 50];
    if (MODE == 0) {
        for (int i = threadIdx.x; i < VARIANTS * 50; i += TPB) {
            const int v = i / 50, q = i - 50 * v, f = q >= 25, k = 4 * (q - 25 * f);
            const uint32_t e = (uint32_t)v * 2654435761u + salt;
            s_obs[i] = make_float4(obs_cell(e, f, k), obs_cell(e, f, k + 1), obs_cell(e, f, k + 2), obs_cell(e, f, k + 3));
        }
        __syncthreads();
    }
    float4 *o = out + (long long)blockIdx.x * TPB * 50;
#pragma unroll 2
    for (int j = threadIdx.x; j < TPB * 50; j += TPB) {
        float4 v;
        if (MODE == 0) {
            const int e = (int)(((unsigned)j * 5243u) >> 18);      // j / 50 for j < 2^15, as in k_step
            v = s_obs[((blockIdx.x * 7 + e) & (VARIANTS - 1)) * 50 + (j - 50 * e)];
        } else if (MODE == 1) {
            const uint32_t h = mix((uint32_t)((long long)blockIdx.x * TPB * 50 + j) ^ salt);
            v = make_float4(__uint_as_float(h), __uint_as_float(mix(h + 1)), __uint_as_float(mix(h + 2)),
                            __uint_as_float(mix(h + 3)));
        } else {
            v = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        o[j] = v;
    }
}
__global__ void k_diff(const uint4 *a, const uint4 *b, size_t n, unsigned long long *bad) {
    unsigned long long c = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        uint4 x = a[i], y = b[i];
        c += (x.x != y.x) | (x.y != y.y) | (x.z != y.z) | (x.w != y.w);
    }
    if (c) atomicAdd(bad, c);
}

typedef CUresult (*PFN_GetAttr)(int *, CUdevice_attribute, CUdevice);
typedef CUresult (*PFN_Gran)(size_t *, const CUmemAllocationProp *, CUmemAllocationGranularity_flags);
typedef CUresult (*PFN_Create)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *, unsigned long long);
typedef CUresult (*PFN_Props)(CUmemAllocationProp *, CUmemGenericAllocationHandle);
typedef CUresult (*PFN_Reserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long);
typedef CUresult (*PFN_Map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
typedef CUresult (*PFN_Access)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t);
typedef CUresult (*PFN_Unmap)(CUdeviceptr, size_t);
typedef CUresult (*PFN_Free)(CUdeviceptr, size_t);
typedef CUresult (*PFN_Release)(CUmemGenericAllocationHandle);

template <typename F>
static F entry(const char *name) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    CK(cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || p == nullptr) {
        fprintf(stderr, "driver entry point %s not found\n", name);
        exit(1);
    }
    return (F)p;
}

struct Stats {
    float med, lo, hi;
};
template <typename L>
static Stats time_it(L launch) {
    for (int i = 0; i < 10; i++) launch();
    std::vector<cudaEvent_t> ev(REPS + 1);
    for (auto &e : ev) CK(cudaEventCreate(&e));
    CK(cudaEventRecord(ev[0]));
    for (int i = 0; i < REPS; i++) {
        launch();
        CK(cudaEventRecord(ev[i + 1]));
    }
    CK(cudaDeviceSynchronize());
    std::vector<float> ms(REPS);
    for (int i = 0; i < REPS; i++) CK(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
    for (auto &e : ev) CK(cudaEventDestroy(e));
    std::sort(ms.begin(), ms.end());
    return {ms[REPS / 2] * 1e3f, ms[0] * 1e3f, ms[REPS - 1] * 1e3f};
}

int main() {
    int dev = 0;
    CK(cudaSetDevice(dev));
    CK(cudaFree(0));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    printf("device: %s (sm_%d%d), %d SMs, L2 %d MB\n", prop.name, prop.major, prop.minor, prop.multiProcessorCount,
           prop.l2CacheSize >> 20);

    auto getAttr = entry<PFN_GetAttr>("cuDeviceGetAttribute");
    auto gran = entry<PFN_Gran>("cuMemGetAllocationGranularity");
    auto create = entry<PFN_Create>("cuMemCreate");
    auto props = entry<PFN_Props>("cuMemGetAllocationPropertiesFromHandle");
    auto reserve = entry<PFN_Reserve>("cuMemAddressReserve");
    auto map = entry<PFN_Map>("cuMemMap");
    auto access = entry<PFN_Access>("cuMemSetAccess");
    auto unmap = entry<PFN_Unmap>("cuMemUnmap");
    auto addrFree = entry<PFN_Free>("cuMemAddressFree");
    auto release = entry<PFN_Release>("cuMemRelease");

    int supported = 0;
    CD(getAttr(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
    printf("CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = %d\n", supported);

    CUmemAllocationProp ap = {};
    ap.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    ap.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    ap.location.id = dev;
    ap.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t g = 0;
    CD(gran(&g, &ap, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    const size_t size = (BYTES + g - 1) / g * g;
    CUmemGenericAllocationHandle h;
    CD(create(&h, size, &ap, 0));
    CUmemAllocationProp got = {};
    CD(props(&got, h));
    printf("compressible allocation: %zu bytes (granularity %zu), compressionType after cuMemCreate = %d (%s)\n", size, g,
           (int)got.allocFlags.compressionType,
           got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC ? "compressible" : "NOT compressible");
    CUdeviceptr cptr = 0;
    CD(reserve(&cptr, size, 0, 0, 0));
    CD(map(cptr, size, 0, h, 0));
    CUmemAccessDesc ad = {};
    ad.location = ap.location;
    ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    CD(access(cptr, size, &ad, 1));

    float4 *plain = nullptr;
    CK(cudaMalloc(&plain, BYTES));
    float4 *comp = reinterpret_cast<float4 *>(cptr);
    const unsigned grid = (unsigned)(N_ENVS / TPB);

    // losslessness: the same obs pattern into both, compared word by word
    unsigned long long *bad;
    CK(cudaMalloc(&bad, 8));
    CK(cudaMemset(bad, 0, 8));
    k_store<0><<<grid, TPB>>>(plain, 0);
    k_store<0><<<grid, TPB>>>(comp, 0);
    k_diff<<<4 * prop.multiProcessorCount, 512>>>((const uint4 *)plain, (const uint4 *)comp, BYTES / 16, bad);
    unsigned long long nbad = 0;
    CK(cudaMemcpy(&nbad, bad, 8, cudaMemcpyDeviceToHost));
    printf("obs pattern: %llu differing 16-byte units between the plain and the compressible buffer\n", nbad);
    CK(cudaGetLastError());

    printf("%-8s %-13s %10s %10s %10s %12s\n", "content", "allocation", "median_us", "min_us", "max_us", "GB/s(median)");
    const char *names[3] = {"obs", "random", "zeros"};
    float4 *bufs[2] = {plain, comp};
    const char *anames[2] = {"cudaMalloc", "comp_generic"};
    // alternate the allocations inside each content so that drift shows up in both
    for (int m = 0; m < 3; m++)
        for (int rep = 0; rep < 2; rep++)
            for (int b = 0; b < 2; b++) {
                uint32_t salt = 0;
                Stats s = time_it([&] {
                    if (m == 0) k_store<0><<<grid, TPB>>>(bufs[b], 0);
                    else if (m == 1) k_store<1><<<grid, TPB>>>(bufs[b], salt++);
                    else k_store<2><<<grid, TPB>>>(bufs[b], 0);
                });
                CK(cudaGetLastError());
                printf("%-8s %-13s %10.1f %10.1f %10.1f %12.0f\n", names[m], anames[b], s.med, s.lo, s.hi, BYTES / (s.med * 1e3));
            }
    for (int rep = 0; rep < 2; rep++)
        for (int b = 0; b < 2; b++) {
            Stats s = time_it([&] { CK(cudaMemsetAsync(bufs[b], 0, BYTES)); });
            printf("%-8s %-13s %10.1f %10.1f %10.1f %12.0f\n", "memset0", anames[b], s.med, s.lo, s.hi, BYTES / (s.med * 1e3));
        }
    fflush(stdout);

    CK(cudaDeviceSynchronize());
    CK(cudaFree(plain));
    CK(cudaFree(bad));
    CD(unmap(cptr, size));
    CD(addrFree(cptr, size));
    CD(release(h));
    return 0;
}

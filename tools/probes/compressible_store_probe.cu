// Drain of the 84x84 Pong rasteriser into compressible memory against ordinary memory.
//
// The same drain as pong_raster_fast_kernel<84>: persistent grid of 8-warp CTAs, a warp draws one (env, agent) stack
// from a global counter and writes its four 7 056-byte frames with 16-byte stores out of its shared-memory frame buffer
// (no rasterisation work).  65 536 envs x 2 agents, 3.7 GB per launch, into two 1.85 GB buffers (one per agent) of
// each kind:
//   cudaMalloc           ordinary device memory
//   VMM                  cuMemCreate + cuMemMap, no compression (separates the VMM mapping from compression)
//   VMM COMP_GENERIC     cuMemCreate with allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC; the granted type
//                        is read back with cuMemGetAllocationPropertiesFromHandle and printed
// Contents: every warp's frame buffer holds one frame of a pool read from a file (real frames: oracle_frames.py), all
// zeros, or random bytes.  Each row: ROUNDS rounds x LAUNCHES launches per buffer kind, the kinds alternating within a
// round; the mean of all launches and the range of the per-round means are printed.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o compressible_store_probe compressible_store_probe.cu
//   python oracle_frames.py frames.bin && ./compressible_store_probe frames.bin
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

constexpr int DD = 84 * 84, NCH = DD / 16, FRAMES = 4, WARPS = 8;
constexpr long long N_ENV = 65536;
constexpr int ROUNDS = 6, LAUNCHES = 10;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)
#define CKD(x) do { CUresult r_ = (x); if (r_ != CUDA_SUCCESS) { printf("%s: CUresult %d\n", #x, (int)r_); exit(1); } } while (0)

template <bool CS> __device__ __forceinline__ void st16(uint4* p, uint4 v) {
    if (CS) asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    else *p = v;
}

template <bool CS>
__global__ void __launch_bounds__(WARPS * 32) drain(uint8_t* obs0, uint8_t* obs1, const uint4* __restrict__ pool, int n_pool,
                                                    unsigned long long* counter) {
    extern __shared__ uint4 smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4* sm = smem + (size_t)warp * NCH;
    const int pick = (int)(((long long)(blockIdx.x * WARPS + warp) * 7919) % n_pool);
    for (int i = lane; i < NCH; i += 32) sm[i] = pool[(size_t)pick * NCH + i];
    __syncwarp();
    const long long n_stacks = N_ENV * 2;
    for (;;) {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(counter, 1ull);
        const long long s = (long long)__shfl_sync(0xffffffffu, t, 0);
        if (s >= n_stacks) break;
        uint4* out = reinterpret_cast<uint4*>(((s & 1) ? obs1 : obs0) + (size_t)(s >> 1) * FRAMES * DD);
        for (int f = 0; f < FRAMES; ++f) {
#pragma unroll
            for (int j = 0; j < (NCH + 31) / 32; ++j) {
                const int c = lane + 32 * j;
                if (c < NCH) st16<CS>(out + (size_t)f * NCH + c, sm[c]);
            }
            __syncwarp();
        }
    }
}

// driver entry points without a link dependency on libcuda
template <class F> F drv(const char* name) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    CK(cudaGetDriverEntryPointByVersion(name, &fn, 12000, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || fn == nullptr) { printf("no driver entry point %s\n", name); exit(1); }
    return reinterpret_cast<F>(fn);
}

struct Buf { uint8_t* p[2]; const char* name; int granted; };

Buf make_vmm(int dev, size_t bytes, bool compress, const char* name) {
    static auto create = drv<decltype(&cuMemCreate)>("cuMemCreate");
    static auto gran = drv<decltype(&cuMemGetAllocationGranularity)>("cuMemGetAllocationGranularity");
    static auto reserve = drv<decltype(&cuMemAddressReserve)>("cuMemAddressReserve");
    static auto map = drv<decltype(&cuMemMap)>("cuMemMap");
    static auto access = drv<decltype(&cuMemSetAccess)>("cuMemSetAccess");
    static auto props = drv<decltype(&cuMemGetAllocationPropertiesFromHandle)>("cuMemGetAllocationPropertiesFromHandle");
    Buf b{{nullptr, nullptr}, name, 0};
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof prop);
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = dev;
    if (compress) prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t g = 0;
    CKD(gran(&g, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    const size_t sz = (bytes + g - 1) / g * g;
    b.granted = 1;
    for (int a = 0; a < 2; ++a) {
        CUmemGenericAllocationHandle h;
        CKD(create(&h, sz, &prop, 0));
        CUmemAllocationProp got;
        memset(&got, 0, sizeof got);
        CKD(props(&got, h));
        if (got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) b.granted = 0;
        CUdeviceptr va = 0;
        CKD(reserve(&va, sz, g, 0, 0));
        CKD(map(va, sz, 0, h, 0));
        CUmemAccessDesc ad;
        memset(&ad, 0, sizeof ad);
        ad.location = prop.location;
        ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        CKD(access(va, sz, &ad, 1));
        b.p[a] = reinterpret_cast<uint8_t*>(va);
    }
    printf("%-22s granularity %zu B, %zu B per agent, compression %s (granted type %d)\n", name, g, sz,
           compress ? "requested" : "not requested", compress ? b.granted : 0);
    return b;
}

template <bool CS>
float time_launches(const Buf& b, const uint4* pool, int n_pool, unsigned long long* counter, int grid, int n) {
    const size_t smem = (size_t)WARPS * NCH * 16;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0));
    for (int i = 0; i < n; ++i) {
        CK(cudaMemsetAsync(counter, 0, 8));
        drain<CS><<<grid, WARPS * 32, smem>>>(b.p[0], b.p[1], pool, n_pool, counter);
    }
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaGetLastError());
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1));
    return ms / n;
}

template <bool CS>
void row(const char* contents, std::vector<Buf>& bufs, const uint4* pool, int n_pool, unsigned long long* counter, int ctas) {
    const size_t smem = (size_t)WARPS * NCH * 16;
    CK(cudaFuncSetAttribute(drain<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = 148 * ctas;
    const double bytes = (double)N_ENV * 2 * FRAMES * DD;
    std::vector<double> sum(bufs.size(), 0.0), lo(bufs.size(), 1e30), hi(bufs.size(), 0.0);
    for (size_t k = 0; k < bufs.size(); ++k) time_launches<CS>(bufs[k], pool, n_pool, counter, grid, 3);   // warm-up
    for (int r = 0; r < ROUNDS; ++r)
        for (size_t k0 = 0; k0 < bufs.size(); ++k0) {
            const size_t k = (r & 1) ? bufs.size() - 1 - k0 : k0;    // alternate the order of the kinds
            const double ms = time_launches<CS>(bufs[k], pool, n_pool, counter, grid, LAUNCHES);
            sum[k] += ms; lo[k] = ms < lo[k] ? ms : lo[k]; hi[k] = ms > hi[k] ? ms : hi[k];
        }
    for (size_t k = 0; k < bufs.size(); ++k) {
        const double ms = sum[k] / ROUNDS;
        printf("%-8s %-15s %d CTAs/SM  %-22s %.4f ms/launch (rounds %.4f-%.4f)  %5.0f GB/s  x%.3f vs %s\n", contents,
               CS ? "st.global.cs.v4" : "st.global.v4", ctas, bufs[k].name, ms, lo[k], hi[k], bytes / ms / 1e6,
               (sum[0] / ROUNDS) / ms, bufs[0].name);
    }
}

int main(int argc, char** argv) {
    if (argc < 2) { printf("usage: %s frames.bin (raw 84x84 uint8 frames)\n", argv[0]); return 2; }
    int dev = 0;
    CK(cudaSetDevice(dev));
    cudaDeviceProp dp;
    CK(cudaGetDeviceProperties(&dp, dev));
    int supported = 0;
    CK(cudaDeviceGetAttribute(&supported, (cudaDeviceAttr)CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
    printf("device %s, %d SMs, generic compression supported: %d\n", dp.name, dp.multiProcessorCount, supported);

    FILE* fp = fopen(argv[1], "rb");
    if (!fp) { printf("cannot open %s\n", argv[1]); return 2; }
    std::vector<uint8_t> real;
    uint8_t tmp[DD];
    while (fread(tmp, 1, DD, fp) == (size_t)DD) real.insert(real.end(), tmp, tmp + DD);
    fclose(fp);
    const int n_pool = (int)(real.size() / DD);
    printf("real-frame pool: %d frames from %s\n", n_pool, argv[1]);
    if (n_pool == 0) return 2;
    std::vector<uint8_t> zeros(real.size(), 0), rnd(real.size());
    std::mt19937 rng(1234);
    for (auto& v : rnd) v = (uint8_t)rng();

    const size_t per_agent = (size_t)N_ENV * FRAMES * DD;
    std::vector<Buf> bufs;
    Buf m{{nullptr, nullptr}, "cudaMalloc", 0};
    CK(cudaMalloc(&m.p[0], per_agent)); CK(cudaMalloc(&m.p[1], per_agent));
    bufs.push_back(m);
    bufs.push_back(make_vmm(dev, per_agent, false, "VMM"));
    bufs.push_back(make_vmm(dev, per_agent, supported != 0, "VMM COMP_GENERIC"));

    uint4* pool;
    unsigned long long* counter;
    CK(cudaMalloc(&pool, real.size()));
    CK(cudaMalloc(&counter, 8));
    struct { const char* name; const std::vector<uint8_t>* data; } contents[] = {{"real", &real}, {"zeros", &zeros}, {"random", &rnd}};
    for (auto& c : contents) {
        CK(cudaMemcpy(pool, c.data->data(), real.size(), cudaMemcpyHostToDevice));
        row<true>(c.name, bufs, pool, n_pool, counter, 2);
        row<false>(c.name, bufs, pool, n_pool, counter, 2);
        if (c.data == &real) row<true>(c.name, bufs, pool, n_pool, counter, 3);
    }
    return 0;
}

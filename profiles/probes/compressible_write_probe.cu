// compressible_write_probe.cu — do the step kernel's float32 rows write faster into compressible memory?
// Two buffers of the headline's [20, 1,048,576, 8, 38] float32 rows (25.5 GB): one from cuMemCreate with
// CU_MEM_ALLOCATION_COMP_GENERIC, one from cudaMalloc.  Every warp writes groups of 32 envs (38,912 B) the way
// tpe_emit_group_tma does: 1,216-byte cp.async.bulk images, at most 3 in flight per warp, L2 evict_first.  The
// images come from a group of real rows staged once in the CTA's shared memory, so the probe times the memory
// system, not the building of the rows.  Variants: evict_normal instead of evict_first; one 38,912-byte image
// per group.  Data sets: real rows (profiles/probes/oracle_rows.py), all-zero rows, random bytes.
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o compressible_write_probe compressible_write_probe.cu \
//        -L/usr/local/cuda/lib64/stubs -lcuda
//   python profiles/probes/oracle_rows.py /tmp/rows.bin && ./compressible_write_probe /tmp/rows.bin
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda.h>
#include <cuda_runtime.h>

constexpr int kEnvBytes = 1216;                  // 8 agents x 38 float32
constexpr int kGroupBytes = 32 * kEnvBytes;      // 38,912 B: one warp's 32 envs
constexpr int kSrcGroups = 1024;                 // 32,768 envs of source rows
constexpr long long kGroups = 20LL * 1048576 / 32;
constexpr size_t kBytes = (size_t)kGroups * kGroupBytes;   // 25,501,368,320 B
constexpr int kWarps = 8;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); exit(1); } } while (0)
#define DK(x) do { CUresult r_ = (x); if (r_ != CUDA_SUCCESS) { const char *s_; cuGetErrorString(r_, &s_); printf("%s:%d %s\n", __FILE__, __LINE__, s_); exit(1); } } while (0)

// group g is written by warp g % (gridDim.x * kWarps); its CTA stages source group blockIdx.x % kSrcGroups
template <int IMG, int RING, bool EVICT_FIRST>
__global__ void __launch_bounds__(kWarps * 32) write_rows(unsigned char *out, const unsigned char *src) {
    extern __shared__ __align__(128) unsigned char tile[];   // [kGroupBytes]
    const uint4 *s = reinterpret_cast<const uint4 *>(src + (size_t)(blockIdx.x % kSrcGroups) * kGroupBytes);
    for (int i = threadIdx.x; i < kGroupBytes / 16; i += blockDim.x) reinterpret_cast<uint4 *>(tile)[i] = s[i];
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    const int lane = threadIdx.x & 31;
    if (lane != 0) return;
    unsigned long long pol;
    if (EVICT_FIRST) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    const unsigned tile_s = (unsigned)__cvta_generic_to_shared(tile);
    const long long warps = (long long)gridDim.x * kWarps;
    for (long long g = blockIdx.x * kWarps + (threadIdx.x >> 5); g < kGroups; g += warps) {
        unsigned char *dst = out + g * kGroupBytes;
        for (int b = 0; b < kGroupBytes / IMG; ++b) {
            asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(RING - 1) : "memory");
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                         ::"l"(dst + b * IMG), "r"(tile_s + b * IMG), "n"(IMG), "l"(pol) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__global__ void read_rows(const uint4 *in, size_t n, unsigned *sink) {
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = __ldcs(in + i);
        acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
    }
    sink[blockIdx.x * blockDim.x + threadIdx.x] = acc.x ^ acc.y ^ acc.z ^ acc.w;
}

struct Pattern { const char *name; void (*launch)(unsigned char *, const unsigned char *, int); };

template <int IMG, int RING, bool EF>
void launch(unsigned char *out, const unsigned char *src, int sms) {
    auto k = write_rows<IMG, RING, EF>;
    static int ctas = 0;
    if (!ctas) {
        CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kGroupBytes));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, k, kWarps * 32, kGroupBytes));
        printf("  (%d B images, ring %d, %s: %d CTAs/SM)\n", IMG, RING, EF ? "evict_first" : "evict_normal", ctas);
    }
    k<<<sms * ctas, kWarps * 32, kGroupBytes>>>(out, src);
}

static float time_ms(void (*fn)(unsigned char *, const unsigned char *, int), unsigned char *out, const unsigned char *src, int sms, int reps) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    fn(out, src, sms);   // warm-up
    CK(cudaEventRecord(e0));
    for (int r = 0; r < reps; ++r) fn(out, src, sms);
    CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1)); CK(cudaGetLastError());
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return ms / reps;
}

static unsigned *g_sink;
static void read_launch(unsigned char *out, const unsigned char *, int sms) {
    read_rows<<<sms * 4, 512>>>(reinterpret_cast<const uint4 *>(out), kBytes / 16, g_sink);
}

int main(int argc, char **argv) {
    if (argc < 2) { printf("usage: %s ROWS.bin   (raw float32 [32768, 8, 38], profiles/probes/oracle_rows.py)\n", argv[0]); return 2; }
    DK(cuInit(0));
    CUdevice dev; DK(cuDeviceGet(&dev, 0));
    CK(cudaSetDevice(0)); CK(cudaFree(nullptr));
    {
        char name[256]; DK(cuDeviceGetName(name, sizeof name, dev));
        int comp = 0, sms = 0, clk = 0;
        DK(cuDeviceGetAttribute(&comp, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
        DK(cuDeviceGetAttribute(&sms, CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT, dev));
        DK(cuDeviceGetAttribute(&clk, CU_DEVICE_ATTRIBUTE_CLOCK_RATE, dev));
        printf("device %s, %d SMs, max SM clock %d MHz, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = %d\n", name, sms, clk / 1000, comp);
        fflush(stdout);
        // read-only query of the power limit and the current clocks
        if (std::system("nvidia-smi -i 0 --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,memory.used,memory.total --format=csv")) printf("(nvidia-smi not available)\n");
    }
    int sms; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));

    // ---- source rows ------------------------------------------------------------------------------------------------
    const size_t src_bytes = (size_t)kSrcGroups * kGroupBytes;
    std::vector<unsigned char> real(src_bytes), rnd(src_bytes);
    FILE *f = fopen(argv[1], "rb");
    if (!f || fread(real.data(), 1, src_bytes, f) != src_bytes) { printf("cannot read %zu B of rows from %s\n", src_bytes, argv[1]); return 2; }
    fclose(f);
    uint64_t x = 0x9E3779B97F4A7C15ull;
    for (size_t i = 0; i < src_bytes; i += 8) { x ^= x << 13; x ^= x >> 7; x ^= x << 17; memcpy(&rnd[i], &x, 8); }
    unsigned char *src_real, *src_zero, *src_rnd;
    CK(cudaMalloc(&src_real, src_bytes)); CK(cudaMalloc(&src_zero, src_bytes)); CK(cudaMalloc(&src_rnd, src_bytes));
    CK(cudaMemcpy(src_real, real.data(), src_bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(src_rnd, rnd.data(), src_bytes, cudaMemcpyHostToDevice));
    CK(cudaMemset(src_zero, 0, src_bytes));
    CK(cudaMalloc(&g_sink, (size_t)sms * 4 * 512 * 4));

    // ---- the two buffers --------------------------------------------------------------------------------------------
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = 0;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    DK(cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    const size_t padded = (kBytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h;
    DK(cuMemCreate(&h, padded, &prop, 0));
    CUmemAllocationProp got = {};
    DK(cuMemGetAllocationPropertiesFromHandle(&got, h));
    CUdeviceptr cptr;
    DK(cuMemAddressReserve(&cptr, padded, gran, 0, 0));
    DK(cuMemMap(cptr, padded, 0, h, 0));
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    DK(cuMemSetAccess(cptr, padded, &acc, 1));
    printf("compressible buffer: %zu B (granularity %zu B), requested compressionType %d, granted compressionType %d\n",
           padded, gran, (int)prop.allocFlags.compressionType, (int)got.allocFlags.compressionType);
    unsigned char *comp = reinterpret_cast<unsigned char *>(cptr), *plain;
    CK(cudaMalloc(&plain, kBytes));
    CK(cudaMemset(comp, 0, kBytes)); CK(cudaMemset(plain, 0, kBytes)); CK(cudaDeviceSynchronize());
    fflush(stdout);

    const Pattern pats[] = {
        {"1216 B images, ring 3, evict_first (kernel)", launch<kEnvBytes, 3, true>},
        {"1216 B images, ring 3, evict_normal", launch<kEnvBytes, 3, false>},
        {"38912 B image per group, evict_first", launch<kGroupBytes, 1, true>},
        {"38912 B image per group, evict_normal", launch<kGroupBytes, 1, false>},
    };
    const struct { const char *name; const unsigned char *src; } data[] = {{"real rows", src_real}, {"zero rows", src_zero}, {"random bytes", src_rnd}};
    const int np = sizeof pats / sizeof pats[0], nd = 3, rounds = 3, reps = 3;
    // wr[d][p][alloc][round], rd[d][p][alloc][round]: GB/s
    std::vector<float> wr(nd * np * 2 * rounds), rd(nd * np * 2 * rounds);
    for (int r = 0; r < rounds; ++r)
        for (int d = 0; d < nd; ++d)
            for (int p = 0; p < np; ++p)
                for (int a = 0; a < 2; ++a) {   // plain, compressible alternately
                    unsigned char *buf = a ? comp : plain;
                    const float w = time_ms(pats[p].launch, buf, data[d].src, sms, reps);
                    const float rr = time_ms(read_launch, buf, nullptr, sms, reps);
                    const int i = ((d * np + p) * 2 + a) * rounds + r;
                    wr[i] = kBytes / 1e6 / w;
                    rd[i] = kBytes / 1e6 / rr;
                }
    // the compressible buffer holds what was written: last write was random bytes, group image, evict_normal
    {
        std::vector<unsigned char> back(kGroupBytes);
        int ctas = 0; CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, write_rows<kGroupBytes, 1, false>, kWarps * 32, kGroupBytes));
        const long long warps = (long long)sms * ctas * kWarps;
        int bad = 0;
        for (const unsigned char *s : {src_real, src_zero, src_rnd}) {
            launch<kGroupBytes, 1, false>(comp, s, sms);
            CK(cudaDeviceSynchronize());
            const std::vector<unsigned char> &host = s == src_real ? real : (s == src_rnd ? rnd : std::vector<unsigned char>(src_bytes, 0));
            for (long long g : {0LL, 1LL, 12345LL, kGroups / 2 + 7, kGroups - 1}) {
                CK(cudaMemcpy(back.data(), comp + g * kGroupBytes, kGroupBytes, cudaMemcpyDeviceToHost));
                const long long sg = ((g % warps) / kWarps) % kSrcGroups;
                bad += memcmp(back.data(), host.data() + sg * kGroupBytes, kGroupBytes) != 0;
            }
        }
        printf("read-back of 15 groups from the compressible buffer: %s\n", bad ? "MISMATCH" : "identical to the source rows");
    }
    printf("\nlogical GB/s (25.5 GB per launch, mean of %d launches after a warm-up), rounds 1..%d, then the median\n", reps, rounds);
    for (int d = 0; d < nd; ++d)
        for (int p = 0; p < np; ++p) {
            float med[2][2];
            for (int a = 0; a < 2; ++a) {
                for (int k = 0; k < 2; ++k) {
                    const float *v = (k ? rd : wr).data() + ((d * np + p) * 2 + a) * rounds;
                    float t[3] = {v[0], v[1], v[2]};
                    std::sort(t, t + 3);
                    med[a][k] = t[1];
                }
                const float *w = wr.data() + ((d * np + p) * 2 + a) * rounds, *q = rd.data() + ((d * np + p) * 2 + a) * rounds;
                printf("%-13s %-44s %-12s write %7.0f %7.0f %7.0f -> %7.0f | read %7.0f %7.0f %7.0f -> %7.0f\n", data[d].name, pats[p].name,
                       a ? "compressible" : "plain", w[0], w[1], w[2], med[a][0], q[0], q[1], q[2], med[a][1]);
            }
            printf("%-13s %-44s compressible / plain: write %.3f, read %.3f\n", data[d].name, pats[p].name, med[1][0] / med[0][0], med[1][1] / med[0][1]);
        }
    CK(cudaFree(plain));
    DK(cuMemUnmap(cptr, padded)); DK(cuMemAddressFree(cptr, padded)); DK(cuMemRelease(h));
    return 0;
}

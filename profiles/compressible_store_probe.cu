// Does the L2's generic compression shorten k_obs's write stream on this B200?  k_obs is bound by its HBM writes (fp32
// view rows, mostly zeros).  This probe times k_obs's store loop -- 37 856-byte shared->global bulk stores, two staging
// buffers, 256 threads and 2 CTAs per SM, 8 chunks per dynamic ticket -- into plain cudaMalloc memory and into memory
// from cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC, alternated, for three payloads: all zeros, dense random bits,
// and real C3 view rows (view.npy of `bench.py --workload c3 --dump-outputs DIR`).  Each CTA loads two chunks of the
// payload into its staging buffers once (CTA b: payload chunks 2b and 2b+1, cycled) and then only stores, so the loop
// runs at the store rate, as k_obs's does.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/compressible_store_probe profiles/compressible_store_probe.cu -lcuda
//   /tmp/compressible_store_probe [DIR/view.npy]
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)
#define DK(x) do { CUresult r_ = (x); if (r_ != CUDA_SUCCESS) { const char *s_; cuGetErrorString(r_, &s_); printf("%s: %s\n", #x, s_); exit(1); } } while (0)

constexpr uint32_t kChunk = 8 * 13 * 13 * 7 * 4;          // 37 856 B: 8 view rows, one bulk store
constexpr int kThreads = 256, kPerTicket = 8;
constexpr size_t kAllocBytes = 524288ull * 4868;          // C3's view + feature blocks: 2.552 GB
constexpr size_t kChunks = 524288 / 8;                    // C3's view rows, 8 per chunk: 2.481 GB written

__global__ void __launch_bounds__(kThreads, 2)
k_store(char *out, const uint4 *src, size_t src_chunks, unsigned long long *ticket) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x;
    for (int b = 0; b < 2; b++) {
        const uint4 *s = src + ((2 * blockIdx.x + b) % src_chunks) * (kChunk / 16);
        for (uint32_t i = tid; i < kChunk / 16; i += kThreads) ((uint4 *)(smem + (size_t)b * kChunk))[i] = s[i];
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid != 0) return;
    int b = 0;
    for (;;) {
        const size_t first = (size_t)atomicAdd(ticket, 1ull) * kPerTicket;
        if (first >= kChunks) break;
        for (size_t c = first; c < first + kPerTicket && c < kChunks; c++, b ^= 1) {
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(out + c * kChunk), "r"((uint32_t)__cvta_generic_to_shared(smem + (size_t)b * kChunk)),
                            "r"(kChunk) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

static std::vector<float> load_npy_f32(const char *path) {
    FILE *f = fopen(path, "rb");
    if (!f) { printf("cannot open %s\n", path); exit(1); }
    unsigned char pre[10];
    if (fread(pre, 1, 10, f) != 10 || memcmp(pre, "\x93NUMPY", 6) != 0) { printf("%s: not an .npy file\n", path); exit(1); }
    size_t hlen = pre[8] | (pre[9] << 8);
    if (pre[6] >= 2) { unsigned char x[2]; if (fread(x, 1, 2, f) != 2) exit(1); hlen |= (size_t)(x[0] | (x[1] << 8)) << 16; }
    std::string hdr(hlen, ' ');
    if (fread(&hdr[0], 1, hlen, f) != hlen) exit(1);
    if (hdr.find("'<f4'") == std::string::npos || hdr.find("'fortran_order': False") == std::string::npos) {
        printf("%s: want little-endian float32 in C order, got %s\n", path, hdr.c_str()); exit(1);
    }
    const long start = ftell(f);
    fseek(f, 0, SEEK_END);
    const size_t n = (size_t)(ftell(f) - start) / 4;
    fseek(f, start, SEEK_SET);
    std::vector<float> v(n);
    if (fread(v.data(), 4, n, f) != n) exit(1);
    fclose(f);
    printf("payload %s: %s\n", path, hdr.c_str());
    return v;
}

struct Mem { char *ptr; size_t size; CUmemGenericAllocationHandle h; bool vmm; int compressed; };

static Mem alloc_compressible(size_t bytes, int dev) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = dev;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    DK(cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    Mem m = {};
    m.size = (bytes + gran - 1) / gran * gran;
    m.vmm = true;
    CUdeviceptr p;
    DK(cuMemAddressReserve(&p, m.size, 0, 0, 0));
    DK(cuMemCreate(&m.h, m.size, &prop, 0));
    CUmemAllocationProp got = {};
    DK(cuMemGetAllocationPropertiesFromHandle(&got, m.h));
    m.compressed = got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
    DK(cuMemMap(p, m.size, 0, m.h, 0));
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    DK(cuMemSetAccess(p, m.size, &acc, 1));
    m.ptr = (char *)p;
    printf("cuMemCreate %zu B (granularity %zu B): compressionType granted = %d (%s)\n", m.size, gran,
           (int)got.allocFlags.compressionType, m.compressed ? "COMP_GENERIC" : "COMP_NONE");
    return m;
}

static void free_mem(Mem &m) {
    if (!m.vmm) { CK(cudaFree(m.ptr)); return; }
    DK(cuMemUnmap((CUdeviceptr)m.ptr, m.size));
    DK(cuMemRelease(m.h));
    DK(cuMemAddressFree((CUdeviceptr)m.ptr, m.size));
}

int main(int argc, char **argv) {
    CK(cudaSetDevice(0));
    cudaDeviceProp dp;
    CK(cudaGetDeviceProperties(&dp, 0));
    int sms = dp.multiProcessorCount, comp_attr = 0;
    CUdevice cdev;
    DK(cuDeviceGet(&cdev, 0));
    DK(cuDeviceGetAttribute(&comp_attr, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, cdev));
    printf("device: %s, %d SMs\n", dp.name, sms);
    if (FILE *p = popen("nvidia-smi -i 0 --query-gpu=power.limit,clocks.max.sm --format=csv,noheader", "r")) {
        char line[256];
        if (fgets(line, sizeof line, p)) printf("power limit, max SM clock: %s", line);
        pclose(p);
    }
    printf("CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = %d\n", comp_attr);

    Mem plain = {};
    plain.size = kAllocBytes;
    CK(cudaMalloc(&plain.ptr, plain.size));
    Mem comp = alloc_compressible(kAllocBytes, 0);

    // payloads: whole chunks, at most 64 MB
    struct Payload { const char *name; std::vector<uint32_t> words; };
    std::vector<Payload> payloads;
    const size_t syn_chunks = 1024, syn_words = syn_chunks * kChunk / 4;
    payloads.push_back({"zeros", std::vector<uint32_t>(syn_words, 0u)});
    {
        std::mt19937 rng(12345);
        std::vector<uint32_t> w(syn_words);
        for (auto &x : w) x = rng();
        payloads.push_back({"dense random", std::move(w)});
    }
    if (argc > 1) {
        std::vector<float> v = load_npy_f32(argv[1]);
        size_t words = std::min(v.size(), (size_t)(64 << 20) / 4) / (kChunk / 4) * (kChunk / 4);
        if (words == 0) { printf("%s holds less than one chunk\n", argv[1]); return 1; }
        std::vector<uint32_t> w(words);
        memcpy(w.data(), v.data(), words * 4);
        payloads.push_back({"C3 view rows", std::move(w)});
    }
    for (auto &p : payloads) {
        size_t nz = 0, zero_sectors = 0, sectors = p.words.size() / 8;
        for (uint32_t x : p.words) nz += x != 0;
        for (size_t s = 0; s < sectors; s++) {
            bool z = true;
            for (int k = 0; k < 8; k++) z &= p.words[s * 8 + k] == 0;
            zero_sectors += z;
        }
        printf("payload %-13s %5zu chunks (%.1f MB): %.1f %% non-zero words, %.1f %% all-zero 32-byte sectors\n", p.name,
               p.words.size() * 4 / kChunk, p.words.size() * 4 / 1e6, 100.0 * nz / p.words.size(), 100.0 * zero_sectors / sectors);
    }

    const int smem = 2 * kChunk;
    CK(cudaFuncSetAttribute(k_store, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_store, kThreads, smem));
    const int grid = sms * std::min(per_sm, 2);
    printf("k_store: %d CTAs (%d per SM) x %d threads, %d B staging, %zu chunks = %.3f GB per launch\n\n", grid,
           grid / sms, kThreads, smem, kChunks, kChunks * kChunk / 1e9);
    unsigned long long *ticket;
    CK(cudaMalloc(&ticket, 8));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    auto run = [&](Mem &m, const uint4 *src, size_t src_chunks) {
        CK(cudaMemsetAsync(ticket, 0, 8));
        CK(cudaEventRecord(e0));
        k_store<<<grid, kThreads, smem>>>(m.ptr, src, src_chunks, ticket);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        CK(cudaGetLastError());
        float ms;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        return ms;
    };
    const int reps = 7;
    std::vector<double> gains;
    for (auto &p : payloads) {
        const size_t src_chunks = p.words.size() * 4 / kChunk;
        uint4 *src;
        CK(cudaMalloc(&src, p.words.size() * 4));
        CK(cudaMemcpy(src, p.words.data(), p.words.size() * 4, cudaMemcpyHostToDevice));
        run(plain, src, src_chunks); run(comp, src, src_chunks);            // warm-up
        std::vector<float> tp, tc;
        for (int r = 0; r < reps; r++) { tp.push_back(run(plain, src, src_chunks)); tc.push_back(run(comp, src, src_chunks)); }
        // the bytes that landed: a spread of chunks read back from both allocations, each must be a payload chunk
        // (which one depends on the CTA that took the ticket)
        bool ok = true;
        std::vector<unsigned char> a(kChunk);
        for (Mem *m : {&plain, &comp})
            for (size_t c : {(size_t)0, kChunks / 3, kChunks / 2 + 7, kChunks - 1}) {
                CK(cudaMemcpy(a.data(), m->ptr + c * kChunk, kChunk, cudaMemcpyDeviceToHost));
                bool found = false;
                for (size_t k = 0; k < src_chunks && !found; k++)
                    found = memcmp(a.data(), (const unsigned char *)p.words.data() + k * kChunk, kChunk) == 0;
                ok &= found;
            }
        std::sort(tp.begin(), tp.end()); std::sort(tc.begin(), tc.end());
        const double bytes = (double)kChunks * kChunk;
        printf("%-13s plain        median %.4f ms  [%.4f .. %.4f]  %5.0f GB/s\n", p.name, tp[reps / 2], tp[0], tp[reps - 1], bytes / tp[reps / 2] / 1e6);
        printf("%-13s compressible median %.4f ms  [%.4f .. %.4f]  %5.0f GB/s  -> %.3fx plain  (read-back %s)\n", p.name,
               tc[reps / 2], tc[0], tc[reps - 1], bytes / tc[reps / 2] / 1e6, tp[reps / 2] / tc[reps / 2], ok ? "matches" : "MISMATCH");
        gains.push_back(tp[reps / 2] / tc[reps / 2]);
        CK(cudaFree(src));
    }
    if (argc > 1)
        printf("\ngate (C3 view rows, compressible >= 1.15x plain): %s (%.3fx)\n", gains.back() >= 1.15 ? "GO" : "NO-GO", gains.back());
    free_mem(comp);
    free_mem(plain);
    CK(cudaFree(ticket));
    return 0;
}

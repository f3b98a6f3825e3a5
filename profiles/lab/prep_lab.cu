// prep_lab.cu - development micro-benchmark for the first kernel of the pipeline (not part of the library).
// Times k_prep (the TMA-ring kernel of the batch pipeline) against the general kernel, a plain copy with the same
// traffic pattern and a device memcpy of the same bytes, on device-generated sky frames or on the bench pool
// (LAB_DATA=1 after dump_pool.py), and checks that the kernels write identical planes and histograms.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -std=c++17 -lineinfo prep_lab.cu -o prep_lab
#include <vector>
#include <string>
#include <cstdlib>
#include <cstring>
#include "../../lfd_b200/csrc/k_prep.cuh"

#define CKL(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e_), __LINE__); exit(1); } } while (0)

__device__ __forceinline__ u32 hash32(u32 x) { x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16; return x; }

// sky noise sigma 0.025 + a few bright blobs + special values
__global__ void k_gen(float* out, size_t n, int W, u32 seed)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        u32 h1 = hash32((u32)i * 2u + seed), h2 = hash32((u32)i * 2u + 1u + seed);
        float u1 = (h1 + 1.0f) * 2.3283064e-10f, u2 = h2 * 2.3283064e-10f;
        float v = 0.025f * sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
        u32 h3 = hash32(h1 ^ 0x9e3779b9u);
        if ((h3 & 0x3ff) == 0) v += (float)(h3 >> 24) * 0.03f;            // star-like pixels up to ~7.6
        if ((h3 & 0xfffff) == 1) v = 300.0f + (float)(h3 >> 20);          // saturating pixels
        if ((h3 & 0xffffff) == 2) v = __int_as_float(0x7fc00000);         // NaN
        if ((h3 & 0xffffff) == 3) v = __int_as_float(0x7f800000);         // inf
        if ((h3 & 0xffffff) == 4) v = 3.0e9f;
        if ((h3 & 0xffffff) == 5) v = 254.5f;
        if ((h3 & 0xffffff) == 6) v = 0.5f;
        if ((h3 & 0xffffff) == 7) v = 1.0f;                                // 1.0 + 0.5 -> 1.5 -> 2 (half even)
        out[i] = v;
    }
}

__global__ void k_gen_mask(u32* m, size_t n, u32 seed)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        u32 h = hash32((u32)(i >> 3) + seed);       // blobs of 8 words
        m[i] = ((h & 0x3f) == 0) ? hash32((u32)i) | 0xff00u : 0u;
    }
}

// byte-swapped copy of the frames: the raw FITS payload the big-endian path reads
__global__ void k_bswap(const u32* __restrict__ in, u32* __restrict__ out, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = __byte_perm(in[i], 0, 0x0123);
}

// reads 16 B, writes 8 B per thread-iteration: the traffic pattern of the prep stage without any arithmetic
__global__ void __launch_bounds__(256) k_plain(const float4* __restrict__ in, uint2* __restrict__ out, size_t n4)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        float4 v = __ldcs(in + i);
        out[i] = make_uint2(__float_as_uint(v.x) & 0x01010101u, __float_as_uint(v.z) & 0x01010101u);
    }
}

int main(int argc, char** argv)
{
    const int B = argc > 1 ? atoi(argv[1]) : 64;
    const int H = 1489, W = 2048;
    Dims d; d.H = H; d.W = W; d.WW = (W + 31) / 32; d.N = H * W; d.NW = H * d.WW;
    float *in, *in_be; u32* mask; u8 *g0[2], *g1[2]; u32* hist[2];
    CKL(cudaMalloc(&in, (size_t)B * d.N * 4));
    CKL(cudaMalloc(&in_be, (size_t)B * d.N * 4));
    CKL(cudaMalloc(&mask, (size_t)B * d.NW * 4));
    for (int k = 0; k < 2; k++) {
        CKL(cudaMalloc(&g0[k], (size_t)B * d.N)); CKL(cudaMalloc(&g1[k], (size_t)B * d.N));
        CKL(cudaMalloc(&hist[k], (size_t)2 * B * 256 * 4));
    }
    void* scratch; CKL(cudaMalloc(&scratch, (size_t)B * d.N * 3));
    k_gen<<<148 * 8, 256>>>(in, (size_t)B * d.N, W, 12345u);
    k_gen_mask<<<148 * 8, 256>>>(mask, (size_t)B * d.NW, 777u);
    CKL(cudaDeviceSynchronize());
    if (getenv("LAB_DATA")) {            // real bench frames written by dump_pool.py
        std::vector<char> buf((size_t)B * d.N * 4);
        FILE* fi = fopen("/tmp/lab_in.bin", "rb"); FILE* fm = fopen("/tmp/lab_mask.bin", "rb");
        if (!fi || !fm) { printf("no /tmp/lab_in.bin\n"); return 1; }
        if (fread(buf.data(), 1, buf.size(), fi) != buf.size()) { printf("short read\n"); return 1; }
        CKL(cudaMemcpy(in, buf.data(), buf.size(), cudaMemcpyHostToDevice));
        size_t mb = (size_t)B * d.NW * 4;
        if (fread(buf.data(), 1, mb, fm) != mb) { printf("short mask read\n"); return 1; }
        CKL(cudaMemcpy(mask, buf.data(), mb, cudaMemcpyHostToDevice));
        fclose(fi); fclose(fm);
        printf("using the bench pool from /tmp\n");
    }
    k_bswap<<<148 * 8, 256>>>(reinterpret_cast<const u32*>(in), reinterpret_cast<u32*>(in_be), (size_t)B * d.N);
    CKL(cudaDeviceSynchronize());
    const float minFlux = 0.02f, addFlux = 0.5f;
    cudaDeviceProp prop; CKL(cudaGetDeviceProperties(&prop, 0));
    const int nsm = prop.multiProcessorCount;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);

    struct Var { std::string name; int id; bool check; };
    std::vector<Var> vars = {{"k_prep_generic (reference)", 0, true}, {"k_prep 3 CTAs/SM G=16 (library)", 316, true}, {"k_prep 3 CTAs/SM G=32", 332, true},
                             {"k_prep 4 CTAs/SM G=16", 116, true}, {"k_prep 4 CTAs/SM G=24", 124, true}, {"k_prep 4 CTAs/SM G=32", 132, true},
                             {"k_prep 4 CTAs/SM G=B", 100 + B, true}, {"plain copy 16B->8B", 20, false}, {"memcpy d2d same bytes", 21, false}};
    int per_sm = 0;
    CKL(cudaFuncSetAttribute(k_prep<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM));
    CKL(cudaFuncSetAttribute(k_prep<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM));
    CKL(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_prep<0, false>, PR_WARPS * 32, PR_SMEM));
    printf("k_prep: %d B dynamic smem, %d CTAs/SM\n", (int)PR_SMEM, per_sm);
    // be: the k_prep variants read the byte-swapped copy; the general kernel always reads the native frames
    auto launch = [&](int id, int slot, int be) {
        u32* h0 = hist[slot]; u32* h1 = hist[slot] + (size_t)B * 256;
        const float* src = be ? in_be : in;
        if (id == 0) {
            int pblocks = (d.N / 4 + 255) / 256; if (pblocks > 1184) pblocks = 1184;
            k_prep_generic<<<dim3(pblocks, B), 256>>>(in, mask, g0[slot], g1[slot], h0, h1, nullptr, d, 0, minFlux, addFlux);
        } else if (id >= 100 && id <= 199) {
            const int G = id - 100 > B ? B : id - 100;
            int rb = nsm * 4 / G; if (rb < 1) rb = 1;
            auto kk = be ? k_prep<0, true, 4> : k_prep<0, false, 4>;
            cudaFuncSetAttribute(kk, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM);
            kk<<<dim3(rb, G), PR_WARPS * 32, PR_SMEM>>>(src, mask, g0[slot], g1[slot], h0, h1, d, B, minFlux, addFlux);
        }
        else if (id >= 200 && id <= 399) {
            const int mb = id / 100, G = id % 100 > B ? B : id % 100;
            auto kk = mb == 3 ? (be ? k_prep<0, true, 3> : k_prep<0, false, 3>) : k_prep<0, false, 2>;   // (100 + G selects the library default)
            cudaFuncSetAttribute(kk, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM);
            int rb = nsm * mb / G; if (rb < 1) rb = 1;
            kk<<<dim3(rb, G), PR_WARPS * 32, PR_SMEM>>>(src, mask, g0[slot], g1[slot], h0, h1, d, B, minFlux, addFlux);
        }
        else if (id == 20) k_plain<<<nsm * 8, 256>>>(reinterpret_cast<const float4*>(in), reinterpret_cast<uint2*>(scratch), (size_t)B * d.N / 4);
        else if (id == 21) cudaMemcpyAsync(scratch, in, (size_t)B * d.N * 3, cudaMemcpyDeviceToDevice, 0);
    };
    // reference outputs from the general kernel (the one the standalone write-back path uses)
    CKL(cudaMemset(hist[0], 0, (size_t)2 * B * 256 * 4));
    launch(0, 0, 0);
    CKL(cudaDeviceSynchronize());
    std::vector<u8> r0((size_t)B * d.N), r1((size_t)B * d.N), t0((size_t)B * d.N), t1((size_t)B * d.N);
    std::vector<u32> rh((size_t)2 * B * 256), th((size_t)2 * B * 256);
    CKL(cudaMemcpy(r0.data(), g0[0], r0.size(), cudaMemcpyDeviceToHost));
    CKL(cudaMemcpy(r1.data(), g1[0], r1.size(), cudaMemcpyDeviceToHost));
    CKL(cudaMemcpy(rh.data(), hist[0], rh.size() * 4, cudaMemcpyDeviceToHost));
    const double bytes = (double)B * d.N * 6.0;
    const char* only = getenv("LAB_ONLY");
    const int R = getenv("LAB_R") ? atoi(getenv("LAB_R")) : 20;
    for (auto& v : vars) {
        if (only && !strstr(only, ("," + std::to_string(v.id) + ",").c_str())) continue;
        CKL(cudaMemset(hist[1], 0, (size_t)2 * B * 256 * 4));
        CKL(cudaMemset(g0[1], 0xee, (size_t)B * d.N)); CKL(cudaMemset(g1[1], 0xee, (size_t)B * d.N));
        launch(v.id, 1, 0);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { printf("%-32s FAILED: %s\n", v.name.c_str(), cudaGetErrorString(e)); return 1; }
        std::string verdict = "n/a";
        if (v.check) {
            CKL(cudaMemcpy(t0.data(), g0[1], t0.size(), cudaMemcpyDeviceToHost));
            CKL(cudaMemcpy(t1.data(), g1[1], t1.size(), cudaMemcpyDeviceToHost));
            CKL(cudaMemcpy(th.data(), hist[1], th.size() * 4, cudaMemcpyDeviceToHost));
            size_t bad0 = 0, bad1 = 0, badh = 0;
            for (size_t i = 0; i < t0.size(); i++) { bad0 += t0[i] != r0[i]; bad1 += t1[i] != r1[i]; }
            for (size_t i = 0; i < th.size(); i++) badh += th[i] != rh[i];
            verdict = (bad0 | bad1 | badh) ? "MISMATCH g0=" + std::to_string(bad0) + " g1=" + std::to_string(bad1) + " hist=" + std::to_string(badh) : "identical";
        }
        for (int i = 0; i < 3; i++) launch(v.id, 1, 0);
        CKL(cudaDeviceSynchronize());
        cudaEventRecord(e0);
        for (int i = 0; i < R; i++) launch(v.id, 1, 0);
        cudaEventRecord(e1);
        CKL(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        printf("%-32s %8.1f us  %7.1f GB/s  frac %.3f  %s\n", v.name.c_str(), 1e3 * ms / R, bytes / (ms / R * 1e-3) * 1e-9,
               bytes / (ms / R * 1e-3) * 1e-9 / 6553.9, verdict.c_str());
    }
    // big-endian input path: k_prep<0, true> on the byte-swapped copy against the general kernel on the native frames
    {
        CKL(cudaMemset(hist[0], 0, (size_t)2 * B * 256 * 4)); CKL(cudaMemset(hist[1], 0, (size_t)2 * B * 256 * 4));
        launch(0, 0, 0); launch(316, 1, 1);
        CKL(cudaDeviceSynchronize());
        CKL(cudaMemcpy(r0.data(), g0[0], r0.size(), cudaMemcpyDeviceToHost)); CKL(cudaMemcpy(t0.data(), g0[1], t0.size(), cudaMemcpyDeviceToHost));
        CKL(cudaMemcpy(r1.data(), g1[0], r1.size(), cudaMemcpyDeviceToHost)); CKL(cudaMemcpy(t1.data(), g1[1], t1.size(), cudaMemcpyDeviceToHost));
        CKL(cudaMemcpy(rh.data(), hist[0], rh.size() * 4, cudaMemcpyDeviceToHost)); CKL(cudaMemcpy(th.data(), hist[1], th.size() * 4, cudaMemcpyDeviceToHost));
        size_t bad = 0, badh = 0, shown = 0;
        for (size_t i = 0; i < t0.size(); i++) {
            const bool b = (t0[i] != r0[i]) || (t1[i] != r1[i]);
            bad += b;
            if (b && shown < 8) {
                shown++;
                u32 raw; CKL(cudaMemcpy(&raw, reinterpret_cast<u32*>(in) + ((i / d.N) * (size_t)d.N + (size_t)(d.H - 1 - (i % d.N) / d.W) * d.W + (i % d.W)), 4, cudaMemcpyDeviceToHost));
                printf("  px %zu native 0x%08x generic (%d,%d) k_prep (%d,%d)\n", i, raw, r0[i], r1[i], t0[i], t1[i]);
            }
        }
        for (size_t i = 0; i < th.size(); i++) badh += th[i] != rh[i];
        printf("big-endian input, k_prep vs k_prep_generic: %s (%zu px, %zu bins)\n", (bad | badh) ? "MISMATCH" : "identical", bad, badh);
    }
    return 0;
}

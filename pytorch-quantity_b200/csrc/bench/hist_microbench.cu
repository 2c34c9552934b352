// hist_microbench.cu -- design-space probe for the statistics kernels on B200.
// Standalone (no torch): generates data on the device, times each variant with CUDA events,
// prints GB/s of algorithmic traffic (4 B/element).  Not part of libpq_sm100.so.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --fmad=false -I../../../include -I.. \
//        hist_microbench.cu -o hist_microbench
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "pq_stats_kernels.cuh"

using namespace pq;

__device__ __forceinline__ unsigned int hash32(unsigned int x)
{
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}

// kind 0: bell (sum of 6 uniforms, signed, dense)  1: relu(bell)  2: constant 1.0  3: uniform(-1,1)
__global__ void gen_kernel(float *x, size_t n, int kind, unsigned int seed)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float acc = 0.f;
        unsigned int h = hash32((unsigned int)i * 2654435761u + seed);
        for (int k = 0; k < 6; ++k) { h = hash32(h + k); acc += (h >> 8) * (1.0f / 16777216.0f); }
        float v = acc - 3.0f;
        if (kind == 1) v = v > 0 ? v : 0.f;
        if (kind == 2) v = 1.0f;
        if (kind == 3) v = (hash32(h) >> 8) * (2.0f / 16777216.0f) - 1.0f;
        x[i] = v;
    }
}

// ---- ceiling: same streaming loop, trivial math -------------------------------------------
__global__ void __launch_bounds__(kStatThreads) read_only_kernel(const float4 *x, size_t nvec, float *out)
{
    float s = 0.f;
    const size_t per = (nvec / kChunkVecs + gridDim.x - 1) / gridDim.x;
    size_t c = blockIdx.x * per, ce = min(c + per, nvec / kChunkVecs);
    for (; c < ce; ++c) {
        float4 v[kVecPerThread];
#pragma unroll
        for (int i = 0; i < kVecPerThread; ++i) v[i] = ld_stream_f4(x + c * kChunkVecs + threadIdx.x + i * kStatThreads);
#pragma unroll
        for (int i = 0; i < kVecPerThread; ++i) s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    if (s == 123.456f) *out = s;
}

// ---- experimental histogram variants over one flat tensor ----------------------------------
// MODE 0: IEEE div + smem atomics (COPIES warp-private copies)      == production arithmetic
// MODE 1: reciprocal multiply (inexact) + smem atomics              -> cost of the division
// MODE 2: IEEE div, no atomics (xor into a register)                -> cost of the atomics
template <int MODE, int COPIES, int THREADS>
__global__ void __launch_bounds__(THREADS) hist_variant_kernel(const float4 *x, size_t nvec, float interval,
                                                              unsigned long long *hist)
{
    extern __shared__ unsigned int sh[];
    for (int i = threadIdx.x; i < COPIES * 2048; i += THREADS) sh[i] = 0;
    __syncthreads();
    unsigned int *mine = sh + ((threadIdx.x >> 5) % COPIES) * 2048;
    const float rcp = 1.0f / interval;
    unsigned int sink = 0;
    constexpr int CV = THREADS * kVecPerThread;
    const size_t nchunk = nvec / CV;
    const size_t per = (nchunk + gridDim.x - 1) / gridDim.x;
    size_t c = blockIdx.x * per, ce = min(c + per, nchunk);
    for (; c < ce; ++c) {
        float4 v[kVecPerThread];
#pragma unroll
        for (int i = 0; i < kVecPerThread; ++i) v[i] = ld_stream_f4(x + c * CV + threadIdx.x + i * THREADS);
#pragma unroll
        for (int i = 0; i < kVecPerThread; ++i) {
            float e[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (e[k] != 0.f) {
                    float q = MODE == 1 ? fabsf(e[k]) * rcp : __fdiv_rn(fabsf(e[k]), interval);
                    int idx = q >= 2047.f ? 2047 : (int)q;
                    if (MODE == 2) sink ^= idx; else atomicAdd(mine + idx, 1u);
                }
            }
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < 2048; b += THREADS) {
        unsigned int cnt = 0;
        for (int k = 0; k < COPIES; ++k) cnt += sh[k * 2048 + b];
        if (cnt) atomicAdd(hist + b, (unsigned long long)cnt);
    }
    if (sink == 0xdeadbeef) hist[0] = sink;
}

// MODE lane16: 32 lane-private copies of 16-bit packed counters (128 KB): bank == lane, so an
// ATOMS never has a bank conflict whatever the data.  Flushed before a 16-bit counter can wrap.
template <int THREADS>
__global__ void __launch_bounds__(THREADS) hist_lane16_kernel(const float4 *x, size_t nvec, float interval,
                                                             unsigned long long *hist)
{
    extern __shared__ unsigned int sh[];       // [1024][32] words, two 16-bit counters per word
    for (int i = threadIdx.x; i < 1024 * 32; i += THREADS) sh[i] = 0;
    __syncthreads();
    const unsigned int lane = threadIdx.x & 31;
    constexpr int CV = THREADS * kVecPerThread;
    constexpr int kFlushEvery = 65535 / ((THREADS / 32) * kVecPerThread * 4);   // chunks per flush
    const size_t nchunk = nvec / CV;
    const size_t per = (nchunk + gridDim.x - 1) / gridDim.x;
    size_t c = blockIdx.x * per, ce = min(c + per, nchunk);
    int since = 0;
    while (true) {
        if (c < ce) {
            float4 v[kVecPerThread];
#pragma unroll
            for (int i = 0; i < kVecPerThread; ++i) v[i] = ld_stream_f4(x + c * CV + threadIdx.x + i * THREADS);
#pragma unroll
            for (int i = 0; i < kVecPerThread; ++i) {
                float e[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (e[k] != 0.f) {
                        float q = __fdiv_rn(fabsf(e[k]), interval);
                        unsigned int idx = q >= 2047.f ? 2047u : (unsigned int)(int)q;
                        atomicAdd(sh + ((idx & 1023u) << 5) + lane, 1u << ((idx >> 10) << 4));
                    }
                }
            }
            ++c; ++since;
        }
        if (since == kFlushEvery || c >= ce) {
            __syncthreads();
            for (int b = threadIdx.x; b < 1024; b += THREADS) {
                unsigned int lo = 0, hi = 0;
                for (int l = 0; l < 32; ++l) {
                    unsigned int w = sh[(b << 5) + ((l + lane) & 31)];   // rotate: conflict-free reads
                    lo += w & 0xffffu; hi += w >> 16;
                    sh[(b << 5) + ((l + lane) & 31)] = 0;
                }
                if (lo) atomicAdd(hist + b, (unsigned long long)lo);
                if (hi) atomicAdd(hist + 1024 + b, (unsigned long long)hi);
            }
            __syncthreads();
            since = 0;
            if (c >= ce) break;
        }
    }
}

template <typename F>
float time_ms(F launch, int iters = 10)
{
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    for (int i = 0; i < 3; ++i) launch();
    cudaEventRecord(a);
    for (int i = 0; i < iters; ++i) launch();
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float ms; cudaEventElapsedTime(&ms, a, b);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(e)); exit(1); }
    return ms / iters;
}

template <int MODE, int COPIES, int THREADS>
void run_variant(const char *name, const float *x, size_t n, float interval, unsigned long long *hist, int ctas_per_sm)
{
    size_t smem = (size_t)COPIES * 2048 * 4;
    auto k = hist_variant_kernel<MODE, COPIES, THREADS>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, THREADS, smem);
    if (ctas_per_sm > occ) ctas_per_sm = occ;
    float ms = time_ms([&] { k<<<148 * ctas_per_sm, THREADS, smem>>>((const float4 *)x, n / 4, interval, hist); });
    printf("  %-34s %8.3f ms  %8.1f GB/s  (occ %d CTA/SM)\n", name, ms, n * 4.0 / ms / 1e6, ctas_per_sm);
}

int main(int argc, char **argv)
{
    size_t n = (size_t)1 << 28;
    if (argc > 1) n = (size_t)atoll(argv[1]);
    float *x; unsigned long long *hist; float *out; unsigned int *mx;
    cudaMalloc(&x, n * 4); cudaMalloc(&hist, 2048 * 8 * 4); cudaMalloc(&out, 4); cudaMalloc(&mx, 64);
    const char *kinds[] = {"bell (dense, signed)", "relu(bell) (50% zeros)", "constant 1.0 (one bin)", "uniform(-1,1)"};
    for (int kind = 0; kind < 4; ++kind) {
        gen_kernel<<<148 * 8, 256>>>(x, n, kind, 1234u + kind);
        cudaMemset(mx, 0, 64);
        // production absmax through the ABI-level table
        SegTable t; t.k = 1; t.ptr[0] = x; t.n[0] = n; t.param[0] = 0.f;
        t.chunk_end[0] = (unsigned int)seg_num_chunks(x, n); t.total_chunks = t.chunk_end[0];
        float ms = time_ms([&] { absmax_multi_kernel<<<148 * 8, kStatThreads>>>(t, mx); });
        unsigned int bits; cudaMemcpy(&bits, mx, 4, cudaMemcpyDeviceToHost);
        float maxv; memcpy(&maxv, &bits, 4);
        float interval = maxv / 2048.f + 1e-12f;
        printf("== %s: n=%zu max=%g interval=%g\n", kinds[kind], n, maxv, interval);
        printf("  %-34s %8.3f ms  %8.1f GB/s\n", "absmax (production)", ms, n * 4.0 / ms / 1e6);
        ms = time_ms([&] { read_only_kernel<<<148 * 8, kStatThreads>>>((const float4 *)x, n / 4, out); });
        printf("  %-34s %8.3f ms  %8.1f GB/s\n", "read-only ceiling", ms, n * 4.0 / ms / 1e6);
        t.param[0] = interval;
        {
            auto k8 = hist_multi_kernel<1, 8>;
            cudaFuncSetAttribute(k8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_smem_bytes(1));
            for (int cps = 3; cps <= 4; ++cps) {
                ms = time_ms([&] { k8<<<148 * cps, kStatThreads, hist_smem_bytes(1)>>>(t, hist); });
                printf("  production fast-div VPT=8, %d CTA/SM   %8.3f ms  %8.1f GB/s\n", cps, ms, n * 4.0 / ms / 1e6);
            }
        }
        run_variant<0, 1, 256>("ieee-div, 1 copy, 256thr", x, n, interval, hist, 8);
        run_variant<0, 2, 256>("ieee-div, 2 copies, 256thr", x, n, interval, hist, 8);
        run_variant<0, 4, 512>("ieee-div, 4 copies, 512thr", x, n, interval, hist, 4);
        run_variant<1, 2, 256>("rcp-mul (inexact), 2 copies", x, n, interval, hist, 8);
        run_variant<2, 2, 256>("ieee-div, NO atomics", x, n, interval, hist, 8);
        {
            auto k = hist_lane16_kernel<512>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
            ms = time_ms([&] { k<<<148, 512, 128 * 1024>>>((const float4 *)x, n / 4, interval, hist); });
            printf("  %-34s %8.3f ms  %8.1f GB/s\n", "lane-private 16-bit, 512thr 1/SM", ms, n * 4.0 / ms / 1e6);
            auto k2 = hist_lane16_kernel<1024>;
            cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
            ms = time_ms([&] { k2<<<148, 1024, 128 * 1024>>>((const float4 *)x, n / 4, interval, hist); });
            printf("  %-34s %8.3f ms  %8.1f GB/s\n", "lane-private 16-bit, 1024thr 1/SM", ms, n * 4.0 / ms / 1e6);
        }
    }
    return 0;
}

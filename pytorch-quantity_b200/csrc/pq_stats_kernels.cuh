// pq_stats_kernels.cuh -- activation / weight statistics kernels (subsystem 1):
//   absmax_multi_kernel : per-tensor max |x|           (distribution_collector.py:70-78)
//   hist_multi_kernel   : 2048-bin |x| histograms      (distribution_collector.py:127-135)
//
// Both are HBM-bound streaming kernels: 4 algorithmic bytes per element per pass.
// One launch covers up to PQ_MAX_SEGMENTS tensors.  Every tensor is cut into chunks of
// kChunkElems elements; each CTA owns a CONTIGUOUS range of chunks, so it touches the
// fewest possible tensors and publishes its private result once per tensor it touched.
#pragma once
#include "pq_common.cuh"

namespace pq {

constexpr int kStatThreads = 256;
constexpr int kVecPerThread = 8;                                 // float4 loads in flight per thread
constexpr int kChunkVecs = kStatThreads * kVecPerThread;         // 2048 float4
constexpr int kChunkElems = kChunkVecs * 4;                      // 8192 elements = 32 KB

// Geometry of one segment: scalar head up to the first 16-byte boundary, float4 body, scalar tail.
struct SegGeom {
    const float *p;
    unsigned long long n;
    unsigned int head;              // scalar elements before the aligned body
    unsigned long long nvec;        // float4 count of the body
    const float4 *body;
    unsigned int tail;              // scalar elements after the body
};

__device__ __forceinline__ SegGeom seg_geom(const SegTable &t, int s)
{
    SegGeom g;
    g.p = t.ptr[s];
    g.n = t.n[s];
    unsigned long long addr = (unsigned long long)g.p;
    unsigned long long head = ((16ull - (addr & 15ull)) & 15ull) >> 2;
    g.head = (unsigned int)(head < g.n ? head : g.n);
    g.nvec = (g.n - g.head) >> 2;
    g.body = reinterpret_cast<const float4 *>(g.p + g.head);
    g.tail = (unsigned int)(g.n - g.head - (g.nvec << 2));
    return g;
}

__host__ __device__ inline unsigned int seg_num_chunks(const float *p, unsigned long long n)
{
    unsigned long long addr = (unsigned long long)p;
    unsigned long long head = ((16ull - (addr & 15ull)) & 15ull) >> 2;
    if (head > n) head = n;
    unsigned long long nvec = (n - head) >> 2;
    unsigned long long c = (nvec + kChunkVecs - 1) / kChunkVecs;
    return (unsigned int)(c ? c : 1);
}

// ------------------------------------------------------------------------------ absmax
__device__ __forceinline__ unsigned int absbits(float v) { return __float_as_uint(v) & 0x7fffffffu; }

// Publish the CTA's maximum of the per-thread values m into *dst: warp redux, ONE atomic per CTA.  Every thread of
// the kStatThreads-wide CTA must call it; s_warp is [kStatThreads / 32] shared words, free again on return.
__device__ __forceinline__ void block_max_publish(unsigned int m, unsigned int *s_warp, unsigned int *dst)
{
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned int w = threadIdx.x < kStatThreads / 32 ? s_warp[threadIdx.x] : 0u;
        w = __reduce_max_sync(0xffffffffu, w);
        if (threadIdx.x == 0 && w != 0) atomicMax(dst, w);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kStatThreads)
absmax_multi_kernel(const __grid_constant__ SegTable tab, unsigned int *__restrict__ max_bits)
{
    __shared__ unsigned int s_warp[kStatThreads / 32];
    const unsigned int per = (tab.total_chunks + gridDim.x - 1) / gridDim.x;
    unsigned int c = blockIdx.x * per;
    const unsigned int c_end = min(c + per, tab.total_chunks);
    if (c >= c_end) return;

    int seg = seg_of_chunk(tab, c);
    unsigned int m = 0;
    while (c < c_end) {
        const SegGeom g = seg_geom(tab, seg);
        const unsigned int seg_first = seg ? tab.chunk_end[seg - 1] : 0;
        const unsigned int seg_last = min(tab.chunk_end[seg], c_end);
        for (; c < seg_last; ++c) {
            const unsigned long long v0 = (unsigned long long)(c - seg_first) * kChunkVecs;
            const float4 *src = g.body + v0;
            const unsigned long long left = g.nvec > v0 ? g.nvec - v0 : 0;
            if (left >= (unsigned long long)kChunkVecs) {
                float4 v[kVecPerThread];
#pragma unroll
                for (int i = 0; i < kVecPerThread; ++i) v[i] = ld_stream_f4(src + threadIdx.x + i * kStatThreads);
#pragma unroll
                for (int i = 0; i < kVecPerThread; ++i)
                    m = max(max(m, max(absbits(v[i].x), absbits(v[i].y))), max(absbits(v[i].z), absbits(v[i].w)));
            } else {
                for (unsigned int i = threadIdx.x; i < (unsigned int)left; i += kStatThreads) {
                    float4 v = ld_stream_f4(src + i);
                    m = max(max(m, max(absbits(v.x), absbits(v.y))), max(absbits(v.z), absbits(v.w)));
                }
            }
            if (c == seg_first) {   // the segment's first chunk also owns the unaligned head / tail
                if (threadIdx.x < g.head) m = max(m, absbits(g.p[threadIdx.x]));
                if (threadIdx.x < g.tail) m = max(m, absbits(g.p[g.n - g.tail + threadIdx.x]));
            }
        }
        block_max_publish(m, s_warp, max_bits + seg);      // this CTA's maximum for the segment
        m = 0;
        ++seg;
    }
}

// ------------------------------------------------------------------- per-channel absmax
// Extension of a1 (no reference counterpart): max |x| per channel of a contiguous
// [outer][channels][inner] tensor.  Same streaming skeleton as absmax_multi_kernel (32 KB chunks,
// 8 x LDG.128 in flight per thread, 4 algorithmic bytes per element); the extra work is finding the
// channel of every float4 without dividing.  A CTA owns a contiguous chunk range, so it divides once
// (64-bit) for its first element and afterwards only needs quotients of numbers below inner + 2^13:
// those come from a multiply-shift with a host-computed 32-bit magic (exact for numerators < 2^31,
// Granlund-Montgomery round-up method).  Maxima are kept per CTA in a shared [channels] array;
// a warp whose 32 float4 lie in one plane (the common case: inner >= 128) folds them with one
// redux.sync and issues ONE shared atomic.
struct ChannelGeom {
    unsigned long long total;       // outer * channels * inner
    unsigned int inner, channels;
    unsigned int m_inner, m_chan;   // magics
    int s_inner, s_chan;            // shifts (31 + ceil(log2 d))
};

__device__ __forceinline__ unsigned int magic_div(unsigned int n, unsigned int m, int s)
{
    return (unsigned int)(((unsigned long long)n * m) >> s);
}

// slow path: the four elements of a float4 that straddles a plane boundary (or inner < 4)
__device__ __forceinline__ void chan_add_straddle(unsigned int *smax, const float4 &v, unsigned int rem, unsigned int ch,
                                                  const ChannelGeom &g)
{
    const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        while (rem >= g.inner) {
            rem -= g.inner;
            if (++ch == g.channels) ch = 0;
        }
        atomicMax(smax + ch, absbits(e[j]));
        ++rem;
    }
}

__global__ void __launch_bounds__(kStatThreads)
absmax_per_channel_kernel(const float *__restrict__ x, const ChannelGeom g, unsigned int head,
                          unsigned long long nvec, unsigned int tail, unsigned int total_chunks,
                          unsigned int *__restrict__ max_bits)
{
    extern __shared__ unsigned int s_cmax[];               // [channels]
    const unsigned int per = (total_chunks + gridDim.x - 1) / gridDim.x;
    unsigned int c = blockIdx.x * per;
    const unsigned int c_end = min(c + per, total_chunks);
    if (c >= c_end) return;
    for (unsigned int i = threadIdx.x; i < g.channels; i += kStatThreads) s_cmax[i] = 0;
    __syncthreads();

    const float4 *body = reinterpret_cast<const float4 *>(x + head);
    // position of this CTA's first body element: plane remainder r0 (< inner) and channel ch0
    const unsigned long long e0 = (unsigned long long)head + (unsigned long long)c * kChunkElems;
    const unsigned long long p0 = e0 / g.inner;
    unsigned int r0 = (unsigned int)(e0 - p0 * g.inner);
    unsigned int ch0 = (unsigned int)(p0 % g.channels);

    for (; c < c_end; ++c) {
        const unsigned long long v0 = (unsigned long long)c * kChunkVecs;
        const float4 *src = body + v0;
        const unsigned long long left = nvec > v0 ? nvec - v0 : 0;
        if (left >= (unsigned long long)kChunkVecs) {
            float4 v[kVecPerThread];
#pragma unroll
            for (int i = 0; i < kVecPerThread; ++i) v[i] = ld_stream_f4(src + threadIdx.x + i * kStatThreads);
#pragma unroll
            for (int i = 0; i < kVecPerThread; ++i) {
                const unsigned int r = r0 + 4u * (threadIdx.x + i * kStatThreads);
                const unsigned int q = magic_div(r, g.m_inner, g.s_inner);
                const unsigned int rem = r - q * g.inner;
                unsigned int ch = ch0 + q;
                ch -= magic_div(ch, g.m_chan, g.s_chan) * g.channels;
                const unsigned int m4 = max(max(absbits(v[i].x), absbits(v[i].y)), max(absbits(v[i].z), absbits(v[i].w)));
                const bool whole = rem + 3u < g.inner;     // all four elements in plane `ch`
                int same;
                __match_all_sync(0xffffffffu, ch, &same);
                if (same && __all_sync(0xffffffffu, whole)) {
                    const unsigned int m = __reduce_max_sync(0xffffffffu, m4);
                    if ((threadIdx.x & 31) == 0) atomicMax(s_cmax + ch, m);
                } else if (whole) {
                    atomicMax(s_cmax + ch, m4);
                } else {
                    chan_add_straddle(s_cmax, v[i], rem, ch, g);
                }
            }
        } else {                                           // last, partial chunk: no warp collectives
            for (unsigned int i = threadIdx.x; i < (unsigned int)left; i += kStatThreads) {
                const float4 w = ld_stream_f4(src + i);
                const unsigned int r = r0 + 4u * i;
                const unsigned int q = magic_div(r, g.m_inner, g.s_inner);
                unsigned int ch = ch0 + q;
                ch -= magic_div(ch, g.m_chan, g.s_chan) * g.channels;
                chan_add_straddle(s_cmax, w, r - q * g.inner, ch, g);
            }
        }
        // advance the CTA's base position by one chunk
        r0 += kChunkElems;
        const unsigned int q = magic_div(r0, g.m_inner, g.s_inner);
        r0 -= q * g.inner;
        ch0 += q;
        ch0 -= magic_div(ch0, g.m_chan, g.s_chan) * g.channels;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {             // the unaligned head / tail scalars (<= 3 each)
        for (unsigned int j = 0; j < head + tail; ++j) {
            const unsigned long long e = j < head ? j : g.total - tail + (j - head);
            atomicMax(s_cmax + (unsigned int)((e / g.inner) % g.channels), absbits(x[e]));
        }
    }
    __syncthreads();
    for (unsigned int i = threadIdx.x; i < g.channels; i += kStatThreads) {
        const unsigned int m = s_cmax[i];
        if (m) atomicMax(max_bits + i, m);
    }
}

// Per-channel absmax, "periodic" variant for small planes (inner < 784: 7x7 feature maps, [N][C] matrices), where
// the kernel above spends its time in per-float4 channel arithmetic and shared atomics (0.62-0.73 of HBM peak).
// One image = channels * inner = P elements with P % 4 == 0, so float4 number j of EVERY image covers the same (at
// most four) channels: a thread owns one float4 column j, walks the images with eight loads in flight keeping four
// running maxima in registers, and only at the end looks up its channels (four real divisions per thread) and
// folds them through a per-CTA shared array (a CTA's 1024 consecutive elements span <= 1024 / inner + 2 channels)
// into one global atomicMax per touched channel.  grid = (float4 columns / 256, image groups).
constexpr int kPerRows = 8;

__global__ void __launch_bounds__(kStatThreads)
absmax_periodic_kernel(const float4 *__restrict__ x, unsigned int vec_per_img, unsigned int images, unsigned int inner,
                       unsigned int *__restrict__ max_bits)
{
    __shared__ unsigned int s_cmax[kStatThreads * 4 + 2];
    for (unsigned int i = threadIdx.x; i < kStatThreads * 4 + 2; i += kStatThreads) s_cmax[i] = 0;
    __syncthreads();
    const unsigned int j = blockIdx.x * kStatThreads + threadIdx.x;
    const unsigned int ch_base = (blockIdx.x * kStatThreads * 4u) / inner;     // channel of the CTA's first element
    if (j < vec_per_img) {
        unsigned int m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        const unsigned int step = gridDim.y;
        unsigned int r = blockIdx.y;
        for (; r + (kPerRows - 1) * step < images; r += kPerRows * step) {
            float4 v[kPerRows];
#pragma unroll
            for (int i = 0; i < kPerRows; ++i) v[i] = ld_stream_f4(x + (size_t)(r + i * step) * vec_per_img + j);
#pragma unroll
            for (int i = 0; i < kPerRows; ++i) {
                m0 = max(m0, absbits(v[i].x)); m1 = max(m1, absbits(v[i].y));
                m2 = max(m2, absbits(v[i].z)); m3 = max(m3, absbits(v[i].w));
            }
        }
        for (; r < images; r += step) {
            const float4 w = ld_stream_f4(x + (size_t)r * vec_per_img + j);
            m0 = max(m0, absbits(w.x)); m1 = max(m1, absbits(w.y)); m2 = max(m2, absbits(w.z)); m3 = max(m3, absbits(w.w));
        }
        const unsigned int e = 4u * j;
        atomicMax(s_cmax + (e / inner - ch_base), m0);
        atomicMax(s_cmax + ((e + 1u) / inner - ch_base), m1);
        atomicMax(s_cmax + ((e + 2u) / inner - ch_base), m2);
        atomicMax(s_cmax + ((e + 3u) / inner - ch_base), m3);
    }
    __syncthreads();
    for (unsigned int i = threadIdx.x; i < kStatThreads * 4 + 2; i += kStatThreads) {
        const unsigned int m = s_cmax[i];
        if (m) atomicMax(max_bits + ch_base + i, m);
    }
}

// ------------------------------------------------------------- calibration forward epilogues
// The elementwise glue around the convolutions of the fp32 calibration forward, one pass each instead of ATen's two
// or three (bias add, ReLU) plus the pass-1 re-read of absmax_multi_kernel:
//   out = a + (bias[channel] or b[i]),   relu_out = relu(out) (optional),   *max_slot = max(*max_slot, bits(max |out|))
// Bit for bit what the unfused forward computes: one IEEE fp32 add (ATen's a + 1 * b), ReLU as ATen's clamp_min
// (NaN passes, else max(v, 0)), and absmax_multi_kernel's order-free integer max over |out| bit patterns.
//   EPI_BIAS4 : the conv epilogue in place (out == a), plane size H*W % 4 == 0: a float4 never leaves its plane, so
//               its channel is two multiply-shift divisions of the float4 index (hw = float4 per plane)
//   EPI_BIAS1 : the same for any plane size (7x7): the channel is found for the first element of the float4 and
//               stepped for the other three (hw = elements per plane)
//   EPI_ADD   : Eltwise, out = a + b out of place
// Grid-stride over float4 with kEpiUnroll float4 per operand in flight per thread; n % 4 tail scalars in CTA 0.
enum EpiMode { EPI_BIAS4 = 0, EPI_BIAS1 = 1, EPI_ADD = 2 };
constexpr int kEpiUnroll = 4;

struct EpiArgs {
    const float *a;             // EPI_BIAS*: the conv output, == out
    const float *b;             // EPI_BIAS*: bias [channels]; EPI_ADD: second addend [n]
    float *out;
    float *relu_out;            // may be null
    unsigned int *max_slot;     // may be null
    unsigned long long n;       // elements; n / 4 < 2^31 (EPI_BIAS1: n < 2^31)
    unsigned int hw, channels;
    unsigned int m_hw, m_chan;  // magic31 multipliers of hw and channels
    int s_hw, s_chan;
};

// ATen's clamp_min(v, 0) (launch_clamp_scalar): NaN propagates, otherwise max(v, 0)
__device__ __forceinline__ float relu_aten(float v) { return isnan(v) ? v : fmaxf(v, 0.0f); }

template <int MODE>
__device__ __forceinline__ float4 epi_load_a(const EpiArgs &p, unsigned int i)
{
    // in place: a coherent streaming load (the same thread overwrites the float4 right after)
    return MODE == EPI_ADD ? ld_stream_f4(reinterpret_cast<const float4 *>(p.a) + i)
                           : __ldcs(reinterpret_cast<const float4 *>(p.a) + i);
}

template <int MODE>
__device__ __forceinline__ float4 epi_load_b(const EpiArgs &p, unsigned int i)
{
    if (MODE == EPI_ADD) return ld_stream_f4(reinterpret_cast<const float4 *>(p.b) + i);
    if (MODE == EPI_BIAS4) {
        const unsigned int plane = magic_div(i, p.m_hw, p.s_hw);
        const unsigned int c = plane - magic_div(plane, p.m_chan, p.s_chan) * p.channels;
        const float v = __ldg(p.b + c);
        return make_float4(v, v, v, v);
    }
    const unsigned int e = 4u * i;
    const unsigned int plane = magic_div(e, p.m_hw, p.s_hw);
    unsigned int rem = e - plane * p.hw;
    unsigned int c = plane - magic_div(plane, p.m_chan, p.s_chan) * p.channels;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[j] = __ldg(p.b + c);
        if (++rem == p.hw) {
            rem = 0;
            if (++c == p.channels) c = 0;
        }
    }
    return make_float4(v[0], v[1], v[2], v[3]);
}

__device__ __forceinline__ void epi_store(const EpiArgs &p, unsigned int i, const float4 &a, const float4 &b,
                                          unsigned int &m)
{
    const float4 o = make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
    __stcs(reinterpret_cast<float4 *>(p.out) + i, o);
    if (p.relu_out)
        reinterpret_cast<float4 *>(p.relu_out)[i] = make_float4(relu_aten(o.x), relu_aten(o.y), relu_aten(o.z),
                                                                relu_aten(o.w));
    m = max(max(m, max(absbits(o.x), absbits(o.y))), max(absbits(o.z), absbits(o.w)));
}

template <int MODE>
__global__ void __launch_bounds__(kStatThreads)
epilogue_kernel(const EpiArgs p)
{
    __shared__ unsigned int s_warp[kStatThreads / 32];
    const unsigned int nvec = (unsigned int)(p.n >> 2);
    const unsigned int stride = gridDim.x * kStatThreads;
    unsigned int i = blockIdx.x * kStatThreads + threadIdx.x;
    unsigned int m = 0;
    for (; i + (kEpiUnroll - 1) * stride < nvec; i += kEpiUnroll * stride) {
        float4 a[kEpiUnroll], b[kEpiUnroll];
#pragma unroll
        for (int u = 0; u < kEpiUnroll; ++u) a[u] = epi_load_a<MODE>(p, i + u * stride);
#pragma unroll
        for (int u = 0; u < kEpiUnroll; ++u) b[u] = epi_load_b<MODE>(p, i + u * stride);
#pragma unroll
        for (int u = 0; u < kEpiUnroll; ++u) epi_store(p, i + u * stride, a[u], b[u], m);
    }
    for (; i < nvec; i += stride) epi_store(p, i, epi_load_a<MODE>(p, i), epi_load_b<MODE>(p, i), m);
    const unsigned long long t = ((unsigned long long)nvec << 2) + blockIdx.x * kStatThreads + threadIdx.x;
    if (t < p.n) {                                         // the n % 4 tail: threads 0..2 of CTA 0
        float b;
        if (MODE == EPI_ADD) b = p.b[t];
        else b = __ldg(p.b + (unsigned int)((t / (MODE == EPI_BIAS4 ? 4ull * p.hw : p.hw)) % p.channels));
        const float o = __fadd_rn(p.a[t], b);
        p.out[t] = o;
        if (p.relu_out) p.relu_out[t] = relu_aten(o);
        m = max(m, absbits(o));
    }
    if (p.max_slot) block_max_publish(m, s_warp, p.max_slot);
}

// --------------------------------------------------------------------------- histogram
// Bin index of the reference: idx = min((int)trunc(fl32(|x| / interval)), 2047) for x != 0, where
// the division is IEEE round-to-nearest.  A literal __fdiv_rn costs MUFU.RCP + FCHK + 5 FFMA + a
// slow-path call per element and caps the kernel at ~63 % of HBM bandwidth; ncu shows the kernel is
// issue-bound, not DRAM- or atomic-bound (profiles/).  The fast path is exact by construction:
//   q0 = RN(a * r) with r = RN(1/d) hoisted per tensor.  Both roundings are <= 2^-24 relative and
//   Q = RN(a/d) is within 2^-24 of a/d, so |q0 - Q| <= 3 * 2^-24 * q < 3.7e-4 for q < 2048.
//   u = RZ(min(q0, 2047.5) + 2048) holds trunc(q0) in mantissa bits [12,23) and the first 12
//   fraction bits f below them.  If 4 <= f < 4092, q0 is >= 2^-10 = 9.8e-4 away from every
//   integer, hence trunc(Q) == trunc(q0).
// Otherwise (0.2 % of elements, plus every exact zero) the element is "ambiguous": the hot loop
// still counts it in bin trunc(q0) (no select, no branch), flags its float4, and the rare redo pass
// takes that count back and files the element with the real IEEE division.  Values at or beyond
// the top bin clamp to 2047.5 and are counted there directly (their true quotient is > 2047).
// NaN inputs are undefined in the reference; here they land in the top bin.
struct HistDiv {
    float d;        // bin width
    float r;        // RN(1/d)
};

__device__ __forceinline__ HistDiv make_hist_div(float interval)
{
    HistDiv h;
    h.d = interval;
    h.r = __frcp_rn(interval);
    return h;
}

// exact (reference-literal) path for one element
__device__ __forceinline__ void hist_add_exact(unsigned int *sh, float v, float interval)
{
    if (v != 0.0f) {                                       // bins are (lo, hi]: zeros are skipped
        const float q = __fdiv_rn(fabsf(v), interval);     // IEEE division, as numpy float32 / float32
        const int idx = q >= 2047.0f ? 2047 : (int)q;      // trunc + clamp (np.minimum(..., 2047))
        atomicAdd(sh + idx, 1u);
    }
}

// Shared-memory layout per CTA: COPIES histograms of 2048 words, each 8 KB-aligned in the shared
// window so that `(bits >> 10) & 0x1ffc | base` is ONE logic op, followed by one trash word per
// CTA (used by the zero-aware variant).
constexpr unsigned int kSlowThreshold = 0xff800000u;

__device__ __forceinline__ unsigned int hist_fast_bits(float v, const HistDiv &h)
{
    const float q0 = fminf(__fmul_rn(fabsf(v), h.r), 2047.5f);
    return __float_as_uint(__fadd_rz(q0, 2048.0f));
}

// f = bits & 0xfff must lie in [4, 4092): shift it to the top of the word and range-check
__device__ __forceinline__ bool hist_is_slow(unsigned int bits)
{
    return (bits * 0x100000u - 0x400000u) >= kSlowThreshold;
}

__device__ __forceinline__ unsigned int hist_fast_addr(unsigned int bits, unsigned int base_addr)
{
    return ((bits >> 10) & 0x1ffcu) | base_addr;
}

// One element on the hot path: exactly one shared atomic, no divergent region.  Returns whether the
// element is ambiguous.
//   ZERO_AWARE == false (dense data): the ambiguous element is counted in its provisional bin; the
//     redo pass un-counts it.
//   ZERO_AWARE == true (a warp switches to it when exact zeros keep flagging): ambiguous elements go
//     to the trash word instead and exact zeros do not raise the flag (+3 instructions).
template <bool ZERO_AWARE>
__device__ __forceinline__ bool hist_add_fast(unsigned int base_addr, unsigned int trash_addr, float v,
                                              const HistDiv &h)
{
    const unsigned int bits = hist_fast_bits(v, h);
    const bool slow = hist_is_slow(bits);
    unsigned int addr = hist_fast_addr(bits, base_addr);
    if (ZERO_AWARE) addr = slow ? trash_addr : addr;
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
    return ZERO_AWARE ? (slow && v != 0.0f) : slow;
}

// redo pass for one element of a flagged float4 (rare)
template <bool ZERO_AWARE>
__device__ __forceinline__ void hist_redo(unsigned int *sh, unsigned int base_addr, float v, const HistDiv &h)
{
    const unsigned int bits = hist_fast_bits(v, h);
    if (!hist_is_slow(bits)) return;                       // was filed correctly by the hot loop
    // Flagged just ABOVE integer 0 (q0 < 2^-10): the true quotient Q = RN(a / d) differs from q0 by less than
    // 3.7e-4, so 0 <= Q < 1 and any non-zero value belongs to bin 0, where the hot loop already counted it (the
    // ambiguity band around an integer only matters from below, and there is nothing below 0).  Heavy-tailed
    // tensors (everything in the lowest bins) flag 0.5 % of their elements this way; they now cost the loop
    // but neither the IEEE division nor two more atomics.
    if ((bits & 0x7ffffcu) == 0u) {
        if (v == 0.0f) {                                   // zeros are not counted at all
            if (!ZERO_AWARE)
                asm volatile("red.shared.add.u32 [%0], -1;" ::"r"(hist_fast_addr(bits, base_addr)) : "memory");
        } else if (ZERO_AWARE) {                           // the hot loop sent it to the trash word
            asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(hist_fast_addr(bits, base_addr)) : "memory");
        }
        return;
    }
    if (!ZERO_AWARE)                                       // take the provisional count back
        asm volatile("red.shared.add.u32 [%0], -1;" ::"r"(hist_fast_addr(bits, base_addr)) : "memory");
    hist_add_exact(sh, v, h.d);
}

// one thread's share of a chunk part: VPT float4 -> bit i of the result flags float4 i
template <bool ZERO_AWARE, int VPT>
__device__ __forceinline__ unsigned int hist_add_vecs(unsigned int base_addr, unsigned int trash_addr,
                                                      const float4 (&v)[VPT], const HistDiv &h)
{
    unsigned int redo = 0;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const bool s0 = hist_add_fast<ZERO_AWARE>(base_addr, trash_addr, v[i].x, h);
        const bool s1 = hist_add_fast<ZERO_AWARE>(base_addr, trash_addr, v[i].y, h);
        const bool s2 = hist_add_fast<ZERO_AWARE>(base_addr, trash_addr, v[i].z, h);
        const bool s3 = hist_add_fast<ZERO_AWARE>(base_addr, trash_addr, v[i].w, h);
        if (s0 | s1 | s2 | s3) redo |= 1u << i;
    }
    return redo;
}

template <bool ZERO_AWARE>
__device__ __forceinline__ void hist_redo_vecs(unsigned int redo, unsigned int *mine, unsigned int mine_addr,
                                               const float4 *psrc, const HistDiv &h)
{
    while (redo) {                                         // rare: re-load the flagged float4s
        const int slot = __ffs(redo) - 1;
        redo &= redo - 1;
        const float4 w = psrc[threadIdx.x + slot * kStatThreads];
        hist_redo<ZERO_AWARE>(mine, mine_addr, w.x, h);
        hist_redo<ZERO_AWARE>(mine, mine_addr, w.y, h);
        hist_redo<ZERO_AWARE>(mine, mine_addr, w.z, h);
        hist_redo<ZERO_AWARE>(mine, mine_addr, w.w, h);
    }
}

// rare path: does any flagged float4 of this thread hold an exact zero?  (re-loads them: nothing stays live
// across the hot loop)
__device__ __forceinline__ bool hist_flagged_has_zero(unsigned int redo, const float4 *psrc)
{
    bool z = false;
    while (redo) {
        const int slot = __ffs(redo) - 1;
        redo &= redo - 1;
        const float4 w = psrc[threadIdx.x + slot * kStatThreads];
        z = z || w.x == 0.0f || w.y == 0.0f || w.z == 0.0f || w.w == 0.0f;
    }
    return z;
}

constexpr size_t hist_smem_bytes(int copies) { return 8192 + (size_t)copies * PQ_HIST_BINS * 4 + 128; }

template <int COPIES, int VPT = kVecPerThread>
__global__ void __launch_bounds__(kStatThreads, VPT <= 4 ? 6 : 4)
hist_multi_kernel(const __grid_constant__ SegTable tab, unsigned long long *__restrict__ hist)
{
    // dynamic shared memory: hist_smem_bytes(COPIES)
    extern __shared__ unsigned int s_raw[];                // 8 KB alignment slack + [COPIES][2048] + trash
    // align the histograms to 8 KB inside the shared window (see hist_fast_addr)
    const unsigned int raw_addr = (unsigned int)__cvta_generic_to_shared(s_raw);
    const unsigned int pad = ((8192u - (raw_addr & 8191u)) & 8191u) >> 2;
    unsigned int *s_hist = s_raw + pad;
    const unsigned int per = (tab.total_chunks + gridDim.x - 1) / gridDim.x;
    unsigned int c = blockIdx.x * per;
    const unsigned int c_end = min(c + per, tab.total_chunks);
    if (c >= c_end) return;

    for (int i = threadIdx.x; i < COPIES * PQ_HIST_BINS; i += kStatThreads) s_hist[i] = 0;
    __syncthreads();
    unsigned int *mine = s_hist + ((threadIdx.x >> 5) % COPIES) * PQ_HIST_BINS;
    const unsigned int mine_addr = (unsigned int)__cvta_generic_to_shared(mine);
    const unsigned int trash_addr = (unsigned int)__cvta_generic_to_shared(s_hist + COPIES * PQ_HIST_BINS);

    int seg = seg_of_chunk(tab, c);
    bool zero_aware = false;                               // warp-uniform
    while (c < c_end) {
        const SegGeom g = seg_geom(tab, seg);
        const float interval = tab.param[seg];
        const HistDiv hd = make_hist_div(interval);
        const unsigned int seg_first = seg ? tab.chunk_end[seg - 1] : 0;
        const unsigned int seg_last = min(tab.chunk_end[seg], c_end);
        for (; c < seg_last; ++c) {
            const unsigned long long v0 = (unsigned long long)(c - seg_first) * kChunkVecs;
            const float4 *src = g.body + v0;
            const unsigned long long left = g.nvec > v0 ? g.nvec - v0 : 0;
            if (left >= (unsigned long long)kChunkVecs) {
#pragma unroll 1
                for (int part = 0; part < kVecPerThread / VPT; ++part) {
                    const float4 *psrc = src + part * VPT * kStatThreads;
                    float4 v[VPT];
#pragma unroll
                    for (int i = 0; i < VPT; ++i) v[i] = ld_stream_f4(psrc + threadIdx.x + i * kStatThreads);
                    if (zero_aware) {
                        const unsigned int redo = hist_add_vecs<true, VPT>(mine_addr, trash_addr, v, hd);
                        hist_redo_vecs<true>(redo, mine, mine_addr, psrc, hd);
                    } else {
                        const unsigned int redo = hist_add_vecs<false, VPT>(mine_addr, trash_addr, v, hd);
                        // a warp that keeps flagging BECAUSE OF exact zeros switches, for the rest of its
                        // chunk range, to the variant that does not flag zeros; flags raised by small
                        // non-zero values (heavy-tailed data: everything in the lowest bins) do not count,
                        // the zero-aware variant would only be slower on them
                        bool many_zeros = false;
                        if (__popc(redo) >= 3) many_zeros = hist_flagged_has_zero(redo, psrc);
                        zero_aware = __any_sync(0xffffffffu, many_zeros);
                        hist_redo_vecs<false>(redo, mine, mine_addr, psrc, hd);
                    }
                }
            } else {
                for (unsigned int i = threadIdx.x; i < (unsigned int)left; i += kStatThreads) {
                    const float4 v = ld_stream_f4(src + i);
                    hist_add_exact(mine, v.x, interval);
                    hist_add_exact(mine, v.y, interval);
                    hist_add_exact(mine, v.z, interval);
                    hist_add_exact(mine, v.w, interval);
                }
            }
            if (c == seg_first) {
                if (threadIdx.x < g.head) hist_add_exact(mine, g.p[threadIdx.x], interval);
                if (threadIdx.x < g.tail) hist_add_exact(mine, g.p[g.n - g.tail + threadIdx.x], interval);
            }
        }
        // publish: fold the copies, add the non-empty bins to the tensor's global histogram
        __syncthreads();
        unsigned long long *out = hist + (size_t)seg * PQ_HIST_BINS;
        for (int b = threadIdx.x; b < PQ_HIST_BINS; b += kStatThreads) {
            unsigned int cnt = 0;
#pragma unroll
            for (int k = 0; k < COPIES; ++k) {
                cnt += s_hist[k * PQ_HIST_BINS + b];
                s_hist[k * PQ_HIST_BINS + b] = 0;
            }
            if (cnt) atomicAdd(out + b, (unsigned long long)cnt);
        }
        __syncthreads();
        ++seg;
    }
}

// ------------------------------------------------------- histogram, any INTERVAL_NUM (configs.yml:23)
// The reference's bin count is a configuration value (distribution_collector.py:52-63); 2048 is only its
// default and is what hist_multi_kernel above is specialised for (exact reciprocal trick, 8 KB-aligned bins).
// Any other count takes this reference-literal kernel: same chunking and multi-tensor table, one IEEE
// division per element, `nbins` shared counters per CTA.  Still a streaming HBM kernel, ~0.6 of peak.
__device__ __forceinline__ void hist_add_exact_n(unsigned int *sh, float v, float interval, int nbins)
{
    if (v != 0.0f) {
        const float q = __fdiv_rn(fabsf(v), interval);
        const int idx = q >= (float)(nbins - 1) ? nbins - 1 : (int)q;     // np.minimum(int32(q), nbins - 1)
        atomicAdd(sh + idx, 1u);
    }
}

__global__ void __launch_bounds__(kStatThreads)
hist_generic_kernel(const __grid_constant__ SegTable tab, int nbins, unsigned long long *__restrict__ hist)
{
    extern __shared__ unsigned int s_bins[];               // [nbins]
    const unsigned int per = (tab.total_chunks + gridDim.x - 1) / gridDim.x;
    unsigned int c = blockIdx.x * per;
    const unsigned int c_end = min(c + per, tab.total_chunks);
    if (c >= c_end) return;
    for (int i = threadIdx.x; i < nbins; i += kStatThreads) s_bins[i] = 0;
    __syncthreads();
    int seg = seg_of_chunk(tab, c);
    while (c < c_end) {
        const SegGeom g = seg_geom(tab, seg);
        const float interval = tab.param[seg];
        const unsigned int seg_first = seg ? tab.chunk_end[seg - 1] : 0;
        const unsigned int seg_last = min(tab.chunk_end[seg], c_end);
        for (; c < seg_last; ++c) {
            const unsigned long long v0 = (unsigned long long)(c - seg_first) * kChunkVecs;
            const float4 *src = g.body + v0;
            const unsigned long long left = g.nvec > v0 ? g.nvec - v0 : 0;
            const unsigned int nv = left >= (unsigned long long)kChunkVecs ? (unsigned int)kChunkVecs : (unsigned int)left;
            for (unsigned int i = threadIdx.x; i < nv; i += 4 * kStatThreads) {
                float4 v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (i + j * kStatThreads < nv) v[j] = ld_stream_f4(src + i + j * kStatThreads);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (i + j * kStatThreads < nv) {
                        hist_add_exact_n(s_bins, v[j].x, interval, nbins);
                        hist_add_exact_n(s_bins, v[j].y, interval, nbins);
                        hist_add_exact_n(s_bins, v[j].z, interval, nbins);
                        hist_add_exact_n(s_bins, v[j].w, interval, nbins);
                    }
            }
            if (c == seg_first) {
                if (threadIdx.x < g.head) hist_add_exact_n(s_bins, g.p[threadIdx.x], interval, nbins);
                if (threadIdx.x < g.tail) hist_add_exact_n(s_bins, g.p[g.n - g.tail + threadIdx.x], interval, nbins);
            }
        }
        __syncthreads();
        unsigned long long *out = hist + (size_t)seg * nbins;
        for (int b = threadIdx.x; b < nbins; b += kStatThreads) {
            const unsigned int cnt = s_bins[b];
            s_bins[b] = 0;
            if (cnt) atomicAdd(out + b, (unsigned long long)cnt);
        }
        __syncthreads();
        ++seg;
    }
}

}  // namespace pq

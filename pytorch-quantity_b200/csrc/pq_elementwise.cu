// pq_elementwise.cu -- bandwidth kernels of the simulation path (SURVEY.md 8 rows a10, a12, a15):
//   fakequant  y = clamp(rint(x * 2^bit), lo, hi) [/ 2^bit]   new_quantity_op.py:48-58, 246-257
//   add_clamp  y = clamp(a + b, lo, hi)                        new_quantity_op.py:166-174
//   quantize NCHW fp32 -> NHWC int8 (input quantiser fused with the layout change)
// One fused pass each: 8 B/element (fakequant), 12 B/element (add), 5 B/element (quantise)
// instead of the reference's 3-4 separate ATen kernels.
#include "pq_common.cuh"

namespace pq {

constexpr int kEwThreads = 256;
constexpr int kEwUnroll = 4;

// clamp that propagates NaN like torch.clamp (fminf/fmaxf would drop it)
__device__ __forceinline__ float clamp_nan(float v, float lo, float hi)
{
    return v < lo ? lo : (v > hi ? hi : v);
}

template <bool DEQUANT>
__device__ __forceinline__ float fq1(float x, float scale, float inv_scale, float lo, float hi)
{
    // torch.round == round-half-even == rintf (default rounding mode); the scale is a power of
    // two, so the multiply is exact and the divide equals a multiply by the exact reciprocal.
    float v = clamp_nan(rintf(__fmul_rn(x, scale)), lo, hi);
    return DEQUANT ? __fmul_rn(v, inv_scale) : v;
}

template <bool DEQUANT>
__global__ void __launch_bounds__(kEwThreads)
fakequant_kernel(const float *__restrict__ x, float *__restrict__ y, size_t n, float scale,
                 float inv_scale, float lo, float hi)
{
    // x and y are 16-byte aligned here (host checks); scalar tail handled by the last threads
    const size_t nvec = n >> 2;
    const float4 *xv = reinterpret_cast<const float4 *>(x);
    float4 *yv = reinterpret_cast<float4 *>(y);
    const size_t stride = (size_t)gridDim.x * kEwThreads;
    size_t i = (size_t)blockIdx.x * kEwThreads + threadIdx.x;
    for (; i + (kEwUnroll - 1) * stride < nvec; i += kEwUnroll * stride) {
        float4 v[kEwUnroll];
#pragma unroll
        for (int u = 0; u < kEwUnroll; ++u) v[u] = ld_stream_f4(xv + i + u * stride);
#pragma unroll
        for (int u = 0; u < kEwUnroll; ++u) {
            v[u].x = fq1<DEQUANT>(v[u].x, scale, inv_scale, lo, hi);
            v[u].y = fq1<DEQUANT>(v[u].y, scale, inv_scale, lo, hi);
            v[u].z = fq1<DEQUANT>(v[u].z, scale, inv_scale, lo, hi);
            v[u].w = fq1<DEQUANT>(v[u].w, scale, inv_scale, lo, hi);
            st_stream_f4(yv + i + u * stride, v[u]);
        }
    }
    for (; i < nvec; i += stride) {
        float4 v = ld_stream_f4(xv + i);
        v.x = fq1<DEQUANT>(v.x, scale, inv_scale, lo, hi);
        v.y = fq1<DEQUANT>(v.y, scale, inv_scale, lo, hi);
        v.z = fq1<DEQUANT>(v.z, scale, inv_scale, lo, hi);
        v.w = fq1<DEQUANT>(v.w, scale, inv_scale, lo, hi);
        st_stream_f4(yv + i, v);
    }
    const size_t t = (nvec << 2) + (size_t)blockIdx.x * kEwThreads + threadIdx.x;
    if (t < n) y[t] = fq1<DEQUANT>(x[t], scale, inv_scale, lo, hi);
}

// unaligned fallback (views with odd offsets): same arithmetic, scalar accesses
template <bool DEQUANT>
__global__ void __launch_bounds__(kEwThreads)
fakequant_scalar_kernel(const float *__restrict__ x, float *__restrict__ y, size_t n, float scale,
                        float inv_scale, float lo, float hi)
{
    for (size_t i = (size_t)blockIdx.x * kEwThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kEwThreads)
        y[i] = fq1<DEQUANT>(x[i], scale, inv_scale, lo, hi);
}

__global__ void __launch_bounds__(kEwThreads)
add_clamp_kernel(const float *__restrict__ a, const float *__restrict__ b, float *__restrict__ y,
                 size_t n, float lo, float hi, int vec_ok)
{
    const size_t stride = (size_t)gridDim.x * kEwThreads;
    size_t i = (size_t)blockIdx.x * kEwThreads + threadIdx.x;
    if (vec_ok) {
        const size_t nvec = n >> 2;
        const float4 *av = reinterpret_cast<const float4 *>(a);
        const float4 *bv = reinterpret_cast<const float4 *>(b);
        float4 *yv = reinterpret_cast<float4 *>(y);
        for (; i + stride < nvec; i += 2 * stride) {
            float4 p0 = ld_stream_f4(av + i), q0 = ld_stream_f4(bv + i);
            float4 p1 = ld_stream_f4(av + i + stride), q1 = ld_stream_f4(bv + i + stride);
            float4 r0, r1;
            r0.x = clamp_nan(__fadd_rn(p0.x, q0.x), lo, hi); r0.y = clamp_nan(__fadd_rn(p0.y, q0.y), lo, hi);
            r0.z = clamp_nan(__fadd_rn(p0.z, q0.z), lo, hi); r0.w = clamp_nan(__fadd_rn(p0.w, q0.w), lo, hi);
            r1.x = clamp_nan(__fadd_rn(p1.x, q1.x), lo, hi); r1.y = clamp_nan(__fadd_rn(p1.y, q1.y), lo, hi);
            r1.z = clamp_nan(__fadd_rn(p1.z, q1.z), lo, hi); r1.w = clamp_nan(__fadd_rn(p1.w, q1.w), lo, hi);
            st_stream_f4(yv + i, r0);
            st_stream_f4(yv + i + stride, r1);
        }
        for (; i < nvec; i += stride) {
            float4 p = ld_stream_f4(av + i), q = ld_stream_f4(bv + i), r;
            r.x = clamp_nan(__fadd_rn(p.x, q.x), lo, hi); r.y = clamp_nan(__fadd_rn(p.y, q.y), lo, hi);
            r.z = clamp_nan(__fadd_rn(p.z, q.z), lo, hi); r.w = clamp_nan(__fadd_rn(p.w, q.w), lo, hi);
            st_stream_f4(yv + i, r);
        }
        const size_t t = (nvec << 2) + (size_t)blockIdx.x * kEwThreads + threadIdx.x;
        if (t < n) y[t] = clamp_nan(__fadd_rn(a[t], b[t]), lo, hi);
    } else {
        for (; i < n; i += stride) y[i] = clamp_nan(__fadd_rn(a[i], b[i]), lo, hi);
    }
}

// stand-alone RightShift / Sp / DeQuantity (inside NewConv2d these live in the GEMM epilogue)
template <int OP>   // 0: rshift-round-clamp, 1: clamp-scale
__global__ void __launch_bounds__(kEwThreads)
unary_kernel(const float *__restrict__ x, float *__restrict__ y, size_t n, float mul, float lo, float hi)
{
    for (size_t i = (size_t)blockIdx.x * kEwThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kEwThreads) {
        const float v = x[i];
        float r;
        if (OP == 0) {
            const float s = __fmul_rn(v, mul);                                  // x / 2^rs, exact
            const float t = __fadd_rn(s, s > 0.0f ? 0.5f : -0.5f);              // :32-37
            r = (float)max(min((int)t, (int)hi), (int)lo);                      // int32 cast truncates; :41
        } else {
            r = __fmul_rn(clamp_nan(v, lo, hi), mul);
        }
        y[i] = r;
    }
}

// NCHW fp32 -> NHWC int8 with channel padding (generic path: any H*W, scalar loads).  One CTA
// transposes a [32 channels][32 pixels] tile through shared memory.
__global__ void __launch_bounds__(256)
quantize_nchw_nhwc_kernel(const float *__restrict__ x, int8_t *__restrict__ q, int C, int HW,
                          int c_pad, float scale)
{
    __shared__ int8_t tile[32][33 + 3];
    const int n = blockIdx.z;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
    const float *src = x + (size_t)n * C * HW;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = c0 + ty + j * 8, p = p0 + tx;
        float v = 0.0f;
        if (c < C && p < HW) v = __ldg(src + (size_t)c * HW + p);
        v = clamp_nan(rintf(__fmul_rn(v, scale)), -128.0f, 127.0f);
        tile[ty + j * 8][tx] = (int8_t)(int)v;
    }
    __syncthreads();
    int8_t *dst = q + (size_t)n * HW * c_pad;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int p = p0 + ty + j * 8, c = c0 + tx;
        if (p < HW && c < c_pad) dst[(size_t)p * c_pad + c] = tile[tx][ty + j * 8];
    }
}

// Fast path (H*W % 4 == 0, 16-byte aligned rows): one CTA converts [32 channels][128 pixels].
// Each warp streams 4 channel rows with 512-byte coalesced LDG.128s (16 values per thread in
// flight), quantises, packs its 4 consecutive channels of one pixel into one 32-bit word and
// stores it to a [128 pixels][32 channels] shared tile; the tile leaves as 16-byte vectors, one
// full 32-byte sector per pixel row.
__device__ __forceinline__ unsigned int q8(float v, float scale)
{
    return (unsigned int)(int)clamp_nan(rintf(__fmul_rn(v, scale)), -128.0f, 127.0f) & 0xffu;
}

__global__ void __launch_bounds__(256)
quantize_nchw_nhwc_vec_kernel(const float *__restrict__ x, int8_t *__restrict__ q, int C, int HW,
                              int c_pad, float scale)
{
    __shared__ __align__(16) unsigned int tile[128][8 + 1];     // 128 pixels x 32 channel bytes (+pad)
    const int n = blockIdx.z;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 128;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float *src = x + ((size_t)n * C + c0 + warp * 4) * HW + p0 + lane * 4;
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = c0 + warp * 4 + j;
        v[j] = (c < C && p0 + lane * 4 < HW) ? ld_stream_f4(reinterpret_cast<const float4 *>(src + (size_t)j * HW))
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    tile[lane * 4 + 0][warp] = q8(v[0].x, scale) | (q8(v[1].x, scale) << 8) | (q8(v[2].x, scale) << 16) | (q8(v[3].x, scale) << 24);
    tile[lane * 4 + 1][warp] = q8(v[0].y, scale) | (q8(v[1].y, scale) << 8) | (q8(v[2].y, scale) << 16) | (q8(v[3].y, scale) << 24);
    tile[lane * 4 + 2][warp] = q8(v[0].z, scale) | (q8(v[1].z, scale) << 8) | (q8(v[2].z, scale) << 16) | (q8(v[3].z, scale) << 24);
    tile[lane * 4 + 3][warp] = q8(v[0].w, scale) | (q8(v[1].w, scale) << 8) | (q8(v[2].w, scale) << 16) | (q8(v[3].w, scale) << 24);
    __syncthreads();
    // 128 pixels x 32 bytes = 256 x 16 bytes: thread t writes half a pixel row
    const int p = threadIdx.x >> 1, half = threadIdx.x & 1;
    if (p0 + p < HW && c0 + half * 16 < c_pad) {
        const uint4 w = make_uint4(tile[p][half * 4 + 0], tile[p][half * 4 + 1], tile[p][half * 4 + 2], tile[p][half * 4 + 3]);
        *reinterpret_cast<uint4 *>(q + ((size_t)n * HW + p0 + p) * c_pad + c0 + half * 16) = w;
    }
}

// Fused input quantiser + explicit im2col for convolutions with very few input channels (the
// ResNet stem, Cin = 3): writes A[m][k] = q(x[n][c][p*sh-ph+r][q*sw-pw+s]) for k = (r*S+s)*C + c,
// zero for padding and for k >= R*S*C (row pitch kp, a multiple of 16).  Padding the channels to
// the 32-byte granularity of the im2col TMA instead would multiply the GEMM K by 10.
// Each warp owns 32 consecutive output pixels: for every k the 32 lanes gather one fp32 each from
// neighbouring input columns (coalesced, L1/L2 hits: every input value is used R*S/(sh*sw) times),
// quantise, and pack four k into a word of a [32 pixels][kp bytes] shared tile (odd word pitch, no
// bank conflicts); the tile -- 32 contiguous rows of A -- then leaves with 128-byte coalesced stores.
constexpr int kIm2colWarps = 8;

// round-half-even + saturate in two instructions (F2I.RN saturates, then an integer clamp)
__device__ __forceinline__ int q8i(float v, float scale)
{
    return max(-128, min(127, __float2int_rn(__fmul_rn(v, scale))));
}

__global__ void __launch_bounds__(kIm2colWarps * 32)
quantize_im2col_kernel(const float *__restrict__ x, int8_t *__restrict__ a, int C, int H, int W, int R, int S,
                       int sh, int sw, int ph, int pw, int P, int Q, int kp, long long M, float scale)
{
    extern __shared__ unsigned int s_mem[];
    const int kw = kp >> 2;                         // words per row
    const int pitch = kw | 1;                       // odd word pitch: conflict-free column access
    unsigned int *s_tile = s_mem + (threadIdx.x >> 5) * 32 * pitch;
    const int lane = threadIdx.x & 31;
    const int HWi = H * W;
    const long long warps_total = (M + 31) / 32;
    for (long long wi = (long long)blockIdx.x * kIm2colWarps + (threadIdx.x >> 5); wi < warps_total;
         wi += (long long)gridDim.x * kIm2colWarps) {
        const long long m = wi * 32 + lane;
        const bool live = m < M;
        const int qx = (int)(m % Q);
        const long long mp = m / Q;
        const int py = (int)(mp % P);
        const long long n = mp / P;
        const float *img = x + n * (long long)C * HWi;
        const int iy0 = py * sh - ph, ix0 = qx * sw - pw;
        int8_t *row = reinterpret_cast<int8_t *>(s_tile + lane * pitch);
        int k = 0;
        for (int r = 0; r < R; ++r) {
            const int iy = iy0 + r;
            const bool rok = live && (unsigned)iy < (unsigned)H;
            for (int s_ = 0; s_ < S; ++s_) {
                const int ix = ix0 + s_;
                const bool ok = rok && (unsigned)ix < (unsigned)W;
                const float *src = img + iy * W + ix;
                for (int c = 0; c < C; ++c, ++k)
                    row[k] = (int8_t)(ok ? q8i(__ldg(src + c * HWi), scale) : 0);
            }
        }
        for (; k < kp; ++k) row[k] = 0;             // K padding
        __syncwarp();
        // 32 rows x kw words are contiguous in A: coalesced word stores
        unsigned int *dst = reinterpret_cast<unsigned int *>(a + wi * 32 * (long long)kp);
        const long long words_live = (M - wi * 32 < 32 ? M - wi * 32 : 32) * kw;
        for (int w = lane; w < 32 * kw; w += 32)
            if (w < words_live) dst[w] = s_tile[(w / kw) * pitch + (w % kw)];
        __syncwarp();
    }
}

// Input quantiser for the small-channel convolution (pq_conv2d_smallc_s8): fp32 NCHW with C <= 8 ->
// zero-padded NHWC image with 8-byte pixels, q[n][h + ph][w + pw][c] = q(x[n][c][h][w]); everything else
// (spatial padding, channel slots c >= C) is written as 0.  One thread per padded pixel: C coalesced fp32
// loads along w, one coalesced 8-byte store.
// Variant for C <= 4 (RGB inputs): two padded rows per thread, every load of both rows issued before the first
// conversion (12 loads in flight for C = 3) and half as many, longer-lived blocks; the channel loop is a
// compile-time 4, so the values stay in 16 registers (a 4-row / 8-channel version needed 94 and was slower).
__global__ void __launch_bounds__(128)
quantize_pad_nhwc8_c4_kernel(const float *__restrict__ x, uint2 *__restrict__ q, int C, int H, int W, int ph, int pw,
                             int Hp, int Wp, float scale)
{
    const int wp = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (wp >= Wp) return;
    const size_t n = blockIdx.z;
    const size_t HW = (size_t)H * W;
    const int hp0 = blockIdx.y * 2;
    float v[2][2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int h = hp0 + r - ph;
        const float *row = x + (n * C * H + (size_t)(h < 0 ? 0 : h)) * (size_t)W;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int w = wp + k - pw;
            const bool ok = (unsigned)h < (unsigned)H && (unsigned)w < (unsigned)W;
#pragma unroll
            for (int c = 0; c < 4; ++c) v[r][k][c] = (ok && c < C) ? __ldg(row + c * HW + w) : 0.0f;
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int hp = hp0 + r;
        if (hp >= Hp) break;
        unsigned int word[2] = {0u, 0u};
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < C) word[k] |= ((unsigned int)q8i(v[r][k][c], scale) & 0xffu) << (c * 8);
        *reinterpret_cast<uint4 *>(q + (n * Hp + hp) * (size_t)Wp + wp) = make_uint4(word[0], 0u, word[1], 0u);
    }
}

// Variant for C <= 4 and W % 4 == 0 (the 224 x 224 RGB stem): one thread per FOUR horizontally adjacent input pixels --
// one LDG.128 per channel instead of four scalar loads, one index computation per twelve values.  The two-row kernel
// above spends 43 instructions per value (ncu: 85 % issue utilisation at 46 % of DRAM bandwidth); this one ~7.  The
// padding ring is written by the threads at the row ends (left / right columns) and by a grid-stride loop over the
// top / bottom rows.
__global__ void __launch_bounds__(256)
quantize_pad_nhwc8_v4_kernel(const float *__restrict__ x, uint2 *__restrict__ q, int C, int H, int W, int ph, int pw,
                             int Hp, int Wp, float scale)
{
    const int wq = W >> 2;                                   // float4 per input row
    const int item = blockIdx.x * 256 + threadIdx.x;
    const size_t n = blockIdx.y;
    uint2 *qimg = q + n * (size_t)Hp * Wp;
    if (item < H * wq) {
        const int h = item / wq, w4 = item - h * wq;
        const size_t plane4 = (size_t)H * wq;                // float4 per channel plane
        const float4 *src = reinterpret_cast<const float4 *>(x) + (n * C * plane4 + (size_t)item);
        float4 v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = c < C ? __ldg(src + c * plane4) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        unsigned int word[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (c < C) {
                word[0] |= ((unsigned int)q8i(v[c].x, scale) & 0xffu) << (c * 8);
                word[1] |= ((unsigned int)q8i(v[c].y, scale) & 0xffu) << (c * 8);
                word[2] |= ((unsigned int)q8i(v[c].z, scale) & 0xffu) << (c * 8);
                word[3] |= ((unsigned int)q8i(v[c].w, scale) & 0xffu) << (c * 8);
            }
        }
        uint2 *row = qimg + (size_t)(h + ph) * Wp;
        uint2 *dst = row + pw + 4 * w4;
#pragma unroll
        for (int k = 0; k < 4; ++k) dst[k] = make_uint2(word[k], 0u);
        if (w4 == 0)
            for (int i = 0; i < pw; ++i) row[i] = make_uint2(0u, 0u);
        if (w4 == wq - 1)
            for (int i = pw + W; i < Wp; ++i) row[i] = make_uint2(0u, 0u);
    }
    const int pad_items = (Hp - H) * Wp;                     // rows above and below the image
    for (int i = item; i < pad_items; i += gridDim.x * 256) {
        const int r = i / Wp, c = i - r * Wp;
        qimg[(size_t)(r < ph ? r : H + r) * Wp + c] = make_uint2(0u, 0u);
    }
}

// Space-to-depth input quantiser for stride-2 small-channel convolutions (C <= 4): the zero-padded image is cut into
// 2 x 2 pixel blocks and every block becomes ONE 16-byte pixel  q[n][i][j][(dy * 2 + dx) * 4 + c] =
// q(x[n][c][2i + dy - pad_t][2j + dx - pad_l])  (0 outside the image and for c >= C).  A 7 x 7 / stride 2 filter is
// then a 4 x 4 / stride 1 filter over 16-byte pixels: its row window is the same 64 bytes, consecutive output columns
// are the same 16 bytes apart (so pq_conv2d_smallc_s8's row kernel runs on it unchanged, see NewConv2d), but it has
// 4 filter rows instead of 7 (8 narrow MMAs per tile instead of 14) and the tensor is half as large (12 of 16 bytes
// carry data instead of 3 of 8).  One thread per block: two rows x C channels of float2 loads, one 16-byte store.
template <bool VEC>
__global__ void __launch_bounds__(256)
quantize_s2d16_kernel(const float *__restrict__ x, uint4 *__restrict__ q, int C, int H, int W, int pad_t, int pad_l,
                      int Hp2, int Wp2, float scale)
{
    const int item = blockIdx.x * 256 + threadIdx.x;
    if (item >= Hp2 * Wp2) return;
    const size_t n = blockIdx.y;
    const int i = item / Wp2, j = item - i * Wp2;
    const int w0 = 2 * j - pad_l;
    const size_t HW = (size_t)H * W;
    // every load is issued before the first conversion (predicated, no control flow in between)
    float2 v[2][4];
    const bool both = w0 >= 0 && w0 + 1 < W;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
        const int h = 2 * i + dy - pad_t;
        const bool rok = (unsigned)h < (unsigned)H;
        const float *row = x + (n * C * H + (rok ? h : 0)) * (size_t)W + (both ? w0 : 0);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            v[dy][c] = make_float2(0.0f, 0.0f);
            if (VEC) {
                if (rok && both && c < C) v[dy][c] = __ldg(reinterpret_cast<const float2 *>(row + c * HW));
            }
        }
    }
    if (!VEC || !both) {                                   // image border / unaligned rows: scalar loads
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
            const int h = 2 * i + dy - pad_t;
            if ((unsigned)h >= (unsigned)H) continue;
            const float *row = x + (n * C * H + h) * (size_t)W;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c < C && (unsigned)w0 < (unsigned)W) v[dy][c].x = __ldg(row + c * HW + w0);
                if (c < C && (unsigned)(w0 + 1) < (unsigned)W) v[dy][c].y = __ldg(row + c * HW + w0 + 1);
            }
        }
    }
    unsigned int word[4] = {0u, 0u, 0u, 0u};               // one word per phase (dy, dx): bytes = channels
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            // (channels >= C and rows / columns outside the image hold 0.0f: q8i(0) == 0)
            word[2 * dy] |= ((unsigned int)q8i(v[dy][c].x, scale) & 0xffu) << (c * 8);
            word[2 * dy + 1] |= ((unsigned int)q8i(v[dy][c].y, scale) & 0xffu) << (c * 8);
        }
    q[n * (size_t)Hp2 * Wp2 + item] = make_uint4(word[0], word[1], word[2], word[3]);
}

__global__ void __launch_bounds__(kEwThreads)
quantize_pad_nhwc8_kernel(const float *__restrict__ x, uint2 *__restrict__ q, int C, int H, int W, int ph, int pw,
                          int Hp, int Wp, float scale)
{
    // grid = (pixel pairs of a padded row, padded rows, images): no integer division anywhere; every thread
    // converts two horizontally adjacent padded pixels and stores them as one 16-byte vector (Wp is even)
    const int wp = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (wp >= Wp) return;
    const int hp = blockIdx.y;
    const size_t n = blockIdx.z;
    const int h = hp - ph;
    const size_t HW = (size_t)H * W;
    unsigned int word[4] = {0u, 0u, 0u, 0u};
    if ((unsigned)h < (unsigned)H) {
        const float *row = x + (n * C * H + h) * (size_t)W;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int w = wp + k - pw;
            if ((unsigned)w < (unsigned)W) {
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    if (c < C) word[2 * k + (c >> 2)] |= ((unsigned int)q8i(__ldg(row + c * HW + w), scale) & 0xffu) << ((c & 3) * 8);
            }
        }
    }
    *reinterpret_cast<uint4 *>(q + (n * Hp + hp) * (size_t)Wp + wp) = make_uint4(word[0], word[1], word[2], word[3]);
}

}  // namespace pq

namespace {
unsigned int ew_grid(size_t work_items)
{
    size_t blocks = (work_items + pq::kEwThreads - 1) / pq::kEwThreads;
    size_t cap = (size_t)pq::kNumSMs * 16;
    if (blocks > cap) blocks = cap;
    return (unsigned int)(blocks ? blocks : 1);
}
bool aligned16(const void *p) { return (((unsigned long long)p) & 15ull) == 0; }
}  // namespace

extern "C" int pq_fakequant_f32(const float *x, float *y, size_t n, int bit, float lo, float hi,
                                int dequant, pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!x || !y || x == y) return PQ_EINVAL;
    if (bit < -126 || bit > 126) return PQ_EUNSUPPORTED;
    const float scale = ldexpf(1.0f, bit), inv = ldexpf(1.0f, -bit);
    cudaStream_t s = (cudaStream_t)stream;
    if (aligned16(x) && aligned16(y)) {
        unsigned int g = ew_grid((n >> 2) / pq::kEwUnroll + 1);
        if (dequant) pq::fakequant_kernel<true><<<g, pq::kEwThreads, 0, s>>>(x, y, n, scale, inv, lo, hi);
        else pq::fakequant_kernel<false><<<g, pq::kEwThreads, 0, s>>>(x, y, n, scale, inv, lo, hi);
    } else {
        unsigned int g = ew_grid(n);
        if (dequant) pq::fakequant_scalar_kernel<true><<<g, pq::kEwThreads, 0, s>>>(x, y, n, scale, inv, lo, hi);
        else pq::fakequant_scalar_kernel<false><<<g, pq::kEwThreads, 0, s>>>(x, y, n, scale, inv, lo, hi);
    }
    return (int)cudaGetLastError();
}

extern "C" int pq_add_clamp_f32(const float *a, const float *b, float *y, size_t n, float lo, float hi,
                                pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!a || !b || !y || y == a || y == b) return PQ_EINVAL;
    const int vec_ok = aligned16(a) && aligned16(b) && aligned16(y);
    unsigned int g = ew_grid(vec_ok ? (n >> 3) + 1 : n);
    pq::add_clamp_kernel<<<g, pq::kEwThreads, 0, (cudaStream_t)stream>>>(a, b, y, n, lo, hi, vec_ok);
    return (int)cudaGetLastError();
}

extern "C" int pq_rshift_f32(const float *x, float *y, size_t n, int rs, float lo, float hi, pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!x || !y) return PQ_EINVAL;
    if (rs < -100 || rs > 100) return PQ_EUNSUPPORTED;
    pq::unary_kernel<0><<<ew_grid(n), pq::kEwThreads, 0, (cudaStream_t)stream>>>(x, y, n, ldexpf(1.0f, -rs), lo, hi);
    return (int)cudaGetLastError();
}

extern "C" int pq_clamp_scale_f32(const float *x, float *y, size_t n, float lo, float hi, float scale,
                                  pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!x || !y) return PQ_EINVAL;
    pq::unary_kernel<1><<<ew_grid(n), pq::kEwThreads, 0, (cudaStream_t)stream>>>(x, y, n, scale, lo, hi);
    return (int)cudaGetLastError();
}

extern "C" int pq_quantize_nchw_to_nhwc_s8(const float *x, int8_t *q, int N, int C, int H, int W, int c_pad,
                                           int ib, pq_stream_t stream)
{
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0) return PQ_EINVAL;
    if (!x || !q) return PQ_EINVAL;
    if (c_pad < C || (c_pad & 15)) return PQ_EUNSUPPORTED;
    if (ib < -126 || ib > 126 || N > 65535) return PQ_EUNSUPPORTED;
    const int HW = H * W;
    if ((c_pad + 31) / 32 > 65535) return PQ_EUNSUPPORTED;
    if ((HW & 3) == 0 && aligned16(x) && aligned16(q)) {
        dim3 grid((HW + 127) / 128, (c_pad + 31) / 32, N);
        pq::quantize_nchw_nhwc_vec_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, q, C, HW, c_pad, ldexpf(1.0f, ib));
    } else {
        dim3 grid((HW + 31) / 32, (c_pad + 31) / 32, N);
        pq::quantize_nchw_nhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, q, C, HW, c_pad, ldexpf(1.0f, ib));
    }
    return (int)cudaGetLastError();
}

extern "C" int pq_quantize_im2col_s8(const float *x, int8_t *a, int N, int C, int H, int W, int R, int S,
                                     int stride_h, int stride_w, int pad_h, int pad_w, int kp, int ib,
                                     pq_stream_t stream)
{
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || R <= 0 || S <= 0 || stride_h <= 0 || stride_w <= 0) return PQ_EINVAL;
    if (!x || !a || pad_h < 0 || pad_w < 0) return PQ_EINVAL;
    if (kp < R * S * C || (kp & 15) || ib < -126 || ib > 126) return PQ_EUNSUPPORTED;
    if (!aligned16(a)) return PQ_EALIGN;
    if (H + 2 * pad_h < R || W + 2 * pad_w < S) return PQ_EINVAL;    // filter larger than the padded input
    const int P = (H + 2 * pad_h - R) / stride_h + 1, Q = (W + 2 * pad_w - S) / stride_w + 1;
    const long long M = (long long)N * P * Q;
    const size_t smem = (size_t)(pq::kIm2colWarps * 32 * ((kp >> 2) | 1)) * sizeof(unsigned int);
    if (smem > 200 * 1024) return PQ_EUNSUPPORTED;
    static size_t attr_smem = 0;
    if (smem > attr_smem) {
        PQ_CUDA_TRY(cudaFuncSetAttribute(pq::quantize_im2col_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
        attr_smem = smem;
    }
    const long long warps = (M + 31) / 32;
    long long blocks = (warps + pq::kIm2colWarps - 1) / pq::kIm2colWarps;
    if (blocks > pq::kNumSMs * 8) blocks = pq::kNumSMs * 8;
    pq::quantize_im2col_kernel<<<(unsigned int)blocks, pq::kIm2colWarps * 32, smem, (cudaStream_t)stream>>>(
        x, a, C, H, W, R, S, stride_h, stride_w, pad_h, pad_w, P, Q, kp, M, ldexpf(1.0f, ib));
    return (int)cudaGetLastError();
}

extern "C" int pq_quantize_nchw_to_padded_nhwc8_s8(const float *x, int8_t *q, int N, int C, int H, int W, int pad_h,
                                                   int pad_w, int Hp, int Wp, int ib, pq_stream_t stream)
{
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || pad_h < 0 || pad_w < 0 || !x || !q) return PQ_EINVAL;
    if (C > 8 || Hp < H + pad_h || Wp < W + pad_w || ib < -126 || ib > 126) return PQ_EUNSUPPORTED;
    if ((((unsigned long long)q) & 15ull) || (Wp & 1)) return PQ_EALIGN;
    if (Hp > 65535 || N > 65535) return PQ_EUNSUPPORTED;
    const int threads = Wp / 2 <= 128 ? 128 : pq::kEwThreads;          // a 224-wide image is 115 pixel pairs per row
    const dim3 grid((unsigned)((Wp / 2 + threads - 1) / threads), (unsigned)Hp, (unsigned)N);
    if (C <= 4 && (W & 3) == 0 && aligned16(x)) {
        const dim3 grid4((unsigned)((H * (W / 4) + 255) / 256), (unsigned)N);
        pq::quantize_pad_nhwc8_v4_kernel<<<grid4, 256, 0, (cudaStream_t)stream>>>(
            x, reinterpret_cast<uint2 *>(q), C, H, W, pad_h, pad_w, Hp, Wp, ldexpf(1.0f, ib));
        return (int)cudaGetLastError();
    }
    if (C <= 4) {
        const dim3 grid2((unsigned)((Wp / 2 + 127) / 128), (unsigned)((Hp + 1) / 2), (unsigned)N);
        pq::quantize_pad_nhwc8_c4_kernel<<<grid2, 128, 0, (cudaStream_t)stream>>>(
            x, reinterpret_cast<uint2 *>(q), C, H, W, pad_h, pad_w, Hp, Wp, ldexpf(1.0f, ib));
        return (int)cudaGetLastError();
    }
    pq::quantize_pad_nhwc8_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(
        x, reinterpret_cast<uint2 *>(q), C, H, W, pad_h, pad_w, Hp, Wp, ldexpf(1.0f, ib));
    return (int)cudaGetLastError();
}

extern "C" int pq_quantize_nchw_to_s2d16_s8(const float *x, int8_t *q, int N, int C, int H, int W, int pad_t, int pad_l,
                                            int Hp2, int Wp2, int ib, pq_stream_t stream)
{
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || pad_t < 0 || pad_l < 0 || Hp2 <= 0 || Wp2 <= 0 || !x || !q) return PQ_EINVAL;
    if (C > 4 || (pad_t & 1) || (pad_l & 1) || ib < -126 || ib > 126 || N > 65535) return PQ_EUNSUPPORTED;
    if ((long long)Hp2 * Wp2 > 0x7fffffffLL) return PQ_EUNSUPPORTED;
    if (!aligned16(q) || (((unsigned long long)x) & 3ull)) return PQ_EALIGN;
    const dim3 grid((unsigned)(((long long)Hp2 * Wp2 + 255) / 256), (unsigned)N);
    const float scale = ldexpf(1.0f, ib);
    // float2 loads need every row start 8-byte aligned: even W and an 8-byte aligned tensor
    if ((W & 1) == 0 && (((unsigned long long)x) & 7ull) == 0)
        pq::quantize_s2d16_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(
            x, reinterpret_cast<uint4 *>(q), C, H, W, pad_t, pad_l, Hp2, Wp2, scale);
    else
        pq::quantize_s2d16_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(
            x, reinterpret_cast<uint4 *>(q), C, H, W, pad_t, pad_l, Hp2, Wp2, scale);
    return (int)cudaGetLastError();
}

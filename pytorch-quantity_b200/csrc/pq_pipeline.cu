// pq_pipeline.cu -- bandwidth kernels of the int8 inter-layer pipeline (SURVEY.md 8(f) n1): the
// reconstructed model keeps activations as int8 NHWC between tensor-core layers instead of
// round-tripping through fp32 NCHW.  Every kernel is exact integer arithmetic that reproduces the
// reference's fp32 composition (Quantity o ReLU / MaxPool / NewAdd), see include/pq_sm100.h.
#include "pq_common.cuh"

namespace pq {

constexpr int kPipeThreads = 256;

// Per-byte signed max on sm_100a: the s8x4 video instructions (__vmaxs4) are EMULATED (~9 LOP3 / PRMT / IMAD per call:
// the ncu source view of the max-pool kernel showed 548 instructions per thread, 74 % issue utilisation at 48 % of DRAM
// bandwidth); the s16x2 ones are hardware (VIMNMX.S16x2).  A 16-bit lane compares its HIGH byte first, so two running
// maxima -- one over w << 8 (bytes 0 and 2 in the high halves), one over w itself (bytes 1 and 3) -- are exact in
// their high bytes whatever the low bytes hold, and one PRMT gathers the four high bytes at the end.
struct Max4 {
    uint32_t e, o;                               // lanes whose high bytes are the maxima of bytes (0, 2) and (1, 3)
};
__device__ __forceinline__ Max4 max4_init(bool relu)
{
    const uint32_t v = relu ? 0u : 0x80008000u;  // 0 or -128 in every high byte
    return Max4{v, v};
}
__device__ __forceinline__ void max4_acc(Max4 &m, uint32_t w)
{
    m.e = __vmaxs2(m.e, w << 8);
    m.o = __vmaxs2(m.o, w);
}
__device__ __forceinline__ uint32_t max4_get(const Max4 &m)
{
    return __byte_perm(m.e, m.o, 0x7351);        // e.b1, o.b1, e.b3, o.b3
}
__device__ __forceinline__ uint32_t relu4_s8(uint32_t v)
{
    Max4 m = max4_init(true);                    // per-byte signed max with 0
    max4_acc(m, v);
    return max4_get(m);
}

__global__ void __launch_bounds__(kPipeThreads)
relu_s8_kernel(const uint4 *__restrict__ x, uint4 *__restrict__ y, size_t nvec, const int8_t *xt, int8_t *yt, size_t n)
{
    const size_t stride = (size_t)gridDim.x * kPipeThreads;
    for (size_t i = (size_t)blockIdx.x * kPipeThreads + threadIdx.x; i < nvec; i += stride) {
        uint4 v = x[i];
        v.x = relu4_s8(v.x); v.y = relu4_s8(v.y); v.z = relu4_s8(v.z); v.w = relu4_s8(v.w);
        y[i] = v;
    }
    const size_t t = (nvec << 4) + (size_t)blockIdx.x * kPipeThreads + threadIdx.x;
    if (t < n) yt[t] = xt[t] > 0 ? xt[t] : (int8_t)0;
}

// int8 NHWC max-pool.  grid = (output rows, images); the threads of a block walk the (output column, 16-channel
// group) pairs of one output row, channel group fastest, so a warp reads contiguous runs of the k input rows and
// nothing is divided per element (the flat-index version spent ~400 instructions per output on 64-bit div / mod).
__global__ void __launch_bounds__(kPipeThreads)
maxpool_nhwc_s8_kernel(const int8_t *__restrict__ x, int8_t *__restrict__ y, int N, int H, int W, int C, int k,
                       int stride, int pad, int P, int Q, int relu)
{
    const int cv = C >> 4;
    const int pp = blockIdx.x;
    const size_t n = blockIdx.y;
    const int items = Q * cv;
    const uint32_t init = relu ? 0u : 0x80808080u;               // -128 per byte == -inf padding
    const int8_t *xin = x + n * (size_t)H * W * C;
    int8_t *yout = y + (n * P + pp) * (size_t)Q * C;
    int q = (int)threadIdx.x / cv, c16 = (int)threadIdx.x - q * cv;
    const int dq = kPipeThreads / cv, dc = kPipeThreads - dq * cv;   // advance of (q, c16) per loop trip
    for (int t = threadIdx.x; t < items; t += kPipeThreads) {
        uint4 m = make_uint4(init, init, init, init);
        if (k == 3) {                              // the usual window: all nine loads in flight, out-of-range taps = init
            uint4 v[9];
            const int8_t *base = xin + c16 * 16;
            const int iy0 = pp * stride - pad, ix0 = q * stride - pad;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const int iy = iy0 + r;
                const int row_off = iy * W * C;                       // (< 2^31: one image)
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int ix = ix0 + s;
                    v[3 * r + s] = ((unsigned)iy < (unsigned)H && (unsigned)ix < (unsigned)W)
                                       ? __ldg(reinterpret_cast<const uint4 *>(base + row_off + ix * C)) : m;
                }
            }
            Max4 a = max4_init(relu != 0), b = a, c = a, d = a;
#pragma unroll
            for (int i = 0; i < 9; ++i) {
                max4_acc(a, v[i].x); max4_acc(b, v[i].y); max4_acc(c, v[i].z); max4_acc(d, v[i].w);
            }
            m = make_uint4(max4_get(a), max4_get(b), max4_get(c), max4_get(d));
        } else
        for (int r = 0; r < k; ++r) {
            const int iy = pp * stride - pad + r;
            if ((unsigned)iy >= (unsigned)H) continue;
            const int8_t *row = xin + (size_t)iy * W * C + c16 * 16;
            for (int s = 0; s < k; ++s) {
                const int ix = q * stride - pad + s;
                if ((unsigned)ix >= (unsigned)W) continue;
                const uint4 v = *reinterpret_cast<const uint4 *>(row + (size_t)ix * C);
                m.x = __vmaxs4(m.x, v.x); m.y = __vmaxs4(m.y, v.y); m.z = __vmaxs4(m.z, v.z); m.w = __vmaxs4(m.w, v.w);
            }
        }
        *reinterpret_cast<uint4 *>(yout + (size_t)q * C + c16 * 16) = m;
        q += dq; c16 += dc;
        if (c16 >= cv) { c16 -= cv; ++q; }
    }
}

// Global average pool of an int8 / int16 NHWC payload -> fp32 [N][C]: nn.AvgPool2d(H) on the de-quantised tensor (the
// tail of ResNet: Eltwise -> ReLU -> AvgPool2d -> View -> NewLinear).  ATen (native/cuda/AveragePool2d.cu) accumulates
// the window in fp32 and divides by the window size.  The addends are multiples of 2^-bit and every partial sum stays
// below 2^24 of them (checked by the caller), so the fp32 sum equals the integer sum in any order:
//   out = fl(fl(S) * 2^-bit / fl(H * W)),   one IEEE division.
// Replaces de-quantise (3 elementwise passes + an NHWC -> NCHW copy of the fp32 tensor) + avg_pool2d: 1.1 GB of traffic
// for ResNet-50 at batch 512, against 0.1 GB read here.  8 channels per thread, lanes = consecutive channel groups.
template <bool IS16>
__global__ void __launch_bounds__(kPipeThreads)
avgpool_global_kernel(const void *__restrict__ x, float *__restrict__ out, int HW, int C, int relu, float scale, float divisor)
{
    const int c0 = (blockIdx.x * kPipeThreads + threadIdx.x) * 8;
    if (c0 >= C) return;
    const size_t n = blockIdx.y;
    int acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (IS16) {
        const int16_t *p = reinterpret_cast<const int16_t *>(x) + n * (size_t)HW * C + c0;
        for (int i0 = 0; i0 < HW; i0 += 8) {                 // eight pixels in flight (a 7 x 7 plane is 49 dependent loads otherwise)
            uint4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                v[u] = i0 + u < HW ? __ldg(reinterpret_cast<const uint4 *>(p + (size_t)(i0 + u) * C)) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    int lo = (int)(short)(w[j] & 0xffffu), hi = (int)w[j] >> 16;
                    if (relu) { lo = max(lo, 0); hi = max(hi, 0); }
                    acc[2 * j] += lo; acc[2 * j + 1] += hi;
                }
            }
        }
    } else {
        const int8_t *p = reinterpret_cast<const int8_t *>(x) + n * (size_t)HW * C + c0;
        for (int i = 0; i < HW; ++i, p += C) {
            const uint2 v = *reinterpret_cast<const uint2 *>(p);
            const uint32_t w[2] = {relu ? relu4_s8(v.x) : v.x, relu ? relu4_s8(v.y) : v.y};
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += (int)(signed char)((w[j >> 2] >> (8 * (j & 3))) & 0xffu);
        }
    }
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __fdiv_rn(__fmul_rn((float)acc[j], scale), divisor);
    float4 *o = reinterpret_cast<float4 *>(out + n * (size_t)C + c0);
    o[0] = make_float4(r[0], r[1], r[2], r[3]);
    o[1] = make_float4(r[4], r[5], r[6], r[7]);
}

struct AddParams {
    const void *a, *b;
    int a_is16, b_is16, a_relu, b_relu;
    int out_relu;                  // a following nn.ReLU fused: s = max(s, 0)
    int a_shift, b_shift;          // o_bit - a_bit, o_bit - b_bit  (>= 0)
    int lo, hi;                    // clamp of the real sum to [-128, 127] in units of 2^-o_bit
    int q_shift;                   // q_bit - o_bit
    int16_t *out16;
    int8_t *out8;
};

__device__ __forceinline__ int add_load(const void *p, int is16, size_t i)
{
    return is16 ? (int)reinterpret_cast<const int16_t *>(p)[i] : (int)reinterpret_cast<const int8_t *>(p)[i];
}

// round_half_even(num * 2^sh) saturated to int8
__device__ __forceinline__ int requant_rne(int num, int sh)
{
    int r;
    if (sh >= 0) {
        r = max(-128, min(127, num)) << sh;      // saturate first: |num| <= 2^15, sh <= 15
    } else {
        const int d = -sh;
        r = (num + (1 << (d - 1)) - 1 + ((num >> d) & 1)) >> d;   // arithmetic shift, ties to even
    }
    return max(-128, min(127, r));
}

__device__ __forceinline__ uint4 ld_nc_u4(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// byte permute with sign replication (selector nibble bit 3): one instruction sign-extends a packed
// int8 / int16 lane to 32 bits
__device__ __forceinline__ int prmt_sx(uint32_t w, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(0u), "r"(sel));
    return (int)d;
}

// 16 consecutive operands of vector index v, sign-extended (one PRMT each)
template <bool IS16>
__device__ __forceinline__ void add_load16(const void *base, size_t v, int (&out)[16])
{
    if (IS16) {
        const uint4 w0 = ld_nc_u4(reinterpret_cast<const uint4 *>(base) + 2 * v);
        const uint4 w1 = ld_nc_u4(reinterpret_cast<const uint4 *>(base) + 2 * v + 1);
        const uint32_t ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            out[2 * j] = prmt_sx(ww[j], 0x9910u);            // bytes 0,1 + sign of byte 1
            out[2 * j + 1] = prmt_sx(ww[j], 0xbb32u);        // bytes 2,3 + sign of byte 3
        }
    } else {
        const uint4 w = ld_nc_u4(reinterpret_cast<const uint4 *>(base) + v);
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            out[4 * j] = prmt_sx(ww[j], 0x8880u);
            out[4 * j + 1] = prmt_sx(ww[j], 0x9991u);
            out[4 * j + 2] = prmt_sx(ww[j], 0xaaa2u);
            out[4 * j + 3] = prmt_sx(ww[j], 0xbbb3u);
        }
    }
}

__device__ __forceinline__ uint2 ld_nc_u2(const uint2 *p)
{
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

// 8 consecutive operands starting at element e (e % 8 == 0): one fully coalesced 16-byte (int16) or
// 8-byte (int8) load per lane
template <bool IS16>
__device__ __forceinline__ void add_load8(const void *base, size_t e, int *out)
{
    if (IS16) {
        const uint4 w = ld_nc_u4(reinterpret_cast<const uint4 *>(reinterpret_cast<const int16_t *>(base) + e));
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            out[2 * j] = prmt_sx(ww[j], 0x9910u);
            out[2 * j + 1] = prmt_sx(ww[j], 0xbb32u);
        }
    } else {
        const uint2 w = ld_nc_u2(reinterpret_cast<const uint2 *>(reinterpret_cast<const int8_t *>(base) + e));
        const uint32_t ww[2] = {w.x, w.y};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            out[4 * j] = prmt_sx(ww[j], 0x8880u);
            out[4 * j + 1] = prmt_sx(ww[j], 0x9991u);
            out[4 * j + 2] = prmt_sx(ww[j], 0xaaa2u);
            out[4 * j + 3] = prmt_sx(ww[j], 0xbbb3u);
        }
    }
}

__device__ __forceinline__ uint32_t pack4_sat_s8(int y0, int y1, int y2, int y3)
{
    uint32_t t, w;
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(y3), "r"(y2), "r"(0));
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(w) : "r"(y1), "r"(y0), "r"(t));
    return w;
}

// 16 elements per thread and iteration: 16 / 32-byte vector loads per operand, two 16-byte stores for the
// int16 sum and one for the int8 requantisation (buffers are 16-byte aligned; scalar tail below).  The
// kernel is instruction-bound before it is HBM-bound, so the per-element chain is kept to ~10
// instructions: PRMT sign-extending unpack, the two input shifts as IMADs (fma pipe), a 2-op clamp, the
// ties-to-even shift in 4 ops and saturation inside the packing instruction.
//   RELU_IN: either operand carries a pending ReLU (rare once the ReLU is fused into the producer)
//   QDOWN  : q_shift < 0 (the usual case: the Eltwise's feat bit is coarser than the exact sum)
template <bool A16, bool B16, bool RELU_IN, bool QDOWN>
__global__ void __launch_bounds__(kPipeThreads)
add_requant_kernel(const AddParams p, size_t n)
{
    const size_t nvec = n >> 4;
    const size_t stride = (size_t)gridDim.x * kPipeThreads;
    const int a_mul = 1 << p.a_shift, b_mul = 1 << p.b_shift;
    const int a_lo = p.a_relu ? 0 : -32768, b_lo = p.b_relu ? 0 : -32768;
    const int d = QDOWN ? -p.q_shift : 0;
    const int rc = QDOWN ? (1 << (d - 1)) - 1 : 0;
    // A warp owns 512 consecutive elements per iteration.  When the whole block lies inside the vector
    // part, lane l takes elements [8l, 8l+8) of each 256-element half, so that every load and store
    // instruction of the warp covers one contiguous run (16-byte accesses with a 32-byte lane stride
    // touched every sector twice); the ragged last block keeps 16 consecutive elements per lane.
    for (size_t v = (size_t)blockIdx.x * kPipeThreads + threadIdx.x; v < nvec; v += stride) {
        int av[16], bv[16], num[16], q[16];
        const bool whole = (v | 31) < nvec;                                // warp-uniform
        const size_t e0 = ((v >> 5) << 9) + ((v & 31) << 3), e1 = e0 + 256;
        if (whole) {
            add_load8<A16>(p.a, e0, av); add_load8<A16>(p.a, e1, av + 8);
            add_load8<B16>(p.b, e0, bv); add_load8<B16>(p.b, e1, bv + 8);
        } else {
            add_load16<A16>(p.a, v, av);
            add_load16<B16>(p.b, v, bv);
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            int x = av[j], y = bv[j];
            if (RELU_IN) { x = max(x, a_lo); y = max(y, b_lo); }
            num[j] = max(p.lo, min(p.hi, x * a_mul + y * b_mul));       // p.lo = 0 with a fused output ReLU
            if (QDOWN) q[j] = (num[j] + rc + ((num[j] >> d) & 1)) >> d;   // ties to even; the pack saturates
            else q[j] = max(-128, min(127, num[j])) << p.q_shift;        // saturate first: |num| <= 2^15
        }
        if (p.out16) {
            uint32_t o16[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o16[j] = __byte_perm((uint32_t)num[2 * j], (uint32_t)num[2 * j + 1], 0x5410);
            uint4 *d0 = whole ? reinterpret_cast<uint4 *>(p.out16 + e0) : reinterpret_cast<uint4 *>(p.out16) + 2 * v;
            uint4 *d1 = whole ? reinterpret_cast<uint4 *>(p.out16 + e1) : d0 + 1;
            *d0 = make_uint4(o16[0], o16[1], o16[2], o16[3]);
            *d1 = make_uint4(o16[4], o16[5], o16[6], o16[7]);
        }
        if (p.out8) {
            const uint2 lo8 = make_uint2(pack4_sat_s8(q[0], q[1], q[2], q[3]), pack4_sat_s8(q[4], q[5], q[6], q[7]));
            const uint2 hi8 = make_uint2(pack4_sat_s8(q[8], q[9], q[10], q[11]), pack4_sat_s8(q[12], q[13], q[14], q[15]));
            uint2 *d0 = whole ? reinterpret_cast<uint2 *>(p.out8 + e0) : reinterpret_cast<uint2 *>(p.out8) + 2 * v;
            uint2 *d1 = whole ? reinterpret_cast<uint2 *>(p.out8 + e1) : d0 + 1;
            *d0 = lo8;
            *d1 = hi8;
        }
    }
    const size_t t = (nvec << 4) + (size_t)blockIdx.x * kPipeThreads + threadIdx.x;
    if (t < n) {
        int x = add_load(p.a, A16, t), y = add_load(p.b, B16, t);
        if (p.a_relu) x = max(x, 0);
        if (p.b_relu) y = max(y, 0);
        const int num = max(p.lo, min(p.hi, (x << p.a_shift) + (y << p.b_shift)));
        if (p.out16) p.out16[t] = (int16_t)num;
        if (p.out8) p.out8[t] = (int8_t)requant_rne(num, p.q_shift);
    }
}


// Concat + the consumer's input quantiser on quantised operands (pq_concat_requant_s8).  HBM-bound:
// 1 (int8) or 2 (int16) bytes read + 1 byte written per element.
struct ConcatParams {
    const void *ptr[PQ_CONCAT_MAX_SOURCES];
    int is16[PQ_CONCAT_MAX_SOURCES], channels[PQ_CONCAT_MAX_SOURCES], off[PQ_CONCAT_MAX_SOURCES];
    int sh[PQ_CONCAT_MAX_SOURCES], relu[PQ_CONCAT_MAX_SOURCES];   // sh = q_bit - bit_i
    int k, c_out_pad;
};

// one thread per (pixel, 16 output channels); every channel count is a multiple of 16
__global__ void __launch_bounds__(kPipeThreads)
concat_requant_vec_kernel(const ConcatParams p, size_t pixels, int8_t *__restrict__ out)
{
    const unsigned int groups = (unsigned int)p.c_out_pad >> 4;
    const size_t total = pixels * groups;
    for (size_t t = (size_t)blockIdx.x * kPipeThreads + threadIdx.x; t < total; t += (size_t)gridDim.x * kPipeThreads) {
        const size_t pix = t / groups;
        const int c0 = (int)(t - pix * groups) << 4;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll 1
        for (int i = 0; i < p.k; ++i) {
            const int c = c0 - p.off[i];
            if (c < 0 || c >= p.channels[i]) continue;
            const size_t v = (pix * (size_t)p.channels[i] + c) >> 4;
            int x[16];
            if (p.is16[i]) add_load16<true>(p.ptr[i], v, x); else add_load16<false>(p.ptr[i], v, x);
            const int lo = p.relu[i] ? 0 : -32768, sh = p.sh[i];
            int q[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) q[j] = requant_rne(max(x[j], lo), sh);
            o = make_uint4(pack4_sat_s8(q[0], q[1], q[2], q[3]), pack4_sat_s8(q[4], q[5], q[6], q[7]),
                           pack4_sat_s8(q[8], q[9], q[10], q[11]), pack4_sat_s8(q[12], q[13], q[14], q[15]));
            break;
        }
        reinterpret_cast<uint4 *>(out)[t] = o;
    }
}

// any channel counts: one thread per output element
__global__ void __launch_bounds__(kPipeThreads)
concat_requant_scalar_kernel(const ConcatParams p, size_t pixels, int8_t *__restrict__ out)
{
    const size_t total = pixels * (size_t)p.c_out_pad;
    for (size_t t = (size_t)blockIdx.x * kPipeThreads + threadIdx.x; t < total; t += (size_t)gridDim.x * kPipeThreads) {
        const size_t pix = t / (unsigned int)p.c_out_pad;
        const int c0 = (int)(t - pix * (unsigned int)p.c_out_pad);
        int q = 0;
        for (int i = 0; i < p.k; ++i) {
            const int c = c0 - p.off[i];
            if (c < 0 || c >= p.channels[i]) continue;
            int x = add_load(p.ptr[i], p.is16[i], pix * (size_t)p.channels[i] + c);
            if (p.relu[i]) x = max(x, 0);
            q = requant_rne(x, p.sh[i]);
            break;
        }
        out[t] = (int8_t)q;
    }
}
__global__ void bias_fold_kernel(const int32_t *__restrict__ b, int n, int rs, int32_t *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int v = max(-128, min(127, b[i]));               // BiasAdd operands are int8-saturated (new_quantity_op.py:148)
    out[i] = v;
    out[n + i] = (rs >= 1 && rs <= 20) ? (1 << (rs - 1)) + v * (1 << rs) : 0;
    // third row: the post-shift saturation bounds as s16x2 pairs of adjacent channels (see requant_packed16):
    //   words [0, n/2): h = 127 + min(b, 0);   words [n/2, n): l = -128 + max(b, 0)
    if ((i & 1) == 0 && i + 1 < n) {
        const int v1 = max(-128, min(127, b[i + 1]));
        const int h0 = 127 + min(v, 0), h1 = 127 + min(v1, 0), l0 = -128 + max(v, 0), l1 = -128 + max(v1, 0);
        out[2 * n + (i >> 1)] = (int32_t)(((uint32_t)(uint16_t)(int16_t)h1 << 16) | (uint32_t)(uint16_t)(int16_t)h0);
        out[2 * n + (n >> 1) + (i >> 1)] = (int32_t)(((uint32_t)(uint16_t)(int16_t)l1 << 16) | (uint32_t)(uint16_t)(int16_t)l0);
    }
}

}  // namespace pq

namespace {
unsigned int pipe_grid(size_t items)
{
    size_t blocks = (items + pq::kPipeThreads - 1) / pq::kPipeThreads;
    const size_t cap = (size_t)pq::kNumSMs * 16;
    if (blocks > cap) blocks = cap;
    return (unsigned int)(blocks ? blocks : 1);
}
bool al16(const void *p) { return (((unsigned long long)p) & 15ull) == 0; }
}  // namespace

extern "C" int pq_relu_s8(const int8_t *x, int8_t *y, size_t n, pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!x || !y) return PQ_EINVAL;
    if (!al16(x) || !al16(y)) return PQ_EALIGN;
    pq::relu_s8_kernel<<<pipe_grid((n >> 4) + 1), pq::kPipeThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(x), reinterpret_cast<uint4 *>(y), n >> 4, x, y, n);
    return (int)cudaGetLastError();
}

extern "C" int pq_maxpool_nhwc_s8(const int8_t *x, int8_t *y, int N, int H, int W, int C, int k, int stride, int pad,
                                  int relu, pq_stream_t stream)
{
    if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || k <= 0 || stride <= 0 || pad < 0 || !x || !y) return PQ_EINVAL;
    if ((C & 15) || pad >= k) return PQ_EUNSUPPORTED;
    if (!al16(x) || !al16(y)) return PQ_EALIGN;
    const int P = (H + 2 * pad - k) / stride + 1, Q = (W + 2 * pad - k) / stride + 1;
    if (P <= 0 || Q <= 0) return PQ_EINVAL;
    if (N > 65535) return PQ_EUNSUPPORTED;
    pq::maxpool_nhwc_s8_kernel<<<dim3((unsigned)P, (unsigned)N), pq::kPipeThreads, 0, (cudaStream_t)stream>>>(
        x, y, N, H, W, C, k, stride, pad, P, Q, relu);
    return (int)cudaGetLastError();
}

extern "C" int pq_avgpool_global_nhwc_f32(const void *x, int is16, int bit, int relu, int N, int HW, int C, float *out,
                                          pq_stream_t stream)
{
    if (N <= 0 || HW <= 0 || C <= 0 || !x || !out) return PQ_EINVAL;
    if ((C & 7) || bit < -100 || bit > 100 || N > 65535) return PQ_EUNSUPPORTED;
    // exactness of the fp32 accumulation the reference performs (see the kernel): |sum| < 2^24 payload units
    if ((long long)HW * (is16 ? 32768 : 128) >= (1LL << 24)) return PQ_EUNSUPPORTED;
    if (!al16(x) || !al16(out)) return PQ_EALIGN;
    const float scale = ldexpf(1.0f, -bit), divisor = (float)HW;
    const dim3 grid((unsigned)((C / 8 + pq::kPipeThreads - 1) / pq::kPipeThreads), (unsigned)N);
    if (is16) pq::avgpool_global_kernel<true><<<grid, pq::kPipeThreads, 0, (cudaStream_t)stream>>>(x, out, HW, C, relu, scale, divisor);
    else pq::avgpool_global_kernel<false><<<grid, pq::kPipeThreads, 0, (cudaStream_t)stream>>>(x, out, HW, C, relu, scale, divisor);
    return (int)cudaGetLastError();
}

extern "C" int pq_add_requant(const void *a, int a_is16, int a_bit, int a_relu, const void *b, int b_is16, int b_bit,
                              int b_relu, size_t n, int flags, int16_t *out16, int8_t *out8, int q_bit,
                              pq_stream_t stream)
{
    if (n == 0) return PQ_OK;
    if (!a || !b || (!out16 && !out8)) return PQ_EINVAL;
    if (!al16(a) || !al16(b) || (out16 && !al16(out16)) || (out8 && !al16(out8))) return PQ_EALIGN;
    const int o_bit = a_bit > b_bit ? a_bit : b_bit;
    const int span = o_bit - (a_bit < b_bit ? a_bit : b_bit);
    if (span > 7 || o_bit < 0 || o_bit > 7 || q_bit - o_bit > 15 || o_bit - q_bit > 15) return PQ_EUNSUPPORTED;
    pq::AddParams p;
    p.a = a; p.b = b; p.a_is16 = a_is16; p.b_is16 = b_is16; p.a_relu = a_relu; p.b_relu = b_relu;
    p.a_shift = o_bit - a_bit; p.b_shift = o_bit - b_bit;
    p.out_relu = flags & PQ_FLAG_RELU;
    p.lo = p.out_relu ? 0 : -128 * (1 << o_bit); p.hi = 127 * (1 << o_bit);
    p.q_shift = q_bit - o_bit; p.out16 = out16; p.out8 = out8;
    const unsigned int grid = pipe_grid((n >> 4) + 16);
    cudaStream_t s = (cudaStream_t)stream;
    const int variant = (a_is16 ? 8 : 0) | (b_is16 ? 4 : 0) | ((a_relu || b_relu) ? 2 : 0) | (p.q_shift < 0 ? 1 : 0);
#define PQ_ADD_CASE(V, A, B, R, Q) \
    case V: pq::add_requant_kernel<A, B, R, Q><<<grid, pq::kPipeThreads, 0, s>>>(p, n); break;
    switch (variant) {
        PQ_ADD_CASE(0, false, false, false, false) PQ_ADD_CASE(1, false, false, false, true)
        PQ_ADD_CASE(2, false, false, true, false) PQ_ADD_CASE(3, false, false, true, true)
        PQ_ADD_CASE(4, false, true, false, false) PQ_ADD_CASE(5, false, true, false, true)
        PQ_ADD_CASE(6, false, true, true, false) PQ_ADD_CASE(7, false, true, true, true)
        PQ_ADD_CASE(8, true, false, false, false) PQ_ADD_CASE(9, true, false, false, true)
        PQ_ADD_CASE(10, true, false, true, false) PQ_ADD_CASE(11, true, false, true, true)
        PQ_ADD_CASE(12, true, true, false, false) PQ_ADD_CASE(13, true, true, false, true)
        PQ_ADD_CASE(14, true, true, true, false) PQ_ADD_CASE(15, true, true, true, true)
    }
#undef PQ_ADD_CASE
    return (int)cudaGetLastError();
}

extern "C" int pq_concat_requant_s8(const pq_concat_src *srcs_host, int k, size_t pixels, int q_bit, int c_out_pad,
                                    int8_t *out, pq_stream_t stream)
{
    if (k < 0 || c_out_pad < 0 || (k > 0 && !srcs_host)) return PQ_EINVAL;
    if (k > PQ_CONCAT_MAX_SOURCES) return PQ_ETOOMANY;
    if (pixels == 0 || c_out_pad == 0) return PQ_OK;
    if (!out) return PQ_EINVAL;
    pq::ConcatParams p;
    p.k = k; p.c_out_pad = c_out_pad;
    int off = 0;
    bool vec = (c_out_pad & 15) == 0 && al16(out);
    for (int i = 0; i < k; ++i) {
        const pq_concat_src &s = srcs_host[i];
        if (s.channels < 0 || (s.channels > 0 && !s.ptr)) return PQ_EINVAL;
        if (q_bit - s.bit > 15 || s.bit - q_bit > 15) return PQ_EUNSUPPORTED;
        if (s.is16 && (((unsigned long long)s.ptr) & 1ull)) return PQ_EALIGN;
        p.ptr[i] = s.ptr; p.is16[i] = s.is16 ? 1 : 0; p.channels[i] = s.channels; p.off[i] = off;
        p.sh[i] = q_bit - s.bit; p.relu[i] = s.relu ? 1 : 0;
        vec = vec && (s.channels & 15) == 0 && al16(s.ptr);
        off += s.channels;
    }
    if (off > c_out_pad) return PQ_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (vec)
        pq::concat_requant_vec_kernel<<<pipe_grid(pixels * (size_t)(c_out_pad >> 4)), pq::kPipeThreads, 0, st>>>(
            p, pixels, out);
    else
        pq::concat_requant_scalar_kernel<<<pipe_grid(pixels * (size_t)c_out_pad), pq::kPipeThreads, 0, st>>>(
            p, pixels, out);
    return (int)cudaGetLastError();
}

extern "C" int pq_bias_fold_s32(const int32_t *bias_q, int n, int rs, int32_t *out, pq_stream_t stream)
{
    if (n < 0) return PQ_EINVAL;
    if (n == 0) return PQ_OK;
    if (!bias_q || !out) return PQ_EINVAL;
    pq::bias_fold_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(bias_q, n, rs, out);
    return (int)cudaGetLastError();
}

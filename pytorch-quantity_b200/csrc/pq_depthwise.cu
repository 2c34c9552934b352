// pq_depthwise.cu -- NewConv2d on a depthwise convolution (groups == in_channels == out_channels; MobileNetV2,
// MnasNet, EfficientNet): Conv -> RightShift -> BiasAdd -> Sp -> DeQuantity (new_quantity_op.py:104-133) on an int8
// NHWC image, one kernel per layer.
//
// A depthwise output is R*S multiply-adds of ONE channel, so there is no reduction for the tensor cores to do: the
// layer is a stencil over int8 NHWC, bound by HBM and by the integer issue rate of the SMs.  Each thread owns 16
// channels (one 16-byte vector) of one output pixel at a time:
//   - the CTA's weights ([R][S] taps x its 16 * G channels) are sign-extended once into shared memory, laid out so
//     that the four LDS.128 of one tap are warp-broadcasts without bank conflicts;
//   - every tap is one 16-byte load of the input pixel (read-only path: the R*S re-reads of each input pixel by its
//     neighbours hit L1 / L2, HBM sees it about once), 16 PRMT sign extensions and 16 IMAD into exact int32
//     accumulators (|acc| <= 49 * 2^14);
//   - zero padding is a skipped tap (runtime tap loops) or a predicated-off load (3 x 3 and 5 x 5, unrolled);
//   - the epilogue is the GEMM's (pq_requant.cuh): requant / requant_folded, the saturating pack, 2^-ob.
// A warp covers 32 / G consecutive output pixels x all G channel groups of the CTA, so the int8 NHWC result leaves in
// 16-byte stores that form 16 * G contiguous bytes per pixel, and the fp32 NCHW result in runs of 32 / G consecutive
// pixels per channel.
#include <cuda.h>

#include "pq_common.cuh"
#include "pq_requant.cuh"

namespace pq {

constexpr int kDwThreads = 256;
constexpr int kDwMaxRS = 7;            // R, S <= 7
constexpr int kDwPixIters = 4;         // output pixels per thread

struct DwParams {
    const int8_t *x;                   // [N][H][W][C]
    const int8_t *w;                   // [R][S][C], zero beyond K
    const int32_t *bias;               // [K]
    const int32_t *bias_c;             // PQ_FLAG_BIAS_FOLDED: [K] 2^(rs-1) + (bias << rs) (see requant_folded), else NULL
    float *out_f32;                    // [N][K][P][Q] or NULL
    int8_t *out_s8;                    // [N][P][Q][K] or NULL
    int H, W, C, K, R, S, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, P, Q, rs, ob, relu;
    int M;                             // N * P * Q
};

// G: 16-channel groups per CTA (blockIdx.y selects the CTA's slice of 16 * G channels, C % (16 * G) == 0).
// KS: R == S == KS known at compile time (3, 5: the taps are unrolled, so the loads of a filter row are in flight
// together and no loop control runs per tap; out-of-image taps are predicated to zero), or 0: any R, S <= 7 in runtime
// loops (one load in flight per tap).
template <int G, int KS>
__global__ void __launch_bounds__(kDwThreads) dw_conv_s8_kernel(const DwParams p)
{
    __shared__ int4 ws[kDwMaxRS * kDwMaxRS * 4 * G];   // [tap][j][group]: channels 16 * group + 4j .. 4j + 3
    constexpr int kPixPerCta = kDwThreads / G;
    const int g = (int)threadIdx.x % G, slot = (int)threadIdx.x / G;
    const int cta_c = (int)blockIdx.y * 16 * G, c0 = cta_c + 16 * g;
    const int R = KS ? KS : p.R, S = KS ? KS : p.S;
    const int taps = R * S;

    pdl_wait();                                        // the producer of x finished and flushed
    for (int i = (int)threadIdx.x; i < taps * 4 * G; i += kDwThreads) {
        const int t = i / (4 * G), j = (i / G) % 4, gg = i % G;
        const uint32_t wv = __ldg(reinterpret_cast<const uint32_t *>(p.w + (size_t)t * p.C + cta_c + 16 * gg + 4 * j));
        ws[i] = make_int4(prmt_sx(wv, 0x8880), prmt_sx(wv, 0x9991), prmt_sx(wv, 0xAAA2), prmt_sx(wv, 0xBBB3));
    }
    __syncthreads();
    pdl_launch_dependents();

    const Requant rq = make_requant(p.rs, p.relu);
    const float dq = __int_as_float((127 - p.ob) << 23);              // 2^-ob, exact
    const int a_hi = 127 * (1 << rq.sh) + rq.half - 1, a_lo = -128 * (1 << rq.sh) - rq.half + 1;
    const int nvalid = p.K - c0;                                      // this thread's channels inside K (may be <= 0)
    const int pq_img = p.P * p.Q;
#pragma unroll 1
    for (int it = 0; it < kDwPixIters; ++it) {
        const int m = ((int)blockIdx.x * kDwPixIters + it) * kPixPerCta + slot;
        if (m >= p.M || nvalid <= 0) continue;
        const int n = m / pq_img, pix = m - n * pq_img;
        const int op = pix / p.Q, oq = pix - op * p.Q;
        const int h0 = op * p.stride_h - p.pad_h, w0 = oq * p.stride_w - p.pad_w;
        int acc[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) acc[c] = 0;
        const int8_t *img = p.x + (size_t)n * p.H * p.W * p.C + c0;
#pragma unroll(KS ? KS : 1)
        for (int r = 0; r < R; ++r) {
            const int ih = h0 + r * p.dil_h;
            if (!KS && (ih < 0 || ih >= p.H)) continue;
            const bool row_ok = ih >= 0 && ih < p.H;
            const int4 *wr = ws + r * S * 4 * G + g;
#pragma unroll(KS ? KS : 1)
            for (int s = 0; s < S; ++s) {
                const int iw = w0 + s * p.dil_w;
                if (!KS && (iw < 0 || iw >= p.W)) continue;
                const bool ok = row_ok && iw >= 0 && iw < p.W;       // outside the image: zero padding
                const uint4 v = ok ? __ldg(reinterpret_cast<const uint4 *>(img + ((size_t)ih * p.W + iw) * p.C))
                                   : make_uint4(0u, 0u, 0u, 0u);
                const uint32_t xw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int4 wt = wr[(s * 4 + j) * G];
                    acc[4 * j] += prmt_sx(xw[j], 0x8880) * wt.x;
                    acc[4 * j + 1] += prmt_sx(xw[j], 0x9991) * wt.y;
                    acc[4 * j + 2] += prmt_sx(xw[j], 0xAAA2) * wt.z;
                    acc[4 * j + 3] += prmt_sx(xw[j], 0xBBB3) * wt.w;
                }
            }
        }
        // RightShift -> BiasAdd -> Sp (+ ReLU), saturated to int8
        int y[16];
        if (p.bias_c) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const int t = c < nvalid ? (p.relu ? requant_folded<true>(acc[c], rq.sh, a_lo, a_hi, __ldg(p.bias_c + c0 + c))
                                                   : requant_folded<false>(acc[c], rq.sh, a_lo, a_hi, __ldg(p.bias_c + c0 + c)))
                                         : 0;
                y[c] = max(-128, min(127, t));
            }
        } else {
#pragma unroll
            for (int c = 0; c < 16; ++c) y[c] = c < nvalid ? requant(acc[c], rq, __ldg(p.bias + c0 + c)) : 0;
        }
        if (p.out_s8) {
            int8_t *o8 = p.out_s8 + (size_t)m * p.K + c0;
            if (nvalid >= 16 && (p.K & 15) == 0) {
                *reinterpret_cast<uint4 *>(o8) = make_uint4(pack4_sat_s8(y[0], y[1], y[2], y[3]), pack4_sat_s8(y[4], y[5], y[6], y[7]),
                                                            pack4_sat_s8(y[8], y[9], y[10], y[11]),
                                                            pack4_sat_s8(y[12], y[13], y[14], y[15]));
            } else {
#pragma unroll
                for (int c = 0; c < 16; ++c)
                    if (c < nvalid) o8[c] = (int8_t)y[c];
            }
        }
        if (p.out_f32) {                                               // DeQuantity, NCHW
            float *of = p.out_f32 + ((size_t)n * p.K + c0) * pq_img + pix;
#pragma unroll
            for (int c = 0; c < 16; ++c)
                if (c < nvalid) of[(size_t)c * pq_img] = (float)y[c] * dq;
        }
    }
}

}  // namespace pq

extern "C" int pq_conv2d_dw_s8(const int8_t *x_nhwc, const int8_t *w_rsc, const int32_t *bias_q,
                               const pq_conv_desc *desc_host, int flags, float *out_f32_nchw, int8_t *out_s8_nhwc,
                               pq_stream_t stream)
{
    if (!x_nhwc || !w_rsc || !bias_q || !desc_host || (!out_f32_nchw && !out_s8_nhwc)) return PQ_EINVAL;
    const pq_conv_desc &d = *desc_host;
    if (d.N <= 0 || d.H <= 0 || d.W <= 0 || d.C <= 0 || d.K <= 0 || d.R <= 0 || d.S <= 0) return PQ_EINVAL;
    if (d.stride_h <= 0 || d.stride_w <= 0 || d.pad_h < 0 || d.pad_w < 0 || d.dil_h <= 0 || d.dil_w <= 0) return PQ_EINVAL;
    if (d.K > d.C) return PQ_EINVAL;
    const int r_eff = (d.R - 1) * d.dil_h + 1, s_eff = (d.S - 1) * d.dil_w + 1;
    if (d.H + 2 * d.pad_h < r_eff || d.W + 2 * d.pad_w < s_eff) return PQ_EINVAL;
    if (d.P != (d.H + 2 * d.pad_h - r_eff) / d.stride_h + 1 || d.Q != (d.W + 2 * d.pad_w - s_eff) / d.stride_w + 1)
        return PQ_EINVAL;
    if (d.C % 16 || d.R > pq::kDwMaxRS || d.S > pq::kDwMaxRS || d.stride_h > 2 || d.stride_w > 2 || d.dil_h > 2 ||
        d.dil_w > 2 || d.pad_h > r_eff - 1 || d.pad_w > s_eff - 1)
        return PQ_EUNSUPPORTED;
    if (d.ob < -100 || d.ob > 100 || d.rs > 24 || d.rs < -24) return PQ_EUNSUPPORTED;
    const long long M = (long long)d.N * d.P * d.Q;
    if (M > 0x7fffffffLL) return PQ_EUNSUPPORTED;
    const int G = d.C % 64 == 0 ? 4 : (d.C % 32 == 0 ? 2 : 1);
    if (d.C / (16 * G) > 65535) return PQ_EUNSUPPORTED;             // grid.y below: one CTA per 16 * G channels
    if ((((uintptr_t)x_nhwc | (uintptr_t)w_rsc | (uintptr_t)out_s8_nhwc) & 15) || (((uintptr_t)bias_q | (uintptr_t)out_f32_nchw) & 3))
        return PQ_EALIGN;

    pq::DwParams p = {};
    p.x = x_nhwc; p.w = w_rsc; p.bias = bias_q;
    p.bias_c = ((flags & PQ_FLAG_BIAS_FOLDED) && d.rs >= 1 && d.rs <= 20 && (d.K & 15) == 0) ? bias_q + d.K : nullptr;
    p.out_f32 = out_f32_nchw; p.out_s8 = out_s8_nhwc;
    p.H = d.H; p.W = d.W; p.C = d.C; p.K = d.K; p.R = d.R; p.S = d.S;
    p.stride_h = d.stride_h; p.stride_w = d.stride_w; p.pad_h = d.pad_h; p.pad_w = d.pad_w;
    p.dil_h = d.dil_h; p.dil_w = d.dil_w; p.P = d.P; p.Q = d.Q; p.rs = d.rs; p.ob = d.ob;
    p.relu = flags & PQ_FLAG_RELU;
    p.M = (int)M;
    const int KS = (d.R == d.S && (d.R == 3 || d.R == 5)) ? d.R : 0;
    const long long pix_per_cta = (long long)pq::kDwThreads / G * pq::kDwPixIters;
    const dim3 grid((unsigned)((M + pix_per_cta - 1) / pix_per_cta), (unsigned)(d.C / (16 * G)));
    const cudaStream_t s = (cudaStream_t)stream;
    switch (G * 8 + KS) {
        case 4 * 8 + 3: return launch_pdl(pq::dw_conv_s8_kernel<4, 3>, grid, pq::kDwThreads, 0, s, p);
        case 4 * 8 + 5: return launch_pdl(pq::dw_conv_s8_kernel<4, 5>, grid, pq::kDwThreads, 0, s, p);
        case 4 * 8: return launch_pdl(pq::dw_conv_s8_kernel<4, 0>, grid, pq::kDwThreads, 0, s, p);
        case 2 * 8 + 3: return launch_pdl(pq::dw_conv_s8_kernel<2, 3>, grid, pq::kDwThreads, 0, s, p);
        case 2 * 8 + 5: return launch_pdl(pq::dw_conv_s8_kernel<2, 5>, grid, pq::kDwThreads, 0, s, p);
        case 2 * 8: return launch_pdl(pq::dw_conv_s8_kernel<2, 0>, grid, pq::kDwThreads, 0, s, p);
        case 1 * 8 + 3: return launch_pdl(pq::dw_conv_s8_kernel<1, 3>, grid, pq::kDwThreads, 0, s, p);
        case 1 * 8 + 5: return launch_pdl(pq::dw_conv_s8_kernel<1, 5>, grid, pq::kDwThreads, 0, s, p);
        default: return launch_pdl(pq::dw_conv_s8_kernel<1, 0>, grid, pq::kDwThreads, 0, s, p);
    }
}

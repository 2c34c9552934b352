/*
 * pq_sm100.h -- C ABI of libpq_sm100.so, the B200 (sm_100a) kernels behind the
 * calibration + simulation hot path of pytorch-quantity.
 *
 * The reference has no FFI: its operator API is plain Python classes over numpy / torch
 * (SURVEY.md 8b).  Each entry point below therefore names the reference Python function
 * whose arithmetic it replaces (paths relative to /root/reference/quantity/); the Python
 * classes of the same names in pytorch-quantity_b200/common/quantity/ bind these symbols
 * through ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the
 *     parameter name ends in _host.  The caller (PyTorch) owns every buffer including
 *     workspaces; the library allocates nothing and keeps no state besides cached
 *     function attributes / TMA descriptors.
 *   - all work is enqueued on `stream` (a cudaStream_t); no call synchronises.
 *   - return 0 on success, a negative PQ_E* for bad arguments / unsupported shapes, or a
 *     positive cudaError_t.  Nothing throws or aborts across the ABI.  There is no CPU
 *     fallback: an unsupported request is an error the Python side raises.
 *   - accumulating entry points (absmax, hist) combine with atomics, so successive
 *     batches, several streams and several tensors compose; results are independent of
 *     launch order (unsigned max / integer add), which is what makes the multi-GPU
 *     merge (NCCL MAX / SUM on the same buffers) bit-exact.
 */
#ifndef PQ_SM100_H
#define PQ_SM100_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *pq_stream_t; /* cudaStream_t */

/* pq_version() of a library built from this header.  Bump it whenever an entry point changes its parameters: ctypes
 * binds by name only, so a stale build would otherwise be called with the wrong arguments without any error. */
#define PQ_VERSION 201

#define PQ_OK 0
#define PQ_EINVAL (-1)       /* null pointer, negative size, bad enum */
#define PQ_EUNSUPPORTED (-2) /* shape / alignment the kernels do not implement */
#define PQ_EALIGN (-3)       /* pointer not aligned as documented */
#define PQ_ETOOMANY (-4)     /* more segments than PQ_MAX_SEGMENTS in one call */

#define PQ_HIST_BINS 2048   /* tools/configs.yml:23 INTERVAL_NUM (the default; the fast histogram kernel) */
#define PQ_HIST_BINS_MAX 8192 /* largest INTERVAL_NUM the generic entry points accept */
#define PQ_KL_TARGET_BIN 128 /* common/quantity/quantizer.py:98 target_bin */
#define PQ_KL_CANDIDATES (PQ_HIST_BINS - PQ_KL_TARGET_BIN)
#define PQ_MAX_SEGMENTS 256 /* tensors per multi-tensor launch */

int pq_version(void); /* PQ_VERSION */
const char *pq_error_string(int code);

/* ---- a1: DistributionCollector.refresh_max_val, common/quantity/distribution_collector.py:70-78
 * max_bits[i] = max(max_bits[i], bits(|x|)) over tensor i, as the uint32 pattern of the
 * fp32 magnitude (monotone for non-NaN floats; reinterpret as float to read it).
 * xs_host / ns_host are HOST arrays of k device pointers / element counts. */
int pq_absmax_multi_f32(const float *const *xs_host, const uint64_t *ns_host, int k,
                        uint32_t *max_bits, pq_stream_t stream);

/* ---- extension of a1 (north_star: "per-channel and per-tensor max-abs"): the reference only ever
 * reduces per tensor (distribution_collector.py:77, tools/pytorch_quantizer.py:639,651), so this entry
 * point has no reference counterpart; its contract is the same reduction taken per channel.
 * x is a contiguous fp32 [outer][channels][inner] tensor (NCHW activations: outer = N, inner = H*W;
 * a weight [K][C][R][S] per output channel: outer = 1, channels = K, inner = C*R*S):
 *   max_bits[c] = max(max_bits[c], bits(max |x[:, c, :]|)),  uint32 pattern as in pq_absmax_multi_f32.
 * Requires channels <= 8192, inner < 2^31 - 2^14 and outer * channels < 2^31. */
int pq_absmax_per_channel_f32(const float *x, uint64_t outer, int channels, uint64_t inner,
                              uint32_t *max_bits, pq_stream_t stream);

/* ---- the elementwise glue of the fp32 calibration forward (tools/pytorch_quantizer.py fuses it during
 * Quantity.activation_quantize), each in ONE pass, bit for bit what the unfused PyTorch forward computes:
 * the IEEE fp32 add of ATen's `a + 1 * b`, nn.ReLU as ATen's clamp_min (NaN passes, else max(v, 0)), and the max
 * as pq_absmax_multi_f32 takes it.
 * pq_conv_epilogue_f32: nn.Conv2d's bias add after cuDNN, in place on a contiguous fp32 NCHW y [N][C][hw]:
 *   y += bias[c];  relu_out = relu(y) when relu_out != NULL;  *max_slot = max(*max_slot, bits(max |y|)) when
 *   max_slot != NULL (one slot of a pq_absmax_multi_f32 max_bits array).
 *   y and relu_out 16-byte aligned; N * C < 2^31, hw < 2^31, N * C * hw < 2^33 (hw % 4 != 0: < 2^31).
 * pq_eltwise_add_f32: Eltwise (fabu_layer.py:5-11), z = a + b out of place over n elements, relu_out and max_slot
 *   as above.  a, b, z, relu_out 16-byte aligned, z and relu_out alias nothing; n < 2^33. */
int pq_conv_epilogue_f32(float *y, const float *bias, int N, int C, uint64_t hw, float *relu_out,
                         uint32_t *max_slot, pq_stream_t stream);
int pq_eltwise_add_f32(const float *a, const float *b, float *z, size_t n, float *relu_out, uint32_t *max_slot,
                       pq_stream_t stream);

/* ---- a3: DistributionCollector._add_to_distribution, distribution_collector.py:127-135
 * for every x != 0:  hist[i][min((int)trunc(fl32(|x| / interval_i)), 2047)] += 1
 * with a correctly rounded fp32 division.  hist is int64 [k][2048] (the reference's int32
 * would overflow at BASELINE.json's 8192-image config; the Python layer narrows to int32
 * when it fits).  intervals_host: HOST array of k fp32 bin widths (a2, :60-61). */
int pq_hist2048_multi_f32(const float *const *xs_host, const uint64_t *ns_host,
                          const float *intervals_host, int k, long long *hist,
                          pq_stream_t stream);

/* ---- a5 + a6: Quantizer.normalize_distribution / threshold_distribution /
 * compute_kl_divergence, common/quantity/quantizer.py:95-174
 * counts: fp64 [k][2048] (integer-valued: int32 counts or the float64 group sums of
 * tools/pytorch_quantizer.py:434-445).  Outputs: threshold[k] (the chosen bin T*, first
 * strict minimum, default 2047) and, if kl != NULL, kl[k][1920] (the divergences for
 * T = 128..2047).  workspace: fp64 [k][pq_kl_workspace_doubles()] scratch.
 * All arithmetic in fp64 in the reference's operation order (numpy pairwise sums
 * included); only log() differs from numpy's by <= 1 ulp. */
size_t pq_kl_workspace_doubles(void);
int pq_kl_search_f64(const double *counts, int k, double *workspace, double *kl,
                     int *threshold, pq_stream_t stream);

/* ---- a3 / a5 / a6 for any INTERVAL_NUM (tools/configs.yml:23; DistributionCollector(interval_num=...),
 * common/quantity/distribution_collector.py:9-22, and `length = distribution.size` in
 * common/quantity/quantizer.py:98-103).  nbins == 2048 forwards to the specialised entry points above.
 * pq_hist_multi_f32: hist is int64 [k][nbins], 1 <= nbins <= PQ_HIST_BINS_MAX (else PQ_EUNSUPPORTED).
 * pq_kl_search_n_f64: counts fp64 [k][nbins], kl (optional) fp64 [k][nbins - 128], 128 < nbins <=
 * PQ_HIST_BINS_MAX (nbins <= 128: PQ_EINVAL -- the reference's candidate loop would be empty), default
 * threshold nbins - 1; workspace fp64 [k][pq_kl_workspace_doubles_n(nbins)]. */
int pq_hist_multi_f32(const float *const *xs_host, const uint64_t *ns_host, const float *intervals_host,
                      int k, int nbins, long long *hist, pq_stream_t stream);
size_t pq_kl_workspace_doubles_n(int nbins);
int pq_kl_search_n_f64(const double *counts, int k, int nbins, double *workspace, double *kl,
                       int *threshold, pq_stream_t stream);

/* ---- a10 / a12: QuanDequan.forward (new_quantity_op.py:246-257) and Quantity.forward (:48-58)
 * y = clamp(rint_half_even(x * 2^bit), lo, hi) [/ 2^bit when dequant != 0].  y must not alias x
 * (inputs are read through the non-coherent path). */
int pq_fakequant_f32(const float *x, float *y, size_t n, int bit, float lo, float hi,
                     int dequant, pq_stream_t stream);

/* ---- a15: NewAdd.forward, new_quantity_op.py:166-174:  y = clamp(a + b, lo, hi). */
int pq_add_clamp_f32(const float *a, const float *b, float *y, size_t n, float lo, float hi,
                     pq_stream_t stream);

/* ---- a14 stand-alone: RightShift.forward, new_quantity_op.py:11-44 on fp32 tensors
 * v = x / 2^rs (rs any sign); r = trunc(v + 0.5) if v > 0 else trunc(v - 0.5); y = clamp(r, lo, hi).
 * (Inside NewConv2d / NewLinear this is fused into the GEMM epilogue; this entry serves the
 * module when it is used on its own.) */
int pq_rshift_f32(const float *x, float *y, size_t n, int rs, float lo, float hi, pq_stream_t stream);

/* ---- Sp.forward (:71-91) and DeQuantity.forward (:61-68) stand-alone:
 * y = clamp(x, lo, hi) * scale  (Sp: scale = 1; DeQuantity: lo/hi = -/+inf, scale = 2^-ob). */
int pq_clamp_scale_f32(const float *x, float *y, size_t n, float lo, float hi, float scale,
                       pq_stream_t stream);

/* ---- a12 (layout-changing form): Quantity.forward fused with the NCHW -> NHWC transpose
 * the tensor-core kernels want:  q[n][h][w][c_pad] = (int8) clamp(rint(x[n][c][h][w] * 2^ib)).
 * Channels c >= C of the padded layout are written as 0. */
int pq_quantize_nchw_to_nhwc_s8(const float *x, int8_t *q, int N, int C, int H, int W, int c_pad,
                                int ib, pq_stream_t stream);

/* ---- a12 for convolutions with very few input channels (the ResNet stem): Quantity.forward fused
 * with an explicit im2col, a[m][k] = q(x[n][c][p*sh-ph+r][q*sw-pw+s]) for k = (r*S+s)*C + c, zero for
 * padding and for k in [R*S*C, kp); m = (n*P + p)*Q + q, row pitch kp bytes (multiple of 16).  The
 * result feeds pq_gemm_s8 with weights laid out [K][R][S][C] and zero-padded to kp. */
int pq_quantize_im2col_s8(const float *x, int8_t *a, int N, int C, int H, int W, int R, int S,
                          int stride_h, int stride_w, int pad_h, int pad_w, int kp, int ib,
                          pq_stream_t stream);

/* ---- a12 + a13 for convolutions with <= 8 input channels, fast form (the ResNet stem): the input
 * quantiser writes a zero-padded NHWC image with 8-byte pixels,
 *   q[n][h + pad_h][w + pad_w][c] = (int8) clamp(rint(x[n][c][h][w] * 2^ib)),  0 elsewhere   ([N][Hp][Wp][8])
 * so that the S taps of one filter row are 8*S contiguous bytes; pq_conv2d_smallc_s8 fetches them for a
 * patch of output pixels with one overlapping-stride tiled TMA per filter row (no im2col matrix in HBM).
 * desc.C must be 8; weights are [K][R][64] int8 = 8 tap slots x 8 channel slots per filter row, zero
 * where s >= S or c >= C.  Requires S <= 8, even stride_w, Hp % stride_h == 0,
 * Hp >= max((P-1)*stride_h + R, H + pad_h), Wp even, Wp >= max((Q-1)*stride_w + 8, W + pad_w).
 * desc.dil_h / dil_w must be 1 (else PQ_EUNSUPPORTED).  Epilogue, flags and outputs as pq_conv2d_s8. */
int pq_quantize_nchw_to_padded_nhwc8_s8(const float *x, int8_t *q, int N, int C, int H, int W, int pad_h,
                                        int pad_w, int Hp, int Wp, int ib, pq_stream_t stream);

/* ---- a13 + a14: NewConv2d.forward / NewLinear.forward, new_quantity_op.py:104-133,177-205
 * (Conv -> RightShift -> BiasAdd -> Sp -> DeQuantity) on int8 operands:
 *   acc  = sum_k a[m][k] * w[n][k]                 int8 x int8 -> int32 (tcgen05 kind::i8)
 *   r    = clamp(round_half_away(acc / 2^rs), -128, 127)              (RightShift, :11-44)
 *   y    = clamp(r + bias_q[n], -128, 127)                            (BiasAdd + Sp, :71-101)
 *   out  = y / 2^ob                                                   (DeQuantity, :61-68)
 * pq_gemm_s8: a is [M][K] row-major int8 (NHWC activations of a 1x1/stride-1 conv, or the
 * input of a Linear), w is [N][K] row-major int8, K % 16 == 0, 16-byte aligned rows.
 * Outputs (either may be NULL): out_f32 written as NCHW fp32 with `hw` pixels per image
 * (hw = 1 gives the plain [M][N] row-major layout of a Linear); out_s8 written [M][N].
 * pq_conv2d_s8: the same on an NHWC image, filter tap (r, s) reading input pixel
 * (p*stride_h - pad_h + r*dil_h, q*stride_w - pad_w + s*dil_w).  Dilated filters (nn.Conv2d(dilation=...) wrapped by
 * NewConv2d; the reference's weight path zero-stuffs such kernels for its target hardware,
 * tools/pytorch_quantizer.py:626-629,679-693) take the im2col-TMA path with the dilation as tap offsets, so no
 * multiply is wasted on stuffed zeros; a 1x1 filter ignores the dilation. */
typedef struct pq_conv_desc {
    int N, H, W, C;          /* input NHWC, C = padded channel count (multiple of 16) */
    int K;                   /* output channels */
    int R, S;                /* filter height / width; weights are [K][R][S][C] int8 */
    int stride_h, stride_w, pad_h, pad_w;
    int P, Q;                /* output height / width: (H + 2*pad_h - ((R-1)*dil_h + 1)) / stride_h + 1, Q alike */
    int rs;                  /* weight_bit + input_bit - output_bit, any sign */
    int ob;                  /* output_bit */
    int dil_h, dil_w;        /* dilation, >= 1 */
} pq_conv_desc;

/* flags of the GEMM / conv entry points (0: the layer as above).
 * PQ_FLAG_RELU fuses a following nn.ReLU into the GEMM / conv epilogue: y = max(y, 0).  It serves SURVEY 8(f) n1, the
 * int8 inter-layer pipeline (no reference counterpart as separate ops; the composition is bit-identical to the
 * reference's fp32-boundary chain because a layer's input_bit is its producer's output_bit in feat.table,
 * tools/pytorch_quantizer.py:468-485). */
#define PQ_FLAG_RELU 1
/* PQ_FLAG_BIAS_FOLDED: bias_q points to int32 [3][N] written by pq_bias_fold_s32 for the SAME rs (N % 16 == 0):
 *   [0] bias   [1] 2^(rs-1) + (bias << rs)
 *   [2] N/2 words of s16x2 pairs (channels 2j, 2j+1)  h = 127 + min(bias, 0),  then N/2 words of pairs
 *       l = -128 + max(bias, 0)
 * The int8-only (staged) epilogue then folds BiasAdd (new_quantity_op.py:128-131) into the rounding add of
 * RightShift (:30-37),  t = (acc + [1] + (acc >> 31)) >> rs = round_half_away(acc / 2^rs) + bias,  with RightShift's
 * saturation (:41) applied to the accumulator (channel-independent bounds) and the second one (:71-91) in the packing
 * instruction; the fused-add epilogue instead replaces both saturations by  clamp(t, l, h)  on packed 16-bit pairs
 * (the composition Sp(Sp(r) + b) is monotone in r and constant beyond the int8 range of r).  Same integers either way.
 * Ignored unless 1 <= rs <= 20 and N % 16 == 0. */
#define PQ_FLAG_BIAS_FOLDED 2
/* PQ_FLAG_NO_WINDOWS (conv only): take the im2col-TMA path even where the patch-window path applies (3x3,
 * stride 1, pad 1, C = 64 / 128, one tile of output channels); both are bit-identical, the flag exists for A/B tests. */
#define PQ_FLAG_NO_WINDOWS 4

int pq_gemm_s8(const int8_t *a, const int8_t *w, const int32_t *bias_q, int M, int N, int K, int rs, int ob, int hw,
               int flags, float *out_f32, int8_t *out_s8, pq_stream_t stream);
int pq_conv2d_s8(const int8_t *x_nhwc, const int8_t *w_krsc, const int32_t *bias_q, const pq_conv_desc *desc_host,
                 int flags, float *out_f32_nchw, int8_t *out_s8_nhwc, pq_stream_t stream);

/* out: int32 [3 * n] (rows [0], [1], [2] above; n even). */
int pq_bias_fold_s32(const int32_t *bias_q, int n, int rs, int32_t *out, pq_stream_t stream);

/* Space-to-depth form of the same input for stride-2 convolutions with C <= 4: 2 x 2 pixel blocks of the zero-padded
 * image as 16-byte pixels, q[n][i][j][(dy * 2 + dx) * 4 + c] = Quantity(ib)(x[n][c][2i + dy - pad_t][2j + dx - pad_l])
 * (0 outside the image / for c >= C); pad_t, pad_l even.  Viewed as [N][Hp2][2 * Wp2][8] it is a valid input of
 * pq_conv2d_smallc_s8 for the equivalent stride-(1, 2) filter of ceil((R + 1) / 2) rows (NewConv2d builds the weights):
 * the ResNet stem then needs 8 instead of 14 tensor-core instructions per tile and reads half the bytes. */
int pq_quantize_nchw_to_s2d16_s8(const float *x, int8_t *q, int N, int C, int H, int W, int pad_t, int pad_l,
                                 int Hp2, int Wp2, int ib, pq_stream_t stream);

int pq_conv2d_smallc_s8(const int8_t *xp, const int8_t *w_krs8, const int32_t *bias_q,
                        const pq_conv_desc *desc_host, int Hp, int Wp, int flags, float *out_f32_nchw,
                        int8_t *out_s8_nhwc, pq_stream_t stream);

/* Global average pool of a quantised NHWC payload (int8, or the int16 exact sum of a NewAdd) at fractional bit `bit`,
 * with an optional pending ReLU: out[N][C] fp32 = nn.AvgPool2d(H)(DeQuantity(x)) bit for bit -- the fp32 window sum of
 * the reference is exact while HW * max|x| < 2^24 (otherwise PQ_EUNSUPPORTED), then one IEEE division by HW as in
 * ATen's avg_pool2d.  The pipeline's replacement for de-quantise + F.avg_pool2d (quantity/model/resnet: AvgPool2d ->
 * View -> NewLinear).  C % 8 == 0. */
int pq_avgpool_global_nhwc_f32(const void *x, int is16, int bit, int relu, int N, int HW, int C, float *out,
                               pq_stream_t stream);

/* y = max(x, 0) on int8 (nn.ReLU on a quantised tensor: relu commutes with the input quantiser). */
int pq_relu_s8(const int8_t *x, int8_t *y, size_t n, pq_stream_t stream);

/* nn.MaxPool2d on int8 NHWC (max commutes with the monotone quantiser); relu != 0 also applies max(.,0).
 * Padding behaves like -inf, as in torch. */
int pq_maxpool_nhwc_s8(const int8_t *x, int8_t *y, int N, int H, int W, int C, int k, int stride, int pad,
                       int relu, pq_stream_t stream);

/* NewAdd.forward (new_quantity_op.py:166-174) on quantised operands, exactly:
 *   s = clamp(a / 2^a_bit + b / 2^b_bit, -128, 127)       a, b: int8 or int16 (a_is16 / b_is16),
 *                                                           a_relu / b_relu apply max(.,0) on load
 *   out16 = s * 2^o_bit (int16, o_bit = max(a_bit, b_bit), exact)      -> the identity shortcut of the next add
 *   out8  = clamp(round_half_even(s * 2^q_bit), -128, 127) (int8)      -> Quantity(q_bit) of the consuming convs
 * flags & PQ_FLAG_RELU: the nn.ReLU that follows the Eltwise is applied to s before both outputs
 * (max(.,0) commutes with the monotone quantiser, so out8 equals Quantity(q_bit)(relu(s))).
 * Either output may be NULL.  Requires 0 <= o_bit - min(a_bit, b_bit) <= 7 and |q_bit - o_bit| <= 15. */
int pq_add_requant(const void *a, int a_is16, int a_bit, int a_relu, const void *b, int b_is16, int b_bit,
                   int b_relu, size_t n, int flags, int16_t *out16, int8_t *out8, int q_bit, pq_stream_t stream);

/* Concat (fabu_layer.py:14-20, left in place by tools/reconstruction.py:219-238) followed by the
 * consumer's input quantiser Quantity(q_bit) (new_quantity_op.py:48-58), on quantised operands: source i is
 * int8 or int16 [pixels][channels_i] (NHWC, channel-last) holding v / 2^bit_i; the output is int8
 * [pixels][c_out_pad] with the sources side by side along the channel axis,
 *   out[p][off_i + c] = clamp(round_half_even(relu_i?(v) * 2^(q_bit - bit_i)), -128, 127),
 * which is exactly Quantity(q_bit)(torch.cat(de-quantised sources, 1)) because every product is an exact
 * fp32 value.  Channels sum(channels_i) .. c_out_pad-1 are zero-filled (tensor-core channel padding).
 * srcs_host is a HOST array of k <= PQ_CONCAT_MAX_SOURCES descriptors; |q_bit - bit_i| <= 15. */
#define PQ_CONCAT_MAX_SOURCES 8
typedef struct pq_concat_src {
    const void *ptr;
    int is16;                /* int16 payload (the exact sum of an Eltwise) instead of int8 */
    int channels;
    int bit;
    int relu;                /* apply max(., 0) on load (a pending nn.ReLU) */
} pq_concat_src;
int pq_concat_requant_s8(const pq_concat_src *srcs_host, int k, size_t pixels, int q_bit, int c_out_pad,
                         int8_t *out, pq_stream_t stream);

/* NewConv2d + NewAdd (+ the nn.ReLU after the Eltwise) in ONE kernel: the conv / GEMM epilogue adds the
 * shortcut operand and writes the exact int16 sum and its int8 requantisation, exactly as pq_add_requant
 * would on the conv's int8 result (which is never written to memory).  conv operand: y at bit `ob` of the
 * conv descriptor; shortcut: int8 or int16 [M][N] row-major (NHWC) at bit shortcut_bit.  N % 16 == 0. */
typedef struct pq_add_desc {
    const void *shortcut;
    int shortcut_is16, shortcut_bit, shortcut_relu;
    int out_relu;            /* nn.ReLU after the Eltwise */
    int q_bit;               /* the Eltwise's feat bit: out8 = Quantity(q_bit)(sum) */
    int16_t *out16;          /* exact sum at o_bit = max(ob, shortcut_bit); may be NULL */
    int8_t *out8;            /* required */
} pq_add_desc;
/* flags: PQ_FLAG_BIAS_FOLDED (bias_q as written by pq_bias_fold_s32); PQ_FLAG_RELU is rejected with PQ_EINVAL
 * (the ReLU of a fused add is add_host->out_relu). */
int pq_conv2d_s8_add(const int8_t *x_nhwc, const int8_t *w_krsc, const int32_t *bias_q, const pq_conv_desc *desc_host,
                     const pq_add_desc *add_host, int flags, pq_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PQ_SM100_H */

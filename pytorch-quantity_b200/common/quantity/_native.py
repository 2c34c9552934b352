"""ctypes binding of libpq_sm100.so (the C ABI declared in include/pq_sm100.h).

PyTorch supplies device memory and streams; every kernel on the calibration / simulation
hot path is one of the hand-written sm_100a kernels behind these symbols.  There is no CPU
or eager fallback: if the library is missing, or a tensor is not on a CUDA device, the
call raises.
"""
import ctypes
import os

import numpy as np
import torch

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
LIB_PATH = os.path.join(_PKG_ROOT, "lib", "libpq_sm100.so")

HIST_BINS = 2048
HIST_BINS_MAX = 8192
KL_TARGET_BIN = 128
KL_CANDIDATES = HIST_BINS - KL_TARGET_BIN
MAX_SEGMENTS = 256
PQ_VERSION = 201             # the header's PQ_VERSION: the entry points below match a library built from it

# every symbol include/pq_sm100.h declares: (restype, argtypes)
_vp, _i, _sz, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t, ctypes.c_float
SYMBOLS = {
    "pq_version": (_i, []),
    "pq_error_string": (ctypes.c_char_p, [_i]),
    "pq_absmax_multi_f32": (_i, [_vp, _vp, _i, _vp, _vp]),
    "pq_absmax_per_channel_f32": (_i, [_vp, ctypes.c_uint64, _i, ctypes.c_uint64, _vp, _vp]),
    "pq_conv_epilogue_f32": (_i, [_vp, _vp, _i, _i, ctypes.c_uint64, _vp, _vp, _vp]),
    "pq_eltwise_add_f32": (_i, [_vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "pq_hist2048_multi_f32": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "pq_kl_workspace_doubles": (_sz, []),
    "pq_kl_search_f64": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "pq_hist_multi_f32": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "pq_kl_workspace_doubles_n": (_sz, [_i]),
    "pq_kl_search_n_f64": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp]),
    "pq_fakequant_f32": (_i, [_vp, _vp, _sz, _i, _f, _f, _i, _vp]),
    "pq_add_clamp_f32": (_i, [_vp, _vp, _vp, _sz, _f, _f, _vp]),
    "pq_rshift_f32": (_i, [_vp, _vp, _sz, _i, _f, _f, _vp]),
    "pq_clamp_scale_f32": (_i, [_vp, _vp, _sz, _f, _f, _f, _vp]),
    "pq_quantize_nchw_to_nhwc_s8": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "pq_quantize_im2col_s8": (_i, [_vp, _vp] + [_i] * 12 + [_vp]),
    "pq_quantize_nchw_to_padded_nhwc8_s8": (_i, [_vp, _vp] + [_i] * 9 + [_vp]),
    "pq_conv2d_smallc_s8": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "pq_quantize_nchw_to_s2d16_s8": (_i, [_vp, _vp] + [_i] * 9 + [_vp]),
    "pq_gemm_s8": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pq_conv2d_s8": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "pq_conv2d_s8_add": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "pq_relu_s8": (_i, [_vp, _vp, _sz, _vp]),
    "pq_maxpool_nhwc_s8": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "pq_avgpool_global_nhwc_f32": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "pq_add_requant": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _sz, _i, _vp, _vp, _i, _vp]),
    "pq_concat_requant_s8": (_i, [_vp, _i, _sz, _i, _i, _vp, _vp]),
    "pq_bias_fold_s32": (_i, [_vp, _i, _i, _vp, _vp]),
}
FLAG_RELU = 1
FLAG_BIAS_FOLDED = 2
FLAG_NO_WINDOWS = 4          # pq_conv2d_s8: force the im2col-TMA path (A/B tests of the patch-window path)


class ConvDesc(ctypes.Structure):
    """struct pq_conv_desc"""
    _fields_ = [(n, ctypes.c_int) for n in
                ("N", "H", "W", "C", "K", "R", "S", "stride_h", "stride_w", "pad_h", "pad_w",
                 "P", "Q", "rs", "ob", "dil_h", "dil_w")]


class AddDesc(ctypes.Structure):
    """struct pq_add_desc"""
    _fields_ = [("shortcut", ctypes.c_void_p), ("shortcut_is16", ctypes.c_int), ("shortcut_bit", ctypes.c_int),
                ("shortcut_relu", ctypes.c_int), ("out_relu", ctypes.c_int), ("q_bit", ctypes.c_int),
                ("out16", ctypes.c_void_p), ("out8", ctypes.c_void_p)]


class ConcatSrc(ctypes.Structure):
    """struct pq_concat_src"""
    _fields_ = [("ptr", ctypes.c_void_p), ("is16", ctypes.c_int), ("channels", ctypes.c_int),
                ("bit", ctypes.c_int), ("relu", ctypes.c_int)]


CONCAT_MAX_SOURCES = 8

_lib = None

# ---- instrumentation used by bench.py: launch counts always; CUDA-event timing of each launch
# on its launching stream when a profile dict is installed with set_profile().
LAUNCHES = {"total": 0}
_profile = None


def set_profile(store):
    """store: None (off) or a dict; every C-ABI launch appends (start_evt, end_evt, alg_bytes)
    to store[kernel_name]."""
    global _profile
    _profile = store


class _Timed:
    def __init__(self, name, kernels, alg_bytes, device):
        self.name, self.kernels, self.alg_bytes, self.device = name, kernels, alg_bytes, device

    def __enter__(self):
        LAUNCHES["total"] += self.kernels
        LAUNCHES[self.name] = LAUNCHES.get(self.name, 0) + self.kernels
        if _profile is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record(torch.cuda.current_stream(self.device))
        return self

    def __exit__(self, *exc):
        if _profile is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record(torch.cuda.current_stream(self.device))
            _profile.setdefault(self.name, []).append((self.start, end, self.alg_bytes))
        return False


def lib():
    """Load the library once.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libpq_sm100.so not found at %s -- build it with `python __graft_entry__.py` "
                "(or `make -C pytorch-quantity_b200/csrc`).  This package has no CPU fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        handle.pq_version.restype, handle.pq_version.argtypes = SYMBOLS["pq_version"]
        if handle.pq_version() != PQ_VERSION:
            raise ImportError(
                "%s is version %d, this package needs %d -- rebuild with `python __graft_entry__.py`"
                % (LIB_PATH, handle.pq_version(), PQ_VERSION))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)          # AttributeError if the .so lacks a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed: %s (code %d)" % (what, lib().pq_error_string(rc).decode(), rc))


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def require_cuda(t, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s needs a CUDA tensor: the B200 path has no CPU fallback" % what)


def to_device_f32(x, device=None):
    """Accept CUDA tensors (fast path) or numpy / CPU tensors (compatibility path: one
    host->device copy, then the same kernels).  Returns a contiguous 1-D fp32 CUDA tensor."""
    if isinstance(x, torch.Tensor):
        t = x.detach()
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x)))
    if not t.is_cuda:
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: pytorch-quantity_b200 has no CPU fallback")
        t = t.to(device or "cuda", non_blocking=True)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous().view(-1)


def _seg_arrays(tensors):
    k = len(tensors)
    ptrs = (ctypes.c_void_p * k)(*[t.data_ptr() if t.numel() else 0 for t in tensors])
    ns = (ctypes.c_uint64 * k)(*[t.numel() for t in tensors])
    return ptrs, ns


def absmax_multi(tensors, max_bits):
    """max_bits (int32 CUDA [>=k], bit patterns of fp32 magnitudes) |= max over each tensor."""
    for lo in range(0, len(tensors), MAX_SEGMENTS):
        part = tensors[lo:lo + MAX_SEGMENTS]
        ptrs, ns = _seg_arrays(part)
        out = max_bits[lo:lo + len(part)]
        with _Timed("absmax", 1, 4 * sum(t.numel() for t in part), max_bits.device):
            check(lib().pq_absmax_multi_f32(ptrs, ns, len(part), out.data_ptr(), _stream(max_bits)),
                  "pq_absmax_multi_f32")


def absmax_per_channel(x, max_bits, channel_dim=1):
    """max_bits (int32 CUDA [C]) |= bit pattern of max |x| over every axis but `channel_dim` of the
    contiguous fp32 CUDA tensor x (extension of a1; see include/pq_sm100.h)."""
    require_cuda(x, "absmax_per_channel")
    if x.dtype != torch.float32:
        raise RuntimeError("fp32 expected, got %s" % x.dtype)
    xc = x.detach().contiguous()
    shape = tuple(xc.shape)
    channel_dim %= len(shape)
    outer = int(np.prod(shape[:channel_dim], dtype=np.int64))
    inner = int(np.prod(shape[channel_dim + 1:], dtype=np.int64))
    C = shape[channel_dim]
    assert max_bits.dtype == torch.int32 and max_bits.numel() >= C and max_bits.is_contiguous()
    with _Timed("absmax_channel", 1, 4 * xc.numel(), xc.device):
        check(lib().pq_absmax_per_channel_f32(xc.data_ptr() if xc.numel() else None, outer, C, inner,
                                              max_bits.data_ptr(), _stream(xc)), "pq_absmax_per_channel_f32")


def _require_f32_contiguous(tensors, what):
    """The fused calibration kernels address fp32 elements of contiguous tensors on one CUDA device."""
    dev = tensors[0].device
    for t in tensors:
        require_cuda(t, what)
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev:
            raise RuntimeError("%s needs contiguous fp32 tensors on %s, got %s %s on %s"
                               % (what, dev, t.dtype, "contiguous" if t.is_contiguous() else "strided", t.device))


def conv_epilogue(y, bias, relu=False, max_slot=None):
    """nn.Conv2d's bias add after a bias-less cuDNN convolution, in place on y (contiguous fp32 CUDA [N][C][H][W]):
    y += bias[c].  Returns relu(y) as a new tensor when `relu`, else None.  max_slot: device address of one int32 of
    an absmax_multi max_bits array that takes max |y|, or None.  Launched on y's current stream."""
    _require_f32_contiguous((y, bias), "conv_epilogue")
    N, C, H, W = y.shape
    if bias.numel() != C:
        raise RuntimeError("conv_epilogue: %d bias values for %d channels" % (bias.numel(), C))
    r = torch.empty_like(y) if relu else None
    with _Timed("conv_epilogue", 1, y.numel() * (12 if relu else 8), y.device):
        check(lib().pq_conv_epilogue_f32(y.data_ptr(), bias.data_ptr(), N, C, H * W, r.data_ptr() if relu else None,
                                         max_slot, _stream(y)), "pq_conv_epilogue_f32")
    return r


def eltwise_add(a, b, relu=False, max_slot=None):
    """Eltwise: a + b for contiguous fp32 CUDA tensors of one shape.  Returns (sum, relu(sum) or None); max_slot as in
    conv_epilogue."""
    _require_f32_contiguous((a, b), "eltwise_add")
    if a.shape != b.shape:
        raise RuntimeError("eltwise_add: shapes %s and %s differ" % (tuple(a.shape), tuple(b.shape)))
    z = torch.empty_like(a)
    r = torch.empty_like(a) if relu else None
    with _Timed("eltwise", 1, a.numel() * (16 if relu else 12), a.device):
        check(lib().pq_eltwise_add_f32(a.data_ptr(), b.data_ptr(), z.data_ptr(), a.numel(),
                                       r.data_ptr() if relu else None, max_slot, _stream(a)),
              "pq_eltwise_add_f32")
    return z, r


def hist_multi(tensors, intervals, hist):
    """hist (int64 CUDA [k][nbins]) += nbins-bin |x| histograms with per-tensor fp32 bin width
    (nbins = hist.shape[1]: 2048 takes the specialised kernel, anything else up to 8192 the generic one)."""
    nbins = int(hist.shape[1])
    for lo in range(0, len(tensors), MAX_SEGMENTS):
        part = tensors[lo:lo + MAX_SEGMENTS]
        ptrs, ns = _seg_arrays(part)
        iv = (ctypes.c_float * len(part))(*[float(v) for v in intervals[lo:lo + len(part)]])
        out = hist[lo:lo + len(part)]
        with _Timed("hist", 1, 4 * sum(t.numel() for t in part), hist.device):
            if nbins == HIST_BINS:
                check(lib().pq_hist2048_multi_f32(ptrs, ns, iv, len(part), out.data_ptr(), _stream(hist)),
                      "pq_hist2048_multi_f32")
            else:
                check(lib().pq_hist_multi_f32(ptrs, ns, iv, len(part), nbins, out.data_ptr(), _stream(hist)),
                      "pq_hist_multi_f32 (INTERVAL_NUM=%d)" % nbins)


def kl_search(counts_f64, want_curves=False):
    """counts_f64: CUDA fp64 [k][nbins].  Returns (threshold int32 [k], kl fp64 [k][nbins - 128] or None)."""
    require_cuda(counts_f64, "kl_search")
    assert counts_f64.dtype == torch.float64 and counts_f64.dim() == 2
    nbins = int(counts_f64.shape[1])
    counts_f64 = counts_f64.contiguous()
    k = counts_f64.shape[0]
    dev = counts_f64.device
    ws = torch.empty(k * lib().pq_kl_workspace_doubles_n(nbins), dtype=torch.float64, device=dev)
    thr = torch.empty(k, dtype=torch.int32, device=dev)
    kl = torch.empty((k, max(nbins - KL_TARGET_BIN, 0)), dtype=torch.float64, device=dev) if want_curves else None
    with _Timed("kl", 3, 8 * counts_f64.numel(), dev):
        check(lib().pq_kl_search_n_f64(counts_f64.data_ptr(), k, nbins, ws.data_ptr(),
                                       kl.data_ptr() if want_curves else None, thr.data_ptr(),
                                       _stream(counts_f64)), "pq_kl_search_n_f64 (INTERVAL_NUM=%d)" % nbins)
    return thr, kl


def bias_fold(bias_i32, rs):
    """int32 [N] quantised bias -> int32 [3N]: the bias, then 2^(rs-1) + (bias << rs) (the per-channel constant
    of the folded int8 epilogue), then the post-shift saturation bounds as s16x2 pairs (PQ_FLAG_BIAS_FOLDED,
    include/pq_sm100.h).  Returned unchanged when the fold does not apply (N % 16 != 0 or rs outside [1, 20])."""
    require_cuda(bias_i32, "bias_fold")
    n = bias_i32.numel()
    if n % 16 or bias_i32.dtype != torch.int32 or not 1 <= int(rs) <= 20:
        return bias_i32
    out = torch.empty(3 * n, dtype=torch.int32, device=bias_i32.device)
    check(lib().pq_bias_fold_s32(bias_i32.contiguous().data_ptr(), n, int(rs), out.data_ptr(), _stream(bias_i32)),
          "pq_bias_fold_s32")
    return out


def conv_out_size(in_hw, kernel, stride, padding, dilation=(1, 1)):
    """(P, Q): output height and width of a convolution, as nn.Conv2d computes them."""
    return ((in_hw[0] + 2 * padding[0] - (kernel[0] - 1) * dilation[0] - 1) // stride[0] + 1,
            (in_hw[1] + 2 * padding[1] - (kernel[1] - 1) * dilation[1] - 1) // stride[1] + 1)


def _conv_desc(N, H, W, C, K, kernel, stride, padding, rs, ob, dilation=(1, 1)):
    P, Q = conv_out_size((H, W), kernel, stride, padding, dilation)
    return ConvDesc(N, H, W, C, K, kernel[0], kernel[1], stride[0], stride[1], padding[0], padding[1], P, Q,
                    int(rs), int(ob), dilation[0], dilation[1])


def _bias_flags(bias_q, n, relu):
    return (FLAG_RELU if relu else 0) | (FLAG_BIAS_FOLDED if bias_q.numel() == 3 * n else 0)


def _flat_out(x):
    require_cuda(x, "elementwise kernel")
    if x.dtype != torch.float32:
        raise RuntimeError("fp32 expected, got %s" % x.dtype)
    xc = x.contiguous()
    return xc, torch.empty_like(xc)


def fakequant(x, bit, lo=-128.0, hi=127.0, dequant=True):
    xc, y = _flat_out(x)
    with _Timed("fakequant", 1, 8 * xc.numel(), xc.device):
        check(lib().pq_fakequant_f32(xc.data_ptr(), y.data_ptr(), xc.numel(), int(bit), lo, hi,
                                     1 if dequant else 0, _stream(xc)), "pq_fakequant_f32")
    return y


def add_clamp(a, b, lo=-128.0, hi=127.0):
    require_cuda(b, "add_clamp")
    if a.shape != b.shape:
        a, b = torch.broadcast_tensors(a, b)
    ac, y = _flat_out(a)
    bc = b.contiguous()
    with _Timed("add_clamp", 1, 12 * ac.numel(), ac.device):
        check(lib().pq_add_clamp_f32(ac.data_ptr(), bc.data_ptr(), y.data_ptr(), ac.numel(), lo, hi,
                                     _stream(ac)), "pq_add_clamp_f32")
    return y


def rshift(x, rs, lo=-128.0, hi=127.0):
    xc, y = _flat_out(x)
    check(lib().pq_rshift_f32(xc.data_ptr(), y.data_ptr(), xc.numel(), int(rs), lo, hi, _stream(xc)),
          "pq_rshift_f32")
    return y


def clamp_scale(x, lo, hi, scale):
    xc, y = _flat_out(x)
    check(lib().pq_clamp_scale_f32(xc.data_ptr(), y.data_ptr(), xc.numel(), lo, hi, scale, _stream(xc)),
          "pq_clamp_scale_f32")
    return y


def quantize_nchw_to_nhwc_s8(x, ib, c_pad):
    require_cuda(x, "quantize_nchw_to_nhwc_s8")
    assert x.dim() == 4 and x.dtype == torch.float32
    xc = x.contiguous()
    N, C, H, W = xc.shape
    q = torch.empty((N, H, W, c_pad), dtype=torch.int8, device=x.device)
    with _Timed("quantize_s8", 1, xc.numel() * 4 + q.numel(), xc.device):
        check(lib().pq_quantize_nchw_to_nhwc_s8(xc.data_ptr(), q.data_ptr(), N, C, H, W, c_pad, int(ib),
                                                _stream(xc)), "pq_quantize_nchw_to_nhwc_s8")
    return q


def quantize_im2col_s8(x, ib, kernel, stride, padding, kp):
    """fp32 NCHW -> int8 [N*P*Q][kp] im2col matrix (small-Cin convolutions)."""
    require_cuda(x, "quantize_im2col_s8")
    assert x.dim() == 4 and x.dtype == torch.float32
    xc = x.contiguous()
    N, C, H, W = xc.shape
    R, S = kernel
    P, Q = conv_out_size((H, W), kernel, stride, padding)
    a = torch.empty((N * P * Q, kp), dtype=torch.int8, device=x.device)
    with _Timed("quantize_s8", 1, xc.numel() * 4 + a.numel(), xc.device):
        check(lib().pq_quantize_im2col_s8(xc.data_ptr(), a.data_ptr(), N, C, H, W, R, S, stride[0], stride[1],
                                          padding[0], padding[1], kp, int(ib), _stream(xc)),
              "pq_quantize_im2col_s8")
    return a, (N, P, Q)


def quantize_pad_nhwc8_s8(x, ib, padding, Hp, Wp):
    """fp32 NCHW (C <= 8) -> zero-padded int8 [N][Hp][Wp][8] for conv2d_smallc_s8."""
    require_cuda(x, "quantize_pad_nhwc8_s8")
    assert x.dim() == 4 and x.dtype == torch.float32
    xc = x.contiguous()
    N, C, H, W = xc.shape
    q = torch.empty((N, Hp, Wp, 8), dtype=torch.int8, device=x.device)
    with _Timed("quantize_s8", 1, xc.numel() * 4 + q.numel(), xc.device):
        check(lib().pq_quantize_nchw_to_padded_nhwc8_s8(xc.data_ptr(), q.data_ptr(), N, C, H, W, padding[0],
                                                        padding[1], Hp, Wp, int(ib), _stream(xc)),
              "pq_quantize_nchw_to_padded_nhwc8_s8")
    return q


def quantize_s2d16_s8(x, ib, pad_tl, Hp2, Wp2):
    """fp32 NCHW (C <= 4) -> int8 [N][Hp2][Wp2][16]: 2 x 2 blocks of the zero-padded image (even pad_tl) as 16-byte
    pixels, the input of the space-to-depth form of a stride-2 small-channel convolution."""
    require_cuda(x, "quantize_s2d16_s8")
    assert x.dim() == 4 and x.dtype == torch.float32
    xc = x.contiguous()
    N, C, H, W = xc.shape
    q = torch.empty((N, Hp2, Wp2, 16), dtype=torch.int8, device=x.device)
    with _Timed("quantize_s8", 1, xc.numel() * 4 + q.numel(), xc.device):
        check(lib().pq_quantize_nchw_to_s2d16_s8(xc.data_ptr(), q.data_ptr(), N, C, H, W, pad_tl[0], pad_tl[1], Hp2, Wp2,
                                                 int(ib), _stream(xc)), "pq_quantize_nchw_to_s2d16_s8")
    return q


def conv2d_smallc_s8(xp, w_krs8, bias_q, in_hw, kernel, stride, padding, rs, ob, want_f32=True, want_s8=False,
                     c_real=None, relu=False, ops=None):
    """xp int8 [N][Hp][Wp][8] (padded), w_krs8 int8 [K][R][64] -> fp32 NCHW and / or int8 NHWC."""
    require_cuda(xp, "conv2d_smallc_s8")
    N, Hp, Wp, _ = xp.shape
    K = w_krs8.shape[0]
    R, S = kernel
    d = _conv_desc(N, in_hw[0], in_hw[1], 8, K, kernel, stride, padding, rs, ob)
    P, Q = d.P, d.Q
    out_f32 = torch.empty((N, K, P, Q), dtype=torch.float32, device=xp.device) if want_f32 else None
    out_s8 = torch.empty((N, P, Q, K), dtype=torch.int8, device=xp.device) if want_s8 else None
    with _Timed("conv_s8", 1, ops or 2 * N * P * Q * K * R * S * (c_real or 8), xp.device):        # int8 ops
        check(lib().pq_conv2d_smallc_s8(xp.data_ptr(), w_krs8.data_ptr(), bias_q.data_ptr(), ctypes.byref(d), Hp, Wp,
                                        _bias_flags(bias_q, K, relu), out_f32.data_ptr() if want_f32 else None,
                                        out_s8.data_ptr() if want_s8 else None, _stream(xp)), "pq_conv2d_smallc_s8")
    return out_f32, out_s8


def gemm_s8(a, w, bias_q, rs, ob, hw=1, want_f32=True, want_s8=False, k_real=None, relu=False):
    """a int8 [M][K], w int8 [N][K], bias_q int32 [N] -> fp32 (NCHW with hw pixels per image,
    or [M][N] when hw == 1) and / or int8 [M][N]."""
    require_cuda(a, "gemm_s8")
    M, K = a.shape
    N = w.shape[0]
    out_f32 = out_s8 = None
    if want_f32:
        out_f32 = torch.empty((M // hw, N, hw) if hw > 1 else (M, N), dtype=torch.float32, device=a.device)
    if want_s8:
        out_s8 = torch.empty((M, N), dtype=torch.int8, device=a.device)
    with _Timed("gemm_s8", 1, 2 * M * N * (k_real or K), a.device):      # "bytes" field carries int8 ops here
        check(lib().pq_gemm_s8(a.data_ptr(), w.data_ptr(), bias_q.data_ptr(), M, N, K, int(rs), int(ob), hw,
                               _bias_flags(bias_q, N, relu), out_f32.data_ptr() if want_f32 else None,
                               out_s8.data_ptr() if want_s8 else None, _stream(a)), "pq_gemm_s8")
    return out_f32, out_s8


def conv2d_s8(x_nhwc, w_krsc, bias_q, stride, padding, rs, ob, want_f32=True, want_s8=False, c_real=None,
              relu=False, dilation=(1, 1), windows=True):
    require_cuda(x_nhwc, "conv2d_s8")
    N, H, W, C = x_nhwc.shape
    K, R, S, C2 = w_krsc.shape
    assert C == C2
    dilation = (int(dilation[0]), int(dilation[1])) if (R, S) != (1, 1) else (1, 1)
    d = _conv_desc(N, H, W, C, K, (R, S), stride, padding, rs, ob, dilation)
    P, Q = d.P, d.Q
    out_f32 = torch.empty((N, K, P, Q), dtype=torch.float32, device=x_nhwc.device) if want_f32 else None
    out_s8 = torch.empty((N, P, Q, K), dtype=torch.int8, device=x_nhwc.device) if want_s8 else None
    with _Timed("conv_s8", 1, 2 * N * P * Q * K * R * S * (c_real or C), x_nhwc.device):   # int8 ops
        check(lib().pq_conv2d_s8(x_nhwc.data_ptr(), w_krsc.data_ptr(), bias_q.data_ptr(), ctypes.byref(d),
                                 _bias_flags(bias_q, K, relu) | (0 if windows else FLAG_NO_WINDOWS),
                                 out_f32.data_ptr() if want_f32 else None,
                                 out_s8.data_ptr() if want_s8 else None, _stream(x_nhwc)), "pq_conv2d_s8")
    return out_f32, out_s8


def conv2d_s8_add(x_nhwc, w_krsc, bias_q, stride, padding, rs, ob, shortcut, shortcut_bit, shortcut_relu, q_bit,
                  out_relu, want16=True, c_real=None):
    """NewConv2d + NewAdd (+ ReLU) in one kernel: returns (int16 exact sum or None, int8 at q_bit), both NHWC.
    `shortcut` is int8 or int16 with the conv output's [N][P][Q][K] shape."""
    require_cuda(x_nhwc, "conv2d_s8_add")
    N, H, W, C = x_nhwc.shape
    K, R, S, C2 = w_krsc.shape
    assert C == C2
    d = _conv_desc(N, H, W, C, K, (R, S), stride, padding, rs, ob)
    P, Q = d.P, d.Q
    assert tuple(shortcut.shape) == (N, P, Q, K) and shortcut.is_contiguous()
    out16 = torch.empty((N, P, Q, K), dtype=torch.int16, device=x_nhwc.device) if want16 else None
    out8 = torch.empty((N, P, Q, K), dtype=torch.int8, device=x_nhwc.device)
    add = AddDesc(shortcut.data_ptr(), 1 if shortcut.dtype == torch.int16 else 0, int(shortcut_bit),
                  1 if shortcut_relu else 0, 1 if out_relu else 0, int(q_bit),
                  out16.data_ptr() if want16 else None, out8.data_ptr())
    with _Timed("conv_add_s8", 1, 2 * N * P * Q * K * R * S * (c_real or C), x_nhwc.device):        # int8 ops
        check(lib().pq_conv2d_s8_add(x_nhwc.data_ptr(), w_krsc.data_ptr(), bias_q.data_ptr(), ctypes.byref(d),
                                     ctypes.byref(add), _bias_flags(bias_q, K, False), _stream(x_nhwc)),
              "pq_conv2d_s8_add")
    return out16, out8


def relu_s8(x):
    require_cuda(x, "relu_s8")
    xc = x.contiguous()
    y = torch.empty_like(xc)
    with _Timed("relu_s8", 1, 2 * xc.numel(), xc.device):
        check(lib().pq_relu_s8(xc.data_ptr(), y.data_ptr(), xc.numel(), _stream(xc)), "pq_relu_s8")
    return y


def maxpool_nhwc_s8(x, k, stride, pad, relu=False):
    require_cuda(x, "maxpool_nhwc_s8")
    N, H, W, C = x.shape
    P, Q = conv_out_size((H, W), (k, k), (stride, stride), (pad, pad))
    y = torch.empty((N, P, Q, C), dtype=torch.int8, device=x.device)
    with _Timed("maxpool_s8", 1, x.numel() + y.numel(), x.device):
        check(lib().pq_maxpool_nhwc_s8(x.data_ptr(), y.data_ptr(), N, H, W, C, k, stride, pad, 1 if relu else 0,
                                       _stream(x)), "pq_maxpool_nhwc_s8")
    return y


def avgpool_global_nhwc(x, bit, relu=False):
    """int8 / int16 NHWC payload at fractional bit `bit` -> fp32 [N][C][1][1] = AvgPool2d over the whole plane of the
    de-quantised tensor (None when the exactness condition of pq_avgpool_global_nhwc_f32 does not hold)."""
    require_cuda(x, "avgpool_global_nhwc")
    N, H, W, C = x.shape
    is16 = x.dtype == torch.int16
    if C % 8 or H * W * (32768 if is16 else 128) >= (1 << 24) or not x.is_contiguous():
        return None
    y = torch.empty((N, C, 1, 1), dtype=torch.float32, device=x.device)
    with _Timed("avgpool_s8", 1, x.numel() * x.element_size() + y.numel() * 4, x.device):
        check(lib().pq_avgpool_global_nhwc_f32(x.data_ptr(), 1 if is16 else 0, int(bit), 1 if relu else 0, N, H * W, C,
                                               y.data_ptr(), _stream(x)), "pq_avgpool_global_nhwc_f32")
    return y


def add_requant(a, a_bit, a_relu, b, b_bit, b_relu, q_bit, want16=True, want8=True, out_relu=False):
    """Exact NewAdd on quantised operands (int8 or int16 tensors of identical shape); out_relu fuses
    the nn.ReLU that follows the Eltwise."""
    require_cuda(a, "add_requant")
    assert a.shape == b.shape and a.is_contiguous() and b.is_contiguous()
    out16 = torch.empty(a.shape, dtype=torch.int16, device=a.device) if want16 else None
    out8 = torch.empty(a.shape, dtype=torch.int8, device=a.device) if want8 else None
    nbytes = a.numel() * (a.element_size() + b.element_size() + (2 if want16 else 0) + (1 if want8 else 0))
    with _Timed("add_requant", 1, nbytes, a.device):
        check(lib().pq_add_requant(a.data_ptr(), 1 if a.dtype == torch.int16 else 0, int(a_bit),
                                   1 if a_relu else 0, b.data_ptr(), 1 if b.dtype == torch.int16 else 0,
                                   int(b_bit), 1 if b_relu else 0, a.numel(), FLAG_RELU if out_relu else 0,
                                   out16.data_ptr() if want16 else None, out8.data_ptr() if want8 else None,
                                   int(q_bit), _stream(a)), "pq_add_requant")
    return out16, out8


def concat_requant_s8(sources, q_bit, c_out_pad=None):
    """Concat along channels + Quantity(q_bit) on quantised NHWC payloads.  sources: list of
    (payload int8 / int16 [N][H][W][C_i], bit, relu).  Returns int8 [N][H][W][c_out_pad]."""
    first = sources[0][0]
    require_cuda(first, "concat_requant_s8")
    N, H, W = first.shape[:3]
    k = len(sources)
    if k > CONCAT_MAX_SOURCES:
        raise RuntimeError("concat_requant_s8: at most %d sources" % CONCAT_MAX_SOURCES)
    arr = (ConcatSrc * k)()
    c_sum = nbytes = 0
    for i, (t, bit, relu) in enumerate(sources):
        assert t.is_contiguous() and tuple(t.shape[:3]) == (N, H, W) and t.dtype in (torch.int8, torch.int16)
        arr[i] = ConcatSrc(t.data_ptr(), 1 if t.dtype == torch.int16 else 0, t.shape[3], int(bit), 1 if relu else 0)
        c_sum += t.shape[3]
        nbytes += t.numel() * t.element_size()
    c_out_pad = c_sum if c_out_pad is None else c_out_pad
    out = torch.empty((N, H, W, c_out_pad), dtype=torch.int8, device=first.device)
    with _Timed("concat_requant", 1, nbytes + out.numel(), first.device):
        check(lib().pq_concat_requant_s8(arr, k, N * H * W, int(q_bit), c_out_pad, out.data_ptr(), _stream(first)),
              "pq_concat_requant_s8")
    return out

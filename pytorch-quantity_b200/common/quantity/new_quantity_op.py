"""Simulation operators (subsystems 3 and 4) with the reference's constructor signatures and
attribute names (quantity/common/quantity/new_quantity_op.py:8-452), executed by the sm_100a
kernels of libpq_sm100.so.

Integer simulation (``ReconModel``): ``NewConv2d`` / ``NewLinear`` run
  Quantity -> Conv/Linear -> RightShift -> BiasAdd -> Sp -> DeQuantity          (:124-133, :197-205)
as: one quantise kernel (fp32 NCHW -> int8 NHWC) + one tcgen05 int8 GEMM / implicit-GEMM
kernel whose epilogue does shift / round-half-away / saturate / bias / saturate / dequantise
and writes the fp32 NCHW tensor the module API promises.  The stand-alone modules
(``Quantity``, ``RightShift``, ``Sp``, ``BiasAdd``, ``DeQuantity``) keep working on their own
through small bandwidth kernels.

Fake-quant simulation (``ReconTest``): ``TestConv`` / ``TestLinear`` fake-quantise weight and
bias once with ``QuanDequan`` and apply ``QuanDequan`` to the layer output (:259-292, :358-389);
the fp32 convolution itself stays the user's cuDNN library call, as in the reference.

Deliberate deviations (all documented in INTEGRATION.md):
  * ``quantized_bias`` is a registered buffer so ``model.cuda()`` moves it (reference quirk Q5);
  * ``TestConv`` / ``TestLinear`` write their text / PNG diagnostics only when the module-level
    switch ``WRITE_DIAGNOSTICS`` is on (they cost 25 s per ResNet-18 in the reference);
  * a missing bias is handled (reference quirk Q6 dereferences a non-existent attribute);
  * 8-bit only (the 16-bit branches of the reference are inconsistent, quirk Q11).
"""
import os

import numpy as np
import torch
import torch.nn as nn

from . import _native

QUANTIZE_BIT = 8                     # new_quantity_op.py:8
WRITE_DIAGNOSTICS = False

# Debug switch for the reference's own exactness limit.  The reference runs the integer convolution as an fp32
# nn.Conv2d on integer-valued tensors (new_quantity_op.py:124-126), which equals int8 x int8 -> int32 only while
# every partial sum stays below 2^24 (and only if the library's convolution is exact: cuDNN's fp32 Winograd is
# not, see tests/test_gpu_vs_reference.py).  The kernels here accumulate in int32 and are always exact, so beyond
# that limit they would legitimately DIFFER from the reference.  With CHECK_ACC_RANGE on, NewConv2d / NewLinear
# re-evaluate their accumulator exactly (float64, slow) on every forward, keep ``max_abs_acc`` on the module and
# warn when it reaches 2^24, so that such a mismatch is explained rather than mysterious.
CHECK_ACC_RANGE = False
S2D_STEM = True            # stride-2 convolutions with <= 4 input channels in space-to-depth form (A/B switch)
FP32_EXACT_LIMIT = 1 << 24


def accumulator_report(model):
    """name -> max |accumulator| seen by every NewConv2d / NewLinear of ``model`` (after forwards run with
    CHECK_ACC_RANGE on); names whose value reached 2^24 are where the reference's fp32 arithmetic stops being
    integer arithmetic."""
    return {name: m.max_abs_acc for name, m in model.named_modules() if getattr(m, "max_abs_acc", None) is not None}


def _range(bits):
    assert bits == 8 or bits == 16, "Not support bit width."
    return (-128.0, 127.0) if bits == 8 else (-32768.0, 32767.0)


class RightShift(nn.Module):
    """acc / 2^rs, round half away from zero, saturate (new_quantity_op.py:11-44)."""

    def __init__(self, bits, rs):
        super().__init__()
        self.rs = rs
        self.Bit_width = bits

    def forward(self, x):
        lo, hi = _range(self.Bit_width)
        return _native.rshift(x, self.rs, lo, hi).view(x.shape)


class Quantity(nn.Module):
    """clamp(round_half_even(x * 2^ib)) -> integer-valued fp32 (new_quantity_op.py:48-58)."""

    def __init__(self, ib):
        super().__init__()
        self.ib = ib

    def forward(self, x):
        lo, hi = _range(QUANTIZE_BIT)
        return _native.fakequant(x, self.ib, lo, hi, dequant=False).view(x.shape)


class DeQuantity(nn.Module):
    """x / 2^ob (new_quantity_op.py:61-68)."""

    def __init__(self, ob):
        super().__init__()
        self.ob = ob

    def forward(self, x):
        return _native.clamp_scale(x, float("-inf"), float("inf"), 2.0 ** -self.ob).view(x.shape)


class Sp(nn.Module):
    """Saturating truncation (new_quantity_op.py:71-91)."""

    def __init__(self, bits):
        super().__init__()
        self.bitwidth = bits

    def forward(self, x):
        lo, hi = _range(self.bitwidth)
        return _native.clamp_scale(x, lo, hi, 1.0).view(x.shape)


class BiasAdd(nn.Module):
    """Plain broadcast add (new_quantity_op.py:95-101); fused into the GEMM epilogue inside
    NewConv2d / NewLinear."""

    def forward(self, x, y):
        return torch.add(x, y)


def _quantize_param(p, bit):
    """clamp(round(p * 2^bit), -128, 127) as int8 (new_quantity_op.py:147-152)."""
    return _native.fakequant(p.detach().float().contiguous(), bit, -128.0, 127.0, dequant=False)


def _pad16(c):
    return (c + 15) // 16 * 16


def _pad32(c):
    return (c + 31) // 32 * 32


class _IntSimBase(nn.Module):
    max_abs_acc = None

    def _check_acc(self, input, layer):
        """Debug path (CHECK_ACC_RANGE): exact float64 re-evaluation of this layer's accumulator."""
        import warnings
        import torch.nn.functional as F
        x = input.dequantize() if hasattr(input, "dequantize") else input
        with torch.no_grad():
            q = torch.clamp(torch.round(x.float() * 2.0 ** self.input_bit), -128.0, 127.0).double()
            w = layer.weight.detach().double()                     # integer-valued after quantity()
            if isinstance(layer, nn.Conv2d):
                acc = F.conv2d(q, w, None, layer.stride, layer.padding, layer.dilation, layer.groups)
            else:
                acc = F.linear(q, w)
            m = float(acc.abs().max()) if acc.numel() else 0.0
        self.max_abs_acc = max(self.max_abs_acc or 0.0, m)
        if m >= FP32_EXACT_LIMIT:
            warnings.warn("%s: |accumulator| reaches %.4g >= 2^24: the reference's fp32 convolution is no longer "
                          "exact integer arithmetic here, so its output may differ from this (exact int32) result"
                          % (type(self).__name__, m))

    def _read_info(self, quantize_infor):
        self.weight_bit = quantize_infor["weight_bit"]
        self.bias_bit = quantize_infor["bias_bit"]
        self.input_bit = quantize_infor["input_bit"]
        self.output_bit = quantize_infor["output_bit"]
        self.rs_bit = self.weight_bit + self.input_bit - self.output_bit
        self.Quan = Quantity(self.input_bit)
        self.RightShift = RightShift(QUANTIZE_BIT, self.rs_bit)
        self.BiasAdd = BiasAdd()
        self.Sp = Sp(QUANTIZE_BIT)
        self.DeQuan = DeQuantity(self.output_bit)

    def _quantize_params(self, layer, out_features):
        """Shared body of NewConv2d.quantity / NewLinear.quantity (:135-163, :208-236)."""
        self.weight = layer.weight
        self.bias = layer.bias
        assert self.weight is not None, "The weight can`t be None"
        w = self.weight.data
        if not w.is_cuda:
            if not torch.cuda.is_available():
                raise RuntimeError("no CUDA device: the integer simulation has no CPU fallback")
            layer.cuda()
            w = layer.weight.data
        b = layer.bias.data if layer.bias is not None else torch.zeros(out_features, device=w.device)
        wq = _quantize_param(w, self.weight_bit).view(w.shape)
        bq = _quantize_param(b, self.bias_bit).view(b.shape)
        # the wrapped layer keeps the integer-valued weights and a zero bias, like the reference
        layer.weight = nn.Parameter(wq)
        layer.bias = nn.Parameter(torch.zeros(out_features, device=w.device))
        self.register_buffer("quantized_bias", bq)                      # fp32, integer-valued
        # [N] bias, followed (when N % 16 == 0 and 1 <= rs <= 20) by the folded constants of the int8 epilogue
        self.register_buffer("_bias_i32", _native.bias_fold(bq.to(torch.int32), self.rs_bit))
        return wq


class NewConv2d(_IntSimBase):
    """Integer-simulated convolution (new_quantity_op.py:104-163).

    quantity() picks the kernel for the layer's shape and builds the weights that kernel reads:
      _payload_channels set   int8 NHWC image with that many (padded) channels -> pq_conv2d_s8 (implicit GEMM)
      _smallc                 <= 8 channels: zero-padded image of 8-byte pixels -> pq_conv2d_smallc_s8 (one TMA
                              per filter row); with _s2d the same kernel on the space-to-depth image (stride 2,
                              <= 4 channels)
      _explicit_im2col        other convolutions with <= 8 channels: explicit im2col matrix -> pq_gemm_s8
      _depthwise              groups == in_channels == out_channels inside the kernel's limits: int8 NHWC image with
                              _payload_channels (padded) channels -> pq_conv2d_dw_s8
      _group_block            other groups > 1 where _grouped_fits (>= 2 input channels per group): int8 NHWC image
                              of in_channels (unpadded) channels -> pq_conv2d_s8 with groups, one launch, output-channel
                              tiles of _group_block channels over grouped_filter weights
      _group_convs            the remaining groups > 1 (channel multiplier > 1 with one input channel per group,
                              shapes outside _grouped_fits): one NewConv2d per group
    Only this class reads these flags: forward() and the int8 pipeline run the layer through _quantize / _run /
    _run_add."""

    # class-level defaults: a model pickled before the depthwise / grouped kernels existed has _group_convs set and
    # neither attribute
    _depthwise = False
    _group_block = 0

    def __init__(self, conv_module, quantize_infor):
        super().__init__()
        self._read_info(quantize_infor)
        self.Conv = conv_module
        self.int8_pipeline = False      # see int8_pipeline.enable_int8_pipeline
        self.quantity()

    def quantity(self):
        conv = self.Conv
        if conv.padding_mode != "zeros" or isinstance(conv.padding, str):
            raise NotImplementedError(
                "NewConv2d(%r): padding_mode=%r / padding=%r is not supported by the sm_100a convolution kernels "
                "(PQ_EUNSUPPORTED: zero padding given as integers only; there is no CPU fallback)"
                % (conv, conv.padding_mode, conv.padding))
        wq = self._quantize_params(conv, conv.out_channels)
        K, C, R, S = wq.shape
        self._dilation = tuple(int(d) for d in conv.dilation) if (R, S) != (1, 1) else (1, 1)
        # channel count of the int8 NHWC operand, None when the layer's kernel reads another layout
        self._payload_channels = None
        # whether _run_add can fuse a following NewAdd into this convolution's epilogue
        self._fuses_add = False
        self._group_convs = None
        self._smallc = self._s2d = self._explicit_im2col = self._depthwise = False
        self._group_block = 0
        if conv.groups != 1:
            if _depthwise_fits(conv):
                # one stencil kernel over the int8 NHWC image; weights [R][S][C_pad], channel-fastest
                self._depthwise = True
                self._dilation = tuple(int(d) for d in conv.dilation)
                self._payload_channels = _pad16(K)
                w_rsc = torch.zeros((R, S, self._payload_channels), dtype=torch.int8, device=wq.device)
                w_rsc[..., :K] = wq[:, 0].permute(1, 2, 0).to(torch.int8)
                self.register_buffer("_w_rsc", w_rsc.contiguous())
                return
            if _grouped_fits(conv):
                # one launch of the GEMM kernel over the whole layer; the weight layout depends on the tile width
                self._group_block = _group_block(conv)
                self._payload_channels = conv.in_channels
                self.register_buffer("_w_krsc", grouped_filter(wq, conv.groups, self._group_block))
                return
            self._build_groups(conv, wq)
            return
        # im2col TMA fetches channel blocks of 32 / 64 / 128 bytes; a 1x1 stride-1 conv is a plain GEMM
        plain = (R, S) == (1, 1) and tuple(conv.stride) == (1, 1) and tuple(conv.padding) == (0, 0)
        if plain or C > 8 or self._dilation != (1, 1):
            # (a dilated filter always takes the im2col-TMA kernel: its taps are TMA offsets)
            self._payload_channels = _pad16(C) if plain else _pad32(C)
            self._fuses_add = self._dilation == (1, 1) and K % 16 == 0
            w_krsc = torch.zeros((K, R, S, self._payload_channels), dtype=torch.int8, device=wq.device)
            w_krsc[..., :C] = wq.permute(0, 2, 3, 1).to(torch.int8)
            self.register_buffer("_w_krsc", w_krsc.contiguous())
        elif S <= 8 and conv.stride[1] % 2 == 0:
            # very few input channels (the ResNet stem): instead of padding C to 32, the windowed small-channel
            # kernel over 8-byte pixels
            self._smallc = True
            w = torch.zeros((K, R, 8, 8), dtype=torch.int8, device=wq.device)       # [K][R][tap slot][channel slot]
            w[:, :, :S, :C] = wq.permute(0, 2, 3, 1).to(torch.int8)
            self.register_buffer("_w_krs8", w.view(K, R, 64).contiguous())
            # Stride 2 with <= 4 channels (the ResNet stem): space-to-depth form.  2 x 2 blocks of the padded image
            # become 16-byte pixels (pq_quantize_nchw_to_s2d16_s8), the R x S / stride-2 filter a ceil((R + 1) / 2)-row
            # stride-1 filter over them: tap (r, s) sits in block (a, b), phase (dy, dx) with
            # (a, dy) = divmod(r + e_h, 2), e_h = padding parity (the padded image starts on an even row).  Same
            # 64-byte row window, rows 16 bytes apart -> the same kernel, 8 instead of 14 MMAs per tile for 7 x 7.
            self._s2d = S2D_STEM and tuple(conv.stride) == (2, 2) and C <= 4 and R <= 7 and S <= 7
            if self._s2d:
                self.register_buffer("_w_s2d", s2d_filter(wq, conv.padding), persistent=False)
        else:
            # the small-channel kernel does not apply (odd stride, wide filter): explicit im2col + GEMM
            self._explicit_im2col = True
            self._k_pad = (R * S * C + 63) // 64 * 64
            w_nk = torch.zeros((K, self._k_pad), dtype=torch.int8, device=wq.device)
            w_nk[:, :R * S * C] = wq.permute(0, 2, 3, 1).reshape(K, -1).to(torch.int8)
            self.register_buffer("_w_nk", w_nk.contiguous())

    def _build_groups(self, conv, wq):
        """groups > 1 (the reference wraps any nn.Conv2d, new_quantity_op.py:104-133): one integer convolution per
        group over its channel slice, built from the already quantised parameters, results concatenated along the
        channel axis -- exactly the definition of a grouped convolution, every group on the tensor-core kernels."""
        G = conv.groups
        Kg, Cg = conv.out_channels // G, conv.in_channels // G
        subs = []
        for g in range(G):
            sub = nn.Conv2d(Cg, Kg, conv.kernel_size, conv.stride, conv.padding, conv.dilation, 1, True).to(wq.device)
            with torch.no_grad():
                # integer-valued parameters scaled back by exact powers of two: re-quantising them is the identity
                sub.weight.copy_(wq[g * Kg:(g + 1) * Kg] * 2.0 ** -self.weight_bit)
                sub.bias.copy_(self.quantized_bias[g * Kg:(g + 1) * Kg] * 2.0 ** -self.bias_bit)
            subs.append(NewConv2d(sub, {"weight_bit": self.weight_bit, "bias_bit": self.bias_bit,
                                        "input_bit": self.input_bit, "output_bit": self.output_bit}))
        self._group_convs = nn.ModuleList(subs)

    def _grouped_forward(self, input):
        x = input.dequantize() if hasattr(input, "dequantize") else input
        Cg = self.Conv.in_channels // self.Conv.groups
        outs = [sub(x[:, g * Cg:(g + 1) * Cg].contiguous()) for g, sub in enumerate(self._group_convs)]
        return torch.cat(outs, 1)

    def forward(self, input):
        if CHECK_ACC_RANGE:
            self._check_acc(input, self.Conv)
        if self._group_convs is not None:
            return self._grouped_forward(input)
        if self.int8_pipeline:
            from .int8_pipeline import conv_forward
            return conv_forward(self, input)
        return self._run(self._quantize(input), True, False, False)[0]   # Quan, Conv+RightShift+BiasAdd+Sp+DeQuan

    # ---- the layer's launch path (not for layers on the per-group path).  An operand is what _quantize returns: the
    # int8 NHWC image [N][H][W][_payload_channels] when _payload_channels is set (a producer's int8 payload at input_bit
    # is one, too), otherwise (int8 tensor in the kernel's layout, (N, H, W) of the input).

    def _quantize(self, x):
        """Quantity(input_bit) of fp32 NCHW x into the operand this layer's kernel reads."""
        conv = self.Conv
        if self._payload_channels is not None:
            return _native.quantize_nchw_to_nhwc_s8(x, self.input_bit, self._payload_channels)
        N, _, H, W = x.shape
        if self._explicit_im2col:
            a, _ = _native.quantize_im2col_s8(x, self.input_bit, conv.kernel_size, conv.stride, conv.padding,
                                              self._k_pad)
            return a, (N, H, W)
        (R, S), (sh, sw), (ph, pw) = conv.kernel_size, conv.stride, conv.padding
        P, Q = _native.conv_out_size((H, W), conv.kernel_size, conv.stride, conv.padding)
        if self._s2d:
            hp2, wp2 = P + self._w_s2d.shape[1] - 1, Q + 3      # blocks the 64-byte row windows of every output touch
            xs = _native.quantize_s2d16_s8(x, self.input_bit, (ph + (ph & 1), pw + (pw & 1)), hp2, wp2)
            # the same bytes as an 8-byte-pixel image of twice the width
            return xs.view(N, hp2, 2 * wp2, 8), (N, H, W)
        Hp = max((P - 1) * sh + R, H + ph)
        Hp = (Hp + sh - 1) // sh * sh
        Wp = max((Q - 1) * sw + 8, W + pw)
        Wp += Wp & 1
        return _native.quantize_pad_nhwc8_s8(x, self.input_bit, (ph, pw), Hp, Wp), (N, H, W)

    def _out_shape(self, operand):
        """(N, K, P, Q) of the layer's output for this operand."""
        conv = self.Conv
        N, H, W = operand.shape[:3] if self._payload_channels is not None else operand[1]
        P, Q = _native.conv_out_size((H, W), conv.kernel_size, conv.stride, conv.padding, self._dilation)
        return N, conv.out_channels, P, Q

    def _run(self, operand, want_f32, want_s8, relu):
        """Conv + RightShift + BiasAdd + Sp (+ the nn.ReLU after the layer when relu) on an operand.  Returns
        (fp32 NCHW after DeQuantity or None, int8 NHWC [N][P][Q][K] or None)."""
        conv = self.Conv
        if self._depthwise:
            return _native.conv2d_dw_s8(operand, self._w_rsc, self._bias_i32, conv.stride, conv.padding, self.rs_bit,
                                        self.output_bit, want_f32=want_f32, want_s8=want_s8, relu=relu,
                                        dilation=self._dilation, channels=conv.out_channels)
        if self._payload_channels is not None:
            grouped = self._group_block != 0
            return _native.conv2d_s8(operand, self._w_krsc, self._bias_i32, conv.stride, conv.padding, self.rs_bit,
                                     self.output_bit, want_f32=want_f32, want_s8=want_s8, c_real=conv.in_channels,
                                     relu=relu, dilation=self._dilation, groups=conv.groups if grouped else 1,
                                     group_block=self._group_block)
        t = operand[0]
        N, K, P, Q = self._out_shape(operand)
        if self._explicit_im2col:
            f32, s8 = _native.gemm_s8(t, self._w_nk, self._bias_i32, self.rs_bit, self.output_bit, hw=P * Q,
                                      want_f32=want_f32, want_s8=want_s8, relu=relu,
                                      k_real=conv.in_channels * conv.kernel_size[0] * conv.kernel_size[1])
            return (f32.view(N, K, P, Q) if want_f32 else None), (s8.view(N, P, Q, K) if want_s8 else None)
        if self._s2d:
            # filter of ra rows x 8 slots, stride (1, 2) over the 8-byte-pixel view
            (R, S), ra = conv.kernel_size, self._w_s2d.shape[1]
            return _native.conv2d_smallc_s8(t, self._w_s2d, self._bias_i32, t.shape[1:3], (ra, 8), (1, 2), (0, 0),
                                            self.rs_bit, self.output_bit, want_f32=want_f32, want_s8=want_s8,
                                            relu=relu, ops=2 * N * P * Q * K * R * S * conv.in_channels)
        return _native.conv2d_smallc_s8(t, self._w_krs8, self._bias_i32, operand[1][1:], conv.kernel_size,
                                        conv.stride, conv.padding, self.rs_bit, self.output_bit, want_f32=want_f32,
                                        want_s8=want_s8, c_real=conv.in_channels, relu=relu)

    def _smallc_forward(self, input, want_f32, want_s8, relu):
        """Quan + the small-channel convolution from fp32 NCHW input, in the form _s2d selects (the space-to-depth
        image or the 8-byte-pixel image; both give the same integers).  Returns what _run returns."""
        return self._run(self._quantize(input), want_f32, want_s8, relu)

    def _run_add(self, operand, shortcut, shortcut_bit, shortcut_relu, q_bit, relu, want16):
        """This layer and the NewAdd of its int8 output with `shortcut` (int8 / int16 NHWC at shortcut_bit), plus the
        nn.ReLU after the add when relu, in one kernel (only where _fuses_add).  Returns (int16 exact sum or None,
        int8 Quantity(q_bit) of it), both NHWC."""
        conv = self.Conv
        return _native.conv2d_s8_add(operand, self._w_krsc, self._bias_i32, conv.stride, conv.padding, self.rs_bit,
                                     self.output_bit, shortcut, shortcut_bit, shortcut_relu, q_bit, relu,
                                     want16=want16, c_real=conv.in_channels)


def _depthwise_fits(conv):
    """A depthwise convolution (channel multiplier 1) of a shape pq_conv2d_dw_s8 implements: R, S <= 7, stride and
    dilation 1 or 2, 0 <= pad <= (R - 1) * dilation (zero padding is checked by quantity())."""
    (R, S), (sh, sw), (ph, pw), (dh, dw) = conv.kernel_size, conv.stride, conv.padding, conv.dilation
    return (conv.groups == conv.in_channels == conv.out_channels and R <= 7 and S <= 7 and sh in (1, 2)
            and sw in (1, 2) and dh in (1, 2) and dw in (1, 2) and 0 <= ph <= (R - 1) * dh and 0 <= pw <= (S - 1) * dw)


def _plain(conv):
    """A 1x1 stride-1 unpadded convolution: the kernel runs it as a plain GEMM over the NHWC image."""
    return tuple(conv.kernel_size) == (1, 1) and tuple(conv.stride) == (1, 1) and tuple(conv.padding) == (0, 0)


def _group_block(conv):
    """The output-channel tile width of the grouped kernel for this layer, or None when no width is legal
    (include/pq_sm100.h): the one that wastes the fewest tensor-core operations (max(1, width / Kg) times the useful
    work), the widest among those (fewer re-reads of the input window)."""
    G, C, K = conv.groups, conv.in_channels, conv.out_channels
    Cg, Kg = C // G, K // G
    box = 16 if _plain(conv) else 32
    best = None
    for b in (256, 128, 64, 32):
        wb = _native.group_window(C, K, G, b)
        if (b % Kg and Kg % b) or K % b or wb % box:
            continue
        if best is None or max(1, b // Kg) < max(1, best // Kg):
            best = b
    return best


def _grouped_fits(conv):
    """A grouped convolution the GEMM kernel runs in one launch: >= 2 input channels per group (one channel per group
    is depthwise or a channel multiplier), unpadded channels in whole TMA boxes (C % 32 == 0; 16 for a 1x1 stride-1
    GEMM) and a legal tile width."""
    G, C, K = conv.groups, conv.in_channels, conv.out_channels
    return (G > 1 and C % G == 0 and K % G == 0 and C // G >= 2 and C % (16 if _plain(conv) else 32) == 0
            and _group_block(conv) is not None)


def grouped_filter(wq, groups, group_block):
    """Integer filter [K][Cg][R][S] of a grouped convolution -> int8 [K][R][S][Wb], the layout pq_conv2d_s8 reads for
    output-channel tiles of group_block channels: the tile starting at channel n0 reads the input-channel window that
    starts at (n0 // Kg) * Cg, Wb = Cg * max(1, group_block // Kg) channels wide, and row k holds its group's Cg
    channels at that group's offset inside the window, zeros elsewhere."""
    K, Cg, R, S = wq.shape
    Kg = K // groups
    wb = Cg * max(1, group_block // Kg)
    k = torch.arange(K, device=wq.device)
    off = (k // Kg) * Cg - (k // group_block * group_block // Kg) * Cg          # group origin - window origin
    idx = (off[:, None] + torch.arange(Cg, device=wq.device))[:, None, None, :].expand(K, R, S, Cg)
    w = torch.zeros((K, R, S, wb), dtype=torch.int8, device=wq.device)
    w.scatter_(3, idx, wq.permute(0, 2, 3, 1).to(torch.int8))
    return w.contiguous()


def s2d_filter(wq, padding):
    """Integer filter [K][C <= 4][R <= 7][S <= 7] of a stride-2 convolution -> int8 [K][ra][64]: the equivalent stride-1
    filter over the space-to-depth image of pq_quantize_nchw_to_s2d16_s8 (16-byte pixels = 2 x 2 blocks, byte
    (dy * 2 + dx) * 4 + c), ra = ceil((R + e_h) / 2) rows of four blocks each.  The padded image starts on an even row /
    column (pad rounded up to even, e = pad & 1), so tap (r, s) lies in block (a, b), phase (dy, dx) with
    (a, dy) = divmod(r + e_h, 2), (b, dx) = divmod(s + e_w, 2)."""
    K, C, R, S = wq.shape
    eh, ew = int(padding[0]) & 1, int(padding[1]) & 1
    ra = ((eh + R - 1) >> 1) + 1
    w2 = torch.zeros((K, ra, 4, 2, 2, 4), dtype=torch.int8, device=wq.device)       # [K][a][b][dy][dx][c]
    for r in range(R):
        a, dy = divmod(eh + r, 2)
        for t in range(S):
            b, dx = divmod(ew + t, 2)
            w2[:, a, b, dy, dx, :C] = wq[:, :, r, t].to(torch.int8)
    return w2.view(K, ra, 64).contiguous()


class NewLinear(_IntSimBase):
    """Integer-simulated fully connected layer (new_quantity_op.py:177-236)."""

    def __init__(self, linear_module, quantize_infor):
        super().__init__()
        self._read_info(quantize_infor)
        self.Linear = linear_module
        self.quantity()

    def quantity(self):
        lin = self.Linear
        wq = self._quantize_params(lin, lin.out_features)
        N, K = wq.shape
        self._k_pad = _pad16(K)
        w = torch.zeros((N, self._k_pad), dtype=torch.int8, device=wq.device)
        w[:, :K] = wq.to(torch.int8)
        self.register_buffer("_w_nk", w.contiguous())

    def forward(self, input):
        if CHECK_ACC_RANGE:
            self._check_acc(input, self.Linear)
        x2 = input.reshape(-1, input.shape[-1])
        # Quan: a [B][K] matrix is NCHW with H = W = 1, so the same kernel quantises and pads it
        q = _native.quantize_nchw_to_nhwc_s8(x2.view(x2.shape[0], x2.shape[1], 1, 1), self.input_bit,
                                             self._k_pad).view(x2.shape[0], self._k_pad)
        out, _ = _native.gemm_s8(q, self._w_nk, self._bias_i32, self.rs_bit, self.output_bit,
                                 k_real=self.Linear.in_features)
        return out.view(*input.shape[:-1], out.shape[-1])


class NewAdd(nn.Module):
    """clamp(x + y, -128, 127) on the de-quantised values (new_quantity_op.py:166-174)."""

    def __init__(self):
        super().__init__()
        self.Sp = Sp(QUANTIZE_BIT)

    def forward(self, x, y):
        if getattr(self, "int8_pipeline", False):
            from .int8_pipeline import add_forward
            out = add_forward(self, x, y)
            if out is not None:
                return out
        lo, hi = _range(QUANTIZE_BIT)
        return _native.add_clamp(x, y, lo, hi).view(torch.broadcast_shapes(x.shape, y.shape))


class QuanDequan(nn.Module):
    """Power-of-two fake quantisation: clamp(round(x * 2^bit)) / 2^bit in one fused kernel
    (new_quantity_op.py:239-257)."""

    def __init__(self, Bitwidth, bit):
        super().__init__()
        self.bitwidth = Bitwidth
        self.bit = bit

    def forward(self, quantized_x):
        lo, hi = (-128.0, 127.0) if self.bitwidth == 8 else (-32768.0, 32767.0)
        return _native.fakequant(quantized_x, self.bit, lo, hi, dequant=True).view(quantized_x.shape)


def _dump_diagnostics(path, name, tag, before, after):
    """Text dump of a parameter before / after fake-quant (new_quantity_op.py:312-326); the
    PNG histograms (:328-337) are drawn only if matplotlib is importable."""
    stem = os.path.join(path, name.replace(".", "_") + "_" + tag)
    with open(stem + ".txt", "a") as f:
        for t in (before, after):
            f.write("  ".join(str(v) for v in t.detach().cpu().numpy().flatten()) + "\n\n\n\n")
    try:
        import matplotlib.pyplot as plt
    except ImportError:
        return
    for suffix, t in (("_o.png", before), ("_q.png", after)):
        fig = plt.figure()
        plt.grid()
        plt.title(tag)
        plt.xlabel("bins")
        plt.ylabel("counter/frequency")
        plt.hist(t.detach().cpu().numpy().flatten(), 2048, density=True, histtype="bar", facecolor="blue")
        fig.savefig(stem + suffix, bbox_inches="tight")
        plt.close(fig)


class _FakeQuantBase(nn.Module):
    def _setup(self, name, module, quantize_infor, new_model_path, out_features):
        self.name = name
        self.path = os.path.join(os.path.dirname(new_model_path or "."), "quantity_results")
        if WRITE_DIAGNOSTICS and not os.path.exists(self.path):
            os.makedirs(self.path)
        self.weight_bit = quantize_infor["weight_bit"]
        self.bias_bit = quantize_infor["bias_bit"]
        self.input_bit = quantize_infor["input_bit"]
        self.output_bit = quantize_infor["output_bit"]
        self.weight_qdp = QuanDequan(QUANTIZE_BIT, self.weight_bit)
        self.bias_qdp = QuanDequan(QUANTIZE_BIT, self.bias_bit)
        self.output_qdp = QuanDequan(QUANTIZE_BIT, self.output_bit)
        self._out_features = out_features

    def _feature_extract(self, layer):
        """Fake-quantise weight and bias once and write them back (:294-309, :392-407)."""
        self.weight = layer.weight
        self.bias = layer.bias
        assert self.weight is not None, "The layer weight can`t be None"
        if not layer.weight.is_cuda:
            if not torch.cuda.is_available():
                raise RuntimeError("no CUDA device: the fake-quant simulation has no CPU fallback")
            layer.cuda()
        w = layer.weight.data
        b = layer.bias.data if layer.bias is not None else torch.zeros(self._out_features, device=w.device)
        w_qdp = self.weight_qdp(w)
        b_qdp = self.bias_qdp(b)
        layer.weight = nn.Parameter(w_qdp)
        layer.bias = nn.Parameter(b_qdp)
        if WRITE_DIAGNOSTICS:
            _dump_diagnostics(self.path, self.name, "weight", w, w_qdp)
            _dump_diagnostics(self.path, self.name, "bias", b, b_qdp)


class TestConv(_FakeQuantBase):
    """Fake-quant convolution (new_quantity_op.py:259-355)."""
    __test__ = False      # not a pytest class

    def __init__(self, name, module, quantize_infor, new_model_path):
        super().__init__()
        self._setup(name, module, quantize_infor, new_model_path, module.out_channels)
        self.Conv = module
        self.feature_extract()

    def feature_extract(self):
        self._feature_extract(self.Conv)

    def forward(self, x):
        return self.output_qdp(self.Conv(x))


class TestLinear(_FakeQuantBase):
    """Fake-quant fully connected layer (new_quantity_op.py:358-452)."""
    __test__ = False

    def __init__(self, name, module, quantize_infor, new_model_path):
        super().__init__()
        self._setup(name, module, quantize_infor, new_model_path, module.out_features)
        self.linear = module
        self.feature_extract()

    def feature_extract(self):
        self._feature_extract(self.linear)

    def forward(self, x):
        return self.output_qdp(self.linear(x))

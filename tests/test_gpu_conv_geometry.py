"""The operand side of the dense int8 convolution over its whole geometry range: how gemm_s8_kernel (plain GEMM,
im2col-TMA, patch windows, the fused add) and the small-channel kernels (conv_rows_s8_kernel and the window mode of
gemm_s8_kernel) find the A bytes of a tile, on every path pq_gemm_s8.cu can choose, against

    acc = float64 F.conv2d of the int8 operands (tuple stride, padding, dilation), rounded to int64   exact: |acc| < 2^53
    y   = clamp(clamp(RightShift(acc, rs)) + b) [ReLU], fp32 = y / 2^ob                   new_quantity_op.py:11-44,124-133

which a CPU test pins to oracle.int_conv_layer on rectangular, asymmetric and dilated layers.  The epilogue's own bit
range is test_gpu_epilogue_matrix.py's; each row here runs the staged int8 store and the generic fp32 + unstaged int8
body (or one fused add).

Each GEOMETRY row names the path it must take (checked against a mirror of the host's choice on the CPU and with
torch.profiler on the GPU).  Every output sits in the middle of a sentinel-filled buffer whose neighbouring bytes must
survive, the input and the weights must be unchanged after the call, and a refused call writes nothing.  LIMITS holds
one row inside and one beyond every geometry limit include/pq_sm100.h documents for pq_conv2d_s8 and
pq_conv2d_smallc_s8; the index limits run at their real size.
"""
import ctypes
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

gpu = pytest.mark.gpu
EINVAL, EUNSUPPORTED, EALIGN = -1, -2, -3
M_LIMIT = 2 ** 31 - 1
SMS = 148                              # the B200's SM count: pick_bn below assumes it (checked on the GPU)
SENTINEL = 0xA5
GUARD = 512                            # bytes on either side; a multiple of 16, so outputs keep their alignment


# ------------------------------------------------------------------------------------------ the exact reference
def right_shift(acc, rs):
    """new_quantity_op.py:11-44 on int64 accumulators: round half away from zero for rs >= 1, else clamp then scale."""
    if rs >= 1:
        half = 1 << (rs - 1)
        r = torch.where(acc >= 0, (acc + half) >> rs, -((half - acc) >> rs))
    else:
        r = acc.clamp(-128, 127) << (-rs)
    return r.clamp(-128, 127)


def epilogue_ref(acc, bias, rs, relu):
    """int64 [M][N] accumulators, int64 [N] bias -> the int8-valued layer output (RightShift, BiasAdd, Sp[, ReLU])."""
    y = (right_shift(acc, rs) + bias.view(1, -1)).clamp(-128, 127)
    return y.clamp(min=0) if relu else y


def dequant_ref(y, ob):
    return (y.double() * 2.0 ** -ob).float()          # exact: |y| <= 128


def round_half_even_shift(v, d):
    """round_half_even(v / 2^d) for int64 v and d >= 1."""
    t = v >> d
    rem = v - (t << d)
    half = 1 << (d - 1)
    return t + ((rem > half) | ((rem == half) & ((t & 1) == 1))).long()


def add_ref(y, ob, sc, sbit, sc_relu, out_relu, q_bit):
    """NewAdd (+ the nn.ReLU after it) of y at bit ob and the shortcut sc at bit sbit, exactly: (int16 sum at
    o_bit = max(ob, sbit), int8 Quantity(q_bit) of it)."""
    o = max(ob, sbit)
    s = sc.clamp(min=0) if sc_relu else sc
    total = ((y << (o - ob)) + (s << (o - sbit))).clamp(-128 << o, 127 << o)
    if out_relu:
        total = total.clamp(min=0)
    q8 = total << (q_bit - o) if q_bit >= o else round_half_even_shift(total, o - q_bit)
    return total, q8.clamp(-128, 127)


def exact_conv(x_nhwc, w_krsc, stride, pad, dil):
    """int64 [N*P*Q][K] accumulators of an NHWC int8 image and [K][R][S][C] int8 weights."""
    acc = F.conv2d(x_nhwc.permute(0, 3, 1, 2).double(), w_krsc.permute(0, 3, 1, 2).double(), None, stride, pad, dil)
    assert acc.numel() == 0 or float(acc.abs().max()) < 2.0 ** 53
    return torch.round(acc).long().permute(0, 2, 3, 1).reshape(-1, w_krsc.shape[0])


# ------------------------------------------------------------------------------------------ the host's path choice
# (BN, BK, STAGES, ADDK, BSLOTS) of the gemm_s8_kernel instantiations (pq_gemm_s8.cu: launch_bn, conv_impl)
PLAIN_STAGES = {32: (8, 9, 9), 64: (8, 9, 9), 128: (6, 9, 9), 256: (4, 8, 9)}      # BK 128, 64, 32
ADD_STAGES = {64: (6, 8, 8), 128: (4, 8, 8), 256: (3, 6, 8)}
DEEP_A = (64, 64, 18, 0, 9)
WIN128 = (128, 128, 3, 0, 9)
ROWS_KERNEL = "conv_rows_s8_kernel"


def inst(bn, bk, add=False):
    st = (ADD_STAGES if add else PLAIN_STAGES)[bn][(128, 64, 32).index(bk)]
    return (bn, bk, st, int(add), st)


def pick_bn(m, n, sms=SMS):
    """pq_gemm_s8.cu pick_bn: the widest tile that leaves every SM two tiles, never wider than N needs."""
    mt = -(-m // 128)
    cap = 256 if n > 128 else (128 if n > 64 else (64 if n > 32 else 32))
    bn = cap
    while bn > 32:
        if mt * -(-n // bn) >= 2 * sms:
            return bn
        bn //= 2
    return 64 if cap > 32 and mt * -(-n // 64) >= sms else 32


def out_size(g):
    (sh, sw), (ph, pw), (dh, dw) = g["st"], g["pad"], g["dil"]
    return ((g["H"] + 2 * ph - (g["R"] - 1) * dh - 1) // sh + 1, (g["W"] + 2 * pw - (g["S"] - 1) * dw - 1) // sw + 1)


def conv_path(g, add=False, no_windows=False, sms=SMS):
    """(path, instantiation) that conv_impl / launch_bn select for a pq_conv2d_s8(_add) geometry."""
    B, C, K, R, S = g["B"], g["C"], g["K"], g["R"], g["S"]
    P, Q = out_size(g)
    M = B * P * Q
    pre = "add/" if add else ""
    if (R, S) == (1, 1) and g["st"] == (1, 1) and g["pad"] == (0, 0):
        bk = 128 if C >= 128 else (64 if C >= 64 else 32)
        bn = pick_bn(M, K, sms)
        return pre + "gemm", inst(max(bn, 64) if add else bn, bk, add)
    if (not add and not no_windows and (R, S) == (3, 3) and g["st"] == (1, 1) and g["pad"] == (1, 1) and
            g["dil"] == (1, 1) and ((C == 64 and K <= 64) or (C == 128 and 64 < K <= 128)) and g["W"] + 2 <= 64):
        tw = 16 if g["W"] + 2 <= 16 else (32 if g["W"] + 2 <= 32 else 64)
        th = 128 // tw
        slot = -(-((th + 2) * tw * C) // 1024) * 1024
        slots = min((18 * 128 * 64 if C == 64 else 3 * 128 * 128) // slot, 18 if C == 64 else 3)
        if slots >= 2 and B * -(-P // th) * 128 <= M_LIMIT:
            return "win/tw%d" % tw, DEEP_A if C == 64 else WIN128
    bk = 128 if C % 128 == 0 else (64 if C % 64 == 0 else 32)
    num_kb = R * S * (C // bk)
    tps = 3 if bk <= 64 and num_kb % 3 == 0 else 1
    bn = pick_bn(M, K, sms)
    if not add and bk == 64 and bn == 64 and K <= 64 and num_kb <= 9 and tps == 3:
        return "im2col/deep", DEEP_A
    return pre + "im2col/bk%d/tps%d" % (bk, tps), inst(max(bn, 64) if add else bn, bk, add)


def smallc_pads(g):
    """(Hp, Wp): the smallest padded image pq_conv2d_smallc_s8 accepts (as NewConv2d._quantize builds it), unless the
    row sets its own."""
    P, Q = out_size(g)
    (sh, sw), (ph, pw) = g["st"], g["pad"]
    hp = max((P - 1) * sh + g["R"], g["H"] + ph)
    hp = -(-hp // sh) * sh
    wp = max((Q - 1) * sw + 8, g["W"] + pw)
    return g.get("Hp", hp), g.get("Wp", wp + (wp & 1))


def rows_fit(R, K, Q, Wp):
    """pq_conv2d_smallc_s8's row-kernel conditions besides stride_w == 2, R <= 8 and the tiles_m limit:
    (stages_fit >= 2, the over-read of the last window rows stays inside one ring slot)."""
    pitch, tiles_q = Wp * 8, -(-Q // 128)
    a_stage = -(-(R * pitch + 2112) // 1024) * 1024
    fixed = 1024 + -(-K // 64) * R * 4096 + 16 * 2048 + 256
    return (227 * 1024 - fixed) // a_stage >= 2, (R - 1) * pitch + (tiles_q * 128 - 1) * 16 + 64 <= a_stage


def smallc_path(g, sms=SMS):
    """(path, kernel) pq_conv2d_smallc_s8 selects: the row kernel, or gemm_s8_kernel's window mode (a_im2col == 2)."""
    P, Q = out_size(g)
    Hp, Wp = smallc_pads(g)
    if g["st"][1] == 2 and g["R"] <= 8:
        fit, no_overread = rows_fit(g["R"], g["K"], Q, Wp)
        if fit and no_overread and g["B"] * P * -(-Q // 128) * 128 <= M_LIMIT:
            return "rows", ROWS_KERNEL
    tw = 16 if Q >= 16 else (8 if Q >= 8 else 4)
    patches = g["B"] * -(-P // (128 // tw)) * -(-Q // tw)
    return "smallc-win/tw%d" % tw, inst(pick_bn(patches * 128, g["K"], sms), 64)


def expected_path(path, g):
    if path.startswith(("rows", "smallc")):
        return smallc_path(g)
    return conv_path(g, add=path.startswith("add/"))


# ------------------------------------------------------------------------------------------ geometry rows
def G(B, H, W, C, K, R, S, st=(1, 1), pad=(0, 0), dil=(1, 1), **kw):
    return dict(B=B, H=H, W=W, C=C, K=K, R=R, S=S, st=st, pad=pad, dil=dil, **kw)


# (path, geometry).  Strides 1 to 8, strides larger than the filter, pads beyond (R - 1) * dil (output pixels lying
# wholly in padding), H / W / P / Q = 1, batch 1, M % 128 != 0 with tiles crossing rows and images at many offsets.
GEOMETRY = [
    # plain GEMM (1x1, stride 1, no padding)
    ("gemm", G(1, 1, 1, 32, 48, 1, 1)),                                        # M = 1
    ("gemm", G(3, 7, 5, 48, 40, 1, 1)),                                        # K blocks 32 + 16 (BK 32)
    ("gemm", G(2, 5, 13, 2048, 24, 1, 1)),
    ("gemm", G(5, 13, 11, 96, 64, 1, 1, dil=(3, 2))),                          # a 1x1 filter ignores the dilation
    # im2col-TMA, BK 32
    ("im2col/bk32/tps1", G(3, 19, 9, 32, 16, 2, 1, st=(3, 1), pad=(0, 1), dil=(2, 1))),
    ("im2col/bk32/tps3", G(4, 6, 15, 96, 40, 2, 3, st=(1, 2), pad=(2, 1))),     # cblocks 3 on a 2x3 filter
    ("im2col/bk32/tps3", G(2, 21, 7, 32, 32, 1, 3, st=(5, 1), pad=(0, 4))),     # 1x3, pad_w > S - 1
    ("im2col/bk32/tps3", G(7, 30, 40, 32, 80, 5, 3, st=(8, 7), pad=(3, 0), dil=(1, 2))),
    ("im2col/bk32/tps3", G(128, 7, 9, 32, 16, 3, 3, pad=(2, 1), dil=(2, 1))),   # 63 pixels an image: every offset
    ("im2col/bk32/tps3", G(1, 1, 4095, 32, 32, 3, 3, st=(1, 2), pad=(1, 1))),   # 131040 input bytes (< 131072)
    ("im2col/bk32/tps3", G(1, 1, 4096, 32, 32, 3, 3, st=(1, 2), pad=(1, 1))),   # 131072
    ("im2col/bk32/tps3", G(2, 1, 2049, 32, 32, 3, 3, st=(1, 2), pad=(1, 1))),   # 131136
    # im2col-TMA, BK 64
    ("im2col/bk64/tps1", G(3, 17, 12, 64, 96, 2, 2, st=(2, 1), pad=(1, 0), dil=(2, 2))),
    ("im2col/bk64/tps1", G(11, 30, 1, 64, 64, 4, 1, st=(2, 1), pad=(1, 0), dil=(2, 1))),   # W = Q = 1
    ("im2col/bk64/tps3", G(3, 9, 20, 192, 48, 1, 2, st=(1, 3), pad=(0, 1))),    # cblocks 3 on a 1x2 filter
    ("im2col/bk64/tps3", G(9, 26, 1, 64, 128, 3, 1, st=(4, 2), pad=(3, 1), dil=(3, 1))),   # W = 1, Q = 2
    ("im2col/deep", G(16, 40, 61, 64, 48, 3, 1, st=(1, 2), pad=(1, 0))),         # deep A, 3x1: num_kb 3
    ("im2col/deep", G(30, 33, 40, 64, 64, 1, 3, st=(2, 1), pad=(0, 2), dil=(1, 3))),
    ("im2col/deep", G(19, 20, 50, 64, 64, 2, 3, pad=(1, 0))),                   # 2x3: num_kb 6
    ("im2col/deep", G(25, 75, 60, 64, 40, 3, 3, st=(2, 3), pad=(2, 1), dil=(2, 1))),
    # im2col-TMA, BK 128
    ("im2col/bk128/tps1", G(2, 9, 17, 128, 64, 1, 3, st=(6, 2), pad=(0, 1))),
    ("im2col/bk128/tps1", G(3, 5, 6, 2048, 16, 2, 3, st=(3, 1), pad=(0, 2), dil=(1, 2))),   # 96 K blocks
    ("im2col/bk128/tps1", G(40, 1, 23, 256, 32, 3, 2, st=(2, 5), pad=(1, 1))),   # H = P = 1
    # patch windows (3x3, stride 1, pad 1): both sides of every window width, and of the K / slot conditions
    ("win/tw16", G(3, 9, 13, 64, 64, 3, 3, pad=(1, 1))),
    ("win/tw16", G(2, 9, 14, 64, 48, 3, 3, pad=(1, 1))),
    ("win/tw32", G(1100, 9, 15, 64, 64, 3, 3, pad=(1, 1))),                    # W + 1 = 16 < W + 2
    ("win/tw32", G(2, 6, 29, 64, 64, 3, 3, pad=(1, 1))),
    ("win/tw32", G(3, 6, 30, 64, 32, 3, 3, pad=(1, 1))),
    ("win/tw64", G(2, 5, 31, 64, 64, 3, 3, pad=(1, 1))),
    ("win/tw64", G(2, 5, 61, 64, 64, 3, 3, pad=(1, 1))),
    ("win/tw64", G(1, 5, 62, 64, 16, 3, 3, pad=(1, 1))),
    ("im2col/bk64/tps3", G(2, 3, 63, 64, 64, 3, 3, pad=(1, 1))),             # W + 2 = 65 > 64
    ("im2col/bk32/tps3", G(2, 9, 65, 96, 64, 3, 3, pad=(1, 1))),               # C = 96, W + 2 > 64
    ("im2col/bk64/tps3", G(2, 9, 14, 64, 65, 3, 3, pad=(1, 1))),               # C = 64, K = 65
    ("im2col/bk64/tps3", G(2, 5, 62, 64, 64, 3, 3, pad=(1, 1), dil=(1, 2))),   # dilated: no windows
    ("win/tw16", G(3, 9, 13, 128, 65, 3, 3, pad=(1, 1))),
    ("win/tw32", G(2, 9, 15, 128, 128, 3, 3, pad=(1, 1))),
    ("win/tw32", G(2, 6, 30, 128, 128, 3, 3, pad=(1, 1))),
    ("im2col/bk128/tps1", G(2, 9, 14, 128, 64, 3, 3, pad=(1, 1))),             # C = 128, K = 64
    ("im2col/bk128/tps1", G(2, 9, 14, 128, 129, 3, 3, pad=(1, 1))),            # C = 128, K = 129
    ("im2col/bk128/tps1", G(2, 5, 31, 128, 96, 3, 3, pad=(1, 1))),             # one 64-wide slot only: im2col
    ("im2col/bk128/tps1", G(1, 5, 62, 128, 128, 3, 3, pad=(1, 1))),
    # pq_conv2d_s8_add in its GEMM and im2col forms
    ("add/gemm", G(3, 7, 9, 64, 48, 1, 1)),
    ("add/gemm", G(1, 1, 130, 2048, 64, 1, 1)),
    ("add/im2col/bk32/tps3", G(4, 6, 15, 96, 64, 2, 3, st=(1, 2), pad=(2, 1))),
    ("add/im2col/bk128/tps1", G(5, 21, 10, 128, 80, 3, 1, st=(2, 3), pad=(0, 2), dil=(2, 1))),
    ("add/im2col/bk32/tps1", G(6, 5, 17, 32, 256, 1, 4, st=(1, 4), pad=(1, 0))),
    # pq_conv2d_smallc_s8 (C = 8): the row kernel ...
    ("rows", G(3, 40, 40, 8, 64, 7, 7, st=(2, 2), pad=(3, 3))),                # the ResNet stem
    ("rows", G(2, 8, 257, 8, 96, 3, 5, st=(3, 2), pad=(2, 1))),                # Q = 128, two n tiles
    ("rows", G(2, 3, 259, 8, 64, 2, 8, st=(1, 2), pad=(0, 3))),                # Q = 129: tiles_q = 2
    ("rows", G(1, 10, 599, 8, 128, 8, 3, st=(1, 2), pad=(0, 1), Wp=990)),       # stages_fit = 2
    ("smallc-win/tw16", G(1, 10, 599, 8, 128, 8, 3, st=(1, 2), pad=(0, 1), Wp=992)),   # stages_fit = 1
    # ... and the window mode (a_im2col == 2) at each tw_shift
    ("smallc-win/tw8", G(2, 20, 30, 8, 48, 9, 2, st=(3, 2), pad=(4, 0))),      # stride_w 2 with R > 8
    ("smallc-win/tw4", G(5, 9, 20, 8, 32, 2, 6, st=(2, 4), pad=(1, 2))),       # Q = 5
    ("smallc-win/tw8", G(2, 12, 45, 8, 32, 3, 3, st=(1, 6))),                  # Q = 8
    ("smallc-win/tw8", G(3, 12, 60, 8, 32, 3, 1, st=(1, 4), pad=(1, 0))),      # Q = 15
    ("smallc-win/tw16", G(2, 30, 122, 8, 40, 5, 8, st=(5, 8), pad=(2, 3))),    # Q = 16, K % 16 != 0
    ("smallc-win/tw16", G(2, 11, 158, 8, 64, 4, 4, st=(2, 4), pad=(1, 1))),    # Q = 40
    ("smallc-win/tw8", G(1, 66, 20, 8, 32, 64, 1, st=(1, 2))),                 # R = 64
]


def row_id(r):
    g = r[1]
    return "%s-b%d-%dx%dx%d-k%d-%dx%d-s%d.%d-p%d.%d-d%d.%d" % (
        r[0], g["B"], g["H"], g["W"], g["C"], g["K"], g["R"], g["S"], *g["st"], *g["pad"], *g["dil"])


# ------------------------------------------------------------------------------------------ launches through ctypes
class Guarded:
    """An output tensor in the middle of a sentinel-filled buffer (skew: extra bytes in front, breaking alignment)."""

    def __init__(self, shape, dtype, skew=0):
        n = int(np.prod(shape))
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        self.buf = torch.full((nbytes + 2 * GUARD + 16,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.lo, self.hi = GUARD + skew, GUARD + skew + nbytes
        self.t = self.buf[self.lo:self.hi].view(dtype).view(shape)

    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        assert bool((self.buf[:self.lo] == SENTINEL).all()), "%s: bytes before the output were overwritten" % what
        assert bool((self.buf[self.hi:] == SENTINEL).all()), "%s: bytes after the output were overwritten" % what

    def untouched(self):
        return bool((self.buf == SENTINEL).all())


def _lib():
    from common.quantity import _native
    return _native.lib()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _flags(bias, n, relu):
    from common.quantity import _native
    return (_native.FLAG_RELU if relu else 0) | (_native.FLAG_BIAS_FOLDED if bias.numel() == 3 * n else 0)


def _desc(g, rs, ob):
    from common.quantity import _native
    P, Q = out_size(g)
    return _native.ConvDesc(g["B"], g["H"], g["W"], g["C"], g["K"], g["R"], g["S"], *g["st"], *g["pad"], P, Q,
                            rs, ob, *g["dil"], 0, 0)


class Conv:
    """Operands, exact accumulators and launches of one geometry (entry: 'conv', 'add' or 'smallc')."""

    def __init__(self, g, entry, seed):
        self.g, self.entry = g, entry
        self.gen = torch.Generator(device="cuda").manual_seed(seed)
        B, H, W, K, R, S = g["B"], g["H"], g["W"], g["K"], g["R"], g["S"]
        self.P, self.Q = out_size(g)
        self.M, self.K = B * self.P * self.Q, K
        if entry == "smallc":                  # zero-padded image of 8-byte pixels, weights [K][R][8 taps][8 channels]
            self.Hp, self.Wp = smallc_pads(g)
            x = self._int8((B, H, W, 8))
            ph, pw = g["pad"]
            self.x = torch.zeros((B, self.Hp, self.Wp, 8), dtype=torch.int8, device="cuda")
            self.x[:, ph:ph + H, pw:pw + W] = x
            w8 = self._int8((K, R, 8, 8))
            w8[:, :, S:] = 0                   # taps s >= S are zero by contract
            self.w = w8.view(K, R, 64).contiguous()
            self.acc = exact_conv(x, w8[:, :, :S].contiguous(), g["st"], g["pad"], g["dil"])
        else:
            self.x = self._int8((B, H, W, g["C"]))
            self.w = self._int8((K, R, S, g["C"]))
            self.acc = exact_conv(self.x, self.w, g["st"], g["pad"], g["dil"])
        self.x0, self.w0 = self.x.clone(), self.w.clone()
        b = torch.randint(-128, 128, (K,), generator=self.gen, device="cuda", dtype=torch.int32)
        b[:4] = torch.tensor([-128, -1, 0, 127][:K], dtype=torch.int32)
        self.bias = b
        mx = int(self.acc.abs().max()) if self.acc.numel() else 0
        self.rs = max(1, min(20, mx.bit_length() - 6))      # outputs spread over the int8 range, few saturate

    def _int8(self, shape):
        return torch.randint(-128, 128, shape, generator=self.gen, device="cuda", dtype=torch.int8)

    def fold(self, rs):
        from common.quantity import _native
        return _native.bias_fold(self.bias, rs)

    def run(self, rs, ob, bias, relu, out, flags=0):
        """One pq_conv2d_s8 / pq_conv2d_smallc_s8 launch; returns (fp32 as [M][K] or None, int8 [M][K] or None)."""
        f32 = Guarded((self.g["B"], self.K, self.P, self.Q), torch.float32) if out in ("f32", "both") else None
        s8 = Guarded((self.M, self.K), torch.int8) if out in ("s8", "both") else None
        fp, sp = (f32.ptr() if f32 else None), (s8.ptr() if s8 else None)
        flags |= _flags(bias, self.K, relu)
        d = _desc(self.g, rs, ob)
        if self.entry == "smallc":
            rc = _lib().pq_conv2d_smallc_s8(self.x.data_ptr(), self.w.data_ptr(), bias.data_ptr(), ctypes.byref(d),
                                            self.Hp, self.Wp, flags, fp, sp, _stream())
        else:
            rc = _lib().pq_conv2d_s8(self.x.data_ptr(), self.w.data_ptr(), bias.data_ptr(), ctypes.byref(d), flags, fp,
                                     sp, _stream())
        assert rc == 0, "launch failed: %s" % _lib().pq_error_string(rc).decode()
        torch.cuda.synchronize()
        for g, name in ((f32, "fp32"), (s8, "int8")):
            if g is not None:
                g.check(name)
        return (f32.t.permute(0, 2, 3, 1).reshape(self.M, self.K) if f32 else None), (s8.t if s8 else None)

    def run_add(self, rs, ob, bias, sc, sbit, q_bit, out_relu):
        o16, o8 = Guarded((self.M, self.K), torch.int16), Guarded((self.M, self.K), torch.int8)
        from common.quantity import _native
        add = _native.AddDesc(sc.data_ptr(), 1 if sc.dtype == torch.int16 else 0, sbit, 0, int(out_relu), q_bit,
                              o16.ptr(), o8.ptr())
        rc = _lib().pq_conv2d_s8_add(self.x.data_ptr(), self.w.data_ptr(), bias.data_ptr(), ctypes.byref(_desc(self.g, rs, ob)),
                                     ctypes.byref(add), _flags(bias, self.K, False), _stream())
        assert rc == 0, "launch failed: %s" % _lib().pq_error_string(rc).decode()
        torch.cuda.synchronize()
        o16.check("int16"), o8.check("int8")
        return o16.t, o8.t

    def check_operands(self):
        assert torch.equal(self.x, self.x0), "the input was modified"
        assert torch.equal(self.w, self.w0), "the weights were modified"


# ------------------------------------------------------------------------------------------ landing checks
def kernel_name(name):
    """('gemm_s8_kernel', (BN, BK, STAGES, ADDK, BSLOTS)) or ('conv_rows_s8_kernel', None) from a demangled name."""
    if ROWS_KERNEL in name:
        return ROWS_KERNEL
    m = re.search(r"gemm_s8_kernel<([^>]*)>", name)
    if not m:
        return None
    vals = []
    for a in m.group(1).split(","):
        a = re.sub(r"\((int|bool)\)", "", a).strip()
        vals.append({"true": 1, "false": 0}[a] if a in ("true", "false") else int(a))
    return tuple(vals)


def launched(fn):
    """(fn's result, names of every CUDA kernel it launched)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_FRESH_ENV = "PQ_CONV_GEOMETRY_FRESH"
_LANDING = {}


def _landing_state():
    """Whether torch.profiler records kernels in this process.  After some sequences of earlier tests in the same
    pytest process it records no CUDA activity at all; the landing checks then cannot be made here, so this file is
    run once more on its own in a fresh process, where every landing check runs, and that run must pass."""
    if not _LANDING:
        recorded = bool(launched(lambda: torch.ones(16, device="cuda").add_(1))[1])
        _LANDING["recorded"] = recorded
        if not recorded:
            assert not os.environ.get(_FRESH_ENV), "torch.profiler records no CUDA kernels in a fresh process"
            r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-p", "no:cacheprovider",
                                "-m", "gpu"], cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                               env=dict(os.environ, **{_FRESH_ENV: "1"}), capture_output=True, text=True, timeout=3600)
            _LANDING["fresh_run"] = (r.returncode, r.stdout[-3000:])
    return _LANDING


def check_landing(fn, kernel):
    """fn() launches exactly one convolution kernel, `kernel` (an instantiation tuple or ROWS_KERNEL); returns fn()."""
    state = _landing_state()
    if not state["recorded"]:
        res = fn()
        rc, out = state["fresh_run"]
        assert rc == 0, "the fresh-process run of this file, which makes the landing checks, failed:\n" + out
        return res
    res, names = launched(fn)
    found = [k for k in map(kernel_name, names) if k]
    assert found == [kernel], (kernel, names)
    return res


@pytest.fixture(scope="module")
def b200():
    assert torch.cuda.get_device_properties(0).multi_processor_count == SMS, "pick_bn above assumes 148 SMs"


# ------------------------------------------------------------------------------------------ geometry rows (GPU)
def check_values(case, rs, bias_kind, relu, out, what, flags=0, kernel=None):
    bias = case.fold(rs) if bias_kind == "fold" else case.bias
    want = epilogue_ref(case.acc, case.bias.long(), rs, relu)
    run = lambda: case.run(rs, 3, bias, relu, out, flags)            # noqa: E731
    f32, s8 = check_landing(run, kernel) if kernel is not None else run()
    if s8 is not None:
        assert torch.equal(s8.long(), want), what
    if f32 is not None:
        assert torch.equal(f32, dequant_ref(want, 3)), what
    return s8


@gpu
@pytest.mark.parametrize("row", GEOMETRY, ids=[row_id(r) for r in GEOMETRY])
def test_geometry_row_vs_exact_convolution(row, b200):
    path, g = row
    entry = "smallc" if path.startswith(("rows", "smallc")) else ("add" if path.startswith("add/") else "conv")
    name, kernel = expected_path(path, g)
    assert name == path, (name, path)
    case = Conv(g, entry, zlib.crc32(row_id(row).encode()))
    rs = case.rs
    want = epilogue_ref(case.acc, case.bias.long(), rs, False)
    assert int((want != want[0, 0]).sum()) > 0 and bool(((want > -128) & (want < 127)).any()), "degenerate row"
    if entry == "add":
        sc = torch.randint(-128, 128, (case.M, case.K), generator=case.gen, device="cuda", dtype=torch.int8)
        for i, (kind, ob, sbit, q, relu) in enumerate((("fold", 4, 3, 4, True), ("plain", 2, 5, 6, False))):
            bias = case.fold(rs) if kind == "fold" else case.bias
            run = lambda: case.run_add(rs, ob, bias, sc, sbit, q, relu)          # noqa: E731
            o16, o8 = check_landing(run, kernel) if i == 0 else run()
            w16, w8 = add_ref(epilogue_ref(case.acc, case.bias.long(), rs, False), ob, sc.long(), sbit, False, relu, q)
            assert torch.equal(o16.long(), w16) and torch.equal(o8.long(), w8), (kind, ob, sbit, q, relu)
        case.check_operands()
        return
    if path.startswith("win"):
        from common.quantity import _native
        # the im2col form first: it leaves its operand bytes in the shared memory the window ring does not fill
        ref8 = check_values(case, rs, "fold", False, "s8", "no windows", _native.FLAG_NO_WINDOWS,
                            conv_path(g, no_windows=True)[1])
        win8 = check_values(case, rs, "fold", False, "s8", "windows", 0, kernel)
        assert torch.equal(win8, ref8)
        check_values(case, min(rs + 1, 24), "plain", True, "both", "windows, generic epilogue")
    else:
        check_values(case, rs, "fold", False, "s8", "staged int8", 0, kernel)
        check_values(case, min(rs + 1, 24), "plain", True, "both", "generic epilogue")
    case.check_operands()


# ------------------------------------------------------------------------------------------ limits
# One row inside and one beyond every limit of the header's text (include/pq_sm100.h).  Fields: entry, the limit it
# probes, geometry, expected return code.  Accepted rows run and are compared with the reference.
def _S(g, **kw):
    """a small-channel geometry (C = 8) with optional Hp / Wp overrides"""
    return dict(g, C=8, **kw)


LIMITS = [
    ("conv", "stride <= 8", G(2, 17, 3, 32, 16, 2, 1, st=(8, 1)), 0),
    ("conv", "stride <= 8", G(2, 17, 3, 32, 16, 2, 1, st=(9, 1)), EUNSUPPORTED),
    ("conv", "stride <= 8", G(2, 3, 17, 32, 16, 1, 2, st=(1, 8)), 0),
    ("conv", "stride <= 8", G(2, 3, 17, 32, 16, 1, 2, st=(1, 9)), EUNSUPPORTED),
    ("conv", "pad <= 128", G(1, 1, 3, 32, 16, 2, 1, pad=(128, 0)), 0),
    ("conv", "pad <= 128", G(1, 1, 3, 32, 16, 2, 1, pad=(129, 0)), EUNSUPPORTED),
    ("conv", "pad <= 128", G(1, 3, 1, 32, 16, 1, 2, pad=(0, 128)), 0),
    ("conv", "pad <= 128", G(1, 3, 1, 32, 16, 1, 2, pad=(0, 129)), EUNSUPPORTED),
    ("conv", "pad - (R-1)*dil <= 127", G(1, 2, 4, 32, 16, 1, 3, pad=(127, 1)), 0),
    ("conv", "pad - (R-1)*dil <= 127", G(1, 2, 4, 32, 16, 1, 3, pad=(128, 1)), EUNSUPPORTED),
    ("conv", "pad - (R-1)*dil <= 127", G(1, 4, 2, 32, 16, 3, 1, pad=(1, 127)), 0),
    ("conv", "pad - (R-1)*dil <= 127", G(1, 4, 2, 32, 16, 3, 1, pad=(1, 128)), EUNSUPPORTED),
    ("conv", "(R-1)*dil - pad <= 128", G(1, 130, 3, 32, 16, 2, 1, dil=(128, 1)), 0),
    ("conv", "(R-1)*dil - pad <= 128", G(1, 130, 3, 32, 16, 2, 1, dil=(129, 1)), EUNSUPPORTED),
    ("conv", "(R-1)*dil - pad <= 128", G(1, 3, 140, 32, 16, 3, 3, pad=(1, 2), dil=(1, 65)), 0),
    ("conv", "(R-1)*dil - pad <= 128", G(1, 140, 140, 32, 16, 3, 3, dil=(65, 65)), EUNSUPPORTED),
    ("conv", "(R-1)*dil + 1 <= 255", G(1, 3, 3, 32, 16, 3, 3, pad=(126, 126), dil=(127, 127)), 0),
    ("conv", "(R-1)*dil + 1 <= 255", G(1, 3, 3, 32, 16, 2, 1, pad=(126, 0), dil=(254, 1)), 0),
    ("conv", "(R-1)*dil + 1 <= 255", G(1, 3, 3, 32, 16, 2, 1, pad=(127, 0), dil=(255, 1)), EUNSUPPORTED),
    ("conv", "(R-1)*dil + 1 <= 255", G(1, 3, 3, 32, 16, 1, 2, pad=(0, 127), dil=(1, 255)), EUNSUPPORTED),
    ("conv", "C % 32 == 0 off the plain path", G(2, 5, 7, 48, 16, 1, 1), 0),
    ("conv", "C % 32 == 0 off the plain path", G(2, 5, 7, 48, 16, 1, 1, st=(2, 1)), EUNSUPPORTED),
    ("conv", "C % 32 == 0 off the plain path", G(2, 5, 7, 64, 16, 1, 1, st=(2, 1)), 0),
    ("conv", "C % 32 == 0 off the plain path", G(2, 5, 7, 48, 16, 3, 3, pad=(1, 1)), EUNSUPPORTED),
    ("conv", "C % 16 == 0", G(2, 5, 7, 16, 16, 1, 1), 0),
    ("conv", "C % 16 == 0", G(2, 5, 7, 40, 16, 1, 1), EALIGN),
    ("smallc", "C == 8", _S(G(1, 12, 30, 8, 32, 3, 3, st=(1, 2), pad=(1, 1))), 0),
    ("smallc", "C == 8", G(1, 12, 30, 16, 32, 3, 3, st=(1, 2), pad=(1, 1)), EUNSUPPORTED),
    ("smallc", "S <= 8", _S(G(1, 12, 30, 8, 32, 3, 8, st=(1, 2), pad=(1, 1))), 0),
    ("smallc", "S <= 8", _S(G(1, 12, 30, 8, 32, 3, 9, st=(1, 2), pad=(1, 1))), EUNSUPPORTED),
    ("smallc", "even stride_w", _S(G(1, 12, 30, 8, 32, 3, 3, st=(1, 4), pad=(1, 1))), 0),
    ("smallc", "even stride_w", _S(G(1, 12, 30, 8, 32, 3, 3, st=(1, 3), pad=(1, 1))), EUNSUPPORTED),
    ("smallc", "R <= 64", _S(G(1, 70, 12, 8, 32, 64, 3, st=(1, 2), pad=(0, 1))), 0),
    ("smallc", "R <= 64", _S(G(1, 70, 12, 8, 32, 65, 3, st=(1, 2), pad=(0, 1))), EUNSUPPORTED),
    ("smallc", "Hp % stride_h == 0", _S(G(1, 11, 12, 8, 32, 2, 3, st=(2, 2)), Hp=12), 0),
    ("smallc", "Hp % stride_h == 0", _S(G(1, 11, 12, 8, 32, 2, 3, st=(2, 2)), Hp=13), EUNSUPPORTED),
    ("smallc", "Hp >= (P-1)*stride_h + R", _S(G(1, 10, 12, 8, 32, 3, 3, st=(1, 2), pad=(1, 1)), Hp=12), 0),
    ("smallc", "Hp >= (P-1)*stride_h + R", _S(G(1, 10, 12, 8, 32, 3, 3, st=(1, 2), pad=(1, 1)), Hp=11), EUNSUPPORTED),
    ("smallc", "Hp >= H + pad_h", _S(G(1, 11, 12, 8, 32, 2, 3, st=(2, 2)), Hp=12), 0),
    ("smallc", "Hp >= H + pad_h", _S(G(1, 11, 12, 8, 32, 2, 3, st=(2, 2)), Hp=10), EUNSUPPORTED),
    ("smallc", "Wp even", _S(G(1, 6, 12, 8, 32, 3, 3, st=(1, 2)), Wp=18), 0),
    ("smallc", "Wp even", _S(G(1, 6, 12, 8, 32, 3, 3, st=(1, 2)), Wp=17), EUNSUPPORTED),
    ("smallc", "Wp >= (Q-1)*stride_w + 8", _S(G(1, 6, 12, 8, 32, 3, 3, st=(1, 2)), Wp=16), 0),
    ("smallc", "Wp >= (Q-1)*stride_w + 8", _S(G(1, 6, 12, 8, 32, 3, 3, st=(1, 2)), Wp=14), EUNSUPPORTED),
    ("smallc", "Wp >= W + pad_w", _S(G(1, 6, 25, 8, 32, 3, 2, st=(1, 8)), Wp=26), 0),
    ("smallc", "Wp >= W + pad_w", _S(G(1, 6, 25, 8, 32, 3, 2, st=(1, 8)), Wp=24), EUNSUPPORTED),
    ("smallc", "dilation 1", _S(G(1, 12, 30, 8, 32, 3, 3, st=(1, 2), pad=(1, 1))), 0),
    ("smallc", "dilation 1", _S(G(1, 12, 30, 8, 32, 3, 3, st=(1, 2), pad=(1, 1), dil=(2, 1))), EUNSUPPORTED),
    ("smallc", "dilation 1", _S(G(1, 12, 30, 8, 32, 3, 3, st=(1, 2), pad=(1, 1), dil=(1, 2))), EUNSUPPORTED),
]
# limits whose rows are the index tests at size (test_*_at_size below)
SIZE_LIMITS = {"conv": ["N*P*Q <= 2^31 - 1"], "smallc": ["patches*128 <= 2^31 - 1"]}


def limit_id(r):
    return "%s-%s-%s" % (r[0], re.sub(r"[^0-9A-Za-z]+", "_", r[1]).strip("_"), "ok" if r[3] == 0 else "refused")


@gpu
@pytest.mark.parametrize("row", LIMITS, ids=[limit_id(r) + "-%d" % i for i, r in enumerate(LIMITS)])
def test_limit_one_step_inside_and_beyond(row, b200):
    entry, _, g, want = row
    case = Conv(g, entry, zlib.crc32(repr(row).encode())) if want == 0 else None
    if case is None:                           # operands sized by the geometry all the same: a refusal must not read
        case = Conv.__new__(Conv)
        case.g, case.entry = g, entry
        case.P, case.Q = out_size(g)
        case.M, case.K = g["B"] * case.P * case.Q, g["K"]
        if entry == "smallc":
            case.Hp, case.Wp = smallc_pads(g)
            case.x = torch.zeros((g["B"], case.Hp, case.Wp, 8), dtype=torch.int8, device="cuda")
            case.w = torch.ones((g["K"], g["R"], 64), dtype=torch.int8, device="cuda")
        else:
            case.x = torch.ones((g["B"], g["H"], g["W"], g["C"]), dtype=torch.int8, device="cuda")
            case.w = torch.ones((g["K"], g["R"], g["S"], g["C"]), dtype=torch.int8, device="cuda")
        outs = (Guarded((g["B"], g["K"], case.P, case.Q), torch.float32), Guarded((case.M, case.K), torch.int8))
        bias = torch.zeros(g["K"], dtype=torch.int32, device="cuda")
        d = _desc(g, 7, 0)
        if entry == "smallc":
            rc = _lib().pq_conv2d_smallc_s8(case.x.data_ptr(), case.w.data_ptr(), bias.data_ptr(), ctypes.byref(d),
                                            case.Hp, case.Wp, 0, outs[0].ptr(), outs[1].ptr(), _stream())
        else:
            rc = _lib().pq_conv2d_s8(case.x.data_ptr(), case.w.data_ptr(), bias.data_ptr(), ctypes.byref(d), 0,
                                     outs[0].ptr(), outs[1].ptr(), _stream())
        torch.cuda.synchronize()
        assert rc == want, (rc, want)
        assert all(o.untouched() for o in outs), "a refused call wrote"
        return
    check_values(case, case.rs, "fold", False, "s8", "inside the limit")
    check_values(case, case.rs, "plain", False, "both", "inside the limit, generic epilogue")
    case.check_operands()


# ------------------------------------------------------------------------------------------ index limits at size
def _chunks(n, step):
    for i in range(0, n, step):
        yield i, min(n, i + step)


@gpu
def test_m_limit_at_size(b200):
    """M = N*P*Q at 2^31 - 1 through pad 127 on 1x1 images: 33025 images of 1x1x32, one 1x1 filter, P = Q = 255, so
    M = 2,147,450,625 is accepted (about 2 GB of int8 output, only each image's centre pixel has a non-zero
    accumulator); 33026 images are refused and write nothing."""
    n_ok, hw, centre = 33025, 255 * 255, 127 * 255 + 127
    g = G(n_ok + 1, 1, 1, 32, 1, 1, 1, pad=(127, 127))
    gen = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randint(-128, 128, (n_ok + 1, 1, 1, 32), generator=gen, device="cuda", dtype=torch.int8)
    w = torch.randint(-128, 128, (1, 1, 1, 32), generator=gen, device="cuda", dtype=torch.int8)
    x0, w0 = x.clone(), w.clone()
    bias = torch.tensor([5], dtype=torch.int32, device="cuda")
    rs = 12
    out = Guarded(((n_ok + 1) * hw,), torch.int8)
    assert (n_ok + 1) * hw > M_LIMIT >= n_ok * hw
    rc = _lib().pq_conv2d_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(), ctypes.byref(_desc(g, rs, 0)), 0, None,
                             out.ptr(), _stream())
    torch.cuda.synchronize()
    assert rc == EUNSUPPORTED and out.untouched()
    g["B"] = n_ok
    rc = check_landing(lambda: _lib().pq_conv2d_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                                   ctypes.byref(_desc(g, rs, 0)), 0, None, out.ptr(), _stream()),
                       inst(32, 32))
    torch.cuda.synchronize()
    assert rc == 0
    assert conv_path(g) == ("im2col/bk32/tps1", inst(32, 32))
    acc = (x[:n_ok, 0, 0].double() @ w[0, 0, 0].double()).round().long()
    centre_want = epilogue_ref(acc.view(-1, 1), bias.long(), rs, False).view(-1).to(torch.int8)
    assert int(centre_want.unique().numel()) > 20
    img = out.t[:n_ok * hw].view(n_ok, hw)
    for a, b in _chunks(n_ok, 4096):
        part = img[a:b]
        assert torch.equal(part[:, centre], centre_want[a:b])
        assert bool((part[:, :centre] == 5).all()) and bool((part[:, centre + 1:] == 5).all()), (a, b)
    assert bool((out.buf[out.lo + n_ok * hw:] == SENTINEL).all()) and bool((out.buf[:out.lo] == SENTINEL).all())
    assert torch.equal(x, x0) and torch.equal(w, w0)


@gpu
def test_patch_window_limit_at_size(b200):
    """Patch windows address patches * 128 GEMM rows in 32 bits: C = K = 128 on 1x1 images (3x3, pad 1: only the
    centre tap reads the image) stays on the windows at 2^24 - 1 images and falls back to im2col at 2^24."""
    n = 1 << 24
    gen = torch.Generator(device="cuda").manual_seed(12)
    x = torch.randint(-128, 128, (n, 1, 1, 128), generator=gen, device="cuda", dtype=torch.int8)
    w = torch.randint(-128, 128, (128, 3, 3, 128), generator=gen, device="cuda", dtype=torch.int8)
    bias = torch.randint(-128, 128, (128,), generator=gen, device="cuda", dtype=torch.int32)
    from common.quantity import _native
    rs = 15
    fold = _native.bias_fold(bias, rs)
    w0 = w.clone()
    x_sum = int(x[::4099].long().sum())
    wc = w[:, 1, 1].double().t().contiguous()
    out = Guarded((n, 128), torch.int8)
    for batch, want_path in ((n - 1, ("win/tw16", WIN128)), (n, ("im2col/bk128/tps1", inst(128, 128)))):
        g = G(batch, 1, 1, 128, 128, 3, 3, pad=(1, 1))
        assert conv_path(g) == want_path
        out.buf.fill_(SENTINEL)
        rc = check_landing(lambda: _lib().pq_conv2d_s8(x.data_ptr(), w.data_ptr(), fold.data_ptr(),
                                                       ctypes.byref(_desc(g, rs, 0)), _native.FLAG_BIAS_FOLDED, None,
                                                       out.ptr(), _stream()), want_path[1])
        torch.cuda.synchronize()
        assert rc == 0
        for a, b in _chunks(batch, 1 << 18):
            acc = (x[a:b, 0, 0].double() @ wc).round().long()
            assert torch.equal(out.t[a:b].long(), epilogue_ref(acc, bias.long(), rs, False)), (batch, a)
        assert bool((out.buf[out.lo + batch * 128:] == SENTINEL).all()) and bool((out.buf[:out.lo] == SENTINEL).all())
    assert int(x[::4099].long().sum()) == x_sum and torch.equal(w, w0)


@gpu
def test_row_kernel_limit_at_size(b200):
    """The row kernel addresses tiles_m * 128 GEMM rows in 32 bits: P = 2, Q = 1 stays on it at 2^23 - 1 images and
    falls back to the window mode of gemm_s8_kernel at 2^23."""
    n, K = 1 << 23, 16
    g = G(n, 3, 3, 8, K, 2, 3, st=(1, 2))
    Hp, Wp = smallc_pads(g)
    assert (Hp, Wp) == (3, 8)
    gen = torch.Generator(device="cuda").manual_seed(13)
    xp = torch.randint(-128, 128, (n, Hp, Wp, 8), generator=gen, device="cuda", dtype=torch.int8)
    w8 = torch.randint(-128, 128, (K, 2, 8, 8), generator=gen, device="cuda", dtype=torch.int8)
    w8[:, :, 3:] = 0
    w = w8.view(K, 2, 64).contiguous()
    wm = w8[:, :, :3].reshape(K, 48).double().t().contiguous()     # rows (r, s, c) of one output pixel's window
    bias = torch.randint(-128, 128, (K,), generator=gen, device="cuda", dtype=torch.int32)
    rs = 11
    out = Guarded((n * 2, K), torch.int8)
    for batch, want_path in ((n - 1, ("rows", ROWS_KERNEL)), (n, ("smallc-win/tw4", inst(32, 64)))):
        g["B"] = batch
        assert smallc_path(g) == want_path
        out.buf.fill_(SENTINEL)
        rc = check_landing(lambda: _lib().pq_conv2d_smallc_s8(xp.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                                              ctypes.byref(_desc(g, rs, 0)), Hp, Wp, 0, None,
                                                              out.ptr(), _stream()), want_path[1])
        torch.cuda.synchronize()
        assert rc == 0
        o = out.t[:batch * 2].view(batch, 2, K)
        for a, b in _chunks(batch, 1 << 20):
            for p in range(2):
                acc = (xp[a:b, p:p + 2, :3].reshape(b - a, 48).double() @ wm).round().long()
                assert torch.equal(o[a:b, p].long(), epilogue_ref(acc, bias.long(), rs, False)), (batch, a, p)
        assert bool((out.buf[out.lo + batch * 2 * K:] == SENTINEL).all()) and bool((out.buf[:out.lo] == SENTINEL).all())


@gpu
def test_small_channel_window_limit_at_size(b200):
    """The window mode of pq_conv2d_smallc_s8 addresses patches * 128 GEMM rows in 32 bits: 1x1 outputs at stride_w 4
    (one 4 x 32 patch an image) are accepted at 2^24 - 1 images and refused at 2^24, writing nothing."""
    n, K = 1 << 24, 16
    g = G(n, 1, 1, 8, K, 1, 1, st=(1, 4))
    Hp, Wp = smallc_pads(g)
    assert (Hp, Wp) == (1, 8)
    gen = torch.Generator(device="cuda").manual_seed(14)
    xp = torch.randint(-128, 128, (n, Hp, Wp, 8), generator=gen, device="cuda", dtype=torch.int8)
    w8 = torch.zeros((K, 1, 8, 8), dtype=torch.int8, device="cuda")
    w8[:, :, 0] = torch.randint(-128, 128, (K, 1, 8), generator=gen, device="cuda", dtype=torch.int8)
    w = w8.view(K, 1, 64).contiguous()
    bias = torch.randint(-128, 128, (K,), generator=gen, device="cuda", dtype=torch.int32)
    rs = 9
    out = Guarded((n, K), torch.int8)
    rc = _lib().pq_conv2d_smallc_s8(xp.data_ptr(), w.data_ptr(), bias.data_ptr(), ctypes.byref(_desc(g, rs, 0)), Hp,
                                    Wp, 0, None, out.ptr(), _stream())
    torch.cuda.synchronize()
    assert rc == EUNSUPPORTED and out.untouched()
    g["B"] = n - 1
    assert smallc_path(g) == ("smallc-win/tw4", inst(32, 64))
    rc = check_landing(lambda: _lib().pq_conv2d_smallc_s8(xp.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                                          ctypes.byref(_desc(g, rs, 0)), Hp, Wp, 0, None, out.ptr(),
                                                          _stream()), inst(32, 64))
    torch.cuda.synchronize()
    assert rc == 0
    wm = w8[:, 0, 0].double().t().contiguous()
    for a, b in _chunks(n - 1, 1 << 20):
        acc = (xp[a:b, 0, 0].double() @ wm).round().long()
        assert torch.equal(out.t[a:b].long(), epilogue_ref(acc, bias.long(), rs, False)), a
    assert bool((out.buf[out.lo + (n - 1) * K:] == SENTINEL).all()) and bool((out.buf[:out.lo] == SENTINEL).all())


# ------------------------------------------------------------------------------------------ NewConv2d
def _layer(C, K, k, st, pad, dil=(1, 1), seed=0):
    """An nn.Conv2d with integer-friendly parameters and the quantisation info that spreads its outputs over int8:
    input bit 4, output bit 3, weights of magnitude <= 127 at weight_bit."""
    R, S = k
    acc = (R * S * C) ** 0.5 * 55 * 60
    rs = max(1, int(np.ceil(np.log2(acc))) - 6)
    info = {"weight_bit": rs - 1, "input_bit": 4, "output_bit": 3, "bias_bit": 3}
    g = torch.Generator().manual_seed(seed)
    conv = nn.Conv2d(C, K, k, st, pad, dil)
    with torch.no_grad():
        conv.weight.copy_((torch.rand(conv.weight.shape, generator=g) * 2 - 1) * 127 * 2.0 ** -info["weight_bit"])
        conv.bias.copy_((torch.rand(K, generator=g) * 2 - 1) * 100 / 8)
    return conv, info


# (C, K, kernel, stride, padding, dilation, input H x W, the path flag NewConv2d must choose)
NEWCONV = [
    (3, 16, (7, 7), (2, 2), (3, 3), (1, 1), (37, 30), "s2d"),                # the stem
    (1, 32, (4, 6), (2, 2), (1, 2), (1, 1), (23, 30), "s2d"),                # even R, R != S, unequal pads
    (2, 8, (5, 3), (2, 2), (2, 0), (1, 1), (19, 16), "s2d"),
    (4, 64, (6, 6), (2, 2), (3, 1), (1, 1), (20, 21), "s2d"),                # odd and unequal pads
    (3, 16, (3, 3), (1, 2), (1, 1), (1, 1), (15, 20), "smallc"),             # stride (1, 2): no space-to-depth
    (5, 16, (3, 5), (1, 2), (1, 2), (1, 1), (14, 25), "smallc"),
    (8, 48, (2, 8), (3, 4), (0, 3), (1, 1), (20, 40), "smallc"),
    (3, 16, (3, 3), (2, 3), (1, 1), (1, 1), (17, 20), "explicit_im2col"),    # odd stride_w
    (6, 24, (2, 9), (1, 2), (0, 4), (1, 1), (10, 30), "explicit_im2col"),    # S > 8
    (1, 32, (5, 5), (1, 1), (2, 2), (1, 1), (16, 16), "explicit_im2col"),
    (9, 32, (3, 2), (2, 1), (1, 0), (1, 2), (15, 12), 32),                   # C = 9..31 -> 32 channels
    (17, 48, (1, 3), (1, 1), (0, 1), (1, 1), (9, 14), 32),
    (31, 16, (5, 1), (1, 3), (2, 0), (2, 1), (20, 11), 32),
    (20, 32, (3, 2), (2, 1), (1, 1), (1, 1), (11, 9), 32),
    (9, 16, (1, 1), (1, 1), (0, 0), (1, 1), (7, 9), 16),                     # plain GEMM: 16 channels
    (3, 16, (3, 3), (1, 1), (2, 2), (2, 2), (12, 13), 32),                   # dilated with few channels
    (64, 64, (3, 3), (1, 1), (1, 1), (1, 1), (14, 15), 64),                  # patch windows
]


def _flag(mod, want):
    """NewConv2d chose the path `want`: a payload channel count, or the flag of another operand layout."""
    got = {f for f in ("s2d", "smallc", "explicit_im2col") if getattr(mod, "_" + f)}
    if isinstance(want, int):
        return mod._payload_channels == want and not got
    return mod._payload_channels is None and got == ({"s2d", "smallc"} if want == "s2d" else {want})


@gpu
@pytest.mark.parametrize("layer", NEWCONV, ids=["c%d-k%d-%dx%d-s%d.%d-p%d.%d-d%d.%d-%s" % (
    l[0], l[1], *l[2], *l[3], *l[4], *l[5], l[7]) for l in NEWCONV])
def test_newconv2d_path_choice_vs_oracle(layer, oracle):
    from common.quantity import NewConv2d
    C, K, k, st, pad, dil, (H, W), want = layer
    conv, info = _layer(C, K, k, st, pad, dil, seed=zlib.crc32(repr(layer).encode()))
    wf, bf = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = (torch.randn((2, C, H, W), generator=torch.Generator().manual_seed(1)) * 4)
    mod = NewConv2d(conv, dict(info))
    assert _flag(mod, want), (want, mod._payload_channels, mod._s2d, mod._smallc, mod._explicit_im2col)
    with torch.no_grad():
        y = mod(x.cuda()).cpu().numpy()
    ref, yi = oracle.int_conv_layer(x.numpy(), wf, bf, info, stride=st, padding=pad, dilation=dil)
    assert np.array_equal(y, ref)
    assert len(np.unique(yi)) > 20


@gpu
@pytest.mark.parametrize("layer", [l for l in NEWCONV if l[5] == (1, 1) and l[1] % 16 == 0 and isinstance(l[7], int)],
                         ids=lambda l: "c%d-k%d-%dx%d" % (l[0], l[1], *l[2]))
def test_newconv2d_fused_add_in_the_int8_pipeline(layer, oracle):
    """Layers where _fuses_add holds, followed by a NewAdd in the int8 pipeline: one pq_conv2d_s8_add launch whose
    exact sum equals the fp32-boundary NewAdd of the oracle's layer output and the shortcut."""
    from common.quantity import NewAdd, NewConv2d, _native
    from common.quantity.int8_pipeline import QTensor
    C, K, k, st, pad, dil, (H, W), _ = layer
    conv, info = _layer(C, K, k, st, pad, dil, seed=zlib.crc32(repr(layer).encode()) + 1)
    wf, bf = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = (torch.randn((2, C, H, W), generator=torch.Generator().manual_seed(2)) * 4)
    mod = NewConv2d(conv, dict(info))
    assert mod._fuses_add
    ref, _ = oracle.int_conv_layer(x.numpy(), wf, bf, info, stride=st, padding=pad, dilation=dil)
    P, Q = ref.shape[2:]
    sbit = 5
    sc = torch.randint(-128, 128, (2, P, Q, K), generator=torch.Generator().manual_seed(3), dtype=torch.int8).cuda()
    add = NewAdd()
    add.output_bit = 4
    mod.int8_pipeline = add.int8_pipeline = True
    before = _native.LAUNCHES.get("conv_add_s8", 0)
    with torch.no_grad():
        out = add(mod(x.cuda()), QTensor((2, K, P, Q), sc.device, q8=sc, q8_bit=sbit)).dequantize().cpu().numpy()
    assert _native.LAUNCHES.get("conv_add_s8", 0) == before + 1
    want = np.clip(ref + sc.permute(0, 3, 1, 2).float().cpu().numpy() * np.float32(2.0 ** -sbit), -128, 127)
    assert np.array_equal(out, want)


@gpu
@pytest.mark.parametrize("conv", [dict(k=3, stride=9), dict(k=3, dilation=65), dict(k=2, padding=129),
                                  dict(k=(1, 3), padding=(128, 1))], ids=["stride9", "dil65", "pad129", "pad128_r1"])
def test_newconv2d_outside_the_kernel_limits_raises_on_first_forward(conv):
    """A legal nn.Conv2d outside the kernels' geometry limits: quantity() succeeds, the first forward raises a
    RuntimeError naming PQ_EUNSUPPORTED (there is no fall-back)."""
    from common.quantity import NewConv2d
    kw = dict(conv)
    k = kw.pop("k")
    layer = nn.Conv2d(32, 16, k, **kw)
    mod = NewConv2d(layer, {"weight_bit": 7, "input_bit": 4, "output_bit": 3, "bias_bit": 3})
    x = torch.randn(1, 32, 140, 140, device="cuda")
    assert mod._payload_channels == 32
    with pytest.raises(RuntimeError, match="PQ_EUNSUPPORTED"):
        mod(x)


# ------------------------------------------------------------------------------------------ CPU checks
def test_reference_equals_oracle_on_rectangular_asymmetric_dilated_layers(oracle):
    """exact_conv + epilogue_ref against the oracle's NewConv2d (int_conv_layer) on integer-valued operands."""
    g = torch.Generator().manual_seed(4)
    for (R, S), st, pad, dil in (((2, 3), (2, 1), (1, 2), (2, 1)), ((1, 5), (3, 2), (0, 3), (1, 2)),
                                 ((4, 1), (1, 4), (3, 0), (1, 1)), ((3, 3), (2, 3), (2, 1), (2, 3))):
        x = torch.randint(-128, 128, (2, 9, 11, 32), generator=g, dtype=torch.int8)
        w = torch.randint(-128, 128, (16, R, S, 32), generator=g, dtype=torch.int8)
        b = torch.randint(-128, 128, (16,), generator=g, dtype=torch.int32)
        acc = exact_conv(x, w, st, pad, dil)
        for wb, ib, ob in ((9, 7, -4), (7, 7, 1), (2, 1, 3), (6, 6, -12)):
            info = {"weight_bit": wb, "input_bit": ib, "output_bit": ob, "bias_bit": 2}
            xf = (x.permute(0, 3, 1, 2).double() * 2.0 ** -ib).float().numpy()
            wf = (w.permute(0, 3, 1, 2).double() * 2.0 ** -wb).float().numpy()
            bf = (b.double() * 2.0 ** -2).float().numpy()
            f32, y = oracle.int_conv_layer(xf, wf, bf, info, stride=st, padding=pad, dilation=dil)
            want = epilogue_ref(acc, b.long(), wb + ib - ob, False)
            P, Q = y.shape[2:]
            assert np.array_equal(want.view(2, P, Q, 16).permute(0, 3, 1, 2).numpy(), y), (R, S, st, pad, dil)
            assert np.array_equal(dequant_ref(want, ob).view(2, P, Q, 16).permute(0, 3, 1, 2).numpy(), f32)


def test_every_row_takes_the_path_it_names():
    """Each GEOMETRY row lands on the path it names, and between them the rows reach every path and instantiation
    the dense convolution selects."""
    kernels = set()
    for path, g in GEOMETRY:
        name, kernel = expected_path(path, g)
        assert name == path, (name, path, g)
        kernels.add(kernel)
        if path.startswith("win"):
            kernels.add(conv_path(g, no_windows=True)[1])
    names = {p for p, _ in GEOMETRY}
    for want in ("gemm", "im2col/bk32/tps1", "im2col/bk32/tps3", "im2col/bk64/tps1", "im2col/bk64/tps3",
                 "im2col/deep", "im2col/bk128/tps1", "win/tw16", "win/tw32", "win/tw64", "add/gemm", "rows",
                 "smallc-win/tw4", "smallc-win/tw8", "smallc-win/tw16"):
        assert want in names, want
    assert any(p.startswith("add/im2col") for p in names)
    assert {DEEP_A, WIN128, ROWS_KERNEL} <= kernels
    # C = 96 and 192 give three channel blocks per tap
    assert {32, 64, 96, 128, 192, 2048} <= {g["C"] for p, g in GEOMETRY}
    # C = 64 at every width around the three window widths (W + 2 = 65 falls back to im2col)
    assert {g["W"] for p, g in GEOMETRY if g["C"] == 64 and g["R"] == g["S"] == 3 and g["st"] == (1, 1) and
            g["pad"] == (1, 1) and g["dil"] == (1, 1)} >= {13, 14, 15, 29, 30, 31, 61, 62, 63}


def test_row_kernel_over_read_is_implied_by_the_wp_requirement():
    """The row kernel's over-read condition, (R-1)*pitch + (tiles_q*128 - 1)*16 + 64 <= a_stage, holds for every
    padded width the entry point accepts (Wp >= (Q-1)*2 + 8): tiles_q*128 <= Q + 127, so the left side is at most
    (R-1)*pitch + 16*(Q-1) + 2096 <= R*pitch + 2032 < a_stage.  That fall-back to the window mode cannot be reached,
    and no row can probe it."""
    for R in range(1, 9):
        for Q in list(range(1, 300)) + [1000, 4096, 65535]:
            for Wp in {(Q - 1) * 2 + 8, (Q - 1) * 2 + 10, 2 * Q + 40}:
                assert rows_fit(R, 64, Q, Wp)[1], (R, Q, Wp)
    assert rows_fit(8, 128, 300, 990) == (True, True) and rows_fit(8, 128, 300, 992) == (False, True)


def test_every_documented_limit_has_an_inside_and_a_beyond_row():
    """Each limit the header documents for pq_conv2d_s8 and pq_conv2d_smallc_s8 (include/pq_sm100.h, marked
    'limit:') has a LIMITS row one step inside (accepted) and one beyond (refused), or a test at size."""
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "pq_sm100.h")).read()
    documented = {"conv": re.findall(r"conv limit: ([^;\n]+?)(?:;|\s*\*/|\n)", header),
                  "smallc": re.findall(r"smallc limit: ([^;\n]+?)(?:;|\s*\*/|\n)", header)}
    assert len(documented["conv"]) >= 6 and len(documented["smallc"]) >= 8, documented
    for entry, limits in documented.items():
        for lim in limits:
            lim = lim.strip()
            if lim in SIZE_LIMITS[entry]:
                continue
            codes = {r[3] == 0 for r in LIMITS if r[0] == entry and r[1] == lim}
            assert codes == {True, False}, (entry, lim)
        assert {r[1] for r in LIMITS if r[0] == entry} <= {x.strip() for x in limits}, entry

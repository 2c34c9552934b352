"""Grouped convolutions on the GEMM kernel (pq_conv2d_s8 with pq_conv_desc.groups > 1, NewConv2d's grouped path) against
an evaluation that shares nothing with the kernel:

    acc = float64 F.conv2d(..., groups=G) of the int8 operands, rounded to int64                exact: |acc| < 2^53
    y   = clamp(clamp(RightShift(acc, rs)) + b) [ReLU], fp32 = y / 2^ob                          new_quantity_op.py:11-44,124-133

Every kernel output is written into the middle of a sentinel-filled buffer; the bytes around it, the input and the
weights must survive.  The layer tests compare with the CPU oracle (oracle.int_conv_layer(..., groups=G)).

Output channels come in whole tiles of group_block >= 32 channels (K % group_block == 0), so K % 16 != 0 cannot occur
on this path; the unstaged int8 store (the generic epilogue's direct stores) is reached with an int8 output that is not
16-byte aligned instead.
"""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

gpu = pytest.mark.gpu

PQ_EINVAL, PQ_EUNSUPPORTED = -1, -2
RS_VALUES = (-24, -8, -1, 0, 1, 2, 7, 13, 20, 21, 24)
OB_VALUES = (-100, -3, 0, 4, 100)
OUTPUTS = ("f32", "s8", "s8_unstaged", "both")
GUARD = 4096                      # sentinel bytes before and after every output


def _legal_blocks(K, G):
    Kg = K // G
    return [b for b in (32, 64, 128, 256) if (b % Kg == 0 or Kg % b == 0) and K % b == 0]


# ------------------------------------------------------------------------------------------ CPU: the weight layout
@pytest.mark.parametrize("C,K,G,stride,dil", [
    (64, 64, 8, 1, 1),            # Cg == Kg
    (32, 128, 8, 1, 1),           # Cg < Kg
    (128, 64, 8, 1, 1),           # Cg > Kg
    (64, 256, 2, 2, 1),           # stride 2, Kg > every block
    (96, 96, 3, 1, 2),            # dilation 2
    (256, 256, 64, 1, 1),         # Cg == Kg == 4 (ResNeXt-50's first stage)
])
def test_grouped_filter_layout(C, K, G, stride, dil):
    """Per tile of every legal group_block: a dense conv over the tile's channel window with its grouped_filter rows equals
    the grouped convolution's output channels of the tile, exactly (float64 on integers)."""
    from common.quantity import _native
    from common.quantity.new_quantity_op import grouped_filter
    g = torch.Generator().manual_seed(C * 7 + K + G)
    Cg, Kg = C // G, K // G
    x = torch.randint(-128, 128, (2, C, 9, 8), generator=g).double()
    wq = torch.randint(-128, 128, (K, Cg, 3, 3), generator=g).float()
    ref = F.conv2d(x, wq.double(), None, stride, dil, dil, G)
    blocks = _legal_blocks(K, G)
    assert blocks
    for b in blocks:
        w = grouped_filter(wq, G, b)
        wb = _native.group_window(C, K, G, b)
        assert w.dtype == torch.int8 and tuple(w.shape) == (K, 3, 3, wb)
        for t in range(K // b):
            o = (t * b // Kg) * Cg
            assert o + wb <= C
            wt = w[t * b:(t + 1) * b].permute(0, 3, 1, 2).double()
            got = F.conv2d(x[:, o:o + wb], wt, None, stride, dil, dil)
            assert torch.equal(got, ref[:, t * b:(t + 1) * b]), (b, t)
        # the rows hold the group's weights and nothing else
        assert int((w != 0).sum()) == int((wq != 0).sum())


def test_grouped_fits_envelope():
    """Which layers NewConv2d routes to the grouped kernel, and the tile width it picks (fewest wasted operations, then
    the widest)."""
    from common.quantity.new_quantity_op import _group_block, _grouped_fits
    cases = [  # (cin, cout, k, stride, pad, groups) -> group_block or None
        ((128, 128, 3, 1, 1, 32), 32), ((256, 256, 3, 2, 1, 32), 32), ((1024, 1024, 3, 1, 1, 32), 32),
        ((64, 64, 3, 1, 1, 2), 32), ((64, 128, 1, 1, 0, 4), 32), ((32, 32, 3, 2, 1, 8), 32),
        ((64, 32, 3, 1, 2, 2), 32), ((256, 256, 3, 1, 1, 2), 128), ((512, 512, 3, 1, 1, 2), 256),
        ((64, 256, 3, 1, 1, 16), 128),          # Cg = 4, Kg = 16: Wb = 8 / 16 at 32 / 64 are not whole boxes
        ((32, 32, 3, 1, 1, 32), None),          # Cg == 1: depthwise / per-group routing
        ((16, 32, 3, 1, 1, 16), None),          # Cg == 1, channel multiplier 2
        ((48, 48, 3, 1, 1, 2), None),           # C % 32 != 0 on the im2col path
        ((48, 96, 1, 1, 0, 3), 32),             # 1x1 GEMM path: C % 16 == 0 is enough, Wb = 16
        ((96, 96, 3, 1, 1, 2), None),           # Kg = 48: no block divides or is a multiple of it
        ((64, 64, 1, 1, 0, 8), 32),             # 1x1 GEMM path: Wb = 32 / 16 boxes
    ]
    for (cin, cout, k, s, p, grp), want in cases:
        conv = nn.Conv2d(cin, cout, k, s, p, groups=grp)
        assert _grouped_fits(conv) == (want is not None), (cin, cout, k, grp)
        if want is not None:
            assert _group_block(conv) == want, (cin, cout, k, grp)


def test_bottleneck_defaults_unchanged():
    """ResNet-50 keeps its exact modules (the goldens depend on them); ResNeXt-50 32x4d has 16 grouped 3x3 layers of 32
    groups and torchvision's parameter count."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pytorch-quantity_b200"))
    from model.resnet import resnet50_fabu, resnext50_32x4d_fabu
    torch.manual_seed(0)
    r50 = resnet50_fabu()
    assert all(m.groups == 1 for m in r50.modules() if isinstance(m, nn.Conv2d))
    assert sum(p.numel() for p in r50.parameters()) == 25557032
    rx = resnext50_32x4d_fabu()
    grouped = [m for m in rx.modules() if isinstance(m, nn.Conv2d) and m.groups > 1]
    assert len(grouped) == 16 and all(m.groups == 32 and m.kernel_size == (3, 3) for m in grouped)
    assert sum(p.numel() for p in rx.parameters()) == 25028904


# ------------------------------------------------------------------------------------------ the exact reference
def right_shift(acc, rs):
    """new_quantity_op.py:11-44 on int64: round half away from zero for rs >= 1, else clamp then scale."""
    if rs >= 1:
        half = 1 << (rs - 1)
        r = torch.where(acc >= 0, (acc + half) >> rs, -((half - acc) >> rs))
    else:
        r = acc.clamp(-128, 127) << (-rs)
    return r.clamp(-128, 127)


def grouped_acc(xq, wq, stride, pad, dil, G):
    """int64 NCHW accumulators of int8 xq [N][C][H][W] with wq [K][Cg][R][S], groups G."""
    acc = F.conv2d(xq.double(), wq.double(), None, stride, pad, dil, G)
    assert acc.abs().max().item() < 2.0 ** 53 if acc.numel() else True
    return acc.round().long()


def epilogue_ref(acc, bias, rs, relu):
    y = (right_shift(acc, rs) + bias.long().view(1, -1, 1, 1)).clamp(-128, 127)
    return y.clamp(min=0) if relu else y


def config(K, RS, C, G, B, stride=(1, 1), pad=(0, 0)):
    """(BN, BK, STAGES, BSLOTS) of the gemm_s8_kernel pq_conv2d_s8 launches for a grouped layer (launch_bn)."""
    from common.quantity import _native
    wb = _native.group_window(C, K, G, B)
    plain = RS == (1, 1) and tuple(stride) == (1, 1) and tuple(pad) == (0, 0)
    if plain:
        bk = 128 if wb >= 128 else (64 if wb >= 64 else 32)
    else:
        bk = 128 if wb % 128 == 0 else (64 if wb % 64 == 0 else 32)
    num_kb = RS[0] * RS[1] * wb // bk
    if not plain and B == 64 and bk == 64 and K <= 64 and num_kb <= 9 and num_kb % 3 == 0:
        return (64, 64, 18, 9)                                   # short-K "deep A" configuration
    st = {256: {128: 4, 64: 8, 32: 9}, 128: {128: 6, 64: 9, 32: 9}, 64: {128: 8, 64: 9, 32: 9},
          32: {128: 8, 64: 9, 32: 9}}[B][bk]
    return (B, bk, st, st)


# (N, H, W, C, K, G, (R, S), stride, pad, dil, group_block)
SWEEP = [
    (2, 13, 11, 32, 32, 8, (3, 3), (1, 1), (1, 1), (1, 1), 32),        # Cg = Kg = 4, 8 groups per tile
    (2, 12, 12, 64, 64, 8, (3, 3), (2, 2), (1, 1), (1, 1), 32),        # Cg = Kg = 8, stride 2
    (1, 9, 10, 128, 128, 8, (5, 5), (1, 1), (2, 2), (1, 1), 32),       # Cg = Kg = 16, 5 x 5
    (2, 11, 9, 128, 128, 4, (3, 3), (1, 1), (2, 2), (2, 2), 32),       # Cg = Kg = 32, dilation 2
    (2, 11, 9, 128, 128, 4, (3, 3), (1, 1), (1, 1), (1, 1), 64),       # Cg = Kg = 32, two groups per tile
    (2, 10, 10, 128, 128, 2, (3, 3), (1, 1), (1, 1), (1, 1), 64),      # Cg = Kg = 64
    (2, 10, 10, 128, 128, 2, (3, 3), (2, 2), (1, 1), (1, 1), 32),      # Kg = 64 > block: two tiles per group
    (2, 10, 10, 128, 128, 2, (3, 3), (1, 1), (1, 1), (1, 1), 128),     # Wb = 128
    (2, 9, 9, 64, 128, 4, (1, 1), (1, 1), (0, 0), (1, 1), 32),         # 1x1 GEMM, Cg < Kg, Wb = 16
    (2, 9, 9, 64, 128, 4, (3, 3), (1, 1), (1, 1), (1, 1), 64),         # Cg < Kg, im2col
    (2, 9, 9, 128, 32, 4, (3, 3), (2, 2), (1, 1), (1, 1), 32),         # Cg > Kg, Wb = 128
    (3, 7, 9, 64, 64, 4, (1, 1), (1, 1), (0, 0), (1, 1), 32),          # 1x1 GEMM, Cg = Kg = 16, M % 128 != 0
    (2, 8, 8, 64, 64, 2, (3, 3), (1, 1), (1, 1), (1, 1), 64),          # one n tile: resident weights, deep A
    (2, 7, 7, 256, 256, 2, (3, 3), (1, 1), (1, 1), (1, 1), 256),       # BN = 256
    (2, 7, 7, 128, 512, 2, (1, 1), (2, 2), (0, 0), (1, 1), 256),       # 1x1 stride 2 (im2col), Wb = 64, BN = 256
    (2, 7, 7, 64, 512, 2, (3, 3), (1, 1), (1, 1), (1, 1), 256),        # Wb = 32, BN = 256
    (2, 7, 7, 64, 256, 2, (3, 3), (1, 1), (1, 1), (1, 1), 128),        # Wb = 32, BN = 128
    (2, 7, 7, 128, 256, 2, (3, 3), (1, 1), (1, 1), (1, 1), 128),       # Wb = 64, BN = 128
    (2, 7, 7, 64, 128, 2, (3, 3), (1, 1), (1, 1), (1, 1), 64),         # Wb = 32, BN = 64
    (2, 7, 7, 256, 128, 2, (3, 3), (1, 1), (1, 1), (1, 1), 64),        # Wb = 128, BN = 64
    (2, 7, 7, 128, 64, 2, (3, 3), (1, 1), (1, 1), (1, 1), 32),         # Wb = 64, BN = 32
    (2, 7, 7, 512, 256, 2, (3, 3), (1, 1), (1, 1), (1, 1), 256),       # Cg > Kg, Wb = 512 (four 128-byte blocks per tap)
]
# every kernel configuration the grouped path can select (BN = group_block, BK from Wb)
GROUPED_CONFIGS = {(32, 32, 9, 9), (32, 64, 9, 9), (32, 128, 8, 8), (64, 32, 9, 9), (64, 64, 9, 9), (64, 64, 18, 9),
                   (64, 128, 8, 8), (128, 32, 9, 9), (128, 64, 9, 9), (128, 128, 6, 6), (256, 32, 9, 9),
                   (256, 64, 8, 8), (256, 128, 4, 4)}


def _sentinel(nbytes, dev):
    return torch.full((nbytes + 2 * GUARD + 16,), 0x5A, dtype=torch.uint8, device=dev)


def call_conv(x_nhwc, w, bias_q, desc, flags, want_f32, want_s8, s8_offset=0, add=None):
    """pq_conv2d_s8 (pq_conv2d_s8_add when add is given) with each output in the middle of a sentinel buffer, the int8
    output s8_offset bytes past a 16-byte boundary.  Returns (rc, f32 NCHW, s8 NHWC); checks the guard bands, and that
    input and weights are unchanged."""
    from common.quantity import _native
    N, K, P, Q = desc.N, desc.K, desc.P, desc.Q
    dev = x_nhwc.device
    x0, w0 = x_nhwc.clone(), w.clone()
    bf = _sentinel(4 * N * K * P * Q, dev) if want_f32 else None
    bs = _sentinel(N * P * Q * K, dev) if want_s8 else None
    lo_s = GUARD + s8_offset
    stream = torch.cuda.current_stream().cuda_stream
    if add is None:
        rc = _native.lib().pq_conv2d_s8(x_nhwc.data_ptr(), w.data_ptr(), bias_q.data_ptr(), ctypes.byref(desc), flags,
                                        bf.data_ptr() + GUARD if want_f32 else None,
                                        bs.data_ptr() + lo_s if want_s8 else None, stream)
    else:
        ad = _native.AddDesc(add.data_ptr(), 0, 3, 0, 0, 3, None, bs.data_ptr() + lo_s)
        rc = _native.lib().pq_conv2d_s8_add(x_nhwc.data_ptr(), w.data_ptr(), bias_q.data_ptr(), ctypes.byref(desc),
                                            ctypes.byref(ad), flags, stream)
    torch.cuda.synchronize()
    out_f32 = out_s8 = None
    if bf is not None:
        assert bool((bf[:GUARD] == 0x5A).all()) and bool((bf[GUARD + 4 * N * K * P * Q:] == 0x5A).all()), "guard band"
    if bs is not None:
        assert bool((bs[:lo_s] == 0x5A).all()) and bool((bs[lo_s + N * P * Q * K:] == 0x5A).all()), "guard band"
    if rc == 0:
        if want_f32:
            out_f32 = bf[GUARD:GUARD + 4 * N * K * P * Q].view(torch.float32).view(N, K, P, Q)
        if want_s8:
            out_s8 = bs[lo_s:lo_s + N * P * Q * K].view(torch.int8).view(N, P, Q, K)
    else:                                          # a rejected call writes nothing
        for buf in (bf, bs):
            if buf is not None:
                assert bool((buf == 0x5A).all()), "a rejected call wrote its output"
    assert torch.equal(x_nhwc, x0) and torch.equal(w, w0), "input or weights modified"
    return rc, out_f32, out_s8


def make_desc(N, H, W, C, K, RS, stride, pad, dil, rs, ob, G, B):
    from common.quantity import _native
    return _native._conv_desc(N, H, W, C, K, RS, stride, pad, rs, ob, dil, G, B)


def operands(N, H, W, C, K, G, RS, seed):
    """int8 x [N][C][H][W], w [K][Cg][R][S] (per-channel magnitudes spread over 2^0..2^-7, channels 0..2 zero so that
    their output is the bias), bias [K] with -128, 127 and 5 on those channels."""
    g = torch.Generator().manual_seed(seed)
    R, S = RS
    x = torch.randint(-128, 128, (N, C, H, W), generator=g, dtype=torch.int32)
    w = torch.randint(-128, 128, (K, C // G, R, S), generator=g, dtype=torch.int32)
    w = w >> (torch.arange(K) % 8).view(K, 1, 1, 1)
    w[:3] = 0
    b = torch.randint(-128, 128, (K,), generator=g, dtype=torch.int32)
    b[:3] = torch.tensor([-128, 127, 5], dtype=torch.int32)
    return x.to(torch.int8).cuda(), w.to(torch.int8).cuda(), b.cuda()


def parse_instantiation(name):
    """(BN, BK, STAGES, ADDK, BSLOTS) of a gemm_s8_kernel name as the profiler prints it."""
    args = [re.sub(r"\((int|bool)\)", "", a).strip() for a in re.search(r"gemm_s8_kernel<([^>]*)>", name).group(1).split(",")]
    return tuple(1 if a == "true" else 0 if a == "false" else int(a) for a in args)


def _gemm_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return names, [parse_instantiation(n) for n in names if "gemm_s8_kernel" in n]


def test_sweep_covers_every_grouped_config():
    assert {config(c[4], c[6], c[3], c[5], c[10], c[7], c[8]) for c in SWEEP} == GROUPED_CONFIGS


@gpu
@pytest.mark.parametrize("case", SWEEP, ids=lambda c: "N%d_%dx%d_C%d_K%d_G%d_%dx%d_s%d_p%d_d%d_B%d" % (
    c[0], c[1], c[2], c[3], c[4], c[5], c[6][0], c[6][1], c[7][0], c[8][0], c[9][0], c[10]))
def test_grouped_kernel_sweep(case):
    from common.quantity import _native
    from common.quantity.new_quantity_op import grouped_filter
    N, H, W, C, K, G, RS, stride, pad, dil, B = case
    x, w, b = operands(N, H, W, C, K, G, RS, seed=C * 131 + K + H)
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    wg = grouped_filter(w, G, B)
    acc = grouped_acc(x, w, stride, pad, dil, G)
    i = 0
    for rs in RS_VALUES:
        for relu in (False, True):
            for folded in (False, True):
                ob = OB_VALUES[i % len(OB_VALUES)]
                outs = OUTPUTS[i % len(OUTPUTS)]
                i += 1
                bias_q = _native.bias_fold(b, rs) if folded else b
                flags = (_native.FLAG_RELU if relu else 0) | (_native.FLAG_BIAS_FOLDED if bias_q.numel() == 3 * K else 0)
                d = make_desc(N, H, W, C, K, RS, stride, pad, dil, rs, ob, G, B)
                rc, f32, s8 = call_conv(x_nhwc, wg, bias_q, d, flags, outs in ("f32", "both"), outs != "f32",
                                        s8_offset=1 if outs == "s8_unstaged" else 0)
                assert rc == 0, (rc, rs, ob)
                y = epilogue_ref(acc, b, rs, relu)
                lo = 0 if relu else -128
                # degenerate-case guard: interior values and both saturation values occur
                assert bool((y == 127).any()) and bool((y == lo).any()) and bool(((y > lo) & (y < 127)).any())
                what = "rs=%d ob=%d relu=%s folded=%s out=%s" % (rs, ob, relu, folded, outs)
                if f32 is not None:
                    assert torch.equal(f32, (y.double() * 2.0 ** -ob).float()), what
                if s8 is not None:
                    assert torch.equal(s8.permute(0, 3, 1, 2).long(), y), what
    # the instantiation this shape selects, and the wrapper's integers
    names, inst = _gemm_kernels(lambda: _native.conv2d_s8(x_nhwc, wg, _native.bias_fold(b, 7), stride, pad, 7, 2,
                                                          want_f32=False, want_s8=True, relu=True, dilation=dil,
                                                          groups=G, group_block=B))
    cfg = config(K, RS, C, G, B, stride, pad)
    assert inst == [(cfg[0], cfg[1], cfg[2], 0, cfg[3])], names
    f32, s8 = _native.conv2d_s8(x_nhwc, wg, _native.bias_fold(b, 7), stride, pad, 7, 2, want_f32=True, want_s8=True,
                                relu=True, dilation=dil, groups=G, group_block=B)
    y = epilogue_ref(acc, b, 7, True)
    assert torch.equal(s8.permute(0, 3, 1, 2).long(), y) and torch.equal(f32, (y.double() / 4).float())


@gpu
@pytest.mark.parametrize("B,RS", [(32, (3, 3)), (64, (3, 3)), (32, (1, 1))])
def test_grouped_single_group_input(B, RS):
    """Only one group's input channels are non-zero: every other group's output is its bias alone, so a tile that reads
    the wrong channel window is visible."""
    from common.quantity import _native
    from common.quantity.new_quantity_op import grouped_filter
    N, H, W, C, K, G = 2, 9, 9, 128, 128, 8                  # Cg = Kg = 16: two groups per 32-channel tile
    x, w, b = operands(N, H, W, C, K, G, RS, seed=77)
    w[:3] = 1
    pad = (RS[0] // 2, RS[1] // 2)
    for live in (0, 3, 5, 7):
        xs = torch.zeros_like(x)
        xs[:, live * 16:(live + 1) * 16] = x[:, live * 16:(live + 1) * 16]
        acc = grouped_acc(xs, w, (1, 1), pad, (1, 1), G)
        assert bool((acc[:, live * 16:(live + 1) * 16] != 0).any())
        d = make_desc(N, H, W, C, K, RS, (1, 1), pad, (1, 1), 4, 0, G, B)
        rc, f32, s8 = call_conv(xs.permute(0, 2, 3, 1).contiguous(), grouped_filter(w, G, B), b, d, 0, True, True)
        assert rc == 0
        y = epilogue_ref(acc, b, 4, False)
        assert torch.equal(s8.permute(0, 3, 1, 2).long(), y) and torch.equal(f32, y.float()), live


@gpu
def test_grouped_argument_limits():
    """Every descriptor that breaks a rule of the grouped layout returns the named error and writes nothing; the Python
    wrapper refuses tensors the kernel would misaddress."""
    from common.quantity import _native

    def run(C=64, K=64, G=2, B=32, RS=(3, 3), pad=(1, 1), wb=None, add=False):
        g = torch.Generator().manual_seed(5)
        x = torch.randint(-128, 128, (2, 6, 7, C), generator=g, dtype=torch.int32).to(torch.int8).cuda()
        if wb is None:
            wb = _native.group_window(C, K, G, B) if C % G == 0 and K % G == 0 and B > 0 else C
        w = torch.randint(-128, 128, (K, RS[0], RS[1], max(wb, 16)), generator=g, dtype=torch.int32)
        b = torch.randint(-128, 128, (K,), generator=g, dtype=torch.int32).cuda()
        d = make_desc(2, 6, 7, C, K, RS, (1, 1), pad, (1, 1), 7, 3, G, B)
        sc = torch.zeros((2, d.P, d.Q, K), dtype=torch.int8, device="cuda") if add else None
        return call_conv(x, w.to(torch.int8).cuda(), b, d, 0, not add, True, add=sc)[0]

    assert run() == 0
    assert run(C=96, K=64, G=3) == PQ_EINVAL                    # G does not divide K
    assert run(C=64, K=96, G=3) == PQ_EINVAL                    # G does not divide C
    assert run(G=-1) == PQ_EINVAL
    for B in (0, 16, 48, 512):
        assert run(B=B) == PQ_EUNSUPPORTED, B
    assert run(C=64, K=96, G=2, B=32) == PQ_EUNSUPPORTED        # Kg = 48: neither a multiple nor a divisor of 32
    assert run(C=96, K=96, G=3, B=64) == PQ_EUNSUPPORTED        # K % 64 != 0
    assert run(C=96, K=96, G=3, B=32) == 0
    assert run(C=64, K=128, G=4, B=32) == PQ_EUNSUPPORTED       # im2col: Wb = 16 is not a whole 32-byte box
    assert run(C=64, K=128, G=4, B=32, RS=(1, 1), pad=(0, 0)) == 0   # the 1x1 GEMM takes 16-byte boxes
    assert run(C=32, K=128, G=4, B=32, RS=(1, 1), pad=(0, 0)) == PQ_EUNSUPPORTED   # Wb = 8
    assert run(C=64, K=128, G=4, B=64) == 0
    assert run(C=64, K=64, G=2, B=32, RS=(1, 1), pad=(0, 0), add=True) == PQ_EUNSUPPORTED   # no fused add
    assert run(C=64, K=64, G=1, B=32, RS=(1, 1), pad=(0, 0), wb=64, add=True) == 0          # the dense layer fuses it
    assert run(G=0, wb=64) == 0 and run(G=1, B=48, wb=64) == 0                          # dense: group_block ignored
    # the wrapper
    x = torch.zeros((1, 4, 4, 64), dtype=torch.int8, device="cuda")
    w = torch.zeros((64, 3, 3, 32), dtype=torch.int8, device="cuda")
    b = torch.zeros(64, dtype=torch.int32, device="cuda")
    for args, kw in (((x.float(), w, b), {}), ((x, w.float(), b), {}), ((x, w, b.long()), {}),
                     ((x.transpose(1, 2), w, b), {}), ((x, w[..., :16], b), {}),
                     ((x, w, torch.zeros(40, dtype=torch.int32, device="cuda")), {}),
                     ((x, w, b), {"c_real": 60}), ((x, w, b), {"group_block": 64})):
        with pytest.raises(RuntimeError):
            _native.conv2d_s8(*args, (1, 1), (1, 1), 7, 3, groups=2, **dict({"group_block": 32}, **kw))
    _native.conv2d_s8(x, w, b, (1, 1), (1, 1), 7, 3, groups=2, group_block=32)


# ------------------------------------------------------------------------------------------ at size
# (input H = W, mid channels, stride) of the 16 grouped 3 x 3 layers of ResNeXt-50 32x4d at 224 x 224, distinct shapes
RESNEXT_GROUPED = [(56, 128, 1), (56, 256, 2), (28, 256, 1), (28, 512, 2), (14, 512, 1), (14, 1024, 2), (7, 1024, 1)]


@gpu
@pytest.mark.parametrize("shape", RESNEXT_GROUPED, ids=["%dx%d_c%d_s%d" % (s[0], s[0], s[1], s[2]) for s in RESNEXT_GROUPED])
def test_resnext50_grouped_at_batch_512_vs_exact_evaluation(shape):
    import common.quantity as cq
    hw, c, stride = shape
    G, batch = 32, 512
    g = torch.Generator(device="cuda").manual_seed(2000 + c + hw)
    x = torch.randn(batch, c, hw, hw, device="cuda", generator=g) * 2.0
    info = {"weight_bit": 8, "input_bit": 5, "output_bit": 4, "bias_bit": 4}
    rs = info["weight_bit"] + info["input_bit"] - info["output_bit"]
    conv = nn.Conv2d(c, c, 3, stride=stride, padding=1, groups=G).cuda()
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, device="cuda", generator=g) * 0.1)
        conv.bias.copy_(torch.randn(c, device="cuda", generator=g) * 2.0)
        wq = torch.clamp(torch.round(conv.weight * 2.0 ** info["weight_bit"]), -128, 127)
        bq = torch.clamp(torch.round(conv.bias * 2.0 ** info["bias_bit"]), -128, 127).long()
        m = cq.NewConv2d(conv, dict(info))
        assert m._group_block and m._group_convs is None
        got = m(x)                                               # fp32 NCHW (reference module boundary)
        m.int8_pipeline = True
        q8 = torch.relu(m(x)).int8_payload()                     # int8 NHWC, ReLU fused into the epilogue
        sat = 0
        for i in range(0, batch, 64):
            q = torch.clamp(torch.round(x[i:i + 64] * 2.0 ** info["input_bit"]), -128, 127)
            y = epilogue_ref(grouped_acc(q, wq, stride, 1, 1, G), bq, rs, False)
            assert torch.equal(got[i:i + 64], y.float() / 16.0), i
            assert torch.equal(q8[i:i + 64].permute(0, 3, 1, 2).long(), y.clamp_min(0)), i
            sat += int(((y == 127) | (y == -128)).sum())
    assert sat < 0.9 * got.numel(), "degenerate test: everything saturates"


# ------------------------------------------------------------------------------------------ NewConv2d routing
INFO = {"weight_bit": 7, "input_bit": 5, "output_bit": 4, "bias_bit": 5}


def _layer(cin, cout, k, stride, pad, dil, groups, seed):
    g = torch.Generator().manual_seed(seed)
    conv = nn.Conv2d(cin, cout, k, stride, pad, dil, groups, bias=True)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.3)
        conv.bias.copy_(torch.randn(cout, generator=g))
    return conv


@gpu
@pytest.mark.parametrize("cin,cout,k,stride,pad,dil,groups,grouped", [
    (128, 128, 3, 1, 1, 1, 32, True),         # ResNeXt-50 stage 1
    (256, 256, 3, 2, 1, 1, 32, True),         # stride 2
    (64, 128, 1, 1, 0, 1, 4, True),           # 1x1 GEMM path
    (64, 32, 3, 1, 2, 2, 2, True),            # dilation 2, Cg > Kg
    (64, 256, 3, 1, 1, 1, 16, True),          # Cg = 4, Kg = 16
    (32, 32, 3, 1, 1, 1, 32, False),          # Cg == 1: depthwise kernel
    (16, 32, 3, 1, 1, 1, 16, False),          # Cg == 1, channel multiplier 2: per-group path
    (48, 48, 3, 1, 1, 1, 2, False),           # C % 32 != 0: per-group path
    (96, 96, 3, 1, 1, 1, 2, False),           # Kg = 48: no legal tile width, per-group path
])
def test_newconv2d_grouped_routing(cin, cout, k, stride, pad, dil, groups, grouped):
    from oracle import pq_oracle as oracle
    from common.quantity import NewConv2d, QTensor, _native
    conv = _layer(cin, cout, k, stride, pad, dil, groups, seed=cin + k + groups)
    w, b = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = np.random.default_rng(cin + k).normal(0, 2, (2, cin, 15, 13)).astype(np.float32)
    ref, _ = oracle.int_conv_layer(x, w, b, INFO, stride=stride, padding=pad, dilation=dil, groups=groups)
    mod = NewConv2d(conv.cuda(), dict(INFO)).eval()
    depthwise = cin == cout == groups
    assert bool(mod._group_block) == grouped and mod._depthwise == depthwise
    assert (mod._group_convs is None) == (grouped or depthwise)
    xt = torch.from_numpy(x).cuda()
    with torch.no_grad():
        names, inst = _gemm_kernels(lambda: mod(xt))
        out = mod(xt)
    assert np.array_equal(out.cpu().numpy(), ref)
    if grouped:
        assert len(inst) == 1 and inst[0][0] == mod._group_block, names
        assert not any("dw_conv_s8_kernel" in n or "cat" in n.lower() for n in names), names
    elif depthwise:
        assert not inst
    else:
        assert len(inst) + sum("conv_rows_s8_kernel" in n for n in names) == groups     # one launch per group
    # int8 pipeline: a grouped layer hands out an int8 payload and a following ReLU runs in its epilogue
    mod.int8_pipeline = True
    relu0 = _native.LAUNCHES.get("relu_s8", 0)
    with torch.no_grad():
        q = mod(xt)
        assert isinstance(q, QTensor) == (grouped or depthwise)
        assert np.array_equal((q.dequantize() if isinstance(q, QTensor) else q).cpu().numpy(), ref)
        qr = F.relu(mod(xt))
        got = qr.dequantize() if isinstance(qr, QTensor) else qr
        assert np.array_equal(got.cpu().numpy(), np.maximum(ref, 0))
    if grouped:
        assert _native.LAUNCHES.get("relu_s8", 0) == relu0


@gpu
def test_intsim_ext_grouped_cases_take_the_grouped_kernel():
    """The grouped cases of the reference-parity goldens (test_newconv2d_dilation_and_groups_vs_golden) now run on the
    grouped kernel, so that test pins the grouped path against the reference's own outputs."""
    from golden import gen_golden as gg
    import common.quantity as cq
    names = {"groups2", "groups4_1x1", "groups8_cg4", "groups2_dil2"}
    seen = set()
    for case in gg.INTSIM_EXT_CASES:
        name, B, Cin, H, W, Cout, k, stride, pad, dil, groups = case[:11]
        if name not in names:
            continue
        _, w, b, info = gg.intsim_ext_tensors(case)
        conv = nn.Conv2d(Cin, Cout, k, stride=stride, padding=pad, dilation=dil, groups=groups)
        m = cq.NewConv2d(conv.cuda(), dict(info))
        assert m._group_block and m._group_convs is None, name
        seen.add(name)
    assert seen == names


@gpu
def test_newconv2d_grouped_pickled_before_kernel_keeps_group_path(tmp_path):
    """A NewConv2d pickled before the grouped kernel existed has _group_convs and no _group_block attribute: it still runs
    its per-group path, with the same result."""
    from oracle import pq_oracle as oracle
    from common.quantity import NewConv2d
    conv = _layer(64, 64, 3, 1, 1, 1, 4, seed=3)
    w, b = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = np.random.default_rng(3).normal(0, 2, (2, 64, 9, 9)).astype(np.float32)
    ref, _ = oracle.int_conv_layer(x, w, b, INFO, stride=1, padding=1, groups=4)
    mod = NewConv2d(conv.cuda(), dict(INFO))
    del mod._group_block, mod._w_krsc
    mod._payload_channels = None
    mod._build_groups(mod.Conv, mod.Conv.weight.detach())
    torch.save(mod, tmp_path / "m.pt")
    mod = torch.load(tmp_path / "m.pt", weights_only=False)
    assert mod._group_block == 0 and "_group_block" not in mod.__dict__
    with torch.no_grad():
        names, inst = _gemm_kernels(lambda: mod(torch.from_numpy(x).cuda()))
        out = mod(torch.from_numpy(x).cuda())
    assert len(inst) == 4
    assert np.array_equal(out.cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------ ResNeXt-50 end to end
def _resnext_recon(tmp_path, in_hw, batch):
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(os.path.dirname(here), "pytorch-quantity_b200", "test"))
    import _models
    import tools
    from common.quantity import merge_bn
    from model.resnet.resnet_fabu import randomize_bn_, resnext50_32x4d_fabu

    def build():
        torch.manual_seed(0)
        net = resnext50_32x4d_fabu(in_hw=in_hw).eval()
        with torch.no_grad():
            randomize_bn_(net, 0)
        return net

    cfg, user = _models.configs(str(tmp_path / "wd"), (3, in_hw, in_hw), 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build(), "cpu"), config=cfg, user_config=user, verbose=False)
        cal = [(torch.randn(batch, 3, in_hw, in_hw, generator=torch.Generator().manual_seed(1 + i)), None)
               for i in range(2)]
        q.activation_quantize(cal)
        q.weight_quantize()
        r = tools.Reconstruction(build(), config=cfg)
        r.merge_bn()
        return r.ReconModel(r.get_quantity_information(), None).cuda().eval()


def _info(m):
    return {"weight_bit": m.weight_bit, "bias_bit": m.bias_bit, "input_bit": m.input_bit, "output_bit": m.output_bit}


@gpu
@pytest.mark.parametrize("in_hw,batch", [(64, 2), (224, 1)])
def test_resnext50_end_to_end(tmp_path, monkeypatch, in_hw, batch):
    from oracle import pq_oracle as oracle
    from common.quantity import GraphedForward, NewConv2d, NewLinear, QTensor, _native, enable_int8_pipeline, int8_pipeline
    model = _resnext_recon(tmp_path, in_hw, batch)
    convs = {n: m for n, m in model.named_modules() if isinstance(m, NewConv2d)}
    grouped = {n for n, m in convs.items() if m.Conv.groups > 1}
    assert len(grouped) == 16 and all(convs[n]._group_block and convs[n]._group_convs is None for n in grouped)
    x = torch.randn(batch, 3, in_hw, in_hw, generator=torch.Generator().manual_seed(42)).cuda()
    seen = {}
    hooks = [m.register_forward_hook(lambda m, i, o, n=n: seen.__setitem__(n, (i[0].detach().cpu().numpy(),
                                                                              o.detach().cpu().numpy())))
             for n, m in model.named_modules() if isinstance(m, (NewConv2d, NewLinear))]
    g0 = _native.LAUNCHES.get("conv_s8", 0)
    with torch.no_grad():
        ref = model(x)
    for h in hooks:
        h.remove()
    assert _native.LAUNCHES.get("conv_s8", 0) - g0 <= len(convs)      # no per-group launches
    assert len(seen) == len(convs) + 1
    # every layer equals the oracle on the input it received
    for n, (xi, yo) in seen.items():
        m = dict(model.named_modules())[n]
        info = _info(m)
        if isinstance(m, NewConv2d):
            c = m.Conv
            w = c.weight.detach().double().cpu().numpy() * 2.0 ** -m.weight_bit
            b = m.quantized_bias.double().cpu().numpy() * 2.0 ** -m.bias_bit
            exp, _ = oracle.int_conv_layer(xi, w.astype(np.float32), b.astype(np.float32), info, stride=c.stride,
                                           padding=c.padding, dilation=c.dilation, groups=c.groups)
        else:
            w = m.Linear.weight.detach().double().cpu().numpy() * 2.0 ** -m.weight_bit
            b = m.quantized_bias.double().cpu().numpy() * 2.0 ** -m.bias_bit
            exp, _ = oracle.int_linear_layer(xi, w.astype(np.float32), b.astype(np.float32), info)
        assert np.array_equal(yo, exp), n

    # int8 pipeline: same logits, and no grouped layer quantises from fp32 -- each reads its producer's int8 payload
    enable_int8_pipeline(model)
    name_of = {id(m): n for n, m in convs.items()}
    in_bits = {}
    conv_forward = int8_pipeline.conv_forward

    def recording_conv_forward(mod, xin):
        in_bits[name_of[id(mod)]] = ((xin.q8_bit if xin._lazy_cat is None else None) if isinstance(xin, QTensor)
                                     else "fp32")
        return conv_forward(mod, xin)
    monkeypatch.setattr(int8_pipeline, "conv_forward", recording_conv_forward)
    quantized = []
    for n, m in convs.items():
        m._quantize = (lambda x, n=n, f=m._quantize: (quantized.append(n), f(x))[1])
    with torch.no_grad():
        out = model(x)
    for m in convs.values():
        del m.__dict__["_quantize"]
    assert torch.equal(out, ref)
    assert not grouped & set(quantized), sorted(grouped & set(quantized))
    assert all(in_bits[n] == convs[n].input_bit for n in grouped)
    fwd = GraphedForward(model, x)
    assert torch.equal(fwd(x), ref)
    enable_int8_pipeline(model, False)

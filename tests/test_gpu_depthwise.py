"""The depthwise convolution (pq_conv2d_dw_s8 and NewConv2d's depthwise path) against an evaluation that shares nothing
with the kernel:

    acc = float64 F.conv2d(..., groups=C) of the int8 operands on the GPU, rounded to int64      exact: |acc| < 2^53
    y   = clamp(clamp(RightShift(acc, rs)) + b) [ReLU], fp32 = y / 2^ob                          new_quantity_op.py:11-44,124-133

Every kernel output is written into the middle of a sentinel-filled buffer; the bytes around it, the input and the
weights must survive.  The layer tests compare with the CPU oracle (oracle.int_conv_layer / int_linear_layer).
"""
import ctypes
import os
import re
import shutil
import subprocess
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
OUTPUTS = ("f32", "s8", "both")
GUARD = 4096                      # sentinel bytes before and after every output


def instantiation(C, RS):
    """(G, KS) of the dw_conv_s8_kernel<G, KS> that pq_conv2d_dw_s8 launches for C padded channels and an R x S filter:
    16-channel groups per CTA, and the unrolled square filter size (0: runtime tap loops)."""
    G = 4 if C % 64 == 0 else (2 if C % 32 == 0 else 1)
    return G, (RS[0] if RS[0] == RS[1] and RS[0] in (3, 5) else 0)


# (C padded, K real, (R, S), stride, pad, dilation, (H, W), N)
SWEEP = [
    (16, 16, (3, 3), (1, 1), (1, 1), (1, 1), (13, 17), 2),
    (32, 24, (3, 3), (2, 2), (1, 0), (1, 1), (13, 17), 3),       # K % 16 != 0 (MobileNetV2's 24 channels)
    (32, 32, (5, 5), (1, 2), (2, 4), (1, 1), (7, 7), 1),         # pad up to the maximum in w only
    (144, 144, (3, 3), (2, 2), (0, 4), (2, 2), (13, 17), 2),     # dilation 2, maximum pad in w
    (144, 144, (3, 5), (1, 2), (2, 3), (1, 1), (13, 17), 2),     # non-square filter
    (960, 960, (3, 3), (1, 1), (1, 1), (1, 1), (7, 7), 2),
    (32, 32, (3, 3), (1, 1), (2, 2), (1, 1), (1, 1), 3),         # 1 x 1 image, maximum pad
    (16, 16, (5, 5), (2, 1), (8, 7), (2, 2), (1, 1), 2),         # 1 x 1 image, dilated maximum pad
    (96, 96, (3, 3), (2, 2), (1, 1), (1, 1), (112, 112), 1),
    (32, 32, (7, 7), (2, 1), (3, 6), (1, 1), (13, 17), 1),       # 7 x 7
    (64, 64, (3, 3), (1, 1), (1, 1), (1, 1), (56, 56), 64),      # many waves of CTAs
    (144, 130, (3, 3), (1, 1), (1, 1), (2, 1), (13, 17), 2),     # K % 16 != 0 across several groups
    (64, 64, (5, 5), (2, 2), (2, 1), (1, 1), (13, 17), 2),
    (128, 120, (7, 5), (1, 2), (6, 2), (1, 1), (9, 11), 2),      # non-square, K % 16 != 0
]


# ------------------------------------------------------------------------------------------ the exact reference
def right_shift(acc, rs):
    """new_quantity_op.py:11-44 on int64: round half away from zero for rs >= 1, else clamp then scale."""
    if rs >= 1:
        half = 1 << (rs - 1)
        r = torch.where(acc >= 0, (acc + half) >> rs, -((half - acc) >> rs))
    else:
        r = acc.clamp(-128, 127) << (-rs)
    return r.clamp(-128, 127)


def dw_acc(xq, wq, stride, pad, dil):
    """int64 NCHW accumulators of the depthwise convolution of int8 xq [N][K][H][W] with wq [K][R][S]."""
    K = wq.shape[0]
    acc = F.conv2d(xq.double(), wq.double().unsqueeze(1), None, stride, pad, dil, K)
    assert acc.abs().max().item() < 2.0 ** 53 if acc.numel() else True
    return acc.round().long()


def epilogue_ref(acc, bias, rs, relu):
    y = (right_shift(acc, rs) + bias.long().view(1, -1, 1, 1)).clamp(-128, 127)
    return y.clamp(min=0) if relu else y


# ------------------------------------------------------------------------------------------ the raw entry point
def _sentinel(nbytes, dev):
    return torch.full((nbytes + 2 * GUARD,), 0x5A, dtype=torch.uint8, device=dev)


def call_dw(x_nhwc, w_rsc, bias_q, desc, flags, want_f32, want_s8):
    """pq_conv2d_dw_s8 with each output in the middle of a sentinel buffer.  Returns (rc, f32 NCHW, s8 NHWC); checks the
    guard bands, and that input and weights are unchanged."""
    from common.quantity import _native
    N, K, P, Q = desc.N, desc.K, desc.P, desc.Q
    dev = x_nhwc.device
    x0, w0 = x_nhwc.clone(), w_rsc.clone()
    bf = _sentinel(4 * N * K * P * Q, dev) if want_f32 else None
    bs = _sentinel(N * P * Q * K, dev) if want_s8 else None
    rc = _native.lib().pq_conv2d_dw_s8(x_nhwc.data_ptr(), w_rsc.data_ptr(), bias_q.data_ptr(), ctypes.byref(desc), flags,
                                      bf.data_ptr() + GUARD if want_f32 else None,
                                      bs.data_ptr() + GUARD if want_s8 else None,
                                      torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out_f32 = out_s8 = None
    for buf in (bf, bs):
        if buf is not None:
            assert bool((buf[:GUARD] == 0x5A).all()) and bool((buf[-GUARD:] == 0x5A).all()), "guard band overwritten"
    if rc == 0:
        if want_f32:
            out_f32 = bf[GUARD:-GUARD].view(torch.float32).view(N, K, P, Q)
        if want_s8:
            out_s8 = bs[GUARD:-GUARD].view(torch.int8).view(N, P, Q, K)
    else:                                          # a rejected call writes nothing
        for buf in (bf, bs):
            if buf is not None:
                assert bool((buf == 0x5A).all()), "a rejected call wrote its output"
    assert torch.equal(x_nhwc, x0) and torch.equal(w_rsc, w0), "input or weights modified"
    return rc, out_f32, out_s8


def make_desc(N, H, W, C, K, RS, stride, pad, dil, rs, ob):
    from common.quantity import _native
    return _native._conv_desc(N, H, W, C, K, RS, stride, pad, rs, ob, dil)


def operands(C, K, RS, H, W, N, seed):
    """int8 x [N][K][H][W], w [K][R][S] (per-channel magnitudes spread over 2^0..2^-7, channels 0..2 zero so that
    their output is the bias), bias [K] with -128, 127 and 5 on those channels; plus the padded NHWC / RSC forms."""
    g = torch.Generator().manual_seed(seed)
    R, S = RS
    x = torch.randint(-128, 128, (N, K, H, W), generator=g, dtype=torch.int32)
    w = torch.randint(-128, 128, (K, R, S), generator=g, dtype=torch.int32)
    w = w >> (torch.arange(K) % 8).view(K, 1, 1)
    w[:3] = 0
    b = torch.randint(-128, 128, (K,), generator=g, dtype=torch.int32)
    b[:3] = torch.tensor([-128, 127, 5], dtype=torch.int32)
    x, w, b = x.to(torch.int8).cuda(), w.to(torch.int8).cuda(), b.cuda()
    x_nhwc = torch.zeros((N, H, W, C), dtype=torch.int8, device="cuda")
    x_nhwc[..., :K] = x.permute(0, 2, 3, 1)
    w_rsc = torch.zeros((R, S, C), dtype=torch.int8, device="cuda")
    w_rsc[..., :K] = w.permute(1, 2, 0)
    return x, w, b, x_nhwc.contiguous(), w_rsc.contiguous()


@gpu
@pytest.mark.parametrize("case", SWEEP, ids=lambda c: "C%d_K%d_%dx%d_s%d%d_p%d%d_d%d%d_%dx%d_N%d" % (
    c[0], c[1], c[2][0], c[2][1], c[3][0], c[3][1], c[4][0], c[4][1], c[5][0], c[5][1], c[6][0], c[6][1], c[7]))
def test_dw_kernel_sweep(case):
    from common.quantity import _native
    C, K, RS, stride, pad, dil, (H, W), N = case
    x, w, b, x_nhwc, w_rsc = operands(C, K, RS, H, W, N, seed=C * 131 + H)
    acc = dw_acc(x, w, stride, pad, dil)
    i = 0
    for rs in RS_VALUES:
        for relu in (False, True):
            for folded in (False, True):
                ob = OB_VALUES[i % len(OB_VALUES)]
                outs = OUTPUTS[i % len(OUTPUTS)] if i % 11 else "both"
                i += 1
                bias_q = _native.bias_fold(b, rs) if folded else b
                flags = (_native.FLAG_RELU if relu else 0) | (_native.FLAG_BIAS_FOLDED if bias_q.numel() == 3 * K else 0)
                d = make_desc(N, H, W, C, K, RS, stride, pad, dil, rs, ob)
                rc, f32, s8 = call_dw(x_nhwc, w_rsc, bias_q, d, flags, outs != "s8", outs != "f32")
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
    # the wrapper returns the same integers
    f32, s8 = _native.conv2d_dw_s8(x_nhwc, w_rsc, _native.bias_fold(b, 7), stride, pad, 7, 2, want_f32=True,
                                   want_s8=True, relu=True, dilation=dil, channels=K)
    y = epilogue_ref(acc, b, 7, True)
    assert torch.equal(s8.permute(0, 3, 1, 2).long(), y) and torch.equal(f32, (y.double() / 4).float())


def _tie_targets(taps):
    """(rs, accumulator) pairs exactly at (j + 1/2) * 2^rs near zero and around both saturation edges, for every rs whose
    tie points a sum of `taps` int8 products can reach."""
    amax = (taps - 1) * 16256 + 127
    out = []
    for rs in range(1, 25):
        for j in (-131, -130, -129, -128, -127, -2, -1, 0, 1, 126, 127, 128):
            a = (2 * j + 1) << (rs - 1)
            if abs(a) <= amax:
                out.append((rs, a))
    return out


def _factor(a, taps):
    """int8 (x, w) per tap with sum x * w == a: w = -128 on all taps but the last (w = 1)."""
    xs, ws = [], []
    rem = a
    for _ in range(taps - 1):
        q = max(-128, min(127, int(round(rem / -128.0))))
        xs.append(q); ws.append(-128)
        rem -= q * -128
    assert -128 <= rem <= 127, (a, rem)
    xs.append(rem); ws.append(1)
    return xs, ws


@gpu
def test_dw_crafted_ties():
    """Accumulators exactly on the rounding ties, near zero and at both saturation edges, for every reachable rs, with
    biases -128, -1, 0 and 127, through the plain and the folded epilogue, with and without ReLU."""
    from common.quantity import _native
    R = S = 7
    taps = R * S
    by_rs = {}
    for rs, a in _tie_targets(taps):
        by_rs.setdefault(rs, []).append(a)
    assert max(by_rs) >= 19 and min(by_rs) == 1
    for rs, targets in sorted(by_rs.items()):
        chans = [(a, bv) for a in targets for bv in (-128, -1, 0, 127)]
        K = (len(chans) + 15) // 16 * 16
        chans += [(0, 0)] * (K - len(chans))
        x = torch.zeros((1, K, R, S), dtype=torch.int8)
        w = torch.zeros((K, R, S), dtype=torch.int8)
        for c, (a, _) in enumerate(chans):
            xs, ws = _factor(a, taps)
            x[0, c] = torch.tensor(xs, dtype=torch.int8).view(R, S)
            w[c] = torch.tensor(ws, dtype=torch.int8).view(R, S)
        b = torch.tensor([bv for _, bv in chans], dtype=torch.int32).cuda()
        x, w = x.cuda(), w.cuda()
        acc = dw_acc(x, w, (1, 1), (0, 0), (1, 1))
        assert acc.view(-1).tolist() == [a for a, _ in chans]
        x_nhwc, w_rsc = x.permute(0, 2, 3, 1).contiguous(), w.permute(1, 2, 0).contiguous()
        for relu in (False, True):
            for folded in (False, True):
                bias_q = _native.bias_fold(b, rs) if folded else b
                flags = (_native.FLAG_RELU if relu else 0) | (_native.FLAG_BIAS_FOLDED if bias_q.numel() == 3 * K else 0)
                d = make_desc(1, R, S, K, K, (R, S), (1, 1), (0, 0), (1, 1), rs, 3)
                rc, f32, s8 = call_dw(x_nhwc, w_rsc, bias_q, d, flags, True, True)
                assert rc == 0
                y = epilogue_ref(acc, b, rs, relu)
                assert torch.equal(s8.permute(0, 3, 1, 2).long(), y), (rs, relu, folded)
                assert torch.equal(f32, (y.double() / 8).float()), (rs, relu, folded)


@gpu
def test_dw_argument_limits():
    """One step past each limit is rejected and writes nothing; one step inside is accepted."""
    from common.quantity import _native

    def run(C=32, K=32, RS=(3, 3), stride=(1, 1), pad=(1, 1), dil=(1, 1), rs=7, ob=3, H=9, W=10):
        g = torch.Generator().manual_seed(5)
        x = torch.randint(-128, 128, (2, H, W, C), generator=g, dtype=torch.int32).to(torch.int8).cuda()
        w = torch.randint(-128, 128, (RS[0], RS[1], C), generator=g, dtype=torch.int32).to(torch.int8).cuda()
        b = torch.randint(-128, 128, (K,), generator=g, dtype=torch.int32).cuda()
        d = make_desc(2, H, W, C, K, RS, stride, pad, dil, rs, ob)
        return call_dw(x, w, b, d, 0, True, True)[0]

    for bad, good in ((dict(rs=25), dict(rs=24)), (dict(rs=-25), dict(rs=-24)), (dict(ob=101), dict(ob=100)),
                      (dict(ob=-101), dict(ob=-100)),
                      (dict(RS=(8, 3), pad=(0, 1)), dict(RS=(7, 3), pad=(0, 1))),
                      (dict(RS=(3, 8), pad=(1, 0)), dict(RS=(3, 7), pad=(1, 0))),
                      (dict(stride=(3, 1)), dict(stride=(2, 1))), (dict(stride=(1, 3)), dict(stride=(1, 2))),
                      (dict(dil=(3, 1)), dict(dil=(2, 1))), (dict(dil=(1, 3)), dict(dil=(1, 2))),
                      (dict(pad=(3, 1)), dict(pad=(2, 1))), (dict(pad=(1, 5), dil=(1, 2)), dict(pad=(1, 4), dil=(1, 2))),
                      (dict(C=24, K=24), dict(C=32, K=24)), (dict(C=8, K=8), dict(C=16, K=8))):
        assert run(**bad) == PQ_EUNSUPPORTED, bad
        assert run(**good) == 0, good
    assert run(C=32, K=33) == PQ_EINVAL
    assert run(C=32, K=32) == 0
    # the Python wrapper refuses tensors the kernel would misaddress before the call
    x = torch.zeros((1, 4, 4, 32), dtype=torch.int8, device="cuda")
    w = torch.zeros((3, 3, 32), dtype=torch.int8, device="cuda")
    b = torch.zeros(32, dtype=torch.int32, device="cuda")
    for args in ((x.float(), w, b), (x, w.float(), b), (x, w, b.long()), (x.transpose(1, 2), w, b),
                 (x, w[..., :16], b), (x, w, torch.zeros(40, dtype=torch.int32, device="cuda"))):
        with pytest.raises(RuntimeError):
            _native.conv2d_dw_s8(*args, (1, 1), (1, 1), 7, 3)


def test_dw_instantiations_match_table():
    """The dw_conv_s8_kernel instantiations of the built library are exactly the (G, KS) pairs SWEEP reaches."""
    from common.quantity import _native
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not installed")
    if not os.path.exists(_native.LIB_PATH):
        pytest.skip("library not built")
    sym = subprocess.run(["cuobjdump", "-symbols", _native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = subprocess.run(["cu++filt"], input=sym, check=True, capture_output=True, text=True).stdout
    found = {tuple(int(a) for a in re.sub(r"\(int\)", "", m.group(1)).split(",")) for line in names.splitlines()
             if "STO_ENTRY" in line for m in [re.search(r"dw_conv_s8_kernel<([^>]*)>", line)] if m}
    assert found == {(g, ks) for g in (1, 2, 4) for ks in (0, 3, 5)}
    assert {instantiation(c[0], c[2]) for c in SWEEP} == found


# ------------------------------------------------------------------------------------------ NewConv2d
INFO = {"weight_bit": 7, "input_bit": 5, "output_bit": 4, "bias_bit": 5}


def _layer(cin, cout, k, stride, pad, dil, groups, seed):
    g = torch.Generator().manual_seed(seed)
    conv = nn.Conv2d(cin, cout, k, stride, pad, dil, groups, bias=True)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.3)
        conv.bias.copy_(torch.randn(cout, generator=g))
    return conv


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@gpu
@pytest.mark.parametrize("cin,cout,k,stride,pad,dil,groups,dw", [
    (144, 144, 3, 2, 1, 1, 144, True),
    (24, 24, 5, 1, 2, 1, 24, True),
    (32, 32, 3, 1, 2, 2, 32, True),
    (16, 32, 3, 1, 1, 1, 16, False),          # channel multiplier 2: per-group path
    (16, 16, 9, 1, 4, 1, 16, False),          # R > 7: per-group path
    (16, 16, 3, 3, 1, 1, 16, False),          # stride 3: per-group path
])
def test_newconv2d_depthwise_routing(cin, cout, k, stride, pad, dil, groups, dw):
    from oracle import pq_oracle as oracle
    from common.quantity import NewConv2d, QTensor
    conv = _layer(cin, cout, k, stride, pad, dil, groups, seed=cin + k)
    w, b = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = np.random.default_rng(cin + k).normal(0, 2, (2, cin, 15, 13)).astype(np.float32)
    ref, y = oracle.int_conv_layer(x, w, b, INFO, stride=stride, padding=pad, dilation=dil, groups=groups)
    mod = NewConv2d(conv.cuda(), dict(INFO)).eval()
    assert mod._depthwise == dw and (mod._group_convs is None) == dw
    xt = torch.from_numpy(x).cuda()
    with torch.no_grad():
        names = _kernels(lambda: mod(xt))
        out = mod(xt)
    assert np.array_equal(out.cpu().numpy(), ref)
    n_dw = sum("dw_conv_s8_kernel" in n for n in names)
    if dw:
        assert n_dw == 1 and not any("gemm_s8_kernel" in n or "conv_rows_s8_kernel" in n for n in names), names
    else:
        assert n_dw == 0
    # int8 pipeline: a depthwise layer hands out an int8 payload and a following ReLU runs in its epilogue; the per-group
    # path keeps returning fp32
    mod.int8_pipeline = True
    with torch.no_grad():
        q = mod(xt)
        assert isinstance(q, QTensor) == dw
        assert np.array_equal((q.dequantize() if dw else q).cpu().numpy(), ref)
        qr = F.relu(mod(xt))
        assert np.array_equal((qr.dequantize() if dw else qr).cpu().numpy(), np.maximum(ref, 0))


@gpu
def test_newconv2d_depthwise_pickled_before_kernel_keeps_group_path():
    """A NewConv2d pickled before the depthwise kernel existed has _group_convs and no _depthwise attribute: it still runs
    its per-group path, with the same result."""
    from oracle import pq_oracle as oracle
    from common.quantity import NewConv2d
    conv = _layer(16, 16, 3, 1, 1, 1, 16, seed=3)
    w, b = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = np.random.default_rng(3).normal(0, 2, (2, 16, 9, 9)).astype(np.float32)
    ref, _ = oracle.int_conv_layer(x, w, b, INFO, stride=1, padding=1, groups=16)
    mod = NewConv2d(conv.cuda(), dict(INFO))
    del mod._depthwise, mod._w_rsc
    mod._payload_channels = None
    mod._build_groups(mod.Conv, mod.Conv.weight.detach())
    assert not mod._depthwise
    with torch.no_grad():
        names = _kernels(lambda: mod(torch.from_numpy(x).cuda()))
        out = mod(torch.from_numpy(x).cuda())
    assert not any("dw_conv_s8_kernel" in n for n in names)
    assert np.array_equal(out.cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------ MobileNetV2
def _mobilenet_recon(tmp_path, in_hw, batch):
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(os.path.dirname(here), "pytorch-quantity_b200", "test"))
    import _models
    import tools
    from common.quantity import merge_bn
    from model.mobilenet import mobilenetv2_fabu
    from model.resnet.resnet_fabu import randomize_bn_

    def build():
        torch.manual_seed(0)
        net = mobilenetv2_fabu(in_hw=in_hw).eval()
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
def test_mobilenetv2_end_to_end(tmp_path, monkeypatch, in_hw, batch):
    from oracle import pq_oracle as oracle
    from common.quantity import GraphedForward, NewConv2d, NewLinear, enable_int8_pipeline
    model = _mobilenet_recon(tmp_path, in_hw, batch)
    convs = {n: m for n, m in model.named_modules() if isinstance(m, NewConv2d)}
    dws = {n for n, m in convs.items() if m.Conv.groups > 1}
    assert len(dws) == 17 and all(convs[n]._depthwise for n in dws)
    x = torch.randn(batch, 3, in_hw, in_hw, generator=torch.Generator().manual_seed(42)).cuda()
    seen = {}
    hooks = [m.register_forward_hook(lambda m, i, o, n=n: seen.__setitem__(n, (i[0].detach().cpu().numpy(),
                                                                              o.detach().cpu().numpy())))
             for n, m in model.named_modules() if isinstance(m, (NewConv2d, NewLinear))]
    with torch.no_grad():
        ref = model(x)
    for h in hooks:
        h.remove()
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

    # int8 pipeline: same logits.  A convolution quantises from fp32 only where its input has no int8 payload it can read:
    # the stem (the image), the consumers of the 24-channel tensors (payload channels != 24 padded to 32), layers whose
    # input_bit differs from the bit of their producer's payload, and the consumers of residual adds that the add kernel
    # declined (operand bits outside its range, or an operand already fp32), which hand over fp32.  Never a depthwise
    # layer: each takes its producer's int8 payload.
    from common.quantity import QTensor, int8_pipeline
    enable_int8_pipeline(model)
    name_of = {id(m): n for n, m in convs.items()}
    in_bits = {}
    conv_forward = int8_pipeline.conv_forward

    def recording_conv_forward(mod, xin):
        in_bits[name_of[id(mod)]] = ((xin.q8_bit if xin._lazy_cat is None else None) if isinstance(xin, QTensor)
                                     else "fp32")
        return conv_forward(mod, xin)
    monkeypatch.setattr(int8_pipeline, "conv_forward", recording_conv_forward)
    add_forward, declined_adds = int8_pipeline.add_forward, []

    def recording_add_forward(mod, a, b):
        out = add_forward(mod, a, b)
        if out is None:
            declined_adds.append(tuple(t.exact_bit() if isinstance(t, QTensor) else "fp32" for t in (a, b)))
        return out
    monkeypatch.setattr(int8_pipeline, "add_forward", recording_add_forward)
    quantized = []
    for n, m in convs.items():
        m._quantize = (lambda x, n=n, f=m._quantize: (quantized.append(n), f(x))[1])
    from common.quantity import _native
    relu0 = _native.LAUNCHES.get("relu_s8", 0)
    dw0 = _native.LAUNCHES.get("conv_dw_s8", 0)
    with torch.no_grad():
        out = model(x)
    for m in convs.values():
        del m.__dict__["_quantize"]
    assert torch.equal(out, ref)
    assert _native.LAUNCHES.get("conv_dw_s8", 0) - dw0 == 17
    assert _native.LAUNCHES.get("relu_s8", 0) == relu0          # every ReLU ran inside its convolution
    c24 = {n for n, m in convs.items() if m.Conv.in_channels == 24}
    other_bit = {n for n, b in in_bits.items() if b not in (None, "fp32") and b != convs[n].input_bit}
    fp32_in = {n for n, b in in_bits.items() if b == "fp32"}
    assert len(c24) == 2 and "features.0" in fp32_in
    assert set(quantized) == fp32_in | c24 | other_bit, (sorted(quantized), sorted(other_bit), sorted(fp32_in))
    assert not dws & set(quantized) and not dws & fp32_in
    assert all(in_bits[n] == convs[n].input_bit for n in dws)
    assert all(convs[n].Conv.kernel_size == (1, 1) for n in (fp32_in | other_bit) - {"features.0"})
    assert bool(declined_adds) == bool(fp32_in - {"features.0"}), declined_adds
    fwd = GraphedForward(model, x)
    assert torch.equal(fwd(x), ref)
    enable_int8_pipeline(model, False)

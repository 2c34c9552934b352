"""GPU parity of the integer simulation (ReconModel): tcgen05 int8 GEMM / implicit-GEMM conv with
the fused shift-round-saturate-bias epilogue, through the C ABI, against the reference's golden
outputs (tests/golden/intsim.npz, tiny_e2e.npz) and the oracle.  Bit-exact."""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

import det_inputs
from conftest import golden_json, load_golden
from golden import gen_golden as gg

pytestmark = pytest.mark.gpu


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.mark.parametrize("M,N,K", [(128, 128, 128), (1, 16, 16), (5, 10, 512), (300, 64, 48), (257, 1000, 208),
                                   (1000, 72, 2048), (4096, 256, 64), (129, 33, 32)])
@pytest.mark.parametrize("rs", [7, 0, -1])
def test_gemm_s8_vs_oracle(oracle, M, N, K, rs):
    from common.quantity import _native
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    a = rng.integers(-128, 128, size=(M, K), dtype=np.int8)
    w = rng.integers(-128, 128, size=(N, K), dtype=np.int8)
    b = rng.integers(-128, 128, size=N).astype(np.int32)
    scale = 1 if rs > 0 else 64          # keep some results inside the clamp range when rs <= 0
    a = (a // scale).astype(np.int8); w = (w // scale).astype(np.int8)
    acc = a.astype(np.int64) @ w.astype(np.int64).T
    y = np.clip(oracle.right_shift(acc, rs) + b[None, :], -128, 127)
    ob = 3
    f32, s8 = _native.gemm_s8(dev(a), dev(w), dev(b), rs, ob, want_f32=True, want_s8=True)
    assert np.array_equal(s8.cpu().numpy().astype(np.int64), y)
    assert np.array_equal(f32.cpu().numpy(), (y / 8.0).astype(np.float32))


@pytest.mark.parametrize("case", gg.INTSIM_CONV_CASES, ids=[c[0] for c in gg.INTSIM_CONV_CASES])
def test_newconv2d_vs_golden(case):
    import common.quantity as cq
    g = load_golden("intsim.npz")
    name, B, Cin, H, W, Cout, k, stride, pad = case[:9]
    x, w, b, info = gg.intsim_conv_tensors(case)
    conv = nn.Conv2d(Cin, Cout, k, stride=stride, padding=pad, bias=b is not None)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(w))
        if b is not None:
            conv.bias.copy_(torch.from_numpy(b))
        m = cq.NewConv2d(conv.cuda(), dict(info))
        y = m(dev(x))
    assert np.array_equal(m.Conv.weight.data.cpu().numpy().astype(np.int8), g["conv/" + name + "/wq"])
    assert np.array_equal(m.quantized_bias.cpu().numpy().astype(np.int32), g["conv/" + name + "/bq"])
    assert y.shape == g["conv/" + name + "/y"].shape
    assert np.array_equal(y.cpu().numpy(), g["conv/" + name + "/y"])


@pytest.mark.parametrize("case", gg.INTSIM_LINEAR_CASES, ids=[c[0] for c in gg.INTSIM_LINEAR_CASES])
def test_newlinear_vs_golden(case):
    import common.quantity as cq
    g = load_golden("intsim.npz")
    name, B, fin, fout = case[:4]
    x, w, b, info = gg.intsim_linear_tensors(case)
    lin = nn.Linear(fin, fout)
    with torch.no_grad():
        lin.weight.copy_(torch.from_numpy(w)); lin.bias.copy_(torch.from_numpy(b))
        y = cq.NewLinear(lin.cuda(), dict(info))(dev(x))
    assert np.array_equal(y.cpu().numpy(), g["linear/" + name + "/y"])


# ResNet-50 layer geometries at a small batch: (Cin, H, W, Cout, k, stride, pad)
R50_SHAPES = [(3, 56, 56, 64, 7, 2, 3), (64, 28, 28, 64, 1, 1, 0), (64, 28, 28, 64, 3, 1, 1),
              (256, 28, 28, 512, 1, 2, 0), (128, 28, 28, 128, 3, 2, 1), (256, 14, 14, 256, 3, 1, 1),
              (512, 7, 7, 2048, 1, 1, 0), (512, 7, 7, 512, 3, 1, 1), (1024, 14, 14, 2048, 1, 2, 0)]


@pytest.mark.parametrize("shape", R50_SHAPES, ids=["%dx%dx%d_k%d_s%d" % (s[0], s[1], s[3], s[4], s[5]) for s in R50_SHAPES])
def test_conv_s8_resnet50_geometries_vs_oracle(oracle, shape):
    import common.quantity as cq
    Cin, H, W, Cout, k, stride, pad = shape
    B = 3
    x = det_inputs.bell(B * Cin * H * W, 300 + Cin, 2.0).reshape(B, Cin, H, W)
    w = det_inputs.bell(Cout * Cin * k * k, 301 + Cin, 0.05).reshape(Cout, Cin, k, k)
    b = det_inputs.bell(Cout, 302 + Cin, 1.0)
    info = {"weight_bit": 9, "input_bit": 5, "output_bit": 4, "bias_bit": 4}
    conv = nn.Conv2d(Cin, Cout, k, stride=stride, padding=pad)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(w)); conv.bias.copy_(torch.from_numpy(b))
        y = cq.NewConv2d(conv.cuda(), dict(info))(dev(x)).cpu().numpy()
    ref, _ = oracle.int_conv_layer(x, w, b, info, stride=stride, padding=pad)
    assert np.array_equal(y, ref)


# small-channel ("stem") convolutions: (B, Cin, H, W, Cout, k, stride, pad) incl. ragged patches (P, Q not
# multiples of the 8 x 16 output patch), one channel, eight channels, 3x3 and 5x5 filters
SMALLC_SHAPES = [(2, 3, 64, 64, 64, 7, 2, 3), (3, 3, 37, 53, 32, 7, 2, 3), (1, 1, 30, 30, 16, 3, 2, 1),
                 (2, 8, 21, 19, 48, 5, 2, 2), (2, 4, 18, 10, 256, 3, 2, 0), (1, 3, 224, 224, 64, 7, 2, 3),
                 (2, 3, 33, 41, 32, 7, 4, 3), (1, 3, 40, 300, 72, 3, 2, 1)]


@pytest.mark.parametrize("shape", SMALLC_SHAPES + [(2, 3, 35, 29, 32, 3, 2, 1), (2, 2, 16, 16, 16, 2, 2, 0),
                                                  (1, 4, 31, 40, 64, 5, 2, 2), (2, 3, 26, 22, 48, 7, 2, 2)],
                         ids=lambda s: "b%d_c%d_%dx%d_o%d_k%d_s%d" % s[:7])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("s2d", [True, False], ids=["s2d", "rows8"])
def test_smallc_conv_vs_oracle_and_im2col(oracle, shape, relu, s2d):
    """pq_quantize_nchw_to_padded_nhwc8_s8 + pq_conv2d_smallc_s8 (overlapping-window TMA) against the oracle's
    integer conv layer and against the explicit-im2col GEMM path, fp32 NCHW and int8 NHWC outputs."""
    import common.quantity as cq
    from common.quantity import _native
    B, Cin, H, W, Cout, k, stride, pad = shape
    x = det_inputs.bell(B * Cin * H * W, 400 + Cin + H, 2.0).reshape(B, Cin, H, W)
    w = det_inputs.bell(Cout * Cin * k * k, 401 + Cin, 0.05).reshape(Cout, Cin, k, k)
    b = det_inputs.bell(Cout, 402 + Cin, 1.0)
    info = {"weight_bit": 9, "input_bit": 5, "output_bit": 4, "bias_bit": 4}
    conv = nn.Conv2d(Cin, Cout, k, stride=stride, padding=pad)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(w)); conv.bias.copy_(torch.from_numpy(b))
        m = cq.NewConv2d(conv.cuda(), dict(info))
        assert m._smallc
        # stride (2, 2) with <= 4 channels takes the space-to-depth form by default; both forms must agree
        if s2d and not m._s2d:
            pytest.skip("not a space-to-depth shape")
        m._s2d = s2d
        f32, s8 = m._smallc_forward(dev(x), want_f32=True, want_s8=True, relu=relu)
    ref, _ = oracle.int_conv_layer(x, w, b, info, stride=stride, padding=pad)
    if relu:
        ref = np.maximum(ref, 0)
    assert np.array_equal(f32.cpu().numpy(), ref)
    assert np.array_equal(s8.permute(0, 3, 1, 2).cpu().numpy().astype(np.float32) / 16.0, ref)
    # the explicit im2col + GEMM path computes the same thing
    kp = (k * k * Cin + 63) // 64 * 64
    wq = m.Conv.weight.data.permute(0, 2, 3, 1).reshape(Cout, -1).to(torch.int8)
    w_nk = torch.zeros((Cout, kp), dtype=torch.int8, device="cuda")
    w_nk[:, :wq.shape[1]] = wq
    a, (N, P, Q) = _native.quantize_im2col_s8(dev(x), 5, (k, k), (stride, stride), (pad, pad), kp)
    _, s8b = _native.gemm_s8(a, w_nk, m._bias_i32, m.rs_bit, 4, hw=1, want_f32=False, want_s8=True, relu=relu)
    assert torch.equal(s8b.view(N, P, Q, Cout), s8)


@pytest.mark.parametrize("M,N,K", [(128, 32, 32), (1000, 48, 64), (4099, 64, 128), (777, 128, 256), (12345, 256, 64),
                                   (300, 512, 128), (130, 1024, 64), (64, 2048, 512), (5000, 80, 96)])
def test_gemm_s8_staged_int8_store(oracle, M, N, K):
    """int8 output through the swizzled shared-memory tile + TMA store (N % 16 == 0), every tile width and ragged
    M / N edges, with and without the fused ReLU.  (Writes outside the output are checked with sentinel-filled
    buffers in test_gpu_epilogue_matrix.py.)"""
    from common.quantity import _native
    rng = np.random.default_rng(M + N + K)
    a = rng.integers(-128, 128, size=(M, K), dtype=np.int8)
    w = rng.integers(-16, 16, size=(N, K), dtype=np.int8)
    b = rng.integers(-128, 128, size=N).astype(np.int32)
    acc = a.astype(np.int64) @ w.astype(np.int64).T
    for relu in (False, True):
        y = np.clip(oracle.right_shift(acc, 6) + b[None, :], -128, 127)
        if relu:
            y = np.maximum(y, 0)
        f32, s8 = _native.gemm_s8(dev(a), dev(w), dev(b), 6, 2, want_f32=True, want_s8=True, relu=relu)
        assert np.array_equal(s8.cpu().numpy().astype(np.int64), y)
        assert np.array_equal(f32.cpu().numpy(), (y / 4.0).astype(np.float32))
        _, s8_only = _native.gemm_s8(dev(a), dev(w), dev(b), 6, 2, want_f32=False, want_s8=True, relu=relu)
        assert torch.equal(s8_only, s8)


def test_tiny_reconmodel_bit_exact(tmp_path):
    """ReconModel of the tiny net: every NewConv2d / NewLinear / NewAdd output equals the reference's."""
    import common.quantity as cq
    import tools
    from test_gpu_e2e import _configs, _tiny_model
    g = load_golden("tiny_e2e.npz")
    j = golden_json(g)
    cfg, user = _configs(tmp_path, (1, 3, 16, 16), 2)
    os.makedirs(cfg["OUTPUT"]["WORK_DIR"], exist_ok=True)
    open(cfg["OUTPUT"]["FEAT_BIT_TABLE"], "w").write(j["after_second_rewrite"]["feat.table"])
    open(cfg["OUTPUT"]["WEIGHT_BIT_TABLE"], "w").write(j["after_second_rewrite"]["weight.table"])
    with torch.no_grad():
        net = _tiny_model(g)
        r = tools.Reconstruction(net, config=cfg)
        r.merge_bn()
        model = r.ReconModel(r.get_quantity_information(), str(tmp_path / "workdir" / "ReconModel.pth")).cuda()
        outs = {}
        for name, mod in model.named_modules():
            if type(mod).__name__ in ("NewConv2d", "NewLinear", "NewAdd"):
                mod.register_forward_hook(lambda m, i, o, name=name: outs.__setitem__(name, o.cpu().numpy()))
        y = model(torch.from_numpy(g["eval_batch"]).cuda()).cpu().numpy()
    for name, val in outs.items():
        assert np.array_equal(val, g["ReconModel/layer/" + name]), name
    assert np.array_equal(y, g["ReconModel/y"])
    # the saved model loads back (classes picklable by qualified name, buffers registered)
    loaded = torch.load(str(tmp_path / "workdir" / "ReconModel.pth"), weights_only=False)
    assert np.array_equal(loaded.cuda()(torch.from_numpy(g["eval_batch"]).cuda()).cpu().numpy(), y)


@pytest.mark.parametrize("M,N,K,rs,relu", [(1000, 64, 64, 7, True), (777, 256, 64, 9, False), (4096, 128, 256, 12, True),
                                           (513, 32, 576, 1, False), (2048, 512, 128, 20, False), (300, 16, 32, 5, True),
                                           (999, 64, 1024, 3, False)])
def test_folded_bias_epilogue_equals_classic(oracle, M, N, K, rs, relu):
    """PQ_FLAG_BIAS_FOLDED against the classic staged epilogue and the oracle, with biases at the int8 extremes and
    accumulators that saturate both ways."""
    from common.quantity import _native
    rng = np.random.default_rng(M + N + rs)
    a = rng.integers(-128, 128, size=(M, K)).astype(np.int8)
    w = rng.integers(-128, 128, size=(N, K)).astype(np.int8)
    a[:7] = 127; w[:5] = 127; w[5:9] = -128                        # extreme accumulators
    bias = rng.integers(-128, 128, size=N).astype(np.int32)
    bias[:4] = [-128, 127, 0, -1]
    ta, tw, tb = torch.from_numpy(a).cuda(), torch.from_numpy(w).cuda(), torch.from_numpy(bias).cuda()
    folded_bias = _native.bias_fold(tb, rs)
    assert folded_bias.numel() == 3 * N and torch.equal(folded_bias[:N], tb)
    b64 = bias.astype(np.int64)
    assert np.array_equal(folded_bias[N:2 * N].cpu().numpy().astype(np.int64), (1 << (rs - 1)) + (b64 << rs))
    pairs = folded_bias[2 * N:].cpu().numpy().view(np.int16).astype(np.int64)       # [h pairs | l pairs], channel order
    assert np.array_equal(pairs[:N], 127 + np.minimum(b64, 0)) and np.array_equal(pairs[N:], -128 + np.maximum(b64, 0))
    _, classic = _native.gemm_s8(ta, tw, tb, rs, 3, want_f32=False, want_s8=True, relu=relu)
    _, folded = _native.gemm_s8(ta, tw, folded_bias, rs, 3, want_f32=False, want_s8=True, relu=relu)
    assert torch.equal(classic, folded)
    acc = a.astype(np.int64) @ w.astype(np.int64).T
    want = np.clip(oracle.right_shift(acc, rs) + bias[None, :], -128, 127)
    if relu:
        want = np.maximum(want, 0)
    assert np.array_equal(folded.cpu().numpy().astype(np.int64), want)
    # the fp32-boundary epilogue ignores the flag and reads the plain bias at the front of the buffer
    f32a, _ = _native.gemm_s8(ta, tw, tb, rs, 3, want_f32=True, want_s8=False)
    f32b, _ = _native.gemm_s8(ta, tw, folded_bias, rs, 3, want_f32=True, want_s8=False)
    assert torch.equal(f32a, f32b)


def test_accumulator_range_debug_check():
    """CHECK_ACC_RANGE (debug): the reference's fp32 convolution is integer arithmetic only below 2^24
    (SURVEY a13); the check records max |acc| per layer and warns where a legitimate divergence can start."""
    import warnings
    import common.quantity as cq
    from common.quantity import new_quantity_op as nq
    info = {"weight_bit": 7, "input_bit": 7, "output_bit": 0, "bias_bit": 0}
    conv = nn.Conv2d(512, 16, 3, padding=1, bias=False)
    with torch.no_grad():
        conv.weight.fill_(1.0)                                     # quantises to +127 everywhere
        m = cq.NewConv2d(conv.cuda(), dict(info))
        x = torch.ones(1, 512, 8, 8, device="cuda")                # quantises to +127 everywhere
        small = cq.NewConv2d(nn.Conv2d(16, 16, 1).cuda(), {"weight_bit": 5, "input_bit": 3, "output_bit": 3, "bias_bit": 3})
        nq.CHECK_ACC_RANGE = True
        try:
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                y = m(x)
                small(torch.randn(2, 16, 4, 4, device="cuda"))
        finally:
            nq.CHECK_ACC_RANGE = False
    assert m.max_abs_acc == 127.0 * 127.0 * 512 * 9 and m.max_abs_acc >= nq.FP32_EXACT_LIMIT     # 74 317 824
    assert any("2^24" in str(v.message) for v in w)
    assert 0 < small.max_abs_acc < nq.FP32_EXACT_LIMIT
    assert float(y.max()) == 127.0                                 # the int32 path itself stays exact and saturates
    model = nn.Sequential(m, small)
    assert set(nq.accumulator_report(model)) == {"0", "1"}


# dilated and grouped convolutions: the reference wraps ANY nn.Conv2d (new_quantity_op.py:104-133)
@pytest.mark.parametrize("case", gg.INTSIM_EXT_CASES, ids=[c[0] for c in gg.INTSIM_EXT_CASES])
@pytest.mark.parametrize("pipeline", [False, True])
def test_newconv2d_dilation_and_groups_vs_golden(oracle, case, pipeline):
    """Dilation = im2col-TMA tap offsets (pq_conv2d_s8 with pq_conv_desc.dil_h / dil_w), groups = one tensor-core
    convolution per group; against the reference's NewConv2d around the same dilated / grouped nn.Conv2d
    (intsim_ext.npz) and the oracle."""
    import common.quantity as cq
    g = load_golden("intsim_ext.npz")
    name, B, Cin, H, W, Cout, k, stride, pad, dil, groups = case[:11]
    x, w, b, info = gg.intsim_ext_tensors(case)
    conv = nn.Conv2d(Cin, Cout, k, stride=stride, padding=pad, dilation=dil, groups=groups)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(w)); conv.bias.copy_(torch.from_numpy(b))
        m = cq.NewConv2d(conv.cuda(), dict(info))
        m.int8_pipeline = pipeline
        y = m(dev(x))
        if pipeline and hasattr(y, "dequantize"):
            y = y.dequantize()
    want = g["conv/" + name + "/y"]
    assert y.shape == want.shape
    assert np.array_equal(y.cpu().numpy(), want)
    ref, _ = oracle.int_conv_layer(x, w, b, info, stride=stride, padding=pad, dilation=dil, groups=groups)
    assert np.array_equal(ref, want)


def test_newconv2d_unsupported_padding_mode_is_a_named_error():
    import common.quantity as cq
    conv = nn.Conv2d(16, 16, 3, padding=1, padding_mode="reflect").cuda()
    with pytest.raises(NotImplementedError, match="PQ_EUNSUPPORTED"):
        cq.NewConv2d(conv, {"weight_bit": 7, "input_bit": 4, "output_bit": 3, "bias_bit": 3})


# Patch-window path (GemmParams a_im2col == 3): (B, C, H, W, K).  Covers every patch shape (2 x 64, 4 x 32, 8 x 16),
# ragged last patches (H not a multiple of TH), the widest rows a patch takes (W + 2 == TW), fewer filters than the
# tile holds and filter counts without the staged int8 store (K % 16 != 0).
WINDOW_SHAPES = [(2, 64, 56, 56, 64), (3, 64, 28, 28, 48), (2, 64, 15, 30, 64), (2, 64, 9, 13, 32), (1, 64, 5, 62, 64),
                 (2, 64, 3, 14, 24), (1, 64, 1, 1, 64), (2, 128, 28, 28, 128), (2, 128, 14, 14, 96), (1, 128, 7, 30, 128),
                 (3, 128, 10, 9, 72), (2, 64, 33, 17, 64)]


@pytest.mark.parametrize("shape", WINDOW_SHAPES, ids=["b%d_c%d_%dx%d_k%d" % s for s in WINDOW_SHAPES])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("folded", [False, True])
def test_conv_patch_windows_equal_im2col_and_exact_evaluation(shape, relu, folded):
    """3x3 / stride 1 / pad 1 convolutions whose A operand is one TMA box per tile read through nine shifted
    shared-memory descriptors: int8 NHWC and fp32 NCHW outputs must equal the im2col-TMA path bit for bit and an
    independent evaluation (float64 convolution of the integer tensors + the integer epilogue of
    new_quantity_op.py:11-44,124-133 in torch int64 ops)."""
    from common.quantity import _native
    B, C, H, W, K = shape
    g = torch.Generator().manual_seed(B * 1000 + C + H * 7 + W * 13 + K)
    x = torch.randint(-128, 128, (B, H, W, C), dtype=torch.int8, generator=g).cuda()
    w = torch.randint(-128, 128, (K, 3, 3, C), dtype=torch.int8, generator=g).cuda()
    bias = torch.randint(-128, 128, (K,), dtype=torch.int32, generator=g).cuda()
    rs, ob = 11, 4
    bq = _native.bias_fold(bias, rs) if folded and K % 16 == 0 else bias
    outs = {}
    for windows in (True, False):
        f32, _ = _native.conv2d_s8(x, w, bq, (1, 1), (1, 1), rs, ob, want_f32=True, want_s8=False, relu=relu,
                                   windows=windows)
        _, s8 = _native.conv2d_s8(x, w, bq, (1, 1), (1, 1), rs, ob, want_f32=False, want_s8=True, relu=relu,
                                  windows=windows)
        outs[windows] = (f32, s8)
    assert torch.equal(outs[True][1], outs[False][1])
    assert torch.equal(outs[True][0], outs[False][0])
    acc = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).double(), w.permute(0, 3, 1, 2).double(), padding=1).long()
    r = torch.where(acc >= 0, (acc + (1 << (rs - 1))) >> rs, -((-acc + (1 << (rs - 1))) >> rs)).clamp(-128, 127)
    y = (r + bias.long().view(1, K, 1, 1)).clamp(-128, 127)
    if relu:
        y = y.clamp(min=0)
    assert torch.equal(outs[True][1].permute(0, 3, 1, 2).long(), y)
    assert torch.equal(outs[True][0], y.float() / 16.0)

"""The int8 inter-layer pipeline (SURVEY 8f n1) must be bit-identical to the fp32-boundary ReconModel,
which in turn is pinned to the reference (tests/test_gpu_intsim.py).  Also unit-tests its kernels
against exact integer / torch restatements."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import golden_json, load_golden

pytestmark = pytest.mark.gpu


def test_relu_and_maxpool_s8():
    from common.quantity import _native
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randint(-128, 128, (3, 17, 19, 32), dtype=torch.int8, device="cuda", generator=g)
    assert torch.equal(_native.relu_s8(x), torch.clamp(x, min=0))
    flat = torch.randint(-128, 128, (1000003,), dtype=torch.int8, device="cuda", generator=g)[3:]   # odd size
    assert torch.equal(_native.relu_s8(flat.clone()), torch.clamp(flat, min=0))
    for (k, s, p) in [(3, 2, 1), (2, 2, 0), (3, 1, 1)]:
        for relu in (False, True):
            y = _native.maxpool_nhwc_s8(x, k, s, p, relu=relu)
            ref = F.max_pool2d(x.permute(0, 3, 1, 2).float(), k, s, p)
            if relu:
                ref = torch.relu(ref)
            assert torch.equal(y.permute(0, 3, 1, 2).float(), ref), (k, s, p, relu)


@pytest.mark.parametrize("abit,bbit,qbit,a16,b16", [(4, 4, 4, False, False), (5, 3, 4, False, False), (3, 6, 7, False, True),
                                                    (6, 6, 2, True, True), (2, 7, 0, True, False), (0, 0, 5, False, False)])
def test_add_requant_exact(abit, bbit, qbit, a16, b16):
    from common.quantity import _native
    rng = np.random.default_rng(abit * 100 + bbit * 10 + qbit)
    n = 100003 + 5
    def operand(is16, bit):
        lim = 127 * 2 ** bit if is16 else 127
        lo = -128 * 2 ** bit if is16 else -128
        return rng.integers(lo, lim + 1, size=n).astype(np.int16 if is16 else np.int8)
    a, b = operand(a16, abit), operand(b16, bbit)
    for arelu, brelu, orelu in ((False, False, False), (True, False, False), (True, True, True), (False, False, True)):
        av = np.maximum(a, 0) if arelu else a
        bv = np.maximum(b, 0) if brelu else b
        # the reference's arithmetic: fp32 sum of the real values, clamp, [the nn.ReLU after the Eltwise,]
        # then the consumer's Quantity(q_bit)
        s = np.clip(av.astype(np.float32) / np.float32(2 ** abit) + bv.astype(np.float32) / np.float32(2 ** bbit),
                    np.float32(-128), np.float32(127))
        if orelu:
            s = np.maximum(s, np.float32(0))
        o = max(abit, bbit)
        ref16 = (s * np.float32(2 ** o)).astype(np.int64)
        assert np.array_equal(ref16, s.astype(np.float64) * 2 ** o)          # exact
        ref8 = np.clip(np.rint(s * np.float32(2.0 ** qbit)), -128, 127).astype(np.int64)
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        o16, o8 = _native.add_requant(ta, abit, arelu, tb, bbit, brelu, qbit, out_relu=orelu)
        assert np.array_equal(o16.cpu().numpy().astype(np.int64), ref16)
        assert np.array_equal(o8.cpu().numpy().astype(np.int64), ref8)


# (B, Cin, H, W, Cout, k, stride, pad, conv_ob, shortcut_bit, q_bit, shortcut int16?)
FUSED_ADD_CASES = [(2, 64, 14, 14, 256, 1, 1, 0, 4, 5, 4, True), (3, 32, 9, 11, 64, 3, 1, 1, 5, 3, 2, False),
                   (2, 128, 7, 7, 512, 1, 1, 0, 3, 6, 6, True), (1, 64, 20, 20, 32, 3, 2, 1, 6, 6, 7, False),
                   (2, 256, 5, 5, 1024, 1, 1, 0, 2, 4, 1, True), (2, 16, 33, 17, 48, 1, 1, 0, 4, 4, 4, False)]


@pytest.mark.parametrize("case", FUSED_ADD_CASES, ids=["c%d_%dx%d_o%d_k%d" % (c[1], c[2], c[3], c[4], c[5]) for c in FUSED_ADD_CASES])
def test_conv_add_fused_equals_conv_then_add(case):
    """pq_conv2d_s8_add (NewConv2d + NewAdd + ReLU in one epilogue; 1x1 stride-1 layers take its GEMM form) against
    the two separate kernels, which are pinned to the reference elsewhere."""
    from common.quantity import _native
    B, Cin, H, W, Cout, k, stride, pad, ob, sbit, qbit, s16 = case
    g = torch.Generator(device="cuda").manual_seed(Cin + Cout)
    x = torch.randint(-128, 128, (B, H, W, Cin), dtype=torch.int8, device="cuda", generator=g)
    w = torch.randint(-20, 21, (Cout, k, k, Cin), dtype=torch.int8, device="cuda", generator=g)
    bias = torch.randint(-128, 128, (Cout,), dtype=torch.int32, device="cuda", generator=g)
    P, Q = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    if s16:
        lim = 127 * 2 ** sbit
        sc = torch.randint(-lim - 2 ** sbit, lim + 1, (B, P, Q, Cout), dtype=torch.int16, device="cuda", generator=g)
    else:
        sc = torch.randint(-128, 128, (B, P, Q, Cout), dtype=torch.int8, device="cuda", generator=g)
    rs = 7
    _, y8 = _native.conv2d_s8(x, w, bias, (stride, stride), (pad, pad), rs, ob, want_f32=False, want_s8=True)
    for sc_relu, out_relu in ((False, False), (False, True), (True, True)):
        ref16, ref8 = _native.add_requant(y8, ob, False, sc, sbit, sc_relu, qbit, out_relu=out_relu)
        o16, o8 = _native.conv2d_s8_add(x, w, bias, (stride, stride), (pad, pad), rs, ob, sc, sbit, sc_relu, qbit, out_relu)
        assert torch.equal(o16, ref16), (sc_relu, out_relu)
        assert torch.equal(o8, ref8), (sc_relu, out_relu)
        _, o8b = _native.conv2d_s8_add(x, w, bias, (stride, stride), (pad, pad), rs, ob, sc, sbit, sc_relu, qbit, out_relu,
                                       want16=False)
        assert torch.equal(o8b, ref8)


def _build_recon(model_name, tmp_path, batch_shape):
    import tools
    from common.quantity import merge_bn
    from bench_sim import build, configs
    cfg, user = configs(str(tmp_path / "wd"), 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build(model_name), "cpu"), config=cfg, user_config=user, verbose=False)
        cal = [(torch.randn(4, 3, 224, 224, generator=torch.Generator().manual_seed(1 + i)), None) for i in range(2)]
        q.activation_quantize(cal)
        q.weight_quantize()
        r = tools.Reconstruction(build(model_name), config=cfg)
        r.merge_bn()
        return r.ReconModel(r.get_quantity_information(), None).cuda().eval()


@pytest.mark.parametrize("model_name,batch,fuse_add", [("r18", 3, False), ("r50", 2, False), ("r50", 2, True), ("r18", 2, True)])
def test_pipeline_equals_fp32_boundary_model(tmp_path, monkeypatch, model_name, batch, fuse_add):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from common.quantity import QTensor, enable_int8_pipeline, NewConv2d, int8_pipeline
    monkeypatch.setattr(int8_pipeline, "FUSE_ADD_INTO_CONV", fuse_add)
    model = _build_recon(model_name, tmp_path, batch)
    x = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(42)).cuda()
    with torch.no_grad():
        ref = model(x)
        ref_layers = {}
        hooks = [m.register_forward_hook(lambda m, i, o, n=n: ref_layers.__setitem__(n, o))
                 for n, m in model.named_modules() if type(m).__name__ in ("NewConv2d", "NewAdd")]
        model(x)
        for h in hooks:
            h.remove()
        enable_int8_pipeline(model)
        from common.quantity import _native as _nat
        relu_launches = _nat.LAUNCHES.get("relu_s8", 0)
        seen = {}
        hooks = [m.register_forward_hook(lambda m, i, o, n=n: seen.__setitem__(n, o))
                 for n, m in model.named_modules() if type(m).__name__ in ("NewConv2d", "NewAdd")]
        out = model(x)
        for h in hooks:
            h.remove()
        # every ReLU behind a convolution ran inside that convolution's epilogue (decided lazily, per request)
        assert _nat.LAUNCHES.get("relu_s8", 0) == relu_launches
    assert not isinstance(out, QTensor)
    assert torch.equal(out, ref)
    n_q = 0
    for name, o in seen.items():
        if isinstance(o, QTensor):
            n_q += 1
            # what a hook on the layer observes is the layer's OWN output (pre-ReLU), as in the fp32-boundary model
            assert torch.equal(o.dequantize(), ref_layers[name]), name
    assert n_q >= 15
    from common.quantity import _native
    if fuse_add:
        assert _native.LAUNCHES.get("conv_add_s8", 0) > 0, "no NewAdd was fused into its producer convolution"
    # the same forward captured once and replayed as a CUDA graph, on the capture batch and on a new one
    from common.quantity import GraphedForward
    fwd = GraphedForward(model, x)
    assert fwd.launches > 0
    assert torch.equal(fwd(x), ref)
    x2 = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(43)).cuda()
    got2 = fwd(x2).clone()
    enable_int8_pipeline(model, False)
    with torch.no_grad():
        assert torch.equal(model(x), ref)
        assert torch.equal(model(x2), got2)


def test_pipeline_fallback_paths_tiny_net(tmp_path):
    """8-channel layers, Concat and odd shapes force the de-quantise fallbacks; the result must not change."""
    import tools
    from common.quantity import enable_int8_pipeline
    from test_gpu_e2e import _configs, _tiny_model
    g = load_golden("tiny_e2e.npz")
    j = golden_json(g)
    cfg, user = _configs(tmp_path, (1, 3, 16, 16), 2)
    os.makedirs(cfg["OUTPUT"]["WORK_DIR"], exist_ok=True)
    open(cfg["OUTPUT"]["FEAT_BIT_TABLE"], "w").write(j["after_second_rewrite"]["feat.table"])
    open(cfg["OUTPUT"]["WEIGHT_BIT_TABLE"], "w").write(j["after_second_rewrite"]["weight.table"])
    with torch.no_grad():
        r = tools.Reconstruction(_tiny_model(g), config=cfg)
        r.merge_bn()
        model = enable_int8_pipeline(r.ReconModel(r.get_quantity_information(), None).cuda())
        y = model(torch.from_numpy(g["eval_batch"]).cuda())
    assert np.array_equal(y.cpu().numpy(), g["ReconModel/y"])


# (channel counts, int16 flags, bits, relu flags, q_bit, c_out_pad)
CONCAT_CASES = [((32, 64, 16), (False, False, False), (4, 4, 4), (False, False, False), 4, 112),      # pure copy
                ((32, 64, 16), (False, True, False), (5, 6, 2), (False, True, False), 4, 128),         # vector path
                ((16, 16), (True, True), (7, 3), (True, True), 0, 32),
                ((8, 8), (False, False), (3, 5), (False, True), 4, 16),                                # scalar path
                ((5, 3, 7), (False, True, False), (1, 6, 4), (True, False, False), 7, 32),
                ((48,), (False,), (2,), (False,), 6, 64)]


@pytest.mark.parametrize("case", CONCAT_CASES, ids=["c" + "_".join(map(str, c[0])) + "_q%d" % c[4] for c in CONCAT_CASES])
def test_concat_requant_vs_oracle(oracle, case):
    """pq_concat_requant_s8 == Quantity(q_bit)(Concat(de-quantised members)) (the reference composition)."""
    from common.quantity import _native
    chans, is16, bits, relus, q_bit, c_pad = case
    rng = np.random.default_rng(sum(chans) + q_bit)
    N, H, W = 3, 7, 9
    srcs, parts = [], []
    for c, w16, bit, relu in zip(chans, is16, bits, relus):
        lo, hi = (-128 * 2 ** bit, 127 * 2 ** bit) if w16 else (-128, 127)
        v = rng.integers(lo, hi + 1, size=(N, H, W, c)).astype(np.int16 if w16 else np.int8)
        v.reshape(-1)[:4] = [lo, hi, 0, -1]
        srcs.append((torch.from_numpy(v).cuda(), bit, relu))
        real = v.astype(np.float32) / np.float32(2.0 ** bit)
        parts.append(np.maximum(real, 0) if relu else real)
    want = oracle.concat_quantize([p.transpose(0, 3, 1, 2) for p in parts], q_bit)      # fp32 NCHW
    got = _native.concat_requant_s8(srcs, q_bit, c_pad).cpu().numpy()
    assert got.shape == (N, H, W, c_pad)
    assert np.array_equal(got[..., :sum(chans)].transpose(0, 3, 1, 2).astype(np.float32), want)
    assert not got[..., sum(chans):].any()                                             # channel padding is zero


def test_concat_requant_errors():
    from common.quantity import _native
    a = torch.zeros((1, 2, 2, 16), dtype=torch.int8, device="cuda")
    with pytest.raises(RuntimeError):
        _native.concat_requant_s8([(a, 4, False)], 4, 8)             # output narrower than the sources
    with pytest.raises(RuntimeError):
        _native.concat_requant_s8([(a, 20, False)], 0, 16)           # shift out of range
    with pytest.raises(RuntimeError):
        _native.concat_requant_s8([(a, 4, False)] * 9, 4, 256)       # too many sources


class _WideCatNet(torch.nn.Module):
    """Concat of 32- and 64-channel branches (vector path of the concat kernel), a nested concat, a ReLU
    between Concat and its consumer, and an Eltwise whose int16 sum feeds a Concat."""

    def __init__(self):
        super().__init__()
        from common.quantity import Concat, Eltwise, View
        nn = torch.nn
        self.stem = nn.Sequential(nn.Conv2d(3, 32, 3, padding=1, bias=False), nn.BatchNorm2d(32), nn.ReLU(False))
        self.a = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1, bias=False), nn.BatchNorm2d(32))
        self.b = nn.Sequential(nn.Conv2d(32, 64, 1, bias=True), nn.BatchNorm2d(64), nn.ReLU(False))
        self.cat1 = Concat()
        self.relu1 = nn.ReLU(False)
        self.c = nn.Sequential(nn.Conv2d(96, 32, 3, padding=1, bias=False), nn.BatchNorm2d(32))
        self.add = Eltwise()
        self.cat2 = Concat()
        self.cat3 = Concat()
        self.d = nn.Sequential(nn.Conv2d(32 + 32 + 96, 48, 1, bias=False), nn.BatchNorm2d(48), nn.ReLU(False))
        self.pool = nn.AvgPool2d(12)
        self.view = View()
        self.fc = nn.Linear(48, 10)

    def forward(self, x):
        s = self.stem(x)
        cat1 = self.relu1(self.cat1(self.a(s), self.b(s)))
        e = self.add(self.c(cat1), s)
        cat3 = self.cat3(self.cat2(e, s), cat1)                     # nested: (Eltwise sum, stem) ++ cat1
        return self.fc(self.view(self.pool(self.d(cat3))))


def test_pipeline_concat_stays_quantised(tmp_path):
    import tools
    from common.quantity import _native, enable_int8_pipeline, merge_bn
    from test_gpu_e2e import _configs

    def build():
        torch.manual_seed(3)
        net = _WideCatNet().eval()
        g = torch.Generator().manual_seed(11)
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
                m.weight.data.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.data.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
        return net

    cfg, user = _configs(tmp_path, (1, 3, 12, 12), 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build(), "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize([(torch.randn(4, 3, 12, 12, generator=torch.Generator().manual_seed(1 + i)), None)
                               for i in range(3)])
        q.weight_quantize()
        r = tools.Reconstruction(build(), config=cfg)
        r.merge_bn()
        model = r.ReconModel(r.get_quantity_information(), None).cuda().eval()
        x = torch.randn(5, 3, 12, 12, generator=torch.Generator().manual_seed(42)).cuda()
        ref = model(x)
        enable_int8_pipeline(model)
        before = _native.LAUNCHES.get("concat_requant", 0)
        out = model(x)
        assert _native.LAUNCHES.get("concat_requant", 0) - before == 2, "Concat consumers did not use the int8 kernel"
        assert torch.equal(out, ref)
        enable_int8_pipeline(model, False)
        assert torch.equal(model(x), ref)


def test_pipeline_add_writes_only_consumed_payloads(tmp_path):
    """The payload census: after one forward every Eltwise knows which of its two outputs is read, and later
    forwards skip the other one (stage-end adds feed only convolutions -> int8 only; the last add feeds the
    average pool -> exact int16 only).  The output stays bit-identical."""
    from common.quantity import NewAdd, _native, enable_int8_pipeline
    model = _build_recon("r18", tmp_path, 2)
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(5)).cuda()
    with torch.no_grad():
        ref = model(x)
        enable_int8_pipeline(model)
        first = model(x)
        def add_launches():            # stand-alone add kernels + adds fused into their producer convolution
            return _native.LAUNCHES.get("add_requant", 0) + _native.LAUNCHES.get("conv_add_s8", 0)
        l0 = add_launches()
        second = model(x)
        launches = add_launches() - l0
    assert torch.equal(first, ref) and torch.equal(second, ref)
    adds = [(n, m) for n, m in model.named_modules() if isinstance(m, NewAdd)]
    assert launches == len(adds) == 8, "steady state: exactly one add kernel per Eltwise"
    kinds = {n: frozenset(m._pipe_seen) for n, m in adds}
    both = frozenset({"s16", "q8"})
    assert kinds[adds[-1][0]] == frozenset({"s16"}), kinds           # feeds AvgPool2d: exact sum only
    q8_only = [n for n, k in kinds.items() if k == frozenset({"q8"})]
    assert len(q8_only) == 3, kinds                                  # the last block of stages 1-3
    assert sum(1 for k in kinds.values() if k == both) == 4, kinds  # blocks followed by an identity shortcut


@pytest.mark.parametrize("shape", [(4, 7, 7, 2048), (3, 7, 7, 64), (2, 14, 14, 24), (2, 1, 1, 8), (5, 4, 4, 512), (2, 16, 16, 40)])
@pytest.mark.parametrize("is16", [False, True])
@pytest.mark.parametrize("relu", [False, True])
def test_avgpool_global_equals_torch_on_dequantised_tensor(shape, is16, relu):
    """pq_avgpool_global_nhwc_f32 (the pipeline's AvgPool2d before the classifier) against F.avg_pool2d of the
    de-quantised fp32 NCHW tensor, as the fp32-boundary model computes it: bit-identical."""
    from common.quantity import _native
    N, H, W, C = shape
    g = torch.Generator().manual_seed(N * 100 + C + (7 if is16 else 0))
    lim = 16384 if is16 else 128
    q = torch.randint(-lim, lim, shape, generator=g, dtype=torch.int16 if is16 else torch.int8).cuda()
    for bit in (6, 0, -2, 11):
        y = _native.avgpool_global_nhwc(q, bit, relu=relu)
        v = q.to(torch.float32) * (2.0 ** -bit)
        if relu:
            v = torch.relu(v)
        ref = torch.nn.functional.avg_pool2d(v.permute(0, 3, 1, 2).contiguous(), (H, W))
        assert y.shape == ref.shape and torch.equal(y, ref)

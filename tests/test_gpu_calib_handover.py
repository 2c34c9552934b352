"""The hand-overs of the fused calibration forward: pq_conv_epilogue_add_f32 (a convolution's epilogue with the Eltwise
that reads its output) and pq_conv_epilogue_maxpool_f32 (the stem's epilogue with the max-pool after its ReLU) against
ATen bit for bit, whole calibration jobs with every fallback of the hand-over, and the hand-over plan on CPU traces."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import ref_models
from test_gpu_calib_fusion import _Head, _bits, _fused_and_unfused, _ref_max, _specials

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------ the kernels
@gpu
@pytest.mark.parametrize("N,C,H,W", [(2, 256, 56, 56), (2, 512, 28, 28), (4, 1024, 14, 14), (64, 2048, 7, 7),
                                     (1, 3, 15, 17), (3, 5, 1, 3)])
def test_conv_epilogue_add_bit_exact(N, C, H, W):
    from common.quantity import _native
    gen = torch.Generator(device="cuda").manual_seed(N * 7919 + C * 31 + H * W)
    y0 = torch.randn(N, C, H, W, device="cuda", generator=gen)
    other = torch.randn(N, C, H, W, device="cuda", generator=gen)
    bias = torch.randn(C, device="cuda", generator=gen)
    _specials(y0, gen, with_nan=True)
    _specials(other, gen, with_nan=N < 4)
    y0.view(-1)[0], other.view(-1)[0], bias[0] = -0.0, -0.0, -0.0
    ref_y = y0.clone().add_(bias.view(1, -1, 1, 1))
    for first in (True, False):                          # the conv output as the Eltwise's first operand, or second
        ref_z = torch.add(ref_y, other) if first else torch.add(other, ref_y)
        for relu in (False, True):
            y = y0.clone()
            mb = torch.zeros(3, dtype=torch.int32, device="cuda")
            z, r = _native.conv_epilogue_add(y, bias, other, not first, relu, mb.data_ptr(), mb.data_ptr() + 8)
            torch.cuda.synchronize()
            assert torch.equal(_bits(y), _bits(ref_y))
            assert torch.equal(_bits(z), _bits(ref_z))
            assert (r is not None) == relu
            if relu:
                assert torch.equal(_bits(r), _bits(ref_z.clamp_min(0)))
            assert torch.equal(mb[:1], _ref_max(ref_y)) and mb[1].item() == 0 and torch.equal(mb[2:], _ref_max(ref_z))
    y = y0.clone()                                       # no max slots
    z, _ = _native.conv_epilogue_add(y, bias, other, False)
    assert torch.equal(_bits(y), _bits(ref_y)) and torch.equal(_bits(z), _bits(torch.add(ref_y, other)))


MAXPOOL_GEOMETRIES = [(k, s, p) for k in (1, 2, 3) for s in range(1, k + 1) for p in range(0, k // 2 + 1)]


@gpu
@pytest.mark.parametrize("k,s,p", MAXPOOL_GEOMETRIES)
@pytest.mark.parametrize("N,C,H,W", [(2, 64, 112, 112), (1, 3, 7, 9), (2, 2, 10, 5), (1, 4, 3, 4), (1, 2, 1, 1)])
def test_conv_epilogue_maxpool_bit_exact(k, s, p, N, C, H, W):
    from common.quantity import _native
    if H + 2 * p < k or W + 2 * p < k:
        pytest.skip("no output")
    gen = torch.Generator(device="cuda").manual_seed(N * 131 + C * 17 + H * W + k * 7 + s * 3 + p)
    y0 = torch.randn(N, C, H, W, device="cuda", generator=gen)
    bias = torch.randn(C, device="cuda", generator=gen)
    _specials(y0, gen, with_nan=True)
    # NaNs with distinct payloads next to each other and signed zeros in one window: the scan order decides
    flat = y0.view(-1)
    nans = torch.tensor([0x7fc00001, 0x7fc00002, 0x7fc00003, 0xffc00004 - (1 << 32)], dtype=torch.int32, device="cuda")
    flat[:4] = nans.view(torch.float32)[:min(4, flat.numel())]
    flat[W:W + 3] = torch.tensor([-0.0, 0.0, -0.0], device="cuda")[:min(3, flat.numel() - W)]
    bias[0] = -0.0
    ref_y = y0.clone().add_(bias.view(1, -1, 1, 1))
    ref_r = ref_y.clamp_min(0)
    ref_p = F.max_pool2d(ref_r, k, s, p)
    y = y0.clone()
    mb = torch.zeros(2, dtype=torch.int32, device="cuda")
    r, pooled = _native.conv_epilogue_maxpool(y, bias, k, s, p, mb.data_ptr() + 4)
    torch.cuda.synchronize()
    assert torch.equal(_bits(y), _bits(ref_y))
    assert torch.equal(_bits(r), _bits(ref_r))
    assert pooled.shape == ref_p.shape and torch.equal(_bits(pooled), _bits(ref_p))
    assert mb[0].item() == 0 and torch.equal(mb[1:], _ref_max(ref_y))


@gpu
def test_epilogue_hand_over_abi_errors():
    from common.quantity import _native
    lib = _native.lib()
    s = torch.cuda.current_stream().cuda_stream
    y = torch.zeros(2, 4, 8, 8, device="cuda")
    o, z, r, pl = (torch.zeros_like(y) for _ in range(4))
    b = torch.zeros(4, device="cuda")
    add = lib.pq_conv_epilogue_add_f32
    assert add(y.data_ptr(), b.data_ptr(), 2, 4, 64, o.data_ptr(), 1, y.data_ptr(), None, None, None, s) == -1
    assert add(y.data_ptr(), b.data_ptr(), 2, 4, 64, o.data_ptr(), 1, z.data_ptr(), o.data_ptr(), None, None, s) == -1
    assert add(y.data_ptr(), b.data_ptr(), 2, 4, 64, o.data_ptr() + 4, 1, z.data_ptr(), None, None, None, s) == -3
    assert add(y.data_ptr(), b.data_ptr(), 0, 4, 64, None, 1, None, None, None, None, s) == 0
    pool = lib.pq_conv_epilogue_maxpool_f32
    args = (y.data_ptr(), b.data_ptr(), 2, 4, 8, 8, r.data_ptr(), pl.data_ptr())
    for k, st, p in ((4, 2, 1), (3, 4, 1), (3, 2, 2), (2, 3, 0), (1, 1, 1)):      # k > 3, s > k, 2 p > k
        assert pool(*args, k, st, p, None, s) == -2, (k, st, p)
    assert pool(y.data_ptr(), b.data_ptr(), 1, 1, 256, 256, r.data_ptr(), pl.data_ptr(), 3, 2, 1, None, s) == -2
    assert pool(y.data_ptr(), b.data_ptr(), 2, 4, 8, 8, None, pl.data_ptr(), 3, 2, 1, None, s) == -1
    assert pool(y.data_ptr(), b.data_ptr(), 2, 4, 8, 8, r.data_ptr(), r.data_ptr(), 3, 2, 1, None, s) == -1
    torch.cuda.synchronize()
    assert not y.any() and not r.any() and not pl.any()
    # the Python wrapper declines what the kernel does not implement, without touching y
    y1 = torch.ones(1, 4, 8, 8, device="cuda")
    assert _native.conv_epilogue_maxpool(y1, b, 5, 2, 2) is None
    assert _native.conv_epilogue_maxpool(y1, b, 3, 2, 1) is not None


# ------------------------------------------------------------------------------ whole calibration jobs
class _Block(nn.Module):
    """conv -> ReLU -> Eltwise(conv(...), other) -> ReLU, with the hand-over's fallbacks as variants; every variant
    behaves like the plain block in the tracing forward (batch 1) and deviates only in the calibration forward."""

    def __init__(self, case):
        super().__init__()
        from common.quantity import Eltwise
        torch.manual_seed(17)
        self.case = case
        self.c1 = nn.Conv2d(3, 8, 3, padding=1)
        self.r1 = nn.ReLU()
        self.c2 = nn.Conv2d(8, 8, 3, padding=1)
        self.sc = nn.Conv2d(8, 8, 1) if case == "shortcut_first" else None
        self.elt = Eltwise()
        self.r2 = nn.ReLU()
        self.head = _Head(8)

    def forward(self, x):
        calib = x.shape[0] > 1
        a = self.r1(self.c1(x))
        if self.case == "shortcut_first":
            s = self.sc(a)
            e = self.elt(self.c2(a), s)
        elif self.case == "conv_is_second":
            e = self.elt(a, self.c2(a))
        else:
            if self.case == "modified_before" and calib:
                a.mul_(1.0)                              # `a` changes its version before c2 runs: no speculation
            y = self.c2(a)
            if self.case == "modified_after" and calib:
                a.mul_(1.0)                              # ... after c2 ran: the speculation is not taken
            other = a * 0.5 if self.case == "other_tensor" and calib else a
            e = self.elt(y, other)
        return self.head(self.r2(e))


def _batches(seed):
    return [(torch.randn(4, 3, 12, 12, generator=torch.Generator().manual_seed(seed + i)).cuda(), None)
            for i in range(2)]


def _job(tmp_path, net, batches, input_shape):
    """_fused_and_unfused, plus how often each fused kernel ran (one job, two batches)."""
    from common.quantity import _native
    store = {}
    _native.set_profile(store)
    try:
        a, _, launches, reduced = _fused_and_unfused(tmp_path, net, batches, input_shape)
    finally:
        _native.set_profile(None)
    torch.cuda.synchronize()
    return a, launches, reduced, {k: len(v) for k, v in store.items() if k.startswith(("conv", "eltwise"))}


@gpu
@pytest.mark.parametrize("case,hit", [("plain", True), ("shortcut_first", True), ("conv_is_second", True),
                                      ("modified_before", False), ("modified_after", False),
                                      ("other_tensor", False)])
def test_eltwise_hand_over_and_fallbacks(case, hit, tmp_path):
    net = _Block(case).eval()
    a, launches, reduced, kinds = _job(tmp_path, net, _batches(40), (1, 3, 12, 12))
    convs = 3 if case == "shortcut_first" else 2
    # pass 1 and pass 2 from the cache: two forwards of two batches
    speculated = 0 if case == "modified_before" else 2
    assert kinds.get("conv_epilogue_add", 0) == speculated
    assert kinds.get("eltwise", 0) == (0 if hit else 2)
    assert launches == {"conv_epilogue": 2 * convs, "eltwise": speculated + kinds.get("eltwise", 0)}
    # the Eltwise's max came from the fused ops either way (hit: confirmed speculation; miss: eltwise_add's own)
    elt = [n for n in a["top_feat_names"] if n.startswith("Eltwise")]
    assert all(set(elt) <= r for r in reduced)


class _TwiceEltwise(nn.Module):
    def __init__(self):
        super().__init__()
        from common.quantity import Eltwise
        torch.manual_seed(19)
        self.c1 = nn.Conv2d(3, 8, 3, padding=1)
        self.c2 = nn.Conv2d(8, 8, 3, padding=1)
        self.elt = Eltwise()
        self.head = _Head(8)
        self.spare = nn.Linear(1, 1)                     # feat.table's one spare name for the second call

    def forward(self, x):
        a = self.c1(x)
        return self.head(self.elt(self.c2(a), self.elt(a, a)))


@gpu
def test_eltwise_that_fires_twice_is_not_handed_over(tmp_path):
    _, launches, _, kinds = _job(tmp_path, _TwiceEltwise().eval(), _batches(50), (1, 3, 12, 12))
    assert "conv_epilogue_add" not in kinds and "eltwise" not in kinds
    assert launches == {"conv_epilogue": 4, "eltwise": 0}


class _Stem(nn.Module):
    def __init__(self, pool):
        super().__init__()
        torch.manual_seed(23)
        self.conv = nn.Conv2d(3, 8, 7, stride=2, padding=3)
        self.relu = nn.ReLU()
        self.pool = pool
        self.head = _Head(8)

    def forward(self, x):
        return self.head(self.pool(self.relu(self.conv(x))))


@gpu
@pytest.mark.parametrize("pool,fused", [(nn.MaxPool2d(3, 2, 1), True), (nn.MaxPool2d(2), True),
                                        (nn.MaxPool2d(5, 1, 2), False), (nn.MaxPool2d(3, 1, 1, ceil_mode=True), False),
                                        (nn.MaxPool2d(3, 1, 1, dilation=2), False)])
def test_stem_max_pool_hand_over(pool, fused, tmp_path):
    batches = [(torch.randn(4, 3, 47, 47, generator=torch.Generator().manual_seed(60 + i)).cuda(), None)
               for i in range(2)]
    net = _Stem(pool).eval()
    net.head.pool = nn.AvgPool2d(pool(torch.zeros(1, 8, 24, 24)).shape[-1])
    _, launches, _, kinds = _job(tmp_path, net, batches, (1, 3, 47, 47))
    assert launches["conv_epilogue"] == 2
    assert kinds.get("conv_epilogue_maxpool", 0) == (2 if fused else 0)


# ---------------------------------------------------------------------------- the plan, on a CPU trace
def _traced(net, shape):
    import tools
    q = tools.Quantity.__new__(tools.Quantity)
    settings = tools._config.load_tool_config(None)["SETTINGS"]
    q._all_op_type, q._cared_op_type = settings["ALL_OP_TYPE"], settings["CARE_OP_TYPE"]
    q._allow_same_tid_op_type = settings["ALLOW_SAME_TID_OP_TYPE"]
    q.cuda_device = torch.device("cpu")
    q.build_net_structure(net, shape)
    return q


@pytest.mark.parametrize("name", ["r18", "r50", "resnext50", "mobilenetv2"])
def test_handover_plan_on_a_cpu_trace(name):
    from common.quantity import merge_bn
    if name in ("r18", "r50"):
        net = ref_models.build_model(name)
    elif name == "resnext50":
        from model.resnet.resnet_fabu import resnext50_32x4d_fabu
        net = resnext50_32x4d_fabu()
    else:
        from model.mobilenet.mobilenetv2_fabu import mobilenetv2_fabu
        net = mobilenetv2_fabu()
    net = merge_bn(net.eval(), "cpu")
    q = _traced(net, (1, 3, 224, 224))
    eltwise, pools = q._handover_plan
    from common.quantity import Eltwise
    units = {"r18": 8, "r50": 16, "resnext50": 16, "mobilenetv2": 10}[name]
    downsample = {"r18": 3, "r50": 4, "resnext50": 4, "mobilenetv2": 0}[name]
    assert len(eltwise) == units == sum(type(m) is Eltwise for m in net.modules())
    for elt, (producer, other, producer_first) in eltwise.items():
        pos = int(elt.rsplit("_", 1)[1])
        # the residual branch's last convolution fires right before the Eltwise, after the other operand's producer
        assert producer.startswith("Conv2d_") and int(producer.rsplit("_", 1)[1]) == pos - 1
        assert int(other.rsplit("_", 1)[1]) < pos - 1
        if name == "mobilenetv2":                       # Eltwise(self.conv(x), x): x is the previous unit's output
            assert producer_first and other.split("_")[0] in ("Conv2d", "Eltwise")
    # a downsampling unit's shortcut convolution completes `Eltwise(left(x), shortcut(x))`; its other operand is
    # the left branch's last convolution
    ds = [e for e, (_, other, first) in eltwise.items() if not first]
    assert len(ds) == downsample and all(eltwise[e][1].startswith("Conv2d_") for e in ds)
    ident = [e for e, (_, other, first) in eltwise.items() if first]
    if name != "mobilenetv2":
        assert all(eltwise[e][1].startswith(("ReLU_", "MaxPool2d_")) for e in ident)
        assert pools == {"Conv2d_1": "MaxPool2d_3"}
    else:
        assert pools == {}


def test_handover_plan_skips_what_it_cannot_take():
    class Net(nn.Module):
        def __init__(self, pool):
            super().__init__()
            from common.quantity import Eltwise
            self.c1 = nn.Conv2d(3, 8, 3, padding=1)
            self.r1 = nn.ReLU()
            self.pool = pool
            self.c2 = nn.Conv2d(8, 8, 1)
            self.r2 = nn.ReLU()                         # c2 has a fused ReLU: it cannot also take the Eltwise
            self.elt = Eltwise()
            self.c3 = nn.Conv2d(8, 8, 1, bias=False)    # not planned
            self.elt2 = Eltwise()

        def forward(self, x):
            a = self.pool(self.r1(self.c1(x)))
            c = self.c2(a)
            e = self.elt(a, c)
            self.r2(c)
            return self.elt2(self.c3(e), e)

    q = _traced(Net(nn.MaxPool2d(3, 2, 1)).eval(), (1, 3, 8, 8))
    assert q._handover_plan == ({}, {"Conv2d_1": "MaxPool2d_3"})
    q = _traced(Net(nn.MaxPool2d(3, 2, 1, ceil_mode=True)).eval(), (1, 3, 8, 8))
    assert q._handover_plan == ({}, {})

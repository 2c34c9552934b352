"""The fused calibration forward: pq_conv_epilogue_f32 / pq_eltwise_add_f32 against ATen bit for bit, whole calibration
jobs fused vs unfused, the cases that must run unfused, and the planning function on a CPU trace."""
import os

import pytest
import torch
import torch.nn as nn

import ref_models

gpu = pytest.mark.gpu


def _specials(t, gen, with_nan):
    """Overwrite a few hundred positions of t with +-0, subnormals and (with_nan) +-inf and NaN."""
    vals = [0.0, -0.0, 1e-40, -1e-40, 1.4e-45, -3e-39]
    if with_nan:
        vals += [float("inf"), float("-inf"), float("nan")]
    flat = t.view(-1)
    idx = torch.randint(0, flat.numel(), (min(300, flat.numel()),), generator=gen, device=t.device)
    flat[idx] = torch.tensor(vals, device=t.device).repeat(len(idx) // len(vals) + 1)[:len(idx)]


def _bits(t):
    return t.contiguous().view(torch.int32)


def _ref_max(t):
    from common.quantity import _native
    mb = torch.zeros(1, dtype=torch.int32, device=t.device)
    _native.absmax_multi([t.reshape(-1)], mb)
    return mb


@gpu
@pytest.mark.parametrize("N", [1, 64])
@pytest.mark.parametrize("C", [3, 64, 2048])
@pytest.mark.parametrize("HW", [49, 196, 784, 3136, 12544, 15 * 17])
def test_conv_epilogue_bit_exact(N, C, HW):
    from common.quantity import _native
    gen = torch.Generator(device="cuda").manual_seed(N * 100003 + C * 17 + HW)
    y0 = torch.randn(N, C, HW, 1, device="cuda", generator=gen)
    bias = torch.randn(C, device="cuda", generator=gen)
    _specials(y0, gen, with_nan=N == 1)
    bias[0] = -0.0
    y0[0, 0] = -0.0                                      # -0 + -0: the sign of zero through the add and the ReLU
    if C > 1:
        bias[1] = 1e-39
    ref = y0 + bias.view(1, -1, 1, 1)
    for relu in (False, True):
        y = y0.clone()
        mb = torch.zeros(2, dtype=torch.int32, device="cuda")
        r = _native.conv_epilogue(y, bias, relu=relu, max_slot=mb.data_ptr() + 4)
        torch.cuda.synchronize()
        assert torch.equal(_bits(y), _bits(ref))
        assert (r is not None) == relu
        if relu:
            assert torch.equal(_bits(r), _bits(torch.relu(ref)))
        assert mb[0].item() == 0 and torch.equal(mb[1:], _ref_max(ref))
    y = y0.clone()                                       # no max slot: nothing but the add
    _native.conv_epilogue(y, bias)
    assert torch.equal(_bits(y), _bits(ref))


@gpu
@pytest.mark.parametrize("n", [1, 3, 4, 49 * 3, 255, 64 * 2048 * 49, 64 * 256 * 3136 + 5])
def test_eltwise_add_bit_exact(n):
    from common.quantity import _native
    gen = torch.Generator(device="cuda").manual_seed(n)
    a = torch.randn(n, device="cuda", generator=gen)
    b = torch.randn(n, device="cuda", generator=gen)
    _specials(a, gen, with_nan=n % 2 == 1)
    _specials(b, gen, with_nan=False)
    a[0], b[0] = -0.0, -0.0
    ref = torch.add(a, b)
    mb = torch.zeros(1, dtype=torch.int32, device="cuda")
    z, r = _native.eltwise_add(a, b, relu=True, max_slot=mb.data_ptr())
    torch.cuda.synchronize()
    assert torch.equal(_bits(z), _bits(ref))
    assert torch.equal(_bits(r), _bits(torch.relu(ref)))
    assert torch.equal(mb, _ref_max(ref))
    z2, r2 = _native.eltwise_add(a, b)
    assert r2 is None and torch.equal(_bits(z2), _bits(ref))


@gpu
def test_epilogue_abi_errors():
    from common.quantity import _native
    lib = _native.lib()
    y = torch.zeros(2, 4, 8, 8, device="cuda")
    b = torch.zeros(4, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    assert lib.pq_conv_epilogue_f32(y.data_ptr(), b.data_ptr(), 2, 4, 64, y.data_ptr(), None, s) == -1
    assert lib.pq_conv_epilogue_f32(y.data_ptr() + 4, b.data_ptr(), 2, 4, 63, None, None, s) == -3
    assert lib.pq_conv_epilogue_f32(y.data_ptr(), b.data_ptr(), 0, 4, 64, None, None, s) == 0
    assert lib.pq_eltwise_add_f32(y.data_ptr(), y.data_ptr(), y.data_ptr(), 512, None, None, s) == -1
    # the Python wrappers refuse what the kernels would misaddress
    with pytest.raises(RuntimeError, match="fp32"):
        _native.conv_epilogue(y.half(), b)
    with pytest.raises(RuntimeError, match="fp32"):
        _native.conv_epilogue(y.transpose(2, 3), b)
    with pytest.raises(RuntimeError, match="bias"):
        _native.conv_epilogue(y, b[:3])
    with pytest.raises(RuntimeError, match="differ"):
        _native.eltwise_add(y, y[:1])
    with pytest.raises(RuntimeError, match="fp32"):
        _native.eltwise_add(y, y.double())


# ------------------------------------------------------------------------------ whole calibration jobs
def _configs(tmp_path, input_shape, n_batches):
    import tools._config as tc
    cfg = tc.load_tool_config(os.path.join(os.path.dirname(tc.__file__), "configs.yml"))
    wd = str(tmp_path / "workdir")
    cfg["OUTPUT"] = {"WORK_DIR": wd, "WEIGHT_BIT_TABLE": wd + "/weight.table", "FEAT_BIT_TABLE": wd + "/feat.table",
                     "WEIGHT_DIR": wd + "/weight", "BIAS_DIR": wd + "/bias", "FINAL_WEIGHT_DIR": wd + "/new_weight",
                     "FINAL_BIAS_DIR": wd + "/new_bias"}
    cfg["SETTINGS"]["MAX_CALI_IMG_NUM"] = n_batches - 1
    user = tc.load_user_config({"PATH": {}, "MODEL": {"INPUT_SHAPE": ",".join(map(str, input_shape))},
                                "PRE_PROCESS": {"IMG": 1}, "SETTINGS": {"DEVICE": "gpu", "GPU": 0}})
    return cfg, user


def _fused_and_unfused(tmp_path, net, batches, input_shape, cache_bytes=None, care=None, autocast=False):
    """(fused result, unfused result, fused launches of each kind, the sets of tensor names whose pass-1 max-abs the
    fused ops took, one per batch) of the same calibration job.  care: CARE_OP_TYPE; autocast: run the job under
    torch.autocast(fp16)."""
    import tools
    from common.quantity import DistributionCollector, _native
    out = {}
    record = DistributionCollector._refresh_max_val_except
    for fuse in (True, False):
        cfg, user = _configs(tmp_path / ("f%d" % fuse), input_shape, len(batches))
        if care is not None:
            cfg["SETTINGS"]["CARE_OP_TYPE"] = care
        reduced = []

        def recording(self, tensors, names):
            reduced.append(set(names))
            return record(self, tensors, names)
        DistributionCollector._refresh_max_val_except = recording
        try:
            with torch.no_grad():
                q = tools.Quantity(net, config=cfg, user_config=user, cache_bytes=cache_bytes, verbose=False)
                q._fuse_calibration = fuse
                before = dict(_native.LAUNCHES)
                with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
                    q.activation_quantize(batches)
                launches = {k: _native.LAUNCHES.get(k, 0) - before.get(k, 0) for k in ("conv_epilogue", "eltwise")}
        finally:
            DistributionCollector._refresh_max_val_except = record
        assert all(vars(m).get("forward") is None for m in net.modules())      # every module restored
        out[fuse] = (q.last_calibration, open(cfg["OUTPUT"]["FEAT_BIT_TABLE"]).read(), launches, reduced)
    (a, ta, la, ra), (b, tb, lb, rb) = out[True], out[False]
    assert all(not r for r in rb)
    assert lb == {"conv_epilogue": 0, "eltwise": 0}
    assert ta == tb and a["top_feat_names"] == b["top_feat_names"]
    for n in a["top_feat_names"]:
        assert repr(a["max_vals"][n]) == repr(b["max_vals"][n]), n
        assert (a["distributions"][n] == b["distributions"][n]).all(), n
    return a, b, la, ra


@gpu
@pytest.mark.parametrize("name,n_batches,batch", [("tiny", 3, 2), ("lenet", 3, 8), ("r18", 2, 4), ("r50", 2, 4)])
def test_fused_calibration_equals_unfused(name, n_batches, batch, tmp_path):
    from common.quantity import merge_bn
    ref_models.set_deterministic()
    net = merge_bn(ref_models.build_model(name), "cpu")
    batches = ref_models.calib_batches(name, n_batches, batch)
    a, _, launches, reduced = _fused_and_unfused(tmp_path, net, batches, ref_models.INPUT_SHAPE[name])
    convs = sum(isinstance(m, nn.Conv2d) and m.bias is not None for m in net.modules())
    assert launches["conv_epilogue"] == n_batches * convs
    # every convolution / Eltwise output got its max in the fused op: pass 1 re-reads only the rest (image, Linear,
    # Concat)
    fused = {n for n in a["top_feat_names"] if n.rsplit("_", 1)[0] in ("Conv2d", "Eltwise")}
    assert len(fused) == convs + launches["eltwise"] // n_batches
    assert reduced == [fused] * n_batches
    # pass 2 from the HBM cache, and the same job with every batch's forward re-run in pass 2 (no max slot there)
    _, _, rerun, reduced = _fused_and_unfused(tmp_path / "rerun", net, batches, ref_models.INPUT_SHAPE[name],
                                              cache_bytes=0)
    assert rerun["conv_epilogue"] == 2 * n_batches * convs
    assert reduced == [fused] * n_batches


class _Head(nn.Module):
    def __init__(self, c):
        super().__init__()
        from common.quantity import View
        self.pool = nn.AvgPool2d(12)
        self.view = View()
        self.fc = nn.Linear(c, 4)

    def forward(self, x):
        return self.fc(self.view(self.pool(x)))


class _TwiceNet(nn.Module):
    def __init__(self):
        super().__init__()
        self.c0 = nn.Conv2d(3, 8, 3, padding=1, bias=False)
        self.c = nn.Conv2d(8, 8, 3, padding=1)
        self.relu = nn.ReLU()
        self.head = _Head(8)
        # never called: feat.table names its lines from named_modules(), one name per module (reference :468-489),
        # so a module that fires twice needs one spare name
        self.spare = nn.Linear(1, 1)

    def forward(self, x):
        return self.head(self.relu(self.c(self.c(self.c0(x)))))


def _one_conv(conv, relu_inplace=False):
    torch.manual_seed(7)
    return nn.Sequential(conv, nn.ReLU(relu_inplace), _Head(conv.out_channels))


@gpu
@pytest.mark.parametrize("case", ["called_twice", "inplace_relu", "no_bias", "reflect", "channels_last", "depthwise",
                                  "autocast"])
def test_unfused_cases_give_the_same_tables(case, tmp_path):
    torch.manual_seed(11)
    cin = 8 if case == "depthwise" else 3
    if case == "called_twice":
        net = _TwiceNet()
    elif case == "depthwise":
        net = _one_conv(nn.Conv2d(8, 8, 3, padding=1, groups=8))
    else:
        net = _one_conv(nn.Conv2d(3, 8, 3, padding=1, bias=case != "no_bias",
                                  padding_mode="reflect" if case == "reflect" else "zeros"),
                        relu_inplace=case == "inplace_relu")
    net = net.eval()
    batches = []
    for i in range(2):
        x = torch.randn(4, cin, 12, 12, generator=torch.Generator().manual_seed(20 + i)).cuda()
        batches.append((x.to(memory_format=torch.channels_last) if case == "channels_last" else x, None))
    _, _, launches, _ = _fused_and_unfused(tmp_path, net, batches, (1, cin, 12, 12), autocast=case == "autocast")
    assert launches["conv_epilogue"] == 0


class _TwoHeadNet(nn.Module):
    """An Eltwise whose output is a second model output: with Eltwise out of CARE_OP_TYPE it is traced but not
    observed."""

    def __init__(self):
        super().__init__()
        from common.quantity import Eltwise
        torch.manual_seed(13)
        self.c1 = nn.Conv2d(3, 8, 3, padding=1)
        self.r1 = nn.ReLU()
        self.c2 = nn.Conv2d(8, 8, 3, padding=1)
        self.elt = Eltwise()
        self.r2 = nn.ReLU()
        self.head = _Head(8)

    def forward(self, x):
        a = self.r1(self.c1(x))
        e = self.r2(self.elt(self.c2(a), a))
        return self.head(a), e


@gpu
def test_fused_op_outside_care_op_type_takes_no_max(tmp_path):
    batches = [(torch.randn(4, 3, 12, 12, generator=torch.Generator().manual_seed(30 + i)).cuda(), None)
               for i in range(2)]
    a, _, launches, reduced = _fused_and_unfused(tmp_path, _TwoHeadNet().eval(), batches, (1, 3, 12, 12),
                                                 care=["Conv2d", "Linear", "Concat"])
    assert a["top_feat_names"] == ["image", "Conv2d_1", "Conv2d_3", "Linear_8"]
    assert launches == {"conv_epilogue": 4, "eltwise": 2}
    assert reduced == [{"Conv2d_1", "Conv2d_3"}] * 2


# ---------------------------------------------------------------------------- the plan, on a CPU trace
class _PlanNet(nn.Module):
    def __init__(self):
        super().__init__()
        from common.quantity import Eltwise
        self.a = nn.Conv2d(3, 8, 3, padding=1)                                  # fused, with its ReLU
        self.ra = nn.ReLU()
        self.shared = nn.Conv2d(8, 8, 1)                                        # fires twice
        self.nobias = nn.Conv2d(8, 8, 1, bias=False)
        self.reflect = nn.Conv2d(8, 8, 3, padding=1, padding_mode="reflect")
        self.b = nn.Conv2d(8, 8, 1)                                             # its output is modified in place
        self.rb = nn.ReLU(inplace=True)
        self.elt = Eltwise()                                                    # fused, with its ReLU
        self.re = nn.ReLU()
        self.c = nn.Conv2d(8, 8, 1)                                             # fused; two ReLU consumers
        self.r1 = nn.ReLU()
        self.r2 = nn.ReLU()

    def forward(self, x):
        a = self.ra(self.a(x))
        b = self.rb(self.b(self.reflect(self.nobias(self.shared(self.shared(a))))))
        c = self.c(self.re(self.elt(b, a)))
        return self.r1(c) + self.r2(c)


def test_fusion_plan_on_a_cpu_trace():
    import tools
    q = tools.Quantity.__new__(tools.Quantity)          # the tracer alone: Quantity() itself needs a GPU
    settings = tools._config.load_tool_config(None)["SETTINGS"]
    q._all_op_type, q._cared_op_type = settings["ALL_OP_TYPE"], settings["CARE_OP_TYPE"]
    q._allow_same_tid_op_type = settings["ALLOW_SAME_TID_OP_TYPE"]
    q.cuda_device = torch.device("cpu")
    net = _PlanNet().eval()
    q.build_net_structure(net, (1, 3, 8, 8))
    assert q._inplace_modified == {"Conv2d_7"}
    plan = q._fusion_plan
    assert list(plan) == ["Conv2d_1", "Eltwise_9", "Conv2d_11"]
    assert plan["Conv2d_1"] == (net.a, net.ra)
    assert plan["Eltwise_9"] == (net.elt, net.re)
    assert plan["Conv2d_11"] == (net.c, None)

"""GPU parity with ZERO tolerance against the reference's results on a B200, stored under tests/golden/.

These tests used to run the UNMODIFIED reference live in a subprocess (baseline/ref_runner.py ``--device gpu``,
quantity/test/user_configs.yml:24, quantity/tools/pytorch_quantizer.py:43-45,291-292): same seeds, same batch
shapes, TF32 off, deterministic algorithms, no autotuning in both arms, so that the fp32 forward is the SAME cuDNN
forward and everything downstream must be identical.  The reference's source is not part of this repository, so
what those runs were compared against is stored as ``vs_reference_<model>.npz`` (tests/golden/gen_vs_reference.py):

  * calibration (quantity/tools/pytorch_quantizer.py:345-489, :592-677): tracer output, per-tensor maxima,
    intervals, the md5 of every merged 2048-bin histogram, thresholds, feat.table, weight.table and the md5 of
    every weight / bias JSON after weight_quantize and after the example script's second rewrite_weight;
  * ReconTest (fake-quant) and ReconModel (integer simulation) forwards: the md5 of every rebuilt layer's output
    (quantity/common/quantity/new_quantity_op.py:124-133, :197-205, :166-174, :280-292, :376-389) with a seeded
    sample of its values, and the logits.

The files were recorded from this repository on a B200 at the commit whose outputs last equalled the reference's
live GPU run in every one of these checks (profiles/r02_pytest_gpu_365.log).  Independently of the CUDA kernels, the
generator recomputed with the CPU oracle (oracle/pq_oracle.py, held to the reference's own golden runs by
tests/test_oracle.py) every calibration statistic, feat.table and every ReconModel layer output before storing them;
each file records that count and the GPU / torch / CUDA / cuDNN versions it was recorded on ("oracle_checked",
"recorded_on").

ReconModel and cuDNN.  The reference expresses int8 x int8 -> int32 as an fp32 ``nn.Conv2d`` on integer-valued
tensors (new_quantity_op.py:124-133), which IS integer arithmetic only if the library's convolution is exact on
integers.  On a GPU, cuDNN picks fp32 Winograd for the 3x3 stride-1 layers, whose transforms are not exact, so the
reference arm these layers equal is its ReconModel forward with ``torch.backends.cudnn`` disabled (ATen's GEMM
convolution, exact below 2^24): hence the name ``ReconModel:nocudnn``.  The layer test re-establishes that
condition on the spot: every NewConv2d / NewLinear's integer operands give the same accumulator in fp32 with cuDNN
disabled as in float64, and no accumulator reaches 2^24.
"""
import hashlib
import os

import numpy as np
import pytest
import torch

import ref_models
from conftest import golden_json, load_golden

pytestmark = pytest.mark.gpu

# model -> (calibration batches x batch size, rebuilt models, evaluation batch)
PLAN = {
    "tiny": ("3x2", ("ReconModel:nocudnn", "ReconTest"), 4),
    "lenet": ("4x8", ("ReconModel:nocudnn", "ReconTest"), 16),
    "r18": ("8x8", ("ReconModel:nocudnn", "ReconTest"), 8),   # BASELINE config 1 (64 images) + config 2 at B = 8
    "r50": ("2x4", ("ReconModel:nocudnn",), 8),               # config 3 / 4 topology at a small size
}
BIT_KEYS = ("weight_bit", "bias_bit", "output_bit", "input_bit")
LAYER_TYPES = ("NewConv2d", "NewLinear", "NewAdd", "TestConv", "TestLinear")
SAMPLE = 64           # values kept per layer output, at seeded positions, to report how far a mismatch is off


def hist_digest(d):
    """md5 of a histogram as float64 bytes: equal digests mean ``np.array_equal`` histograms."""
    return hashlib.md5(np.asarray(d, dtype=np.float64).tobytes()).hexdigest()


def golden_name(name):
    return "vs_reference_%s.npz" % name


def _golden(name):
    g = load_golden(golden_name(name))
    return g, golden_json(g)


def _configs(workdir, input_shape, max_cali):
    import tools._config as tc
    cfg = tc.load_tool_config(os.path.join(os.path.dirname(tc.__file__), "configs.yml"))
    wd = str(workdir)
    cfg["OUTPUT"] = {"WORK_DIR": wd, "WEIGHT_BIT_TABLE": wd + "/weight.table",
                     "FEAT_BIT_TABLE": wd + "/feat.table", "WEIGHT_DIR": wd + "/weight",
                     "BIAS_DIR": wd + "/bias", "FINAL_WEIGHT_DIR": wd + "/new_weight",
                     "FINAL_BIAS_DIR": wd + "/new_bias"}
    cfg["SETTINGS"]["MAX_CALI_IMG_NUM"] = max_cali
    user = tc.load_user_config({"PATH": {}, "MODEL": {"INPUT_SHAPE": ",".join(map(str, input_shape))},
                                "PRE_PROCESS": {"IMG": 1}, "SETTINGS": {"DEVICE": "gpu", "GPU": 0}})
    return cfg, user


def _snapshot(cfg):
    out = cfg["OUTPUT"]
    snap = {"feat.table": open(out["FEAT_BIT_TABLE"]).read(), "weight.table": open(out["WEIGHT_BIT_TABLE"]).read()}
    for key, sub in (("WEIGHT_DIR", "weight"), ("BIAS_DIR", "bias"), ("FINAL_WEIGHT_DIR", "new_weight"),
                     ("FINAL_BIAS_DIR", "new_bias")):
        for fn in sorted(os.listdir(out[key])):
            snap[sub + "/" + fn] = hashlib.md5(open(os.path.join(out[key], fn), "rb").read()).hexdigest()
    return snap


def calibrate(name, workdir):
    """The whole calibration job of PLAN[name] through this repository's tools: activation_quantize, weight_quantize
    and the example script's second rewrite_weight.  Returns (Quantity, last_calibration, snapshot after
    weight_quantize, snapshot after the second rewrite)."""
    import common.quantity as cq
    import tools
    ref_models.set_deterministic()
    n_batches, batch = (int(v) for v in PLAN[name][0].split("x"))
    cfg, user = _configs(workdir, ref_models.INPUT_SHAPE[name], n_batches - 1)
    with torch.no_grad():
        net = cq.merge_bn(ref_models.build_model(name), "cpu")
        q = tools.Quantity(net, config=cfg, user_config=user, verbose=False)
        q.activation_quantize(ref_models.calib_batches(name, n_batches, batch))
        cal = q.last_calibration
        q.weight_quantize()
        snap1 = _snapshot(cfg)
        q.rewrite_weight()
        snap2 = _snapshot(cfg)
    return q, cal, snap1, snap2


def rebuilt(name, mode, tables, workdir, pipeline=False):
    """This repository's Reconstruction on the given feat.table / weight.table.  Returns (model, quantity
    information)."""
    import tools
    os.makedirs(workdir, exist_ok=True)
    cfg, _user = _configs(workdir, ref_models.INPUT_SHAPE[name], 0)
    open(cfg["OUTPUT"]["FEAT_BIT_TABLE"], "w").write(tables["feat.table"])
    open(cfg["OUTPUT"]["WEIGHT_BIT_TABLE"], "w").write(tables["weight.table"])
    net = ref_models.build_model(name)
    r = tools.Reconstruction(net, config=cfg)
    r.merge_bn()
    net.eval()
    info = r.get_quantity_information()
    model = getattr(r, mode)(info, os.path.join(workdir, mode + ".pth")).cuda()
    if pipeline:
        from common.quantity.int8_pipeline import enable_int8_pipeline
        enable_int8_pipeline(model)
    return model, info


def exactness(m, xin):
    """The reference's ReconModel computes int8 x int8 as an fp32 ``nn.Conv2d`` / ``nn.Linear`` on integer-valued
    operands; with cuDNN disabled that is exact as long as every accumulator stays below 2^24.  This evaluates the
    layer's operands (its input quantiser and integer weights) both ways: the fp32 library result with cuDNN disabled
    against float64."""
    import torch.nn.functional as F
    xq = m.Quan(xin)
    with torch.backends.cudnn.flags(enabled=False):
        if type(m).__name__ == "NewConv2d":
            c = m.Conv
            got = F.conv2d(xq, c.weight, None, c.stride, c.padding, c.dilation, c.groups)
            want = F.conv2d(xq.double(), c.weight.double(), None, c.stride, c.padding, c.dilation, c.groups)
        else:
            got = F.linear(xq, m.Linear.weight)
            want = F.linear(xq.double(), m.Linear.weight.double())
    return {"inexact_fraction": float((got.double() != want).double().mean()),
            "max_abs_acc": float(want.abs().max())}


def layer_outputs(name, spec, tables, workdir, self_check=False):
    """Forward of the rebuilt model on the evaluation batch.  Returns ({layer: (md5, sample)} in forward order,
    logits, quantity information, {layer: exactness(...)} of every NewConv2d / NewLinear when ``self_check``).  The
    md5 is over the output's float32 bytes with -0.0 folded into 0.0, so equal digests mean ``torch.equal``
    outputs."""
    ref_models.set_deterministic()
    outs, checks = {}, {}

    def keep(lname):
        def _h(m, i, o):
            a = (o.detach() + 0.0).cpu().numpy()
            idx = np.random.default_rng(0).integers(0, a.size, SAMPLE)
            outs[lname] = (hashlib.md5(a.tobytes()).hexdigest(), a.reshape(-1)[idx])
            if self_check and type(m).__name__ in ("NewConv2d", "NewLinear"):
                checks[lname] = exactness(m, i[0])
        return _h

    with torch.no_grad():
        model, info = rebuilt(name, spec.split(":")[0], tables, workdir)
        for lname, mod in model.named_modules():
            if type(mod).__name__ in LAYER_TYPES:
                mod.register_forward_hook(keep(lname))
        y = model(ref_models.eval_batch(name, PLAN[name][2]).cuda())
    return outs, y.cpu(), info, checks


def _check_bits(info, ref):
    for lname, d in ref["quantity_information"].items():
        for key in BIT_KEYS:
            assert info[lname][key] == d[key], (lname, key)


@pytest.mark.parametrize("name", ["tiny", "lenet", "r18", "r50"])
def test_calibration_byte_identical_to_reference_on_gpu(name, tmp_path):
    _g, ref = _golden(name)
    q, cal, snap1, snap2 = calibrate(name, tmp_path / "workdir")
    assert dict(q.net_info) == ref["net_info"] and list(q.net_info) == list(ref["net_info"])
    assert q.cared_op_layer_names == ref["cared_op_layer_names"]
    assert q.get_merge_groups(q.net_info) == ref["merge_groups"]
    top = cal["top_feat_names"]
    assert top == ["image"] + list(ref["net_info"])
    for n in top:                                              # statistics: exact
        assert float(cal["max_vals"][n]) == ref["max_vals"][n], ("max", n)
        assert float(cal["intervals"][n]) == ref["intervals"][n], ("interval", n)
        d = cal["distributions"][n]
        assert hist_digest(d) == ref["dist_md5"][n], ("histogram", n, float(np.sum(d)), ref["dist_total"][n])
        assert float(cal["thresholds"][n]) == ref["thresholds"][n], ("threshold", n)
    assert snap1 == ref["after_weight_quantize"]               # tables as text, every JSON by md5: zero tolerance
    assert snap2 == ref["after_second_rewrite"]


@pytest.mark.parametrize("name,spec", [("tiny", "ReconTest"), ("tiny", "ReconModel:nocudnn"), ("lenet", "ReconTest"),
                                       ("lenet", "ReconModel:nocudnn"), ("r18", "ReconTest"),
                                       ("r18", "ReconModel:nocudnn"), ("r50", "ReconModel:nocudnn")])
def test_rebuilt_model_layers_equal_reference_on_gpu(name, spec, tmp_path):
    g, ref = _golden(name)
    outs, y, info, checks = layer_outputs(name, spec, ref["after_second_rewrite"], str(tmp_path / "workdir"),
                                          self_check=spec == "ReconModel:nocudnn")
    _check_bits(info, ref)
    names = list(ref[spec + "/layer_md5"])                     # forward order
    assert list(outs) == names and len(names) > 0
    for lname in names:
        md5, sample = outs[lname]
        want = g[spec + "/sample/" + lname]
        assert md5 == ref[spec + "/layer_md5"][lname], (spec, lname, float(np.abs(sample - want).max()),
                                                       float((sample != want).mean()))
    assert torch.equal(y, torch.from_numpy(g[spec + "/y"]))
    # the reference arm these layers equal is exact integer arithmetic: every accumulator exact, far below 2^24
    assert len(checks) > 0 or spec != "ReconModel:nocudnn"
    for lname, sc in checks.items():
        assert sc["inexact_fraction"] == 0.0 and sc["max_abs_acc"] < 2 ** 24, (lname, sc)


@pytest.mark.parametrize("name", ["tiny", "r18", "r50"])
def test_int8_pipeline_logits_equal_reference_on_gpu(name, tmp_path):
    """The opt-in int8 inter-layer pipeline (SURVEY 8f n1) against the reference's ReconModel logits."""
    g, ref = _golden(name)
    ref_models.set_deterministic()
    with torch.no_grad():
        model, info = rebuilt(name, "ReconModel", ref["after_second_rewrite"], str(tmp_path / "workdir"),
                              pipeline=True)
        _check_bits(info, ref)
        y = model(ref_models.eval_batch(name, PLAN[name][2]).cuda())
    assert torch.equal(y.float().cpu(), torch.from_numpy(g["ReconModel:nocudnn/y"]))


"""Record tests/golden/vs_reference_<model>.npz, what tests/test_gpu_vs_reference.py compares against.

    python tests/golden/gen_vs_reference.py [--out DIR] [model ...]

Needs a B200: the values are those of the cuDNN fp32 forward and this repository's kernels on that GPU.  Run it only
from a tree whose outputs equal the reference's (the files were recorded at such a commit, see the test module); a
file recorded from a tree that computes something else would turn the tests into a check against that tree.  To
catch that, every value that the CPU oracle (oracle/pq_oracle.py, the restatement of the reference's arithmetic that
tests/test_oracle.py holds to the reference's own golden runs) can compute is recomputed by it, independently of the
CUDA kernels, and the file is not written unless all of them agree:
  * calibration: the same fp32 forward's hooked activations through oracle.calibrate give the maxima, intervals,
    histograms, thresholds and feat.table;
  * ReconModel: every NewConv2d / NewLinear / NewAdd output from that layer's own input through the oracle's
    int_conv_layer / int_linear_layer / add_clamp.
The software stack and GPU of the recording are stored beside the values ("recorded_on").

Per model: one ``json`` entry (tracer output, merge groups, per-tensor maxima / intervals / thresholds, the md5 and
total count of every merged histogram, the tables as text and the md5 of every weight / bias JSON, the per-layer
quantity information and output md5 of each rebuilt model), each rebuilt model's logits and a seeded sample of every
layer output.
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np
import torch

GOLDEN = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(GOLDEN)
REPO = os.path.dirname(TESTS)
for p in (os.path.join(REPO, "pytorch-quantity_b200"), REPO, TESTS):
    if p not in sys.path:
        sys.path.insert(0, p)

import test_gpu_vs_reference as t  # noqa: E402


def oracle_calibration(name, net_info, cared, workdir):
    """Maxima, intervals, histograms, thresholds and feat.table lines of the CPU oracle on the hooked activations of
    the same fp32 forward (a fresh copy of the model, the same batches)."""
    import common.quantity as cq
    import ref_models
    import tools
    from oracle import pq_oracle as oracle
    oracle.build()
    ref_models.set_deterministic()
    n_batches, batch = (int(v) for v in t.PLAN[name][0].split("x"))
    cfg, user = t._configs(workdir, ref_models.INPUT_SHAPE[name], n_batches - 1)
    top = ["image"] + list(net_info)
    feats = []
    with torch.no_grad():
        q = tools.Quantity(cq.merge_bn(ref_models.build_model(name), "cpu"), config=cfg, user_config=user,
                           verbose=False)
        named, hooks = q.regist_hook_outfeature(q.model)
        for x, _ in ref_models.calib_batches(name, n_batches, batch):
            q._forward_device(q.model, x.cuda())
            feats.append({n: named[n].detach().cpu().numpy().reshape(-1) for n in top})
        for h in hooks:
            h.remove()
    r = oracle.calibrate(feats, top, net_info, q.get_merge_groups(q.net_info), return_all=True)
    lines = oracle.feat_table_lines(top, cared, net_info, r["bits"])
    return r, "\n".join(lines) + "\n"


def oracle_layers(name, tables, workdir):
    """Number of ReconModel layers checked: each NewConv2d / NewLinear / NewAdd output against the oracle evaluated
    on that layer's own input."""
    from oracle import pq_oracle as oracle
    ref_models = t.ref_models
    ref_models.set_deterministic()
    bad, n = [], 0
    with torch.no_grad():
        model, _info = t.rebuilt(name, "ReconModel", tables, workdir)

        def check(lname):
            def _h(m, i, o):
                nonlocal n
                got = o.detach().cpu().numpy()
                kind = type(m).__name__
                if kind == "NewAdd":
                    want = oracle.add_clamp(i[0].cpu().numpy(), i[1].cpu().numpy())
                else:
                    info = {k: getattr(m, k) for k in t.BIT_KEYS}
                    w = m.weight.detach().cpu().numpy()
                    b = None if m.bias is None else m.bias.detach().cpu().numpy()
                    x = i[0].detach().cpu().numpy()
                    if kind == "NewConv2d":
                        c = m.Conv
                        want, _y = oracle.int_conv_layer(x, w, b, info, c.stride, c.padding, c.dilation, c.groups)
                    else:
                        want, _y = oracle.int_linear_layer(x, w, b, info)
                n += 1
                if not np.array_equal(got, want):
                    bad.append(lname)
            return _h

        for lname, mod in model.named_modules():
            if type(mod).__name__ in ("NewConv2d", "NewLinear", "NewAdd"):
                mod.register_forward_hook(check(lname))
        model(ref_models.eval_batch(name, t.PLAN[name][2]).cuda())
    assert n > 0 and not bad, ("ReconModel layers differ from the oracle", bad)
    return n


def record(name, workdir):
    q, cal, snap1, snap2 = t.calibrate(name, os.path.join(workdir, "calib"))
    res = {"net_info": {k: {"inputs": v["inputs"], "type": v["type"]} for k, v in q.net_info.items()},
           "cared_op_layer_names": q.cared_op_layer_names, "merge_groups": q.get_merge_groups(q.net_info),
           "after_weight_quantize": snap1, "after_second_rewrite": snap2}
    arrays = {}
    for key in ("max_vals", "intervals", "thresholds"):
        res[key] = {n: float(v) for n, v in cal[key].items()}
    res["dist_md5"] = {n: t.hist_digest(d) for n, d in cal["distributions"].items()}
    res["dist_total"] = {n: float(np.sum(d)) for n, d in cal["distributions"].items()}
    r, feat_table = oracle_calibration(name, res["net_info"], q.cared_op_layer_names, os.path.join(workdir, "oracle"))
    for n in cal["top_feat_names"]:
        assert float(r["max_vals"][n]) == res["max_vals"][n], ("oracle max", n)
        assert float(r["intervals"][n]) == res["intervals"][n], ("oracle interval", n)
        assert t.hist_digest(r["dists"][n]) == res["dist_md5"][n], ("oracle histogram", n)
        assert float(r["thresholds"][n]) == res["thresholds"][n], ("oracle threshold", n)
    assert feat_table == snap1["feat.table"], "oracle feat.table"
    res["oracle_checked"] = {"calibration_tensors": len(cal["top_feat_names"]),
                             "reconmodel_layers": oracle_layers(name, snap2, os.path.join(workdir, "oracle_rm"))}
    res["recorded_on"] = {"gpu": torch.cuda.get_device_name(0), "torch": torch.__version__,
                          "cuda": torch.version.cuda, "cudnn": torch.backends.cudnn.version()}
    for spec in t.PLAN[name][1]:
        outs, y, info, _checks = t.layer_outputs(name, spec, snap2, os.path.join(workdir, spec.replace(":", "_")))
        res[spec + "/layer_md5"] = {lname: md5 for lname, (md5, _s) in outs.items()}
        for lname, (_m, sample) in outs.items():
            arrays[spec + "/sample/" + lname] = sample
        arrays[spec + "/y"] = y.numpy()
        res["quantity_information"] = {k: {key: v[key] for key in t.BIT_KEYS} for k, v in info.items()}
    arrays["json"] = np.frombuffer(json.dumps(res).encode(), dtype=np.uint8)
    return arrays


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=GOLDEN)
    ap.add_argument("models", nargs="*", default=list(t.PLAN))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the golden values are those of a B200"
    os.makedirs(args.out, exist_ok=True)
    for name in args.models:
        with tempfile.TemporaryDirectory(prefix="pq_gen_vs_ref_") as wd:
            arrays = record(name, wd)
        path = os.path.join(args.out, t.golden_name(name))
        np.savez_compressed(path, **arrays)
        print("%s: %d arrays, %.0f kB" % (path, len(arrays), os.path.getsize(path) / 1e3), flush=True)


if __name__ == "__main__":
    main()

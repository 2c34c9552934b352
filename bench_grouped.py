#!/usr/bin/env python
"""Grouped convolutions of the integer simulation: the distinct grouped 3 x 3 layers of ResNeXt-50 32x4d (224 x 224)
one by one, and the whole ResNeXt-50 ReconModel forward.

    python bench_grouped.py [--batch 512] [--iters 20] [--group-batch 32] [--no-model] [--out FILE]

Per layer (plain NewConv2d, seeded weights, fixed bits), at --batch:
  s8       int8 NHWC in -> int8 NHWC out with the following nn.ReLU fused, the pipeline form (NewConv2d._run)
  f32      int8 NHWC in -> fp32 NCHW out (the module boundary)
  groups   the per-group path (one NewConv2d per group, as a model pickled before the grouped kernel runs it),
           fp32 NCHW in and out, at --group-batch images and scaled to --batch
Each time is the mean over --iters launches timed one by one with CUDA events, the 256 MB L2 flush buffer rewritten
before each launch.  Useful int8 ops 2 * M * K * R * S * Cg; the tensor cores issue group_block / Kg times as many
when Kg < group_block ("MMA ops").  Algorithmic bytes of the s8 form: the input image once and the output once; the
HBM floor is those bytes over a device-to-device copy peak measured in the same process.

Whole model (unless --no-model): ResNeXt-50 calibrated with tools.Quantity on two seeded batches of 4, then the
ReconModel forward at --batch images: fp32 boundary, int8 pipeline eager and GraphedForward, with this library's
launches per forward.
"""
import argparse
import copy
import os
import sys
import tempfile

import torch
import torch.nn as nn

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "pytorch-quantity_b200")
for p in (PKG, REPO):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_depthwise import card, copy_peak, timed          # noqa: E402  (same card line, copy peak and L2 flush)

# (input H = W, channels, stride, layers of that shape) of the grouped 3 x 3 layers of ResNeXt-50 32x4d at 224 x 224
GROUPED_LAYERS = [(56, 128, 1, 3), (56, 256, 2, 1), (28, 256, 1, 3), (28, 512, 2, 1), (14, 512, 1, 5),
                  (14, 1024, 2, 1), (7, 1024, 1, 2)]
GROUPS = 32
INFO = {"weight_bit": 8, "input_bit": 5, "output_bit": 4, "bias_bit": 4}


def layer_table(batch, group_batch, iters, peak, lines):
    from common.quantity import NewConv2d
    lines.append("per layer: batch %d (groups: batch %d, scaled), mean of %d launches, L2 flushed before each" % (
        batch, group_batch, iters))
    lines.append("%-3s %-15s %3s %4s %9s %9s %10s %9s %9s %11s %8s %6s" % (
        "#", "HxW C s", "n", "blk", "s8 ms", "f32 ms", "groups ms", "Gop", "MMA Gop", "bytes s8", "TOP/s", "floor%"))
    tot = {"s8": 0.0, "f32": 0.0, "groups": 0.0, "bytes": 0, "ops": 0}
    for i, (hw, c, s, n) in enumerate(GROUPED_LAYERS):
        g = torch.Generator().manual_seed(200 + i)
        conv = nn.Conv2d(c, c, 3, s, 1, groups=GROUPS)
        with torch.no_grad():
            conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.1)
            conv.bias.copy_(torch.randn(c, generator=g) * 0.5)
        conv_old = copy.deepcopy(conv)
        mod = NewConv2d(conv.cuda(), dict(INFO)).eval()
        blk = mod._group_block
        p = (hw + 2 - 3) // s + 1
        cg = kg = c // GROUPS
        ops = 2 * batch * p * p * c * 9 * cg
        mma_ops = ops * max(1, blk // kg)
        nbytes = batch * c * (hw * hw + p * p)
        x = torch.randint(-128, 128, (batch, hw, hw, c), generator=g, dtype=torch.int32).to(torch.int8).cuda()
        row = {}
        with torch.no_grad():
            row["s8"] = timed(lambda: mod._run(x, False, True, True), iters)
            row["f32"] = timed(lambda: mod._run(x, True, False, False), iters)
        del x
        # the per-group path on the same layer
        old = NewConv2d(conv_old.cuda(), dict(INFO)).eval()
        del old._group_block, old._w_krsc
        old._payload_channels = None
        old._build_groups(old.Conv, old.Conv.weight.detach())
        xf = torch.randn(group_batch, c, hw, hw, generator=g).cuda()
        with torch.no_grad():
            row["groups"] = timed(lambda: old(xf), max(3, iters // 4)) * batch / group_batch
        del xf, old
        floor = nbytes / peak
        lines.append("%-3d %-15s %3d %4d %9.4f %9.4f %10.2f %9.1f %9.1f %11d %8.1f %6.1f" % (
            i, "%dx%d %d %d" % (hw, hw, c, s), n, blk, row["s8"] * 1e3, row["f32"] * 1e3, row["groups"] * 1e3,
            ops / 1e9, mma_ops / 1e9, nbytes, ops / row["s8"] / 1e12, 100 * floor / row["s8"]))
        for k in ("s8", "f32", "groups"):
            tot[k] += n * row[k]
        tot["bytes"] += n * nbytes
        tot["ops"] += n * ops
        torch.cuda.empty_cache()
    floor = tot["bytes"] / peak
    lines.append("all 16 layers (shape x n): s8+relu %.3f ms, f32 %.3f ms, per-group path %.1f ms; %.1f G useful int8 "
                 "ops, %.3f GB int8 in + out" % (tot["s8"] * 1e3, tot["f32"] * 1e3, tot["groups"] * 1e3,
                                                tot["ops"] / 1e9, tot["bytes"] / 1e9))
    lines.append("HBM floor at the measured copy peak %.3f ms; s8+relu / floor = %.2f" % (
        floor * 1e3, tot["s8"] / floor))


def whole_model(batch, iters, lines):
    sys.path.insert(0, os.path.join(PKG, "test"))
    import _models
    import tools
    from common.quantity import GraphedForward, _native, enable_int8_pipeline, merge_bn
    wd = tempfile.mkdtemp(prefix="pq_bench_grouped_")
    cfg, user = _models.configs(wd, (3, 224, 224), 2)
    with torch.no_grad():
        net, _ = _models.build("resnext50_32x4d")
        q = tools.Quantity(merge_bn(net, "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize([(torch.randn(4, 3, 224, 224, generator=torch.Generator().manual_seed(1 + i)), None)
                               for i in range(2)])
        q.weight_quantize()
        r = tools.Reconstruction(_models.build("resnext50_32x4d")[0], config=cfg)
        r.merge_bn()
        model = r.ReconModel(r.get_quantity_information(), None).cuda().eval()
        x = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(7)).cuda()
        res = {}
        for name, pipe in (("fp32 boundary", False), ("int8 pipeline", True)):
            enable_int8_pipeline(model, pipe)
            ref = model(x)
            l0 = _native.LAUNCHES["total"]
            model(x)
            launches = _native.LAUNCHES["total"] - l0
            res[name] = ref
            lines.append("%-16s %9.3f ms/forward, %d launches of this library" % (
                name, timed(lambda: model(x), iters) * 1e3, launches))
        assert torch.equal(res["fp32 boundary"], res["int8 pipeline"])
        fwd = GraphedForward(model, x)
        assert torch.equal(fwd(x), res["int8 pipeline"])
        lines.append("%-16s %9.3f ms/forward, %d launches of this library in the graph" % (
            "GraphedForward", timed(lambda: fwd(x), iters) * 1e3, fwd.launches))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--group-batch", type=int, default=32, help="batch of the per-group path column (scaled)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--no-model", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_grouped.py needs a GPU")
    torch.backends.cudnn.benchmark = False
    peak = copy_peak()
    lines = ["card: %s" % card(), "copy peak (1 GiB device-to-device, read + write): %.2f TB/s" % (peak / 1e12)]
    layer_table(args.batch, args.group_batch, args.iters, peak, lines)
    if not args.no_model:
        lines.append("ResNeXt-50 32x4d ReconModel, batch %d, 224 x 224:" % args.batch)
        whole_model(args.batch, max(5, args.iters // 4), lines)
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

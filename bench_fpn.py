#!/usr/bin/env python
"""Nearest-neighbour upsampling in the integer simulation: the semantic FPN (model/fpn) end to end, and the two kernels
that read an upsampled operand through index tables.

    python bench_fpn.py [--batch 16] [--hw 512] [--iters 20] [--out FILE]

Whole model: the FPN calibrated with tools.Quantity on two seeded batches of 2, then the ReconModel forward at --batch
images of --hw x --hw: fp32 boundary, int8 pipeline eager and GraphedForward (the output read as fp32 each time), with
this library's launches per forward; the three outputs must be equal.

Kernels, at the FPN's own shapes for --batch images: each top-down add (int8 lateral + int16 sum of the level above,
read x2 through the tables; int16 sum and int8 out written) and the head Concat (four 128-channel levels, three of them
read x2 / x4 / x8 through the tables, written as the 512-channel int8 operand of the fuse convolution).  Each time is
the mean over --iters launches timed one by one with CUDA events, the 256 MB L2 flush buffer rewritten before each.
Algorithmic bytes: each operand read once at its own resolution and each output written once; GB/s over the kernel
time and its fraction of a device-to-device copy measured in the same process.
"""
import argparse
import os
import sys
import tempfile

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "pytorch-quantity_b200")
for p in (PKG, REPO):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_depthwise import card, copy_peak, timed   # noqa: E402


def kernel_table(batch, hw, iters, peak, lines):
    from common.quantity import _native, int8_pipeline
    g = torch.Generator(device="cuda").manual_seed(3)

    def s8(*shape):
        return torch.randint(-128, 128, shape, dtype=torch.int32, device="cuda", generator=g).to(torch.int8)

    def s16(*shape):
        return torch.randint(-128 * 16, 127 * 16 + 1, shape, dtype=torch.int32, device="cuda",
                             generator=g).to(torch.int16)

    def tables(h, w, scale):
        req = int8_pipeline.nearest_request(4, scale_factor=scale)
        t = int8_pipeline.nearest_tables((h, w), req, torch.device("cuda"))
        return t.map_h, t.map_w

    lines.append("kernels: batch %d at %d x %d, mean of %d launches, L2 flushed before each" % (batch, hw, hw, iters))
    lines.append("%-34s %10s %12s %9s %7s" % ("kernel", "ms", "bytes", "GB/s", "copy%"))
    for level, side in (("P4", hw // 16), ("P3", hw // 8), ("P2", hw // 4)):
        lat, up = s8(batch, side, side, 256), s16(batch, side // 2, side // 2, 256)
        mh, mw = tables(side // 2, side // 2, 2)
        nbytes = lat.numel() * (1 + 2 + 1) + up.numel() * 2
        t = timed(lambda: _native.add_requant_nearest(lat, 3, False, up, 4, False, mh, mw, 2), iters)
        lines.append("%-34s %10.4f %12d %9.0f %7.1f" % ("add_requant_nearest %s (%dx%d)" % (level, side, side),
                                                         t * 1e3, nbytes, nbytes / t / 1e9, 100 * nbytes / t / peak))
    side = hw // 4
    srcs, nbytes = [], 0
    for f in (1, 2, 4, 8):
        x = s8(batch, side // f, side // f, 128)
        srcs.append((x, 3, False, None if f == 1 else tables(side // f, side // f, f)))
        nbytes += x.numel()
    nbytes += batch * side * side * 512
    t = timed(lambda: _native.concat_requant_nearest_s8(srcs, (side, side), 2, 512), iters)
    lines.append("%-34s %10.4f %12d %9.0f %7.1f" % ("concat_requant_nearest head (%dx%d)" % (side, side), t * 1e3,
                                                     nbytes, nbytes / t / 1e9, 100 * nbytes / t / peak))


def whole_model(batch, hw, iters, lines):
    sys.path.insert(0, os.path.join(PKG, "test"))
    import _models
    import tools
    from common.quantity import GraphedForward, QTensor, _native, enable_int8_pipeline, merge_bn
    wd = tempfile.mkdtemp(prefix="pq_bench_fpn_")
    cfg, user = _models.configs(wd, (3, hw, hw), 2)
    plain = lambda y: y.dequantize() if isinstance(y, QTensor) else y     # read the output as fp32
    with torch.no_grad():
        net, _ = _models.build("fpn_r50")
        q = tools.Quantity(merge_bn(net, "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize([(torch.randn(2, 3, hw, hw, generator=torch.Generator().manual_seed(1 + i)), None)
                               for i in range(2)])
        q.weight_quantize()
        r = tools.Reconstruction(_models.build("fpn_r50")[0], config=cfg)
        r.merge_bn()
        model = r.ReconModel(r.get_quantity_information(), None).cuda().eval()
        x = torch.randn(batch, 3, hw, hw, generator=torch.Generator().manual_seed(7)).cuda()
        res = {}
        for name, pipe in (("fp32 boundary", False), ("int8 pipeline", True)):
            enable_int8_pipeline(model, pipe)
            res[name] = plain(model(x)).clone()
            l0 = _native.LAUNCHES["total"]
            plain(model(x))
            launches = _native.LAUNCHES["total"] - l0
            lines.append("%-16s %9.3f ms/forward, %d launches of this library" % (
                name, timed(lambda: plain(model(x)), iters) * 1e3, launches))
        assert torch.equal(res["fp32 boundary"], res["int8 pipeline"])
        fwd = GraphedForward(model, x)
        assert torch.equal(fwd(x), res["int8 pipeline"])
        lines.append("%-16s %9.3f ms/forward, %d launches of this library in the graph" % (
            "GraphedForward", timed(lambda: fwd(x), iters) * 1e3, fwd.launches))
        lines.append("outputs of the three forwards equal: yes")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--hw", type=int, default=512)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fpn.py needs a GPU")
    torch.backends.cudnn.benchmark = False
    peak = copy_peak()
    lines = ["card: %s" % card(), "copy peak (1 GiB device-to-device, read + write): %.2f TB/s" % (peak / 1e12)]
    kernel_table(args.batch, args.hw, args.iters, peak, lines)
    lines.append("semantic FPN (ResNet-50) ReconModel, batch %d, %d x %d:" % (args.batch, args.hw, args.hw))
    whole_model(args.batch, args.hw, max(5, args.iters // 4), lines)
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

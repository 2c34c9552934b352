#!/usr/bin/env python
"""Windowed average pooling in the integer simulation: the ResNet-50-D (model/resnet, deep stem and avg-down
shortcuts) end to end, and the kernel that pools a quantised payload straight into its consumer's int8 operand.

    python bench_resnetd.py [--batch 512] [--hw 224] [--iters 20] [--out FILE]

Kernels, at the three avg-down shapes for --batch images (the int16 Eltwise sums at 256 x 56^2, 512 x 28^2 and
1024 x 14^2 for 224^2 inputs, AvgPool2d(2, 2, ceil_mode=True, count_include_pad=False), a pending ReLU on load, int8
NHWC out): pq_avgpool_requant_s8 against what the pipeline ran before it for the same bytes in the same process --
de-quantise to fp32 NCHW (as QTensor.dequantize), F.avg_pool2d, then the consumer's Quantity(ib) into its NHWC operand
(pq_quantize_nchw_to_nhwc_s8) -- whose result must be equal.  Each time is the mean over --iters calls timed one by
one with CUDA events, the 256 MB L2 flush buffer rewritten before each.  Algorithmic bytes: the int16 payload read once
and the int8 operand written once; GB/s over the time and its fraction of a device-to-device copy measured in the same
process.

Whole model: ResNet-50-D calibrated with tools.Quantity on two seeded batches of 2, then the ReconModel forward at
--batch images of --hw x --hw: fp32 boundary, int8 pipeline eager and GraphedForward, with this library's launches per
forward; the three outputs must be equal.
"""
import argparse
import os
import sys
import tempfile

import torch
import torch.nn.functional as F

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "pytorch-quantity_b200")
for p in (PKG, REPO):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_depthwise import card, copy_peak, timed   # noqa: E402

WINDOW = (2, 2, 2, 2, 0, 0, 1, 0, 0)   # AvgPool2d(2, 2, ceil_mode=True, count_include_pad=False), as the kernel takes it


def kernel_table(batch, hw, iters, peak, lines):
    from common.quantity import _native
    g = torch.Generator(device="cuda").manual_seed(3)
    bit, ib = 4, 2
    lines.append("kernels: batch %d, int16 in at bit %d with a pending ReLU, int8 NHWC out at bit %d, mean of %d calls, "
                 "L2 flushed before each" % (batch, bit, ib, iters))
    lines.append("%-40s %10s %12s %9s %7s" % ("kernel", "ms", "bytes", "GB/s", "copy%"))
    for C, side in ((256, hw // 4), (512, hw // 8), (1024, hw // 16)):
        x = torch.randint(-128 * 16, 127 * 16 + 1, (batch, side, side, C), dtype=torch.int32, device="cuda",
                          generator=g).to(torch.int16)
        new = lambda: _native.avgpool_requant_s8(x, bit, True, WINDOW, ib, C)

        def parent():
            v = torch.relu(x.to(torch.float32) * (2.0 ** -bit)).permute(0, 3, 1, 2).contiguous()
            y = F.avg_pool2d(v, 2, 2, 0, True, False)
            return _native.quantize_nchw_to_nhwc_s8(y, ib, C)
        assert torch.equal(new(), parent()), (C, side)
        P = (side + 1) // 2
        nbytes = x.numel() * 2 + batch * P * P * C
        for name, fn in (("pq_avgpool_requant_s8", new), ("parent: dequantize+avg_pool2d+Quantity", parent)):
            t = timed(fn, iters)
            lines.append("%-40s %10.4f %12d %9.0f %7.1f" % ("%s %dx%d^2" % (name, C, side), t * 1e3, nbytes,
                                                             nbytes / t / 1e9, 100 * nbytes / t / peak))


def whole_model(batch, hw, iters, lines):
    sys.path.insert(0, os.path.join(PKG, "test"))
    import _models
    import tools
    from common.quantity import GraphedForward, QTensor, _native, enable_int8_pipeline, merge_bn
    from model.resnet import resnet50d_fabu
    from model.resnet.resnet_fabu import randomize_bn_

    def build():
        torch.manual_seed(0)
        net = resnet50d_fabu(in_hw=hw).eval()
        with torch.no_grad():
            randomize_bn_(net, 0)
        return net
    wd = tempfile.mkdtemp(prefix="pq_bench_resnetd_")
    cfg, user = _models.configs(wd, (3, hw, hw), 2)
    plain = lambda y: y.dequantize() if isinstance(y, QTensor) else y     # read the output as fp32
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build(), "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize([(torch.randn(2, 3, hw, hw, generator=torch.Generator().manual_seed(1 + i)), None)
                               for i in range(2)])
        q.weight_quantize()
        r = tools.Reconstruction(build(), config=cfg)
        r.merge_bn()
        model = r.ReconModel(r.get_quantity_information(), None).cuda().eval()
        x = torch.randn(batch, 3, hw, hw, generator=torch.Generator().manual_seed(7)).cuda()
        res = {}
        for name, pipe in (("fp32 boundary", False), ("int8 pipeline", True)):
            enable_int8_pipeline(model, pipe)
            res[name] = plain(model(x)).clone()
            l0 = dict(_native.LAUNCHES)
            plain(model(x))
            launches = _native.LAUNCHES["total"] - l0["total"]
            pools = _native.LAUNCHES.get("avgpool_requant", 0) - l0.get("avgpool_requant", 0)
            lines.append("%-16s %9.3f ms/forward, %d launches of this library (%d avgpool_requant)" % (
                name, timed(lambda: plain(model(x)), iters) * 1e3, launches, pools))
        assert torch.equal(res["fp32 boundary"], res["int8 pipeline"])
        fwd = GraphedForward(model, x)
        assert torch.equal(fwd(x), res["int8 pipeline"])
        lines.append("%-16s %9.3f ms/forward, %d launches of this library in the graph" % (
            "GraphedForward", timed(lambda: fwd(x), iters) * 1e3, fwd.launches))
        lines.append("outputs of the three forwards equal: yes")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--hw", type=int, default=224)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resnetd.py needs a GPU")
    torch.backends.cudnn.benchmark = False
    peak = copy_peak()
    lines = ["card: %s" % card(), "copy peak (1 GiB device-to-device, read + write): %.2f TB/s" % (peak / 1e12)]
    kernel_table(args.batch, args.hw, args.iters, peak, lines)
    lines.append("ResNet-50-D ReconModel, batch %d, %d x %d:" % (args.batch, args.hw, args.hw))
    whole_model(args.batch, args.hw, max(5, args.iters // 4), lines)
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

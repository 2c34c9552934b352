#!/usr/bin/env python
"""Depthwise convolutions of the integer simulation: the 17 depthwise layers of MobileNetV2 (224 x 224) one by one, and
the whole MobileNetV2 ReconModel forward.

    python bench_depthwise.py [--batch 512] [--iters 20] [--layer-batch-forward 512] [--no-model] [--out FILE]

Per layer (plain NewConv2d, seeded weights, fixed bits), at --batch:
  fwd      the module's fp32-boundary forward (fp32 NCHW in and out), at --layer-batch-forward images
  s8       int8 NHWC in -> int8 NHWC out, the pipeline form (NewConv2d._run on its own operand)
  s8+relu  the same with the following nn.ReLU fused, as the pipeline runs MobileNetV2
  f32      int8 NHWC in -> fp32 NCHW out (the module boundary)
Each time is the mean over --iters launches timed one by one with CUDA events, the 256 MB L2 flush buffer rewritten
before each launch.  Algorithmic bytes: the input image once and the output once (int8 1 B, fp32 4 B per element);
GB/s over the kernel time; fraction of a device-to-device copy peak measured in the same process.  A tree whose
NewConv2d has no int8 depthwise path (per-group path) reports only `fwd`.

Whole model (unless --no-model): MobileNetV2 calibrated with tools.Quantity on two seeded batches of 4, then the
ReconModel forward at --batch images: fp32 boundary, int8 pipeline eager and GraphedForward, with this library's
launches per forward.
"""
import argparse
import os
import subprocess
import sys
import tempfile

import torch
import torch.nn as nn

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "pytorch-quantity_b200")
for p in (PKG, REPO):
    if p not in sys.path:
        sys.path.insert(0, p)

# (input H = W, channels, stride) of the 3 x 3 depthwise layers of MobileNetV2 at 224 x 224, in network order
DW_LAYERS = ([(112, 32, 1), (112, 96, 2), (56, 144, 1), (56, 144, 2)] + [(28, 192, 1)] * 2 + [(28, 192, 2)]
             + [(14, 384, 1)] * 4 + [(14, 576, 1)] * 2 + [(14, 576, 2)] + [(7, 960, 1)] * 3)
INFO = {"weight_bit": 7, "input_bit": 4, "output_bit": 4, "bias_bit": 5}
HBM_COPY_PEAK_DESIGN = 6.46e12          # DESIGN.md section 6, for the computed floor


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name()


def copy_peak():
    """Bytes moved per second by a 1 GiB device-to-device copy (read + write)."""
    n = 1 << 30
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e9
    for _ in range(10):
        s.record(); b.copy_(a); e.record(); torch.cuda.synchronize()
        best = min(best, s.elapsed_time(e) / 1e3)
    return 2 * n / best


_FLUSH = None


def timed(fn, iters):
    """Mean seconds of fn() over iters launches, each after an L2 flush, each bracketed by its own events."""
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for s, e in ev:
        _FLUSH.fill_(1)
        s.record(); fn(); e.record()
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in ev) / iters / 1e3


def layer_table(batch, fwd_batch, iters, peak, lines):
    from common.quantity import NewConv2d
    has_dw = hasattr(NewConv2d, "_depthwise")
    lines.append("per layer: batch %d (fwd: batch %d), mean of %d launches, L2 flushed before each" % (
        batch, fwd_batch, iters))
    lines.append("%-3s %-13s %10s %10s %10s %10s %12s %9s %7s" % (
        "#", "HxW C s", "fwd ms", "s8 ms", "s8+relu ms", "f32 ms", "bytes s8", "GB/s s8r", "copy%"))
    tot = {"fwd": 0.0, "s8": 0.0, "s8r": 0.0, "f32": 0.0, "bytes": 0}
    for i, (hw, c, s) in enumerate(DW_LAYERS):
        g = torch.Generator().manual_seed(100 + i)
        conv = nn.Conv2d(c, c, 3, s, 1, groups=c)
        with torch.no_grad():
            conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.2)
            conv.bias.copy_(torch.randn(c, generator=g) * 0.5)
        mod = NewConv2d(conv.cuda(), dict(INFO)).eval()
        xf = torch.randn(fwd_batch, c, hw, hw, generator=g).cuda()
        with torch.no_grad():
            t_fwd = timed(lambda: mod(xf), max(3, iters // 4) if not has_dw else iters)
        del xf
        p = (hw + 2 - 3) // s + 1
        nbytes = batch * c * (hw * hw + p * p)
        row = {"fwd": t_fwd}
        if has_dw:
            x = torch.randint(-128, 128, (batch, hw, hw, c), generator=g, dtype=torch.int32).to(torch.int8).cuda()
            with torch.no_grad():
                row["s8"] = timed(lambda: mod._run(x, False, True, False), iters)
                row["s8r"] = timed(lambda: mod._run(x, False, True, True), iters)
                row["f32"] = timed(lambda: mod._run(x, True, False, False), iters)
            del x
            gbs = nbytes / row["s8r"]
            lines.append("%-3d %-13s %10.4f %10.4f %10.4f %10.4f %12d %9.0f %7.1f" % (
                i, "%dx%d %d %d" % (hw, hw, c, s), row["fwd"] * 1e3, row["s8"] * 1e3, row["s8r"] * 1e3,
                row["f32"] * 1e3, nbytes, gbs / 1e9, 100 * gbs / peak))
        else:
            lines.append("%-3d %-13s %10.4f %10s %10s %10s %12d" % (i, "%dx%d %d %d" % (hw, hw, c, s), t_fwd * 1e3,
                                                                 "-", "-", "-", nbytes))
        for k, v in row.items():
            tot[k] += v
        tot["bytes"] += nbytes
        torch.cuda.empty_cache()
    lines.append("sum: fwd %.3f ms (batch %d)" % (tot["fwd"] * 1e3, fwd_batch))
    if has_dw:
        floor = tot["bytes"] / peak
        lines.append("sum: s8 %.3f ms, s8+relu %.3f ms, f32 %.3f ms; %.3f GB int8 in + out" % (
            tot["s8"] * 1e3, tot["s8r"] * 1e3, tot["f32"] * 1e3, tot["bytes"] / 1e9))
        lines.append("HBM floor at the measured copy peak %.3f ms (at %.2f TB/s: %.3f ms); s8+relu / floor = %.2f" % (
            floor * 1e3, HBM_COPY_PEAK_DESIGN / 1e12, tot["bytes"] / HBM_COPY_PEAK_DESIGN * 1e3, tot["s8r"] / floor))


def whole_model(batch, iters, lines):
    sys.path.insert(0, os.path.join(PKG, "test"))
    import _models
    import tools
    from common.quantity import GraphedForward, _native, enable_int8_pipeline, merge_bn
    wd = tempfile.mkdtemp(prefix="pq_bench_dw_")
    cfg, user = _models.configs(wd, (3, 224, 224), 2)
    with torch.no_grad():
        net, _ = _models.build("mobilenetv2")
        q = tools.Quantity(merge_bn(net, "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize([(torch.randn(4, 3, 224, 224, generator=torch.Generator().manual_seed(1 + i)), None)
                               for i in range(2)])
        q.weight_quantize()
        r = tools.Reconstruction(_models.build("mobilenetv2")[0], config=cfg)
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
    ap.add_argument("--layer-batch-forward", type=int, default=None, help="batch of the fp32-boundary forward column")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--no-model", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_depthwise.py needs a GPU")
    torch.backends.cudnn.benchmark = False
    peak = copy_peak()
    lines = ["card: %s" % card(), "copy peak (1 GiB device-to-device, read + write): %.2f TB/s" % (peak / 1e12)]
    layer_table(args.batch, args.layer_batch_forward or args.batch, args.iters, peak, lines)
    if not args.no_model:
        lines.append("MobileNetV2 ReconModel, batch %d, 224 x 224:" % args.batch)
        whole_model(args.batch, max(5, args.iters // 4), lines)
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

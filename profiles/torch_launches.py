"""Launch list of one calibration job of the bench workload under torch.profiler, plus the bandwidth of the fused
calibration-forward kernels against a copy peak measured in the same process.

    python profiles/torch_launches.py OUT.txt [--steps K]

Workload: bench.py's (ResNet-50, BN folded, micro-batch 64, inputs resident in HBM), K batches through
Quantity.activation_quantize after a warm-up job; pass 2 is served from the HBM activation cache.  The list gives
every kernel's count, total time and share; then, per plane size, the algorithmic GB/s of pq::epilogue_kernel
(conv epilogue: 8 bytes per element, 12 with the ReLU output; Eltwise: 12 / 16) and of absmax_multi_kernel, over the
copy peak: a CUDA-event-timed clone of a 4 GiB tensor (8 bytes per element moved).  A conv output is read back
right after cuDNN wrote it, so part of it still comes from L2: the conv epilogue can exceed the copy peak.
Profiler-traced, so the host side is slower than in bench.py: compare kernel times and shares, not the step time."""
import argparse
import os
import subprocess
import sys
import tempfile
from collections import defaultdict

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench  # noqa: E402  (puts the package on sys.path)
import torch  # noqa: E402


def copy_peak_gbs(nbytes=4 << 30, iters=10):
    x = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").normal_()
    for _ in range(3):
        y = x.clone()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(iters):
        y = x.clone()
    e.record()
    torch.cuda.synchronize()
    del x, y
    return 2.0 * nbytes * iters / (s.elapsed_time(e) * 1e-3) / 1e9


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        return torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--steps", type=int, default=4)
    args = ap.parse_args()
    from torch.profiler import ProfilerActivity, profile
    import tools
    from common.quantity import _native
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    _native.lib()
    net = bench.build_model()
    workdir = tempfile.mkdtemp(prefix="pq_launches_")
    warm = [bench.make_batch(10_000 + i, device="cuda") for i in range(3)]
    bench.run_job(net, bench.ShardedBatches(warm, 3, 0, 1), 3, workdir, 0, 1)
    batches = [bench.make_batch(i, device="cuda") for i in range(args.steps)]
    cfg, user = bench.tool_configs(workdir, args.steps)
    q = tools.Quantity(net, config=cfg, user_config=user, verbose=False)     # the (unfused) tracing forward
    rec, shapes = {}, {"conv_epilogue": [], "eltwise": []}
    for kind, fname in (("conv_epilogue", "conv_epilogue"), ("eltwise", "eltwise_add")):
        def wrap(fn, kind=kind):                   # the tensor shape of every fused launch, in order
            def call(t, *a, **k):
                shapes[kind].append(tuple(t.shape))
                return fn(t, *a, **k)
            return call
        setattr(_native, fname, wrap(getattr(_native, fname)))
    torch.cuda.synchronize()
    _native.set_profile(rec)                       # per launch, in order: (start, end, algorithmic bytes)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        q.activation_quantize(bench.ShardedBatches(batches, args.steps, 0, 1))
        torch.cuda.synchronize()
    _native.set_profile(None)
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and not e.name.startswith(("Memcpy", "Memset"))]
    kernels.sort(key=lambda e: e.time_range.start)
    peak = copy_peak_gbs()

    per = defaultdict(lambda: [0, 0.0])
    for e in kernels:
        per[e.name][0] += 1
        per[e.name][1] += e.device_time / 1e3
    total = sum(v[1] for v in per.values())
    lines = ["# torch.profiler (CUDA activity) of Quantity.activation_quantize on the bench workload: %d batches of 64, "
             "ResNet-50, pass 2 from the HBM cache; after a 3-batch warm-up job" % args.steps,
             "# card: %s" % card(),
             "# %d launches, %.3f ms of kernel time (%.3f ms per batch)" % (len(kernels), total, total / args.steps),
             "%-100s %6s %10s %6s" % ("kernel", "count", "total_ms", "share")]
    for name, (n, ms) in sorted(per.items(), key=lambda kv: -kv[1][1]):
        lines.append("%-100s %6d %10.3f %5.1f%%" % (name[:100], n, ms, 100 * ms / total))
    ours = sum(ms for name, (n, ms) in per.items() if "pq::" in name)
    lines.append("# kernels of this repo (pq::*): %.3f ms = %.1f%% of the kernel time" % (ours, 100 * ours / total))
    for bad in ("CUDAFunctor_add", "launch_clamp_scalar"):
        lines.append("# launches whose name contains %s: %d" % (bad, sum(n for name, (n, _) in per.items()
                                                                        if bad in name)))

    # the k-th launch of a kind in the trace is the k-th _Timed record of that kind
    lines.append("# copy peak, same process: clone of a 4 GiB fp32 tensor, %.1f GB/s" % peak)
    lines.append("%-44s %6s %10s %9s %8s" % ("pq kernel, tensor shape, bytes per launch", "count", "GB", "GB/s",
                                             "of copy"))
    for kind, match in (("conv_epilogue", "epilogue_kernel<0>|epilogue_kernel<1>"), ("eltwise", "epilogue_kernel<2>"),
                        ("absmax", "absmax_multi_kernel")):
        ev = [e for e in kernels if any(m in e.name for m in match.split("|"))]
        recs = rec.get(kind, [])
        assert len(ev) == len(recs), (kind, len(ev), len(recs))
        groups = defaultdict(lambda: [0, 0, 0.0])
        labels = shapes.get(kind) or [()] * len(recs)
        for e, (_s, _e, nbytes), shape in zip(ev, recs, labels):
            g = groups[(shape, nbytes)]
            g[0] += 1
            g[1] += nbytes
            g[2] += e.device_time / 1e3
        for (shape, nbytes), (n, b, ms) in sorted(groups.items(), key=lambda kv: (kv[0][0][2:], kv[0])):
            gbs = b / (ms * 1e-3) / 1e9
            label = "%s %s %d" % (kind, "x".join(map(str, shape)), nbytes)
            lines.append("%-44s %6d %10.3f %9.1f %8.3f" % (label, n, b / 1e9, gbs, gbs / peak))
    text = "\n".join(lines) + "\n"
    with open(args.out, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- headline benchmark of the calibration hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], the configuration the metric "calib images/sec (hist+KL)"
is quoted on): ResNet-50 (fabu-style, BN folded, random init) calibration on synthetic
3x224x224 images, micro-batch 64 per rank.  One STEP = one micro-batch taken through the whole
hot path: fp32 forward with device-resident hooks, pass-1 max-abs of the 71 observed tensors,
pass-2 2048-bin histograms; the job ends with the NCCL MAX / SUM merge, the KL threshold search
of all 71 tensors and the feat.table bits.  The timed region is the whole job for K steps per
rank; value = N*K*64 images / max-over-ranks device time.  Weak scaling: per-rank work fixed.

  value : inputs resident in HBM before the timed region (tools.Quantity.activation_quantize
          on device tensors).
  e2e   : the same public call on HOST batches in pinned memory; the H2D copy of every batch and
          the D2H read of maxima / histograms / thresholds are inside the timed region.
  roofline : the dominant kernel of this repo (pq_hist2048_multi_f32, HBM-bound, 4 algorithmic
          bytes per element per launch), timed live with CUDA events on its launching stream.
  cpu_baseline / --impl reference : the UNMODIFIED reference (staged byte copy baseline/_ref, run by
          baseline/ref_runner.py in its own process with DEVICE: cpu and WORKER_NUM = host cores) through its
          own Quantity.activation_quantize on a bounded sample of the same workload ("kind": "reference");
          falls back to the oracle port ("kind": "port") only if nothing is staged.
Extra keys measured after the timed region (rank 0, N = 1): "c3_full" (the whole 8192-image job of BASELINE
config 3, honest cache / re-forward split; every rank at any N), "recontest" (config 2), "reconmodel" (config 4)
each with the reference's own modules timed eager on this same GPU, "c1" (config 1: this repo on the GPU next to
the unmodified reference on the host cores, same 64 images).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "pytorch-quantity_b200")
for p in (PKG, REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

MICRO_BATCH = 64
IMG_SHAPE = (3, 224, 224)
METRIC = "calib images/sec (hist+KL)"
UNIT = "images/s"
WORKLOAD = "ResNet-50 224x224 calibration (max-abs + 2048-bin hist + KL search), micro-batch 64 per GPU"


def build_model():
    from model.resnet.resnet_fabu import randomize_bn_, resnet50_fabu
    from common.quantity import merge_bn
    torch.manual_seed(0)
    net = resnet50_fabu().eval()
    with torch.no_grad():
        randomize_bn_(net, 0)
        merge_bn(net, "cpu")
    return net


def make_batch(index, batch=MICRO_BATCH, device="cpu", pin=False):
    g = torch.Generator().manual_seed(1 + index)
    x = torch.randn(batch, *IMG_SHAPE, generator=g)
    if device != "cpu":
        return x.to(device)
    return x.pin_memory() if pin else x


def tool_configs(workdir, n_batches):
    import tools._config as tc
    cfg = tc.load_tool_config(os.path.join(os.path.dirname(tc.__file__), "configs.yml"))
    cfg["OUTPUT"] = {"WORK_DIR": workdir, "WEIGHT_BIT_TABLE": workdir + "/weight.table",
                     "FEAT_BIT_TABLE": workdir + "/feat.table", "WEIGHT_DIR": workdir + "/weight",
                     "BIAS_DIR": workdir + "/bias", "FINAL_WEIGHT_DIR": workdir + "/new_weight",
                     "FINAL_BIAS_DIR": workdir + "/new_bias"}
    cfg["SETTINGS"]["MAX_CALI_IMG_NUM"] = n_batches - 1
    user = tc.load_user_config({"PATH": {}, "MODEL": {"INPUT_SHAPE": "1,3,224,224"},
                                "PRE_PROCESS": {"IMG": 1}, "SETTINGS": {"DEVICE": "gpu", "GPU": 0}})
    return cfg, user


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc, self.first = gpu_index, [], None, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)   # (the recipe's period:
            # every poll takes driver locks; at 100 ms the polled `value` job came out up to 4 % below the unpolled e2e job)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self, wait_s=3.0):
        """Call right before the timed region: waits until nvidia-smi has delivered its first sample (its NVML
        start-up takes driver locks for ~50 ms and must not land inside the timed region) and discards what
        was sampled so far."""
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < wait_s:
            time.sleep(0.02)
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        self.thread.join(timeout=2)
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows[self.first:] or self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        loaded = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full
    capture of this same bench command (profiles/rNN_traffic.json, written by profiles/summarize.py)."""
    for tag in ("r02", "r01"):                     # the latest committed capture
        try:
            with open(os.path.join(REPO, "profiles", tag + "_traffic.json")) as f:
                return float(json.load(f)[kernel]["dram_bytes_per_launch"])
        except (OSError, KeyError, ValueError):
            continue
    return None


def fakequant_bandwidth(n_elems=1 << 28, iters=10):
    """Second half of BASELINE.json's metric: QuanDequan (pq_fakequant_f32) GB/s on a 1 GiB fp32 tensor
    (larger than L2), 8 algorithmic bytes per element, CUDA events on the launching stream."""
    from common.quantity import _native
    x = torch.randn(n_elems, device="cuda")
    for _ in range(3):
        y = _native.fakequant(x, 4)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(iters):
        y = _native.fakequant(x, 4)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / iters
    del x, y
    return 8.0 * n_elems / (ms * 1e-3) / 1e9, ms


# ----------------------------------------------------------------------------- our arm
def run_job(net, batches, n_global, workdir, rank, world):
    """One whole calibration job through the public API; returns (seconds on device, Quantity)."""
    import tools
    cfg, user = tool_configs(workdir, n_global)
    q = tools.Quantity(net, config=cfg, user_config=user, verbose=False)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    q.activation_quantize(batches)
    end.record()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    ms = start.elapsed_time(end)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    return ms / 1e3, q


class ShardedBatches:
    """A global list of n_global batches of which only this rank's (index % world == rank) exist."""

    def __init__(self, mine, n_global, rank, world):
        self.mine, self.n, self.rank, self.world = mine, n_global, rank, world

    def __iter__(self):
        for i in range(self.n):
            yield (self.mine[i // self.world], None) if i % self.world == self.rank else None


def ours(args):
    from common.quantity import _native
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.backends.cudnn.allow_tf32 = False           # the forward stays true fp32, like the reference
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = os.environ.get("PQ_BENCH_NO_AUTOTUNE") != "1"   # off under ncu
    _native.lib()
    net = build_model()
    workdir = tempfile.mkdtemp(prefix="pq_bench_rank%d_" % rank)
    K, W = args.steps, max(args.warmup, 3)

    # warm-up: W steps through the same job shape (cuDNN autotune, allocator, kernels)
    # (pinned host batches: the warm-up also exercises the copy stream / H2D path the e2e job uses)
    warm = [make_batch(10_000 + rank * W + i, pin=True) for i in range(W)]
    _, qw = run_job(net, ShardedBatches(warm, W * world, rank, world), W * world, workdir, rank, world)
    del warm
    # Pre-size the caching allocator's pool for the K-batch activation cache so that no cudaMalloc
    # lands inside the timed region: allocate one block of the expected size and release it to the pool.
    per_batch = qw.timings["cached_bytes"] // max(1, qw.timings["cached_batches"])
    free, _total = torch.cuda.mem_get_info()
    want = min(int((K + 2) * per_batch * 1.05), int(free * 0.8))
    if want > 0:
        torch.empty(want, dtype=torch.uint8, device="cuda")

    # ---- value: inputs resident in HBM ---------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                    # started early: see ClockSampler.mark
    dev_batches = [make_batch(rank + world * i, device="cuda") for i in range(K)]
    prof = {}
    _native.set_profile(prof)
    l0 = _native.LAUNCHES["total"]
    if rank == 0:
        sampler.mark()
    try:
        secs, q = run_job(net, ShardedBatches(dev_batches, K * world, rank, world), K * world, workdir, rank, world)
    finally:                               # nvidia-smi must not outlive a failed run
        clocks = sampler.stop() if rank == 0 else None
    launches = _native.LAUNCHES["total"] - l0
    _native.set_profile(None)
    torch.cuda.synchronize()
    value = world * K * MICRO_BATCH / secs
    timings = dict(q.timings)
    bits_image = q.last_calibration["bits"]["image"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, q.last_calibration)
    del dev_batches

    def kernel_stats(name):
        rows = prof.get(name, [])
        if not rows:
            return None
        ms = [s.elapsed_time(e) for s, e, _ in rows]
        nbytes = [b for _, _, b in rows]
        return {"launches": len(rows), "avg_ms": sum(ms) / len(ms), "avg_bytes": sum(nbytes) / len(nbytes),
                "total_ms": sum(ms)}

    hist, amax, kl = kernel_stats("hist"), kernel_stats("absmax"), kernel_stats("kl")
    peak, peak_src = peaks()
    achieved = hist["avg_bytes"] / (hist["avg_ms"] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "pq::hist_multi_kernel (pq_hist2048_multi_f32)",
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": ncu_traffic("hist_multi"), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": hist["avg_bytes"], "avg_launch_ms": round(hist["avg_ms"], 4),
                "absmax_GBps": round(amax["avg_bytes"] / (amax["avg_ms"] * 1e-3) / 1e9, 1),
                "kl_ms_per_job": round(kl["total_ms"], 3), "kl_us_per_tensor": round(kl["total_ms"] * 1e3 / 71, 1),
                "stats_share_of_step": round((hist["total_ms"] + amax["total_ms"]) / (secs * 1e3), 4)}

    # ---- e2e: host batches in pinned memory through the same public call ---------------------
    host_batches = [make_batch(rank + world * i, pin=True) for i in range(K)]
    e_secs, q2 = run_job(net, ShardedBatches(host_batches, K * world, rank, world), K * world, workdir, rank, world)
    n_fwd_pass2 = K - q2.timings.get("cached_batches", 0)
    h2d = (K + n_fwd_pass2) * MICRO_BATCH * int(np.prod(IMG_SHAPE)) * 4 / K
    d2h = (71 * 4 + 71 * 2048 * 8 + 71 * 4) / K
    e2e = {"value": round(world * K * MICRO_BATCH / e_secs, 2), "unit": UNIT,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "phases_s": {k: round(v, 4) for k, v in q2.timings.items() if k.endswith("_s")}}
    assert q2.last_calibration["bits"]["image"] == bits_image
    del host_batches

    fq_gbps, fq_ms = fakequant_bandwidth()
    extras = {}
    if not args.no_extras:
        t0 = time.perf_counter()
        for _ in range(int(os.environ.get("PQ_BENCH_C3_REPEAT", "1"))):
            extras["c3_full"] = c3_full_job(net, workdir, rank, world)
        _note(t0, "c3_full")
        torch.cuda.empty_cache()
        if rank == 0 and world == 1 and os.environ.get("PQ_BENCH_ONLY_C3") != "1":   # (development: c3_full only)
            extras.update(sim_extras(peak))
            t0 = time.perf_counter()
            extras["c1"] = c1_extra()
            _note(t0, "c1")
    line = None
    if rank == 0:
        cpu = cpu_baseline(sample_images=args.cpu_sample) if world == 1 and not args.no_cpu_baseline else None
        line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": round(secs * 1e3 / K, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "global_batch": world * MICRO_BATCH, "images": world * K * MICRO_BATCH,
                           "observed_tensors": 71, "elements_per_image": 16784872,
                           "l2": "inputs larger than L2 (4.3 GB of activations per step)",
                           "pass2": "%d of %d steps served from the HBM activation cache"
                                    % (timings.get("cached_batches", 0), K),
                           "parallelism": "dp%d" % world},
                "roofline": roofline, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
                "fakequant": {"GBps": round(fq_gbps, 1), "frac_of_hbm_peak": round(fq_gbps / peak, 4),
                              "elements": 1 << 28, "ms": round(fq_ms, 4), "algorithmic_bytes_per_element": 8},
                "phases_s": {k: round(v, 4) for k, v in timings.items() if k.endswith("_s")}}
        if cpu:
            line["cpu_baseline"] = cpu
        line.update(extras)
    if world > 1:
        torch.distributed.destroy_process_group()
    return line



def dump_outputs(out_dir, cal):
    """What the timed job hands its caller (Quantity.last_calibration after the merge over ranks), as float64 arrays
    whose rows follow the observed tensors in forward order ("image" first): <key>.npy of shape [71] for the
    per-tensor scalars and distributions.npy of shape [71, 2048] for the histograms."""
    os.makedirs(out_dir, exist_ok=True)
    names = cal["top_feat_names"]
    for key in ("max_vals", "intervals", "thresholds", "threshold_bins", "bits"):
        np.save(os.path.join(out_dir, key + ".npy"), np.array([float(cal[key][n]) for n in names], np.float64))
    np.save(os.path.join(out_dir, "distributions.npy"),
            np.stack([np.asarray(cal["distributions"][n], np.float64) for n in names]))


# ------------------------------------------------------------------------ extras (after the timed region)
class CycledBatches:
    """n_global batches of which this rank owns every world-th; the owned ones cycle through a small pool of
    distinct pinned host batches (synthetic data: throughput does not depend on the pixel values)."""

    def __init__(self, pool, n_global, rank, world):
        self.pool, self.n, self.rank, self.world = pool, n_global, rank, world

    def __iter__(self):
        for i in range(self.n):
            yield (self.pool[(i // self.world) % len(self.pool)], None) if i % self.world == self.rank else None


def _alloc_stats(tag):
    s = torch.cuda.memory_stats()
    free, _total = torch.cuda.mem_get_info()
    print("[bench] %s: reserved %.1f GB, allocated %.1f GB, device-free %.1f GB, segments %d, cudaMalloc calls %d, "
          "allocator retries %d" % (tag, s["reserved_bytes.all.current"] / 1e9, s["allocated_bytes.all.current"] / 1e9,
                                    free / 1e9, s["segment.all.current"], s["num_device_alloc"], s["num_alloc_retries"]),
          file=sys.stderr, flush=True)


def c3_full_job(net, workdir, rank, world, total_images=8192):
    """BASELINE config 3 at its stated size: 8192 images = 128 micro-batches of 64 shared by the ranks, host batches,
    through the public call.  At N = 1 the 550 GB of observed activations do not fit the HBM cache, so most of
    pass 2 re-runs the forward; from N = 4 on everything is served from the cache."""
    n_global = total_images // MICRO_BATCH
    pool = [make_batch(50_000 + rank * 16 + i, pin=True) for i in range(min(16, n_global // world))]
    trace = os.environ.get("PQ_BENCH_C3_TRACE") == "1"          # per-batch device times of pass 1 + allocator statistics
    if trace:
        import common.quantity.distribution_collector as dc
        events, orig = [], dc.DistributionCollector.refresh_max_val

        def traced(self, feats):
            r = orig(self, feats)
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            events.append(e)
            return r
        dc.DistributionCollector.refresh_max_val = traced
        _alloc_stats("c3_full before")
    try:
        secs, q = run_job(net, CycledBatches(pool, n_global, rank, world), n_global, workdir, rank, world)
    finally:
        if trace:
            dc.DistributionCollector.refresh_max_val = orig
    if trace:
        _alloc_stats("c3_full after")
        ms = [events[i].elapsed_time(events[i + 1]) for i in range(len(events) - 1)]
        for a in range(0, len(ms), 16):
            print("[bench]   pass-1 batches %3d-%3d device ms: %s" % (a + 2, min(a + 17, len(ms) + 1),
                  " ".join("%5.1f" % v for v in ms[a:a + 16])), file=sys.stderr, flush=True)
    t = q.timings
    print("[bench] c3_full rank %d: %s" % (rank, {k: (round(v, 3) if isinstance(v, float) else v) for k, v in t.items()}),
          file=sys.stderr, flush=True)
    return {"images": total_images, "steps_per_rank": t["batches"], "seconds": round(secs, 3),
            "images_per_s": round(total_images / secs, 1),
            "pass2_from_hbm_cache": t["cached_batches"], "pass2_forward_reruns": t["batches"] - t["cached_batches"],
            "cache_GB": round(t["cached_bytes"] / 1e9, 1),
            "phases_s": {k: round(v, 3) for k, v in t.items() if k.endswith("_s")},
            "inputs": "pinned host batches (H2D inside the timed region), %d distinct batches cycled" % len(pool)}


def _sim_workdir(name, tag):
    """Tables for the simulation extras: a short calibration of the same seeded model through this repo's tools."""
    import tempfile
    import ref_models
    import tools
    from common.quantity import merge_bn
    workdir = tempfile.mkdtemp(prefix="pq_bench_%s_" % tag)
    cfg, user = tool_configs(workdir, 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(ref_models.build_model(name), "cpu"), config=cfg, user_config=user, verbose=False)
        q.activation_quantize(ref_models.calib_batches(name, 2, 16))
        q.weight_quantize(write_json=False)              # Reconstruction reads the two tables only
    return workdir, cfg


def _rebuilt(name, mode, cfg):
    import ref_models
    import tools
    with torch.no_grad():
        r = tools.Reconstruction(ref_models.build_model(name), config=cfg)
        r.merge_bn()
        return getattr(r, mode)(r.get_quantity_information(), None).cuda().eval()


def _note(t0, what):
    print("[bench] %-40s %.1f s" % (what, time.perf_counter() - t0), file=sys.stderr, flush=True)


def sim_extras(peak_hbm, iters=5):
    """BASELINE configs 2 and 4 in the driver-run line: this repository's ReconTest / ReconModel forwards and, on
    the same GPU in the same run, the reference's own modules run eager (baseline/ref_runner.py --device gpu)."""
    import bench_sim
    import ref_models
    from common.quantity import enable_int8_pipeline
    ref_models.set_deterministic()      # the same library flags as the reference arm (baseline/ref_runner.py)
    out = {}
    t0 = time.perf_counter()
    # ---- config 2: ResNet-18 ReconTest, batch 256
    B = 256
    workdir, cfg = _sim_workdir("r18", "c2")
    model = _rebuilt("r18", "ReconTest", cfg)
    x = ref_models.eval_batch("r18", B).cuda()
    ms, stats, launches, y = bench_sim.timed_forward(model, x, iters)
    fq = stats.get("fakequant", {})
    rec = {"workload": "ResNet-18 224x224 ReconTest (fake-quant) inference, batch %d" % B, "ms_per_forward": round(ms, 3),
           "images_per_s": round(B / (ms * 1e-3), 1), "gpu_launches_per_forward": launches,
           "fakequant_ms_per_forward": round(fq.get("ms_per_fwd", 0.0), 4)}
    if fq.get("ms_per_fwd"):
        rec["fakequant_GBps"] = round(fq["alg_bytes_per_fwd"] / (fq["ms_per_fwd"] * 1e-3) / 1e9, 1)
        rec["fakequant_frac_of_hbm_peak"] = round(rec["fakequant_GBps"] / peak_hbm, 4)
    _note(t0, "recontest: this repo")
    if reference_staged():
        res, arrays = run_reference("r18", "c2", "--device", "gpu", "--tables-from", workdir, "--recon", "ReconTest",
                                    "--eval", B, "--time-forward", iters)
        rec["reference_eager_ms"] = round(statistics.median(res["ReconTest/forward_ms"]), 3)
        rec["reference_build_s"] = round(res["seconds_build_ReconTest"], 1)
        rec["logits_equal_reference"] = bool(np.array_equal(np.load(arrays)["ReconTest/y"], y.cpu().numpy()))
    out["recontest"] = rec
    _note(t0, "recontest: + reference eager")
    del model, x, y
    torch.cuda.empty_cache()
    # ---- config 4: ResNet-50 ReconModel, batch 512
    B = 512
    workdir, cfg = _sim_workdir("r50", "c4")
    model = _rebuilt("r50", "ReconModel", cfg)
    x = ref_models.eval_batch("r50", B).cuda()
    ms32, stats32, launches32, y32 = bench_sim.timed_forward(model, x, iters)
    enable_int8_pipeline(model, True)
    ms8, stats8, launches8, y8 = bench_sim.timed_forward(model, x, iters)
    gms, glaunches, gy = bench_sim.timed_graph(model, x, iters)
    peak8 = bench_sim.int8_peak_tops()
    rec = {"workload": "ResNet-50 224x224 ReconModel (integer simulation) inference, batch %d" % B,
           "fp32_boundary_ms_per_forward": round(ms32, 3), "int8_pipeline_ms_per_forward": round(ms8, 3),
           "int8_pipeline_graph_ms_per_forward": round(gms, 3), "images_per_s": round(B / (gms * 1e-3), 1),
           "gpu_launches_per_forward": launches8, "int8_peak_TOPS_measured": round(peak8, 1),
           "pipeline_equals_fp32_boundary": bool(torch.equal(y8, y32) and torch.equal(gy, y32)), "kernels": {}}
    ops = ms_conv = 0.0
    for kname, st in stats8.items():
        k = {"launches": st["launches_per_fwd"], "ms": round(st["ms_per_fwd"], 4)}
        if kname in ("conv_s8", "gemm_s8", "conv_add_s8"):
            ops += st["alg_bytes_per_fwd"]
            ms_conv += st["ms_per_fwd"]
            k["TOPS"] = round(st["alg_bytes_per_fwd"] / (st["ms_per_fwd"] * 1e-3) / 1e12, 1)
        elif st["ms_per_fwd"] > 0:
            k["GBps"] = round(st["alg_bytes_per_fwd"] / (st["ms_per_fwd"] * 1e-3) / 1e9, 1)
            k["frac_of_hbm_peak"] = round(k["GBps"] / peak_hbm, 4)
        rec["kernels"][kname] = k
    if ms_conv > 0:
        rec["conv_ms_per_forward"] = round(ms_conv, 3)
        rec["conv_TOPS"] = round(ops / (ms_conv * 1e-3) / 1e12, 1)
        rec["frac_of_int8_peak"] = round(rec["conv_TOPS"] / peak8, 4)
    _note(t0, "reconmodel: this repo")
    if reference_staged():
        res, arrays = run_reference("r50", "c4", "--device", "gpu", "--tables-from", workdir, "--recon",
                                    "ReconModel,ReconModel:nocudnn", "--eval", B, "--time-forward", 3,
                                    "--exact-batch", 32)
        rec["reference_eager_ms"] = round(statistics.median(res["ReconModel/forward_ms"]), 3)
        ref_y = np.load(arrays)
        # the exact arm (cuDNN's fp32 Winograd is not exact on integers, see tests/test_gpu_vs_reference.py) on the
        # first 32 images: ATen's GEMM convolution loops over the samples and would take minutes at batch 512
        y_np = y32.cpu().numpy()
        rec["logits_equal_reference_exact_conv"] = bool(np.array_equal(ref_y["ReconModel:nocudnn/y"], y_np[:32]))
        rec["logits_equal_reference_exact_conv_images"] = 32
        rec["logits_equal_reference_cudnn"] = bool(np.array_equal(ref_y["ReconModel/y"], y_np))
    out["reconmodel"] = rec
    _note(t0, "reconmodel: + reference eager")
    del model, x
    torch.cuda.empty_cache()
    return out


def c1_extra():
    """BASELINE config 1 (ResNet-18, 64 images as 8 batches of 8): this repository on the GPU next to the UNMODIFIED
    reference on the host cores, both running the whole job (calibration + weight quantisation + rewrite)."""
    import tempfile
    import ref_models
    import tools
    from common.quantity import merge_bn
    workdir = tempfile.mkdtemp(prefix="pq_bench_c1_")
    cfg, user = tool_configs(workdir, 8)
    batches = ref_models.calib_batches("r18", 8, 8)
    with torch.no_grad():
        net = merge_bn(ref_models.build_model("r18"), "cpu")
        q = tools.Quantity(net, config=cfg, user_config=user, verbose=False)
        for _ in range(2):                                  # second run: warm allocator / kernels
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            q.activation_quantize(batches)
            torch.cuda.synchronize()
            t_act = time.perf_counter() - t0
        q.weight_quantize()
        t_all = time.perf_counter() - t0
    rec = {"workload": "ResNet-18 224x224 calibration, 64 images (8 batches of 8), feat.table + weight.table + JSON",
           "ours_activation_quantize_s": round(t_act, 4), "ours_whole_job_s": round(t_all, 3),
           "ours_images_per_s": round(64 / t_act, 1)}
    if reference_staged():
        res, _ = run_reference("r18", "c1", "--device", "cpu", "--calib", "8x8")
        ours_feat = open(cfg["OUTPUT"]["FEAT_BIT_TABLE"]).read()
        ours_weight = open(cfg["OUTPUT"]["WEIGHT_BIT_TABLE"]).read()
        ref_feat = res["after_weight_quantize"]["feat.table"]
        rec.update({
            "reference_cpu_activation_quantize_s": round(res["seconds_activation_quantize"], 1),
            "reference_cpu_weight_quantize_s": round(res["seconds_weight_quantize"], 1),
            "reference_cpu_images_per_s": round(64 / res["seconds_activation_quantize"], 2),
            "reference_cores": res["worker_num"], "host_cores": os.cpu_count(),
            "weight_table_identical": ours_weight == res["after_second_rewrite"]["weight.table"],
            # cuDNN forward here, MKLDNN forward there: byte-identity of feat.table is asserted GPU-vs-GPU in the tests
            "feat_table_lines_differing_vs_cpu_forward": sum(a != b for a, b in zip(ours_feat.split("\n"),
                                                                                      ref_feat.split("\n")))})
    return rec

# ------------------------------------------------------------------- CPU baseline / reference arm
def cpu_calibration_sample(n_images, batch, threads):
    """The reference's CPU algorithm on `n_images` synthetic images: torch CPU fp32 forward with
    hooks (both passes, like pytorch_quantizer.py:379-426), oracle max-abs / histograms per tensor
    fanned out over `threads` host threads (the reference fans out over a process pool), then the
    oracle KL search for all tensors.  Returns seconds."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pq_oracle as oracle
    oracle.build()
    torch.set_num_threads(threads)
    net = build_model()
    feats = {}
    order = []

    def hook(name):
        def _h(m, i, o):
            if not feats:
                feats["image"] = i[0].detach().numpy().reshape(-1)
            feats[name] = o.detach().numpy().reshape(-1)
        return _h

    for name, m in net.named_modules():
        if type(m).__name__ in ("Conv2d", "Linear", "Eltwise"):
            m.register_forward_hook(hook(name))
            order.append(name)
    names = ["image"] + order
    batches = [make_batch(i, batch) for i in range(max(1, n_images // batch))]
    pool = ThreadPoolExecutor(threads)
    t0 = time.perf_counter()
    maxes = {n: 0 for n in names}
    with torch.no_grad():
        for x in batches:                                           # pass 1
            feats.clear()
            net(x)
            for n, m in zip(names, pool.map(lambda n: oracle.absmax_update(maxes[n], feats[n]), names)):
                maxes[n] = m
        intervals = {n: oracle.interval(maxes[n]) for n in names}
        hists = {n: np.zeros(2048, np.int64) for n in names}
        for x in batches:                                           # pass 2
            feats.clear()
            net(x)
            for n, h in zip(names, pool.map(lambda n: oracle.hist(feats[n], intervals[n]), names)):
                hists[n] += h
    bits = list(pool.map(lambda n: oracle.quantize_distribution(hists[n], intervals[n])[0], names))
    secs = time.perf_counter() - t0
    assert len(bits) == 71
    return secs, len(batches) * batch


RUNNER = os.path.join(REPO, "baseline", "ref_runner.py")


def reference_staged():
    return os.path.isdir(os.path.join(REPO, "baseline", "_ref", "quantity", "common", "quantity"))


def run_reference(model, out_tag, *flags, timeout=1500):
    """baseline/ref_runner.py (the unmodified reference) in its own process; returns (result.json, arrays path)."""
    import tempfile
    out = tempfile.mkdtemp(prefix="pq_ref_%s_" % out_tag)
    cmd = [sys.executable, RUNNER, "--model", model, "--out", out] + [str(f) for f in flags]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    if p.returncode != 0:
        raise RuntimeError("reference runner failed: " + p.stdout[-1500:])
    with open(os.path.join(out, "result.json")) as f:
        return json.load(f), os.path.join(out, "arrays.npz")


def reference_calibration(n_batches, batch, warmup=0):
    """The reference's own two-pass calibration job (Quantity.activation_quantize, pytorch_quantizer.py:345-489:
    fp32 CPU forward x2, numpy max-abs, the per-element Python histogram loop in a process pool, the pure-Python
    KL search of all 71 tensors) on n_batches x batch synthetic images of the bench workload."""
    res, _ = run_reference("r50", "calib", "--device", "cpu", "--calib", "%dx%d" % (n_batches, batch),
                           "--calib-only-activations", "--warmup-batches", warmup)
    return res["seconds_activation_quantize"], n_batches * batch, res["worker_num"]


def cpu_baseline(sample_images=8):
    if not reference_staged():
        threads = os.cpu_count() or 1
        secs, n = cpu_calibration_sample(16, 8, threads)
        return {"value": round(n / secs, 3), "unit": UNIT, "cores": threads, "kind": "port",
                "sample": "%d images through torch-CPU fp32 forward x2 + oracle max-abs/hist + oracle KL search "
                          "(baseline/_ref not staged)" % n}
    secs, n, workers = reference_calibration(max(1, sample_images // 2), 2)
    return {"value": round(n / secs, 3), "unit": UNIT, "cores": workers, "kind": "reference",
            "sample": "the unmodified reference (baseline/_ref, DEVICE: cpu, WORKER_NUM %d of %d host cores): one whole "
                      "Quantity.activation_quantize job on %d images (%d batches of 2) of the same ResNet-50 workload, "
                      "%.1f s" % (workers, os.cpu_count() or 1, n, n // 2, secs)}


def reference_arm(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return None
    K, W = args.steps, max(args.warmup, 1)
    if reference_staged():
        per_step = 2                                   # bounded sample: a step is one batch of 2 images
        secs, n, workers = reference_calibration(K, per_step, warmup=W)
        value = round(n / secs, 3)
        return {
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": K, "warmup": W,
            "ms_per_step": round(secs * 1e3 / K, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the same keys as the GPU arm's config, with this arm's truthful values: the same workload, a bounded
            # sample of it per step (2 images instead of 64) -- rates are per image
            "config": {"workload": WORKLOAD, "global_batch": per_step, "images": n, "observed_tensors": 71,
                       "elements_per_image": 16784872,
                       "l2": "host memory (the reference copies every activation to numpy)",
                       "pass2": "every step re-runs the forward (reference :415-426)", "parallelism": "cpu%d" % workers,
                       "job": "one whole activation_quantize job of %d batches (both passes + KL search of 71 tensors)" % K},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "reference",
                             "sample": "unmodified reference (baseline/_ref), DEVICE: cpu, WORKER_NUM %d: %d steps of %d "
                                       "images, %d warm-up forwards" % (workers, K, per_step, W)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    threads = os.cpu_count() or 1
    per_step = 8                                       # bounded sample: 8 images per step
    for _ in range(min(W, 1)):
        cpu_calibration_sample(per_step, per_step, threads)
    k_eff = min(K, 6)                                   # keep the whole run within a few minutes
    secs, n = cpu_calibration_sample(per_step * k_eff, per_step, threads)
    value = round(n / secs, 3)
    return ({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": k_eff, "warmup": W,
        "ms_per_step": round(secs * 1e3 / k_eff, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_images_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d steps of %d images; torch-CPU forward x2 + oracle statistics + KL"
                                   % (k_eff, per_step)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip c3_full / recontest / reconmodel / c1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed job computed as DIR/<name>.npy (float64; the "
                         "inputs are seeded, so two builds can be compared output for output).  cuDNN autotuning "
                         "may pick other fp32 convolutions from run to run, which moves maxima and histograms in "
                         "the last bits; PQ_BENCH_NO_AUTOTUNE=1 turns it off, so that cuDNN's heuristics choose "
                         "the algorithms")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    # the drop-in classes print progress like the reference does; keep stdout to the ONE JSON line
    real_stdout = sys.stdout
    sys.stdout = sys.stderr
    try:
        with tempfile.TemporaryDirectory(prefix="pq_bench_") as tmp:
            tempfile.tempdir = tmp          # every work directory of the run lives here and goes with it
            line = reference_arm(args) if args.impl == "reference" else ours(args)
    finally:
        tempfile.tempdir = None
        sys.stdout = real_stdout
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()

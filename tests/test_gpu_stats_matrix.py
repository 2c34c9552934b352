"""Every statistics and KL kernel of the calibration side (pq_stats.cu, pq_stats_kernels.cuh, pq_kl.cu), over its whole
argument range, against references that share no code with the kernels:

    max-abs     the maximum of |x| in float64, compared as the fp32 bit pattern (non-NaN inputs: the header defines
                the max only for those)
    histogram   q = float32(|x|.astype(float64) / float64(d)); +-0 skipped; q >= nbins - 1 and NaN -> bin nbins - 1;
                else bin trunc(q).  float64 carries 53 >= 2 * 24 + 2 bits, so rounding the quotient to float64 and
                then to float32 gives the correctly rounded fp32 quotient (subnormal and overflowing results included).
                Pinned to oracle.hist on finite inputs below.
    epilogues   float32(float64(a) + float64(b)) (exact for the same reason), max(v, 0), and the max-abs above
    KL          oracle.kl_search(oracle.normalize(counts)), which test_oracle.py pins to the reference goldens;
                curves within rtol 1e-9, thresholds exact

Segment tables cover zero-length segments (null pointers) first, last and between, every 4-byte offset, one chunk,
one chunk + 1 element, many chunks, and tables of more than 148 * 8 chunks where CTAs start mid-segment and one CTA
spans several segments.  Every output sits in a sentinel-filled buffer whose neighbouring bytes must survive; the
accumulating outputs (max_bits, histograms) are pre-seeded and must be max-ed / added into, not overwritten.  Each
row names the kernel its launch must land on (checked with torch.profiler), and KERNELS lists every kernel of the
three files with the test that reaches it.
"""
import ctypes
import os
import re
import shutil
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
EINVAL, EUNSUPPORTED, EALIGN, ETOOMANY = -1, -2, -3, -4
FLT_MAX = float(np.finfo(np.float32).max)
CHUNK = 8192                          # kChunkElems
CTAS = 148 * 8                        # the statistics kernels' grid cap
SENTINEL = 0xA5
GUARD = 512                           # bytes on either side; a multiple of 16, so outputs stay 16-byte aligned
NANS = np.array([0x7FC00000, 0xFFC00000, 0x7F800001, 0x7FA00000, 0xFFFFFFFF], dtype=np.uint32).view(np.float32)


def _lib():
    from common.quantity import _native
    return _native.lib()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _seed(*key):
    return zlib.crc32(repr(key).encode()) & 0xFFFF


class Guarded:
    """An output tensor in the middle of a sentinel-filled buffer."""

    def __init__(self, shape, dtype):
        n = int(np.prod(shape))
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        self.buf = torch.full((nbytes + 2 * GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.lo, self.hi = GUARD, GUARD + nbytes
        self.t = self.buf[self.lo:self.hi].view(dtype).view(shape)

    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        assert bool((self.buf[:self.lo] == SENTINEL).all()), "%s: bytes before the output were overwritten" % what
        assert bool((self.buf[self.hi:] == SENTINEL).all()), "%s: bytes after the output were overwritten" % what


def _untouched(*gs):
    return all(bool((g.buf == SENTINEL).all()) for g in gs)


# ------------------------------------------------------------------------------------------ kernel names
def kernel_id(name):
    """'hist_multi_kernel<1,8>' from a demangled name in either spelling: cu++filt's
    'void pq::epilogue_kernel<(int)1>(pq::EpiArgs)' or the profiler's '...<1>(...)'."""
    s = re.sub(r"\(int\)(-?\d+)", r"\1", name)
    m = re.search(r"pq::(\w+)(<[^>()]*>)?", s)
    return m.group(1) + (m.group(2) or "").replace(" ", "") if m else None


def launched(fn):
    """Names of every CUDA kernel fn() launched."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_FRESH_ENV = "PQ_STATS_MATRIX_FRESH"
_LANDING = {}


def _landing_state():
    """Whether torch.profiler records kernels in this process.  After some sequences of earlier tests in the same
    pytest process it records no CUDA activity at all; the landing checks then cannot be made here, so this file is
    run once more on its own in a fresh process, where every landing check runs, and that run must pass."""
    if not _LANDING:
        recorded = bool(launched(lambda: torch.ones(16, device="cuda").add_(1)))
        _LANDING["recorded"] = recorded
        if not recorded:
            assert not os.environ.get(_FRESH_ENV), "torch.profiler records no CUDA kernels in a fresh process"
            r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-p", "no:cacheprovider",
                                "-m", "gpu"], cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                               env=dict(os.environ, **{_FRESH_ENV: "1"}), capture_output=True, text=True, timeout=3600)
            _LANDING["fresh_run"] = (r.returncode, r.stdout[-3000:])
    return _LANDING


def check_landing(fn, kernels):
    """fn() launches exactly `kernels` (a list of kernel ids, in order)."""
    state = _landing_state()
    if state["recorded"]:
        names = launched(fn)
        assert [k for k in map(kernel_id, names) if k] == list(kernels), (kernels, names)
    else:
        fn()
        rc, out = state["fresh_run"]
        assert rc == 0, "the fresh-process run of this file, which makes the landing checks, failed:\n" + out


# ------------------------------------------------------------------------------------------ references
def absmax_bits_ref(x):
    """uint32 bit pattern of max |x| (float64 maximum of non-NaN float32 values; exact)."""
    x = np.asarray(x, dtype=np.float32)
    if x.size == 0:
        return 0
    assert not np.isnan(x).any()
    return int(np.array([np.abs(x.astype(np.float64)).max()], dtype=np.float32).view(np.uint32)[0])


def hist_ref(x, d, nbins):
    """int64 [nbins]: the contract of pq_hist_multi_f32 (module docstring)."""
    x = np.asarray(x, dtype=np.float32)
    x = x[x != 0]                                            # NaN != 0: kept
    with np.errstate(all="ignore"):
        q = (np.abs(x.astype(np.float64)) / np.float64(np.float32(d))).astype(np.float32)
    top = q >= nbins - 1
    top |= np.isnan(q)
    idx = np.where(top, nbins - 1, np.trunc(np.where(top, 0, q)).astype(np.int64))
    return np.bincount(idx, minlength=nbins).astype(np.int64)


def _f32(v):
    return np.array(v, dtype=np.float32)


def neighbours(v, ulps=3):
    """float32 v and its +-1..ulps neighbours (finite, non-negative ones)."""
    v = _f32(v).ravel()
    out = [v]
    up, down = v.copy(), v.copy()
    with np.errstate(over="ignore"):
        for _ in range(ulps):
            up, down = np.nextafter(up, np.float32(np.inf)), np.nextafter(down, np.float32(0))
            out += [up, down]
    r = np.concatenate(out)
    return r[np.isfinite(r)]


def hist_values(d, nbins, seed):
    """Crafted float32 values for bin width d: +-3 ulps around every bin edge b * d that matters (0, 1, 2, the
    middle, the top bin's edges and beyond), q exactly nbins - 1 and one ulp below it, subnormal x, +-0, +-inf,
    +-FLT_MAX, quiet / negative / signalling NaN, and noise.  Signs alternate; the length is odd, so a tiled copy puts
    every value in every lane of a float4."""
    d = np.float32(d)
    top = nbins - 1
    bins = np.array(sorted({0, 1, 2, 3, nbins // 2, top - 1, top, top + 1, nbins + 1, 2 * nbins}), dtype=np.float64)
    with np.errstate(all="ignore"):
        edges = (bins * np.float64(d)).astype(np.float32)
        q_top = np.float32(top)
        exact = np.array([q_top, np.nextafter(q_top, np.float32(0)), np.float32(nbins)], dtype=np.float64)
        exact = (exact * np.float64(d)).astype(np.float32)
    rng = np.random.default_rng(seed)
    with np.errstate(over="ignore"):                         # d = FLT_MAX: noise beyond the range is +inf
        noise = (rng.uniform(0, nbins + 2, 61) * np.float64(d)).astype(np.float32)
    specials = np.array([0.0, -0.0, 2.0 ** -149, 3 * 2.0 ** -149, 2.0 ** -130, 2.0 ** -126, np.inf, -np.inf, FLT_MAX,
                         -FLT_MAX], dtype=np.float32)
    v = np.concatenate([neighbours(edges), neighbours(exact, 1), noise, specials, NANS])
    sign = np.where(np.arange(v.size) % 2, np.float32(-1), np.float32(1))
    with np.errstate(invalid="ignore"):
        v = np.where(np.isnan(v), v, v * sign).astype(np.float32)
    return v if v.size % 2 else np.append(v, np.float32(0.5) * d)


# ------------------------------------------------------------------------------------------ segment tables
def table(name):
    """[(n, offset in elements)] of one multi-tensor launch; n = 0 is a null pointer."""
    if name == "k1_one_chunk":
        return [(CHUNK, 0)]
    if name == "k1_chunk_plus_one":
        return [(CHUNK + 1, 0)]
    if name == "k2_offsets":
        return [(CHUNK + 1, 1), (3 * CHUNK + 4 * 37 + 2, 3)]
    if name == "k255_tiny":                                   # n in {1, 2, 3} at every offset, zero-length between
        return [(0, 0) if i in (0, 97, 254) else (1 + i % 3, (i // 3) % 4) for i in range(255)]
    if name == "k256_mixed":
        sizes = (0, 1, 2, 3, 5, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK + 7, 3 * CHUNK + 4 * 37 + 1)
        t = [(sizes[i % len(sizes)], i % 4) for i in range(256)]
        t[0] = t[255] = (0, 0)
        return t
    if name == "many_chunks":
        return [(0, 0), (40 * CHUNK + 4 * 37 + 3, 1), (0, 0), (17 * CHUNK + 2, 2), (0, 0)]
    if name == "ctas_start_mid_segment":                      # 40 x 38 chunks > 148 * 8: two chunks per CTA
        return [(37 * CHUNK + 4 * i + 1 + i % 3, i % 4) for i in range(40)]
    if name == "cta_spans_segments":                          # ~2560 chunks: three per CTA, over 1-chunk segments
        return [(2500 * CHUNK - 1, 3)] + [(0, 0) if i % 7 == 3 else (CHUNK - 4 * (i % 5) + i % 4, i % 4)
                                          for i in range(60)]
    raise KeyError(name)


TABLES = ("k1_one_chunk", "k1_chunk_plus_one", "k2_offsets", "k255_tiny", "k256_mixed", "many_chunks",
          "ctas_start_mid_segment", "cta_spans_segments")


def total_chunks(segs):
    t = 0
    for s in segs:
        n = 0 if s is None else s.numel()
        head = min(((16 - (s.data_ptr() & 15)) & 15) >> 2, n) if n else 0
        t += max(1, -(-((n - head) // 4) // 2048))
    return t


def place(arrays):
    """Device segments at their offsets: a fresh allocation per segment (256-byte aligned), viewed `off` in."""
    segs = []
    for a, off in arrays:
        if a.size == 0:
            segs.append(None)
            continue
        buf = torch.empty(a.size + off + 4, dtype=torch.float32, device="cuda")
        v = buf[off:off + a.size]
        v.copy_(torch.from_numpy(a))
        segs.append(v)
    return segs


def seg_args(segs):
    k = len(segs)
    ptrs = (ctypes.c_void_p * k)(*[None if s is None else s.data_ptr() for s in segs])
    ns = (ctypes.c_uint64 * k)(*[0 if s is None else s.numel() for s in segs])
    return ptrs, ns


def positions(s):
    """Index of one element per position class of device segment s: 'head' (unaligned scalars), 'tail', 'partial'
    (last partial chunk), 'lane0'..'lane3' (a float4 lane in a full chunk)."""
    n = s.numel()
    head = min(((16 - (s.data_ptr() & 15)) & 15) >> 2, n)
    nvec = (n - head) // 4
    tail = n - head - 4 * nvec
    full, part = nvec // 2048, nvec % 2048
    p = {}
    if head:
        p["head"] = head - 1
    if tail:
        p["tail"] = n - 1
    if part:
        p["partial"] = head + 4 * (full * 2048 + part // 2) + 1
    if full:
        v = (full * 2048) * 5 // 7
        for lane in range(4):
            p["lane%d" % lane] = head + 4 * v + lane
    return p


POS = ("head", "tail", "partial", "lane0", "lane1", "lane2", "lane3")


# ------------------------------------------------------------------------------------------ 1. absmax_multi
def absmax_segment(n, i, rnd, seed):
    """float32 data of segment i in round rnd, and the position class its single maximum goes to (or None)."""
    rng = np.random.default_rng(seed)
    kind = ("noise", "noise", "neg0", "pm0", "subnormal", "fltmax", "inf", "-inf")[i % 8]
    if kind == "neg0":
        return np.full(n, -0.0, dtype=np.float32), None, None
    if kind == "pm0":
        return np.where(rng.random(n) < 0.5, np.float32(0), np.float32(-0.0)).astype(np.float32), None, None
    if kind == "subnormal":
        x = (rng.integers(1, 1 << 20, n) * 2.0 ** -149).astype(np.float32) * np.where(rng.random(n) < 0.5, -1, 1)
        peak = np.float32(-(2 ** 22) * 2.0 ** -149)
    else:
        x = rng.uniform(-1, 1, n).astype(np.float32)
        peak = {"noise": np.float32(-1.5 - rnd), "fltmax": np.float32(-FLT_MAX),
                "inf": np.float32(np.inf), "-inf": np.float32(-np.inf)}[kind]
    return x.astype(np.float32), peak, POS[(i + rnd) % len(POS)]


def run_absmax(name, rounds):
    lib = _lib()
    spec = table(name)
    for rnd in range(rounds):
        data = []
        for i, (n, off) in enumerate(spec):
            x, peak, pos = absmax_segment(n, i, rnd, _seed(name, i, rnd))
            data.append((x, off, peak, pos))
        segs = place([(x, off) for x, off, _, _ in data])
        for s, (x, off, peak, pos) in zip(segs, data):
            if s is None or peak is None:
                continue
            p = positions(s)
            idx = p.get(pos, p[sorted(p)[0]])
            x[idx] = peak
            s[idx] = float(peak)
        k = len(spec)
        ref = np.array([absmax_bits_ref(x) for x, _, _, _ in data], dtype=np.int64)
        seed = np.array([0 if i % 3 == 0 else (r >> 1 if i % 3 == 1 else min(r + 12345, 0x7F800000))
                         for i, r in enumerate(ref)], dtype=np.int64)
        out = Guarded((k,), torch.int32)
        out.t.copy_(torch.from_numpy(seed.astype(np.uint32).view(np.int32)))
        ptrs, ns = seg_args(segs)

        def run():
            assert lib.pq_absmax_multi_f32(ptrs, ns, k, out.ptr(), _stream()) == 0
        check_landing(run, ["absmax_multi_kernel"]) if rnd == 0 else run()
        torch.cuda.synchronize()
        out.check(name)
        got = out.t.cpu().numpy().view(np.uint32).astype(np.int64)
        bad = np.nonzero(got != np.maximum(seed, ref))[0]
        assert bad.size == 0, (name, rnd, bad[:8], got[bad[:8]], ref[bad[:8]], seed[bad[:8]])
    return total_chunks(segs)


@gpu
@pytest.mark.parametrize("name", TABLES)
def test_absmax_multi(name):
    chunks = run_absmax(name, 2 if name == "cta_spans_segments" else len(POS))
    if name == "ctas_start_mid_segment":
        assert CTAS < chunks < 2 * CTAS
    if name == "cta_spans_segments":
        assert chunks > 2 * CTAS


@gpu
def test_absmax_multi_257_tensors_through_native():
    """257 tensors: _native.absmax_multi splits them into two launches at MAX_SEGMENTS."""
    from common.quantity import _native
    k = 257
    xs, ref = [], []
    for i in range(k):
        n = (0, 1, 3, 1000, CHUNK + 3)[i % 5]
        x, peak, _ = absmax_segment(n, i, 0, _seed("k257", i))
        if peak is not None and n:
            x[n // 2] = peak
        xs.append(torch.from_numpy(x).cuda())
        ref.append(absmax_bits_ref(x))
    out = Guarded((k,), torch.int32)
    out.t.zero_()
    check_landing(lambda: _native.absmax_multi(xs, out.t), ["absmax_multi_kernel"] * 2)
    torch.cuda.synchronize()
    out.check("k257")
    assert np.array_equal(out.t.cpu().numpy().view(np.uint32), np.array(ref, dtype=np.uint32))


@gpu
def test_collector_reads_an_all_negative_zero_max_as_int_zero():
    import common.quantity as cq
    col = cq.DistributionCollector(["z", "x"])
    col.refresh_max_val({"z": torch.full((1001,), -0.0, device="cuda"), "x": torch.tensor([-0.0, -2.5], device="cuda")})
    mv = col.max_vals
    assert type(mv["z"]) is int and mv["z"] == 0
    assert mv["x"] == np.float32(2.5)


# ------------------------------------------------------------------------------------------ 2. per-channel max-abs
def per_channel_case(outer, channels, inner, off, seed):
    """[outer][channels][inner] noise below 1; channel 2j's maximum on the LAST element of one of its planes and
    channel 2j + 1's on the FIRST element of the plane right after it; channel 2 all -0.0; channel 5 peaks at -inf."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1, 1, (outer, channels, inner)).astype(np.float32)
    for c in range(channels):
        o = (c // 2) % outer
        x[o, c, inner - 1 if c % 2 == 0 else 0] = np.float32((2 + rng.integers(0, 1000)) * (-1) ** c)
    if channels > 2:
        x[:, 2, :] = -0.0
    if channels > 5:
        x[outer - 1, 5, inner // 2] = -np.inf
    buf = torch.empty(x.size + off + 4, dtype=torch.float32, device="cuda")
    t = buf[off:off + x.size]
    t.copy_(torch.from_numpy(x.ravel()))
    ref = np.abs(x.astype(np.float64)).max(axis=(0, 2)).astype(np.float32).view(np.uint32).astype(np.int64)
    return t, ref


def per_channel_kernel(outer, channels, inner, ptr):
    per_img = channels * inner
    periodic = inner < 784 and outer >= 16 and per_img % 4 == 0 and ptr % 16 == 0
    return "absmax_periodic_kernel" if periodic else "absmax_per_channel_kernel"


def run_per_channel(outer, channels, inner, off, landing=True):
    t, ref = per_channel_case(outer, channels, inner, off, _seed(outer, channels, inner, off))
    seed = np.where(np.arange(channels) % 3 == 1, 0x7F000000, 0).astype(np.int64)
    out = Guarded((channels,), torch.int32)
    out.t.copy_(torch.from_numpy(seed.astype(np.uint32).view(np.int32)))

    def run():
        assert _lib().pq_absmax_per_channel_f32(t.data_ptr(), outer, channels, inner, out.ptr(), _stream()) == 0
    if landing:
        check_landing(run, [per_channel_kernel(outer, channels, inner, t.data_ptr())])
    else:
        run()
    torch.cuda.synchronize()
    out.check("per-channel")
    got = out.t.cpu().numpy().view(np.uint32).astype(np.int64)
    bad = np.nonzero(got != np.maximum(seed, ref))[0]
    assert bad.size == 0, ((outer, channels, inner, off), bad[:8], got[bad[:8]], ref[bad[:8]])


# (outer, channels, inner, offset in elements): the variant line (inner 783 / 784, outer 15 / 16, C * inner % 4 of
# 0 / 2, 16- against 4-byte alignment), tiny planes, and 1 / 8191 / 8192 channels
PER_CHANNEL_ROWS = [
    (16, 8, 783, 0), (16, 8, 784, 0), (15, 8, 783, 0), (16, 2, 783, 0), (16, 8, 783, 1), (16, 8, 783, 4),
    (16, 8, 784, 3), (64, 32, 1, 0), (40, 16, 2, 0), (40, 7, 3, 0), (20, 3, 5, 0), (17, 4, 5, 0), (33, 6, 3, 2),
    (3, 1, 5000, 0), (2, 8191, 3, 1), (1, 8192, 7, 0), (16, 8192, 1, 0), (200, 64, 49, 0), (5, 64, 3136, 2),
]


@gpu
@pytest.mark.parametrize("row", PER_CHANNEL_ROWS, ids=["o%d_c%d_i%d_off%d" % r for r in PER_CHANNEL_ROWS])
def test_absmax_per_channel(row):
    run_per_channel(*row)


@gpu
@pytest.mark.parametrize("k", range(1, 21))
def test_absmax_per_channel_inner_around_powers_of_two(k):
    """inner = 2^k - 1, 2^k, 2^k + 1: the multiply-shift division of the plane index at every magic shift."""
    for inner in (2 ** k - 1, 2 ** k, 2 ** k + 1):
        if inner < 1:
            continue
        channels = 3 if inner > 4096 else 6
        outer = max(2, min(64, (1 << 21) // (channels * inner)))
        run_per_channel(outer, channels, inner, k % 4, landing=(inner == 2 ** k + 1))


# inner near 2^31 (1.52e9 = 2^30.5): the largest plane remainders the multiply-shift divides.  Here the plane of a
# float4 that starts on the last element of plane 0 is only exact with the magic's shift of 31 + ceil(log2 inner).
BIG_INNER = 1519152477


@gpu
def test_absmax_per_channel_plane_of_1_5e9_elements():
    lib = _lib()
    inner, channels = BIG_INNER, 2
    x = torch.zeros(channels * inner, dtype=torch.float32, device="cuda")
    x[inner - 1] = -7.0                                     # last element of plane 0, at a float4 start
    x[inner] = 3.0                                          # first element of plane 1
    x[2 * inner - 1] = 5.0
    assert (x.data_ptr() // 4 + inner - 1) % 4 == 0
    out = Guarded((channels,), torch.int32)
    out.t.zero_()

    def run():
        assert lib.pq_absmax_per_channel_f32(x.data_ptr(), 1, channels, inner, out.ptr(), _stream()) == 0
    check_landing(run, ["absmax_per_channel_kernel"])
    torch.cuda.synchronize()
    out.check("big plane")
    assert out.t.view(torch.float32).cpu().tolist() == [7.0, 5.0]
    del x
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------ 3. epilogues
def epi_operands(n, seed):
    """float32: noise, +-0, subnormals, +-FLT_MAX (sums overflow to inf), +-inf, never inf - inf."""
    rng = np.random.default_rng(seed)
    a = rng.normal(0, 3, n).astype(np.float32)
    sp = np.array([0.0, -0.0, 2.0 ** -149, -2.0 ** -140, FLT_MAX, -FLT_MAX, np.inf, -np.inf, 1e-30], dtype=np.float32)
    a[::5] = np.resize(sp, a[::5].size)
    return a


def epi_ref(a, b):
    with np.errstate(over="ignore"):
        o = (a.astype(np.float64) + b.astype(np.float64)).astype(np.float32)
    return o, np.maximum(o, np.float32(0))


# (entry, N, C, hw or n, kernel)
EPI_ROWS = [
    ("conv", 2, 3, 64, "epilogue_kernel<0>"), ("conv", 64, 64, 784, "epilogue_kernel<0>"),
    ("conv", 2, 5, 49, "epilogue_kernel<1>"), ("conv", 3, 7, 1, "epilogue_kernel<1>"),
    ("conv", 32, 512, 49, "epilogue_kernel<1>"), ("add", 1, 1, 1001, "epilogue_kernel<2>"),
    ("add", 1, 1, 4096 * 1200 + 3, "epilogue_kernel<2>"),
]


@gpu
@pytest.mark.parametrize("row", EPI_ROWS, ids=["%s_%d_%d_%d" % r[:4] for r in EPI_ROWS])
def test_epilogue(row):
    entry, N, C, hw, kernel = row
    lib = _lib()
    n = N * C * hw
    a = epi_operands(n, _seed(row))
    if entry == "conv":
        bias = np.random.default_rng(_seed(row, "b")).normal(0, 2, C).astype(np.float32)
        bias[:3] = np.resize(np.array([-0.0, FLT_MAX, 2.0 ** -145], dtype=np.float32), min(3, C))
        b_full = np.broadcast_to(bias[None, :, None], (N, C, hw)).ravel()
        b_dev = torch.from_numpy(bias).cuda()
    else:
        b_full = epi_operands(n, _seed(row, "b"))
        b_full[np.isinf(a)] = 1.0                            # never inf - inf: the max of a NaN is out of scope
        b_dev = torch.from_numpy(b_full).cuda()
    o_ref, r_ref = epi_ref(a, b_full)
    m_ref = absmax_bits_ref(o_ref)
    for relu in (True, False):
        y = Guarded((n,), torch.float32)
        y.t.copy_(torch.from_numpy(a))
        z = Guarded((n,), torch.float32) if entry == "add" else None
        r = Guarded((n,), torch.float32)
        slots = Guarded((3,), torch.int32)
        slots.t.copy_(torch.tensor([0x11, 0x3F000000, 0x22], dtype=torch.int32))
        slot = slots.ptr() + 4
        rp = r.ptr() if relu else None

        def run():
            if entry == "conv":
                rc = lib.pq_conv_epilogue_f32(y.ptr(), b_dev.data_ptr(), N, C, hw, rp, slot, _stream())
            else:
                rc = lib.pq_eltwise_add_f32(y.ptr(), b_dev.data_ptr(), z.ptr(), n, rp, slot, _stream())
            assert rc == 0
        check_landing(run, [kernel]) if relu else run()
        torch.cuda.synchronize()
        out = y if entry == "conv" else z
        for g in (y, r, slots) + ((z,) if z else ()):
            g.check(row)
        assert np.array_equal(out.t.cpu().numpy().view(np.uint32), o_ref.view(np.uint32)), row
        if relu:
            assert np.array_equal(r.t.cpu().numpy(), r_ref), row
        else:
            assert _untouched(r)
        got = slots.t.cpu().numpy().view(np.uint32)
        assert got[0] == 0x11 and got[2] == 0x22 and got[1] == max(0x3F000000, m_ref), (row, got, m_ref)


# ------------------------------------------------------------------------------------------ 4. histograms
NORMAL_INTERVALS = (2.0 ** -126, 1e-12, 1e35, FLT_MAX, 0.0123456, 3.0, 1.7e-20, 2.0 ** -3, 7.1e-7, 0.3)
SUBNORMAL_INTERVALS = (2.0 ** -149, 3 * 2.0 ** -149, 2.0 ** -140, 1e-40, 2.0 ** -127, float(np.nextafter(
    np.float32(2.0 ** -126), np.float32(0))))


def intervals_for(k, pool, seed):
    rng = np.random.default_rng(seed)
    extra = (2.0 ** rng.uniform(-60, 60, k)).astype(np.float32)
    return np.array([pool[i % len(pool)] if i % 2 == 0 else extra[i] for i in range(k)], dtype=np.float32)


def zero_dense(n, d, seed):
    """Every float4 holds an exact zero; the rest are ambiguous values (one ulp around bin edges) and values just
    above 0 and just below 1: a warp flags all its float4s because of zeros and switches to the zero-aware variant."""
    rng = np.random.default_rng(seed)
    d = np.float32(d)
    with np.errstate(over="ignore"):
        edges = (np.arange(0, 40, dtype=np.float64) * np.float64(d)).astype(np.float32)
    amb = np.concatenate([neighbours(edges, 1), neighbours(np.array([d], dtype=np.float32) * np.float32(1e-4), 1)])
    x = rng.choice(amb, n).astype(np.float32)
    x[::4] = 0.0
    x[2::8] = -0.0
    return x


def hist_case(name, nbins, pool, zero_rows=False):
    spec = table(name)
    ivs = intervals_for(len(spec), pool, _seed(name, nbins, pool))
    arrays = []
    for i, ((n, off), d) in enumerate(zip(spec, ivs)):
        if zero_rows and i % 3 == 1 and n >= 2 * CHUNK:
            x = zero_dense(n, d, _seed(name, i))
        else:
            v = hist_values(d, nbins, _seed(name, nbins, i))
            x = np.resize(np.roll(v, i * 7), n).astype(np.float32)
        arrays.append((x, off))
    return spec, ivs, arrays


def run_hist(name, nbins, pool, kernel, zero_rows=False):
    lib = _lib()
    spec, ivs, arrays = hist_case(name, nbins, pool, zero_rows)
    k = len(spec)
    segs = place(arrays)
    ref = np.stack([hist_ref(x, d, nbins) for (x, _), d in zip(arrays, ivs)])
    seed = np.random.default_rng(_seed(name, "seed")).integers(0, 1 << 40, (k, nbins)).astype(np.int64)
    out = Guarded((k, nbins), torch.int64)
    out.t.copy_(torch.from_numpy(seed))
    ptrs, ns = seg_args(segs)
    iv = (ctypes.c_float * k)(*[float(d) for d in ivs])

    def run():
        if nbins == 2048:
            rc = lib.pq_hist2048_multi_f32(ptrs, ns, iv, k, out.ptr(), _stream())
        else:
            rc = lib.pq_hist_multi_f32(ptrs, ns, iv, k, nbins, out.ptr(), _stream())
        assert rc == 0
    check_landing(run, [kernel])
    torch.cuda.synchronize()
    out.check(name)
    got = out.t.cpu().numpy() - seed
    for i in range(k):
        if not np.array_equal(got[i], ref[i]):
            diff = np.nonzero(got[i] != ref[i])[0]
            raise AssertionError("%s seg %d (n=%d, d=%r): bins %s got %s want %s"
                                 % (name, i, spec[i][0], float(ivs[i]), diff[:8], got[i][diff[:8]], ref[i][diff[:8]]))


@gpu
@pytest.mark.parametrize("name", TABLES)
def test_hist2048(name):
    run_hist(name, 2048, NORMAL_INTERVALS, "hist_multi_kernel<1,8>", zero_rows=True)


@gpu
@pytest.mark.parametrize("name", ("k2_offsets", "many_chunks", "k256_mixed"))
def test_hist2048_subnormal_intervals(name):
    """A subnormal bin width (1 / d overflows fp32 below 1 / FLT_MAX): the call divides literally."""
    run_hist(name, 2048, SUBNORMAL_INTERVALS, "hist_generic_kernel")


@gpu
def test_hist2048_nan_lands_in_the_top_bin_wherever_it_sits():
    """A NaN (and inf / inf) counts in bin 2047 in the unaligned head, a full chunk, the last partial chunk and the
    tail alike."""
    lib = _lib()
    n = 2 * CHUNK + 4 * 5 + 2
    seg = place([(np.full(n, 0.5, dtype=np.float32), 1), (np.full(n, np.inf, dtype=np.float32), 1)])
    for s in seg[:1]:
        for idx in positions(s).values():
            s[idx] = float("nan")
    out = Guarded((2, 2048), torch.int64)
    out.t.zero_()
    ptrs, ns = seg_args(seg)
    iv = (ctypes.c_float * 2)(1.0, float("inf"))
    assert lib.pq_hist2048_multi_f32(ptrs, ns, iv, 2, out.ptr(), _stream()) == 0
    torch.cuda.synchronize()
    got = out.t.cpu().numpy()
    npos = len(positions(seg[0]))
    assert got[0, 2047] == npos and got[0, 0] == n - npos and got[0].sum() == n
    assert got[1, 2047] == n and got[1].sum() == n


GENERIC_NBINS = (1, 2, 3, 127, 129, 2047, 2049, 4095, 8192)


@gpu
@pytest.mark.parametrize("nbins", GENERIC_NBINS)
def test_hist_generic(nbins):
    for name in ("k2_offsets", "many_chunks", "k255_tiny"):
        run_hist(name, nbins, NORMAL_INTERVALS + SUBNORMAL_INTERVALS, "hist_generic_kernel")
    if nbins in (3, 2049):
        run_hist("ctas_start_mid_segment", nbins, NORMAL_INTERVALS, "hist_generic_kernel")


# ------------------------------------------------------------------------------------------ 5. KL search
KL_NBINS = (129, 130, 136, 255, 256, 257, 1000, 2047, 2048, 2049, 4096, 8191, 8192)
FAMILIES = ("zero", "spike0", "spike127", "spike128", "spike_last", "upper", "zero_runs", "big_odd", "noise")


def kl_family(fam, nbins, seed):
    """float64 integer counts [nbins]."""
    rng = np.random.default_rng(seed)
    c = np.zeros(nbins)
    if fam.startswith("spike"):
        c[{"spike0": 0, "spike127": 127, "spike128": 128, "spike_last": nbins - 1}[fam]] = rng.integers(1, 10 ** 6)
    elif fam == "upper":                                      # no mass below bin 128
        c[128:] = rng.integers(0, 5000, nbins - 128)
    elif fam == "zero_runs":                                  # zero runs longer than one target bin (count = 1e-12)
        c[:] = np.round(1e5 * np.exp(-((np.arange(nbins) / (0.3 * nbins)) ** 2))) + 1
        run = nbins // 128 + 2
        for s in range(3, nbins - run, 5 * run):
            c[s:s + run] = 0
    elif fam == "big_odd":                                    # odd counts above 2^24: float32 rounds them
        c[:] = 2 * rng.integers(1 << 23, 1 << 29, nbins) + 1
        c[rng.integers(0, nbins, nbins // 4)] = 0
    elif fam == "noise":
        c[:] = np.round(np.abs(rng.normal(0, 1, nbins)) * 1e4 * np.exp(-np.arange(nbins) / (0.2 * nbins)))
    return c


def kl_ref(oracle, counts):
    return oracle.kl_search(oracle.normalize(counts))


def kl_kernels(nbins):
    return ["kl_prepare_kernel", "kl_candidate_kernel<%d>" % (2048 if nbins <= 2048 else 8192), "kl_argmin_kernel"]


def run_kl(oracle, counts, landing=False, refs=None):
    lib = _lib()
    k, nbins = counts.shape
    cand = nbins - 128
    dev = torch.from_numpy(counts).cuda()
    ws = torch.empty(k * lib.pq_kl_workspace_doubles_n(nbins), dtype=torch.float64, device="cuda")
    thr = Guarded((k,), torch.int32)
    kl = Guarded((k, cand), torch.float64)

    def run():
        assert lib.pq_kl_search_n_f64(dev.data_ptr(), k, nbins, ws.data_ptr(), kl.ptr(), thr.ptr(), _stream()) == 0
    check_landing(run, kl_kernels(nbins)) if landing else run()
    torch.cuda.synchronize()
    thr.check("thresholds")
    kl.check("curves")
    got_t, got_kl = thr.t.cpu().numpy(), kl.t.cpu().numpy()
    for i in range(k):
        t, curve = refs[i] if refs else kl_ref(oracle, counts[i])
        np.testing.assert_allclose(got_kl[i], curve, rtol=1e-9, atol=1e-300, err_msg="row %d" % i)
        assert got_t[i] == t, (i, got_t[i], t)


@gpu
@pytest.mark.parametrize("nbins", KL_NBINS)
def test_kl_search(oracle, nbins):
    fams = [kl_family(f, nbins, _seed(f, nbins)) for f in FAMILIES]
    refs = [kl_ref(oracle, c) for c in fams]
    run_kl(oracle, np.stack(fams[7:8]), landing=True, refs=refs[7:8])                 # k = 1
    run_kl(oracle, np.stack(fams[:7]), refs=refs[:7])                                 # k = 7
    order = np.random.default_rng(nbins).permutation(np.resize(np.arange(len(fams)), 300 if nbins <= 2049 else 30))
    run_kl(oracle, np.stack([fams[j] for j in order]), refs=[refs[j] for j in order])  # every family, mixed


@gpu
def test_kl_int64_counts_above_2_31_through_quantizer(oracle):
    import common.quantity as cq
    rng = np.random.default_rng(31)
    names = ["a", "b", "c"]
    counts = {n: (2 * rng.integers(1 << 30, 1 << 33, 2048) + 1) * (rng.random(2048) < 0.7) for n in names}
    counts["c"][300:] = 0
    dists = {n: torch.from_numpy(c.astype(np.int64)).cuda() for n, c in counts.items()}
    intervals = {n: np.float32(0.01 * (i + 1)) for i, n in enumerate(names)}
    q = cq.Quantizer(names, keep_curves=True)
    q.quantize(dists, intervals)
    curves = q.kl_curves.cpu().numpy()
    for i, n in enumerate(names):
        assert counts[n].max() > 2 ** 31
        t, curve = kl_ref(oracle, counts[n].astype(np.float64))
        np.testing.assert_allclose(curves[i], curve, rtol=1e-9, atol=1e-300)
        assert q.threshold_bin[n] == t and q.bits[n] == oracle.threshold_to_bit(t, intervals[n])[0]


@gpu
def test_kl_65535_tensors_per_call_and_more_through_native(oracle):
    """The C entry point takes k = 65535 and refuses 65536 (writing nothing); _native.kl_search splits 65536."""
    from common.quantity import _native
    lib = _lib()
    nbins = 129
    distinct = [kl_family(FAMILIES[j % len(FAMILIES)], nbins, _seed("k64k", j)) for j in range(97)]
    refs = [kl_ref(oracle, c) for c in distinct]
    rows = np.arange(65536) * 31 % 97
    counts = torch.from_numpy(np.stack(distinct)[rows]).cuda()
    want_kl = np.array([refs[j][1][0] for j in rows])
    ws = torch.empty(65536 * lib.pq_kl_workspace_doubles_n(nbins), dtype=torch.float64, device="cuda")
    for k, rc_want in ((65536, EUNSUPPORTED), (65535, 0)):
        thr, kl = Guarded((k,), torch.int32), Guarded((k, 1), torch.float64)
        rc = lib.pq_kl_search_n_f64(counts.data_ptr(), k, nbins, ws.data_ptr(), kl.ptr(), thr.ptr(), _stream())
        torch.cuda.synchronize()
        assert rc == rc_want
        if rc_want:
            assert _untouched(thr, kl)
            continue
        thr.check("65535")
        kl.check("65535")
        np.testing.assert_allclose(kl.t.cpu().numpy()[:, 0], want_kl[:k], rtol=1e-9, atol=1e-300)
        assert (thr.t.cpu().numpy() == 128).all()
    got = {}

    def run():
        got["thr"], got["kl"] = _native.kl_search(counts, want_curves=True)
    check_landing(run, kl_kernels(nbins) * 2)
    torch.cuda.synchronize()
    np.testing.assert_allclose(got["kl"].cpu().numpy()[:, 0], want_kl, rtol=1e-9, atol=1e-300)
    assert (got["thr"].cpu().numpy() == 128).all()


# ------------------------------------------------------------------------------------------ 6. argument limits
@gpu
def test_one_step_beyond_each_limit():
    """One step beyond each argument limit returns the documented code and writes nothing; one step inside is
    accepted."""
    lib = _lib()
    s = _stream()
    x = torch.ones(6 * CHUNK, device="cuda")               # also holds the 5 chunks a truncated count would read

    def call_multi(ptrs, ns, ivs=None, nbins=2048, want=0):
        k = len(ptrs)
        pa = (ctypes.c_void_p * max(k, 1))(*ptrs)
        na = (ctypes.c_uint64 * max(k, 1))(*ns)
        iv = (ctypes.c_float * max(k, 1))(*(ivs if ivs is not None else [1.0] * k))
        m = Guarded((max(k, 1),), torch.int32)
        h = Guarded((max(k, 1), nbins), torch.int64)
        rcs = [lib.pq_absmax_multi_f32(pa, na, k, m.ptr(), s) if ivs is None else None,
               lib.pq_hist2048_multi_f32(pa, na, iv, k, h.ptr(), s) if nbins == 2048 else
               lib.pq_hist_multi_f32(pa, na, iv, k, nbins, h.ptr(), s)]
        torch.cuda.synchronize()
        for rc in rcs:
            assert rc in (None, want), (rcs, want, k)
        if want:
            assert _untouched(m, h)
        else:
            m.check("accepted")
            h.check("accepted")

    p = x.data_ptr()
    # segment count
    call_multi([p] * 257, [8] * 257, want=ETOOMANY)
    call_multi([p] * 256, [8] * 256)
    call_multi([p] * 257, [8] * 257, ivs=[1.0] * 257, nbins=1000, want=ETOOMANY)
    # null pointer with n > 0, misaligned pointer
    call_multi([p, None], [8, 1], want=EINVAL)
    call_multi([p, None], [8, 0])
    call_multi([p + 2], [8], want=EALIGN)
    call_multi([p + 4], [8])
    # intervals: 0, -0, NaN, -1 refused, the smallest subnormal accepted
    for bad in (0.0, -0.0, float("nan"), -1.0):
        for nb in (2048, 1000):
            call_multi([p, p], [8, 8], ivs=[1.0, bad], nbins=nb, want=EINVAL)
    call_multi([p], [CHUNK], ivs=[2.0 ** -149])
    call_multi([p], [CHUNK], ivs=[2.0 ** -149], nbins=1000)
    # nbins
    call_multi([p], [8], ivs=[1.0], nbins=1)
    call_multi([p], [8], ivs=[1.0], nbins=8192)
    for nb, want in ((0, EINVAL), (-3, EINVAL), (8193, EUNSUPPORTED)):
        pa, na, iv = (ctypes.c_void_p * 1)(p), (ctypes.c_uint64 * 1)(8), (ctypes.c_float * 1)(1.0)
        h = Guarded((1, 16), torch.int64)
        assert lib.pq_hist_multi_f32(pa, na, iv, 1, nb, h.ptr(), s) == want
        assert _untouched(h)
    # a table of more than 2^32 - 1 chunks, refused before any launch: one huge segment, and two that fit alone
    call_multi([p], [(1 << 32) * CHUNK], want=EUNSUPPORTED)
    call_multi([p], [(1 << 32) * CHUNK + 5 * CHUNK], want=EUNSUPPORTED)
    call_multi([p, p], [((1 << 32) - 1) * CHUNK] * 2, want=EUNSUPPORTED)

    # pq_absmax_per_channel_f32
    def per_channel(ptr, outer, channels, inner, want):
        m = Guarded((max(channels, 1),), torch.int32)
        m.t.zero_()
        rc = lib.pq_absmax_per_channel_f32(ptr, outer, channels, inner, m.ptr(), s)
        torch.cuda.synchronize()
        assert rc == want, (outer, channels, inner, rc)
        if want:
            assert bool((m.t == 0).all())
        m.check("per-channel limit")
    big = torch.ones(8192 * 7, device="cuda")
    per_channel(big.data_ptr(), 1, 8193, 1, EUNSUPPORTED)
    per_channel(big.data_ptr(), 1, 8192, 7, 0)
    per_channel(big.data_ptr(), 1, -1, 7, EINVAL)
    per_channel(None, 1, 4, 7, EINVAL)
    per_channel(big.data_ptr() + 2, 1, 4, 7, EALIGN)
    per_channel(big.data_ptr() + 4, 1, 4, 7, 0)
    per_channel(big.data_ptr(), 1, 1, (1 << 31) - (1 << 14), EUNSUPPORTED)
    per_channel(big.data_ptr(), 1 << 18, 8192, 1, EUNSUPPORTED)                  # outer * channels = 2^31
    per_channel(big.data_ptr(), 1 << 20, 1, 1 << 30, EUNSUPPORTED)              # 2^37 chunks
    per_channel(big.data_ptr(), 0, 4, 7, 0)

    # the two epilogue entry points
    y = Guarded((4096,), torch.float32)
    y2 = Guarded((4096,), torch.float32)
    b = torch.zeros(4096, device="cuda")
    slot = Guarded((1,), torch.int32)

    def epi(rc, *gs):
        torch.cuda.synchronize()
        assert rc[0] == rc[1], rc
        if rc[1]:
            assert _untouched(y, y2, slot, *gs)
    yp, bp, y2p, sp = y.ptr(), b.data_ptr(), y2.ptr(), slot.ptr()
    epi((lib.pq_conv_epilogue_f32(yp, bp, -1, 4, 16, None, sp, s), EINVAL))
    epi((lib.pq_conv_epilogue_f32(yp, bp, 1, 0, 16, None, sp, s), EINVAL))
    epi((lib.pq_conv_epilogue_f32(yp, bp, 1, 4, 16, yp, sp, s), EINVAL))
    epi((lib.pq_conv_epilogue_f32(yp + 4, bp, 1, 4, 16, None, sp, s), EALIGN))
    epi((lib.pq_conv_epilogue_f32(yp, bp, 1, 4, 16, y2p + 4, sp, s), EALIGN))
    epi((lib.pq_conv_epilogue_f32(yp, bp + 2, 1, 4, 16, None, sp, s), EALIGN))
    epi((lib.pq_conv_epilogue_f32(yp, bp, 1, 4, 1 << 31, None, sp, s), EUNSUPPORTED))
    epi((lib.pq_conv_epilogue_f32(yp, bp, 1 << 16, 1 << 15, 4, None, sp, s), EUNSUPPORTED))
    epi((lib.pq_conv_epilogue_f32(yp, bp, 5, 1, (1 << 31) - 4, None, sp, s), EUNSUPPORTED))   # n >= 2^33
    epi((lib.pq_conv_epilogue_f32(yp, bp, 2, 1, (1 << 30) + 1, None, sp, s), EUNSUPPORTED))   # 7x7-like, >= 2^31
    epi((lib.pq_conv_epilogue_f32(yp, bp, 0, 4, 16, None, sp, s), 0))
    epi((lib.pq_eltwise_add_f32(yp, bp, yp, 16, None, sp, s), EINVAL))
    epi((lib.pq_eltwise_add_f32(yp, bp, y2p, 16, y2p, sp, s), EINVAL))
    epi((lib.pq_eltwise_add_f32(yp, bp, y2p, 16, bp, sp, s), EINVAL))
    epi((lib.pq_eltwise_add_f32(yp + 4, bp, y2p, 16, None, sp, s), EALIGN))
    epi((lib.pq_eltwise_add_f32(yp, bp, y2p, 1 << 33, None, sp, s), EUNSUPPORTED))
    epi((lib.pq_eltwise_add_f32(yp, bp, y2p, 0, None, sp, s), 0))
    y.t.zero_()
    slot.t.zero_()
    assert lib.pq_conv_epilogue_f32(yp, bp, 1, 4, 16, None, sp, s) == 0
    assert lib.pq_eltwise_add_f32(yp, bp, y2p, 4093, None, sp, s) == 0
    torch.cuda.synchronize()
    y2.check("eltwise accepted")
    assert bool((y2.t[:4093] == 0).all()) and bool((y2.t.view(torch.uint8)[4 * 4093:] == SENTINEL).all())

    # KL
    c = torch.ones((2, 8192), dtype=torch.float64, device="cuda")
    ws = torch.empty(2 * 3 * 8192, dtype=torch.float64, device="cuda")
    for nb, k, want in ((128, 1, EINVAL), (129, 1, 0), (8193, 1, EUNSUPPORTED), (8192, 1, 0), (200, -1, EINVAL),
                        (200, 0, 0), (200, 65536, EUNSUPPORTED)):
        thr = Guarded((2,), torch.int32)
        kl = Guarded((2, 8192), torch.float64)
        rc = lib.pq_kl_search_n_f64(c.data_ptr(), k, nb, ws.data_ptr(), kl.ptr(), thr.ptr(), s)
        torch.cuda.synchronize()
        assert rc == want, (nb, k, rc)
        if want or k == 0:
            assert _untouched(thr, kl)
        else:
            thr.check("kl")
            kl.check("kl")
    thr = Guarded((1,), torch.int32)
    assert lib.pq_kl_search_n_f64(None, 1, 200, ws.data_ptr(), None, thr.ptr(), s) == EINVAL
    assert lib.pq_kl_search_n_f64(c.data_ptr(), 1, 200, None, None, thr.ptr(), s) == EINVAL
    torch.cuda.synchronize()
    assert _untouched(thr)


# ------------------------------------------------------------------------------------------ kernel census
# Every kernel of pq_stats.cu / pq_stats_kernels.cuh / pq_kl.cu and the test whose rows land on it.
KERNELS = {
    "absmax_multi_kernel": "test_absmax_multi",
    "absmax_per_channel_kernel": "test_absmax_per_channel",
    "absmax_periodic_kernel": "test_absmax_per_channel",
    "epilogue_kernel<0>": "test_epilogue",
    "epilogue_kernel<1>": "test_epilogue",
    "epilogue_kernel<2>": "test_epilogue",
    "hist_multi_kernel<1,8>": "test_hist2048",
    "hist_generic_kernel": "test_hist_generic",
    "kl_prepare_kernel": "test_kl_search",
    "kl_candidate_kernel<2048>": "test_kl_search",
    "kl_candidate_kernel<8192>": "test_kl_search",
    "kl_argmin_kernel": "test_kl_search",
}
FAMILY_NAMES = {k.split("<")[0] for k in KERNELS}
ROW_KERNELS = ({per_channel_kernel(o, c, i, 16 if off % 4 == 0 else 4) for o, c, i, off in PER_CHANNEL_ROWS} |
               {r[-1] for r in EPI_ROWS} | {k for nb in KL_NBINS for k in kl_kernels(nb)} |
               {"absmax_multi_kernel", "hist_multi_kernel<1,8>", "hist_generic_kernel"})


def library_kernels():
    from common.quantity import _native
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not installed")
    sym = subprocess.run(["cuobjdump", "-symbols", _native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = subprocess.run(["cu++filt"], input=sym, check=True, capture_output=True, text=True).stdout
    return {kernel_id(line) for line in names.splitlines() if "STO_ENTRY" in line}


def test_kernel_table_equals_library_symbols():
    """KERNELS is exactly the library's statistics / KL kernels (every instantiation): one added without a row here
    fails, and every kernel is the landing target of some row."""
    found = library_kernels()
    assert len(KERNELS) == 12
    assert {k for k in found if k.split("<")[0] in FAMILY_NAMES} == set(KERNELS)
    for test in set(KERNELS.values()):
        assert callable(globals().get(test)), test
    assert ROW_KERNELS == set(KERNELS)


def test_kernel_id_spellings():
    assert kernel_id("void pq::hist_multi_kernel<1, 8>(pq::SegTable, unsigned long long *)") == "hist_multi_kernel<1,8>"
    assert kernel_id("void pq::epilogue_kernel<(int)2>(pq::EpiArgs)") == "epilogue_kernel<2>"
    assert kernel_id("pq::kl_argmin_kernel(const double *, int *, pq::KlGeom)") == "kl_argmin_kernel"
    assert kernel_id("void at::native::vectorized_elementwise_kernel<4>(int)") is None


# ------------------------------------------------------------------------------------------ CPU: the references
def test_hist_reference_equals_oracle(oracle):
    """hist_ref is oracle.hist (the C restatement of the reference) on finite inputs, subnormal widths included."""
    rng = np.random.default_rng(3)
    for nbins in (1, 3, 129, 2048, 8192):
        for d in NORMAL_INTERVALS + SUBNORMAL_INTERVALS + (1.0, 2.5e-3):
            v = hist_values(d, nbins, 1)
            v = v[np.isfinite(v)]
            with np.errstate(over="ignore"):
                x = np.concatenate([v, rng.normal(0, 1, 2000).astype(np.float32) * np.float32(d) * nbins])
            assert np.array_equal(hist_ref(x, d, nbins), oracle.hist(x, np.float32(d), nbins)), (nbins, d)


def test_hist_reference_nan_and_infinite_quotients():
    h = hist_ref(np.concatenate([NANS, _f32([np.inf, -np.inf, 0.0, -0.0, 1.0])]), np.float32(np.inf), 16)
    assert h[15] == len(NANS) + 2 and h[0] == 1 and h.sum() == len(NANS) + 3
    assert hist_ref(_f32([FLT_MAX, 2.0 ** -149]), 2.0 ** -149, 2048).tolist()[2047] == 1


def test_crafted_values_reach_the_ambiguous_band():
    """The crafted widths put values where RN(|x| * RN(1/d)) truncates below the correctly rounded quotient (the
    fast path's provisional bin is wrong and only the redo pass files the element), including just below 1, and
    the zero-dense rows hold such values next to their zeros."""
    below_one = wrong = 0
    for d in NORMAL_INTERVALS + tuple(intervals_for(40, NORMAL_INTERVALS, 9)):
        d = np.float32(d)
        for v in (hist_values(d, 2048, 0), zero_dense(4096, d, 0)):
            a = np.abs(v[np.isfinite(v) & (v != 0)])
            with np.errstate(all="ignore"):
                q0 = np.minimum(a * (np.float32(1) / d), np.float32(2047.5)).astype(np.float32)
                q = (a.astype(np.float64) / np.float64(d)).astype(np.float32)
            lo = np.trunc(q0) < np.trunc(np.minimum(q, 2047))
            wrong += int(lo.sum())
            below_one += int((lo & (q0 < 1)).sum())
    assert wrong > 50 and below_one > 5, (wrong, below_one)


def test_kl_families_have_the_intended_shape(oracle):
    for nbins in (129, 2048):
        fams = {f: kl_family(f, nbins, _seed(f, nbins)) for f in FAMILIES}
        for f in ("zero", "spike0"):                            # exact ties: the first candidate must win
            t, curve = kl_ref(oracle, fams[f])
            assert t == 128 and (curve == curve[0]).all() and curve[0] < 66666, f
        c = fams["big_odd"]
        assert (c % 2 == 1).sum() > nbins // 2 and c.max() > 2 ** 24
        assert (c.astype(np.float32).astype(np.float64) != c).any()
        z = fams["zero_runs"]
        run = max(len(r) for r in "".join("0" if v == 0 else "1" for v in z).split("1"))
        assert run > nbins / 128
        assert fams["upper"][:128].sum() == 0 and fams["upper"][128:].sum() > 0

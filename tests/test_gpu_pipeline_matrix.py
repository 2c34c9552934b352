"""Every kernel of the int8 pipeline (pq_pipeline.cu) and of the elementwise / input-quantiser library
(pq_elementwise.cu), over its whole argument range, against references that share no code with the kernels:

    quantisers   clamp(round(x.double() * 2**ib), -128, 127), then torch indexing (permute, F.unfold, padding)
    max-pool     F.max_pool2d of the fp32 NCHW tensor [ReLU]             (max is exact on int8 values)
    avg-pool     F.avg_pool2d of the de-quantised fp32 NCHW tensor        (the fp32-boundary model's own operation)
    add          the exact int64 NewAdd of test_gpu_epilogue_matrix.add_ref, tied to oracle.add_clamp below
    concat       oracle.concat_quantize of the de-quantised sources
    fp32 kernels numpy fp32 restatements of NewAdd / RightShift / Sp / DeQuantity, pinned to intsim.npz below;
                 compared as bit patterns, so the sign of a zero counts

For the quantisers, clamp(round(x.double() * 2**ib), -128, 127) equals the fp32 arithmetic of Quantity(ib)
(rint(x * 2^ib) in fp32, then the clamp) for every finite or infinite x and |ib| <= 126: the float64 product of a
float32 and a power of two in that range is exact, and wherever the fp32 product overflows (to +-inf) or underflows
(to a subnormal or zero, |product| < 2^-126 < 1/2) the rounded, clamped result is the same (saturated, or 0).
NaN is out of scope: the int8 format has no NaN.

Every output is written into the middle of a sentinel-filled buffer (Guarded): every byte of the output must equal
the reference, so bytes a kernel fails to write show up as 0xA5, and the guard bytes around it must survive.  Each
row names the kernel its launch must land on (checked with torch.profiler).  KERNELS lists every kernel of the two
files with the test that reaches it, and test_kernel_table_equals_library_symbols keeps that list complete.
"""
import os
import re
import shutil
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import det_inputs
from conftest import load_golden
from test_gpu_epilogue_matrix import SENTINEL, Guarded, _stream, add_ref

gpu = pytest.mark.gpu
EINVAL, EUNSUPPORTED, EALIGN, ETOOMANY = -1, -2, -3, -4
CAP_THREADS = 148 * 16 * 256          # the bandwidth kernels' grid cap (kNumSMs * 16 blocks of 256 threads)
FLT_MAX = float(np.finfo(np.float32).max)
IBS = (-126, -20, -1, 0, 1, 4, 7, 20, 126)


def _lib():
    from common.quantity import _native
    return _native.lib()


# ------------------------------------------------------------------------------------------ kernel names
def kernel_id(name):
    """'quantize_s2d16_kernel<true>' from a demangled name in either spelling: cu++filt's
    'void pq::quantize_s2d16_kernel<(bool)1>(const float *, ...)' or the profiler's '...<true>(...)'."""
    s = re.sub(r"\(bool\)1", "true", name)
    s = re.sub(r"\(bool\)0", "false", s)
    s = re.sub(r"\(int\)(-?\d+)", r"\1", s)
    m = re.search(r"pq::(\w+)(<[^>()]*>)?", s)
    return m.group(1) + (m.group(2) or "").replace(" ", "") if m else None


def launched(fn):
    """Names of every CUDA kernel fn() launched."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_FRESH_ENV = "PQ_PIPELINE_MATRIX_FRESH"
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


def check_landing(fn, kernel):
    state = _landing_state()
    if state["recorded"]:
        names = launched(fn)
        assert [k for k in map(kernel_id, names) if k] == [kernel], (kernel, names)
    else:
        fn()
        rc, out = state["fresh_run"]
        assert rc == 0, "the fresh-process run of this file, which makes the landing checks, failed:\n" + out


def _tf(b):
    return "true" if b else "false"


def add_kernel(a16, b16, relu_in, qdown):
    return "add_requant_kernel<%s,%s,%s,%s>" % (_tf(a16), _tf(b16), _tf(relu_in), _tf(qdown))


# ------------------------------------------------------------------------------------------ crafted inputs
def crafted_values(ib):
    """float32: every tie (m + 1/2) * 2^-ib for m in -131..130 that is a finite float (across both saturation edges:
    127.5 -> 127, -128.5 -> -128, -129.5 -> -128), the float neighbours of each tie, and the specials.  Odd length,
    so a tiled copy puts every value in every lane of a 4- or 16-wide vector."""
    ties = (np.arange(-131, 131, dtype=np.float64) + 0.5) * 2.0 ** -ib
    ties = ties[np.abs(ties) <= FLT_MAX].astype(np.float32)
    assert np.array_equal(ties.astype(np.float64) * 2.0 ** ib % 1, np.full(len(ties), 0.5))
    up, down = np.nextafter(ties, np.float32(np.inf)), np.nextafter(ties, np.float32(-np.inf))
    specials = np.array([0.0, -0.0, np.inf, -np.inf, FLT_MAX, -FLT_MAX, 2.0 ** -149, -2.0 ** -149, 2.0 ** -126,
                         -2.0 ** -126], dtype=np.float32)
    v = np.concatenate([ties, up, down, specials])
    return v if len(v) % 2 else np.append(v, np.float32(1.0))


def crafted(shape, ib, seed):
    """A float32 CUDA tensor of `shape`: the crafted values of `ib` tiled over it (so they reach every lane, tile edge
    and image border), every seventh element bell-shaped noise spanning the int8 range."""
    n = int(np.prod(shape))
    v = np.resize(crafted_values(ib), n)
    noise = np.clip(det_inputs.bell(n, seed, 40.0).astype(np.float64) * 2.0 ** -ib, -FLT_MAX, FLT_MAX)
    v[3::7] = noise.astype(np.float32)[3::7]
    return torch.from_numpy(v.reshape(shape)).cuda()


def q_ref(x, ib):
    """Quantity(ib) of fp32 x as int64 (see the module docstring for why float64 is exact here)."""
    return torch.round(x.double() * 2.0 ** ib).clamp(-128, 127).long()


def offset_view(t, elems=1):
    """A copy of t that starts `elems` elements into its allocation (4 bytes for fp32: not 8- or 16-byte aligned)."""
    buf = torch.empty(t.numel() + elems, dtype=t.dtype, device=t.device)
    v = buf[elems:].view(t.shape)
    v.copy_(t)
    return v


def _seed(*key):
    return zlib.crc32(repr(key).encode()) & 0xFFFF


# ------------------------------------------------------------------------------------------ 1. input quantisers
# (N, C, H, W, c_pad, x at a 4-byte offset, kernel)
NHWC_ROWS = [
    (2, 40, 12, 12, 64, False, "quantize_nchw_nhwc_vec_kernel"),    # C % 32 != 0, HW = 144: a ragged 128-pixel tile
    (1, 3, 8, 16, 96, False, "quantize_nchw_nhwc_vec_kernel"),      # c_pad > C over three 32-channel tiles
    (2, 64, 28, 28, 64, False, "quantize_nchw_nhwc_vec_kernel"),
    (3, 17, 7, 4, 48, False, "quantize_nchw_nhwc_vec_kernel"),
    (2, 64, 7, 7, 64, False, "quantize_nchw_nhwc_kernel"),          # 7 x 7 planes
    (300, 1000, 1, 1, 1008, False, "quantize_nchw_nhwc_kernel"),    # NewLinear
    (2, 5, 9, 11, 32, False, "quantize_nchw_nhwc_kernel"),          # odd planes
    (2, 24, 4, 8, 48, True, "quantize_nchw_nhwc_kernel"),           # aligned shape, unaligned view
]


@gpu
@pytest.mark.parametrize("row", NHWC_ROWS, ids=["n%d_c%d_%dx%d_p%d%s" % (r[:5] + ("_off" if r[5] else "",))
                                                for r in NHWC_ROWS])
def test_quantize_nchw_to_nhwc(row):
    N, C, H, W, c_pad, off, kernel = row
    lib = _lib()
    for i, ib in enumerate(IBS):
        x = crafted((N, C, H, W), ib, _seed(row, ib))
        if off:
            x = offset_view(x)
        out = Guarded((N, H, W, c_pad), torch.int8)

        def run():
            assert lib.pq_quantize_nchw_to_nhwc_s8(x.data_ptr(), out.ptr(), N, C, H, W, c_pad, ib, _stream()) == 0
        if i == 0:
            check_landing(run, kernel)
        run()
        torch.cuda.synchronize()
        out.check("ib=%d" % ib)
        want = torch.zeros((N, H, W, c_pad), dtype=torch.long, device="cuda")
        want[..., :C] = q_ref(x, ib).permute(0, 2, 3, 1)
        assert torch.equal(out.t.long(), want), ib


# (N, C, H, W, R, S, stride (h, w), pad (h, w), extra kp bytes beyond R*S*C rounded up to 16)
IM2COL_ROWS = [
    (2, 3, 23, 19, 7, 7, (2, 2), (3, 3), 0),        # the ResNet stem's geometry
    (1, 1, 9, 13, 1, 1, (1, 1), (0, 0), 0),
    (2, 8, 11, 10, 3, 3, (1, 1), (1, 1), 0),
    (2, 8, 11, 10, 3, 3, (1, 1), (1, 1), 32),
    (1, 5, 17, 15, 5, 5, (3, 2), (2, 0), 0),
    (3, 2, 12, 12, 5, 3, (4, 4), (3, 1), 16),
    (1, 4, 10, 10, 7, 5, (1, 3), (3, 2), 0),
    (1, 6, 8, 9, 3, 7, (2, 1), (0, 3), 48),
    (2, 7, 6, 5, 1, 3, (2, 4), (0, 1), 0),
    (7, 3, 224, 224, 3, 3, (1, 1), (1, 1), 0),      # M = 351232 > 1184 * 8 * 32: the grid-stride loop runs
]


@gpu
@pytest.mark.parametrize("row", IM2COL_ROWS, ids=["n%d_c%d_%dx%d_r%ds%d_st%d%d_p%d%d_kx%d" % (r[:6] + r[6] + r[7] + r[8:])
                                                  for r in IM2COL_ROWS])
def test_quantize_im2col(row):
    N, C, H, W, R, S, (sh, sw), (ph, pw), extra = row
    kp = (R * S * C + 15) // 16 * 16 + extra
    P, Q = (H + 2 * ph - R) // sh + 1, (W + 2 * pw - S) // sw + 1
    M = N * P * Q
    lib = _lib()
    big = M > 1184 * 8 * 32
    for i, ib in enumerate((4, 126, -126) if big else IBS):
        x = crafted((N, C, H, W), ib, _seed(row, ib))
        out = Guarded((M, kp), torch.int8)

        def run():
            assert lib.pq_quantize_im2col_s8(x.data_ptr(), out.ptr(), N, C, H, W, R, S, sh, sw, ph, pw, kp, ib,
                                             _stream()) == 0
        if i == 0:
            check_landing(run, "quantize_im2col_kernel")
        run()
        torch.cuda.synchronize()
        out.check("ib=%d" % ib)
        cols = F.unfold(q_ref(x, ib).double(), (R, S), padding=(ph, pw), stride=(sh, sw))     # [N][C*R*S][P*Q]
        cols = cols.view(N, C, R * S, P * Q).permute(0, 3, 2, 1).reshape(M, R * S * C)        # k = (r*S + s)*C + c
        want = torch.zeros((M, kp), dtype=torch.long, device="cuda")
        want[:, :R * S * C] = cols.long()
        assert torch.equal(out.t.long(), want), ib


def smallc_padded_size(H, W, R, S, sh, sw, ph, pw):
    """Hp, Wp as NewConv2d._quantize computes them for the small-channel convolution."""
    P, Q = (H + 2 * ph - R) // sh + 1, (W + 2 * pw - S) // sw + 1
    Hp = max((P - 1) * sh + R, H + ph)
    Hp = (Hp + sh - 1) // sh * sh
    Wp = max((Q - 1) * sw + 8, W + pw)
    return Hp, Wp + (Wp & 1)


# (N, C, H, W, conv (R, S, sh, sw, ph, pw), extra (Hp, Wp), x at a 4-byte offset, kernel)
PAD8_ROWS = [
    (2, 3, 20, 24, (7, 7, 2, 2, 3, 3), (0, 0), False, "quantize_pad_nhwc8_v4_kernel"),
    (1, 1, 5, 8, (3, 3, 1, 2, 1, 1), (0, 0), False, "quantize_pad_nhwc8_v4_kernel"),
    (3, 4, 9, 12, (3, 5, 1, 2, 1, 2), (20, 10), False, "quantize_pad_nhwc8_v4_kernel"),  # deep ring: grid-stride rows
    (2, 3, 15, 17, (7, 7, 2, 2, 3, 3), (0, 0), False, "quantize_pad_nhwc8_c4_kernel"),
    (1, 2, 7, 9, (3, 3, 1, 2, 1, 1), (0, 0), False, "quantize_pad_nhwc8_c4_kernel"),     # odd Hp (9)
    (2, 4, 6, 7, (3, 3, 1, 2, 1, 1), (3, 2), False, "quantize_pad_nhwc8_c4_kernel"),
    (2, 3, 10, 16, (5, 5, 2, 2, 2, 2), (1, 0), True, "quantize_pad_nhwc8_c4_kernel"),    # W % 4 == 0, unaligned view
    (1, 5, 9, 10, (3, 3, 1, 2, 1, 1), (0, 0), False, "quantize_pad_nhwc8_kernel"),
    (2, 6, 7, 13, (5, 5, 2, 2, 2, 2), (2, 4), False, "quantize_pad_nhwc8_kernel"),
    (1, 7, 12, 8, (3, 3, 1, 2, 0, 0), (0, 0), False, "quantize_pad_nhwc8_kernel"),
    (2, 8, 11, 300, (3, 3, 1, 2, 1, 1), (1, 2), False, "quantize_pad_nhwc8_kernel"),    # Wp / 2 > 128: 256 threads
]


@gpu
@pytest.mark.parametrize("row", PAD8_ROWS, ids=["n%d_c%d_%dx%d_r%d_e%d%d%s" % (r[:4] + (r[4][0],) + r[5] + ("_off" if r[6] else "",))
                                                for r in PAD8_ROWS])
def test_quantize_pad_nhwc8(row):
    N, C, H, W, (R, S, sh, sw, ph, pw), (eh, ew), off, kernel = row
    Hp, Wp = smallc_padded_size(H, W, R, S, sh, sw, ph, pw)
    Hp, Wp = Hp + eh, Wp + ew
    lib = _lib()
    for i, ib in enumerate(IBS):
        x = crafted((N, C, H, W), ib, _seed(row, ib))
        if off:
            x = offset_view(x)
        out = Guarded((N, Hp, Wp, 8), torch.int8)

        def run():
            assert lib.pq_quantize_nchw_to_padded_nhwc8_s8(x.data_ptr(), out.ptr(), N, C, H, W, ph, pw, Hp, Wp, ib,
                                                           _stream()) == 0
        if i == 0:
            check_landing(run, kernel)
        run()
        torch.cuda.synchronize()
        out.check("ib=%d" % ib)
        want = torch.zeros((N, Hp, Wp, 8), dtype=torch.long, device="cuda")
        want[:, ph:ph + H, pw:pw + W, :C] = q_ref(x, ib).permute(0, 2, 3, 1)
        assert torch.equal(out.t.long(), want), ib


def s2d_ref(q, pad_t, pad_l, Hp2, Wp2):
    """q[n][i][j][(dy*2 + dx)*4 + c] = q(x[n][c][2i + dy - pad_t][2j + dx - pad_l]), 0 outside / for c >= C."""
    N, C, H, W = q.shape
    canvas = torch.zeros((N, 4, max(2 * Hp2, pad_t + H), max(2 * Wp2, pad_l + W)), dtype=torch.long, device=q.device)
    canvas[:, :C, pad_t:pad_t + H, pad_l:pad_l + W] = q
    canvas = canvas[:, :, :2 * Hp2, :2 * Wp2].reshape(N, 4, Hp2, 2, Wp2, 2)
    return canvas.permute(0, 2, 4, 3, 5, 1).reshape(N, Hp2, Wp2, 16)


# (N, C, H, W, pad_t, pad_l, Hp2, Wp2, x at a 4-byte offset, kernel)
S2D_ROWS = [
    (2, 3, 14, 16, 2, 2, 11, 14, "", "quantize_s2d16_kernel<true>"),      # ResNet-stem-like, blocks beyond the image
    (1, 1, 6, 8, 0, 0, 3, 4, "", "quantize_s2d16_kernel<true>"),
    (2, 4, 9, 10, 4, 2, 9, 9, "", "quantize_s2d16_kernel<true>"),
    (1, 2, 7, 12, 0, 4, 6, 11, "", "quantize_s2d16_kernel<true>"),
    (2, 3, 13, 15, 2, 2, 10, 12, "", "quantize_s2d16_kernel<false>"),     # odd W
    (1, 4, 5, 9, 4, 0, 6, 7, "", "quantize_s2d16_kernel<false>"),
    (1, 1, 8, 7, 0, 2, 5, 6, "", "quantize_s2d16_kernel<false>"),
    (2, 3, 12, 16, 2, 2, 9, 11, "off", "quantize_s2d16_kernel<false>"),   # even W, x at a 4-byte offset
    (1, 2, 6, 6, 4, 4, 3, 3, "", "quantize_s2d16_kernel<true>"),          # the output ends inside the padding
]


@gpu
@pytest.mark.parametrize("row", S2D_ROWS, ids=["n%d_c%d_%dx%d_p%d%d_%dx%d%s" % (r[:8] + ("_" + r[8] if r[8] else "",))
                                               for r in S2D_ROWS])
def test_quantize_s2d16(row):
    N, C, H, W, pt, pl, Hp2, Wp2, off, kernel = row
    lib = _lib()
    for i, ib in enumerate(IBS):
        x = crafted((N, C, H, W), ib, _seed(row, ib))
        if off:
            x = offset_view(x)
        out = Guarded((N, Hp2, Wp2, 16), torch.int8)

        def run():
            assert lib.pq_quantize_nchw_to_s2d16_s8(x.data_ptr(), out.ptr(), N, C, H, W, pt, pl, Hp2, Wp2, ib,
                                                    _stream()) == 0
        if i == 0:
            check_landing(run, kernel)
        run()
        torch.cuda.synchronize()
        out.check("ib=%d" % ib)
        assert torch.equal(out.t.long(), s2d_ref(q_ref(x, ib), pt, pl, Hp2, Wp2)), ib


# ------------------------------------------------------------------------------------------ 2. pipeline kernels
def pool_operand(shape, seed):
    """int8 NHWC: uniform values, image 0's top half all -128, and all-negative windows in the last image."""
    N, H, W, C = shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(-128, 128, shape, generator=g, device="cuda", dtype=torch.int8)
    x[0, :max(1, H // 2)] = -128
    x[-1, :, :max(1, W // 2)] = torch.randint(-128, 0, x[-1, :, :max(1, W // 2)].shape, generator=g, device="cuda",
                                              dtype=torch.int8)
    return x


def maxpool_ref(x, k, s, p, relu):
    y = F.max_pool2d(x.permute(0, 3, 1, 2).float(), k, s, p)
    if relu:
        y = y.clamp(min=0)
    return y.permute(0, 2, 3, 1).long()


# (N, H, W, C, k, stride, pad): k = 3 takes the unrolled path, every other k the generic one
MAXPOOL_ROWS = [
    (2, 9, 11, 16, 3, 2, 1),
    (2, 13, 7, 48, 3, 1, 1),          # C = 48: (q, c16) wraps its channel group (dc)
    (2, 8, 60, 272, 3, 2, 1),         # Q * C / 16 = 510 > 256: a second trip
    (2, 5, 6, 4112, 3, 1, 1),         # C / 16 = 257 > 256 threads: dq == 0
    (2, 10, 10, 64, 3, 4, 0),         # stride > k
    (2, 7, 9, 16, 1, 1, 0),
    (2, 8, 8, 48, 2, 2, 1),
    (2, 11, 13, 272, 4, 3, 2),
    (2, 12, 9, 64, 5, 2, 2),
    (2, 6, 7, 4112, 2, 1, 1),
    (2, 9, 9, 48, 2, 3, 0),           # stride > k
    (2, 5, 70, 272, 5, 1, 1),         # Q * C / 16 = 1122
    (2, 17, 40, 16, 4, 1, 2),
    (1, 6, 5, 96, 5, 3, 0),
]


@gpu
@pytest.mark.parametrize("row", MAXPOOL_ROWS, ids=["n%d_%dx%d_c%d_k%d_s%d_p%d" % r for r in MAXPOOL_ROWS])
def test_maxpool(row):
    N, H, W, C, k, s, p = row
    lib = _lib()
    x = pool_operand((N, H, W, C), _seed(row))
    P, Q = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    for relu in (False, True):
        out = Guarded((N, P, Q, C), torch.int8)

        def run():
            assert lib.pq_maxpool_nhwc_s8(x.data_ptr(), out.ptr(), N, H, W, C, k, s, p, int(relu), _stream()) == 0
        if not relu:
            check_landing(run, "maxpool_nhwc_s8_kernel")
        run()
        torch.cuda.synchronize()
        out.check("relu=%s" % relu)
        assert torch.equal(out.t.long(), maxpool_ref(x, k, s, p, relu)), relu


@gpu
def test_maxpool_resnet_stem_at_size():
    """The ResNet stem's pool at batch 512: 512 x 112 x 112 x 64, k 3, stride 2, pad 1."""
    N, H, W, C = 512, 112, 112, 64
    x = pool_operand((N, H, W, C), 9)
    for relu in (False, True):
        out = Guarded((N, 56, 56, C), torch.int8)
        assert _lib().pq_maxpool_nhwc_s8(x.data_ptr(), out.ptr(), N, H, W, C, 3, 2, 1, int(relu), _stream()) == 0
        torch.cuda.synchronize()
        out.check("stem")
        assert torch.equal(out.t.long(), maxpool_ref(x, 3, 2, 1, relu)), relu


def avgpool_operand(N, HW, C, is16, seed):
    """image 0 all at the payload's maximum, image 1 all at its minimum, the rest uniform over the payload range."""
    lo, hi = (-32768, 32767) if is16 else (-128, 127)
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(lo, hi + 1, (N, HW, 1, C), generator=g, device="cuda", dtype=torch.int32)
    x[0], x[1] = hi, lo
    return x.to(torch.int16 if is16 else torch.int8)


def avgpool_ref(x, bit, relu):
    v = x.float() * 2.0 ** -bit                       # exact: a payload times a power of two in the fp32 range
    if relu:
        v = torch.relu(v)
    return F.avg_pool2d(v.permute(0, 3, 1, 2).contiguous(), v.shape[1:3]).view(v.shape[0], v.shape[3])


# (HW, C, int16 payload); HW 511 is the last int16 and 131071 the last int8 plane with |sum| < 2^24 payload units
AVGPOOL_ROWS = [(hw, c, is16) for is16, hws in ((False, (1, 49, 511, 131071)), (True, (1, 49, 511)))
                for hw in hws for c in (8, 2048, 2056, 4096) if not (hw == 131071 and c == 4096)]


@gpu
@pytest.mark.parametrize("row", AVGPOOL_ROWS, ids=["hw%d_c%d_%s" % (r[0], r[1], "s16" if r[2] else "s8") for r in AVGPOOL_ROWS])
def test_avgpool_global(row):
    HW, C, is16 = row
    N = 3
    lib = _lib()
    x = avgpool_operand(N, HW, C, is16, _seed(row))
    for i, (bit, relu) in enumerate((b, r) for b in (-100, -7, 0, 7, 100) for r in (False, True)):
        out = Guarded((N, C), torch.float32)

        def run():
            assert lib.pq_avgpool_global_nhwc_f32(x.data_ptr(), int(is16), bit, int(relu), N, HW, C, out.ptr(),
                                                  _stream()) == 0
        if i == 0:
            check_landing(run, "avgpool_global_kernel<%s>" % _tf(is16))
        run()
        torch.cuda.synchronize()
        out.check("bit=%d relu=%s" % (bit, relu))
        want = avgpool_ref(x, bit, relu)
        assert torch.equal(out.t.view(torch.int32), want.view(torch.int32)), (bit, relu)


@gpu
def test_avgpool_one_step_beyond_the_exact_plane_falls_back():
    """HW * max|payload| = 2^24: PQ_EUNSUPPORTED with the output untouched, the wrapper returns None, and a QTensor
    pooled in pipeline mode takes the de-quantising path with the same result."""
    from common.quantity import QTensor, _native
    for is16, HW, shape in ((False, 131072, (2, 512, 256)), (True, 512, (2, 16, 32))):
        N, H, W = shape
        C = 16
        x = avgpool_operand(N, HW, C, is16, HW).view(N, H, W, C)
        out = Guarded((N, C), torch.float32)
        assert _lib().pq_avgpool_global_nhwc_f32(x.data_ptr(), int(is16), 3, 0, N, HW, C, out.ptr(), _stream()) \
            == EUNSUPPORTED
        torch.cuda.synchronize()
        assert _untouched(out)
        assert _lib().pq_avgpool_global_nhwc_f32(x.data_ptr(), int(is16), 3, 0, N, HW - 1, C, out.ptr(), _stream()) == 0
        torch.cuda.synchronize()
        assert bool((out.buf[:out.lo] == SENTINEL).all()) and bool((out.buf[out.hi:] == SENTINEL).all())
        assert _native.avgpool_global_nhwc(x, 3) is None
        kw = dict(s16=x, s16_bit=3) if is16 else dict(q8=x, q8_bit=3)
        qt = QTensor((N, C, H, W), x.device, **kw)
        got = F.avg_pool2d(qt, (H, W))
        want = F.avg_pool2d((x.float() * 2.0 ** -3).permute(0, 3, 1, 2).contiguous(), (H, W))
        assert not isinstance(got, QTensor) and torch.equal(got, want)


# ---- add_requant
ADD_NS = (1, 15, 16, 17, 511, 512, 513, 100003, 16 * 606208 + 5)      # the last one runs the grid-stride loop


def add_operands(n, a16, abit, b16, bbit, q_bit, seed):
    """Operands of n elements: payload extremes, operand pairs whose sum sits at the clamp bounds and one either side,
    exact ties (2j + 1) * 2^(d - 1) of the requantisation shift d (j near 0 and at both saturation edges, both signs),
    then uniform values."""
    o = max(abit, bbit)
    sa, sb = o - abit, o - bbit
    lim = lambda is16: (-32768, 32767) if is16 else (-128, 127)
    (alo, ahi), (blo, bhi) = lim(a16), lim(b16)
    pairs = [(alo, blo), (ahi, bhi), (alo, bhi), (ahi, blo), (0, 0), (-1, 1), (alo, 0), (0, bhi)]
    targets = [-128 << o, 127 << o]
    targets = [t + d for t in targets for d in (-1, 0, 1)]
    d = o - q_bit
    if d >= 1:
        targets += [(2 * j + 1) << (d - 1) for j in (-130, -129, -128, -3, -2, -1, 0, 1, 2, 126, 127, 128)]
    rng = np.random.default_rng(seed)
    for t in targets:                    # the operand without a shift takes any integer: solve for it
        for _ in range(4):
            if sa == 0:
                b = int(rng.integers(blo, bhi + 1)) if _ else 0
                a = t - (b << sb)
            else:
                a = int(rng.integers(alo, ahi + 1)) if _ else 0
                b = t - (a << sa)
            if alo <= a <= ahi and blo <= b <= bhi:
                pairs.append((a, b))
    a = rng.integers(alo, ahi + 1, size=n)
    b = rng.integers(blo, bhi + 1, size=n)
    k = min(n, len(pairs))
    crafted_pairs = np.array(pairs, dtype=np.int64)
    a[:k], b[:k] = crafted_pairs[:k, 0], crafted_pairs[:k, 1]
    if n > 2 * len(pairs):               # and once more at the end (the scalar tail)
        a[-len(pairs):], b[-len(pairs):] = crafted_pairs[:, 0], crafted_pairs[:, 1]
    dt = lambda is16: torch.int16 if is16 else torch.int8
    return torch.from_numpy(a).to(dt(a16)), torch.from_numpy(b).to(dt(b16))


def run_add(a, abit, arelu, b, bbit, brelu, q_bit, out_relu, want16, want8, kernel=None):
    n = a.numel()
    o16 = Guarded((n,), torch.int16) if want16 else None
    o8 = Guarded((n,), torch.int8) if want8 else None

    def run():
        rc = _lib().pq_add_requant(a.data_ptr(), int(a.dtype == torch.int16), abit, int(arelu), b.data_ptr(),
                                   int(b.dtype == torch.int16), bbit, int(brelu), n, int(out_relu),
                                   o16.ptr() if o16 else None, o8.ptr() if o8 else None, q_bit, _stream())
        assert rc == 0, rc
    if kernel:
        check_landing(run, kernel)
    run()
    torch.cuda.synchronize()
    s16, q8 = add_ref(a.long().clamp(min=0) if arelu else a.long(), abit, b.long(), bbit, brelu, out_relu, q_bit)
    what = (a.dtype, abit, arelu, b.dtype, bbit, brelu, q_bit, out_relu, n)
    for g, want in ((o16, s16), (o8, q8)):
        if g is not None:
            g.check(str(what))
            assert torch.equal(g.t.long(), want), what


# one bit setting per (RELU_IN, QDOWN): (abit, arelu, bbit, brelu, q_bit, out_relu)
ADD_BITS = {(False, False): (4, False, 2, False, 6, False), (False, True): (7, False, 3, False, 0, True),
            (True, False): (3, True, 3, False, 3, False), (True, True): (0, False, 6, True, -9, True)}


@gpu
@pytest.mark.parametrize("a16,b16,relu_in,qdown", [(a, b, r, q) for a in (False, True) for b in (False, True)
                                                   for r in (False, True) for q in (False, True)],
                         ids=lambda v: str(int(v)))
def test_add_requant_instantiations_and_sizes(a16, b16, relu_in, qdown):
    abit, arelu, bbit, brelu, q_bit, out_relu = ADD_BITS[(relu_in, qdown)]
    kernel = add_kernel(a16, b16, relu_in, qdown)
    for n in ADD_NS:
        a, b = (t.cuda() for t in add_operands(n, a16, abit, b16, bbit, q_bit, _seed(kernel, n)))
        for i, (w16, w8) in enumerate(((True, True), (True, False), (False, True))):
            run_add(a, abit, arelu, b, bbit, brelu, q_bit, out_relu, w16, w8,
                    kernel if n == 100003 and i == 0 else None)


@gpu
@pytest.mark.parametrize("o_bit", range(8))
def test_add_requant_bit_grid(o_bit):
    """Every admissible (o_bit, span, q_shift) with either operand the finer one, at n = 517 (vector part + tail)."""
    i = 0
    for span in range(8):
        for q_shift in range(-15, 16):
            for a_finer in (False, True):
                abit, bbit = (o_bit, o_bit - span) if a_finer else (o_bit - span, o_bit)
                a16, b16, arelu, brelu, out_relu = (i & 1, i & 2, i % 5 == 0, i % 7 == 0, i % 3 == 0)
                i += 1
                a, b = (t.cuda() for t in add_operands(517, bool(a16), abit, bool(b16), bbit, o_bit + q_shift, i))
                run_add(a, abit, arelu, b, bbit, brelu, o_bit + q_shift, out_relu, True, True)


# ---- concat_requant
def concat_source(pixels, c, is16, bit, q_bit, seed, offset=0):
    """[pixels][c] payload: uniform, with the exact ties of the shift q_bit - bit and both payload extremes planted."""
    lo, hi = (-32768, 32767) if is16 else (-128, 127)
    rng = np.random.default_rng(seed)
    v = rng.integers(lo, hi + 1, size=pixels * c)
    d = bit - q_bit
    plant = [lo, hi, 0, -1]
    if d >= 1:
        plant += [t for j in range(-131, 131) for t in ((2 * j + 1) << (d - 1),) if lo <= t <= hi]
    k = min(len(plant), v.size)
    v[:k] = plant[:k]
    v[-k:] = plant[:k]
    t = torch.from_numpy(v.reshape(pixels, c)).to(torch.int16 if is16 else torch.int8).cuda()
    return offset_view(t, offset) if offset else t


# (pixels, sources ((channels, int16, bit, relu, element offset), ...), q_bit, c_out_pad, kernel)
CONCAT_ROWS = [
    (1000, ((16, False, 4, False, 0), (32, True, 9, True, 0), (48, False, -3, False, 0)), 4, 112, "vec"),
    (777, tuple((16, i % 2 == 1, 4 - sh, i % 3 == 0, 0) for i, sh in enumerate((-15, -8, -1, 0, 1, 7, 14, 15))), 4, 144,
     "vec"),
    (501, tuple((c, i % 2 == 0, 2 - sh, i % 2 == 1, 0) for i, (c, sh) in
                enumerate(zip((5, 3, 7, 1, 9, 2, 4, 6), (15, -15, 3, -3, 0, 8, -8, 1)))), 2, 48, "scalar"),
    (300, ((1, True, 7, False, 0),), 0, 16, "scalar"),
    (640, ((32, False, 5, False, 0), (16, False, 3, True, 1), (16, True, 9, False, 0)), 5, 64, "scalar"),  # unaligned
    (160000, ((16, True, 6, True, 0), (32, False, 2, False, 0)), 4, 64, "vec"),        # pixels * groups > grid cap
    (20000, ((24, False, 1, False, 0), (13, True, 10, True, 0)), -1, 48, "scalar"),    # pixels * c_out_pad > cap
    (96, ((16, False, 0, False, 0),), 0, 16, "vec"),                                  # a plain copy
]


@gpu
@pytest.mark.parametrize("row", CONCAT_ROWS, ids=["p%d_k%d_q%d_c%d_%s" % (r[0], len(r[1]), r[2], r[3], r[4])
                                                  for r in CONCAT_ROWS])
def test_concat_requant_vs_oracle(oracle, row):
    from common.quantity import _native
    pixels, spec, q_bit, c_pad, kind = row
    srcs = [concat_source(pixels, c, is16, bit, q_bit, _seed(row, i), off) for i, (c, is16, bit, relu, off) in
            enumerate(spec)]
    arr = (_native.ConcatSrc * len(spec))(*[_native.ConcatSrc(t.data_ptr(), int(s[1]), s[0], s[2], int(s[3]))
                                            for t, s in zip(srcs, spec)])
    out = Guarded((pixels, c_pad), torch.int8)

    def run():
        assert _lib().pq_concat_requant_s8(arr, len(spec), pixels, q_bit, c_pad, out.ptr(), _stream()) == 0
    check_landing(run, "concat_requant_%s_kernel" % kind)
    torch.cuda.synchronize()
    out.check("concat")
    parts = []
    for t, (c, is16, bit, relu, off) in zip(srcs, spec):
        real = t.cpu().numpy().astype(np.float32) / np.float32(2.0 ** bit)
        parts.append(np.maximum(real, np.float32(0)) if relu else real)
    want = oracle.concat_quantize(parts, q_bit)
    c_sum = sum(s[0] for s in spec)
    got = out.t.cpu().numpy()
    assert np.array_equal(got[:, :c_sum].astype(np.float32), want)
    assert not got[:, c_sum:].any()


# ---- relu_s8
@gpu
@pytest.mark.parametrize("n", (1, 15, 16, 17, 10 ** 6 + 3, 2 * 16 * CAP_THREADS + 9))
def test_relu_s8(n):
    x = torch.from_numpy(np.resize(np.arange(-128, 128, dtype=np.int8), n + 7)[7:].copy()).cuda()   # all 256 bytes
    out = Guarded((n,), torch.int8)

    def run():
        assert _lib().pq_relu_s8(x.data_ptr(), out.ptr(), n, _stream()) == 0
    check_landing(run, "relu_s8_kernel")
    torch.cuda.synchronize()
    out.check("relu")
    assert torch.equal(out.t, x.clamp(min=0))


# ------------------------------------------------------------------------------------------ 3. stand-alone fp32
def _f32(v):
    return np.asarray(v, dtype=np.float32)


def add_clamp_ref(a, b, lo, hi):
    """NewAdd (new_quantity_op.py:166-174): fp32 a + b, then torch.clamp (which keeps the sign of a zero)."""
    s = (_f32(a) + _f32(b)).astype(np.float32)
    return np.where(s < lo, np.float32(lo), np.where(s > hi, np.float32(hi), s)).astype(np.float32)


def rshift_ref(x, rs, lo, hi):
    """RightShift (new_quantity_op.py:11-44): v = x / 2^rs in fp32, trunc(v +- 0.5) as an int32, clamp -> fp32."""
    s = (_f32(x) * np.float32(2.0 ** -rs)).astype(np.float32)
    t = np.where(s > 0, s + np.float32(0.5), s - np.float32(0.5)).astype(np.float32)
    assert np.all(np.abs(t) < 2.0 ** 31)
    return np.clip(np.trunc(t).astype(np.int64), int(lo), int(hi)).astype(np.float32)


def clamp_scale_ref(x, lo, hi, scale):
    """Sp / DeQuantity: torch.clamp(x, lo, hi) * scale in fp32."""
    x = _f32(x)
    c = np.where(x < lo, np.float32(lo), np.where(x > hi, np.float32(hi), x)).astype(np.float32)
    with np.errstate(over="ignore"):
        return (c * np.float32(scale)).astype(np.float32)


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.int32)


def _f32_out(n, off):
    return Guarded((n,), torch.float32, skew=4 if off else 0)


def _dev(v, off=False):
    t = torch.from_numpy(_f32(v)).cuda()
    return offset_view(t) if off else t


@gpu
@pytest.mark.parametrize("n", (1, 2, 3, 4, 5, 7, 4099, (1 << 20) + 3, 2 * 8 * CAP_THREADS + 3))
def test_add_clamp(n):
    a = det_inputs.bell(n, 61, 90.0)
    b = det_inputs.bell(n, 62, 90.0)
    special = np.array([(-0.0, -0.0), (0.0, -0.0), (3.5, -3.5), (np.inf, 1.0), (-np.inf, 5.0), (127.0, 0.5),
                        (-128.0, -0.5), (100.0, 27.0), (-100.0, -28.0), (-0.25, 0.25), (1e-45, -0.0)], np.float32)
    k = min(n, len(special))
    a[-k:], b[-k:] = special[:k, 0], special[:k, 1]
    for lo, hi in ((-128.0, 127.0), (-32768.0, 32767.0), (-np.inf, np.inf)):
        for off in (None, "a", "b", "y"):             # the vector path, then each operand off 16-byte alignment
            out = _f32_out(n, off == "y")
            ta, tb = _dev(a, off == "a"), _dev(b, off == "b")

            def run():
                assert _lib().pq_add_clamp_f32(ta.data_ptr(), tb.data_ptr(), out.ptr(), n, lo, hi, _stream()) == 0
            check_landing(run, "add_clamp_kernel") if off in (None, "a") and lo == -128.0 else run()
            torch.cuda.synchronize()
            out.check("add_clamp")
            assert np.array_equal(_bits(out.t.cpu().numpy()), _bits(add_clamp_ref(a, b, lo, hi))), (lo, off)


@gpu
@pytest.mark.parametrize("rs", (-100, -24, 0, 1, 24, 100))
def test_rshift(rs):
    k = np.arange(-300, 300, dtype=np.float64)
    ties = (k + 0.5) * 2.0 ** rs                           # quotients exactly +-k.5
    near = np.concatenate([k * 2.0 ** rs, ties]).astype(np.float32)
    near = np.concatenate([near, np.nextafter(near, np.float32(np.inf)), np.nextafter(near, np.float32(-np.inf))])
    big = (np.array([3e6, -3e6, 2.0 ** 22, -2.0 ** 22, 128.0, -129.0]) * 2.0 ** rs).astype(np.float32)   # saturation
    noise = (det_inputs.bell(70001, 63, 200.0).astype(np.float64) * 2.0 ** rs).astype(np.float32)
    x = np.concatenate([near, big, np.array([0.0, -0.0, 2.0 ** -149, -2.0 ** -149], np.float32), noise])
    n = x.size
    for lo, hi in ((-128.0, 127.0), (-32768.0, 32767.0)):
        for off in (False, True):
            out = _f32_out(n, off)
            t = _dev(x, off)

            def run():
                assert _lib().pq_rshift_f32(t.data_ptr(), out.ptr(), n, rs, lo, hi, _stream()) == 0
            check_landing(run, "unary_kernel<0>") if not off and lo == -128.0 else run()
            torch.cuda.synchronize()
            out.check("rshift")
            assert np.array_equal(_bits(out.t.cpu().numpy()), _bits(rshift_ref(x, rs, lo, hi))), (lo, off)


@gpu
@pytest.mark.parametrize("n", (1, 5, 70001, 2 * CAP_THREADS + 5))
def test_clamp_scale(n):
    x = np.resize(np.concatenate([det_inputs.bell(4093, 64, 300.0),
                                  np.array([0.0, -0.0, np.inf, -np.inf, FLT_MAX, -FLT_MAX, 2.0 ** -149, 127.5, -128.5],
                                           np.float32)]), n)
    cases = [(-128.0, 127.0, 1.0), (-np.inf, np.inf, 2.0 ** -5), (-np.inf, np.inf, 2.0 ** 100),
             (-np.inf, np.inf, 2.0 ** -100), (-32768.0, 32767.0, 0.5), (0.0, 127.0, 1.0)]
    for i, (lo, hi, scale) in enumerate(cases):
        out = _f32_out(n, i % 2 == 1)
        t = _dev(x, i % 3 == 2)

        def run():
            assert _lib().pq_clamp_scale_f32(t.data_ptr(), out.ptr(), n, lo, hi, scale, _stream()) == 0
        check_landing(run, "unary_kernel<1>") if i == 0 else run()
        torch.cuda.synchronize()
        out.check("clamp_scale")
        assert np.array_equal(_bits(out.t.cpu().numpy()), _bits(clamp_scale_ref(x, lo, hi, scale))), (lo, hi, scale)


# ------------------------------------------------------------------------------------------ 4. kernel census
# Every kernel of pq_pipeline.cu and pq_elementwise.cu and the test that reaches it (with a landing check).
KERNELS = {
    "relu_s8_kernel": "test_relu_s8",
    "maxpool_nhwc_s8_kernel": "test_maxpool",
    "avgpool_global_kernel<false>": "test_avgpool_global",
    "avgpool_global_kernel<true>": "test_avgpool_global",
    **{add_kernel(a, b, r, q): "test_add_requant_instantiations_and_sizes"
       for a in (False, True) for b in (False, True) for r in (False, True) for q in (False, True)},
    "concat_requant_vec_kernel": "test_concat_requant_vs_oracle",
    "concat_requant_scalar_kernel": "test_concat_requant_vs_oracle",
    "bias_fold_kernel": "test_gpu_parity.py (and the folded-bias rows of test_gpu_epilogue_matrix.py)",
    "fakequant_kernel<false>": "test_gpu_parity.py",
    "fakequant_kernel<true>": "test_gpu_parity.py",
    "fakequant_scalar_kernel<false>": "test_gpu_parity.py",
    "fakequant_scalar_kernel<true>": "test_gpu_parity.py",
    "add_clamp_kernel": "test_add_clamp",
    "unary_kernel<0>": "test_rshift",
    "unary_kernel<1>": "test_clamp_scale",
    "quantize_nchw_nhwc_kernel": "test_quantize_nchw_to_nhwc",
    "quantize_nchw_nhwc_vec_kernel": "test_quantize_nchw_to_nhwc",
    "quantize_im2col_kernel": "test_quantize_im2col",
    "quantize_pad_nhwc8_v4_kernel": "test_quantize_pad_nhwc8",
    "quantize_pad_nhwc8_c4_kernel": "test_quantize_pad_nhwc8",
    "quantize_pad_nhwc8_kernel": "test_quantize_pad_nhwc8",
    "quantize_s2d16_kernel<false>": "test_quantize_s2d16",
    "quantize_s2d16_kernel<true>": "test_quantize_s2d16",
}
# The library's other kernels (every instantiation of each) and the test file that covers them.
OTHER_KERNELS = {
    "gemm_s8_kernel": "test_gpu_epilogue_matrix.py",
    "conv_rows_s8_kernel": "test_gpu_epilogue_matrix.py",
    "dw_conv_s8_kernel": "test_gpu_depthwise.py",
    "absmax_multi_kernel": "test_gpu_stats_matrix.py",
    "absmax_per_channel_kernel": "test_gpu_stats_matrix.py",
    "absmax_periodic_kernel": "test_gpu_stats_matrix.py",
    "hist_multi_kernel": "test_gpu_stats_matrix.py",
    "hist_generic_kernel": "test_gpu_stats_matrix.py",
    "epilogue_kernel": "test_gpu_stats_matrix.py",
    "kl_prepare_kernel": "test_gpu_stats_matrix.py",
    "kl_candidate_kernel": "test_gpu_stats_matrix.py",
    "kl_argmin_kernel": "test_gpu_stats_matrix.py",
}
ROW_KERNELS = ({r[-1] for r in NHWC_ROWS} | {"quantize_im2col_kernel"} | {r[-1] for r in PAD8_ROWS} |
               {r[-1] for r in S2D_ROWS} | {"concat_requant_%s_kernel" % r[-1] for r in CONCAT_ROWS})


def library_kernels():
    from common.quantity import _native
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not installed")
    sym = subprocess.run(["cuobjdump", "-symbols", _native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = subprocess.run(["cu++filt"], input=sym, check=True, capture_output=True, text=True).stdout
    return {kernel_id(line) for line in names.splitlines() if "STO_ENTRY" in line}


def test_kernel_table_equals_library_symbols():
    """KERNELS is exactly the library's pipeline / elementwise kernels and every other kernel belongs to a family in
    OTHER_KERNELS: a kernel added without a row here fails."""
    found = library_kernels()
    assert len(KERNELS) == 38
    assert {k for k in found if k.split("<")[0] not in OTHER_KERNELS} == set(KERNELS)
    assert {k.split("<")[0] for k in found} >= set(OTHER_KERNELS)
    for test in set(KERNELS.values()):
        assert test.endswith(")") or test.endswith(".py") or callable(globals().get(test)), test
    assert ROW_KERNELS <= set(KERNELS)


def test_kernel_id_spellings():
    assert kernel_id("void pq::add_requant_kernel<(bool)1, (bool)0, (bool)0, (bool)1>(pq::AddParams, unsigned long)") \
        == "add_requant_kernel<true,false,false,true>"
    assert kernel_id("void pq::add_requant_kernel<true, false, false, true>(pq::AddParams, unsigned long)") \
        == "add_requant_kernel<true,false,false,true>"
    assert kernel_id("void pq::unary_kernel<(int)1>(const float *, float *, unsigned long, float, float, float)") \
        == "unary_kernel<1>"
    assert kernel_id("pq::maxpool_nhwc_s8_kernel(const signed char *, signed char *, int, int)") \
        == "maxpool_nhwc_s8_kernel"
    assert kernel_id("void pq::gemm_s8_kernel<128, 64, 8, true, 8>(CUtensorMap)") == "gemm_s8_kernel<128,64,8,true,8>"
    assert kernel_id("void at::native::vectorized_elementwise_kernel<4>(int)") is None


# ------------------------------------------------------------------------------------------ argument limits
def _untouched(*gs):
    return all(bool((g.buf == SENTINEL).all()) for g in gs)


def _written(g):
    g.check("accepted")
    return not bool((g.t.view(torch.uint8) == SENTINEL).all())


@gpu
def test_one_step_beyond_each_limit():
    """One step beyond each argument limit returns the documented code and leaves the sentinels untouched; one step
    inside is accepted and writes."""
    from common.quantity import _native
    lib = _lib()
    s = _stream()
    g = torch.Generator(device="cuda").manual_seed(17)

    def expect(call, want, *outs):
        rc = call()
        torch.cuda.synchronize()
        assert rc == want, (rc, want)
        for o in outs:
            assert (_written(o) if want == 0 else _untouched(o))

    # max-pool: C % 16, N
    x = torch.randint(-128, 128, (4, 5, 5, 48), generator=g, device="cuda", dtype=torch.int8)
    for C, want in ((24, EUNSUPPORTED), (40, EUNSUPPORTED), (32, 0), (48, 0)):
        o = Guarded((4, 3, 3, C), torch.int8)
        expect(lambda: lib.pq_maxpool_nhwc_s8(x.data_ptr(), o.ptr(), 4, 5, 5, C, 3, 2, 1, 0, s), want, o)
    xn = torch.randint(-128, 128, (65536, 1, 1, 16), generator=g, device="cuda", dtype=torch.int8)
    for N, want in ((65536, EUNSUPPORTED), (65535, 0)):
        o = Guarded((N, 1, 1, 16), torch.int8)
        expect(lambda: lib.pq_maxpool_nhwc_s8(xn.data_ptr(), o.ptr(), N, 1, 1, 16, 1, 1, 0, 0, s), want, o)
    # avgpool: C % 8, bit
    xa = torch.randint(-128, 128, (2, 9, 24), generator=g, device="cuda", dtype=torch.int8)
    for C, bit, want in ((12, 0, EUNSUPPORTED), (20, 0, EUNSUPPORTED), (16, 0, 0), (8, 101, EUNSUPPORTED),
                         (8, -101, EUNSUPPORTED), (8, 100, 0), (8, -100, 0)):
        o = Guarded((2, C), torch.float32)
        expect(lambda: lib.pq_avgpool_global_nhwc_f32(xa.data_ptr(), 0, bit, 0, 2, 9, C, o.ptr(), s), want, o)
    # add: span, o_bit, q_shift
    a = torch.randint(-128, 128, (100,), generator=g, device="cuda", dtype=torch.int8)
    for abit, bbit, q, want in ((7, -1, 7, EUNSUPPORTED), (7, 0, 7, 0), (-1, -1, -1, EUNSUPPORTED), (0, 0, 0, 0),
                                (8, 8, 8, EUNSUPPORTED), (7, 7, 7, 0), (4, 4, 20, EUNSUPPORTED), (4, 4, 19, 0),
                                (4, 4, -12, EUNSUPPORTED), (4, 4, -11, 0), (3, 1, 19, EUNSUPPORTED), (3, 1, -13, EUNSUPPORTED)):
        o16, o8 = Guarded((100,), torch.int16), Guarded((100,), torch.int8)
        expect(lambda: lib.pq_add_requant(a.data_ptr(), 0, abit, 0, a.data_ptr(), 0, bbit, 0, 100, 0, o16.ptr(),
                                          o8.ptr(), q, s), want, o16, o8)
    # concat: k, shift, odd int16 pointer
    c8 = torch.randint(-128, 128, (64, 16), generator=g, device="cuda", dtype=torch.int8)
    c16 = torch.randint(-32768, 32767, (64 * 16 + 1,), generator=g, device="cuda", dtype=torch.int32).to(torch.int16)

    def concat(srcs, q, c_pad, o):
        arr = (_native.ConcatSrc * len(srcs))(*srcs)
        return lambda: lib.pq_concat_requant_s8(arr, len(srcs), 64, q, c_pad, o.ptr(), s)
    for k, want in ((9, ETOOMANY), (8, 0)):
        o = Guarded((64, 16 * k), torch.int8)
        expect(concat([_native.ConcatSrc(c8.data_ptr(), 0, 16, 4, 0)] * k, 4, 16 * k, o), want, o)
    for bit, want in ((20, EUNSUPPORTED), (-12, EUNSUPPORTED), (19, 0), (-11, 0)):
        o = Guarded((64, 16), torch.int8)
        expect(concat([_native.ConcatSrc(c8.data_ptr(), 0, 16, bit, 0)], 4, 16, o), want, o)
    for ptr, want in ((c16.data_ptr() + 1, EALIGN), (c16.data_ptr() + 2, 0)):
        o = Guarded((64, 16), torch.int8)
        expect(concat([_native.ConcatSrc(ptr, 1, 16, 9, 0)], 4, 16, o), want, o)
    # quantisers: c_pad % 16, ib, C, s2d pad parity, Wp parity
    xf = crafted((2, 8, 6, 8), 4, 5)
    for c_pad, ib, want in ((24, 4, EUNSUPPORTED), (32, 4, 0), (16, 127, EUNSUPPORTED), (16, -127, EUNSUPPORTED),
                            (16, 126, 0), (16, -126, 0)):
        o = Guarded((2, 6, 8, c_pad), torch.int8)
        expect(lambda: lib.pq_quantize_nchw_to_nhwc_s8(xf.data_ptr(), o.ptr(), 2, 8, 6, 8, c_pad, ib, s), want, o)
    for ib, want in ((127, EUNSUPPORTED), (-127, EUNSUPPORTED), (126, 0), (-126, 0)):
        o = Guarded((2 * 6 * 8, 80), torch.int8)
        expect(lambda: lib.pq_quantize_im2col_s8(xf.data_ptr(), o.ptr(), 2, 8, 6, 8, 3, 3, 1, 1, 1, 1, 80, ib, s),
               want, o)
    for C, ib, Wp, want in ((9, 4, 10, EUNSUPPORTED), (8, 4, 10, 0), (8, 127, 10, EUNSUPPORTED),
                            (8, -127, 10, EUNSUPPORTED), (8, 126, 10, 0), (8, 4, 11, EALIGN)):
        o = Guarded((2, 8, Wp, 8), torch.int8)
        xc = crafted((2, C, 6, 8), 4, 6)
        expect(lambda: lib.pq_quantize_nchw_to_padded_nhwc8_s8(xc.data_ptr(), o.ptr(), 2, C, 6, 8, 1, 1, 8, Wp, ib, s),
               want, o)
    for C, pt, pl, ib, want in ((5, 2, 2, 4, EUNSUPPORTED), (4, 2, 2, 4, 0), (4, 1, 2, 4, EUNSUPPORTED),
                                (4, 2, 3, 4, EUNSUPPORTED), (4, 2, 2, 127, EUNSUPPORTED), (4, 2, 2, -127, EUNSUPPORTED),
                                (4, 2, 2, -126, 0)):
        o = Guarded((2, 5, 6, 16), torch.int8)
        xc = crafted((2, C, 6, 8), 4, 7)
        expect(lambda: lib.pq_quantize_nchw_to_s2d16_s8(xc.data_ptr(), o.ptr(), 2, C, 6, 8, pt, pl, 5, 6, ib, s),
               want, o)


# ------------------------------------------------------------------------------------------ argument-boundary fixes
@gpu
def test_maxpool_padding_over_half_the_window_is_refused():
    """torch refuses pad > k / 2; so does the kernel (PQ_EUNSUPPORTED, nothing written), and a QTensor in pipeline
    mode raises torch's own error, as the fp32-boundary model does."""
    from common.quantity import QTensor
    x = pool_operand((2, 9, 9, 16), 21)
    for k, p in ((3, 2), (2, 2), (1, 1), (5, 3)):
        P = (9 + 2 * p - k) // 2 + 1
        o = Guarded((2, P, P, 16), torch.int8)
        assert _lib().pq_maxpool_nhwc_s8(x.data_ptr(), o.ptr(), 2, 9, 9, 16, k, 2, p, 0, _stream()) == EUNSUPPORTED
        torch.cuda.synchronize()
        assert _untouched(o), (k, p)
    qt = QTensor((2, 16, 9, 9), x.device, q8=x, q8_bit=3)
    with pytest.raises(RuntimeError) as got:
        F.max_pool2d(qt, 3, 2, 2)
    with pytest.raises(RuntimeError) as want:
        F.max_pool2d(qt.dequantize(), 3, 2, 2)
    assert str(got.value) == str(want.value)


@gpu
def test_window_larger_than_the_padded_input_is_refused():
    """H + 2 pad < k (or W): PQ_EINVAL from max-pool and the im2col quantiser, although C's truncating division gives a
    1 x 1 output.  The output here is empty (passed as the address of its guard: an empty tensor's data_ptr() is NULL),
    so whatever a launch wrote would land in the guard."""
    lib = _lib()
    x = torch.randint(-128, 128, (1, 2, 2, 16), device="cuda", dtype=torch.int8)
    for H, W, k, st, p in ((1, 1, 2, 2, 0), (2, 1, 3, 2, 0), (1, 2, 4, 3, 1), (2, 2, 3, 2, 0)):
        o = Guarded((0,), torch.int8)
        assert lib.pq_maxpool_nhwc_s8(x.data_ptr(), o.buf.data_ptr() + o.lo, 1, H, W, 16, k, st, p, 0, _stream()) \
            == EINVAL, (H, W, k)
        torch.cuda.synchronize()
        assert _untouched(o), (H, W, k)
    xf = crafted((1, 1, 2, 2), 4, 3)
    for H, W, R, S, st, p in ((1, 1, 2, 2, 2, 0), (2, 2, 3, 3, 2, 0), (2, 2, 1, 3, 2, 0), (2, 1, 3, 1, 2, 0)):
        o = Guarded((0,), torch.int8)
        assert lib.pq_quantize_im2col_s8(xf.data_ptr(), o.buf.data_ptr() + o.lo, 1, 1, H, W, R, S, st, st, p, p, 16, 4,
                                         _stream()) \
            == EINVAL, (H, W, R, S)
        torch.cuda.synchronize()
        assert _untouched(o), (H, W, R, S)


@gpu
def test_maxpool_image_size_limit():
    """One image of 2^31 bytes or more is PQ_EUNSUPPORTED, checked before the pointers (no buffer needed, nothing
    launched); one step inside passes that check and stops at the NULL pointers."""
    lib = _lib()
    for (H, W, C), want in (((1 << 15, 1 << 12, 16), EUNSUPPORTED), ((1, 1 << 27, 16), EUNSUPPORTED),
                            ((46341, 2897, 16), EUNSUPPORTED), ((1 << 15, (1 << 12) - 1, 16), EINVAL)):
        assert lib.pq_maxpool_nhwc_s8(None, None, 1, H, W, C, 3, 2, 1, 0, _stream()) == want, (H, W, C)


# ------------------------------------------------------------------------------------------ CPU checks
def test_crafted_values_are_exact_ties_and_neighbours():
    for ib in IBS:
        v = crafted_values(ib)
        assert len(v) % 2 == 1
        t = v.astype(np.float64) * 2.0 ** ib
        finite = np.isfinite(t)
        assert np.sum(t[finite] % 1 == 0.5) >= (8 if ib < -120 else 262)
        if abs(ib) < 100:
            assert {127.5, -128.5, -129.5} <= set(t[finite].tolist())


def test_quantiser_reference_equals_oracle(oracle):
    """q_ref (float64) equals the oracle's fp32 Quantity on the crafted values of every ib (inf included)."""
    for ib in IBS:
        v = crafted_values(ib)
        v = np.concatenate([v, (det_inputs.bell(5001, ib & 0xff, 40.0).astype(np.float64) * 2.0 ** -ib).clip(
            -FLT_MAX, FLT_MAX).astype(np.float32)])
        with np.errstate(over="ignore"):
            want = oracle.quantize_input(v, ib)
        assert np.array_equal(q_ref(torch.from_numpy(v), ib).numpy(), want.astype(np.int64)), ib


def test_add_reference_equals_oracle(oracle):
    """add_ref on integer payloads equals the oracle's NewAdd on the de-quantised values, then Quantity(q_bit)."""
    for i, (abit, bbit, q_bit, a16, b16, arelu, brelu, orelu) in enumerate(
            ((4, 2, 6, False, True, False, False, False), (7, 0, -8, True, True, True, False, True),
             (0, -7, 15, True, False, False, True, False), (3, 3, 3, False, False, True, True, True),
             (7, 7, -8, False, False, False, False, False))):
        a, b = add_operands(3001, a16, abit, b16, bbit, q_bit, i)
        a, b = a.long(), b.long()
        av, bv = (a.clamp(min=0) if arelu else a), (b.clamp(min=0) if brelu else b)
        s16, q8 = add_ref(av, abit, b, bbit, brelu, orelu, q_bit)
        s = oracle.add_clamp(av.numpy().astype(np.float32) / np.float32(2.0 ** abit),
                             bv.numpy().astype(np.float32) / np.float32(2.0 ** bbit))
        if orelu:
            s = np.maximum(s, np.float32(0))
        o = max(abit, bbit)
        assert np.array_equal(s16.numpy(), (s.astype(np.float64) * 2.0 ** o).astype(np.int64))
        assert np.array_equal(q8.numpy(), oracle.quantize_input(s, q_bit).astype(np.int64))


def test_fp32_restatements_equal_intsim_golden():
    """rshift_ref / add_clamp_ref bit for bit against the reference's RightShift and NewAdd outputs (intsim.npz)."""
    g = load_golden("intsim.npz")
    accs = np.arange(-1100, 1100, dtype=np.float32)
    for rs in (-2, 0, 1, 3, 7):
        assert np.array_equal(_bits(rshift_ref(accs, rs, -128.0, 127.0)), _bits(g["rshift/rs%d" % rs])), rs
    a, c = det_inputs.bell(4096, 41, 60.0), det_inputs.bell(4096, 42, 60.0)
    assert np.array_equal(_bits(add_clamp_ref(a, c, -128.0, 127.0)), _bits(g["add/y"]))


def test_s2d_reference_on_a_small_image():
    """s2d_ref against the header formula evaluated element by element."""
    q = torch.arange(2 * 3 * 5 * 7).view(2, 3, 5, 7) - 100
    pt, pl, Hp2, Wp2 = 2, 4, 5, 6
    got = s2d_ref(q, pt, pl, Hp2, Wp2)
    for n in range(2):
        for i in range(Hp2):
            for j in range(Wp2):
                for dy in range(2):
                    for dx in range(2):
                        for c in range(4):
                            h, w = 2 * i + dy - pt, 2 * j + dx - pl
                            v = int(q[n, c, h, w]) if c < 3 and 0 <= h < 5 and 0 <= w < 7 else 0
                            assert int(got[n, i, j, (dy * 2 + dx) * 4 + c]) == v

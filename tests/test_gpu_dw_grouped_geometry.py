"""The depthwise (pq_conv2d_dw_s8, dw_conv_s8_kernel<G, KS>) and grouped (pq_conv2d_s8 with desc.groups > 1, modes 0 and
1 of gemm_s8_kernel) convolutions over their whole geometry range, on every kernel they reach, against

    acc = float64 F.conv2d of the int8 operands (tuple stride, padding, dilation, groups), rounded to int64   |acc| < 2^53
    y   = clamp(clamp(RightShift(acc, rs)) + b) [ReLU], fp32 = y / 2^ob                   new_quantity_op.py:11-44,124-133

which a CPU test pins to oracle.int_conv_layer(..., groups=...) on rectangular, asymmetric and dilated layers.  The
epilogue's own bit range is test_gpu_depthwise.py's and test_gpu_grouped.py's; here each row runs the plain and the
folded bias, the int8-only, the fp32-only and both outputs, ReLU on and off.

Each row names the instantiation it must reach (checked against a mirror of the host's choice on the CPU and with
torch.profiler on the GPU).  Every output sits in the middle of a sentinel-filled buffer whose neighbouring bytes must
survive, the input, the weights and the bias must be unchanged after the call, and a refused call writes nothing.  The
depthwise limits the header lists ('dw limit:') each have a row one step inside and one beyond; the index limits run at
their real size.
"""
import ctypes
import itertools
import os
import re
import shutil
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from test_gpu_conv_geometry import (EALIGN, EINVAL, EUNSUPPORTED, M_LIMIT, SENTINEL, SMS, Guarded, _chunks, _lib,
                                    _stream, dequant_ref, epilogue_ref, kernel_name, launched, right_shift)
from test_gpu_grouped import GROUPED_CONFIGS

gpu = pytest.mark.gpu
DW_THREADS, DW_PIX_ITERS = 256, 4          # pq_depthwise.cu: kDwThreads, kDwPixIters
DW_GRID_Y = 65535
OBS = (-3, 0, 2, 5, 9)


def out_size(g):
    (sh, sw), (ph, pw), (dh, dw) = g["st"], g["pad"], g["dil"]
    return ((g["H"] + 2 * ph - (g["R"] - 1) * dh - 1) // sh + 1, (g["W"] + 2 * pw - (g["S"] - 1) * dw - 1) // sw + 1)


def _flags(bias, k, relu):
    from common.quantity import _native
    return (_native.FLAG_RELU if relu else 0) | (_native.FLAG_BIAS_FOLDED if bias.numel() == 3 * k else 0)


# ------------------------------------------------------------------------------------------ the host's choices
def dw_inst(C, R, S):
    """(G, KS) of the dw_conv_s8_kernel pq_conv2d_dw_s8 launches: 16-channel groups per CTA, unrolled square filter."""
    G = 4 if C % 64 == 0 else (2 if C % 32 == 0 else 1)
    return G, (R if R == S and R in (3, 5) else 0)


def grouped_choice(g):
    """(instantiation (BN, BK, STAGES, ADDK, BSLOTS), tps, resident weights) pq_conv2d_s8 selects for a grouped layer
    (conv_impl, gemm_impl, launch_bn, launch_cfg)."""
    from common.quantity import _native
    C, K, G, B = g["C"], g["K"], g["G"], g["B"]
    wb = _native.group_window(C, K, G, B)
    plain = (g["R"], g["S"]) == (1, 1) and g["st"] == (1, 1) and g["pad"] == (0, 0)
    if plain:                                      # mode 0: the box may reach past the window, weights zero-filled
        bk = 128 if wb >= 128 else (64 if wb >= 64 else 32)
        num_kb, tps = -(-wb // bk), 1
    else:
        bk = 128 if wb % 128 == 0 else (64 if wb % 64 == 0 else 32)
        num_kb = g["R"] * g["S"] * wb // bk
        tps = 3 if bk <= 64 and num_kb % 3 == 0 else 1
    if not plain and bk == 64 and B == 64 and K <= 64 and num_kb <= 9 and tps == 3:
        inst = (64, 64, 18, 0, 9)                  # short-K "deep A"
    else:
        st = {256: {128: 4, 64: 8, 32: 9}, 128: {128: 6, 64: 9, 32: 9}, 64: {128: 8, 64: 9, 32: 9},
              32: {128: 8, 64: 9, 32: 9}}[B][bk]
        inst = (B, bk, st, 0, st)
    return inst, tps, int(K <= B and num_kb <= inst[4])


def grouped_name(g):
    inst, tps, res = grouped_choice(g)
    mode = "gemm" if (g["R"], g["S"]) == (1, 1) and g["st"] == (1, 1) and g["pad"] == (0, 0) else "im2col"
    return "%s/%d.%d.%d.%d/tps%d/%s" % (mode, inst[0], inst[1], inst[2], inst[4], tps, "res" if res else "str")


def kname(name):
    """('dw', G, KS) or a gemm_s8_kernel instantiation tuple from a demangled kernel name, else None."""
    m = re.search(r"dw_conv_s8_kernel<([^>]*)>", name)
    if m:
        return ("dw",) + tuple(int(re.sub(r"\(int\)", "", a).strip()) for a in m.group(1).split(","))
    k = kernel_name(name)
    return k if isinstance(k, tuple) else None


# ------------------------------------------------------------------------------------------ landing checks
_FRESH_ENV = "PQ_DW_GROUPED_GEOMETRY_FRESH"
_LANDING = {}


def _landing_state():
    """Whether torch.profiler records kernels in this process.  After some sequences of earlier tests in the same
    pytest process it records no CUDA activity at all; the landing checks then cannot be made here, so this file is
    run once more on its own in a fresh process, where every landing check runs, and that run must pass."""
    if not _LANDING:
        recorded = bool(launched(lambda: torch.ones(16, device="cuda").add_(1))[1])
        _LANDING["recorded"] = recorded
        if not recorded:
            assert not os.environ.get(_FRESH_ENV), "torch.profiler records no CUDA kernels in a fresh process"
            r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-p", "no:cacheprovider",
                                "-m", "gpu"], cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                               env=dict(os.environ, **{_FRESH_ENV: "1"}), capture_output=True, text=True, timeout=3600)
            _LANDING["fresh_run"] = (r.returncode, r.stdout[-3000:])
    return _LANDING


def check_landing(fn, kernel):
    """fn() launches exactly one convolution kernel, `kernel` (('dw', G, KS) or a gemm_s8_kernel tuple)."""
    state = _landing_state()
    if not state["recorded"]:
        res = fn()
        rc, out = state["fresh_run"]
        assert rc == 0, "the fresh-process run of this file, which makes the landing checks, failed:\n" + out
        return res
    res, names = launched(fn)
    found = [k for k in map(kname, names) if k]
    assert found == [kernel], (kernel, names)
    return res


@pytest.fixture(scope="module")
def b200():
    assert torch.cuda.get_device_properties(0).multi_processor_count == SMS, "the tile walks below assume 148 SMs"


# ------------------------------------------------------------------------------------------ depthwise rows
def D(N, H, W, C, K, R, S, st=(1, 1), pad=(0, 0), dil=(1, 1)):
    return dict(N=N, H=H, W=W, C=C, K=K, R=R, S=S, st=st, pad=pad, dil=dil)


DW_CHANNELS = {1: (16, 48, 80), 2: (96, 160, 32), 4: (192, 960, 64)}
DW_FILTERS = {3: ((3, 3),), 5: ((5, 5),), 0: ((1, 7), (7, 1), (2, 6), (4, 3), (1, 1), (7, 7), (2, 2), (4, 4))}
DW_IMAGES = ((9, 13), (1, 11), (12, 1), (7, 8), (3, 17), (15, 10), (2, 2), (11, 5))
STEPS = ((1, 1), (1, 2), (2, 1), (2, 2))


def _dw_sweep():
    """Every (G, KS) at every stride (1|2) x (1|2) and dilation (1|2) x (1|2); pads 0, 1 and (R-1)*dil chosen per
    dimension (pad_h != pad_w on most rows); K = C, 1, C - 1, C - 15 and 16 of C = 64; images from 1 x 1 up."""
    rows = []
    for G, KS in itertools.product((1, 2, 4), (3, 5, 0)):
        for j, (st, dil) in enumerate(itertools.product(STEPS, STEPS)):
            C = DW_CHANNELS[G][j % 3]
            R, S = DW_FILTERS[KS][j % len(DW_FILTERS[KS])]
            mh, mw = (R - 1) * dil[0], (S - 1) * dil[1]
            ph, pw = min((0, 1, mh)[j % 3], mh), min((mw, 0, 1)[j % 3], mw)
            K = (C, 1, C - 1, C - 15, 16 if C == 64 else C)[j % 5]
            H, W = DW_IMAGES[(j + 3 * G + KS) % len(DW_IMAGES)]
            H, W = max(H, (R - 1) * dil[0] + 1 - 2 * ph), max(W, (S - 1) * dil[1] + 1 - 2 * pw)
            rows.append(((G, KS), D(1 + j % 3, H, W, C, K, R, S, st, (ph, pw), dil)))
    return rows


DW_ROWS = _dw_sweep() + [
    # images smaller than the dilated filter (legal only through padding)
    ((1, 0), D(2, 3, 3, 16, 16, 7, 7, pad=(12, 12), dil=(2, 2))),
    ((4, 3), D(1, 2, 2, 64, 61, 3, 3, pad=(2, 2), dil=(2, 2))),
    ((2, 5), D(3, 4, 1, 96, 96, 5, 5, st=(2, 1), pad=(8, 4), dil=(2, 1))),
    # P = 1, Q = 1
    ((1, 0), D(2, 1, 7, 48, 48, 1, 7, st=(2, 2), pad=(0, 3))),
    ((2, 0), D(3, 9, 1, 32, 31, 7, 1, st=(1, 2), pad=(3, 0))),
    ((4, 3), D(1, 3, 3, 192, 177, 3, 3, st=(2, 2))),
    # many CTAs along x, M % (1024 / G) != 0, P * Q odd: a warp's 32 / G pixels cross image boundaries
    ((1, 3), D(3, 37, 41, 16, 15, 3, 3, pad=(1, 0))),
    ((2, 5), D(5, 33, 29, 160, 145, 5, 5, st=(2, 1), pad=(2, 3), dil=(1, 2))),
    ((4, 0), D(7, 21, 19, 960, 959, 2, 6, st=(1, 2), pad=(1, 2))),
    ((4, 0), D(9, 11, 13, 64, 16, 4, 4, st=(2, 1), pad=(3, 0), dil=(1, 2))),           # K = 16 of C = 64
    ((1, 0), D(4, 25, 23, 80, 1, 7, 7, pad=(3, 6), dil=(1, 2))),                       # K = 1
]
DW_SATURATED = D(2, 7, 7, 16, 16, 7, 7)           # all -128 operands: |acc| = 49 * 2^14 everywhere


def dw_row_id(r):
    g = r[1]
    return "G%d.KS%d-n%d-%dx%d-c%d-k%d-%dx%d-s%d.%d-p%d.%d-d%d.%d" % (
        *r[0], g["N"], g["H"], g["W"], g["C"], g["K"], g["R"], g["S"], *g["st"], *g["pad"], *g["dil"])


def dw_exact(x_nhwc, w_rsc, K, st, pad, dil):
    """int64 [N*P*Q][K] accumulators of the depthwise convolution of channels < K."""
    acc = F.conv2d(x_nhwc[..., :K].permute(0, 3, 1, 2).double(), w_rsc[..., :K].permute(2, 0, 1).unsqueeze(1).double(),
                   None, st, pad, dil, K)
    assert acc.numel() == 0 or float(acc.abs().max()) < 2.0 ** 53
    return torch.round(acc).long().permute(0, 2, 3, 1).reshape(-1, K)


def _desc(g, rs, ob):
    from common.quantity import _native
    return _native._conv_desc(g["N"], g["H"], g["W"], g["C"], g["K"], (g["R"], g["S"]), g["st"], g["pad"], rs, ob,
                              g["dil"], g.get("G", 1), g.get("B", 0))


class Case:
    """Operands, exact accumulators and launches of one depthwise ('dw') or grouped ('grouped') geometry."""

    def __init__(self, g, kind, seed, fill=None):
        self.g, self.kind = g, kind
        self.gen = torch.Generator(device="cuda").manual_seed(seed)
        N, H, W, C, K, R, S = g["N"], g["H"], g["W"], g["C"], g["K"], g["R"], g["S"]
        self.P, self.Q = out_size(g)
        self.M, self.K = N * self.P * self.Q, K
        self.x = self._int8((N, H, W, C)) if fill is None else torch.full((N, H, W, C), fill, dtype=torch.int8,
                                                                           device="cuda")
        if kind == "dw":
            w = self._int8((R, S, C)) if fill is None else torch.full((R, S, C), fill, dtype=torch.int8, device="cuda")
            w[..., K:] = 0                                 # zero beyond K by contract
            self.w = w
            self.acc = dw_exact(self.x, w, K, g["st"], g["pad"], g["dil"])
        else:
            from common.quantity.new_quantity_op import grouped_filter
            wq = self._int8((K, C // g["G"], R, S))
            self.w = grouped_filter(wq, g["G"], g["B"])
            acc = F.conv2d(self.x.permute(0, 3, 1, 2).double(), wq.double(), None, g["st"], g["pad"], g["dil"], g["G"])
            assert acc.numel() == 0 or float(acc.abs().max()) < 2.0 ** 53
            self.acc = torch.round(acc).long().permute(0, 2, 3, 1).reshape(-1, K)
        b = torch.randint(-128, 128, (K,), generator=self.gen, device="cuda", dtype=torch.int32)
        b[:4] = torch.tensor([-128, -1, 0, 127][:K], dtype=torch.int32)
        self.bias = b
        mx = int(self.acc.abs().max()) if self.acc.numel() else 0
        self.rs = max(1, min(20, mx.bit_length() - 6))     # outputs spread over the int8 range, few saturate
        self.x0, self.w0 = self.x.clone(), self.w.clone()

    def _int8(self, shape):
        return torch.randint(-128, 128, shape, generator=self.gen, device="cuda", dtype=torch.int8)

    def fold(self, rs):
        """the folded [3K] bias with PQ_FLAG_BIAS_FOLDED; where K % 16 != 0 (which bias_fold leaves alone) a [3K]
        buffer whose tail is noise, which the kernel must ignore"""
        from common.quantity import _native
        f = _native.bias_fold(self.bias, rs)
        if f.numel() == 3 * self.K:
            return f
        noise = torch.randint(-2 ** 31, 2 ** 31 - 1, (2 * self.K,), generator=self.gen, device="cuda", dtype=torch.int32)
        return torch.cat([self.bias, noise])

    def launch(self, rs, ob, bias_ptr, flags, fp, sp):
        entry = _lib().pq_conv2d_dw_s8 if self.kind == "dw" else _lib().pq_conv2d_s8
        return entry(self.x.data_ptr(), self.w.data_ptr(), bias_ptr, ctypes.byref(_desc(self.g, rs, ob)), flags, fp,
                     sp, _stream())

    def run(self, rs, ob, bias, relu, out, s8_skew=0, f32_skew=0):
        """One launch; returns (fp32 as [M][K] or None, int8 [M][K] or None)."""
        f32 = Guarded((self.g["N"], self.K, self.P, self.Q), torch.float32, f32_skew) if out in ("f32", "both") else None
        s8 = Guarded((self.M, self.K), torch.int8, s8_skew) if out in ("s8", "both") else None
        b0 = bias.clone()
        rc = self.launch(rs, ob, bias.data_ptr(), _flags(bias, self.K, relu), f32.ptr() if f32 else None,
                         s8.ptr() if s8 else None)
        assert rc == 0, "launch failed: %s" % _lib().pq_error_string(rc).decode()
        torch.cuda.synchronize()
        for gd, name in ((f32, "fp32"), (s8, "int8")):
            if gd is not None:
                gd.check(name)
        assert torch.equal(bias, b0), "the bias was modified"
        return (f32.t.permute(0, 2, 3, 1).reshape(self.M, self.K) if f32 else None), (s8.t if s8 else None)

    def check_operands(self):
        assert torch.equal(self.x, self.x0), "the input was modified"
        assert torch.equal(self.w, self.w0), "the weights were modified"


def check_values(case, rs, ob, bias_kind, relu, out, kernel=None):
    bias = case.fold(rs) if bias_kind == "fold" else case.bias
    want = epilogue_ref(case.acc, case.bias.long(), rs, relu)
    run = lambda: case.run(rs, ob, bias, relu, out)                      # noqa: E731
    f32, s8 = check_landing(run, kernel) if kernel is not None else run()
    what = "rs=%d ob=%d bias=%s relu=%s out=%s" % (rs, ob, bias_kind, relu, out)
    if s8 is not None:
        assert torch.equal(s8.long(), want), what
    if f32 is not None:
        assert torch.equal(f32, dequant_ref(want, ob)), what


def run_row(case, kernel, seed):
    """Plain and folded bias; int8-only, fp32-only and both outputs; ReLU off and on; rs and ob spread over rows."""
    rs, ob = case.rs, OBS[seed % len(OBS)]
    want = epilogue_ref(case.acc, case.bias.long(), rs, False)
    if want.numel() >= 16:
        assert int((want != want[0, 0]).sum()) > 0 and bool(((want > -128) & (want < 127)).any()), "degenerate row"
    check_values(case, rs, ob, "fold", False, "s8", kernel)
    check_values(case, min(rs + 1, 24), OBS[(seed + 1) % len(OBS)], "plain", True, "f32")
    check_values(case, max(rs - 1, 1), ob, "fold" if seed & 1 else "plain", bool(seed & 2), "both")
    case.check_operands()


@gpu
@pytest.mark.parametrize("row", DW_ROWS, ids=[dw_row_id(r) for r in DW_ROWS])
def test_depthwise_row_vs_exact_convolution(row, b200):
    inst, g = row
    assert dw_inst(g["C"], g["R"], g["S"]) == inst
    seed = zlib.crc32(dw_row_id(row).encode())
    run_row(Case(g, "dw", seed), ("dw",) + inst, seed)


@gpu
def test_depthwise_all_minus_128_saturates(b200):
    """7 x 7 with every operand -128: acc = 49 * 2^14 on every pixel and channel, and every output saturates to 127."""
    case = Case(DW_SATURATED, "dw", 1, fill=-128)
    assert bool((case.acc == 49 * 2 ** 14).all())
    for rs, relu, kind, out in ((1, False, "fold", "s8"), (12, True, "fold", "both"), (7, False, "plain", "f32"),
                                (-3, True, "plain", "s8")):
        assert bool((right_shift(case.acc, rs) == 127).all())
        check_values(case, rs, 2, kind, relu, out, ("dw", 1, 0) if rs == 1 else None)
    case.check_operands()


@gpu
def test_depthwise_output_and_bias_alignment(b200):
    """out_s8 16 bytes past a boundary runs, 8 bytes past is PQ_EALIGN; out_f32 and the bias 4 bytes past run, 2 bytes
    past are PQ_EALIGN; a refused call writes nothing."""
    g = D(2, 9, 11, 32, 32, 3, 3, pad=(1, 1))
    case = Case(g, "dw", 2)
    want = epilogue_ref(case.acc, case.bias.long(), case.rs, True)
    f32, s8 = case.run(case.rs, 3, case.bias, True, "s8", s8_skew=16)
    assert torch.equal(s8.long(), want)
    f32, s8 = case.run(case.rs, 3, case.bias, True, "f32", f32_skew=4)
    assert torch.equal(f32, dequant_ref(want, 3))
    shifted = torch.cat([torch.zeros(1, dtype=torch.int32, device="cuda"), case.bias])      # bias 4 bytes past 16
    out = Guarded((case.M, case.K), torch.int8)
    assert case.launch(case.rs, 3, shifted.data_ptr() + 4, _native_flag("relu"), None, out.ptr()) == 0
    torch.cuda.synchronize()
    out.check("int8")
    assert torch.equal(out.t.long(), want)
    for s8_skew, f32_skew, bias_off in ((8, 0, 0), (0, 2, 0), (0, 0, 2)):
        outs = (Guarded((g["N"], g["K"], case.P, case.Q), torch.float32), Guarded((case.M, case.K), torch.int8, s8_skew))
        rc = case.launch(case.rs, 3, shifted.data_ptr() + (bias_off or 4), 0, outs[0].ptr() + f32_skew, outs[1].ptr())
        torch.cuda.synchronize()
        assert rc == EALIGN, (s8_skew, f32_skew, bias_off, rc)
        assert all(o.untouched() for o in outs), "a refused call wrote"
    case.check_operands()


def _native_flag(name):
    from common.quantity import _native
    return {"relu": _native.FLAG_RELU, "fold": _native.FLAG_BIAS_FOLDED}[name]


# ------------------------------------------------------------------------------------------ depthwise limits
# (limit as the header words it, geometry, expected return code); accepted rows run and are compared.
DW_LIMITS = [
    ("R, S <= 7", D(2, 9, 9, 32, 32, 7, 3, pad=(3, 1)), 0),
    ("R, S <= 7", D(2, 9, 9, 32, 32, 8, 3, pad=(3, 1)), EUNSUPPORTED),
    ("R, S <= 7", D(2, 9, 9, 32, 32, 3, 7, pad=(1, 3)), 0),
    ("R, S <= 7", D(2, 9, 9, 32, 32, 3, 8, pad=(1, 3)), EUNSUPPORTED),
    ("stride <= 2", D(2, 9, 9, 32, 32, 3, 3, st=(2, 1)), 0),
    ("stride <= 2", D(2, 9, 9, 32, 32, 3, 3, st=(3, 1)), EUNSUPPORTED),
    ("stride <= 2", D(2, 9, 9, 32, 32, 3, 3, st=(1, 2)), 0),
    ("stride <= 2", D(2, 9, 9, 32, 32, 3, 3, st=(1, 3)), EUNSUPPORTED),
    ("dilation <= 2", D(2, 9, 9, 32, 32, 3, 3, dil=(2, 1)), 0),
    ("dilation <= 2", D(2, 9, 9, 32, 32, 3, 3, dil=(3, 1)), EUNSUPPORTED),
    ("dilation <= 2", D(2, 9, 9, 32, 32, 3, 3, dil=(1, 2)), 0),
    ("dilation <= 2", D(2, 9, 9, 32, 32, 3, 3, dil=(1, 3)), EUNSUPPORTED),
    ("pad <= (R-1)*dil", D(2, 5, 6, 16, 16, 5, 3, pad=(8, 1), dil=(2, 1)), 0),
    ("pad <= (R-1)*dil", D(2, 5, 6, 16, 16, 5, 3, pad=(9, 1), dil=(2, 1)), EUNSUPPORTED),
    ("pad <= (R-1)*dil", D(2, 5, 6, 16, 16, 3, 4, pad=(1, 6), dil=(1, 2)), 0),
    ("pad <= (R-1)*dil", D(2, 5, 6, 16, 16, 3, 4, pad=(1, 7), dil=(1, 2)), EUNSUPPORTED),
    ("C % 16 == 0", D(2, 5, 6, 16, 8, 3, 3, pad=(1, 1)), 0),
    ("C % 16 == 0", D(2, 5, 6, 8, 8, 3, 3, pad=(1, 1)), EUNSUPPORTED),
    ("C % 16 == 0", D(2, 5, 6, 48, 40, 3, 3, pad=(1, 1)), 0),
    ("C % 16 == 0", D(2, 5, 6, 40, 40, 3, 3, pad=(1, 1)), EUNSUPPORTED),
    # the launch grid: C / (16 * G) CTAs along y, at most 65535 (N = H = W = 1)
    ("C / (16*G) <= 65535", D(1, 1, 1, 16 * 65535, 16 * 65535, 3, 3, pad=(1, 1)), 0),
    ("C / (16*G) <= 65535", D(1, 1, 1, 16 * 65537, 16 * 65537, 3, 3, pad=(1, 1)), EUNSUPPORTED),
    ("C / (16*G) <= 65535", D(1, 1, 1, 32 * 65535, 32 * 65535 - 5, 3, 3, pad=(1, 1)), 0),
    ("C / (16*G) <= 65535", D(1, 1, 1, 32 * 65537, 32 * 65537, 3, 3, pad=(1, 1)), EUNSUPPORTED),
    ("C / (16*G) <= 65535", D(1, 1, 1, 64 * 65535, 64 * 65535, 1, 1), 0),
    ("C / (16*G) <= 65535", D(1, 1, 1, 64 * 65536, 64 * 65536, 1, 1), EUNSUPPORTED),
]
DW_SIZE_LIMITS = ["N*P*Q <= 2^31 - 1"]           # test_depthwise_m_limit_at_size


def dw_limit_id(r):
    return "%s-%s-C%d" % (re.sub(r"[^0-9A-Za-z]+", "_", r[0]).strip("_"), "ok" if r[2] == 0 else "refused", r[1]["C"])


def _center_tap_acc(x, w, K):
    """int64 [N][K] accumulators of a 1 x 1 image under a filter whose only tap inside the image is the centre one."""
    R, S = w.shape[:2]
    return x[:, 0, 0, :K].long() * w[R // 2, S // 2, :K].long().view(1, -1)


@gpu
@pytest.mark.parametrize("row", DW_LIMITS, ids=[dw_limit_id(r) + "-%d" % i for i, r in enumerate(DW_LIMITS)])
def test_depthwise_limit_one_step_inside_and_beyond(row, b200):
    _, g, want = row
    seed = zlib.crc32(repr(row).encode())
    if want == 0 and g["C"] <= 4096:
        run_row(Case(g, "dw", seed), ("dw",) + dw_inst(g["C"], g["R"], g["S"]), seed)
        return
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(-128, 128, (g["N"], g["H"], g["W"], g["C"]), generator=gen, device="cuda", dtype=torch.int8)
    w = torch.randint(-128, 128, (g["R"], g["S"], g["C"]), generator=gen, device="cuda", dtype=torch.int8)
    w[..., g["K"]:] = 0
    bias = torch.randint(-128, 128, (g["K"],), generator=gen, device="cuda", dtype=torch.int32)
    x0, w0, b0 = x.clone(), w.clone(), bias.clone()
    P, Q = out_size(g)
    M = g["N"] * P * Q
    outs = (Guarded((g["N"], g["K"], P, Q), torch.float32), Guarded((M, g["K"]), torch.int8))
    call = lambda: _lib().pq_conv2d_dw_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(),        # noqa: E731
                                          ctypes.byref(_desc(g, 9, 1)), 0, outs[0].ptr(), outs[1].ptr(), _stream())
    if want != 0:
        rc = call()
        torch.cuda.synchronize()
        assert rc == want, (rc, want)
        assert all(o.untouched() for o in outs), "a refused call wrote"
        # nothing is left behind for the next launch to report
        t = torch.ones(1 << 20, device="cuda").add_(1)
        torch.cuda.synchronize()
        assert float(t.sum()) == 2.0 * (1 << 20)
    else:                                              # the widths at the grid limit: centre tap only, P = Q = 1
        rc = check_landing(call, ("dw",) + dw_inst(g["C"], g["R"], g["S"]))
        torch.cuda.synchronize()
        assert rc == 0
        y = epilogue_ref(_center_tap_acc(x, w, g["K"]), bias.long(), 9, False)
        outs[0].check("fp32"), outs[1].check("int8")
        assert torch.equal(outs[1].t.long(), y) and torch.equal(outs[0].t.view(M, g["K"]), dequant_ref(y, 1))
        assert int(y.unique().numel()) > 100
    assert torch.equal(x, x0) and torch.equal(w, w0) and torch.equal(bias, b0)


# ------------------------------------------------------------------------------------------ depthwise at size
@gpu
def test_depthwise_m_limit_at_size(b200):
    """M = N*P*Q at 2^31 - 1: 1 x 1 x 16 images under a 7 x 7 filter at dilation 2 and pad 12 give P = Q = 13 (169
    pixels an image); K = 1.  12,707,003 images (M = 2,147,483,507, about 2.1 GB of int8 output) are accepted, one image
    more is refused and writes nothing.  Output pixel (p, q) sees the image's one pixel through tap ((12 - p) / 2,
    (12 - q) / 2) when p and q are even, and nothing otherwise, so each image's output is a function of its own pixel:
    it is compared in chunks against a table over the 256 byte values.  This guards the 32-bit m of the kernel, which
    stays in range because kDwThreads / G * kDwPixIters is a power of two."""
    n_ok, hw = 12707003, 169
    g = D(n_ok + 1, 1, 1, 16, 1, 7, 7, pad=(12, 12), dil=(2, 2))
    assert out_size(g) == (13, 13) and (n_ok + 1) * hw > M_LIMIT >= n_ok * hw
    gen = torch.Generator(device="cuda").manual_seed(21)
    x = torch.randint(-128, 128, (n_ok + 1, 1, 1, 16), generator=gen, device="cuda", dtype=torch.int8)
    w = torch.zeros((7, 7, 16), dtype=torch.int8, device="cuda")
    w[..., 0] = torch.randint(-128, 128, (7, 7), generator=gen, device="cuda", dtype=torch.int8)
    bias = torch.tensor([-7], dtype=torch.int32, device="cuda")
    rs = 3
    x_sum, w0 = int(x[::4099].long().sum()), w.clone()
    out = Guarded(((n_ok + 1) * hw,), torch.int8)
    rc = _lib().pq_conv2d_dw_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(), ctypes.byref(_desc(g, rs, 0)), 0, None,
                                out.ptr(), _stream())
    torch.cuda.synchronize()
    assert rc == EUNSUPPORTED and out.untouched()
    g["N"] = n_ok
    rc = check_landing(lambda: _lib().pq_conv2d_dw_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                                      ctypes.byref(_desc(g, rs, 0)), 0, None, out.ptr(), _stream()),
                       ("dw", 1, 0))
    torch.cuda.synchronize()
    assert rc == 0
    # table[v + 128] = the 169 outputs of an image whose pixel is v
    vals = torch.arange(-128, 128, device="cuda", dtype=torch.int8).view(256, 1, 1, 1).expand(256, 1, 1, 16).contiguous()
    table = epilogue_ref(dw_exact(vals, w, 1, (1, 1), (12, 12), (2, 2)), bias.long(), rs, False).view(256, hw)
    assert int(table.unique().numel()) > 50
    table = table.to(torch.int8)
    img = out.t[:n_ok * hw].view(n_ok, hw)
    for a, b in _chunks(n_ok, 1 << 20):
        assert torch.equal(img[a:b], table[x[a:b, 0, 0, 0].long() + 128]), a
    assert bool((out.buf[out.lo + n_ok * hw:] == SENTINEL).all()) and bool((out.buf[:out.lo] == SENTINEL).all())
    assert int(x[::4099].long().sum()) == x_sum and torch.equal(w, w0)


def dw_band_acc(x, n, w_rsc, K, st, pad, dil, p0, p1):
    """int64 [p1 - p0][Q][K] accumulators of output rows p0 .. p1 - 1 of image n, from the input rows they read."""
    H, W = x.shape[1], x.shape[2]
    R = w_rsc.shape[0]
    lo = p0 * st[0] - pad[0]
    hi = (p1 - 1) * st[0] - pad[0] + (R - 1) * dil[0] + 1
    band = torch.zeros((hi - lo, W, K), dtype=torch.int8, device=x.device)
    a, b = max(lo, 0), min(hi, H)
    band[a - lo:b - lo] = x[n, a:b, :, :K]
    acc = F.conv2d(band.permute(2, 0, 1).unsqueeze(0).double(), w_rsc[..., :K].permute(2, 0, 1).unsqueeze(1).double(),
                   None, st, (0, pad[1]), dil, K)
    return torch.round(acc[0]).long().permute(1, 2, 0)


@gpu
def test_depthwise_big_image_at_size(b200):
    """One image of 11586 x 11586 x 16 = 2,147,766,336 bytes (over 2^31) and a batch of two (over 2^32 bytes), 3 x 3,
    stride 2, pad 1: bands of output rows on both sides of each 2^31-byte boundary of the input, and at the edges of
    both images, against a reference cropped to the input rows they read."""
    HW, C = 11586, 16
    img_bytes = HW * HW * C
    assert img_bytes > 2 ** 31 and 2 * img_bytes > 2 ** 32
    g = D(2, HW, HW, C, C, 3, 3, st=(2, 2), pad=(1, 1))
    P, Q = out_size(g)
    gen = torch.Generator(device="cuda").manual_seed(22)
    x = torch.randint(-128, 128, (2, HW, HW, C), generator=gen, device="cuda", dtype=torch.int8)
    w = torch.randint(-128, 128, (3, 3, C), generator=gen, device="cuda", dtype=torch.int8)
    bias = torch.randint(-128, 128, (C,), generator=gen, device="cuda", dtype=torch.int32)
    x_sum, w0 = int(x[:, ::97, ::89].long().sum()), w.clone()
    rs = 13
    out = Guarded((2 * P * Q * C,), torch.int8)
    rc = check_landing(lambda: _lib().pq_conv2d_dw_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                                      ctypes.byref(_desc(g, rs, 0)), _native_flag("relu"), None,
                                                      out.ptr(), _stream()), ("dw", 1, 3))
    torch.cuda.synchronize()
    assert rc == 0
    o = out.t.view(2, P, Q, C)
    row_bytes = HW * C
    bands = {(0, 0), (0, P - 3), (1, 0), (1, P - 3)}
    for boundary in (2 ** 31, 2 ** 32):
        n, h = divmod(boundary // row_bytes, HW)
        bands.add((n, max(0, h // 2 - 3)))                 # output rows whose input rows straddle the boundary
    checked = 0
    for n, p0 in sorted(bands):
        p1 = min(P, p0 + 6)
        want = epilogue_ref(dw_band_acc(x, n, w, C, (2, 2), (1, 1), (1, 1), p0, p1).reshape(-1, C), bias.long(), rs,
                            True)
        assert torch.equal(o[n, p0:p1].reshape(-1, C).long(), want), (n, p0)
        checked += 1
    assert checked == 6
    out.check("int8")
    assert int(x[:, ::97, ::89].long().sum()) == x_sum and torch.equal(w, w0)


# ------------------------------------------------------------------------------------------ grouped rows
def GG(N, H, W, C, K, G, B, R, S, st=(1, 1), pad=(0, 0), dil=(1, 1)):
    return dict(N=N, H=H, W=W, C=C, K=K, G=G, B=B, R=R, S=S, st=st, pad=pad, dil=dil)


# (name: mode / BN.BK.STAGES.BSLOTS / tps / resident or streamed weights, geometry)
GROUPED_ROWS = [
    # R != S
    ("im2col/32.32.9.9/tps3/str", GG(2, 9, 13, 64, 64, 2, 32, 1, 3, pad=(0, 1))),
    ("im2col/32.64.9.9/tps3/str", GG(3, 11, 7, 128, 64, 4, 32, 3, 1, st=(2, 1), pad=(1, 0))),
    ("im2col/64.32.9.9/tps1/str", GG(2, 6, 20, 64, 128, 2, 64, 1, 7, st=(1, 2), pad=(0, 3))),
    ("im2col/128.128.6.6/tps1/str", GG(2, 12, 10, 256, 256, 8, 128, 5, 3, pad=(2, 1), dil=(1, 2))),
    # strides 1 to 8, stride_h != stride_w, strides larger than the filter
    ("im2col/32.32.9.9/tps3/str", GG(2, 30, 25, 64, 64, 2, 32, 3, 3, st=(4, 3), pad=(1, 1))),
    ("im2col/32.32.9.9/tps1/str", GG(2, 40, 17, 96, 96, 3, 32, 2, 2, st=(8, 5), pad=(0, 1))),
    ("im2col/64.64.9.9/tps3/str", GG(1, 19, 30, 128, 128, 4, 64, 3, 3, st=(6, 7), pad=(2, 0))),
    ("im2col/32.32.9.9/tps1/str", GG(3, 13, 25, 64, 64, 2, 32, 1, 2, st=(3, 8), pad=(0, 1))),
    # dil_h != dil_w
    ("im2col/32.32.9.9/tps3/str", GG(2, 17, 15, 64, 64, 4, 32, 3, 3, pad=(2, 1), dil=(2, 1))),
    ("im2col/64.32.9.9/tps3/str", GG(2, 13, 16, 128, 256, 4, 64, 2, 3, st=(2, 1), pad=(1, 3), dil=(3, 2))),
    # pads asymmetric and beyond (R - 1) * dil: output pixels wholly in padding
    ("im2col/32.32.9.9/tps3/str", GG(2, 5, 9, 64, 64, 2, 32, 3, 3, st=(1, 2), pad=(4, 0))),
    ("im2col/64.64.18.9/tps3/res", GG(1, 3, 4, 64, 64, 2, 64, 1, 3, pad=(3, 5))),
    # H, W, P, Q = 1 and batch 1
    ("im2col/32.32.9.9/tps1/str", GG(1, 1, 1, 64, 64, 2, 32, 1, 1, st=(2, 2))),
    ("im2col/64.32.9.9/tps3/str", GG(3, 1, 19, 64, 128, 2, 64, 1, 3, st=(1, 2), pad=(0, 1))),
    ("im2col/32.64.9.9/tps3/str", GG(4, 17, 1, 128, 64, 2, 32, 3, 1, st=(2, 1), pad=(1, 0))),
    ("im2col/32.32.9.9/tps3/str", GG(5, 3, 9, 64, 64, 2, 32, 3, 3, st=(2, 8), pad=(0, 1))),   # P = 1, Q = 2
    # tiles crossing images, M % 128 != 0
    ("im2col/32.32.9.9/tps3/str", GG(5, 7, 9, 64, 64, 2, 32, 3, 3, pad=(1, 1))),
    ("im2col/128.64.9.9/tps3/res", GG(7, 5, 11, 64, 128, 2, 128, 3, 3, st=(1, 2), pad=(1, 1))),
    # 1 x 1 off the plain path (pad > 0, stride 2): im2col
    ("im2col/32.32.9.9/tps1/str", GG(2, 9, 9, 64, 64, 2, 32, 1, 1, pad=(1, 0))),
    ("im2col/64.32.9.9/tps1/str", GG(3, 10, 11, 128, 256, 4, 64, 1, 1, st=(2, 2))),
    # plain 1 x 1: Wb = 16, 48, 80, 144 -- BK exceeds Wb or does not divide it; the box reads into the next group's
    # channels or past C and meets zero weights
    ("gemm/32.32.9.9/tps1/str", GG(3, 7, 9, 64, 128, 4, 32, 1, 1)),
    ("gemm/32.32.9.9/tps1/str", GG(2, 9, 9, 96, 64, 2, 32, 1, 1)),
    ("gemm/32.64.9.9/tps1/str", GG(2, 8, 7, 160, 64, 2, 32, 1, 1)),
    ("gemm/32.128.8.8/tps1/str", GG(2, 7, 9, 288, 64, 2, 32, 1, 1)),
    # window origins inside a CTA's tile walk: > 148 tiles, n-tile counts 8 and 64 (not dividing 148), so one
    # 32-tile batch of produce_a spans several channel windows
    ("im2col/32.32.9.9/tps3/str", GG(13, 14, 14, 256, 256, 8, 32, 3, 3, pad=(1, 1))),
    ("gemm/32.32.9.9/tps1/str", GG(12, 10, 10, 256, 256, 8, 32, 1, 1)),
    ("im2col/32.32.9.9/tps3/str", GG(3, 10, 10, 2048, 2048, 64, 32, 3, 3, pad=(1, 1))),
    ("gemm/32.32.9.9/tps1/str", GG(2, 9, 17, 2048, 2048, 64, 32, 1, 1)),
    # Wb > BK with two or more n tiles: c0 + cb * BK at non-zero origins
    ("im2col/32.128.8.8/tps1/str", GG(2, 7, 7, 512, 64, 2, 32, 3, 3, pad=(1, 1))),
    ("im2col/32.128.8.8/tps1/str", GG(2, 6, 5, 1024, 64, 2, 32, 3, 1, st=(1, 2), pad=(1, 0))),
    ("gemm/32.128.8.8/tps1/str", GG(3, 9, 7, 512, 64, 2, 32, 1, 1)),
    # tpg > 1 at B = 256 (Kg = 512), and Cg = 2 (G = C / 2)
    ("im2col/256.128.4.4/tps1/str", GG(2, 7, 7, 1024, 1024, 2, 256, 3, 3, pad=(1, 1))),
    ("im2col/32.32.9.9/tps3/str", GG(3, 9, 11, 64, 64, 32, 32, 3, 3, pad=(1, 1))),
    ("im2col/64.64.9.9/tps3/str", GG(2, 9, 11, 128, 128, 64, 64, 3, 3, st=(2, 1), pad=(1, 1))),
    # the remaining tile configurations, resident and streamed weights
    ("im2col/32.64.9.9/tps1/str", GG(2, 9, 8, 128, 64, 2, 32, 2, 2, pad=(1, 0))),
    ("im2col/64.128.8.8/tps1/res", GG(2, 8, 9, 256, 64, 2, 64, 1, 3, pad=(0, 1))),
    ("im2col/64.128.8.8/tps1/str", GG(2, 8, 9, 256, 128, 2, 64, 1, 3, pad=(0, 1))),
    ("im2col/128.32.9.9/tps3/res", GG(2, 9, 9, 32, 128, 2, 128, 3, 3, pad=(1, 1))),
    ("im2col/128.32.9.9/tps3/str", GG(2, 9, 9, 64, 256, 2, 128, 3, 3, pad=(1, 1))),
    ("im2col/128.64.9.9/tps1/str", GG(2, 9, 9, 128, 256, 2, 128, 2, 2, pad=(1, 1))),
    ("im2col/256.32.9.9/tps3/str", GG(2, 7, 9, 64, 512, 2, 256, 3, 3, pad=(1, 1))),
    ("im2col/256.32.9.9/tps3/res", GG(2, 7, 9, 32, 256, 2, 256, 1, 3, pad=(0, 1))),
    ("im2col/256.64.8.8/tps3/str", GG(2, 7, 7, 128, 512, 2, 256, 3, 3, pad=(1, 1))),
    ("im2col/256.64.8.8/tps1/res", GG(2, 7, 7, 64, 256, 2, 256, 2, 2, pad=(1, 1))),
    ("gemm/64.64.9.9/tps1/res", GG(2, 9, 9, 64, 64, 2, 64, 1, 1)),
    # 3 x 3 / stride 1 / pad 1 at C = 64 and 128 (the dense layer's patch-window shapes) stay on im2col when grouped
    ("im2col/32.32.9.9/tps3/str", GG(2, 14, 14, 64, 64, 2, 32, 3, 3, pad=(1, 1))),
    ("im2col/128.128.6.6/tps1/str", GG(2, 9, 13, 128, 128, 2, 128, 3, 3, pad=(1, 1))),
]


def grouped_row_id(r):
    g = r[1]
    return "%s-n%d-%dx%dx%d-k%d-g%d-b%d-%dx%d-s%d.%d-p%d.%d-d%d.%d" % (
        r[0].replace("/", "."), g["N"], g["H"], g["W"], g["C"], g["K"], g["G"], g["B"], g["R"], g["S"], *g["st"],
        *g["pad"], *g["dil"])


@gpu
@pytest.mark.parametrize("row", GROUPED_ROWS, ids=[grouped_row_id(r) for r in GROUPED_ROWS])
def test_grouped_row_vs_exact_convolution(row, b200):
    name, g = row
    assert grouped_name(g) == name
    seed = zlib.crc32(grouped_row_id(row).encode())
    run_row(Case(g, "grouped", seed), grouped_choice(g)[0], seed)


# TMA's im2col corner limits under grouping: one step inside and one beyond each
GROUPED_LIMITS = [
    ("pad <= 128", GG(1, 1, 3, 64, 64, 2, 32, 2, 1, pad=(128, 0)), 0),
    ("pad <= 128", GG(1, 1, 3, 64, 64, 2, 32, 2, 1, pad=(129, 0)), EUNSUPPORTED),
    ("pad - (R-1)*dil <= 127", GG(1, 2, 4, 64, 64, 2, 32, 1, 3, pad=(127, 1)), 0),
    ("pad - (R-1)*dil <= 127", GG(1, 2, 4, 64, 64, 2, 32, 1, 3, pad=(128, 1)), EUNSUPPORTED),
    ("(R-1)*dil - pad <= 128", GG(1, 130, 3, 64, 64, 2, 32, 2, 1, dil=(128, 1)), 0),
    ("(R-1)*dil - pad <= 128", GG(1, 130, 3, 64, 64, 2, 32, 2, 1, dil=(129, 1)), EUNSUPPORTED),
]


@gpu
@pytest.mark.parametrize("row", GROUPED_LIMITS, ids=["%s-%s" % (re.sub(r"[^0-9A-Za-z]+", "_", r[0]).strip("_"),
                                                                  "ok" if r[2] == 0 else "refused")
                                                      for r in GROUPED_LIMITS])
def test_grouped_corner_limits(row, b200):
    _, g, want = row
    seed = zlib.crc32(repr(row).encode())
    case = Case(g, "grouped", seed)
    if want == 0:
        run_row(case, grouped_choice(g)[0], seed)
        return
    outs = (Guarded((g["N"], g["K"], case.P, case.Q), torch.float32), Guarded((case.M, case.K), torch.int8))
    rc = case.launch(7, 0, case.bias.data_ptr(), 0, outs[0].ptr(), outs[1].ptr())
    torch.cuda.synchronize()
    assert rc == want and all(o.untouched() for o in outs), rc
    case.check_operands()


@gpu
def test_grouped_m_limit_refused(b200):
    """M = N*P*Q = 2^31 exactly (32768 images of 2 x 2 x 64 at pad 127 under a 1 x 1 filter: P = Q = 256) is refused
    and writes nothing.  The accepted side, M = 2^31 - 1, would need at least 64 GB of int8 output (a grouped layer has
    K >= 32), so it does not run here; the index arithmetic it shares with the dense layer runs at full size in
    test_gpu_conv_geometry.py::test_m_limit_at_size."""
    g = GG(32768, 2, 2, 64, 64, 2, 32, 1, 1, pad=(127, 127))
    assert out_size(g) == (256, 256) and g["N"] * 256 * 256 == 2 ** 31
    x = torch.ones((g["N"], 2, 2, 64), dtype=torch.int8, device="cuda")
    w = torch.ones((64, 1, 1, 32), dtype=torch.int8, device="cuda")
    bias = torch.zeros(64, dtype=torch.int32, device="cuda")
    outs = (Guarded((4096,), torch.float32), Guarded((4096,), torch.int8))       # small: nothing may be written
    rc = _lib().pq_conv2d_s8(x.data_ptr(), w.data_ptr(), bias.data_ptr(), ctypes.byref(_desc(g, 7, 0)), 0,
                             outs[0].ptr(), outs[1].ptr(), _stream())
    torch.cuda.synchronize()
    assert rc == EUNSUPPORTED and all(o.untouched() for o in outs)


# ------------------------------------------------------------------------------------------ NewConv2d
INFO = {"weight_bit": 7, "input_bit": 5, "output_bit": 4, "bias_bit": 5}

# (cin, cout, kernel, stride, padding, dilation, groups, (H, W)); groups == cin == cout: depthwise
NEWCONV = [
    (24, 24, (3, 3), (1, 2), (1, 0), (2, 1), 24, (13, 17)),
    (40, 40, (1, 7), (2, 2), (0, 6), (1, 2), 40, (9, 20)),
    (64, 64, (7, 1), (1, 1), (3, 0), (1, 1), 64, (15, 6)),
    (96, 96, (5, 5), (2, 2), (4, 2), (1, 1), 96, (11, 12)),
    (16, 16, (7, 7), (1, 1), (12, 12), (2, 2), 16, (3, 3)),
    (32, 32, (2, 2), (2, 1), (1, 0), (1, 1), 32, (10, 9)),
    (17, 17, (3, 3), (2, 2), (2, 1), (1, 1), 17, (1, 9)),
    (64, 64, (1, 3), (1, 1), (0, 1), (1, 1), 2, (9, 13)),
    (128, 64, (3, 1), (2, 1), (1, 0), (1, 1), 4, (11, 7)),
    (64, 128, (1, 7), (1, 2), (0, 3), (1, 1), 2, (6, 20)),
    (96, 96, (3, 3), (3, 2), (2, 1), (2, 1), 3, (17, 12)),
    (64, 64, (3, 3), (8, 5), (4, 0), (1, 1), 2, (20, 17)),
    (64, 64, (1, 1), (2, 2), (0, 0), (1, 1), 2, (9, 10)),
    (48, 96, (1, 1), (1, 1), (0, 0), (1, 1), 3, (7, 9)),
    (64, 64, (3, 3), (1, 1), (4, 1), (1, 1), 32, (5, 9)),
    (512, 64, (3, 3), (1, 1), (1, 1), (1, 1), 2, (5, 6)),
]


def _layer(cin, cout, k, stride, pad, dil, groups, seed):
    g = torch.Generator().manual_seed(seed)
    conv = nn.Conv2d(cin, cout, k, stride, pad, dil, groups, bias=True)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 0.3)
        conv.bias.copy_(torch.randn(cout, generator=g))
    return conv


@gpu
@pytest.mark.parametrize("layer", NEWCONV, ids=["c%d-k%d-%dx%d-s%d.%d-p%d.%d-d%d.%d-g%d" % (
    l[0], l[1], *l[2], *l[3], *l[4], *l[5], l[6]) for l in NEWCONV])
def test_newconv2d_vs_oracle_and_int8_pipeline(layer, oracle):
    """NewConv2d on a depthwise or grouped layer of each geometry class equals the oracle; in the int8 pipeline it
    returns a QTensor with the same values, and a following ReLU runs inside its epilogue."""
    from common.quantity import NewConv2d, QTensor, _native
    cin, cout, k, st, pad, dil, groups, (H, W) = layer
    conv = _layer(cin, cout, k, st, pad, dil, groups, seed=zlib.crc32(repr(layer).encode()))
    w, b = conv.weight.detach().numpy().copy(), conv.bias.detach().numpy().copy()
    x = np.random.default_rng(cin + groups).normal(0, 2, (2, cin, H, W)).astype(np.float32)
    ref, yi = oracle.int_conv_layer(x, w, b, INFO, stride=st, padding=pad, dilation=dil, groups=groups)
    mod = NewConv2d(conv.cuda(), dict(INFO)).eval()
    depthwise = cin == cout == groups
    assert mod._depthwise == depthwise and bool(mod._group_block) == (not depthwise) and mod._group_convs is None
    xt = torch.from_numpy(x).cuda()
    with torch.no_grad():
        out = mod(xt)
    assert np.array_equal(out.cpu().numpy(), ref)
    assert len(np.unique(yi)) > 20
    mod.int8_pipeline = True
    relu0 = _native.LAUNCHES.get("relu_s8", 0)
    with torch.no_grad():
        q = mod(xt)
        assert isinstance(q, QTensor)
        assert np.array_equal(q.dequantize().cpu().numpy(), ref)
        qr = F.relu(mod(xt))
        assert isinstance(qr, QTensor)
        assert np.array_equal(qr.dequantize().cpu().numpy(), np.maximum(ref, 0))
    assert _native.LAUNCHES.get("relu_s8", 0) == relu0


@gpu
@pytest.mark.parametrize("C", [16 * 65537, 32 * 65537, 64 * 65536])
def test_newconv2d_depthwise_wider_than_the_grid_raises_on_first_forward(C):
    """A depthwise layer wider than the launch grid allows: NewConv2d builds it on the depthwise kernel, the first
    forward raises a RuntimeError naming PQ_EUNSUPPORTED (there is no fall-back)."""
    from common.quantity import NewConv2d
    conv = nn.Conv2d(C, C, 3, 1, 1, groups=C).cuda()
    mod = NewConv2d(conv, dict(INFO))
    assert mod._depthwise and mod._payload_channels == C
    with pytest.raises(RuntimeError, match="PQ_EUNSUPPORTED"):
        mod(torch.randn(1, C, 1, 1, device="cuda"))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ CPU checks
def test_reference_equals_oracle_on_depthwise_and_grouped_layers(oracle):
    """dw_exact and the grouped F.conv2d + epilogue_ref against the oracle's NewConv2d (int_conv_layer(groups=...)) on
    integer-valued operands, rectangular filters, asymmetric stride and padding, and dilation."""
    gen = torch.Generator().manual_seed(4)
    for (R, S), st, pad, dil, groups, C in (((2, 3), (2, 1), (1, 2), (2, 1), 32, 32), ((1, 5), (1, 2), (0, 4), (1, 2), 16, 16),
                                            ((3, 1), (2, 2), (2, 0), (1, 1), 4, 64), ((5, 3), (1, 3), (3, 1), (2, 2), 2, 32)):
        K = C
        x = torch.randint(-128, 128, (2, 11, 13, C), generator=gen, dtype=torch.int8)
        wq = torch.randint(-128, 128, (K, C // groups, R, S), generator=gen, dtype=torch.int8)
        b = torch.randint(-128, 128, (K,), generator=gen, dtype=torch.int32)
        if groups == C:
            acc = dw_exact(x, wq[:, 0].permute(1, 2, 0).contiguous(), K, st, pad, dil)
        else:
            acc = F.conv2d(x.permute(0, 3, 1, 2).double(), wq.double(), None, st, pad, dil, groups)
            acc = torch.round(acc).long().permute(0, 2, 3, 1).reshape(-1, K)
        for wb, ib, ob in ((9, 7, -4), (7, 7, 1), (2, 1, 3)):
            info = {"weight_bit": wb, "input_bit": ib, "output_bit": ob, "bias_bit": 2}
            xf = (x.permute(0, 3, 1, 2).double() * 2.0 ** -ib).float().numpy()
            wf = (wq.double() * 2.0 ** -wb).float().numpy()
            bf = (b.double() * 2.0 ** -2).float().numpy()
            f32, y = oracle.int_conv_layer(xf, wf, bf, info, stride=st, padding=pad, dilation=dil, groups=groups)
            want = epilogue_ref(acc, b.long(), wb + ib - ob, False)
            P, Q = y.shape[2:]
            assert np.array_equal(want.view(2, P, Q, K).permute(0, 3, 1, 2).numpy(), y), (R, S, groups)
            assert np.array_equal(dequant_ref(want, ob).view(2, P, Q, K).permute(0, 3, 1, 2).numpy(), f32)


def test_depthwise_rows_cover_the_geometry():
    """Every (G, KS) at every stride and dilation combination, pads 0, 1 and the maximum per dimension, the filter
    shapes, edge images and channel counts the rows are meant to reach."""
    seen = {}
    for inst, g in DW_ROWS:
        assert dw_inst(g["C"], g["R"], g["S"]) == inst, (inst, g)
        assert g["pad"][0] <= (g["R"] - 1) * g["dil"][0] and g["pad"][1] <= (g["S"] - 1) * g["dil"][1]
        seen.setdefault(inst, set()).add((g["st"], g["dil"]))
    assert set(seen) == {(G, KS) for G in (1, 2, 4) for KS in (3, 5, 0)}
    assert all(v == set(itertools.product(STEPS, STEPS)) for v in seen.values())
    gs = [g for _, g in DW_ROWS]
    for dim, k in ((0, "R"), (1, "S")):
        pads = {("max" if g["pad"][dim] == (g[k] - 1) * g["dil"][dim] else g["pad"][dim]) for g in gs if g[k] > 1}
        assert {0, 1, "max"} <= pads
    assert sum(g["pad"][0] != g["pad"][1] for g in gs) > len(gs) // 2
    assert {(1, 7), (7, 1), (2, 6), (4, 3), (1, 1), (7, 7), (2, 2), (4, 4)} <= {(g["R"], g["S"]) for g in gs}
    pq = [out_size(g) for g in gs]
    assert any(g["H"] == 1 for g in gs) and any(g["W"] == 1 for g in gs) and any(g["N"] == 1 for g in gs)
    assert any(p == 1 for p, _ in pq) and any(q == 1 for _, q in pq)
    assert any(g["H"] < (g["R"] - 1) * g["dil"][0] + 1 and g["W"] < (g["S"] - 1) * g["dil"][1] + 1 for g in gs)
    big = [(g, p * q) for g, (p, q) in zip(gs, pq) if g["N"] * p * q > DW_THREADS // dw_inst(g["C"], 1, 1)[0] * DW_PIX_ITERS]
    assert any(g["N"] * n % (1024 // dw_inst(g["C"], 1, 1)[0]) and n % 2 for g, n in big)
    assert {16, 48, 80, 96, 160, 192, 960} <= {g["C"] for g in gs}
    assert any(g["C"] // (16 * dw_inst(g["C"], 1, 1)[0]) >= 3 for g in gs)          # several CTAs along y
    kinds = {"K=1" if g["K"] == 1 else "C-1" if g["K"] == g["C"] - 1 else "C-15" if g["K"] == g["C"] - 15 else
             "16/64" if (g["K"], g["C"]) == (16, 64) else "C" if g["K"] == g["C"] else "other" for g in gs}
    assert {"K=1", "C-1", "C-15", "16/64", "C"} <= kinds
    # K % 16 != 0 inside a CTA of G = 2 and G = 4
    assert {dw_inst(g["C"], 1, 1)[0] for g in gs if g["K"] % 16} >= {1, 2, 4}


def test_grouped_rows_take_the_instantiation_they_name():
    """Each grouped row's name is the host's choice; between them the rows reach every configuration the grouped path
    can select, both tps, resident and streamed weights, the Wb / BK cases and the window walks they are meant to."""
    from common.quantity import _native
    from common.quantity.new_quantity_op import _group_block  # noqa: F401  (the same package the rows use)
    configs, tps, res = set(), set(), set()
    for name, g in GROUPED_ROWS:
        assert grouped_name(g) == name, (name, grouped_name(g), g)
        inst, t, r = grouped_choice(g)
        configs.add((inst[0], inst[1], inst[2], inst[4]))
        tps.add(t), res.add(r)
        Kg = g["K"] // g["G"]
        assert g["C"] % g["G"] == 0 and g["K"] % g["G"] == 0 and g["K"] % g["B"] == 0
        assert g["B"] % Kg == 0 or Kg % g["B"] == 0
    assert configs == GROUPED_CONFIGS and tps == {1, 3} and res == {0, 1}
    plain = [g for n, g in GROUPED_ROWS if n.startswith("gemm")]
    assert {16, 48, 80, 144} <= {_native.group_window(g["C"], g["K"], g["G"], g["B"]) for g in plain}

    def tiles(g):
        P, Q = out_size(g)
        return -(-g["N"] * P * Q // 128), g["K"] // g["B"]
    walks = {n_t for n, g in GROUPED_ROWS for m_t, n_t in [tiles(g)] if m_t * n_t > SMS and SMS % n_t}
    assert {8, 64} <= walks
    wide = [g for n, g in GROUPED_ROWS if n.startswith("im2col") and grouped_choice(g)[0][1] == 128 and
            _native.group_window(g["C"], g["K"], g["G"], g["B"]) in (256, 512) and tiles(g)[1] >= 2]
    assert {256, 512} <= {_native.group_window(g["C"], g["K"], g["G"], g["B"]) for g in wide}
    assert any(g["B"] == 256 and g["K"] // g["G"] == 512 for _, g in GROUPED_ROWS)                   # tpg = 2
    assert any(g["C"] // g["G"] == 2 for _, g in GROUPED_ROWS)
    assert {(1, 3), (3, 1), (1, 7), (5, 3)} <= {(g["R"], g["S"]) for _, g in GROUPED_ROWS}
    assert set(range(1, 9)) <= {s for _, g in GROUPED_ROWS for s in g["st"]}


def test_depthwise_and_grouped_fits_envelope():
    """NewConv2d's routing envelope, one step across each clause of _depthwise_fits and _grouped_fits."""
    from common.quantity.new_quantity_op import _depthwise_fits, _grouped_fits

    def dw(**kw):
        a = dict(k=(3, 3), s=(1, 1), p=(1, 1), d=(1, 1))
        a.update(kw)
        return _depthwise_fits(nn.Conv2d(32, 32, a["k"], a["s"], a["p"], a["d"], groups=32))
    assert dw(k=(7, 3), p=(3, 1)) and not dw(k=(8, 3), p=(3, 1))
    assert dw(k=(3, 7), p=(1, 3)) and not dw(k=(3, 8), p=(1, 3))
    assert dw(s=(2, 1)) and not dw(s=(3, 1)) and dw(s=(1, 2)) and not dw(s=(1, 3))
    assert dw(d=(2, 1)) and not dw(d=(3, 1)) and dw(d=(1, 2)) and not dw(d=(1, 3))
    assert dw(p=(2, 1)) and not dw(p=(3, 1)) and dw(p=(1, 2)) and not dw(p=(1, 3))
    assert dw(p=(4, 1), d=(2, 1)) and not dw(p=(5, 1), d=(2, 1))
    assert not _depthwise_fits(nn.Conv2d(32, 64, 3, 1, 1, groups=32))                  # channel multiplier 2

    def gp(cin, cout, groups, k=3, s=1, p=1):
        return _grouped_fits(nn.Conv2d(cin, cout, k, s, p, groups=groups))
    assert gp(64, 64, 32) and not gp(32, 32, 32)                                       # Cg = 2 / Cg = 1
    assert gp(64, 64, 2) and not gp(48, 48, 2) and not gp(80, 80, 5)                  # C % 32
    assert gp(48, 96, 3, 1, 1, 0) and not gp(40, 80, 5, 1, 1, 0)                      # plain 1 x 1: C % 16
    assert not gp(48, 96, 3, 1, 2, 0) and not gp(48, 96, 3, 1, 1, 1)                  # 1 x 1 off the plain path


def test_every_depthwise_limit_has_an_inside_and_a_beyond_row():
    """Each limit the header documents for pq_conv2d_dw_s8 ('dw limit:') has a row one step inside and one beyond, or
    a test at size; the grid-limit rows sit at the three widths either side of it."""
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "pq_sm100.h")).read()
    documented = [s.strip() for s in re.findall(r"dw limit: ([^;\n]+?)(?:;|\s*\*/|\n)", header)]
    assert len(documented) >= 7, documented
    for lim in documented:
        if lim in DW_SIZE_LIMITS:
            continue
        assert {r[2] == 0 for r in DW_LIMITS if r[0] == lim} == {True, False}, lim
    assert {r[0] for r in DW_LIMITS} <= set(documented)
    grid = {(r[1]["C"], r[2]) for r in DW_LIMITS if r[0] == "C / (16*G) <= 65535"}
    for G in (1, 2, 4):
        ok = [c for c, rc in grid if rc == 0 and dw_inst(c, 3, 3)[0] == G]
        bad = [c for c, rc in grid if rc != 0 and dw_inst(c, 3, 3)[0] == G]
        assert ok == [16 * G * 65535] and len(bad) == 1 and bad[0] // (16 * G) == 65536 + (G < 4), (G, ok, bad)


def _cuobjdump():
    for tool in ("cuobjdump", "cu++filt"):
        if shutil.which(tool) is None and not os.path.exists(os.path.join("/usr/local/cuda/bin", tool)):
            pytest.skip("%s not installed" % tool)
    return [shutil.which(t) or os.path.join("/usr/local/cuda/bin", t) for t in ("cuobjdump", "cu++filt")]


def test_rows_reach_every_instantiation_of_the_library():
    """The dw_conv_s8_kernel instantiations of the built library are exactly the (G, KS) the depthwise rows reach, and
    every gemm_s8_kernel configuration the grouped rows reach is in the library."""
    from common.quantity import _native
    if not os.path.exists(_native.LIB_PATH):
        pytest.skip("library not built")
    objdump, filt = _cuobjdump()
    sym = subprocess.run([objdump, "-symbols", _native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = subprocess.run([filt], input=sym, check=True, capture_output=True, text=True).stdout
    entries = [line for line in names.splitlines() if "STO_ENTRY" in line]
    dws = {kname(line)[1:] for line in entries if "dw_conv_s8_kernel" in line}
    assert dws == {inst for inst, _ in DW_ROWS}
    gemms = {kname(line) for line in entries if "gemm_s8_kernel" in line}
    assert {grouped_choice(g)[0] for _, g in GROUPED_ROWS} <= gemms

"""Windowed average pooling kept int8 in the pipeline: the kernel pq_avgpool_requant_s8 (a new overload of
avgpool_global_kernel, AvgPoolParams), the lazy pooled views of int8_pipeline and the ResNet-50-D of the model zoo.

The kernel is compared byte for byte with Quantity(q_bit) of ATen's F.avg_pool2d on the de-quantised fp32 NCHW tensor,
computed on the device with torch.round (half to even) and a clamp, which share no code with the kernel.  Outputs sit
in sentinel-filled buffers; inputs must be unchanged afterwards; torch.profiler shows which overload each call lands on.
"""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

gpu = pytest.mark.gpu
EINVAL, EUNSUPPORTED = -1, -2
SENTINEL = 0xA5
GUARD = 4096
HERE = os.path.dirname(os.path.abspath(__file__))


def _pipe():
    from common.quantity import int8_pipeline
    return int8_pipeline


# ------------------------------------------------------------------------------------------ CPU: argument rules
META = torch.device("meta")


def _meta_q(shape=(2, 16, 7, 9), s16=False, bit=3):
    from common.quantity import QTensor
    return QTensor(shape, META, s16_bit=bit) if s16 else QTensor(shape, META, q8_bit=bit)


# (positional args, keyword args, becomes a pooled view) on a 2 x 16 x 7 x 9 int8 QTensor
DECLINE_ROWS = [
    ((2,), {}, True), ((3, 2, 1), {}, True), ((3, 2, 1, True, False, 5), {}, True),
    (((2, 3), (1, 2), (1, 1)), {}, True), (([3], [2], [1]), {}, True), ((3, [], 0), {}, True),
    ((), dict(kernel_size=2, stride=2, ceil_mode=True, count_include_pad=False), True),
    ((3,), dict(divisor_override=-4), True), ((3,), dict(divisor_override=2 ** 31 - 1), True),
    ((7, 1), {}, True), ((1,), {}, True),
    ((3,), dict(divisor_override=0), False),                  # torch refuses it
    ((3,), dict(divisor_override=2 ** 31), False),            # beyond int32
    ((3, 2, 2), {}, False),                                   # pad > k / 2: torch refuses it
    ((8,), {}, False),                                        # output too small: torch refuses it
    ((3, 0), {}, False), ((3, 2, -1), {}, False), ((2.0,), {}, False), (((2, 2, 2),), {}, False),
    ((3, 2, 1, False, True, None, "surplus"), {}, False), ((), dict(kernel_size=3, bogus=1), False),
]


@pytest.mark.parametrize("row", range(len(DECLINE_ROWS)))
def test_decline_rules(row):
    """Which F.avg_pool2d argument sets, positional and keyword, become a pooled view (meta QTensors: host logic)."""
    args, kwargs, taken = DECLINE_ROWS[row]
    v = _pipe()._avgpool(_meta_q(), *args, **kwargs)
    assert (v is not None and v._lazy_pool is not None) == taken
    if taken:
        want = F.avg_pool2d(torch.empty(2, 16, 7, 9, device=META), *args, **kwargs).shape
        assert v.shape == want and v.exact_bit() is None and not v.has_q8()


@pytest.mark.parametrize("kw", [dict(kernel_size=3, stride=2, padding=1), dict(kernel_size=(2, 3), ceil_mode=True),
                                dict(kernel_size=2, stride=2, ceil_mode=True, count_include_pad=False),
                                dict(kernel_size=3, divisor_override=7)])
def test_decline_rules_module_form(kw):
    """nn.AvgPool2d passes every argument positionally; the same window results as from the keyword call."""
    m = nn.AvgPool2d(**kw)
    args = (m.kernel_size, m.stride, m.padding, m.ceil_mode, m.count_include_pad, m.divisor_override)
    a, b = _pipe()._avgpool(_meta_q(), *args), _pipe()._avgpool(_meta_q(), **kw)
    assert a._lazy_pool.window == b._lazy_pool.window and a.shape == b.shape


def test_decline_rules_source_and_limits():
    """Sources and sizes the kernel does not take are left to ATen; the whole-plane pool keeps its own path."""
    from common.quantity import QTensor, _native
    p = _pipe()
    assert p._avgpool(_meta_q((16, 7, 9)), 3) is None                                   # 3-D
    assert p._avgpool(_meta_q((2, 12, 7, 9)), 3) is None                                # C % 8
    assert p._avgpool(_meta_q((2, 24, 7, 9)), 3) is not None
    assert p._avgpool(_meta_q(bit=32), 3) is None and p._avgpool(_meta_q(bit=-32), 3) is None
    assert p._avgpool(_meta_q(bit=31), 3) is not None and p._avgpool(_meta_q(bit=-31), 3) is not None
    assert p._avgpool(QTensor((2, 16, 7, 9), META), 3) is None                          # no payload
    # exactness: kh*kw*(32768 | 128) < 2^24
    big = (2, 16, 520, 520)
    assert p._avgpool(_meta_q(big, s16=True), (7, 73)) is not None
    assert p._avgpool(_meta_q(big, s16=True), (8, 64)) is None
    assert p._avgpool(_meta_q(big, s16=False), (8, 64)) is not None
    assert p._avgpool(_meta_q((1, 16, 1, 131072)), (1, 131071)) is not None
    assert p._avgpool(_meta_q((1, 16, 1, 131072)), (1, 131072)) is None
    # N*P*Q <= 2^31 - 1
    assert p._avgpool(_meta_q((2 ** 31 - 1, 16, 1, 3)), (1, 2), (1, 2)) is not None
    assert p._avgpool(_meta_q((2, 16, 1, 2 ** 30)), 1) is None
    # lazy concatenation, nearest view and pooled view as sources
    a, b = _meta_q(), _meta_q()
    cat = p._concat([a, b], 1)
    assert cat is not None and p._avgpool(cat, 3) is None
    up = p._upsample(a, (), {"scale_factor": 2})
    assert up is not None and p._avgpool(up, 3) is None
    v = p._avgpool(a, 3, 1, 1)
    assert p._avgpool(v, 3) is None
    # a pooled view is not an exact payload: Concat, NewAdd, max-pool and upsample take the fp32 path
    assert p._concat([v, v], 1) is None and p._upsample(v, (), {"scale_factor": 2}) is None
    assert p._maxpool(v, 3, 1, 1) is None
    import types
    assert p.add_forward(types.SimpleNamespace(output_bit=3), v, v) is None
    # the pooled view carries a later ReLU
    r = v.with_relu()
    assert r._lazy_pool is v._lazy_pool and r.relu_pending
    # the whole-plane pool keeps the global kernel's path, whatever the other arguments
    calls = []
    orig = _native.avgpool_global_nhwc
    _native.avgpool_global_nhwc = lambda x, bit, relu=False: calls.append((bit, relu)) or "global"
    try:
        q = QTensor((2, 16, 7, 9), META, q8=torch.empty((2, 7, 9, 16), dtype=torch.int8, device=META), q8_bit=3)
        assert p._avgpool(q, (7, 9)) == "global" and p._avgpool(q, kernel_size=[7, 9], stride=1) == "global"
        assert p._avgpool(q, (7, 9), padding=1) is None and p._avgpool(q, (7, 9), divisor_override=3) is None
        assert calls == [(3, False), (3, False)]
    finally:
        _native.avgpool_global_nhwc = orig


def test_output_size_matches_aten():
    """The binding's P, Q equal F.avg_pool2d's over odd sizes, where ceil_mode adds a clipped last window."""
    from common.quantity import _native
    n = 0
    for H in (1, 2, 3, 5, 7, 8, 13):
        for W in (1, 4, 6, 9, 11):
            for kh, kw in ((1, 2), (2, 3), (3, 2), (4, 1), (5, 3), (7, 2)):
                for s in (1, 2, 3):
                    for p in range(kh // 2 + 1):
                        for ceil in (False, True):
                            win = (kh, kw, s, s + 1, p, kw // 2, int(ceil), 1, 0)
                            try:
                                want = F.avg_pool2d(torch.zeros(1, 1, H, W), (kh, kw), (s, s + 1), (p, kw // 2), ceil)
                            except RuntimeError:
                                with pytest.raises(RuntimeError):
                                    _native.avgpool_out_size((H, W), win)
                                continue
                            assert _native.avgpool_out_size((H, W), win) == tuple(want.shape[2:])
                            n += 1
    assert n > 1000


def _trace(build, hw):
    import tools._config as tc
    from common.quantity import merge_bn
    from tools.pytorch_quantizer import Quantity
    cfg = tc.load_tool_config(os.path.join(os.path.dirname(HERE), "pytorch-quantity_b200", "tools", "configs.yml"))
    st = cfg["SETTINGS"]
    q = object.__new__(Quantity)
    q._cared_op_type, q._all_op_type = st["CARE_OP_TYPE"], st["ALL_OP_TYPE"]
    q._allow_same_tid_op_type, q._merge_op_type = st["ALLOW_SAME_TID_OP_TYPE"], st["MERGE_OP_YTPE"]
    q.verbose, q.rank, q.cuda_device = False, 0, torch.device("cpu")
    torch.manual_seed(0)
    return q, q.build_net_structure(merge_bn(build().eval(), "cpu"), (1, 3, hw, hw))


def test_resnet50d_traces_avg_down_to_the_eltwise(capsys):
    """The tracer splices each avg-down pool out (AvgPool2d is in ALL_OP_TYPE, not cared): the shortcut convolution of
    every stride-2 unit reads the preceding Eltwise, and the merge groups are those of a ResNet-50 whose first unit of
    each later stage pairs its last convolution with that shortcut."""
    from model.resnet import resnet50d_fabu
    q, net = _trace(lambda: resnet50d_fabu(in_hw=64), 64)
    kinds = [i["type"] for i in net.values()]
    assert kinds.count("Conv2d") == 3 + 16 * 3 + 4 and kinds.count("Eltwise") == 16 and kinds.count("Linear") == 1
    assert set(kinds) == {"Conv2d", "Eltwise", "Linear"}
    adds = [(n, i["inputs"]) for n, i in net.items() if i["type"] == "Eltwise"]
    # the first unit of stages 2..4: Eltwise(last conv of the unit, shortcut conv); the shortcut reads the previous add
    firsts = [adds[3], adds[7], adds[13]]
    for k, (n, (left, short)) in enumerate(firsts):
        prev = adds[(3, 7, 13)[k] - 1][0]
        assert net[short]["inputs"] == [prev], (n, short, net[short]["inputs"])
        assert net[left]["inputs"] != [prev]
    assert [n for n, _ in adds[:4]] == ["Eltwise_14", "Eltwise_21", "Eltwise_28", "Eltwise_37"]
    assert adds[3][1] == ["Conv2d_34", "Conv2d_36"] and net["Conv2d_36"]["inputs"] == ["Eltwise_28"]
    groups = q.get_merge_groups(net)
    assert len(groups) == 16 and groups[-1] == ["Conv2d_12", "Conv2d_13"]
    assert ["Conv2d_34", "Conv2d_36"] in groups and ["Conv2d_64", "Conv2d_66"] in groups
    assert ["Conv2d_108", "Conv2d_110"] in groups
    assert net["Conv2d_3"]["inputs"] == ["Conv2d_1"] and net["Conv2d_5"]["inputs"] == ["Conv2d_3"]   # the deep stem


# ------------------------------------------------------------------------------------------ CPU: limits in the header
AT_SIZE = 2 ** 31 - 1
# (limit as the header words it, (N, H, W, C, c_out_pad, kh, kw, ph, pw, is16, bit, q_bit), expected return code); the
# row at size runs in test_avgpool_pixel_limit_inside_at_size
LIMITS = [
    ("kh*kw*(32768 | 128) < 2^24", (1, 7, 73, 8, 16, 7, 73, 0, 0, True, 3, 3), 0),
    ("kh*kw*(32768 | 128) < 2^24", (1, 8, 64, 8, 16, 8, 64, 0, 0, True, 3, 3), EUNSUPPORTED),
    ("kh*kw*(32768 | 128) < 2^24", (1, 1, 131071, 8, 16, 1, 131071, 0, 0, False, 3, 3), 0),
    ("kh*kw*(32768 | 128) < 2^24", (1, 1, 131072, 8, 16, 1, 131072, 0, 0, False, 3, 3), EUNSUPPORTED),
    # kh*kw*32768 = 2^75 does not fit in 64 bits: the check must not wrap
    ("kh*kw*(32768 | 128) < 2^24", (1, 2 ** 30, 2 ** 30, 8, 16, 2 ** 30, 2 ** 30, 0, 0, True, 3, 3), EUNSUPPORTED),
    ("2*pad <= k", (1, 5, 5, 8, 16, 3, 2, 1, 1, False, 3, 3), 0),
    ("2*pad <= k", (1, 5, 5, 8, 16, 3, 3, 2, 1, False, 3, 3), EUNSUPPORTED),
    ("2*pad <= k", (1, 5, 5, 8, 16, 3, 3, 1, 2, False, 3, 3), EUNSUPPORTED),
    ("C % 8 == 0", (1, 5, 5, 8, 16, 3, 3, 1, 1, False, 3, 3), 0),
    ("C % 8 == 0", (1, 5, 5, 12, 16, 3, 3, 1, 1, False, 3, 3), EUNSUPPORTED),
    ("C % 8 == 0", (1, 5, 5, 4, 16, 3, 3, 1, 1, False, 3, 3), EUNSUPPORTED),
    ("c_out_pad % 16 == 0", (1, 5, 5, 24, 32, 3, 3, 1, 1, False, 3, 3), 0),
    ("c_out_pad % 16 == 0", (1, 5, 5, 24, 24, 3, 3, 1, 1, False, 3, 3), EUNSUPPORTED),
    ("c_out_pad % 16 == 0", (1, 5, 5, 24, 40, 3, 3, 1, 1, False, 3, 3), EUNSUPPORTED),
    ("N*P*Q <= 2^31 - 1", (AT_SIZE, 1, 1, 8, 16, 1, 1, 0, 0, False, 3, 3), 0),
    ("N*P*Q <= 2^31 - 1", (2, 1, 2 ** 30, 8, 16, 1, 1, 0, 0, False, 3, 3), EUNSUPPORTED),
    ("|bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, True, 31, 3), 0),
    ("|bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, True, -31, 3), 0),
    ("|bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, True, 32, 3), EUNSUPPORTED),
    ("|bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, True, -32, 3), EUNSUPPORTED),
    ("|q_bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, False, 3, 31), 0),
    ("|q_bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, False, 3, -31), 0),
    ("|q_bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, False, 3, 32), EUNSUPPORTED),
    ("|q_bit| <= 31", (1, 5, 5, 8, 16, 3, 3, 1, 1, False, 3, -32), EUNSUPPORTED),
]


def _header():
    return open(os.path.join(os.path.dirname(HERE), "include", "pq_sm100.h")).read()


def test_every_avgpool_limit_has_an_inside_and_a_beyond_row():
    documented = [s.strip() for s in re.findall(r"avgpool limit: ([^;\n]+?)(?:;|\s*\*/|\n)", _header())]
    assert len(documented) == 7 and {r[0] for r in LIMITS} == set(documented), documented
    for lim in documented:
        assert {r[2] == 0 for r in LIMITS if r[0] == lim} == {True, False}, lim


# ------------------------------------------------------------------------------------------ GPU helpers
def _lib():
    from common.quantity import _native
    return _native.lib()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class Guarded:
    """A device buffer of `shape` / `dtype` in the middle of sentinel bytes."""

    def __init__(self, shape, dtype=torch.int8):
        n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
        self.buf = torch.full((GUARD + n + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.t = self.buf[GUARD:GUARD + n].view(dtype).view(shape)

    def ptr(self):
        return self.t.data_ptr()

    def guards_intact(self):
        return bool((self.buf[:GUARD] == SENTINEL).all()) and bool((self.buf[-GUARD:] == SENTINEL).all())

    def untouched(self):
        return bool((self.buf == SENTINEL).all())


def launched(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_FRESH_ENV = "PQ_AVGPOOL_FRESH"
_STATE = {}


def profiler_records():
    """Whether torch.profiler records CUDA kernels in this process.  After some sequences of earlier tests in one pytest
    process it records none at all; the tests of this file that check kernel names then run once more in a fresh
    process, which must pass."""
    if "recorded" not in _STATE:
        _STATE["recorded"] = bool(launched(lambda: torch.ones(16, device="cuda").add_(1)))
        if not _STATE["recorded"]:
            assert not os.environ.get(_FRESH_ENV), "torch.profiler records no CUDA kernels in a fresh process"
            r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-p", "no:cacheprovider",
                                "-m", "gpu", "-k", "landing or resnet50d_end_to_end"], cwd=os.path.dirname(HERE),
                               env=dict(os.environ, **{_FRESH_ENV: "1"}), capture_output=True, text=True, timeout=3600)
            _STATE["fresh"] = (r.returncode, r.stdout[-3000:])
    return _STATE["recorded"]


def fresh_run_passed():
    rc, out = _STATE["fresh"]
    assert rc == 0, "the fresh-process run of this file, which makes the kernel-name checks, failed:\n" + out


def _payload(shape, is16, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lo, hi = (-32768, 32767) if is16 else (-128, 127)
    v = torch.randint(lo, hi + 1, shape, dtype=torch.int32, device="cuda", generator=g)
    v.view(-1)[:4] = torch.tensor([lo, hi, 0, -1], dtype=torch.int32)
    return v.to(torch.int16 if is16 else torch.int8).contiguous()


def reference(x, bit, relu, win, q_bit, c_pad, out_relu=False):
    """Quantity(q_bit)(F.avg_pool2d(de-quantised x)) by ATen on the device, int8 NHWC [N][P][Q][c_pad]."""
    kh, kw, sh, sw, ph, pw, ceil, cip, div = win
    v = x.float() * 2.0 ** -bit                        # exact: a payload times a power of two in the fp32 range
    if relu:
        v = torch.relu(v)
    y = F.avg_pool2d(v.permute(0, 3, 1, 2).contiguous(), (kh, kw), (sh, sw), (ph, pw), bool(ceil), bool(cip),
                     div or None)
    if out_relu:
        y = torch.relu(y)
    q = torch.clamp(torch.round(y * 2.0 ** q_bit), -128, 127).to(torch.int8).permute(0, 2, 3, 1)
    out = torch.zeros(q.shape[:3] + (c_pad,), dtype=torch.int8, device=x.device)
    out[..., :q.shape[3]] = q
    return out


def run_kernel(x, bit, relu, win, q_bit, c_pad, out_relu=False, out=None):
    from common.quantity import _native
    N, H, W, C = x.shape
    P, Q = _native.avgpool_out_size((H, W), win)
    g = out or Guarded((N, P, Q, c_pad))
    rc = _lib().pq_avgpool_requant_s8(x.data_ptr(), int(x.dtype == torch.int16), bit, int(relu) | 2 * int(out_relu),
                                      N, H, W, C, ctypes.byref(_native.PoolDesc(*win)), q_bit, c_pad, g.ptr(), _stream())
    return rc, g


# ------------------------------------------------------------------------------------------ GPU: kernel against ATen
def _rows():
    """(N, H, W, C, c_pad, (kh, kw, sh, sw, ph, pw), is16, relu, bit, q_bit): every kh != kw in 1..7, strides 1-3 and
    pads 0..k/2 per dimension, C in {8, 16, 24, 48, 256} with c_pad = C (where it is a multiple of 16) and padded, int8
    and int16 with and without the ReLU on load, bits across their range.  Each row runs every ceil_mode,
    count_include_pad and divisor (None, positive, negative)."""
    rows, i = [], 0
    cs = (8, 16, 24, 48, 256)
    bits = (-31, -9, -2, 0, 3, 7, 15, 31)
    for kh in range(1, 8):
        for kw in range(1, 8):
            if kh == kw:
                continue
            C = cs[i % 5]
            c_pad = C if C % 16 == 0 and i % 2 else (C + 15) // 16 * 16 + 16 * (i % 3 == 0)
            sh, sw = 1 + i % 3, 1 + (i // 3) % 3
            ph, pw = i % (kh // 2 + 1), (i // 2) % (kw // 2 + 1)
            H, W = kh + 3 + i % 4, kw + 2 + (i * 7) % 9                      # odd and even sizes
            is16, relu = bool(i % 2), bool((i // 2) % 2)
            bit = bits[i % 8]
            q_bit = max(-31, min(31, bit + (-3, -1, 0, 1, 2, 5)[i % 6] - (8 if is16 else 0)))
            q_bit = {5: 31, 6: -31}.get(i % 11, q_bit)                        # both ends of the q_bit range
            rows.append((1 + i % 3, H, W, C, c_pad, (kh, kw, sh, sw, ph, pw), is16, relu, bit, q_bit))
            i += 1
    return rows


ROWS = _rows()
GRID_ROW = (2, 11, 80, 256, 256, (3, 2, 1, 2, 1, 1), True, True, 4, -3)        # Q * c_pad / 8 = 1280 > 256 threads
ROWS.append(GRID_ROW)


@gpu
@pytest.mark.parametrize("row", range(len(ROWS)))
def test_kernel_against_aten(row):
    N, H, W, C, c_pad, geo, is16, relu, bit, q_bit = ROWS[row]
    x = _payload((N, H, W, C), is16, row)
    x0 = x.clone()
    for ceil in (False, True):
        for cip in (False, True):
            for div in (0, 3, -5):
                win = geo + (int(ceil), int(cip), div)
                try:
                    want = reference(x, bit, relu, win, q_bit, c_pad)
                except RuntimeError:
                    continue                            # ceil_mode may leave no legal output for some geometries
                for out_relu in (False, True) if div == 0 else (False,):
                    w = reference(x, bit, relu, win, q_bit, c_pad, out_relu) if out_relu else want
                    rc, g = run_kernel(x, bit, relu, win, q_bit, c_pad, out_relu)
                    torch.cuda.synchronize()
                    assert rc == 0, (win, rc)
                    assert g.guards_intact(), win
                    assert torch.equal(g.t, w), (win, out_relu, (g.t != w).nonzero()[:5].tolist())
    assert torch.equal(x, x0)


def test_rows_cover_the_sweep():
    pairs = {r[5][:2] for r in ROWS}
    assert {(a, b) for a in range(1, 8) for b in range(1, 8) if a != b} <= pairs
    assert {r[5][2] for r in ROWS} == {1, 2, 3} and {r[5][3] for r in ROWS} == {1, 2, 3}
    assert {r[3] for r in ROWS} == {8, 16, 24, 48, 256}
    assert any(r[3] == r[4] for r in ROWS) and any(r[4] > r[3] for r in ROWS)
    assert {(r[6], r[7]) for r in ROWS} == {(a, b) for a in (False, True) for b in (False, True)}
    assert {-31, 31} <= {r[8] for r in ROWS} and {-31, 31} <= {r[9] for r in ROWS}
    N, H, W, C, c_pad, geo = GRID_ROW[:6]
    Q = (W + 2 * geo[5] - geo[1]) // geo[3] + 1
    assert Q * c_pad // 8 > 256                         # the threads of a block go round the row loop more than once


@gpu
def test_kernel_rounding_and_ties():
    """Crafted rows.  Ties: 2 x 2 windows whose only nonzero tap is m, divisor 4 and q_bit = bit + 1, so the scaled
    value is m / 2: every odd m is an exact .5 tie (both signs, rounded to even).  Rounding: a 1 x 511 int16 window near
    the payload maximum divided by 511 and by the override 3, where the fp32 quotient is rounded."""
    N, H, W, C = 2, 6, 8, 256
    x = torch.zeros((N, H, W, C), dtype=torch.int8, device="cuda")
    x[:, ::2, ::2, :] = (torch.arange(C, device="cuda") - 128).to(torch.int8)
    for win in ((2, 2, 2, 2, 0, 0, 0, 1, 0), (2, 2, 2, 2, 0, 0, 1, 0, 4)):
        rc, g = run_kernel(x, 5, False, win, 6, C)
        torch.cuda.synchronize()
        want = reference(x, 5, False, win, 6, C)
        assert rc == 0 and g.guards_intact() and torch.equal(g.t, want)
        ties = torch.arange(C, device="cuda") - 128
        assert torch.equal(g.t[0, 0, 0].long(), torch.round(ties / 2.0).long())       # half to even
    x = _payload((2, 3, 600, 16), True, 5)
    g = torch.Generator(device="cuda").manual_seed(6)
    x[1] = (32767 - torch.randint(0, 64, (3, 600, 16), generator=g, device="cuda")).to(torch.int16)
    for div in (0, 3, -3):
        win = (1, 511, 1, 89, 0, 0, 0, 1, div)
        for bit, q_bit in ((0, -8), (3, -5), (-2, -10)):
            rc, g = run_kernel(x, bit, False, win, q_bit if div == 0 else q_bit - 8, 16)
            torch.cuda.synchronize()
            want = reference(x, bit, False, win, q_bit if div == 0 else q_bit - 8, 16)
            assert rc == 0 and g.guards_intact() and torch.equal(g.t, want), (div, bit)
            assert len(torch.unique(want)) > 1


# ------------------------------------------------------------------------------------------ GPU: limits
@gpu
@pytest.mark.parametrize("row", [r for r in LIMITS if r[1][0] != AT_SIZE],
                         ids=lambda r: "%s-%d" % (re.sub(r"\W", "", r[0]), r[2]))
def test_avgpool_limit_one_step_inside_and_beyond(row):
    """A row inside a limit runs and writes its output; a row beyond is PQ_EUNSUPPORTED and writes nothing."""
    from common.quantity import _native
    _, (N, H, W, C, c_pad, kh, kw, ph, pw, is16, bit, q_bit), want = row
    win = (kh, kw, 1, 1, ph, pw, 0, 1, 0)
    small = N * H * W * C <= 1 << 24
    x = _payload((N, H, W, C) if small else (1, 1, 1, 16), is16, 3)
    try:
        P, Q = _native.avgpool_out_size((H, W), win)
    except RuntimeError:
        P = Q = 1                                       # arguments torch refuses: the library refuses them first
    g = Guarded((N, P, Q, c_pad) if small else (1, 1, 1, 16))
    rc = _lib().pq_avgpool_requant_s8(x.data_ptr(), int(is16), bit, 0, N, H, W, C, ctypes.byref(_native.PoolDesc(*win)), q_bit,
                                      c_pad, g.ptr(), _stream())
    torch.cuda.synchronize()
    assert rc == want
    if want == 0:
        assert g.guards_intact() and torch.equal(g.t, reference(x, bit, False, win, q_bit, c_pad))
    else:
        assert g.untouched()


@gpu
def test_avgpool_pixel_limit_inside_at_size():
    """N*P*Q = 2^31 - 1 (a prime: 2^31 - 1 images of one pixel) runs; the output is checked at both ends and the
    sentinels after it."""
    n = AT_SIZE
    need = n * (8 + 16) + (1 << 30)
    torch.cuda.empty_cache()                           # earlier at-size tests leave blocks in the cache
    if torch.cuda.mem_get_info()[0] < need:
        pytest.skip("needs %d GB of free device memory" % (need >> 30))
    from common.quantity import _native
    x = torch.full((n, 1, 1, 8), 5, dtype=torch.int8, device="cuda")
    x[-1] = -7
    g = Guarded((n, 1, 1, 16))
    assert _lib().pq_avgpool_requant_s8(x.data_ptr(), 0, 3, 0, n, 1, 1, 8, ctypes.byref(_native.PoolDesc(1, 1, 1, 1, 0, 0, 0, 1, 0)),
                                        4, 16, g.ptr(), _stream()) == 0
    torch.cuda.synchronize()
    assert g.guards_intact()
    assert bool((g.t[:1 << 20, ..., :8] == 10).all()) and bool((g.t[-(1 << 20):-1, ..., :8] == 10).all())
    assert bool((g.t[-1, ..., :8] == -14).all()) and bool((g.t[-1, ..., 8:] == 0).all())
    assert bool((g.t[:1 << 20, ..., 8:] == 0).all())


@gpu
def test_avgpool_long_row_at_size():
    """One output row of more than 2^31 (column, 8-channel group) pairs: Q = 2^23 + 1 columns of c_out_pad = 2048
    channels (2^31 + 256 pairs, 16 GB) from an 8-channel 1 x 1 pool.  Every pixel is written: the requantised input in
    channels 0..7, zeros after it, sentinels intact."""
    Q = 2 ** 23 + 1
    need = Q * (8 + 2048) + (1 << 30)
    torch.cuda.empty_cache()                           # earlier at-size tests leave blocks in the cache
    if torch.cuda.mem_get_info()[0] < need:
        pytest.skip("needs %d GB of free device memory" % (need >> 30))
    from common.quantity import _native
    g0 = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randint(-63, 64, (1, 1, Q, 8), generator=g0, device="cuda", dtype=torch.int32).to(torch.int8)
    g = Guarded((1, 1, Q, 2048))
    assert _lib().pq_avgpool_requant_s8(x.data_ptr(), 0, 3, 0, 1, 1, Q, 8,
                                        ctypes.byref(_native.PoolDesc(1, 1, 1, 1, 0, 0, 0, 1, 0)), 4, 2048, g.ptr(),
                                        _stream()) == 0
    torch.cuda.synchronize()
    assert g.guards_intact()
    assert torch.equal(g.t[..., :8], (x.to(torch.int16) * 2).to(torch.int8))          # bit 3 -> 4: exactly 2x
    assert int(torch.count_nonzero(g.t[..., 8:])) == 0


@gpu
def test_avgpool_window_end_past_int_max_at_size():
    """W = 2^31 - 1 with a 1 x 3 window, right pad 1 and stride 2^30 - 1: the last window ends at W + 1 = 2^31 and is
    clipped to W.  Each of the three windows (left edge, interior, right edge) equals ATen's pool of a small slice
    holding the same taps and the same edge, for both count_include_pad."""
    W, s = 2 ** 31 - 1, 2 ** 30 - 1
    need = W * 8 + (1 << 30)
    torch.cuda.empty_cache()                           # earlier at-size tests leave blocks in the cache
    if torch.cuda.mem_get_info()[0] < need:
        pytest.skip("needs %d GB of free device memory" % (need >> 30))
    from common.quantity import _native
    x = torch.zeros((1, 1, W, 8), dtype=torch.int8, device="cuda")
    g0 = torch.Generator(device="cuda").manual_seed(12)
    for lo in (0, s - 1, W - 3):
        x[:, :, lo:lo + 3] = torch.randint(-128, 128, (1, 1, 3, 8), generator=g0, device="cuda",
                                           dtype=torch.int32).to(torch.int8)
    for cip in (0, 1):
        win = (1, 3, 1, s, 0, 1, 0, cip, 0)
        assert _native.avgpool_out_size((1, W), win) == (1, 3)
        g = Guarded((1, 1, 3, 16))
        assert _lib().pq_avgpool_requant_s8(x.data_ptr(), 0, 3, 0, 1, 1, W, 8, ctypes.byref(_native.PoolDesc(*win)),
                                            5, 16, g.ptr(), _stream()) == 0
        torch.cuda.synchronize()
        assert g.guards_intact()
        small = (1, 3, 1, 1, 0, 1, 0, cip, 0)
        left = reference(x[:, :, :2].contiguous(), 3, False, small, 5, 16)[:, :, 0]
        inner = reference(x[:, :, s - 1:s + 2].contiguous(), 3, False, (1, 3, 1, 1, 0, 0, 0, cip, 0), 5, 16)[:, :, 0]
        right = reference(x[:, :, W - 2:].contiguous(), 3, False, small, 5, 16)[:, :, 1]
        assert torch.equal(g.t[:, :, 0], left) and torch.equal(g.t[:, :, 1], inner), cip
        assert torch.equal(g.t[:, :, 2], right), (cip, g.t[:, :, 2], right)


@gpu
def test_avgpool_invalid_arguments():
    """Arguments torch itself refuses, and malformed calls, are PQ_EINVAL and write nothing."""
    from common.quantity import _native
    x = _payload((1, 5, 5, 16), False, 1)
    g = Guarded((1, 5, 5, 16))
    ok = (3, 3, 1, 1, 1, 1, 0, 1, 0)
    call = lambda win, C=16, c_pad=16, relu=0, ptr=x.data_ptr(), desc=True: _lib().pq_avgpool_requant_s8(
        ptr, 0, 3, relu, 1, 5, 5, C, ctypes.byref(_native.PoolDesc(*win)) if desc else None, 3, c_pad, g.ptr(), _stream())
    for win in ((0, 3, 1, 1, 0, 0, 0, 1, 0), (3, 3, 0, 1, 0, 0, 0, 1, 0), (3, 3, 1, 1, -1, 0, 0, 1, 0),
                (8, 3, 1, 1, 0, 0, 0, 1, 0)):
        assert call(win) == EINVAL, win
    assert call(ok, c_pad=0) == EINVAL and call(ok, relu=4) == EINVAL and call(ok, ptr=None) == EINVAL
    assert call(ok, desc=False) == EINVAL and call(ok, C=0) == EINVAL
    torch.cuda.synchronize()
    assert g.untouched()
    assert call(ok) == 0


@gpu
def test_landing():
    """pq_avgpool_requant_s8 runs the AvgPoolParams overload of avgpool_global_kernel (int8 and int16); the whole-plane
    entry point still runs the original overload."""
    from common.quantity import _native
    for is16 in (False, True):
        x = _payload((2, 9, 9, 32), is16, 7)
        win = (2, 2, 2, 2, 0, 0, 1, 0, 0)
        if profiler_records():
            g = Guarded((2, 5, 5, 32))                    # (its fill is not part of the profiled launch)
            names = launched(lambda: run_kernel(x, 2, True, win, 1, 32, out=g))
            assert len(names) == 1 and "avgpool_global_kernel" in names[0] and "AvgPoolParams" in names[0], names
            assert ("true" if is16 else "false") in names[0] or ("(bool)1" if is16 else "(bool)0") in names[0]
            names = launched(lambda: _native.avgpool_global_nhwc(x, 2))
            assert len(names) == 1 and "avgpool_global_kernel" in names[0] and "AvgPoolParams" not in names[0], names
        else:
            fresh_run_passed()


# ------------------------------------------------------------------------------------------ GPU: pipeline
INFO = {"weight_bit": 7, "input_bit": 4, "output_bit": 3, "bias_bit": 4}


def _qconv(cin, cout, k, seed, groups=1, info=INFO):
    from common.quantity import NewConv2d
    torch.manual_seed(seed)
    conv = nn.Conv2d(cin, cout, k, padding=k // 2, groups=groups)
    return NewConv2d(conv.cuda(), dict(info)).cuda().eval()


def _sources(x, C):
    """(name, QTensor source, its fp32-boundary value): a conv's int8 payload, with a ReLU pending, and a NewAdd's
    int16 sum, with and without the ReLU after it."""
    from common.quantity import NewAdd
    c1, c2 = _qconv(16, C, 3, 1), _qconv(16, C, 1, 2)
    add = NewAdd().cuda()
    add.output_bit = 2
    out = []
    for pipe in (True, False):
        for m in (c1, c2, add):
            m.int8_pipeline = pipe
        a, b = c1(x), c2(x)
        s = add(a, b)
        out.append({"conv": a, "conv relu": F.relu(a), "add": s, "add relu": F.relu(add(c1(x), c2(x)))})
    return [(k, out[0][k], out[1][k]) for k in out[0]]


POOL_ARGS = [((2, 2), dict(ceil_mode=True, count_include_pad=False)), ((3, 2, 1), {}),
             ((3,), dict(stride=1, padding=1, count_include_pad=False)), (((2, 3), (1, 2), (1, 1), True), {}),
             ((2,), dict(divisor_override=-3))]


@gpu
@pytest.mark.parametrize("pa", range(len(POOL_ARGS)))
def test_pipeline_pool_equals_fp32_boundary(pa):
    """A pool of each source, with a ReLU before or after, consumed by a 1x1, 3x3, depthwise and grouped NewConv2d, is
    torch.equal to the fp32-boundary model, and each consumer reads it through pq_avgpool_requant_s8."""
    from common.quantity import QTensor, _native
    args, kw = POOL_ARGS[pa]
    C = 32
    x = torch.randn(2, 16, 11, 9, generator=torch.Generator().manual_seed(pa)).cuda()
    cons = {"1x1": _qconv(C, 16, 1, 5, info=dict(INFO, input_bit=2)), "3x3": _qconv(C, 24, 3, 6),
            "dw": _qconv(C, C, 3, 7, groups=C, info=dict(INFO, input_bit=5)), "grouped": _qconv(C, 64, 3, 8, groups=2, info=dict(INFO, input_bit=1))}
    assert cons["dw"]._depthwise and cons["grouped"]._group_block
    with torch.no_grad():
        for name, q, ref in _sources(x, C):
            for after in (False, True):
                v = F.avg_pool2d(q, *args, **kw)
                want = F.avg_pool2d(ref, *args, **kw)
                if after:
                    v, want = F.relu(v), F.relu(want)
                assert isinstance(v, QTensor) and v._lazy_pool is not None, name
                assert torch.equal(v.dequantize(), want), name
                for cname, m in cons.items():
                    m.int8_pipeline = True
                    n0 = _native.LAUNCHES.get("avgpool_requant", 0)
                    got = m(v).dequantize()
                    assert _native.LAUNCHES.get("avgpool_requant", 0) == n0 + 1, (name, cname)
                    m.int8_pipeline = False
                    assert torch.equal(got, m(want)), (name, after, cname)


@gpu
def test_pipeline_declined_consumers_and_arguments():
    """Every other consumer of a pooled view, and every declined argument set, gives ATen's result on the
    de-quantised tensor: torch.equal to the fp32-boundary model."""
    from common.quantity import NewAdd, QTensor, _native
    C = 32
    x = torch.randn(2, 16, 12, 10, generator=torch.Generator().manual_seed(3)).cuda()
    add = NewAdd().cuda()
    add.output_bit = 1
    with torch.no_grad():
        for name, q, ref in _sources(x, C):
            v, w = F.avg_pool2d(q, 3, 2, 1), F.avg_pool2d(ref, 3, 2, 1)
            add.int8_pipeline = True
            s = add(v, v)
            add.int8_pipeline = False
            checks = {
                "add": (s, add(w, w)),
                "cat": (torch.cat([v, F.relu(v)], 1), torch.cat([w, F.relu(w)], 1)),
                "maxpool": (F.max_pool2d(v, 2), F.max_pool2d(w, 2)),
                "pool of pool": (F.avg_pool2d(v, 2, 1), F.avg_pool2d(w, 2, 1)),
                "global pool": (F.avg_pool2d(v, v.shape[2:]), F.avg_pool2d(w, w.shape[2:])),
                "view": (v.reshape(2, -1), w.reshape(2, -1)),
                "upsample": (F.interpolate(v, scale_factor=2), F.interpolate(w, scale_factor=2)),
                "user code": (v * 3 + 1, w * 3 + 1),
            }
            for k, (got, want) in checks.items():
                got = got.dequantize() if isinstance(got, QTensor) else got
                assert torch.equal(got, want), (name, k)
            # consumers outside the kernel's limits (q_bit beyond 31, channel padding off the 16 grid) are not served
            lp = v._lazy_pool
            assert lp.supported(31, 32) and not lp.supported(32, 32) and not lp.supported(-32, 32)
            assert not lp.supported(4, 24) and not lp.supported(4, 16)
            assert _native.avgpool_requant_s8(*_pipe()._operand(q), lp.window, 32, 32) is None
            # argument sets the pipeline leaves to ATen
            for args, kw in (((3,), dict(divisor_override=2 ** 31)), ((2.0,), {})):
                try:
                    want = F.avg_pool2d(ref, *args, **kw)
                except (RuntimeError, TypeError) as e:
                    with pytest.raises(type(e)):
                        F.avg_pool2d(q, *args, **kw)
                    continue
                got = F.avg_pool2d(q, *args, **kw)
                assert not isinstance(got, QTensor) and torch.equal(got, want), (name, args, kw)
            for args in ((3, 2, 2), (13,), (3, 0)):
                with pytest.raises(RuntimeError):
                    F.avg_pool2d(q, *args)


# ------------------------------------------------------------------------------------------ GPU: ResNet-50-D end to end
def _resnetd_recon(tmp_path, in_hw, batch):
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "pytorch-quantity_b200", "test"))
    import _models
    import tools
    from common.quantity import merge_bn
    from model.resnet import resnet50d_fabu
    from model.resnet.resnet_fabu import randomize_bn_

    def build():
        torch.manual_seed(0)
        net = resnet50d_fabu(in_hw=in_hw).eval()
        with torch.no_grad():
            randomize_bn_(net, 0)
        return net

    wd = str(tmp_path / "wd")
    cfg, user = _models.configs(wd, (3, in_hw, in_hw), 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build(), "cpu"), config=cfg, user_config=user, verbose=False)
        cal = [(torch.randn(batch, 3, in_hw, in_hw, generator=torch.Generator().manual_seed(1 + i)), None)
               for i in range(2)]
        q.activation_quantize(cal)
        q.weight_quantize()
        r = tools.Reconstruction(build(), config=cfg)
        r.merge_bn()
        return r.ReconModel(r.get_quantity_information(), None).cuda().eval()


@gpu
def test_resnet50d_end_to_end(tmp_path):
    from oracle import pq_oracle as oracle
    from common.quantity import GraphedForward, NewConv2d, _native, enable_int8_pipeline
    model = _resnetd_recon(tmp_path, 64, 2)
    convs = {n: m for n, m in model.named_modules() if isinstance(m, NewConv2d)}
    assert len(convs) == 55
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(42)).cuda()
    seen = {}
    hooks = [m.register_forward_hook(lambda m, i, o, n=n: seen.__setitem__(n, (i[0].detach().cpu().numpy(),
                                                                              o.detach().cpu().numpy())))
             for n, m in convs.items()]
    with torch.no_grad():
        ref = model(x)
    for h in hooks:
        h.remove()
    assert ref.shape == (2, 1000) and len(seen) == len(convs)
    for n, (xi, yo) in seen.items():
        m = convs[n]
        c = m.Conv
        info = {"weight_bit": m.weight_bit, "bias_bit": m.bias_bit, "input_bit": m.input_bit,
                "output_bit": m.output_bit}
        w = c.weight.detach().double().cpu().numpy() * 2.0 ** -m.weight_bit
        b = m.quantized_bias.double().cpu().numpy() * 2.0 ** -m.bias_bit
        exp, _ = oracle.int_conv_layer(xi, w.astype(np.float32), b.astype(np.float32), info, stride=c.stride,
                                       padding=c.padding, dilation=c.dilation, groups=c.groups)
        assert np.array_equal(yo, exp), n

    enable_int8_pipeline(model)
    with torch.no_grad():
        model(x)                    # the first forward takes each add's census of the payloads its consumers read
        l0 = dict(_native.LAUNCHES)
        recorded = profiler_records()
        names = launched(lambda: model(x)) if recorded else model(x)
        out = model(x)
    d = {k: _native.LAUNCHES.get(k, 0) - l0.get(k, 0) for k in _native.LAUNCHES}
    assert torch.equal(out, ref)
    assert d.get("avgpool_requant", 0) == 2 * 3          # the three avg-down pools, in both forwards
    assert d.get("quantize_s8", 0) == 2 * 2              # the stem's and the classifier's quantisers only
    if recorded:
        assert sum("avgpool_global_kernel" in n and "AvgPoolParams" in n for n in names) == 3
        assert not any("avg_pool" in n.lower() for n in names), [n for n in names if "avg" in n.lower()]
    else:
        fresh_run_passed()
    fwd = GraphedForward(model, x)
    assert torch.equal(fwd(x), ref)
    enable_int8_pipeline(model, False)

"""Nearest-neighbour upsampling kept int8 in the pipeline: index tables from ATen's own rule, the two kernels that read
an operand through them (pq_add_requant_nearest, pq_concat_requant_nearest_s8), the lazy nearest views of
int8_pipeline, and the semantic FPN of the model zoo end to end.

The kernels are compared byte for byte with their same-resolution counterparts (pq_add_requant, pq_concat_requant_s8)
applied to the operand gathered with torch indexing, which share no code with the table reads.  Outputs sit in
sentinel-filled buffers; inputs must be unchanged afterwards; torch.profiler shows which overload each call lands on.
"""
import ctypes
import os
import re
import shutil
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


def _pipe():
    from common.quantity import int8_pipeline
    return int8_pipeline


# ------------------------------------------------------------------------------------------ CPU: argument rules
MODES = ("nearest", "nearest-exact", "bilinear", "bicubic", "area", "linear", "trilinear")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("antialias", (False, True))
@pytest.mark.parametrize("align_corners", (None, False, True))
@pytest.mark.parametrize("ndim", (3, 4, 5))
def test_decline_rules(mode, antialias, align_corners, ndim):
    """Only mode='nearest' on a 4-D input, without antialias or align_corners, becomes a nearest view."""
    req = _pipe().nearest_request(ndim, size=None, scale_factor=2.0, mode=mode, align_corners=align_corners,
                                  recompute_scale_factor=None, antialias=antialias)
    taken = mode == "nearest" and not antialias and align_corners is None and ndim == 4
    assert (req is not None) == taken
    if taken:
        assert req == (None, 2.0, None)


def test_decline_rules_positional_and_defaults():
    nr = _pipe().nearest_request
    assert nr(4, None, [2, 3]) == (None, (2, 3), None)            # F.interpolate's default mode is 'nearest'
    assert nr(4, [9, 11]) == ((9, 11), None, None)
    assert nr(4, None, 1.7, "nearest", None, True) == (None, 1.7, True)
    assert nr(4, None, 2, "nearest-exact") is None
    with pytest.raises(TypeError):
        nr(4, None, 2, "nearest", None, None, False, "surplus")


GEOMETRIES = [  # (H, W, F.interpolate keyword arguments)
    (5, 7, dict(scale_factor=2)), (5, 7, dict(scale_factor=3)), (5, 7, dict(scale_factor=(2, 1))),
    (6, 9, dict(scale_factor=1.7)), (6, 9, dict(scale_factor=1.7, recompute_scale_factor=True)),
    (6, 9, dict(size=(9, 11))), (6, 9, dict(size=13)), (8, 10, dict(scale_factor=0.5)),
    (7, 9, dict(scale_factor=(3, 0.5))), (1, 1, dict(scale_factor=4)), (1, 6, dict(size=(3, 2))),
]


@pytest.mark.parametrize("H,W,kw", GEOMETRIES, ids=[str(i) for i in range(len(GEOMETRIES))])
def test_tables_gather_equals_interpolate(H, W, kw):
    """Gathering through the tables equals F.interpolate(mode='nearest') for every geometry (CPU)."""
    p = _pipe()
    req = p.nearest_request(4, **kw)
    t = p.nearest_tables((H, W), req, torch.device("cpu"))
    x = torch.randn(2, 3, H, W, generator=torch.Generator().manual_seed(H * W))
    ref = F.interpolate(x, mode="nearest", **kw)
    assert t.map_h.dtype == torch.int32 and tuple(ref.shape[2:]) == (t.map_h.numel(), t.map_w.numel())
    assert torch.equal(x[:, :, t.map_h.long()][:, :, :, t.map_w.long()], ref)
    assert p.nearest_tables((H, W), req, torch.device("cpu")) is t            # cached per geometry


@pytest.mark.parametrize("C,N,hw,taken", [(24, 2, 8, False), (19, 2, 8, False), (32, 2, 8, True), (16, 2 ** 15, 256, False),
                                         (16, 2 ** 15 - 1, 256, True)])
def test_view_add_outside_add_limits_is_declined(C, N, hw, taken):
    """A NewAdd with one upsampled operand becomes a lazy nearest add only inside pq_add_requant_nearest's limits
    (C % 16 == 0, N*P*Q <= 2^31 - 1); otherwise add_forward declines and the add takes the fp32 path.  A NewConv2d
    reading an upsampled tensor beyond the pixel limit quantises the de-quantised tensor instead.  (Meta tensors: the
    rules are host logic.)"""
    import types
    from common.quantity import QTensor
    p = _pipe()
    meta = torch.device("meta")
    lat = QTensor((N, C, hw, hw), meta, q8_bit=3)
    v = p._upsample(QTensor((N, C, hw // 2, hw // 2), meta, q8_bit=3), (), {"scale_factor": 2, "mode": "nearest"})
    assert v is not None and v._lazy_cat.view_source() is not None
    assert (p.add_forward(types.SimpleNamespace(output_bit=3), lat, v) is not None) == taken
    assert (p.add_forward(types.SimpleNamespace(output_bit=3), v, lat) is not None) == taken
    assert v._lazy_cat.supported(3) == (N * hw * hw <= 2 ** 31 - 1)


def _fpn_trace():
    import torch
    import tools._config as tc
    from common.quantity import merge_bn
    from model.fpn import fpn_r50_fabu
    from tools.pytorch_quantizer import Quantity
    here = os.path.dirname(os.path.abspath(__file__))
    cfg = tc.load_tool_config(os.path.join(os.path.dirname(here), "pytorch-quantity_b200", "tools", "configs.yml"))
    st = cfg["SETTINGS"]
    q = object.__new__(Quantity)
    q._cared_op_type, q._all_op_type = st["CARE_OP_TYPE"], st["ALL_OP_TYPE"]
    q._allow_same_tid_op_type, q._merge_op_type = st["ALLOW_SAME_TID_OP_TYPE"], st["MERGE_OP_YTPE"]
    q.verbose, q.rank, q.cuda_device = False, 0, torch.device("cpu")
    torch.manual_seed(0)
    net = q.build_net_structure(merge_bn(fpn_r50_fabu().eval(), "cpu"), (1, 3, 64, 64))
    return q, net


def test_fpn_traces_to_expected_merge_groups(capsys):
    """The tracer sees every upsample (UpsamplingNearest2d is in ALL_OP_TYPE, not cared) and splices it out, so each
    top-down Eltwise groups its lateral with the producer of the upsampled level, and the head Concats nest."""
    q, net = _fpn_trace()
    merges = [(n, i["inputs"]) for n, i in net.items() if i["type"] in ("Eltwise", "Concat")]
    assert [n for n, _ in merges[-6:]] == ["Eltwise_123", "Eltwise_126", "Eltwise_129", "Concat_135", "Concat_139",
                                           "Concat_143"]
    assert dict(merges[-6:]) == {
        "Eltwise_123": ["Conv2d_121", "Conv2d_120"],      # lateral4(C4) + Up(P5 = lateral5(C5))
        "Eltwise_126": ["Conv2d_124", "Eltwise_123"],     # lateral3(C3) + Up(P4)
        "Eltwise_129": ["Conv2d_127", "Eltwise_126"],     # lateral2(C2) + Up(P3)
        "Concat_135": ["Conv2d_130", "Conv2d_132"],       # head2(P2), Up(head3(P3))
        "Concat_139": ["Concat_135", "Conv2d_136"],
        "Concat_143": ["Concat_139", "Conv2d_140"]}
    groups = q.get_merge_groups(net)
    assert groups[:5] == [["Concat_139", "Conv2d_140"], ["Concat_135", "Conv2d_136"], ["Conv2d_130", "Conv2d_132"],
                          ["Conv2d_127", "Eltwise_126"], ["Conv2d_124", "Eltwise_123"]]
    convs = [n for n, i in net.items() if i["type"] == "Conv2d"]
    assert len(convs) == 53 + 4 + 4 + 2                   # ResNet-50 body, laterals, level heads, fuse + classifier


# ------------------------------------------------------------------------------------------ GPU: kernels
def _lib():
    from common.quantity import _native
    return _native.lib()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class Guarded:
    """A device buffer of `shape` / `dtype` in the middle of sentinel bytes."""

    def __init__(self, shape, dtype):
        n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
        self.buf = torch.full((GUARD + n + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.t = self.buf[GUARD:GUARD + n].view(dtype).view(shape)

    def ptr(self):
        return self.t.data_ptr()

    def guards_intact(self):
        return bool((self.buf[:GUARD] == SENTINEL).all()) and bool((self.buf[-GUARD:] == SENTINEL).all())

    def untouched(self):
        return bool((self.buf == SENTINEL).all())


def _operand(shape, is16, bit, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lo, hi = (-128 * 2 ** bit, 127 * 2 ** bit) if is16 else (-128, 127)
    v = torch.randint(lo, hi + 1, shape, dtype=torch.int32, device="cuda", generator=g)
    v.view(-1)[:4] = torch.tensor([lo, hi, 0, -1], dtype=torch.int32)
    return v.to(torch.int16 if is16 else torch.int8).contiguous()


def _tables(hw, kw):
    p = _pipe()
    return p.nearest_tables(hw, p.nearest_request(4, **kw), torch.device("cuda"))


def _gather(x, t):
    """NHWC x read at (n, map_h[p], map_w[q]) by torch indexing."""
    return x[:, t.map_h.long()][:, :, t.map_w.long()].contiguous()


def _tf(b):
    return "true" if b else "false"


def launched(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_FRESH_ENV = "PQ_UPSAMPLE_FRESH"
_STATE = {}


def profiler_records():
    """Whether torch.profiler records CUDA kernels in this process.  After some sequences of earlier tests in one pytest
    process it records none at all; the tests of this file that check kernel names (the kernel rows, the census and
    the FPN end to end) then run once more in a fresh process, which must pass."""
    if "recorded" not in _STATE:
        _STATE["recorded"] = bool(launched(lambda: torch.ones(16, device="cuda").add_(1)))
        if not _STATE["recorded"]:
            assert not os.environ.get(_FRESH_ENV), "torch.profiler records no CUDA kernels in a fresh process"
            r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-p", "no:cacheprovider",
                                "-m", "gpu", "-k", "nearest_kernel or census or fpn_end_to_end"],
                               cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                               env=dict(os.environ, **{_FRESH_ENV: "1"}), capture_output=True, text=True, timeout=3600)
            _STATE["fresh"] = (r.returncode, r.stdout[-3000:])
    return _STATE["recorded"]


def fresh_run_passed():
    rc, out = _STATE["fresh"]
    assert rc == 0, "the fresh-process run of this file, which makes the kernel-name checks, failed:\n" + out


def check_landing(fn, want):
    """fn() launches exactly one kernel, whose demangled name contains `want` (overload id and params struct)."""
    if profiler_records():
        names = launched(fn)
        assert len(names) == 1 and want in names[0].replace(" ", ""), (want, names)
        _STATE.setdefault("reached", set()).add(names[0])
    else:
        fn()
        fresh_run_passed()


ADD_OVERLOADS = [(a16, b16, relu_in, qdown) for a16 in (False, True) for b16 in (False, True)
                 for relu_in in (False, True) for qdown in (False, True)]
# (N, H, W, C, F.interpolate keyword arguments): x2, x3, (2, 1), 1.7 with and without recompute_scale_factor, explicit
# size, downscaling 0.5, H / W / N = 1, C from 16 to 2048, and source pixel counts not a multiple of the block
ADD_GEOMS = [
    (2, 5, 7, 16, dict(scale_factor=2)), (1, 4, 3, 48, dict(scale_factor=3)), (3, 6, 5, 32, dict(scale_factor=(2, 1))),
    (2, 6, 9, 64, dict(scale_factor=1.7)), (2, 6, 9, 64, dict(scale_factor=1.7, recompute_scale_factor=True)),
    (1, 7, 5, 256, dict(size=(9, 11))), (2, 10, 8, 32, dict(scale_factor=0.5)), (1, 1, 9, 16, dict(scale_factor=2)),
    (2, 9, 1, 16, dict(scale_factor=3)), (1, 1, 1, 2048, dict(scale_factor=4)), (1, 3, 3, 1024, dict(scale_factor=2)),
    (4, 13, 11, 272, dict(scale_factor=2)),
    (4, 160, 160, 48, dict(scale_factor=2)),
]
GRID_THREADS = 148 * 16 * 256          # the bandwidth kernels' grid cap: kNumSMs * 16 blocks of 256 threads


def test_add_rows_take_the_grid_stride_loop_with_a_carry():
    """One add row has more (pixel, 16-channel group) items than the capped grid has threads, with a group count that
    does not divide the grid: its threads go round the loop more than once and advance their group with a carry."""
    rows = []
    for N, H, W, C, kw in ADD_GEOMS:
        t = _pipe().nearest_tables((H, W), _pipe().nearest_request(4, **kw), torch.device("cpu"))
        items = N * t.map_h.numel() * t.map_w.numel() * C // 16
        rows.append(items > GRID_THREADS and GRID_THREADS % (C // 16) != 0)
    assert any(rows)


def _add_case(a16, b16, relu_in, qdown, geom, out_relu, outs, seed):
    N, H, W, C, kw = geom
    t = _tables((H, W), kw)
    P, Q = t.map_h.numel(), t.map_w.numel()
    abit, bbit = (6, 3) if a16 else (2, 5)
    o_bit = max(abit, bbit)
    qbit = o_bit - 3 if qdown else o_bit + 2
    a = _operand((N, P, Q, C), a16, abit, seed)
    b = _operand((N, H, W, C), b16, bbit, seed + 1)
    a0, b0 = a.clone(), b.clone()
    arelu, brelu = (relu_in, False) if seed % 2 else (False, relu_in)
    want16, want8 = outs in ("s16", "both"), outs in ("q8", "both")
    # the reference: pq_add_requant on the gathered operand
    bg = _gather(b, t)
    ref16 = torch.empty((N, P, Q, C), dtype=torch.int16, device="cuda")
    ref8 = torch.empty((N, P, Q, C), dtype=torch.int8, device="cuda")
    flags = 1 if out_relu else 0
    assert _lib().pq_add_requant(a.data_ptr(), int(a16), abit, int(arelu), bg.data_ptr(), int(b16), bbit, int(brelu),
                                 a.numel(), flags, ref16.data_ptr(), ref8.data_ptr(), qbit, _stream()) == 0
    g16, g8 = Guarded((N, P, Q, C), torch.int16), Guarded((N, P, Q, C), torch.int8)
    call = lambda: _lib().pq_add_requant_nearest(
        a.data_ptr(), int(a16), abit, int(arelu), b.data_ptr(), int(b16), bbit, int(brelu), N, P, Q, C, H, W,
        t.map_h.data_ptr(), t.map_w.data_ptr(), flags, g16.ptr() if want16 else None, g8.ptr() if want8 else None,
        qbit, _stream())
    rc = []
    check_landing(lambda: rc.append(call()),
                  "add_requant_kernel<%s,%s,%s,%s>(pq::AddNearestParams" % tuple(map(_tf, (a16, b16, relu_in, qdown))))
    torch.cuda.synchronize()
    assert rc == [0]
    assert torch.equal(a, a0) and torch.equal(b, b0)
    assert g16.guards_intact() and g8.guards_intact()
    assert torch.equal(g16.t, ref16) if want16 else g16.untouched()
    assert torch.equal(g8.t, ref8) if want8 else g8.untouched()


@gpu
@pytest.mark.parametrize("overload", ADD_OVERLOADS, ids=["a16=%d,b16=%d,relu=%d,qdown=%d" % o for o in ADD_OVERLOADS])
def test_add_nearest_kernel_every_overload(overload):
    for i, geom in enumerate(ADD_GEOMS):
        _add_case(*overload, geom, out_relu=bool(i % 3 == 1), outs=("both", "s16", "q8")[i % 3], seed=7 * i + 1)


# concat sources: (channels, is16, bit, relu, geometry of this member or None for the output resolution)
CONCAT_CASES = [
    # vector path: every channel count % 16 == 0
    ((2, 6, 10), [(32, False, 3, False, dict(scale_factor=2)), (16, True, 5, True, None)], 4, 48),
    ((1, 6, 10), [(64, True, 6, False, dict(scale_factor=1.7)), (32, False, 2, False, dict(scale_factor=(3, 0.5))),
                 (16, False, 1, True, None)], 3, 128),
    ((2, 9, 11), [(128, False, 4, False, dict(size=(9, 11)))], 4, 128),
    ((3, 8, 8), [(16, True, 7, True, dict(scale_factor=0.5))], 0, 32),
    ((1, 1, 1), [(2048, False, 4, False, dict(scale_factor=1))], 6, 2048),
    ((2, 11, 17), [(48, False, 4, False, dict(scale_factor=1.7, recompute_scale_factor=True))], 5, 64),
    # scalar path: a channel count or the padding off the 16 grid
    ((2, 6, 10), [(3, False, 3, True, dict(scale_factor=2)), (5, True, 4, False, None)], 4, 16),
    ((1, 6, 9), [(24, False, 2, False, dict(scale_factor=(2, 1))), (16, False, 3, False, dict(scale_factor=3))], 3, 45),
    ((1, 1, 9), [(7, True, 5, False, dict(scale_factor=(1, 3)))], 2, 7),
    # more work than the capped grid: vector threads and scalar warps go round their loops more than once
    ((4, 320, 320), [(48, False, 3, False, dict(scale_factor=2)), (16, True, 5, False, None)], 4, 80),
    ((2, 160, 160), [(3, False, 3, False, dict(scale_factor=4)), (5, True, 4, True, None)], 4, 16),
]


def test_concat_rows_take_the_grid_stride_loop():
    """The vector kernel has more (pixel, group) items than the grid has threads on one row, and the scalar kernel
    (one warp per pixel) more pixels than the grid has warps on another."""
    vec = [N * P * Q * c_pad // 16 for (N, P, Q), m, _, c_pad in CONCAT_CASES
           if c_pad % 16 == 0 and all(c % 16 == 0 for c, *_ in m)]
    scalar = [N * P * Q for (N, P, Q), m, _, c_pad in CONCAT_CASES if c_pad % 16 or any(c % 16 for c, *_ in m)]
    assert max(vec) > GRID_THREADS and max(scalar) > GRID_THREADS // 32


def _src_hw(out_nhw, kw):
    """A source height / width that F.interpolate(**kw) maps to the output's (searching small sizes)."""
    N, P, Q = out_nhw
    p = _pipe()

    def out_hw(H, W):
        try:
            t = p.nearest_tables((H, W), p.nearest_request(4, **kw), torch.device("cpu"))
        except RuntimeError:                            # an empty output: ATen refuses it
            return None
        return t.map_h.numel(), t.map_w.numel()
    # the output height depends on H only and the width on W only: search them one at a time
    H = next(h for h in range(1, 4 * P + 4) if (out_hw(h, 4 * Q + 3) or (0,))[0] == P)
    W = next(w for w in range(1, 4 * Q + 4) if out_hw(H, w) == (P, Q))
    return H, W


@gpu
@pytest.mark.parametrize("case", range(len(CONCAT_CASES)))
def test_concat_nearest_kernel(case):
    from common.quantity import _native
    (N, P, Q), members, q_bit, c_pad = CONCAT_CASES[case]
    arr = (_native.ConcatNearestSrc * len(members))()
    ref_srcs, keep = (_native.ConcatSrc * len(members))(), []
    vec = c_pad % 16 == 0
    for i, (c, is16, bit, relu, kw) in enumerate(members):
        if kw is None:
            x = _operand((N, P, Q, c), is16, bit, 100 * case + i)
            arr[i] = _native.ConcatNearestSrc(x.data_ptr(), int(is16), c, bit, int(relu), P, Q, None, None)
            xg = x
        else:
            H, W = _src_hw((N, P, Q), kw)
            t = _tables((H, W), kw)
            x = _operand((N, H, W, c), is16, bit, 100 * case + i)
            arr[i] = _native.ConcatNearestSrc(x.data_ptr(), int(is16), c, bit, int(relu), H, W, t.map_h.data_ptr(),
                                              t.map_w.data_ptr())
            xg = _gather(x, t)
        vec = vec and c % 16 == 0
        ref_srcs[i] = _native.ConcatSrc(xg.data_ptr(), int(is16), c, bit, int(relu))
        keep.append((x, x.clone(), xg))
    ref = torch.empty((N, P, Q, c_pad), dtype=torch.int8, device="cuda")
    assert _lib().pq_concat_requant_s8(ref_srcs, len(members), N * P * Q, q_bit, c_pad, ref.data_ptr(), _stream()) == 0
    g = Guarded((N, P, Q, c_pad), torch.int8)
    rc = []
    check_landing(lambda: rc.append(_lib().pq_concat_requant_nearest_s8(arr, len(members), N, P, Q, q_bit, c_pad,
                                                                        g.ptr(), _stream())),
                  "concat_requant_%s_kernel(pq::ConcatNearestParams" % ("vec" if vec else "scalar"))
    torch.cuda.synchronize()
    assert rc == [0] and g.guards_intact() and torch.equal(g.t, ref)
    assert all(torch.equal(x, x0) for x, x0, _ in keep)


# ------------------------------------------------------------------------------------------ GPU: limits
# (limit as the header words it, entry point, (N, P, Q, C), expected return code).  The rows at size (N*P*Q = 2^31 - 1)
# run in test_nearest_pixel_limit_inside_at_size; the others in test_nearest_limit_one_step_inside_and_beyond.
AT_SIZE = 2 ** 31 - 1
NEAREST_LIMITS = [
    ("C % 16 == 0", "add", (1, 4, 4, 16), 0), ("C % 16 == 0", "add", (1, 4, 4, 17), EUNSUPPORTED),
    ("C % 16 == 0", "add", (1, 4, 4, 15), EUNSUPPORTED), ("C % 16 == 0", "add", (1, 4, 4, 48), 0),
    ("C % 16 == 0", "add", (1, 4, 4, 47), EUNSUPPORTED),
    ("N*P*Q <= 2^31 - 1", "add", (AT_SIZE, 1, 1, 16), 0), ("N*P*Q <= 2^31 - 1", "concat", (AT_SIZE, 1, 1, 16), 0),
    ("N*P*Q <= 2^31 - 1", "add", (2, 1, 2 ** 30, 16), EUNSUPPORTED),
    ("N*P*Q <= 2^31 - 1", "concat", (2, 1, 2 ** 30, 16), EUNSUPPORTED),
    ("N*P*Q <= 2^31 - 1", "add", (2 ** 16, 2 ** 8, 2 ** 7, 16), EUNSUPPORTED),
]


def _header():
    return open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "pq_sm100.h")).read()


def test_every_nearest_limit_has_an_inside_and_a_beyond_row():
    """Each limit the header documents for the nearest entry points ('nearest limit:') has a row one step inside and
    one beyond, on each entry point it names (the pixel limit binds both)."""
    documented = [s.strip() for s in re.findall(r"nearest limit: ([^;\n]+?)(?:;|\s*\*/|\n)", _header())]
    assert documented == ["C % 16 == 0", "N*P*Q <= 2^31 - 1"], documented
    assert {r[0] for r in NEAREST_LIMITS} == set(documented)
    for lim in documented:
        entries = ("add",) if lim.startswith("C ") else ("add", "concat")
        for e in entries:
            assert {r[3] == 0 for r in NEAREST_LIMITS if r[0] == lim and r[1] == e} == {True, False}, (lim, e)


@gpu
@pytest.mark.parametrize("row", [r for r in NEAREST_LIMITS if r[2][0] != AT_SIZE],
                         ids=lambda r: "%s-%s-%s" % (r[1], r[0].replace(" ", ""), "x".join(map(str, r[2]))))
def test_nearest_limit_one_step_inside_and_beyond(row):
    """A row inside a limit runs and writes its output; a row beyond is PQ_EUNSUPPORTED and writes nothing."""
    from common.quantity import _native
    _, entry, (N, P, Q, C), want = row
    t = _tables((2, 2), dict(scale_factor=2))
    small = N * P * Q * C <= 1 << 20                   # beyond rows never touch their (small) buffers
    a = torch.zeros((N, P, Q, C) if small else (1, 4, 4, 16), dtype=torch.int8, device="cuda")
    b = torch.ones((1, 2, 2, C), dtype=torch.int8, device="cuda")
    mh = _tables((2, 2), dict(size=(P, Q))) if small else t
    g = Guarded(a.shape, torch.int8)
    if entry == "add":
        rc = _lib().pq_add_requant_nearest(a.data_ptr(), 0, 3, 0, b.data_ptr(), 0, 3, 0, N, P, Q, C, 2, 2,
                                           mh.map_h.data_ptr(), mh.map_w.data_ptr(), 0, None, g.ptr(), 3, _stream())
    else:
        src = (_native.ConcatNearestSrc * 1)(_native.ConcatNearestSrc(b.data_ptr(), 0, C, 3, 0, 2, 2,
                                                                      mh.map_h.data_ptr(), mh.map_w.data_ptr()))
        rc = _lib().pq_concat_requant_nearest_s8(src, 1, N, P, Q, 3, C, g.ptr(), _stream())
    torch.cuda.synchronize()
    assert rc == want
    if want == 0:
        assert g.guards_intact() and bool((g.t == 1).all())      # 0 + 1 at bit 3, or 1 requantised at bit 3
    else:
        assert g.untouched()


@gpu
def test_nearest_invalid_arguments():
    from common.quantity import _native
    t = _tables((2, 2), dict(scale_factor=2))
    b = torch.zeros((1, 2, 2, 32), dtype=torch.int8, device="cuda")
    g = Guarded((1, 4, 4, 32), torch.int8)
    add = lambda C, mh: _lib().pq_add_requant_nearest(g.ptr(), 0, 3, 0, b.data_ptr(), 0, 3, 0, 1, 4, 4, C, 2, 2, mh,
                                                      t.map_w.data_ptr(), 0, None, g.ptr(), 3, _stream())
    assert add(16, None) == EINVAL and add(0, t.map_h.data_ptr()) == EINVAL
    same_res_mismatch = (_native.ConcatNearestSrc * 1)(_native.ConcatNearestSrc(b.data_ptr(), 0, 32, 3, 0, 2, 2, None,
                                                                                None))
    assert _lib().pq_concat_requant_nearest_s8(same_res_mismatch, 1, 1, 4, 4, 3, 32, g.ptr(), _stream()) == EINVAL
    torch.cuda.synchronize()
    assert g.untouched()


@gpu
def test_nearest_pixel_limit_inside_at_size():
    """N*P*Q = 2^31 - 1 (a prime, so N = 2^31 - 1 images of one pixel) runs on both entry points; the outputs are
    checked at both ends and against the sentinel after them."""
    need = 2 * (2 ** 31 - 1) * 16 + (1 << 30)
    if torch.cuda.mem_get_info()[0] < need:
        pytest.skip("needs %d GB of free device memory" % (need >> 30))
    from common.quantity import _native
    n = 2 ** 31 - 1
    t = _tables((1, 1), dict(scale_factor=1))
    x = torch.full((n, 1, 1, 16), 5, dtype=torch.int8, device="cuda")
    x[-1] = -7
    g = Guarded((n, 1, 1, 16), torch.int8)
    src = (_native.ConcatNearestSrc * 1)(_native.ConcatNearestSrc(x.data_ptr(), 0, 16, 3, 0, 1, 1, t.map_h.data_ptr(),
                                                                  t.map_w.data_ptr()))
    assert _lib().pq_concat_requant_nearest_s8(src, 1, n, 1, 1, 4, 16, g.ptr(), _stream()) == 0
    torch.cuda.synchronize()
    assert g.guards_intact() and bool((g.t[:1 << 20] == 10).all()) and bool((g.t[-1] == -14).all())
    assert bool((g.t[-(1 << 20):-1] == 10).all())
    # the add: a = x, b = the one source pixel of every image (x itself, read through the 1x1 tables)
    assert _lib().pq_add_requant_nearest(x.data_ptr(), 0, 3, 0, x.data_ptr(), 0, 3, 0, n, 1, 1, 16, 1, 1,
                                         t.map_h.data_ptr(), t.map_w.data_ptr(), 0, None, g.ptr(), 3, _stream()) == 0
    torch.cuda.synchronize()
    assert g.guards_intact() and bool((g.t[:1 << 20] == 10).all()) and bool((g.t[-1] == -14).all())
    assert bool((g.t[-(1 << 20):-1] == 10).all())


@gpu
def test_census_every_nearest_overload_reached():
    """Every kernel of the library that takes a nearest params struct is one a test above lands on."""
    if shutil.which("cuobjdump") is None or shutil.which("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not installed")
    from common.quantity import _native
    sym = subprocess.run(["cuobjdump", "-symbols", _native.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = subprocess.run(["cu++filt"], input=sym, check=True, capture_output=True, text=True).stdout
    ids = set()
    for line in names.splitlines():
        if "STO_ENTRY" in line and "NearestParams" in line:
            s = line[line.index("pq::"):].replace("(bool)1", "true").replace("(bool)0", "false").replace(" ", "")
            ids.add(s[:s.index("NearestParams")])
    assert len(ids) == 18, sorted(ids)
    for o in ADD_OVERLOADS:
        _add_case(*o, ADD_GEOMS[0], out_relu=False, outs="both", seed=3)
    for case in (0, 6):
        test_concat_nearest_kernel(case)
    if _STATE.get("recorded"):
        reached = {n.replace(" ", "") for n in _STATE["reached"]}
        for i in ids:
            assert any(r.startswith("void" + i) or r.startswith(i) or i in r for r in reached), i


# ------------------------------------------------------------------------------------------ GPU: pipeline
def _qconv(cin, cout, info, seed):
    from common.quantity import NewConv2d
    torch.manual_seed(seed)
    conv = nn.Conv2d(cin, cout, 3, padding=1)
    m = NewConv2d(conv.cuda(), dict(info)).cuda().eval()
    return m


INFO = {"weight_bit": 7, "input_bit": 4, "output_bit": 3, "bias_bit": 4}


def _sources(x):
    """(name, QTensor source, its fp32-boundary value): lazy conv, pending ReLU, NewAdd int16 sum, lazy Concat and a
    composed view."""
    from common.quantity import NewAdd
    c1, c2 = _qconv(16, 32, INFO, 1), _qconv(16, 32, INFO, 2)
    add = NewAdd().cuda()
    add.output_bit = 2
    out = []
    for pipe in (True, False):
        for m in (c1, c2, add):
            m.int8_pipeline = pipe
        a, b = c1(x), c2(x)
        s = add(a, b)
        out.append({"lazy conv": a, "pending relu": F.relu(b), "add int16": s, "lazy concat": torch.cat([a, F.relu(b)], 1),
                    "composed view": F.interpolate(a, scale_factor=(2, 1), mode="nearest")})
    return [(k, out[0][k], out[1][k]) for k in out[0]]


@gpu
@pytest.mark.parametrize("kw", [dict(scale_factor=2), dict(scale_factor=1.7), dict(size=(9, 11)),
                                dict(scale_factor=0.5), dict(scale_factor=3, recompute_scale_factor=True)],
                         ids=["x2", "x1.7", "size", "x0.5", "x3-recompute"])
def test_pipeline_interpolate_equals_dequantised(kw):
    """F.interpolate on each QTensor source is a lazy view equal to F.interpolate of the de-quantised tensor, and a
    NewConv2d / Concat / NewAdd reading the view equals the fp32-boundary model's layer on that tensor."""
    from common.quantity import NewAdd, QTensor, _native
    x = torch.randn(2, 16, 6, 8, generator=torch.Generator().manual_seed(5)).cuda()
    with torch.no_grad():
        for name, q, ref in _sources(x):
            v = F.interpolate(q, mode="nearest", **kw)
            want = F.interpolate(ref, mode="nearest", **kw)
            assert isinstance(v, QTensor) and v._upsample is not None, name
            assert torch.equal(v.dequantize(), want), name
            cons = _qconv(v.shape[1], 16, dict(INFO, input_bit=2), 9)
            cons.int8_pipeline = True
            before = _native.LAUNCHES.get("concat_requant_nearest", 0)
            got = cons(v).dequantize()
            assert _native.LAUNCHES.get("concat_requant_nearest", 0) == before + 1, name
            cons.int8_pipeline = False
            assert torch.equal(got, cons(want)), name
            cat = torch.cat([F.relu(v), v], 1)
            assert torch.equal(cat.dequantize(), torch.cat([F.relu(want), want], 1)), name
            if v._lazy_cat.view_source() is not None:
                lat = _qconv(16, v.shape[1], INFO, 4)
                lat.int8_pipeline = True
                xl = F.interpolate(x, size=tuple(v.shape[2:]), mode="nearest")
                add = NewAdd().cuda()
                add.output_bit, add.int8_pipeline = 3, True
                n0 = _native.LAUNCHES.get("add_requant_nearest", 0)
                s = add(lat(xl), v)
                assert isinstance(s, QTensor) and torch.equal(s.dequantize(), add(lat(xl), v).dequantize())
                assert _native.LAUNCHES.get("add_requant_nearest", 0) > n0, name
                lat.int8_pipeline = add.int8_pipeline = False
                assert torch.equal(s.dequantize(), add(lat(xl), want)), name
                assert torch.equal(F.relu(s).dequantize(), F.relu(add(lat(xl), want))), name


@gpu
@pytest.mark.parametrize("C", [19, 24, 32])
def test_pipeline_view_add_outside_add_limits(C):
    """An FCN-style `score_skip + Up(score)` whose channel count is off the 16 grid (19 classes, a 24-channel decoder)
    is outside pq_add_requant_nearest's limits: the add takes the fp32 path, and its result and the convolution reading
    it are torch.equal to the fp32-boundary model.  At C = 32 the same graph runs the nearest add."""
    from common.quantity import NewAdd, QTensor, _native
    x = torch.randn(2, 16, 12, 10, generator=torch.Generator().manual_seed(C)).cuda()
    skip, score, head = _qconv(16, C, INFO, 11), _qconv(16, C, INFO, 12), _qconv(C, 16, dict(INFO, input_bit=2), 13)
    add = NewAdd().cuda()
    add.output_bit = 2
    outs = {}
    with torch.no_grad():
        for pipe in (True, False):
            for m in (skip, score, head, add):
                m.int8_pipeline = pipe
            n0 = _native.LAUNCHES.get("add_requant_nearest", 0)
            s = add(skip(x), F.interpolate(score(x[:, :, ::2, ::2]), scale_factor=2, mode="nearest"))
            y = head(F.relu(s))
            if pipe:                                    # the add ran for the convolution's int8 operand
                assert isinstance(s, QTensor) == (C % 16 == 0)
                assert _native.LAUNCHES.get("add_requant_nearest", 0) - n0 == (C % 16 == 0)
            outs[pipe] = (s.dequantize() if isinstance(s, QTensor) else s,
                          y.dequantize() if isinstance(y, QTensor) else y)
    assert torch.equal(outs[True][0], outs[False][0]) and torch.equal(outs[True][1], outs[False][1])


@gpu
@pytest.mark.parametrize("mode,extra", [("nearest-exact", {}), ("bilinear", {}), ("bilinear", dict(antialias=True)),
                                        ("bicubic", dict(align_corners=True)), ("area", {})])
def test_pipeline_declined_modes_fall_back(mode, extra):
    from common.quantity import QTensor
    x = torch.randn(2, 16, 6, 8, generator=torch.Generator().manual_seed(6)).cuda()
    with torch.no_grad():
        for name, q, ref in _sources(x):
            got = F.interpolate(q, scale_factor=2, mode=mode, **extra)
            assert not isinstance(got, QTensor), name
            assert torch.equal(got, F.interpolate(ref, scale_factor=2, mode=mode, **extra)), name


# ------------------------------------------------------------------------------------------ GPU: FPN end to end
def _fpn_recon(tmp_path, in_hw, batch, fuse=True):
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(os.path.dirname(here), "pytorch-quantity_b200", "test"))
    import _models
    import tools
    from common.quantity import merge_bn
    from model.fpn import fpn_r50_fabu
    from model.resnet.resnet_fabu import randomize_bn_

    def build():
        torch.manual_seed(0)
        net = fpn_r50_fabu().eval()
        with torch.no_grad():
            randomize_bn_(net, 0)
        return net

    wd = str(tmp_path / ("wd_fused" if fuse else "wd_plain"))
    cfg, user = _models.configs(wd, (3, in_hw, in_hw), 2)
    with torch.no_grad():
        q = tools.Quantity(merge_bn(build(), "cpu"), config=cfg, user_config=user, verbose=False)
        q._fuse_calibration = fuse
        cal = [(torch.randn(batch, 3, in_hw, in_hw, generator=torch.Generator().manual_seed(1 + i)), None)
               for i in range(2)]
        q.activation_quantize(cal)
        stats = (q.last_calibration, open(os.path.join(wd, "feat.table")).read())
        q.weight_quantize()
        r = tools.Reconstruction(build(), config=cfg)
        r.merge_bn()
        return r.ReconModel(r.get_quantity_information(), None).cuda().eval(), q, stats


@gpu
def test_fpn_calibration_fused_equals_unfused(tmp_path):
    """Calibration with the fused calibration forward on and off: identical maxima, histograms and feat.table."""
    _, _, (a, ta) = _fpn_recon(tmp_path, 64, 2, fuse=True)
    _, _, (b, tb) = _fpn_recon(tmp_path, 64, 2, fuse=False)
    assert ta == tb and a["top_feat_names"] == b["top_feat_names"]
    for n in a["top_feat_names"]:
        assert repr(a["max_vals"][n]) == repr(b["max_vals"][n]), n
        assert (a["distributions"][n] == b["distributions"][n]).all(), n


@gpu
def test_fpn_end_to_end(tmp_path, monkeypatch):
    from oracle import pq_oracle as oracle
    from common.quantity import GraphedForward, NewAdd, NewConv2d, QTensor, _native, enable_int8_pipeline, \
        int8_pipeline
    model, _, _ = _fpn_recon(tmp_path, 64, 2)
    convs = {n: m for n, m in model.named_modules() if isinstance(m, NewConv2d)}
    assert len(convs) == 63
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(42)).cuda()
    seen = {}
    hooks = [m.register_forward_hook(lambda m, i, o, n=n: seen.__setitem__(n, (i[0].detach().cpu().numpy(),
                                                                              o.detach().cpu().numpy())))
             for n, m in convs.items()]
    with torch.no_grad():
        ref = model(x)
    for h in hooks:
        h.remove()
    assert ref.shape == (2, 19, 64, 64) and len(seen) == len(convs)
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
    name_of = {id(m): n for n, m in convs.items()}
    in_kind = {}
    conv_forward = int8_pipeline.conv_forward

    def recording_conv_forward(mod, xin):
        in_kind[name_of[id(mod)]] = "fp32" if not isinstance(xin, QTensor) else (
            "view" if xin._upsample is not None else "cat" if xin._lazy_cat is not None else xin.q8_bit)
        return conv_forward(mod, xin)
    monkeypatch.setattr(int8_pipeline, "conv_forward", recording_conv_forward)
    quantized = []
    for n, m in convs.items():
        m._quantize = (lambda x, n=n, f=m._quantize: (quantized.append(n), f(x))[1])
    add_forward, declined = int8_pipeline.add_forward, []

    def recording_add_forward(mod, a, b):
        out = add_forward(mod, a, b)
        if out is None:
            declined.append(mod)
        return out
    monkeypatch.setattr(int8_pipeline, "add_forward", recording_add_forward)
    with torch.no_grad():
        model(x).dequantize()       # the first forward takes each add's census of the payloads its consumers read
    l0 = dict(_native.LAUNCHES)
    with torch.no_grad():
        recorded = profiler_records()
        names = launched(lambda: model(x).dequantize()) if recorded else model(x).dequantize()   # read: lazy until then
        out = model(x)
    for m in convs.values():
        del m.__dict__["_quantize"]
    d = {k: _native.LAUNCHES.get(k, 0) - l0.get(k, 0) for k in _native.LAUNCHES}
    assert torch.equal(out, ref)
    top_down = [m for n, m in model.named_modules() if isinstance(m, NewAdd) and n in ("add4", "add3", "add2")]
    assert len(top_down) == 3
    assert declined == []                                           # every add stays quantised, top-down ones too
    assert d.get("add_requant_nearest", 0) == 2 * 3                 # every top-down add, in both forwards
    assert d.get("concat_requant_nearest", 0) == 2 * 1              # the head Concat: one launch
    assert d.get("concat_requant", 0) == 0
    # the convolutions that quantise from fp32: the stem (the image) and those whose input bit differs from the bit of
    # their producer's payload (conv_forward's identity test declines; quantised from the de-quantised tensor)
    other_bit = {n for n, k in in_kind.items() if k not in ("fp32", "view", "cat") and k != convs[n].input_bit}
    fp32_in = {n for n, k in in_kind.items() if k == "fp32"}
    assert fp32_in == {"stem.0"}, sorted(fp32_in)
    assert set(quantized) == fp32_in | other_bit, (sorted(quantized), sorted(other_bit))
    assert in_kind["fuse.0"] == "cat"
    if recorded:
        ups = [n for n in names if "upsample" in n.lower()]
        assert len(ups) == 1, ups                                    # the final user-facing x4 only
        assert sum("add_requant_kernel" in n and "AddNearestParams" in n for n in names) == 3
        assert sum("concat_requant" in n and "ConcatNearestParams" in n for n in names) == 1
    else:
        fresh_run_passed()
    fwd = GraphedForward(model, x)
    assert torch.equal(fwd(x), ref)
    enable_int8_pipeline(model, False)


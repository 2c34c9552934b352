"""CPU-only checks: the C-ABI library loads and exports every symbol the header declares,
host-side logic (JSON writer, re-writer, bit reader, graph pruning / merge groups) agrees
with the reference's golden outputs.  No compute kernels are launched."""
import json
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, REPO, golden_json, load_golden


def _header():
    return open(os.path.join(REPO, "include", "pq_sm100.h")).read()


def test_library_exports_every_declared_symbol():
    from common.quantity import _native
    header = _header()
    declared = set(re.findall(r"\b(pq_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_native.SYMBOLS), declared ^ set(_native.SYMBOLS)
    lib = _native.lib()
    for name in declared:
        assert hasattr(lib, name), name
    version = int(re.search(r"#define PQ_VERSION (\d+)", header).group(1))
    assert lib.pq_version() == version == _native.PQ_VERSION
    assert b"PQ_EINVAL" in lib.pq_error_string(-1)
    assert lib.pq_kl_workspace_doubles() >= 2048 + 2 * 1920


def test_ctypes_signatures_match_the_header():
    """ctypes passes surplus arguments through without complaint, so a stale argtypes list or struct layout would
    misbind silently: every SYMBOLS entry must take as many parameters as the header declares, and the ctypes
    structures must have the header structs' fields in the same order."""
    from common.quantity import _native
    header = re.sub(r"/\*.*?\*/", "", _header(), flags=re.S)
    decls = re.findall(r"^[a-z_0-9 ]+\**\s*\**(pq_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", header, flags=re.M)
    assert {name for name, _ in decls} == set(_native.SYMBOLS)
    for name, params in decls:
        params = params.strip()
        count = 0 if params in ("", "void") else params.count(",") + 1
        assert len(_native.SYMBOLS[name][1]) == count, name
    for struct, cls in (("pq_conv_desc", _native.ConvDesc), ("pq_add_desc", _native.AddDesc),
                        ("pq_concat_src", _native.ConcatSrc)):
        body = re.search(r"typedef struct %s \{(.*?)\}" % struct, header, flags=re.S).group(1)
        fields = [re.findall(r"\w+", part)[-1] for decl in body.split(";") if decl.strip() for part in decl.split(",")]
        assert fields == [f[0] for f in cls._fields_], struct


def test_product_never_imports_oracle():
    pkg = os.path.join(REPO, "pytorch-quantity_b200")
    for root, _d, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(root, f)).read()
                assert "oracle" not in text.replace("# oracle-free", ""), os.path.join(root, f)


def test_no_cpu_fallback_without_cuda():
    import torch
    import common.quantity as cq
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError):
        cq.QuanDequan(8, 3)(torch.zeros(4))
    with pytest.raises(RuntimeError):
        cq.DistributionCollector(["a"]).refresh_max_val({"a": np.zeros(4, np.float32)})
    with pytest.raises(RuntimeError):
        cq.Quantizer(["a"]).quantize({"a": np.ones(2048, np.int32)}, {"a": np.float32(0.1)})


def test_json_writer_is_byte_identical_to_json_dump():
    from tools._jsonio import dumps_int_array
    rng = np.random.default_rng(0)
    for shape in [(5,), (3, 4), (2, 3, 3, 3), (4, 1, 1, 1), (1,), (2, 0), (7, 2, 1), (1, 1, 1, 1), (40,), (3, 40), (2, 3, 40),
                  (64, 3, 7, 7), (5, 33), (33, 5), (2, 17, 2), (9, 2, 2, 2, 2), (2, 70000), (16, 8, 3, 3)]:
        for lo, hi in ((-128, 128), (-99999, 100000), (0, 1), (-40000, 40000), (-3000000, 3000000)):
            a = rng.integers(lo, hi, size=shape).astype(np.int32)        # (beyond 5 digits: the plain path)
            assert dumps_int_array(a) == json.dumps(a.tolist(), indent=4), (shape, lo)
    a8 = rng.integers(-128, 128, size=(3, 2)).astype(np.int8)
    assert dumps_int_array(a8) == json.dumps(a8.tolist(), indent=4)


def test_rewriter_and_bit_reader_vs_golden(tmp_path):
    """BiasReWriter on a hand-computed case: bias alignment, int8 wrap-around (quirk Q8),
    MAX_SHIFT cap, table rewrite (tools/rewriter.py:38-140).  The reference-produced files are
    compared byte-for-byte in tests/test_gpu_e2e.py."""
    from common.quantity import BitReader
    from tools import BiasReWriter
    from tools._jsonio import dump_int_array
    wd = tmp_path
    for sub in ("weight", "bias", "new_weight", "new_bias"):
        os.makedirs(wd / sub)
    old_bias = {"a": 3, "b": 9}
    new_bias = {"a": 5, "b": 4}
    dump_int_array(np.array([100, -100, 50, 1], np.int32), str(wd / "bias" / "a.bias.json"))
    dump_int_array(np.array([100, -100, 48, 16, 24, 8], np.int32), str(wd / "bias" / "b.bias.json"))
    open(wd / "weight.table", "w").write("a.weight 7\na.bias 3\nb.weight 14\nb.bias 9\n")
    open(wd / "feat.table", "w").write("image 4\na 5 4\nb 4 5\n")
    dump_int_array(np.array([[100, -100], [3, 127]], np.int32), str(wd / "weight" / "a.weight.json"))
    dump_int_array(np.array([[64, -128], [2, 6]], np.int32), str(wd / "weight" / "b.weight.json"))
    rw = BiasReWriter(str(wd / "weight"), str(wd / "bias"), str(wd / "new_weight"), str(wd / "new_bias"),
                      str(wd / "weight.table"), str(wd / "feat.table"), max_shift_limit=12)
    wb, bb = rw.get_weight_info()
    fb, ib = rw.get_feat_info()
    assert dict(wb) == {"a": 7, "b": 14} and dict(bb) == old_bias and fb == {"image": 4, "a": 5, "b": 4}
    rw.rewrite_bias_table(bb, fb)
    rw.rewrite_bias_dir(bb, fb)
    assert json.load(open(wd / "new_bias" / "a.bias.json")) == [-112, 112, -56, 4]      # x4, int8 wrap (quirk Q8)
    assert json.load(open(wd / "new_bias" / "b.bias.json")) == [3, -3, 2, 0, 1, 0]      # /32, half-even
    need, nw = rw.max_shift_limit_weight(fb, ib, wb)
    assert need and nw == {"a": 7, "b": 11}                                             # 14+5-4=15 > 12 -> 11
    rw.rewrite_weight_table(wb, nw)
    rw.rewrite_weight_dir(wb, nw)
    assert open(wd / "weight.table").read() == "a.weight 7\na.bias 5\nb.weight 11\nb.bias 4\n"
    assert json.load(open(wd / "new_weight" / "b.weight.json")) == [[8, -16], [0, 1]]
    r = BitReader(feat_table=str(wd / "feat.table"), weight_table=str(wd / "weight.table"))
    assert r.get_feat_info()[1]["b"] == ["5"]


def test_graph_pruning_and_merge_groups_host_logic():
    """prune_net_info / get_merge_groups on the reference's own un-pruned trace of the tiny net."""
    from collections import OrderedDict
    from tools.pytorch_quantizer import Quantity
    g = load_golden("tiny_e2e.npz")
    j = golden_json(g)
    q = object.__new__(Quantity)
    q._cared_op_type = ["Conv2d", "Linear", "Eltwise", "Concat"]
    q._merge_op_type = ["Eltwise", "Concat"]
    q.verbose, q.rank = False, 0
    full = OrderedDict([
        ("Conv2d_1", {"inputs": [], "type": "Conv2d"}),
        ("ReLU_2", {"inputs": ["Conv2d_1"], "type": "ReLU"}),
        ("MaxPool2d_3", {"inputs": ["ReLU_2"], "type": "MaxPool2d"}),
        ("Conv2d_4", {"inputs": ["MaxPool2d_3"], "type": "Conv2d"}),
        ("Conv2d_5", {"inputs": ["MaxPool2d_3"], "type": "Conv2d"}),
        ("Concat_6", {"inputs": ["Conv2d_4", "Conv2d_5"], "type": "Concat"}),
        ("ReLU_7", {"inputs": ["Concat_6"], "type": "ReLU"}),
        ("Conv2d_8", {"inputs": ["ReLU_7"], "type": "Conv2d"}),
        ("Eltwise_9", {"inputs": ["Conv2d_8", "MaxPool2d_3"], "type": "Eltwise"}),
        ("ReLU_10", {"inputs": ["Eltwise_9"], "type": "ReLU"}),
        ("Conv2d_11", {"inputs": ["ReLU_10"], "type": "Conv2d"}),
        ("Eltwise_12", {"inputs": ["Conv2d_11", "ReLU_10"], "type": "Eltwise"}),
        ("ReLU_13", {"inputs": ["Eltwise_12"], "type": "ReLU"}),
        ("AvgPool2d_14", {"inputs": ["ReLU_13"], "type": "AvgPool2d"}),
        ("View_15", {"inputs": ["AvgPool2d_14"], "type": "View"}),
        ("Linear_16", {"inputs": ["View_15"], "type": "Linear"}),
    ])
    keep = [n for n, i in full.items() if i["type"] in q._cared_op_type]
    pruned = q.prune_net_info(full, keep)
    assert pruned == j["net_info"] and list(pruned) == list(j["net_info"])
    assert q.get_merge_groups(pruned) == j["merge_groups"]


# Public surface of the reference's common.quantity package (quantity/common/quantity/__init__.py:1-6), recorded by
# inspecting the unmodified reference: constructor / function parameters (name, default) and forward() parameters.
_REQ = object()
REFERENCE_SURFACE = {
    "DistributionCollector": ([("tensor_list", _REQ), ("interval_num", 2048), ("statistic", 1), ("worker_num", 1),
                               ("debug", False)], None,
                              ["add_to_distributions", "distribution_intervals", "distributions", "max_vals", "refresh_max_val"]),
    "Quantizer": ([("tensor_list", _REQ), ("worker_num", 1), ("debug", False)], None,
                  ["bits", "quantize", "threshold_value"]),
    "BitReader": ([("feat_table", None), ("weight_table", None)], None, ["get_feat_info", "get_weight_info"]),
    "merge_bn": ([("model", _REQ), ("device", "cpu")], None, []),
    "walk_dirs": ([("dir_name", _REQ), ("file_type", None)], None, []),
    "tid": ([("tensor", _REQ)], None, []),
    "Eltwise": ([], ["x", "y"], []), "Concat": ([], ["x", "y", "dim"], []), "Identity": ([], ["x"], []),
    "View": ([], ["x"], []),
    "RightShift": ([("bits", _REQ), ("rs", _REQ)], ["x"], []), "Sp": ([("bits", _REQ)], ["x"], []),
    "BiasAdd": ([], ["x", "y"], []),
    "NewConv2d": ([("conv_module", _REQ), ("quantize_infor", _REQ)], ["input"], ["quantity"]),
    "NewAdd": ([], ["x", "y"], []),
    "NewLinear": ([("linear_module", _REQ), ("quantize_infor", _REQ)], ["input"], ["quantity"]),
    "QuanDequan": ([("Bitwidth", _REQ), ("bit", _REQ)], ["quantized_x"], []),
    "TestConv": ([("name", _REQ), ("module", _REQ), ("quantize_infor", _REQ), ("new_model_path", _REQ)], ["x"], []),
    "TestLinear": ([("name", _REQ), ("module", _REQ), ("quantize_infor", _REQ), ("new_model_path", _REQ)], ["x"], []),
    "Quantity": ([("ib", _REQ)], ["x"], []), "DeQuantity": ([("ob", _REQ)], ["x"], []),
}


def test_public_surface_matches_the_reference():
    """Same 21 names, same leading constructor / function parameters (names and defaults; extra trailing keyword
    parameters such as ``device`` are allowed), same forward() parameter names, same public members."""
    import inspect
    import common.quantity as cq
    assert sorted(cq.__all__) == sorted(REFERENCE_SURFACE)
    for name, (params, fwd, members) in REFERENCE_SURFACE.items():
        obj = getattr(cq, name)
        sig = inspect.signature(obj.__init__ if inspect.isclass(obj) else obj)
        got = [p for p in sig.parameters.values() if p.name != "self" and p.kind in (p.POSITIONAL_OR_KEYWORD,)]
        assert len(got) >= len(params), name
        for have, (pname, default) in zip(got, params):
            assert have.name == pname, (name, have.name, pname)
            if default is _REQ:
                assert have.default is inspect.Parameter.empty, (name, pname)
            else:
                assert have.default == default, (name, pname)
        for extra in got[len(params):]:
            assert extra.default is not inspect.Parameter.empty, (name, extra.name)   # extensions must be optional
        if fwd is not None:
            fparams = [p for p in inspect.signature(obj.forward).parameters if p != "self"]
            assert fparams[:len(fwd)] == fwd, (name, fparams)
        for m in members:
            assert hasattr(obj, m), (name, m)


def test_tools_surface_matches_the_reference():
    """quantity/tools/__init__.py:1-3 exports Quantity, Reconstruction, BiasReWriter with these entry points."""
    import inspect
    import tools
    for cls, methods in (("Quantity", ["activation_quantize", "weight_quantize", "rewrite_weight", "build_net_structure",
                                       "get_merge_groups", "preprocess", "dilation_to_zero_padding", "init_dir"]),
                         ("Reconstruction", ["merge_bn", "get_quantity_information", "ReconModel", "ReconTest"]),
                         ("BiasReWriter", ["get_weight_info", "get_feat_info", "rewrite_bias_table", "rewrite_bias_dir",
                                           "max_shift_limit_weight", "rewrite_weight_table", "rewrite_weight_dir"])):
        obj = getattr(tools, cls)
        for m in methods:
            assert callable(getattr(obj, m)), (cls, m)
    assert list(inspect.signature(tools.Quantity.__init__).parameters)[:2] == ["self", "model"]
    assert list(inspect.signature(tools.Reconstruction.__init__).parameters)[:2] == ["self", "model"]
    for m in ("ReconModel", "ReconTest"):               # reconstruction.py:175, :243
        assert list(inspect.signature(getattr(tools.Reconstruction, m)).parameters) == \
            ["self", "all_quantize_infor", "new_model_path"], m


def test_space_to_depth_filter_mapping_equals_stride2_convolution():
    """new_quantity_op.s2d_filter + the layout of pq_quantize_nchw_to_s2d16_s8, emulated in torch on the CPU: the
    stride-1 filter over 16-byte space-to-depth pixels must reproduce the stride-2 convolution (odd sizes, odd / even /
    zero padding, 1-4 channels, non-square filters)."""
    import torch
    import torch.nn.functional as F
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "_nqo_src", os.path.join(os.path.dirname(__file__), "..", "pytorch-quantity_b200", "common", "quantity",
                                 "new_quantity_op.py"))
    src = open(spec.origin).read()
    ns = {"torch": torch}
    start = src.index("def s2d_filter(")
    exec(src[start:src.index("class NewLinear(")], ns)           # the pure-torch helper, without importing the CUDA package
    s2d_filter = ns["s2d_filter"]
    g = torch.Generator().manual_seed(0)
    for (C, H, W, K, R, S, ph, pw) in [(3, 20, 20, 4, 7, 7, 3, 3), (3, 13, 17, 5, 7, 7, 3, 3), (1, 12, 12, 3, 3, 3, 1, 1),
                                       (4, 10, 9, 2, 5, 5, 2, 2), (3, 11, 14, 2, 3, 3, 0, 0), (2, 9, 9, 3, 7, 5, 3, 2),
                                       (3, 16, 16, 2, 2, 2, 0, 0), (3, 15, 12, 2, 6, 4, 2, 1)]:
        x = torch.randint(-128, 128, (2, C, H, W), generator=g).double()
        w = torch.randint(-128, 128, (K, C, R, S), generator=g).double()
        ref = F.conv2d(x, w, stride=2, padding=(ph, pw))
        P, Q = ref.shape[2], ref.shape[3]
        w2 = s2d_filter(w, (ph, pw)).double()
        ra = w2.shape[1]
        pt, pl = ph + (ph & 1), pw + (pw & 1)
        hp2, wp2 = P + ra - 1, Q + 3
        xs = torch.zeros(2, hp2, wp2, 2, 2, 4, dtype=torch.float64)
        for i in range(hp2):
            for dy in range(2):
                h = 2 * i + dy - pt
                if not 0 <= h < H:
                    continue
                for j in range(wp2):
                    for dx in range(2):
                        ww = 2 * j + dx - pl
                        if 0 <= ww < W:
                            xs[:, i, j, dy, dx, :C] = x[:, :, h, ww]
        xs = xs.view(2, hp2, wp2 * 16)
        out = torch.zeros_like(ref)
        for p in range(P):
            for q in range(Q):
                for a in range(ra):
                    out[:, :, p, q] += xs[:, p + a, q * 16:q * 16 + 64] @ w2[:, a, :].T
        assert torch.equal(out, ref), (C, H, W, K, R, S, ph, pw)


def test_rewriter_reuses_arrays_it_wrote_and_reparses_foreign_files(tmp_path):
    """tools/_jsonio.written_array: the array behind a file this process wrote is reused only while the file is
    unchanged; a file modified (or written) by somebody else is parsed again."""
    import time
    from tools._jsonio import dump_int_array, written_array
    p = str(tmp_path / "w.json")
    a = np.arange(-6, 6, dtype=np.int32).reshape(3, 4)
    dump_int_array(a, p)
    got = written_array(p)
    assert got is not None and np.array_equal(got, a) and got is not a
    assert np.array_equal(np.array(json.load(open(p))), a)
    time.sleep(0.01)
    with open(p, "w") as f:                                  # same size, other content, later mtime
        f.write(open(p).read().replace("5", "4"))
    assert written_array(p) is None
    assert written_array(str(tmp_path / "missing.json")) is None
    q = str(tmp_path / "foreign.json")
    json.dump(a.tolist(), open(q, "w"), indent=4)
    assert written_array(q) is None

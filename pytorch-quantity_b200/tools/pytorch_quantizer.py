"""Calibration driver (reference: quantity/tools/pytorch_quantizer.py:19-693).

``Quantity(model)`` traces the model, ``activation_quantize(batches)`` runs the two-pass
calibration and writes ``feat.table``, ``weight_quantize()`` writes ``weight.table`` and the
per-parameter JSON, ``rewrite_weight()`` finalises them -- same entry points, same files.

What is different from the reference, by design (B200-first):
  * hooks keep the observed activations ON THE DEVICE (the reference copies every one to
    the host, :509,:513) and hand the whole batch to two multi-tensor CUDA kernels, one
    launch per pass per batch (max-abs, 2048-bin histograms);
  * pass 1 caches as many batches of observed activations in HBM as fit (180 GB per GPU),
    so pass 2 re-runs the fp32 forward only for the batches that did not fit;
  * calibration batches shard data-parallel over ``torch.distributed`` ranks; the per-tensor
    maxima merge with all_reduce(MAX) and the integer histograms with all_reduce(SUM), so the
    tables are bit-identical for any rank count;
  * the KL threshold search for all tensors is one GPU launch sequence;
  * during calibration the bias add after every cuDNN convolution, each Eltwise and the out-of-place nn.ReLU that
    follows either run as one native kernel that also takes the pass-1 max-abs (plan_calibration_fusion); the
    convolution that completes an Eltwise's operands also computes the Eltwise, and the stem's convolution the
    max-pool after its ReLU (plan_calibration_handover), all with bit-identical results;
  * producer/consumer links are traced by tensor identity instead of a value hash.
"""
import json
import math
import os
import time
from collections import Counter, OrderedDict

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from common.quantity import DistributionCollector, Eltwise, Quantizer, _native

from ._config import load_tool_config, load_user_config
from ._jsonio import dump_int_array
from .rewriter import BiasReWriter


def _dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def _barrier():
    """Rank 0 alone writes the tables / JSON; the other ranks must not run ahead and read partial files."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()


def plan_calibration_fusion(net, modules, inplace_modified):
    """Which modules the calibration forward runs as fused native ops, decided from one trace of
    Quantity.build_net_structure (``net``: tracer name -> {"inputs", "type"}, ``modules``: tracer name -> module).

    Returns {tracer name: (module, relu)} for every module that fired exactly once, whose output no later op modifies
    in place, and that is
      * an nn.Conv2d with the plain nn.Conv2d forward, an fp32 bias and zero padding: cuDNN convolves without the bias
        and pq_conv_epilogue_f32 adds it, or
      * an Eltwise: pq_eltwise_add_f32.
    ``relu`` is the output's only traced nn.ReLU consumer when that ReLU is out of place, has the plain forward and
    fired once (the fused op then writes its output too), else None.  Without torch's backend selector the fused
    convolution could not tell whether cuDNN would run it, so no convolution is planned (Eltwise does not depend on
    it).  What depends on the call (grad mode, autocast, contiguous fp32 tensors on the device, the cuDNN backend)
    the fused forwards check every time.  Modules outside CARE_OP_TYPE are planned too; their fused ops take no
    max-abs, since the collector does not observe their outputs."""
    calls = Counter(id(m) for m in modules.values())
    consumers = {}
    for name, info in net.items():
        for src in info["inputs"]:
            consumers.setdefault(src, []).append(name)

    def once(m):
        return calls[id(m)] == 1 and "forward" not in vars(m)

    can_select = hasattr(torch._C, "_select_conv_backend")
    plan = OrderedDict()
    for name, m in modules.items():
        if not once(m) or name in inplace_modified:
            continue
        conv = (can_select and isinstance(m, nn.Conv2d) and type(m).forward is nn.Conv2d.forward
                and type(m)._conv_forward is nn.Conv2d._conv_forward and m.bias is not None
                and m.bias.dtype == torch.float32 and m.padding_mode == "zeros" and not isinstance(m.padding, str))
        if not (conv or type(m) is Eltwise):
            continue
        relus = [modules[c] for c in consumers.get(name, ()) if isinstance(modules[c], nn.ReLU)]
        relu = relus[0] if len(relus) == 1 else None
        if relu is not None and (type(relu).forward is not nn.ReLU.forward or relu.inplace or not once(relu)):
            relu = None
        plan[name] = (m, relu)
    return plan


def plan_calibration_handover(net, modules, plan):
    """The hand-overs between the fused ops of ``plan`` (plan_calibration_fusion), from the same trace.  Returns
    (eltwise, pools):
      * eltwise: {Eltwise tracer name: (producer, other, producer_first)} for every planned Eltwise whose two operands
        come from two traced modules, where ``producer`` -- the operand producer that fires last -- is a planned
        convolution without a fused ReLU.  Its fused forward also computes the Eltwise (pq_conv_epilogue_add_f32)
        when the traced tensor ``other`` of the other operand exists unmodified; ``producer_first``: the producer's
        output is the Eltwise's first operand.
      * pools: {convolution tracer name: MaxPool2d tracer name} for every planned
        convolution whose fused ReLU's only consumer is a plain nn.MaxPool2d without indices, dilation or ceil_mode
        that fired once: its fused forward also computes the pooled output (pq_conv_epilogue_maxpool_f32)."""
    calls = Counter(id(m) for m in modules.values())
    consumers = {}
    for name, info in net.items():
        for src in info["inputs"]:
            consumers.setdefault(src, []).append(name)
    name_of = {id(m): n for n, m in modules.items()}

    def pos(name):
        return int(name.rsplit("_", 1)[1])

    eltwise = OrderedDict()
    for name, (m, _relu) in plan.items():
        srcs = net[name]["inputs"]
        if type(m) is not Eltwise or len(srcs) != 2 or srcs[0] == srcs[1]:
            continue
        last = max(srcs, key=pos)
        if last in plan and isinstance(plan[last][0], nn.Conv2d) and plan[last][1] is None:
            eltwise[name] = (last, srcs[1] if last == srcs[0] else srcs[0], last == srcs[0])

    def pair(v):
        return tuple(v) if isinstance(v, (tuple, list)) else (v, v)

    pools = OrderedDict()
    for name, (m, relu) in plan.items():
        if relu is None or not isinstance(m, nn.Conv2d):
            continue
        relu_name = name_of[id(relu)]
        after = consumers.get(relu_name, [])
        if len(after) != 1:
            continue
        pool = modules[after[0]]
        if (type(pool) is nn.MaxPool2d and calls[id(pool)] == 1 and "forward" not in vars(pool)
                and not pool.return_indices and not pool.ceil_mode and pair(pool.dilation) == (1, 1)
                and len(set(pair(pool.kernel_size))) == 1 and len(set(pair(pool.stride))) == 1
                and len(set(pair(pool.padding))) == 1):
            pools[name] = after[0]
    return eltwise, pools


class _CalibrationFusion:
    """The fused forwards of a plan (plan_calibration_fusion) and its hand-overs (plan_calibration_handover) for one
    activation_quantize call: install() sets them as instance attributes, remove() restores the modules.

    Each fused op is one native launch on the stream current at the call.  While ``collect`` is set (pass 1) a fused
    op whose output the collector observes (``slots``: tensor name -> its max_bits slot) also takes the max |x| of
    that output into the slot, provided it runs at its traced position in the forward (the calibration hooks' count),
    and adds the name to ``reduced``; refresh_max_val then skips those tensors.

    A fused op may also compute a consumer's output speculatively: the convolution its ReLU's (and the stem's
    max-pool's), the convolution that completes an Eltwise's operands the Eltwise's.  The consumer returns it only if
    it is called with the very tensors, unmodified; any other call runs the consumer's own forward.  Every module's
    output is complete when the module returns.  A speculated Eltwise takes its max |z| into a pending slot; fold()
    moves it to max_bits only when the Eltwise took z at its traced position."""

    def __init__(self, plan, handover, modules, hook_state, slots, max_bits, device):
        self.collect = False
        self.reduced = set()
        self._state = hook_state
        self._device = device
        eltwise, pools = handover
        name_of = {id(m): n for n, m in modules.items()}
        # Per forward (begin() clears them): the outputs of fused ops and of handed-over ReLUs / max-pools that an
        # Eltwise hand-over reads as its other operand (tracer name -> (tensor, _version)), and the speculated Eltwise
        # outputs (tracer name -> (a, a._version, b, b._version, z, relu(z) or None)).
        self._others = {other for _, other, _ in eltwise.values()}
        self._outputs = {}
        self._speculated = {}
        # max |z| of a speculated Eltwise: pending[i] for max_bits[i], folded in once the hand-over is confirmed
        self._max_bits = max_bits
        self._pending = torch.zeros_like(max_bits) if max_bits is not None and eltwise else None
        self._published = set()     # pending indices written this forward
        self._confirmed = set()     # ... and confirmed
        self._forwards = []         # (module, fused forward), all built before any module is touched
        for name, (m, relu) in plan.items():
            relu_stash = [None] if relu is not None else None
            pos = int(name.rsplit("_", 1)[1])
            if isinstance(m, nn.Conv2d):
                adds = [(e, other, first, slots.get(e), plan[e][1] is not None)
                        for e, (producer, other, first) in eltwise.items() if producer == name]
                pool = None
                if name in pools:
                    pool = (modules[pools[name]], [None])
                    self._forwards.append((pool[0], self._pool(pool[0], pools[name], pool[1])))
                fwd = self._conv(m, name, pos, slots.get(name), relu_stash, adds[0] if adds else None, pool)
            else:
                fwd = self._eltwise(m, name, pos, slots.get(name), relu_stash)
            self._forwards.append((m, fwd))
            if relu is not None:
                self._forwards.append((relu, self._relu(relu, name_of[id(relu)], relu_stash)))
        self._patched = []

    def install(self):
        for m, forward in self._forwards:
            m.forward = forward
            self._patched.append(m)

    def remove(self):
        for m in self._patched:
            del m.forward
        self._patched = []
        self.begin()

    def begin(self):
        """A forward begins: nothing the last one computed can be handed over any more."""
        self._outputs.clear()
        self._speculated.clear()

    def fold(self):
        """Pass 1, after a forward: the confirmed speculative maxima into max_bits (an integer max, order-free like
        the kernels' atomicMax), the others dropped, the pending slots cleared for the next forward."""
        if not self._published:
            return
        for i in self._published - self._confirmed:
            self._pending[i] = 0
        if self._confirmed:
            torch.maximum(self._max_bits, self._pending, out=self._max_bits)
        self._pending.zero_()
        self._published.clear()
        self._confirmed.clear()

    def _fusable(self, t):
        return (isinstance(t, torch.Tensor) and t.device == self._device and t.dtype == torch.float32
                and t.is_contiguous() and t.data_ptr() % 16 == 0)

    def _at_position(self, pos):
        return self.collect and self._state["idx"] == pos - 1

    def _slot(self, name, pos, slot):
        if slot is not None and self._at_position(pos):
            self.reduced.add(name)
            return slot
        return None

    def _output(self, name, t):
        if name in self._others:
            self._outputs[name] = (t, t._version)

    def _conv(self, m, name, pos, slot, relu_stash, add, pool):
        own = m.forward
        cudnn = {}                  # input shape -> does cuDNN run this convolution (bias included)?

        def on_cudnn(x):
            # only on the cuDNN backend is the bias a separate add after the convolution (ATen's
            # output.add_(bias)); the slow and depthwise kernels accumulate it.  A selector that cannot be asked
            # (a changed private signature) means: not fused.
            try:
                return torch._C._select_conv_backend(x, m.weight, m.bias, m.stride, m.padding, m.dilation, False,
                                                     (0, 0), m.groups) == torch._C._ConvBackend.Cudnn
            except (TypeError, RuntimeError):
                return False

        def epilogue(y):
            max_slot = self._slot(name, pos, slot)
            if add is not None:
                elt, other_name, first, elt_slot, elt_relu = add
                got = self._outputs.get(other_name)
                if got is not None and got[0]._version == got[1] and self._fusable(got[0]) \
                        and got[0].shape == y.shape:
                    other = got[0]
                    i = max_z = None
                    if elt_slot is not None and self.collect:
                        i = (elt_slot - self._max_bits.data_ptr()) // 4
                        max_z = self._pending.data_ptr() + 4 * i
                        self._published.add(i)
                    z, r = _native.conv_epilogue_add(y, m.bias, other, not first, elt_relu, max_slot, max_z)
                    a, b = (y, other) if first else (other, y)
                    self._speculated[elt] = (a, a._version, b, b._version, z, r, i)
                    return
            if pool is not None:
                k, s, p = (v if isinstance(v, int) else v[0]
                           for v in (pool[0].kernel_size, pool[0].stride, pool[0].padding))
                got = _native.conv_epilogue_maxpool(y, m.bias, k, s, p, max_slot)
                if got is not None:
                    relu_stash[0] = (y, y._version, got[0])
                    pool[1][0] = (got[0], got[0]._version, got[1])
                    return
            r = _native.conv_epilogue(y, m.bias, relu_stash is not None, max_slot)
            if relu_stash is not None:
                relu_stash[0] = (y, y._version, r)

        def forward(x):
            # under autocast the convolution runs in 16 bits with the bias cast alongside: the module's own forward
            if (torch.is_grad_enabled() or torch.is_autocast_enabled(self._device.type) or not self._fusable(x)
                    or x.dim() != 4):
                return own(x)
            ok = cudnn.get(x.shape)
            if ok is None:
                ok = cudnn[x.shape] = on_cudnn(x)
            if not ok:
                return own(x)
            y = F.conv2d(x, m.weight, None, m.stride, m.padding, m.dilation, m.groups)
            if y.dtype != torch.float32 or not y.is_contiguous():     # (a channels_last weight) ATen's own bias add
                return y.add_(m.bias.reshape(1, -1, 1, 1))
            epilogue(y)
            self._output(name, y)
            return y
        return forward

    def _eltwise(self, m, name, pos, slot, relu_stash):
        own = m.forward

        def forward(a, b):
            spec = self._speculated.pop(name, None)
            if spec is not None and a is spec[0] and a._version == spec[1] and b is spec[2] and b._version == spec[3]:
                z, r, i = spec[4], spec[5], spec[6]
                if i is not None and self._slot(name, pos, slot) is not None:
                    self._confirmed.add(i)
            else:
                # (torch.add is not an autocast op: fp32 operands give the fp32 sum with autocast on or off)
                if torch.is_grad_enabled() or not (self._fusable(a) and self._fusable(b)) or a.shape != b.shape:
                    return own(a, b)
                z, r = _native.eltwise_add(a, b, relu_stash is not None, self._slot(name, pos, slot))
            if relu_stash is not None:
                relu_stash[0] = (z, z._version, r)
            self._output(name, z)
            return z
        return forward

    def _relu(self, relu, name, stash):
        own = relu.forward

        def forward(x):
            st, stash[0] = stash[0], None
            if st is not None and x is st[0] and x._version == st[1]:
                self._output(name, st[2])
                return st[2]
            return own(x)
        return forward

    def _pool(self, pool, name, stash):
        own = pool.forward

        def forward(x):
            st, stash[0] = stash[0], None
            if st is not None and x is st[0] and x._version == st[1]:
                self._output(name, st[2])
                return st[2]
            return own(x)
        return forward


class Quantity(object):

    def __init__(self, model, config=None, user_config=None, cache_bytes=None, verbose=True):
        self.config = load_tool_config(config)
        self.user_config = load_user_config(user_config)
        self.verbose = verbose
        self.rank, self.world_size = _dist_info()
        self.init_dir()

        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: pytorch-quantity_b200 has no CPU fallback")
        self.device = self.user_config["SETTINGS"]["DEVICE"]      # kept; execution is always CUDA
        if self.world_size == 1:
            self.cuda_device = torch.device("cuda", int(self.user_config["SETTINGS"].get("GPU", 0)))
        else:
            self.cuda_device = torch.device("cuda", torch.cuda.current_device())

        settings = self.config["SETTINGS"]
        self._cared_op_type = settings["CARE_OP_TYPE"]
        self._all_op_type = settings["ALL_OP_TYPE"]
        self._allow_same_tid_op_type = settings["ALLOW_SAME_TID_OP_TYPE"]
        self._merge_op_type = settings["MERGE_OP_YTPE"]
        self._max_img_num = settings["MAX_CALI_IMG_NUM"]
        self._log("max_img_num", self._max_img_num)
        # The reference leaves the caller's model alone (:57); here it must live on the GPU (no CPU fallback), but
        # its train/eval mode is the caller's business exactly as in the reference.
        self.model = model.to(self.cuda_device)
        if self.model.training:
            import warnings
            warnings.warn("Quantity: the model is in training mode (Dropout / un-merged BatchNorm would perturb the "
                          "statistics); the reference does not switch modes either -- call model.eval() first")
        self.input_size = tuple(int(v) for v in str(self.user_config["MODEL"]["INPUT_SHAPE"]).split(","))
        self.layers_num = 0
        self.name_to_param = OrderedDict()
        self.cache_bytes = cache_bytes
        self._begin_forward = lambda: None
        self._inplace_modified = set()
        self._fuse_calibration = True      # False: the calibration forward runs the model's own forwards only
        self.net_info = self.build_net_structure(self.model, self.input_size, self.device)
        self.cared_op_layer_names = self.get_cared_op_names(self.model)
        self._DKL_weight = False
        self.timings = {}

    def _log(self, *a):
        if self.verbose and self.rank == 0:
            print(*a)

    # ------------------------------------------------------------------ graph tracing
    def build_net_structure(self, model, input_size, device="cpu"):
        """One forward on torch.rand(INPUT_SHAPE) with a hook on every ALL_OP_TYPE module;
        tensors are named ``<Class>_<k>`` in hook firing order and linked producer -> consumer
        (reference :65-197, which links by a value hash; here by tensor identity)."""
        all_op_type = self._all_op_type
        allow_same = self._allow_same_tid_op_type
        net = OrderedDict()
        producer_of = {}            # id(tensor) -> tracer name of its latest producer
        keep_alive = []             # tensors stay referenced so ids cannot be recycled
        hooks = []
        orphan = []
        observed = []               # (tracer name, tensor, version at hook time): what calibration will record
        modules = OrderedDict()     # tracer name -> the module that fired

        def _hook(m, inputs, output):
            kind = type(m).__name__
            name = "%s_%i" % (kind, len(net) + 1)
            if name in net:
                raise NotImplementedError("module called twice (shared parameters): %s" % name)
            srcs = []
            for t in inputs:
                if not isinstance(t, torch.Tensor):
                    continue
                if id(t) in producer_of:
                    srcs.append(producer_of[id(t)])
                elif len(net) != 0:
                    orphan.append(name)       # only the first layer may read the network input
            if any(t is output for t in inputs if isinstance(t, torch.Tensor)) and kind not in allow_same:
                raise ValueError("Same input and output id, the op {} is useful?".format(name))
            if not net and inputs and isinstance(inputs[0], torch.Tensor):
                observed.append(("image", inputs[0], inputs[0]._version))
            net[name] = {"inputs": srcs, "type": kind}
            modules[name] = m
            producer_of[id(output)] = name    # in-place / pass-through ops take over the tensor
            keep_alive.append((inputs, output))
            if isinstance(output, torch.Tensor):
                observed.append((name, output, output._version))

        for m in model.modules():
            if type(m).__name__ in all_op_type:
                hooks.append(m.register_forward_hook(_hook))
        x = torch.rand(*input_size, device=self.cuda_device)
        with torch.no_grad():
            model(x)
        for h in hooks:
            h.remove()
        assert not orphan, "Can't find the input tensor of {} \n {}".format(orphan[0], net)
        self.layers_num = len(net)
        # Tensors a later in-place op (nn.ReLU(inplace=True), ``out += residual``) overwrites after their hook
        # fired.  The reference snapshots every hooked output to numpy at hook time (:509,:513), so it records the
        # pre-modification values; the calibration hooks below keep device references and therefore clone
        # exactly these tensors (and only these) to record the same values.
        self._inplace_modified = {n for n, t, v in observed if t._version != v}
        self._fusion_plan = plan_calibration_fusion(net, modules, self._inplace_modified)
        self._handover_plan = plan_calibration_handover(net, modules, self._fusion_plan)
        self._traced_modules = modules
        keep = [n for n, info in net.items() if info["type"] in self._cared_op_type]
        return self.prune_net_info(net, keep)

    def get_cared_op_names(self, model):
        return [name for name, module in model.named_modules()
                if type(module).__name__ in self._cared_op_type]

    def prune_net_info(self, net_info, keep_node_list):
        """Drop un-cared nodes and splice their (single) input through, so every cared node's
        inputs are cared nodes (reference :207-249)."""
        keep = set(keep_node_list)

        def resolve(name):
            while name is not None and name not in keep:
                ins = net_info[name]["inputs"]
                assert len(ins) <= 1, (ins, name)
                name = ins[0] if ins else None
            return name

        pruned = OrderedDict()
        for name, info in net_info.items():
            if name in keep:
                pruned[name] = {"inputs": [resolve(i) for i in info["inputs"]], "type": info["type"]}
        return pruned

    def get_merge_groups(self, net):
        """For every Eltwise / Concat (last first): the cared producers of its inputs
        (reference :298-341)."""
        merge_layer = [n for n, info in net.items() if info["type"] in self._merge_op_type]
        merge_layer.reverse()
        self._log("merge layers:", merge_layer)
        seen = set()

        def bottoms_of(name):
            if name in seen:
                return []
            seen.add(name)
            out = []
            for b in net[name]["inputs"]:
                if net[b]["type"] not in self._cared_op_type:
                    out.extend(bottoms_of(b))
                else:
                    out.append(b)
            return out

        groups = []
        for layer in merge_layer:
            names = bottoms_of(layer)
            self._log(layer, names)
            if names:
                groups.append(names)
        return groups

    # ---------------------------------------------------------------------- data input
    def preprocess(self, image):
        """Modes of reference :252-284: 1 = items of a loader ``(img, label)``; 2 = path of a
        .npy file.  Mode 0 (image files) is dead code in the reference (quirk Q3)."""
        option = int(self.user_config["PRE_PROCESS"]["IMG"])
        if option == 1:
            img, _ = image
            return img
        if option == 2:
            arr = torch.as_tensor(np.load(image))
            return arr.view(1, *arr.shape)
        raise NotImplementedError("PRE_PROCESS.IMG mode %r" % option)

    def net_forward(self, net, image_path):
        img = self.preprocess(image_path)
        if not img.is_cuda:
            img = img.to(self.cuda_device, non_blocking=True)
        self._forward_device(net, img)

    def _forward_device(self, net, img):
        self._begin_forward()
        with torch.no_grad():
            net(img)

    def _device_batches(self, images_files, skip=None):
        """This rank's batches as device tensors, ``(index, tensor or None)``: the host->device copy of
        batch i+1 is issued on a copy stream while batch i is being processed (pinned host batches
        overlap completely).  ``skip(index)`` true: nothing is copied and None is yielded."""
        dev = self.cuda_device
        copy_stream = None

        def stage(item):
            nonlocal copy_stream
            i, image = item
            if skip is not None and skip(i):
                return i, None, None
            img = self.preprocess(image)
            if img.is_cuda:
                return i, img, None
            if copy_stream is None:
                copy_stream = torch.cuda.Stream(dev)
            # The buffer comes from the compute stream's allocator pool (no cudaMalloc once the pool is warm);
            # the copy stream may touch it only after everything already queued on the compute stream.
            main = torch.cuda.current_stream(dev)
            staged = torch.empty(img.shape, dtype=img.dtype, device=dev)
            ready = torch.cuda.Event()
            ready.record(main)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ready)
                staged.copy_(img, non_blocking=True)
                done = torch.cuda.Event()
                done.record(copy_stream)
            return i, staged, done

        pending = None
        for item in self._my_batches(images_files):
            ahead = stage(item)
            if pending is not None:
                yield self._claim(pending)
            pending = ahead
        if pending is not None:
            yield self._claim(pending)

    def _claim(self, staged):
        i, img, done = staged
        if done is not None:
            torch.cuda.current_stream(self.cuda_device).wait_event(done)
        return i, img

    # --------------------------------------------------------------- activation hooks
    def regist_hook_outfeature(self, model):
        """Hooks that record 'image' and the output of every cared op of the current forward
        as device tensors (reference :491-524 copies them to numpy)."""
        out_feat = OrderedDict()
        hooks = []
        cared = self._cared_op_type
        state = {"idx": 0}
        versions = {}
        clone = self._inplace_modified
        self._feat_versions = versions
        self._feat_state = state

        def _begin():
            state["idx"] = 0
            out_feat.clear()
            versions.clear()

        def _keep(name, t):
            t = t.detach()
            if name in clone:
                t = t.clone()              # a later in-place op overwrites it (found by build_net_structure)
            out_feat[name] = t
            versions[name] = t._version

        def _hook(m, inputs, output):
            if state["idx"] >= self.layers_num:
                _begin()                   # a new forward started without _begin_forward (plain ``model(x)``, :497-500)
            if state["idx"] == 0:
                _keep("image", inputs[0])
            state["idx"] += 1
            kind = type(m).__name__
            if kind in cared:
                _keep("%s_%i" % (kind, state["idx"]), output)

        for m in model.modules():
            if type(m).__name__ in self._all_op_type:
                hooks.append(m.register_forward_hook(_hook))
        self._begin_forward = _begin
        return out_feat, hooks

    def _check_unmodified(self, feats):
        """The observed tensors are device references, not the host snapshots of the reference (:509,:513): a
        tensor modified in place after its hook fired would silently yield post-modification statistics."""
        for name, t in feats.items():
            v = self._feat_versions.get(name) if feats is self._named_feats_live else None
            if v is not None and t._version != v:
                raise RuntimeError(
                    "calibration tensor %r was modified in place after it was observed (nn.ReLU(inplace=True), "
                    "`out += residual`, ...) in a way the tracing forward did not show; the reference records "
                    "the value at hook time. Use out-of-place ops for data-dependent control flow." % name)

    def _my_batches(self, images_files):
        """Batches 0..MAX_CALI_IMG_NUM (reference :381), round-robin over data-parallel ranks."""
        for i, image in enumerate(images_files):
            if i > self._max_img_num:
                break
            if i % self.world_size == self.rank:
                yield i, image

    # ------------------------------------------------------------------- calibration
    def activation_quantize(self, images_files):
        settings = self.config["SETTINGS"]
        interval_num = settings["INTERVAL_NUM"]
        table_file = self.config["OUTPUT"]["FEAT_BIT_TABLE"]
        merge_groups = self.get_merge_groups(self.net_info)
        top_feat_names = ["image"] + list(self.net_info.keys())

        collector = DistributionCollector(top_feat_names, interval_num=interval_num,
                                          statistic=settings["STATISTIC"],
                                          worker_num=settings["WORKER_NUM"], device=self.cuda_device)
        quantizer = Quantizer(top_feat_names, worker_num=settings["WORKER_NUM"], device=self.cuda_device)
        named_feats, hooks = self.regist_hook_outfeature(self.model)
        self._named_feats_live = named_feats

        # HBM activation cache for pass 2
        budget = self.cache_bytes
        if budget is None:
            free, _total = torch.cuda.mem_get_info(self.cuda_device)
            # memory the caching allocator already holds but is not using is just as available
            pooled = torch.cuda.memory_reserved(self.cuda_device) - torch.cuda.memory_allocated(self.cuda_device)
            budget = int((free + pooled) * 0.6)
        cache, cached_bytes, n_cached = {}, 0, 0

        t0 = time.perf_counter()
        n_mine = 0
        plan = self._fusion_plan if self._fuse_calibration else {}
        # max slots only for the tensors the collector observes (CARE_OP_TYPE); the other fused ops take no max
        slots = {n: collector._max_slot(n) for n in plan if n in top_feat_names}
        handover = self._handover_plan if self._fuse_calibration else ({}, {})
        fusion = _CalibrationFusion(plan, handover, self._traced_modules, self._feat_state, slots,
                                    collector.device_state()[0] if slots else None, self.cuda_device)
        try:
            fusion.install()
            fusion.collect = True
            for i, img in self._device_batches(images_files):                    # pass 1  (:379-390)
                fusion.reduced.clear()
                fusion.begin()
                self._forward_device(self.model, img)
                self._check_unmodified(named_feats)
                feats = {n: named_feats[n] for n in top_feat_names}
                fusion.fold()
                collector._refresh_max_val_except(feats, fusion.reduced)
                nbytes = sum(t.numel() * t.element_size() for t in feats.values())
                if cached_bytes + nbytes <= budget:
                    cache[i] = feats
                    cached_bytes += nbytes
                    n_cached += 1
                n_mine += 1
            if n_mine == 0:
                collector.refresh_max_val({n: torch.zeros(0, device=self.cuda_device) for n in top_feat_names})
            collector.all_reduce_max()
            self._log("max_vals", collector.max_vals)
            distribution_intervals = collector.distribution_intervals
            t1 = time.perf_counter()

            def group_has_eltwise(names):
                return any(self.net_info[n]["type"] == "Eltwise" for n in names)

            for names in merge_groups:                                           # (:396-411)
                assert len(names) > 1
                if group_has_eltwise(names):
                    continue
                widest = 0
                for n in names:
                    widest = max(widest, distribution_intervals[n])
                for n in names:
                    distribution_intervals[n] = widest

            self._log("Collect histograms of activations:")
            fusion.collect = False
            for i, img in self._device_batches(images_files, skip=lambda i: i in cache):   # pass 2  (:415-426)
                if img is None:
                    feats = cache.pop(i)
                else:
                    fusion.begin()
                    self._forward_device(self.model, img)
                    self._check_unmodified(named_feats)
                    feats = {n: named_feats[n] for n in top_feat_names}
                collector.add_to_distributions(feats)
            if n_mine == 0:
                collector.add_to_distributions({n: torch.zeros(0, device=self.cuda_device) for n in top_feat_names})
            cache.clear()
            collector.all_reduce_hist()
        finally:
            fusion.remove()
            for h in hooks:
                h.remove()
        named_feats.clear()                # the last forward's activations (4.3 GB for ResNet-50 at batch 64) go back to the pool
        distributions = collector.distributions
        t2 = time.perf_counter()

        for names in merge_groups:                                           # (:432-445)
            if group_has_eltwise(names):
                continue
            total = np.zeros(interval_num)
            for n in names:
                total += distributions[n]
            for n in names:
                distributions[n] = total

        quantizer.quantize(distributions, distribution_intervals)           # (:448)
        bits = quantizer.bits
        for names in merge_groups:                                           # (:453-465)
            elt_idx, found = 0, False
            for i, n in enumerate(names):
                if self.net_info[n]["type"] == "Eltwise":
                    elt_idx, found = i, True
            if found:
                conv_id = 1 - elt_idx                                        # 2-member groups (quirk Q4)
                self._log("bit conv:eltwise ", bits[names[conv_id]], bits[names[elt_idx]])
                bits[names[conv_id]] = bits[names[elt_idx]]
        t3 = time.perf_counter()

        lines, first = [], True                                              # (:468-489)
        for i, feat_name in enumerate(top_feat_names):
            if feat_name == "image":
                line = "image " + str(bits["image"])
            elif first:
                line = self.cared_op_layer_names[i - 1] + " " + str(bits[feat_name]) + " " + str(bits["image"])
                first = False
            elif len(self.net_info[feat_name]["inputs"]) > 0:
                line = self.cared_op_layer_names[i - 1] + " " + str(bits[feat_name])
                for inp in self.net_info[feat_name]["inputs"]:
                    line += " " + str(bits[inp])
            else:
                raise NotImplementedError(self.net_info[feat_name])
            lines.append(line)
        if self.rank == 0:
            with open(table_file, "w") as f:
                for line in lines:
                    f.write(line + "\n")
        _barrier()
        self.timings.update(pass1_s=t1 - t0, pass2_s=t2 - t1, kl_s=t3 - t2,
                            batches=n_mine, cached_batches=n_cached, cached_bytes=cached_bytes)
        self.last_calibration = dict(bits=dict(bits), intervals=dict(distribution_intervals),
                                     thresholds=dict(quantizer.threshold_value),
                                     threshold_bins=dict(quantizer.threshold_bin),
                                     distributions=distributions, max_vals=dict(collector.max_vals),
                                     top_feat_names=top_feat_names, merge_groups=merge_groups,
                                     table_lines=lines)
        return lines

    # -------------------------------------------------------------------------- files
    def init_dir(self):
        out = self.config["OUTPUT"]
        if self.rank == 0:
            for key in ("WORK_DIR", "WEIGHT_DIR", "BIAS_DIR", "FINAL_WEIGHT_DIR", "FINAL_BIAS_DIR"):
                os.makedirs(out[key], exist_ok=True)
        _barrier()

    def rewrite_weight(self):
        """Align bias bits to the output bits and cap the shift (reference :553-590)."""
        if self.rank == 0:
            self._rewrite_weight_rank0()
        _barrier()

    def _rewrite_weight_rank0(self):
        out = self.config["OUTPUT"]
        rewriter = BiasReWriter(out["WEIGHT_DIR"], out["BIAS_DIR"], out["FINAL_WEIGHT_DIR"],
                                out["FINAL_BIAS_DIR"], out["WEIGHT_BIT_TABLE"], out["FEAT_BIT_TABLE"],
                                max_shift_limit=self.config["SETTINGS"]["MAX_SHIFT"])
        weight_bits, bias_bits = rewriter.get_weight_info()
        feat_bits, infeat_bits = rewriter.get_feat_info()
        unmatched = set(bias_bits) ^ set(feat_bits)
        if unmatched:
            self._log("These layers not include params but we care about their features:", unmatched)
        self._log("Align bias bit:")
        rewriter.rewrite_bias_table(bias_bits, feat_bits)
        rewriter.rewrite_bias_dir(bias_bits, feat_bits)
        self._log("Add max shift limitation:")
        need, new_weight = rewriter.max_shift_limit_weight(feat_bits, infeat_bits, weight_bits)
        if need:
            self._log("rewirte weight!!!!")
            rewriter.rewrite_weight_table(weight_bits, new_weight)
            rewriter.rewrite_weight_dir(weight_bits, new_weight)
        self._log("Done!")

    def weight_quantize(self, write_json=True):
        """Per-parameter max-abs -> bit, int8 values -> JSON, weight.table (reference :592-677).
        The max-abs of all parameters is one multi-tensor kernel launch; rounding / clamping is
        the fake-quant kernel without the dequantise step.  ``write_json=False`` (not a reference option) writes
        only weight.table -- all that Reconstruction needs -- and skips the per-parameter JSON files and the
        rewriter pass over them, which are 100 % host serialisation time."""
        settings, out = self.config["SETTINGS"], self.config["OUTPUT"]
        names, shapes, flats = [], {}, []
        for name, param in self.model.named_parameters():
            if not name.endswith("weight") and not name.endswith("bias"):
                print("[WARNING]", " not supported param: {}".format(name))
                continue
            module = self.model
            for part in name.split(".")[:-1]:
                module = getattr(module, part)
            data = param.detach()
            if name.endswith("weight") and isinstance(module, nn.Conv2d):
                if module.dilation != (1, 1) and not settings["SUPPORT_DILATION"]:
                    data = self.dilation_to_zero_padding(data, module.dilation)
            names.append(name)
            shapes[name] = tuple(data.shape)
            flats.append(data.contiguous().view(-1).float())

        collector = DistributionCollector(names, interval_num=settings["INTERVAL_NUM"],
                                          statistic=settings["STATISTIC"], device=self.cuda_device)
        params = dict(zip(names, flats))
        collector.refresh_max_val(params)
        max_vals = collector.max_vals
        self._log("max vals:", max_vals)
        bits_co = {}
        if self._DKL_weight:                                                 # (:644-648)
            quantizer = Quantizer(names, device=self.cuda_device)
            collector.add_to_distributions(params)
            quantizer.quantize(collector.distributions, collector.distribution_intervals)
            bits_co = quantizer.bits
        else:
            for name in names:                                               # (:650-653)
                bits_co[name] = int(8 - 1 - math.ceil(math.log(max_vals[name], 2)))

        table, writes = [], []
        for name in names:
            bit = bits_co[name]
            q = _native.fakequant(params[name], bit, -128.0, 127.0, dequant=False)   # around + clip
            table.append(name + " " + str(bit))
            if self.rank != 0 or not write_json:
                continue
            content = q.to(torch.int32).view(shapes[name]).cpu().numpy()
            if name.endswith("weight"):
                writes.append((content, os.path.join(out["WEIGHT_DIR"], name + ".json")))
            elif name.endswith("bias"):
                writes.append((content, os.path.join(out["BIAS_DIR"], name + ".json")))
            else:
                raise NotImplementedError(name)
        if writes:
            # the files are independent and the writer is numpy (the GIL is released in its large array operations):
            # a few host threads, largest tensors first
            writes.sort(key=lambda w: -w[0].size)
            workers = max(1, min(8, os.cpu_count() or 1, len(writes)))
            if workers == 1:
                for content, path in writes:
                    dump_int_array(content, path)
            else:
                from concurrent.futures import ThreadPoolExecutor
                with ThreadPoolExecutor(workers) as pool:
                    list(pool.map(lambda w: dump_int_array(*w), writes))
        if self.rank == 0:
            with open(out["WEIGHT_BIT_TABLE"], "w") as f:
                for line in table:
                    f.write(line + "\n")
        _barrier()
        if write_json:
            self.rewrite_weight()

    def dilation_to_zero_padding(self, tensor, dilation):
        """Zero-stuff a dilated kernel (reference :679-693); dilation (2, 2) only."""
        assert tensor.shape[2] == tensor.shape[3] and tuple(dilation) == (2, 2), "Not support."
        k = tensor.shape[2]
        out = torch.zeros(tensor.shape[0], tensor.shape[1], 2 * k - 1, 2 * k - 1,
                          dtype=torch.float32, device=tensor.device)
        out[..., ::2, ::2] = tensor
        return out

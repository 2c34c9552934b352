"""Int8 inter-layer pipeline for the integer simulation (SURVEY.md 8(f) n1; opt-in).

The reference's ``NewConv2d`` de-quantises its result to fp32 NCHW and the next ``NewConv2d``
quantises it again (new_quantity_op.py:124-133).  In feat.table a layer's input bit IS its producer's
output bit (tools/pytorch_quantizer.py:468-485), so that round trip is the identity on the int8
values: ``Quantity(ib)(y / 2^ob) == y`` when ``ib == ob``.  With the pipeline enabled the tensor-core
layers hand each other int8 NHWC payloads wrapped in a lazy ``QTensor``:

    NewConv2d -> QTensor(int8 NHWC, bit)            epilogue stores int8 (ReLU fused when it follows)
    nn.ReLU / nn.MaxPool2d on a QTensor             stay int8 (both commute with the monotone quantiser)
    NewAdd(QTensor, QTensor)                        exact integer sum: int16 (for the next identity
                                                    shortcut) + int8 at the Eltwise's feat bit (for convs);
                                                    evaluated lazily so that a following nn.ReLU is fused
    Concat(QTensor, QTensor) / torch.cat(dim=1)     lazy: the consuming NewConv2d asks for the concatenation at
                                                    ITS input bit and one bandwidth kernel (pq_concat_requant_s8)
                                                    writes the channel-padded int8 NHWC operand directly
    anything else (AvgPool2d, user code)            the QTensor de-quantises itself to fp32 NCHW first

so the final output is bit-identical to the fp32-boundary model while HBM traffic drops ~4x.
``enable_int8_pipeline(model)`` turns it on for a model built by ``Reconstruction.ReconModel``.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _native


# NewConv2d + NewAdd (+ ReLU) in one kernel (pq_conv2d_s8_add): the convolution's int8 result never touches
# memory.  Bit-identical to conv followed by pq_add_requant; on ResNet-50 batch 512 the 16 fused launches take
# 3.02 ms against 1.19 + 2.52 ms for the separate kernels (forward 6.83 -> 6.19 ms), so it is on by default.
# PQ_FUSE_ADD=0 switches it off (A/B measurements).
import os as _os
FUSE_ADD_INTO_CONV = _os.environ.get("PQ_FUSE_ADD", "1") != "0"

_METADATA = {"__get__", "size", "dim", "numel", "element_size", "ndimension", "is_floating_point", "__len__",
             "get_device", "is_complex", "nelement"}


class _LazyConv:
    """A NewConv2d whose kernel has not run yet.  It runs when the first consumer asks for the int8 payload, by
    which time it is known whether an nn.ReLU was applied in between: that ReLU is then fused into the conv
    epilogue.  The decision is taken per request, not from module adjacency, so whoever observes the conv's OWN
    output (a forward hook on the NewConv2d, ``seq[0](x)`` on its own, a sliced Sequential) still gets pre-ReLU
    values, exactly like the fp32-boundary model.  If the only consumer is a NewAdd, the add (and the ReLU after
    it) can run inside the conv's epilogue and the conv result never touches memory."""

    def __init__(self, mod, operand):
        self.mod, self.operand = mod, operand          # the NewConv2d and its operand (see NewConv2d._quantize)
        self.out = {}                                  # relu -> int8 NHWC payload

    def get(self, relu):
        if relu not in self.out:
            if relu and False in self.out:             # both asked for (rare): ReLU of the payload already there
                self.out[True] = _native.relu_s8(self.out[False])
            else:
                self.out[relu] = self.mod._run(self.operand, False, True, relu)[1]
        return self.out[relu]


class _LazyAdd:
    """A NewAdd whose kernel has not run yet: it runs when the first consumer asks for a payload, by
    which time it is known whether an nn.ReLU sits between the Eltwise and that consumer.

    It also writes only the payloads somebody reads.  The exact int16 sum is needed by an identity
    shortcut (the next NewAdd) or a de-quantising consumer; the int8 requantisation by convolutions.  Which
    of the two a given Eltwise feeds is a property of the (static) model, so the module keeps a census of
    the kinds requested in earlier forwards (``mod._pipe_seen``) and the kernel skips the other output --
    at the end of a ResNet stage nobody reads the int16 sum, which saves 2 of 6 bytes per element there.
    A request for a kind that was not produced simply re-runs the kernel with both (first forward only)."""

    def __init__(self, x, y, q_bit, mod=None):
        self.x, self.y = x, y                          # operand QTensors (not yet materialised)
        self.q_bit = q_bit
        self.mod = mod
        self.done = {}                                 # relu -> {"s16": tensor, "q8": tensor}

    @staticmethod
    def _fusable(t):
        lc = t._lazy_conv
        return FUSE_ADD_INTO_CONV and lc is not None and lc.mod._fuses_add and not lc.out and not t.relu_pending

    def get(self, relu, kind):
        """kind: "s16" (exact sum) or "q8" (Quantity(q_bit) of it).  Returns the dict of payloads held."""
        seen = getattr(self.mod, "_pipe_seen", None) if self.mod is not None else None
        have = self.done.get(relu)
        if have is None or kind not in have:
            wants = set(seen) if seen else set()
            wants.add(kind)
            if have:                                   # a second kind after all: produce both
                wants = {"s16", "q8"}
            want16, want8 = "s16" in wants, "q8" in wants
            x, y = self.x, self.y
            if not self._fusable(x) and self._fusable(y):
                x, y = y, x
            if self._fusable(x):                       # conv + add (+ relu) in one kernel (always writes int8)
                lc = x._lazy_conv
                sc, sc_bit, sc_relu = _operand(y)
                s16, q8 = lc.mod._run_add(lc.operand, sc, sc_bit, sc_relu, self.q_bit, relu, want16)
            else:
                (a, abit, arelu), (b, bbit, brelu) = _operand(x), _operand(y)
                s16, q8 = _native.add_requant(a, abit, arelu, b, bbit, brelu, self.q_bit, want16=want16,
                                              want8=want8, out_relu=relu)
            have = {}
            if s16 is not None:
                have["s16"] = s16
            if q8 is not None:
                have["q8"] = q8
            self.done[relu] = have
        if seen is not None:
            seen.add(kind)
        return have


class _LazyCat:
    """torch.cat(members, 1) that has not run yet.  The reference leaves Concat in fp32
    (tools/reconstruction.py:219-238) and the consumer's Quantity(ib) quantises the result, so the exact
    int8 operand is ``clamp(rint(member * 2^ib))`` per member -- computed here from the members' most
    exact integer payloads once the consumer (and so ib and its channel padding) is known."""

    def __init__(self, members):
        self.members = []                              # (QTensor, extra_relu), nested concatenations flattened
        for m in members:
            if m._lazy_cat is not None:
                self.members += [(t, r or m.relu_pending) for t, r in m._lazy_cat.members]
            else:
                self.members.append((m, False))
        self.done = {}

    def supported(self, q_bit):
        return len(self.members) <= _native.CONCAT_MAX_SOURCES and all(
            t.exact_bit() is not None and abs(q_bit - t.exact_bit()) <= 15 for t, _ in self.members)

    def get(self, q_bit, c_pad, relu):
        key = (q_bit, c_pad, relu)
        if key not in self.done:
            srcs = []
            for t, extra in self.members:
                payload, bit, r = _operand(t)
                srcs.append((payload, bit, r or extra or relu))
            self.done[key] = _native.concat_requant_s8(srcs, q_bit, c_pad)
        return self.done[key]

    def dequantize(self):
        parts = [torch.relu(t.dequantize()) if extra else t.dequantize() for t, extra in self.members]
        return torch.cat(parts, 1)


class QTensor(torch.Tensor):
    """A float32 NCHW tensor that exists only as quantised payloads until somebody needs the floats."""

    @staticmethod
    def __new__(cls, shape, device, **kw):
        return torch.Tensor._make_wrapper_subclass(cls, shape, dtype=torch.float32, device=device,
                                                   requires_grad=False)

    def __init__(self, shape, device, q8=None, q8_bit=None, s16=None, s16_bit=None, relu_pending=False,
                 nonneg=False, lazy=None, lazy_conv=None, lazy_cat=None):
        self.channels = int(shape[1])                  # plain attribute: tensor.shape on a subclass costs a dispatch
        self._q8, self.q8_bit = q8, q8_bit             # int8 NHWC, value = q8 / 2^q8_bit (after pending relu)
        self._s16, self.s16_bit = s16, s16_bit         # int16 NHWC exact value (outputs of NewAdd)
        self.relu_pending = relu_pending               # a ReLU was applied logically but not to the payloads
        self.nonneg = nonneg                           # payloads are already >= 0
        self._lazy = lazy                              # _LazyAdd: payloads appear on first use
        self._lazy_conv = lazy_conv                    # _LazyConv: the int8 payload appears on first use
        self._lazy_cat = lazy_cat                      # _LazyCat: payload exists per (consumer bit, padding)
        self._q8_relu = None

    def exact_bit(self):
        """Fractional bit of the most exact payload, without materialising anything."""
        return self.s16_bit if self.s16_bit is not None else self.q8_bit

    def _materialize(self, kind):
        if self._lazy_conv is not None:
            relu = self.relu_pending
            self._q8 = self._lazy_conv.get(relu)       # a pending ReLU is applied by the conv epilogue
            self._lazy_conv = None
            self._q8_relu = None
            self.nonneg = self.nonneg or relu
        if self._lazy is not None and (self._s16 if kind == "s16" else self._q8) is None:
            relu = self.relu_pending
            have = self._lazy.get(relu, kind)           # the pending ReLU is applied by the add kernel
            self._s16, self._q8 = have.get("s16"), have.get("q8")   # one provenance: never mix relu / non-relu
            self._q8_relu = None
            self.nonneg = self.nonneg or relu

    def has_q8(self):
        """An int8 payload exists or can be produced (no kernel runs)."""
        return self._q8 is not None or self._lazy is not None or self._lazy_conv is not None

    @property
    def q8(self):
        self._materialize("q8")
        return self._q8

    @property
    def s16(self):
        if self.s16_bit is None:
            return None
        self._materialize("s16")
        return self._s16

    def __repr__(self):
        return "QTensor(shape=%s, q8_bit=%s, s16_bit=%s, relu_pending=%s)" % (
            tuple(self.shape), self.q8_bit, self.s16_bit, self.relu_pending)

    # ---- payload access -------------------------------------------------------------------
    def int8_payload(self):
        """int8 NHWC with any pending ReLU applied (materialised once)."""
        self._materialize("q8")
        if not self.relu_pending or self.nonneg:
            return self.q8
        if self._q8_relu is None:
            self._q8_relu = _native.relu_s8(self.q8)
        return self._q8_relu

    def dequantize(self):
        """fp32 NCHW, exactly what the fp32-boundary model would hold here (cold path: plain torch ops)."""
        if self._lazy_cat is not None:
            v = self._lazy_cat.dequantize()
            return torch.relu(v) if self.relu_pending else v
        if self.s16_bit is not None:
            v = self.s16.to(torch.float32) * (2.0 ** -self.s16_bit)
        else:
            v = self.q8.to(torch.float32) * (2.0 ** -self.q8_bit)
        if self.relu_pending and not self.nonneg:
            v = torch.relu(v)
        return v.permute(0, 3, 1, 2).contiguous()

    def with_relu(self):
        if self.nonneg:
            return self
        return QTensor(self.shape, self.device, q8=self._q8, q8_bit=self.q8_bit, s16=self._s16,
                       s16_bit=self.s16_bit, relu_pending=True, lazy=self._lazy, lazy_conv=self._lazy_conv,
                       lazy_cat=self._lazy_cat)

    # ---- dispatch -------------------------------------------------------------------------
    @classmethod
    def __torch_dispatch__(cls, func, types, args=(), kwargs=None):
        # ATen-level calls that slipped past __torch_function__: compute on the de-quantised floats
        return func(*_plain_tree(args), **_plain_tree(kwargs or {}))

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        if func in (F.relu, torch.relu, torch.Tensor.relu) and isinstance(args[0], QTensor) \
                and not kwargs.get("inplace", False) and len(args) == 1:
            return args[0].with_relu()
        if func is torch.cat:
            out = _concat(*args, **kwargs)
            if out is not None:
                return out
        if func is F.max_pool2d and isinstance(args[0], QTensor):
            out = _maxpool(args[0], *args[1:], **kwargs)
            if out is not None:
                return out
        if func is F.avg_pool2d and isinstance(args[0], QTensor):
            out = _avgpool(args[0], *args[1:], **kwargs)
            if out is not None:
                return out
        # metadata queries are answered by the wrapper itself (no payload is touched)
        if getattr(func, "__name__", "") in _METADATA:
            with torch._C.DisableTorchFunctionSubclass():
                return func(*args, **kwargs)

        def plain(a):
            if isinstance(a, QTensor):
                return a.dequantize()
            if isinstance(a, (list, tuple)):
                return type(a)(plain(v) for v in a)
            return a

        with torch._C.DisableTorchFunctionSubclass():
            return func(*plain(args), **{k: plain(v) for k, v in kwargs.items()})


def _plain_tree(obj):
    from torch.utils._pytree import tree_map
    return tree_map(lambda a: a.dequantize() if isinstance(a, QTensor) else a, obj)


def _pair(v):
    return (v, v) if isinstance(v, int) else tuple(v)


def _concat(tensors, dim=0, out=None):
    """torch.cat of QTensors along the channel axis stays quantised (lazily, see _LazyCat)."""
    if out is not None or dim not in (1, -3) or not isinstance(tensors, (list, tuple)) or len(tensors) < 1:
        return None
    if not all(isinstance(t, QTensor) and t.dim() == 4 for t in tensors):
        return None
    first = tensors[0]
    if any(t.shape[0] != first.shape[0] or t.shape[2:] != first.shape[2:] for t in tensors):
        return None
    if any(t._lazy_cat is None and t.exact_bit() is None for t in tensors):
        return None
    lazy = _LazyCat(tensors)
    if len(lazy.members) > _native.CONCAT_MAX_SOURCES:
        return None
    shape = (first.shape[0], sum(t.shape[1] for t in tensors), first.shape[2], first.shape[3])
    return QTensor(shape, first.device, lazy_cat=lazy, nonneg=all(t.nonneg for t in tensors))


def _maxpool(x, kernel_size, stride=None, padding=0, dilation=1, ceil_mode=False, return_indices=False):
    k, s, p = _pair(kernel_size), _pair(stride if stride is not None else kernel_size), _pair(padding)
    if k[0] != k[1] or s[0] != s[1] or p[0] != p[1] or _pair(dilation) != (1, 1) or ceil_mode or return_indices:
        return None
    if not x.has_q8() or x.channels % 16:               # payload channels == logical channels
        return None
    q8 = x.q8
    relu = x.relu_pending and not x.nonneg
    y = _native.maxpool_nhwc_s8(q8, k[0], s[0], p[0], relu=relu)
    N, P, Q, C = y.shape
    return QTensor((N, x.shape[1], P, Q), x.device, q8=y, q8_bit=x.q8_bit, nonneg=x.nonneg or relu)


def _avgpool(x, kernel_size, stride=None, padding=0, ceil_mode=False, count_include_pad=True, divisor_override=None):
    """F.avg_pool2d over the WHOLE plane (ResNet's AvgPool2d before the classifier) straight from the most exact
    payload: fp32 [N][C][1][1], bit-identical to pooling the de-quantised tensor (pq_avgpool_global_nhwc_f32)."""
    k = _pair(kernel_size)
    if k != (x.shape[2], x.shape[3]) or _pair(padding) != (0, 0) or divisor_override is not None:
        return None
    if x._lazy_cat is not None or x.channels % 8:
        return None
    relu = x.relu_pending                          # (read before a lazy producer consumes it)
    if x.s16_bit is not None:
        payload, bit = x.s16, x.s16_bit
    elif x.has_q8():
        payload, bit = x.q8, x.q8_bit
    else:
        return None
    if payload.shape[3] != x.channels:             # padded payload channels
        return None
    return _native.avgpool_global_nhwc(payload, bit, relu=relu and not x.nonneg)


def conv_forward(mod, x):
    """NewConv2d.forward in pipeline mode: the operand is the producer's int8 payload, the lazy concatenation at this
    layer's input bit, or else the layer's own quantiser applied to the de-quantised input."""
    c = mod._payload_channels
    operand = None
    if isinstance(x, QTensor):
        if x._lazy_cat is not None:
            if c is not None and x.channels <= c and x._lazy_cat.supported(mod.input_bit):
                operand = x._lazy_cat.get(mod.input_bit, c, x.relu_pending and not x.nonneg)  # Concat + Quantity(ib)
        elif c is not None and x.has_q8() and x.q8_bit == mod.input_bit and x.channels == c:
            operand = x.int8_payload()                           # Quantity(ib) is the identity here
    if operand is None:
        if isinstance(x, QTensor):
            x = x.dequantize()
        operand, device = mod._quantize(x), x.device
    else:
        device = operand.device
    # deferred: the ReLU that may follow is fused on demand, and a NewAdd consumer can absorb the whole convolution
    return QTensor(mod._out_shape(operand), device, q8_bit=mod.output_bit, lazy_conv=_LazyConv(mod, operand))


def _operand(t):
    """(payload, bit, relu) of the most exact representation of a QTensor."""
    if t.s16_bit is not None:
        payload, bit = t.s16, t.s16_bit                # (materialises a lazy add, fusing its ReLU)
    else:
        payload, bit = t.q8, t.q8_bit
    return payload, bit, t.relu_pending and not t.nonneg


def add_forward(mod, x, y):
    """NewAdd.forward in pipeline mode; returns None when the operands are not both quantised."""
    if not (isinstance(x, QTensor) and isinstance(y, QTensor)) or x.shape != y.shape:
        return None
    q_bit = getattr(mod, "output_bit", None)
    abit, bbit = x.exact_bit(), y.exact_bit()
    if q_bit is None or abit is None or bbit is None:
        return None
    o_bit = max(abit, bbit)
    if not (0 <= o_bit <= 7) or o_bit - min(abit, bbit) > 7 or abs(q_bit - o_bit) > 15:
        return None
    if not hasattr(mod, "_pipe_seen"):
        mod._pipe_seen = set()                         # payload kinds this Eltwise's consumers have asked for
    return QTensor(x.shape, x.device, q8_bit=q_bit, s16_bit=o_bit, lazy=_LazyAdd(x, y, q_bit, mod))


def enable_int8_pipeline(model, enabled=True):
    """Switch a ReconModel to the int8 inter-layer pipeline (or back).  Nothing is decided from module adjacency:
    a ReLU after a convolution is fused into its epilogue when the (lazy) convolution finally runs for a consumer
    that sits behind that ReLU (see _LazyConv)."""
    from .new_quantity_op import NewAdd, NewConv2d
    for m in model.modules():
        if isinstance(m, (NewConv2d, NewAdd)):
            m.int8_pipeline = enabled
    return model


class GraphedForward:
    """One captured forward of a (pipeline-enabled) ReconModel for a fixed input shape, replayed as a
    CUDA graph: the ~90 kernel launches, tensor-map encodes and Python dispatch of a ResNet-50 forward
    collapse into one graph launch.  The arithmetic is the captured kernels', so outputs are unchanged.

        fwd = GraphedForward(model, example_batch);  y = fwd(batch)      # y is overwritten by the next call
    """

    def __init__(self, model, example, warmup=2):
        if not example.is_cuda:
            raise RuntimeError("GraphedForward needs a CUDA example batch: no CPU fallback")
        self.model = model
        self.static_in = example.detach().clone()
        with torch.no_grad():
            side = torch.cuda.Stream(device=example.device)
            side.wait_stream(torch.cuda.current_stream(example.device))
            with torch.cuda.stream(side):
                for _ in range(warmup):                # lazy one-time setup must not land in the capture
                    model(self.static_in)
            torch.cuda.current_stream(example.device).wait_stream(side)
            torch.cuda.synchronize(example.device)
            self.graph = torch.cuda.CUDAGraph()
            l0 = _native.LAUNCHES["total"]
            with torch.cuda.graph(self.graph):
                self.static_out = model(self.static_in)
            self.launches = _native.LAUNCHES["total"] - l0     # kernels of this library inside the graph

    def __call__(self, x):
        if x.shape != self.static_in.shape:
            raise RuntimeError("GraphedForward was captured for shape %s" % (tuple(self.static_in.shape),))
        self.static_in.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.static_out

"""Activation / weight statistics on the GPU (subsystem 1).

Drop-in for the reference class (quantity/common/quantity/distribution_collector.py:7-147):
same constructor, same ``refresh_max_val`` / ``add_to_distributions`` calls, same
``max_vals`` / ``distribution_intervals`` / ``distributions`` properties and the same
"call-first" asserts -- but the running maxima and the 2048-bin histograms live in HBM and
are updated by two multi-tensor sm_100a kernels (pq_absmax_multi_f32,
pq_hist2048_multi_f32) instead of numpy reductions and a per-element Python loop fanned out
over a multiprocessing.Pool.  Values of the ``tensors`` dict may be CUDA tensors (the fast
path: nothing leaves the device) or numpy arrays / CPU tensors (uploaded once).

State kept on the device:
  _max_bits  int32 [n]        bit pattern of the running max |x| (order-free atomicMax)
  _hist      int64 [n][2048]  running counts (order-free atomicAdd)
so the merge over data-parallel ranks is ``all_reduce(MAX)`` / ``all_reduce(SUM)`` on these two
buffers (``all_reduce_max`` / ``all_reduce_hist``) and is bit-identical for any rank count.
"""
import numpy as np
import torch

from . import _native


class DistributionCollector:

    def __init__(self, tensor_list, interval_num=2048, statistic=1, worker_num=1, debug=False,
                 device=None):
        # INTERVAL_NUM is a configuration value in the reference (tools/configs.yml:23); 2048 runs the specialised
        # histogram kernel, any other count up to 8192 the generic one
        if int(interval_num) != interval_num or not (1 <= interval_num <= _native.HIST_BINS_MAX):
            raise ValueError("INTERVAL_NUM must be an integer in [1, %d] (PQ_EUNSUPPORTED beyond: shared-memory "
                             "histogram), got %r" % (_native.HIST_BINS_MAX, interval_num))
        interval_num = int(interval_num)
        self._tensor_list = tensor_list
        self._interval_num = interval_num
        self._statistic = statistic
        self._worker_num = worker_num        # accepted for compatibility; the GPU needs no pool
        self._debug = debug
        self._device = torch.device(device) if device is not None else None
        self._max_bits = None
        self._hist = None
        self._max_vals = {name: 0 for name in tensor_list}
        self._distributions = {}
        self._max_dirty = False
        self._hist_dirty = False
        self._max_vals_refreshed_flag = False
        self._added_to_distributions_flag = False

    # ------------------------------------------------------------------ device state
    def _ensure_state(self, sample):
        if self._max_bits is not None:
            return
        if self._device is None:
            if isinstance(sample, torch.Tensor) and sample.is_cuda:
                self._device = sample.device
            else:
                if not torch.cuda.is_available():
                    raise RuntimeError("no CUDA device: DistributionCollector has no CPU fallback")
                self._device = torch.device("cuda", torch.cuda.current_device())
        n = len(self._tensor_list)
        self._max_bits = torch.zeros(n, dtype=torch.int32, device=self._device)
        self._hist = torch.zeros((n, self._interval_num), dtype=torch.int64, device=self._device)

    def _gather(self, tensors, skip=()):
        """The tensors as flat fp32 device tensors in tensor_list order; those named in `skip` as empty ones."""
        first = next(iter(tensors.values())) if len(tensors) else None
        self._ensure_state(first)
        empty = torch.empty(0, device=self._device) if skip else None
        return [empty if name in skip else _native.to_device_f32(tensors[name], self._device)
                for name in self._tensor_list]

    # ------------------------------------------------------------------- reference API
    @property
    def max_vals(self):
        assert self._max_vals_refreshed_flag, "Please use refresh_max_val() first."
        if self._max_dirty:
            vals = self._max_bits.view(torch.float32).cpu().numpy()     # one D2H per pass
            for name, v in zip(self._tensor_list, vals):
                # the reference's ``max(0, np.float32)`` keeps the python int 0 until a value exceeds it
                self._max_vals[name] = np.float32(v) if v > 0 else 0
            self._max_dirty = False
        return self._max_vals

    @property
    def distribution_intervals(self):
        """Bin width per tensor: statistic * max / interval_num + 1e-12, an np.float32 under
        numpy-2 promotion exactly as in distribution_collector.py:60-61."""
        assert self._max_vals_refreshed_flag, "Please use refresh_max_val() first."
        max_vals = self.max_vals
        intervals = {}
        for name in self._tensor_list:
            intervals[name] = self._statistic * max_vals[name] / self._interval_num + 1e-12
        self._distribution_intervals = intervals
        return intervals

    @property
    def distributions(self):
        assert self._added_to_distributions_flag, "Please use add_to_distributions() first."
        if self._hist_dirty:
            h = self._hist.cpu().numpy()                                  # one D2H per pass
            fits = int(h.max(initial=0)) < 2 ** 31
            for i, name in enumerate(self._tensor_list):
                # int32 like distribution_collector.py:41 whenever the counts fit
                self._distributions[name] = h[i].astype(np.int32) if fits else h[i].copy()
            self._hist_dirty = False
        return self._distributions

    def refresh_max_val(self, tensors):
        """Pass 1: running max |x| of every tensor (distribution_collector.py:70-78)."""
        self._refresh_max_val_except(tensors, ())

    def _refresh_max_val_except(self, tensors, reduced):
        """refresh_max_val for the tensors not named in `reduced`: those already went into their max_bits slots
        (max_slot) while they were computed, the fused ops of the calibration forward.  They stay in the one
        absmax_multi launch as empty segments."""
        self._max_vals_refreshed_flag = True
        _native.absmax_multi(self._gather(tensors, reduced), self._max_bits)
        self._max_dirty = True

    def _max_slot(self, name):
        """Device address of the int32 max_bits slot of tensor `name`: the max_slot of a fused op."""
        self._ensure_state(None)
        return self._max_bits.data_ptr() + 4 * self._tensor_list.index(name)

    def add_to_distributions(self, tensors):
        """Pass 2: accumulate the 2048-bin |x| histograms (distribution_collector.py:80-135)."""
        if self._debug and self._added_to_distributions_flag:
            return
        self._added_to_distributions_flag = True
        if not hasattr(self, "_distribution_intervals"):
            print("interval:", self.distribution_intervals)
        flat = self._gather(tensors)
        intervals = [np.float32(self._distribution_intervals[name]) for name in self._tensor_list]
        _native.hist_multi(flat, intervals, self._hist)
        self._hist_dirty = True

    # ------------------------------------------- per-channel maxima (extension; no reference counterpart)
    def refresh_channel_max_val(self, tensors, channel_dim=1):
        """Running max |x| per channel of every listed tensor that has a channel axis (north_star item 1,
        "per-channel and per-tensor max-abs").  The reference reduces per tensor only
        (distribution_collector.py:77); this is the same reduction kept per channel, one
        pq_absmax_per_channel_f32 launch per tensor, state int32 bit patterns on the device."""
        if not hasattr(self, "_chan_bits"):
            self._chan_bits = {}
        for name in self._tensor_list:
            x = tensors[name]
            if not (isinstance(x, torch.Tensor) and x.is_cuda):
                x = _native.to_device_f32(x, self._device).view(np.shape(tensors[name]))
            if x.dim() <= channel_dim:
                continue
            if name not in self._chan_bits:
                self._chan_bits[name] = torch.zeros(x.shape[channel_dim], dtype=torch.int32, device=x.device)
            _native.absmax_per_channel(x.float(), self._chan_bits[name], channel_dim)

    @property
    def channel_max_vals(self):
        """dict name -> np.float32 [C] (one D2H per tensor)."""
        assert hasattr(self, "_chan_bits"), "Please use refresh_channel_max_val() first."
        return {name: b.view(torch.float32).cpu().numpy() for name, b in self._chan_bits.items()}

    def all_reduce_channel_max(self, group=None):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            for name in self._tensor_list:
                if name in getattr(self, "_chan_bits", {}):
                    dist.all_reduce(self._chan_bits[name], op=dist.ReduceOp.MAX, group=group)

    # ------------------------------------------------------- multi-GPU merge (new; SURVEY 8e)
    def device_state(self):
        """(max_bits int32 [n], hist int64 [n][2048]) on the device."""
        return self._max_bits, self._hist

    def all_reduce_max(self, group=None):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            self._ensure_state(None)
            # non-negative fp32 bit patterns order like the floats: integer MAX is exact
            dist.all_reduce(self._max_bits, op=dist.ReduceOp.MAX, group=group)
            self._max_dirty = True
            self._max_vals_refreshed_flag = True

    def all_reduce_hist(self, group=None):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            self._ensure_state(None)
            dist.all_reduce(self._hist, op=dist.ReduceOp.SUM, group=group)
            self._hist_dirty = True
            self._added_to_distributions_flag = True

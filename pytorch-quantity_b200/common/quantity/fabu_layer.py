"""Model-authoring operators (reference: quantity/common/quantity/fabu_layer.py:5-36).

The calibration tracer only sees ``nn.Module`` calls, so a model that wants its residual
adds, concatenations and flattens observed (and later replaced, e.g. Eltwise -> NewAdd)
must express them with these modules instead of ``+`` / ``torch.cat`` / ``.view``.
They stay ordinary PyTorch ops; during calibration Quantity.activation_quantize runs Eltwise (and the
nn.ReLU after it) as one native kernel with the same result (tools/pytorch_quantizer.py, plan_calibration_fusion)."""
import torch
from torch import nn


class Eltwise(nn.Module):
    """Element-wise sum of two feature maps (fabu_layer.py:5-11)."""

    def forward(self, x, y):
        return torch.add(x, y)


class Concat(nn.Module):
    """Concatenation of two feature maps, channel axis by default (fabu_layer.py:14-20)."""

    def forward(self, x, y, dim=1):
        return torch.cat([x, y], dim)


class Identity(nn.Module):
    """What ``merge_bn`` leaves in place of a folded BatchNorm2d (fabu_layer.py:23-29)."""

    def forward(self, x):
        return x


class View(nn.Module):
    """Flatten to (batch, -1); returns a fresh tensor so the tracer can tell producer from
    consumer (fabu_layer.py:31-36)."""

    def forward(self, x):
        return x.reshape(x.shape[0], -1).clone()

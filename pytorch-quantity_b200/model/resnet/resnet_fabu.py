"""ImageNet-topology ResNet-18 / ResNet-50 authored under the tracer's rules.

The reference ships only a CIFAR ResNet-18 written this way
(quantity/model/resnet/ResNet_18_fabu.py:11-70); its ImageNet ResNets
(quantity/model/resnet/ResNet.py:161-217) use ``out += residual`` and in-place ReLU,
which the hook-based tracer cannot follow (README.md:48-50: every operation must be an
nn.Module, no functional ops).  BASELINE.json's configs are ResNet-18/50 at 224x224, so
this file provides that topology with the authoring rules of the fabu file:
``Eltwise`` for the residual add, ``View`` for the flatten, non-in-place ReLU, and each
BatchNorm2d registered right after its Conv2d so ``merge_bn`` can fold it
(quantity/common/quantity/utils.py:10-16).

It imports ``common.quantity`` by that name on purpose: the same file runs on top of the
reference package (golden generation) and on top of this repository's drop-in package.
"""
import torch.nn as nn

from common.quantity import Eltwise, View


def _conv_bn(cin, cout, k, stride, pad, groups=1):
    return [nn.Conv2d(cin, cout, kernel_size=k, stride=stride, padding=pad, groups=groups, bias=False),
            nn.BatchNorm2d(cout)]


class BasicUnit(nn.Module):
    """3x3 -> 3x3 residual unit (ResNet-18/34)."""
    expansion = 1

    def __init__(self, cin, width, stride):
        super().__init__()
        cout = width * self.expansion
        self.left = nn.Sequential(
            *_conv_bn(cin, width, 3, stride, 1), nn.ReLU(False),
            *_conv_bn(width, cout, 3, 1, 1))
        self.shortcut = nn.Sequential()
        if stride != 1 or cin != cout:
            self.shortcut = nn.Sequential(*_conv_bn(cin, cout, 1, stride, 0))
        self.Eltwise = Eltwise()
        self.relu = nn.ReLU(False)

    def forward(self, x):
        return self.relu(self.Eltwise(self.left(x), self.shortcut(x)))


class BottleneckUnit(BasicUnit):
    """1x1 -> 3x3(stride) -> 1x1 residual unit (ResNet-50/101), stride on the 3x3 like
    quantity/model/resnet/ResNet.py:31-61.  With groups > 1 it is the ResNeXt unit: the 3x3 is a grouped convolution
    of width * base_width / 64 * groups channels (torchvision's ResNeXt definition).  With avg_down it is the ResNet-D
    unit (He et al., "Bag of Tricks for Image Classification with Convolutional Neural Networks", 2019): a stride-2
    shortcut averages 2 x 2 blocks first and then applies a stride-1 1x1 convolution, so no activation is skipped."""
    expansion = 4

    def __init__(self, cin, width, stride, groups=1, base_width=64, avg_down=False):
        nn.Module.__init__(self)
        cout = width * self.expansion
        mid = width * base_width // 64 * groups
        self.left = nn.Sequential(
            *_conv_bn(cin, mid, 1, 1, 0), nn.ReLU(False),
            *_conv_bn(mid, mid, 3, stride, 1, groups), nn.ReLU(False),
            *_conv_bn(mid, cout, 1, 1, 0))
        self.shortcut = nn.Sequential()
        if avg_down and stride != 1:
            self.shortcut = nn.Sequential(nn.AvgPool2d(stride, stride, ceil_mode=True, count_include_pad=False),
                                          *_conv_bn(cin, cout, 1, 1, 0))
        elif stride != 1 or cin != cout:
            self.shortcut = nn.Sequential(*_conv_bn(cin, cout, 1, stride, 0))
        self.Eltwise = Eltwise()
        self.relu = nn.ReLU(False)


class FabuResNet(nn.Module):
    def __init__(self, unit, depths, num_classes=1000, in_hw=224, deep_stem=False, **unit_kw):
        super().__init__()
        if deep_stem:       # ResNet-C / -D: three 3x3 convolutions in place of the 7x7
            self.stem = nn.Sequential(*_conv_bn(3, 32, 3, 2, 1), nn.ReLU(False), *_conv_bn(32, 32, 3, 1, 1),
                                      nn.ReLU(False), *_conv_bn(32, 64, 3, 1, 1), nn.ReLU(False))
        else:
            self.stem = nn.Sequential(*_conv_bn(3, 64, 7, 2, 3), nn.ReLU(False))
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        stages, cin = [], 64
        for i, (width, n) in enumerate(zip((64, 128, 256, 512), depths)):
            units = []
            for j in range(n):
                units.append(unit(cin, width, (1 if i == 0 else 2) if j == 0 else 1, **unit_kw))
                cin = width * unit.expansion
            stages.append(nn.Sequential(*units))
        self.layer1, self.layer2, self.layer3, self.layer4 = stages
        self.avgpool = nn.AvgPool2d(in_hw // 32)
        self.view = View()
        self.fc = nn.Linear(cin, num_classes)

    def forward(self, x):
        x = self.maxpool(self.stem(x))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        return self.fc(self.view(self.avgpool(x)))


def resnet18_fabu(num_classes=1000, in_hw=224):
    return FabuResNet(BasicUnit, (2, 2, 2, 2), num_classes, in_hw)


def resnet50_fabu(num_classes=1000, in_hw=224):
    return FabuResNet(BottleneckUnit, (3, 4, 6, 3), num_classes, in_hw)


def resnet50d_fabu(num_classes=1000, in_hw=224):
    """ResNet-50-D: the deep stem and avg-down shortcuts (AvgPool2d(2, 2, ceil_mode=True, count_include_pad=False)
    -> 1x1 conv -> BN) on every stride-2 unit."""
    return FabuResNet(BottleneckUnit, (3, 4, 6, 3), num_classes, in_hw, deep_stem=True, avg_down=True)


def resnext50_32x4d_fabu(num_classes=1000, in_hw=224):
    return FabuResNet(BottleneckUnit, (3, 4, 6, 3), num_classes, in_hw, groups=32, base_width=4)


def randomize_bn_(model, seed=0):
    """SURVEY.md 8(d) synthetic-weight recipe: default inits under manual_seed(seed),
    every BN randomised so that folding it changes the conv (call before merge_bn)."""
    import torch
    g = torch.Generator().manual_seed(seed + 12345)
    for m in model.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
    return model

"""MobileNetV2 (Sandler et al., 2018; width 1.0, 224 x 224) authored under the tracer's rules, like resnet_fabu.py:
``Eltwise`` for the residual add, ``View`` for the flatten, non-in-place ``nn.ReLU``, and each BatchNorm2d registered
right after its Conv2d so ``merge_bn`` can fold it.

The paper's ReLU6 is replaced by ReLU: ``ReLU6`` is not among the tracer's operator types (``ALL_OP_TYPE`` in
tools/configs.yml), so calibration could not follow it.  The network is otherwise the standard one: a 3 x 3 stride-2
stem of 32 channels, 17 inverted-residual blocks from the (t, c, n, s) table below (1 x 1 expansion by t, 3 x 3
depthwise, linear 1 x 1 projection, identity shortcut where stride is 1 and the width is kept), a 1 x 1 convolution
to 1280 channels, global average pooling and the classifier.

It imports ``common.quantity`` by that name, as resnet_fabu.py does.
"""
import torch.nn as nn

from common.quantity import Eltwise, View

# expansion t, output channels c, repeats n, stride of the first repeat s
INVERTED_RESIDUAL_SETTING = ((1, 16, 1, 1), (6, 24, 2, 2), (6, 32, 3, 2), (6, 64, 4, 2), (6, 96, 3, 1),
                             (6, 160, 3, 2), (6, 320, 1, 1))


def _conv_bn_relu(cin, cout, k, stride, groups=1, relu=True):
    layers = [nn.Conv2d(cin, cout, kernel_size=k, stride=stride, padding=k // 2, groups=groups, bias=False),
              nn.BatchNorm2d(cout)]
    return layers + [nn.ReLU(False)] if relu else layers


class InvertedResidual(nn.Module):
    def __init__(self, cin, cout, stride, t):
        super().__init__()
        hidden = cin * t
        layers = _conv_bn_relu(cin, hidden, 1, 1) if t != 1 else []
        layers += _conv_bn_relu(hidden, hidden, 3, stride, groups=hidden)        # depthwise
        layers += _conv_bn_relu(hidden, cout, 1, 1, relu=False)                  # linear projection
        self.conv = nn.Sequential(*layers)
        self.use_res = stride == 1 and cin == cout
        if self.use_res:
            self.Eltwise = Eltwise()

    def forward(self, x):
        return self.Eltwise(self.conv(x), x) if self.use_res else self.conv(x)


class MobileNetV2Fabu(nn.Module):
    def __init__(self, num_classes=1000, in_hw=224):
        super().__init__()
        layers, cin = _conv_bn_relu(3, 32, 3, 2), 32
        for t, c, n, s in INVERTED_RESIDUAL_SETTING:
            for i in range(n):
                layers.append(InvertedResidual(cin, c, s if i == 0 else 1, t))
                cin = c
        layers += _conv_bn_relu(cin, 1280, 1, 1)
        self.features = nn.Sequential(*layers)
        self.avgpool = nn.AvgPool2d(in_hw // 32)
        self.view = View()
        self.classifier = nn.Linear(1280, num_classes)

    def forward(self, x):
        return self.classifier(self.view(self.avgpool(self.features(x))))


def mobilenetv2_fabu(num_classes=1000, in_hw=224):
    return MobileNetV2Fabu(num_classes, in_hw)

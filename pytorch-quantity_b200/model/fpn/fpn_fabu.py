"""Semantic FPN (Kirillov et al., "Panoptic Feature Pyramid Networks", 2019) on the ResNet-50 of resnet_fabu, authored
under the tracer's rules.

The reference's tracer lists ``UpsamplingNearest2d`` among its operator types (tools/configs.yml:21-22), the operator
of FPN necks and segmentation heads.  This file is such a network:

    backbone    the stem and layer1..layer4 of resnet50_fabu (C2..C5 at 1/4 .. 1/32; no pooling, no fc)
    top-down    P5 = lateral5(C5);  P_i = Eltwise(lateral_i(C_i), UpsamplingNearest2d(2)(P_{i+1})),  1x1 laterals
                to 256 channels
    head        per level a 3x3 conv + BN + ReLU to 128 channels, upsampled to 1/4 scale; the four levels merged with
                nested two-input Concats, a 3x3 conv + BN + ReLU, a 1x1 classifier to num_classes and a final x4
                upsample to the input resolution

Every upsample is a module of its own (the tracer refuses a module called twice), every ReLU is a non-in-place
nn.ReLU and every BatchNorm2d is registered right after its Conv2d so ``merge_bn`` folds it.
"""
import torch.nn as nn

from common.quantity import Concat, Eltwise

from ..resnet.resnet_fabu import BottleneckUnit, FabuResNet, _conv_bn


class SemanticFPNFabu(nn.Module):
    def __init__(self, num_classes=19, fpn_channels=256, head_channels=128):
        super().__init__()
        body = FabuResNet(BottleneckUnit, (3, 4, 6, 3))
        self.stem, self.maxpool = body.stem, body.maxpool
        self.layer1, self.layer2, self.layer3, self.layer4 = body.layer1, body.layer2, body.layer3, body.layer4
        self.lateral2, self.lateral3, self.lateral4, self.lateral5 = (
            nn.Conv2d(c, fpn_channels, kernel_size=1) for c in (256, 512, 1024, 2048))
        self.up5, self.up4, self.up3 = (nn.UpsamplingNearest2d(scale_factor=2) for _ in range(3))
        self.add4, self.add3, self.add2 = Eltwise(), Eltwise(), Eltwise()
        self.head2, self.head3, self.head4, self.head5 = (
            nn.Sequential(*_conv_bn(fpn_channels, head_channels, 3, 1, 1), nn.ReLU(False)) for _ in range(4))
        self.head_up3, self.head_up4, self.head_up5 = (nn.UpsamplingNearest2d(scale_factor=s) for s in (2, 4, 8))
        self.cat3, self.cat4, self.cat5 = Concat(), Concat(), Concat()
        self.fuse = nn.Sequential(*_conv_bn(4 * head_channels, head_channels, 3, 1, 1), nn.ReLU(False))
        self.classifier = nn.Conv2d(head_channels, num_classes, kernel_size=1)
        self.up_out = nn.UpsamplingNearest2d(scale_factor=4)

    def forward(self, x):
        c2 = self.layer1(self.maxpool(self.stem(x)))
        c3 = self.layer2(c2)
        c4 = self.layer3(c3)
        c5 = self.layer4(c4)
        p5 = self.lateral5(c5)
        p4 = self.add4(self.lateral4(c4), self.up5(p5))
        p3 = self.add3(self.lateral3(c3), self.up4(p4))
        p2 = self.add2(self.lateral2(c2), self.up3(p3))
        s = self.cat3(self.head2(p2), self.head_up3(self.head3(p3)))
        s = self.cat4(s, self.head_up4(self.head4(p4)))
        s = self.cat5(s, self.head_up5(self.head5(p5)))
        return self.up_out(self.classifier(self.fuse(s)))


def fpn_r50_fabu(num_classes=19):
    return SemanticFPNFabu(num_classes)

"""CPU oracle for the Resnet34_8s backbone -- TEST INFRASTRUCTURE, NOT THE PRODUCT.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` leg may import this file.  The shipped path
(``pytorch-dense-correspondence_b200``) never imports anything under ``oracle/``.

This is a plain PyTorch fp32 restatement of the reference's backbone.  The
arithmetic itself (Conv2d / BatchNorm2d / ReLU / MaxPool2d / bilinear upsample)
is third-party: torch (reference pin torch 1.1.0, docker/install_pytorch.sh:6-7);
what is restated here is the reference's *wiring* of those ops:

  external/pytorch-segmentation-detection/vision/torchvision/models/resnet.py
      conv3x3              :20-37    (pad = dilation for a 3x3 kernel)
      BasicBlock           :40-69
      ResNet.__init__      :112-180  (He-normal conv init :174-180)
      ResNet._make_layer   :183-229  (stride -> dilation once output_stride is hit,
                                      and the dilation is applied to block 0 too)
      ResNet.forward       :231-265
      resnet34             :290-308
  external/pytorch-segmentation-detection/pytorch_segmentation_detection/models/resnet_dilated.py
      Resnet34_8s          :283-322  (fc = Conv2d(512, D, 1), N(0, 0.01) / 0 init,
                                      upsample_bilinear == align_corners=True)

Parity pin: ``oracle/make_golden.py`` imports the real reference modules from
/root/reference (in the build container), loads this oracle's seeded state_dict
into them and checks bit-equality of the outputs before writing tests/golden/.
The reference holds no golden vectors / known-answer tests of its own for this
path (SURVEY.md section 8c), so "the reference executed on seeded inputs" is the
pin.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F


def conv3x3(in_planes, out_planes, stride=1, dilation=1):
    # resnet.py:20-37 -- "full padding" of a dilated 3x3 == dilation
    upsampled = (3 - 1) * (dilation - 1) + 3
    pad = (upsampled - 1) // 2
    return nn.Conv2d(in_planes, out_planes, kernel_size=3, stride=stride,
                     padding=pad, dilation=dilation, bias=False)


class BasicBlock(nn.Module):
    # resnet.py:40-69
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None, dilation=1):
        super().__init__()
        self.conv1 = conv3x3(inplanes, planes, stride, dilation=dilation)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = conv3x3(planes, planes, dilation=dilation)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        residual = x
        out = self.relu(self.bn1(self.conv1(x)))
        out = self.bn2(self.conv2(out))
        if self.downsample is not None:
            residual = self.downsample(x)
        out = out + residual
        return self.relu(out)


class ResNetFullyConv(nn.Module):
    """resnet.py:112-265 configured as resnet34(fully_conv=True, output_stride=8,
    remove_avg_pool_layer=True) with the fc already replaced by the 1x1 scoring conv
    (resnet_dilated.py:298)."""

    def __init__(self, layers=(3, 4, 6, 3), num_classes=3, output_stride=8):
        super().__init__()
        self.output_stride = output_stride
        self.current_stride = 4
        self.current_dilation = 1
        self.inplanes = 64
        self.conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        self.layer1 = self._make_layer(64, layers[0])
        self.layer2 = self._make_layer(128, layers[1], stride=2)
        self.layer3 = self._make_layer(256, layers[2], stride=2)
        self.layer4 = self._make_layer(512, layers[3], stride=2)
        self.fc = nn.Conv2d(512, num_classes, 1)
        # resnet.py:174-180 (He-normal on every conv, BN gamma=1 beta=0) ...
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()
        # ... then resnet_dilated.py:305-308 for the scoring layer
        self.fc.weight.data.normal_(0, 0.01)
        self.fc.bias.data.zero_()

    def _make_layer(self, planes, blocks, stride=1):
        # resnet.py:183-229
        downsample = None
        if stride != 1 or self.inplanes != planes:
            if self.current_stride == self.output_stride:
                self.current_dilation = self.current_dilation * stride
                stride = 1
            else:
                self.current_stride = self.current_stride * stride
            downsample = nn.Sequential(
                nn.Conv2d(self.inplanes, planes, kernel_size=1, stride=stride, bias=False),
                nn.BatchNorm2d(planes))
        layers = [BasicBlock(self.inplanes, planes, stride, downsample,
                             dilation=self.current_dilation)]
        self.inplanes = planes
        for _ in range(1, blocks):
            layers.append(BasicBlock(self.inplanes, planes, dilation=self.current_dilation))
        return nn.Sequential(*layers)

    def forward(self, x):
        # resnet.py:231-265 with remove_avg_pool_layer=True, fully_conv=True
        x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        return self.fc(x)


class Resnet34_8s(nn.Module):
    """resnet_dilated.py:283-322.  State-dict keys are ``resnet34_8s.*`` exactly like
    the reference (218 entries at any D)."""

    def __init__(self, num_classes=1000):
        super().__init__()
        self.resnet34_8s = ResNetFullyConv((3, 4, 6, 3), num_classes=num_classes)

    def forward(self, x, feature_alignment=False):
        if feature_alignment:
            raise NotImplementedError("feature_alignment is off on the hot path (rd.py:314)")
        size = x.shape[2:]
        x = self.resnet34_8s(x)
        # nn.functional.upsample_bilinear(size=) == interpolate(bilinear, align_corners=True)
        return F.interpolate(x, size=tuple(size), mode="bilinear", align_corners=True)


# Intra-op CPU threads tests/golden/backbone_*.npz and train_step_*.npz were written with.  The CPU convolutions split
# their weight-gradient reductions per thread, and at the golden sizes a different split can flip a ReLU / max-pool
# decision: the oracle's first-layer gradient at D=16 is 2.9e-3 (relative) off the stored one with 16 threads, ~2e-6 with
# 1, 2, 4, 32 or 64, and bit-equal with 8.  Comparisons with those vectors run with this many threads.
GOLDEN_CPU_THREADS = 8


def seeded_oracle(D=3, seed=0):
    """The weights every parity test uses: the oracle's own init under a fixed CPU seed."""
    g = torch.random.get_rng_state()
    torch.manual_seed(seed)
    net = Resnet34_8s(num_classes=D)
    torch.random.set_rng_state(g)
    return net


def process_network_output(image_pred, N, D, H, W):
    """dense_correspondence_network.py:303-319."""
    return image_pred.view(N, D, W * H).permute(0, 2, 1)

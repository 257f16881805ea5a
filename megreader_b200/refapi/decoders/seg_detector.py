"""DB text-detection head with the reference's surface (decoders/seg_detector.py:7-147): constructor, module tree, state-dict keys
(in2..in5, out2..out5, binarize.{0,1,3,4,6}, thresh.{0,1,3,4,6}) and weights_init are the same.

    features (c2, c3, c4, c5) -> 1x1 lateral convs, nearest x2 top-down adds, 3x3 convs to C/4 with nearest up-sampling to 1/4
    -> fuse (N, C, H/4, W/4) -> binarize / thresh: 3x3 conv, BN, ReLU, 2x2 stride-2 transposed conv, BN, ReLU, 2x2 stride-2
    transposed conv to one channel, sigmoid -> binary, thresh;  thresh_binary = 1 / (1 + exp(-k (binary - thresh)))

On CUDA tensors the two sigmoids and the step function run as one kernel each way (megreader_b200/db.py, csrc/db_head.cu) on the
outputs of binarize[:-1] / thresh[:-1]; on CPU tensors the framework composition below runs.  Every convolution, transposed
convolution and BatchNorm is an ordinary module, so megreader_b200.conv_engine.use_engine_convs can put them on its kernels."""
from collections import OrderedDict

import torch
import torch.nn as nn


class SegDetector(nn.Module):
    def __init__(self, in_channels=[64, 128, 256, 512], inner_channels=256, k=10, bias=False, adaptive=False, smooth=False,
                 serial=False, *args, **kwargs):
        super().__init__()
        self.k = k
        self.serial = serial
        self.up5 = nn.Upsample(scale_factor=2, mode='nearest')
        self.up4 = nn.Upsample(scale_factor=2, mode='nearest')
        self.up3 = nn.Upsample(scale_factor=2, mode='nearest')
        quarter = inner_channels // 4
        self.in5 = nn.Conv2d(in_channels[-1], inner_channels, 1, bias=bias)
        self.in4 = nn.Conv2d(in_channels[-2], inner_channels, 1, bias=bias)
        self.in3 = nn.Conv2d(in_channels[-3], inner_channels, 1, bias=bias)
        self.in2 = nn.Conv2d(in_channels[-4], inner_channels, 1, bias=bias)
        self.out5 = nn.Sequential(nn.Conv2d(inner_channels, quarter, 3, padding=1, bias=bias), nn.Upsample(scale_factor=8, mode='nearest'))
        self.out4 = nn.Sequential(nn.Conv2d(inner_channels, quarter, 3, padding=1, bias=bias), nn.Upsample(scale_factor=4, mode='nearest'))
        self.out3 = nn.Sequential(nn.Conv2d(inner_channels, quarter, 3, padding=1, bias=bias), nn.Upsample(scale_factor=2, mode='nearest'))
        self.out2 = nn.Conv2d(inner_channels, quarter, 3, padding=1, bias=bias)
        self.binarize = nn.Sequential(
            nn.Conv2d(inner_channels, quarter, 3, padding=1, bias=bias), nn.BatchNorm2d(quarter), nn.ReLU(inplace=True),
            nn.ConvTranspose2d(quarter, quarter, 2, 2), nn.BatchNorm2d(quarter), nn.ReLU(inplace=True),
            nn.ConvTranspose2d(quarter, 1, 2, 2), nn.Sigmoid())
        self.binarize.apply(self.weights_init)
        self.adaptive = adaptive
        if adaptive:
            self.thresh = self._init_thresh(inner_channels, serial=serial, smooth=smooth, bias=bias)
            self.thresh.apply(self.weights_init)
        for m in (self.in5, self.in4, self.in3, self.in2, self.out5, self.out4, self.out3, self.out2):
            m.apply(self.weights_init)

    def weights_init(self, m):
        name = m.__class__.__name__
        if 'Conv' in name:
            nn.init.kaiming_normal_(m.weight.data)
        elif 'BatchNorm' in name:
            m.weight.data.fill_(1.)
            m.bias.data.fill_(1e-4)

    def _init_thresh(self, inner_channels, serial=False, smooth=False, bias=False):
        quarter = inner_channels // 4
        self.thresh = nn.Sequential(
            nn.Conv2d(inner_channels + (1 if serial else 0), quarter, 3, padding=1, bias=bias), nn.BatchNorm2d(quarter),
            nn.ReLU(inplace=True),
            self._init_upsample(quarter, quarter, smooth=smooth, bias=bias), nn.BatchNorm2d(quarter), nn.ReLU(inplace=True),
            self._init_upsample(quarter, 1, smooth=smooth, bias=bias), nn.Sigmoid())
        return self.thresh

    def _init_upsample(self, in_channels, out_channels, smooth=False, bias=False):
        if not smooth:
            return nn.ConvTranspose2d(in_channels, out_channels, 2, 2)
        inter = in_channels if out_channels == 1 else out_channels
        layers = [nn.Upsample(scale_factor=2, mode='nearest'), nn.Conv2d(in_channels, inter, 3, 1, 1, bias=bias)]
        if out_channels == 1:
            layers.append(nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=1, padding=1, bias=True))
        # the reference hands the list itself to nn.Sequential, which raises TypeError: smooth=True never builds there either
        return nn.Sequential(layers)

    def forward(self, features, gt=None, masks=None, training=False):
        fuse = self._fuse(features)
        if not fuse.is_cuda:
            return self._forward_framework(fuse)
        from megreader_b200 import db
        x_b = self.binarize[:-1](fuse).float().contiguous()
        if not self.adaptive:
            binary, _, _ = db.maps(x_b, x_b, self.k)
            return OrderedDict(binary=binary)
        if self.serial:
            binary, _, _ = db.maps(x_b, x_b, self.k)
            fuse = torch.cat((fuse, nn.functional.interpolate(binary.to(fuse.dtype), fuse.shape[2:])), 1)
        x_t = self.thresh[:-1](fuse).float().contiguous()
        binary, thresh, thresh_binary = db.maps(x_b, x_t, self.k)
        return OrderedDict(binary=binary, thresh=thresh, thresh_binary=thresh_binary)

    def _fuse(self, features):
        c2, c3, c4, c5 = features
        in5, in4, in3, in2 = self.in5(c5), self.in4(c4), self.in3(c3), self.in2(c2)
        out4 = self.up5(in5) + in4        # 1/16
        out3 = self.up4(out4) + in3       # 1/8
        out2 = self.up3(out3) + in2       # 1/4
        return torch.cat((self.out5(in5), self.out4(out4), self.out3(out3), self.out2(out2)), 1)

    def _forward_framework(self, fuse):
        """The reference's composition after the fused features (the CPU path; bench_db.py's library arm on the GPU)."""
        binary = self.binarize(fuse)
        result = OrderedDict(binary=binary)
        if self.adaptive:
            if self.serial:
                fuse = torch.cat((fuse, nn.functional.interpolate(binary, fuse.shape[2:])), 1)
            thresh = self.thresh(fuse)
            result.update(thresh=thresh, thresh_binary=self.step_function(binary, thresh))
        return result

    def step_function(self, x, y):
        return torch.reciprocal(1 + torch.exp(-self.k * (x - y)))

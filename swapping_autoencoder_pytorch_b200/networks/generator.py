"""Generator / decoder G: (structure code, texture code) -> image.
Architecture and sub-module names of reference models/networks/generator.py:9-161."""
import math

import torch
import torch.nn.functional as F

from .. import util
from ..stylegan2_layers import ConvLayer, EqualLinear, StyledConv, ToRGB
from ..stylegan2_op import add_scale, conv2d_residual, spatial_style_native, upsample2x_add_scale
from .base_network import BaseNetwork

_INV_SQRT2 = 1.0 / math.sqrt(2.0)


def _is_plain_pointwise(layer):
    """ConvLayer that is nothing but a bias-free 1x1 stride-1 convolution (the generator's head skip connections)"""
    mods = layer._modules
    conv = mods["Conv"]
    return (set(mods) == {"Conv"} and conv.bias is None and conv.weight.shape[2] == 1 and conv.weight.shape[3] == 1
            and conv.stride == 1 and conv.padding == 0)


class UpsamplingBlock(torch.nn.Module):
    """two styled convs, the first upsampling x2 (reference generator.py:9-20; unused by the resnet generator)"""

    def __init__(self, inch, outch, styledim, blur_kernel=[1, 3, 3, 1], use_noise=False):
        super().__init__()
        self.inch, self.outch, self.styledim = inch, outch, styledim
        self.conv1 = StyledConv(inch, outch, 3, styledim, upsample=True, blur_kernel=blur_kernel, use_noise=use_noise)
        self.conv2 = StyledConv(outch, outch, 3, styledim, upsample=False, use_noise=use_noise)

    def forward(self, x, style):
        return self.conv2(self.conv1(x, style), style)


class ResolutionPreservingResnetBlock(torch.nn.Module):
    """reference generator.py:23-36"""

    def __init__(self, opt, inch, outch, styledim):
        super().__init__()
        self.conv1 = StyledConv(inch, outch, 3, styledim, upsample=False)
        self.conv2 = StyledConv(outch, outch, 3, styledim, upsample=False)
        self.skip = ConvLayer(inch, outch, 1, activate=False, bias=False) if inch != outch else torch.nn.Identity()

    def forward(self, x, style):
        skip = self.skip
        if isinstance(skip, ConvLayer) and _is_plain_pointwise(skip):
            # (skip(x) + res) / sqrt(2) with the factor folded into conv2's activation gain and the skip filter's scale:
            # the merge is a plain add in the 1x1 conv's epilogue and its backward needs no scaling pass
            res = self.conv2(self.conv1(x, style), style, out_scale=_INV_SQRT2)
            conv = skip._modules["Conv"]
            return conv2d_residual(x, conv.weight, res, 1.0, stride=conv.stride, padding=conv.padding,
                                   wscale=conv.scale * _INV_SQRT2)
        res = self.conv2(self.conv1(x, style), style)
        return add_scale(skip(x), res, _INV_SQRT2)


class UpsamplingResnetBlock(torch.nn.Module):
    """reference generator.py:39-53: residual branch upsamples with a transposed modulated conv, the skip branch
    with a 1x1 conv + bilinear x2."""

    def __init__(self, inch, outch, styledim, blur_kernel=[1, 3, 3, 1], use_noise=False):
        super().__init__()
        self.inch, self.outch, self.styledim = inch, outch, styledim
        self.conv1 = StyledConv(inch, outch, 3, styledim, upsample=True, blur_kernel=blur_kernel, use_noise=use_noise)
        self.conv2 = StyledConv(outch, outch, 3, styledim, upsample=False, use_noise=use_noise)
        self.skip = ConvLayer(inch, outch, 1, activate=True, bias=True) if inch != outch else torch.nn.Identity()

    def forward(self, x, style):
        if isinstance(self.skip, ConvLayer) and self.outch % 4 == 0:
            # both branches arrive pre-scaled by 1/sqrt(2) (folded into their activation gains; bilinear interpolation
            # is linear), so "bilinear x2 + merge" is one kernel with unit scale and the residual branch's gradient is
            # the block's output gradient itself
            res = self.conv2(self.conv1(x, style), style, out_scale=_INV_SQRT2)
            return upsample2x_add_scale(self.skip(x, out_scale=_INV_SQRT2), res, 1.0)
        res = self.conv2(self.conv1(x, style), style)
        skip = self.skip(x)
        if skip.shape[1] % 4 == 0:
            return upsample2x_add_scale(skip, res, _INV_SQRT2)      # bilinear x2 + merge in one kernel
        skip = F.interpolate(skip, scale_factor=2, mode='bilinear', align_corners=False)
        return add_scale(skip, res, _INV_SQRT2)


class GeneratorModulation(torch.nn.Module):
    """per-channel affine of the structure code predicted from the texture code (reference generator.py:56-67)"""

    def __init__(self, styledim, outch):
        super().__init__()
        self.scale = EqualLinear(styledim, outch)
        self.bias = EqualLinear(styledim, outch)

    def forward(self, x, style):
        if style.ndimension() <= 2:
            return x * self.scale(style)[:, :, None, None] + self.bias(style)[:, :, None, None]
        size = (x.size(2), x.size(3))
        if spatial_style_native():
            # code map: scale and bias are affine in the code, so they are evaluated at the map's resolution and their
            # spatial_code_ch-channel results interpolated (exact, bilinear weights sum to 1) — the global_code_ch-channel map
            # never reaches the structure code's grid
            return (x * F.interpolate(self.scale(style), size=size, mode='bilinear', align_corners=False)
                    + F.interpolate(self.bias(style), size=size, mode='bilinear', align_corners=False))
        style = F.interpolate(style, size=size, mode='bilinear', align_corners=False)
        return x * self.scale(style) + self.bias(style)


class StyleGAN2ResnetGenerator(BaseNetwork):
    @staticmethod
    def modify_commandline_options(parser, is_train):
        parser.add_argument("--netG_scale_capacity", default=1.0, type=float)
        parser.add_argument("--netG_num_base_resnet_layers", default=2, type=int)
        parser.add_argument("--netG_use_noise", type=util.str2bool, nargs='?', const=True, default=True)
        parser.add_argument("--netG_resnet_ch", type=int, default=256)
        return parser

    def __init__(self, opt):
        super().__init__(opt)
        n_up = opt.netE_num_downsampling_sp
        blur = [1, 3, 3, 1] if opt.use_antialias else [1]
        self.global_code_ch = opt.global_code_ch + opt.num_classes
        self.add_module("SpatialCodeModulation", GeneratorModulation(self.global_code_ch, opt.spatial_code_ch))

        ch = opt.spatial_code_ch
        n_head = opt.netG_num_base_resnet_layers
        for i in range(n_head):
            nxt = max(opt.spatial_code_ch, round((i + 1) / n_head * self.nf(0)))   # widen gradually
            self.add_module("HeadResnetBlock%d" % i, ResolutionPreservingResnetBlock(opt, ch, nxt, self.global_code_ch))
            ch = nxt
        for j in range(n_up):
            nxt = self.nf(j + 1)
            self.add_module("UpsamplingResBlock%d" % (2 ** (4 + j)),
                            UpsamplingResnetBlock(ch, nxt, self.global_code_ch, blur, opt.netG_use_noise))
            ch = nxt
        self.add_module("ToRGB", ToRGB(ch, self.global_code_ch, blur_kernel=blur))

    def nf(self, num_up):
        ch = 128 * (2 ** (self.opt.netE_num_downsampling_sp - num_up))
        return int(min(512, ch) * self.opt.netG_scale_capacity)

    def forward(self, spatial_code, global_code):
        spatial_code = util.normalize(spatial_code)
        global_code = util.normalize(global_code)
        x = self.SpatialCodeModulation(spatial_code, global_code)
        for i in range(self.opt.netG_num_base_resnet_layers):
            x = getattr(self, "HeadResnetBlock%d" % i)(x, global_code)
        for j in range(self.opt.netE_num_downsampling_sp):
            x = getattr(self, "UpsamplingResBlock%d" % (2 ** (4 + j)))(x, global_code)
        return self.ToRGB(x, global_code, None)

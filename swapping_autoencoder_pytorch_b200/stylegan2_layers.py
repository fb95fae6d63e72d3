"""Operator surface of the hot path — drop-in for reference ``models/networks/stylegan2_layers.py``.

Same class names, constructor signatures, attribute names, parameter shapes and ``state_dict`` keys as the
reference (so its checkpoints load and its networks / loss graph run unchanged), but every conv / FIR /
bias-activation is one of the sm_100a kernels behind ``include/sae_b200.h`` and activations are stored
channels-last.  Per-class citations point at the reference file (paths relative to the reference checkout).

Differences that are deliberate (B200-first):
* ``ModulatedConv2d`` never materialises ``batch`` copies of the weight and never runs a grouped conv: with
  ``new_demodulation`` (reference :258) the layer *is* a dense convolution of the style-scaled input with one
  demodulated filter (SURVEY.md §0.1), so it is ``modulate`` (one pass, TF32-rounded) + one implicit GEMM.
* ``StyledConv`` folds NoiseInjection + bias + leaky-ReLU into a single pass.
"""
import math
import random
from collections import OrderedDict

import torch
from torch import nn
from torch.nn import functional as F

from .stylegan2_op.blocks import FirSpec, ResBlockSpec, fir_noise_bias_act, fused_blocks_enabled, resblock
from .stylegan2_op import (FusedLeakyReLU, add_scale, conv2d, conv2d_bias_act, conv2d_noise_bias_act, conv2d_residual,
                           conv_transpose2d, fused_leaky_relu, fused_noise_bias_leaky_relu, linear, memo, modulate,
                           modulate_spatial, modulated_conv2d, modulated_conv_ok, reflect_pad, spatial_style_native, torgb,
                           upfirdn2d)

_SQRT2 = math.sqrt(2.0)


class PixelNorm(nn.Module):
    """reference :19-24"""

    def forward(self, input):
        return input * torch.rsqrt(input.square().mean(dim=1, keepdim=True) + 1e-8)


def make_kernel(k):
    """1-D taps -> normalised separable 2-D FIR (reference :27-35)."""
    k = torch.as_tensor(k, dtype=torch.float32)
    if k.dim() == 1:
        k = torch.outer(k, k)
    return k / k.sum()


def _taps_1d(k, gain=1.0):
    """host-side 1-D factors of make_kernel(k) * gain when k is a 1-D tap list: outer(t, t) == make_kernel(k) * gain"""
    try:
        vals = [float(v) for v in k]
    except TypeError:
        return None
    tot = sum(vals)
    g = math.sqrt(gain)
    t = tuple(v / tot * g for v in vals)
    return (t, t)


def _split_pad(p, extra0=0, extra1=0):
    return (p + 1) // 2 + extra0, p // 2 + extra1


class Upsample(nn.Module):
    """FIR upsampling by ``factor`` (reference :38-56)."""

    def __init__(self, kernel, factor=2):
        super().__init__()
        self.factor = factor
        self.register_buffer('kernel', make_kernel(kernel) * (factor ** 2))
        self.taps = _taps_1d(kernel, factor ** 2)
        self.pad = _split_pad(self.kernel.shape[0] - factor, extra0=factor - 1)

    def forward(self, input):
        return upfirdn2d(input, self.kernel, up=self.factor, down=1, pad=self.pad, taps=self.taps)


class Downsample(nn.Module):
    """FIR downsampling by ``factor`` (reference :59-87)."""

    def __init__(self, kernel, factor=2, pad=None, reflection_pad=False):
        super().__init__()
        self.factor = factor
        self.register_buffer('kernel', make_kernel(kernel))
        self.taps = _taps_1d(kernel)
        self.reflection = reflection_pad
        self.pad = _split_pad(self.kernel.shape[0] - factor if pad is None else pad)

    def forward(self, input):
        pad = self.pad
        if self.reflection:
            input = F.pad(input, (pad[0], pad[1], pad[0], pad[1]), mode='reflect')
            pad = (0, 0)
        return upfirdn2d(input, self.kernel, up=1, down=self.factor, pad=pad, taps=self.taps)


class Blur(nn.Module):
    """Padded FIR, up = down = 1 (reference :90-112)."""

    def __init__(self, kernel, pad, upsample_factor=1, reflection_pad=False):
        super().__init__()
        self.taps = _taps_1d(kernel, upsample_factor ** 2 if upsample_factor > 1 else 1.0)
        kernel = make_kernel(kernel)
        if upsample_factor > 1:
            kernel = kernel * (upsample_factor ** 2)
        self.register_buffer('kernel', kernel)
        self.pad = pad
        self.reflection = reflection_pad
        if self.reflection:
            self.reflection_pad = nn.ReflectionPad2d((pad[0], pad[1], pad[0], pad[1]))
            self.pad = (0, 0)

    def forward(self, input, down=1):
        """``down`` (extension): decimate the blurred result — used when the consumer is a stride-2 1x1 convolution,
        which only ever reads the even positions (blur-then-subsample == subsample-of-blur)."""
        if self.reflection:
            input = reflect_pad(input, self.reflection_pad.padding)
        return upfirdn2d(input, self.kernel, down=down, pad=self.pad, taps=self.taps)


class EqualConv2d(nn.Module):
    """Equalised-learning-rate conv (reference :115-150)."""

    def __init__(self, in_channel, out_channel, kernel_size, stride=1, padding=0, bias=True, lr_mul=1.0):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(out_channel, in_channel, kernel_size, kernel_size))
        self.scale = 1 / math.sqrt(in_channel * kernel_size ** 2) * lr_mul
        self.stride = stride
        self.padding = padding
        self.bias = nn.Parameter(torch.zeros(out_channel)) if bias else None

    def forward(self, input):
        return conv2d(input, self.weight, bias=self.bias, stride=self.stride, padding=self.padding, wscale=self.scale)

    def __repr__(self):
        o, i, k, _ = self.weight.shape
        return f'{self.__class__.__name__}({i}, {o}, {k}, stride={self.stride}, padding={self.padding})'


class EqualLinear(nn.Module):
    """Equalised-learning-rate linear with optional fused leaky-ReLU (reference :153-195)."""

    def __init__(self, in_dim, out_dim, bias=True, bias_init=0, lr_mul=1, activation=None):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(out_dim, in_dim).div_(lr_mul))
        self.bias = nn.Parameter(torch.zeros(out_dim).fill_(bias_init)) if bias else None
        self.activation = activation
        self.scale = (1 / math.sqrt(in_dim)) * lr_mul
        self.lr_mul = lr_mul

    def forward(self, input):
        if input.dim() > 2:
            out = conv2d(input, self.weight[:, :, None, None], wscale=self.scale)
        else:
            out = linear(input, self.weight, wscale=self.scale)
        if self.activation:
            return fused_leaky_relu(out, self.bias * self.lr_mul)
        if self.bias is not None:
            b = self.bias * self.lr_mul
            out = out + (b.view(1, -1, 1, 1) if out.dim() > 2 else b)
        return out

    def __repr__(self):
        return f'{self.__class__.__name__}({self.weight.shape[1]}, {self.weight.shape[0]})'


class ScaledLeakyReLU(nn.Module):
    """reference :198-207"""

    def __init__(self, negative_slope=0.2):
        super().__init__()
        self.negative_slope = negative_slope

    def forward(self, input):
        return F.leaky_relu(input, negative_slope=self.negative_slope) * _SQRT2


class ModulatedConv2d(nn.Module):
    """Style-modulated convolution (reference :210-325), ``new_demodulation`` semantics only:
    the *style vector* is RMS-normalised, the input is multiplied by it, and the (style-independent) filter is
    L2-normalised per output channel."""

    def __init__(self, in_channel, out_channel, kernel_size, style_dim, demodulate=True, upsample=False,
                 downsample=False, blur_kernel=[1, 3, 3, 1]):
        super().__init__()
        self.eps = 1e-8
        self.kernel_size = kernel_size
        self.in_channel = in_channel
        self.out_channel = out_channel
        self.upsample = upsample
        self.downsample = downsample
        if upsample:
            factor = 2
            p = (len(blur_kernel) - factor) - (kernel_size - 1)
            self.blur = Blur(blur_kernel, pad=_split_pad(p, extra0=factor - 1, extra1=1), upsample_factor=factor)
        if downsample:
            factor = 2
            p = (len(blur_kernel) - factor) + (kernel_size - 1)
            self.blur = Blur(blur_kernel, pad=_split_pad(p))
        self.scale = 1 / math.sqrt(in_channel * kernel_size ** 2)
        self.padding = kernel_size // 2
        self.weight = nn.Parameter(torch.randn(1, out_channel, in_channel, kernel_size, kernel_size))
        self.modulation = EqualLinear(style_dim, in_channel, bias_init=1)
        self.demodulate = demodulate
        self.new_demodulation = True

    def __repr__(self):
        return (f'{self.__class__.__name__}({self.in_channel}, {self.out_channel}, {self.kernel_size}, '
                f'upsample={self.upsample}, downsample={self.downsample})')

    def filter(self):
        """scale * W, demodulated per output channel: [Cout, Cin, k, k] (reference :285-292; identical for
        every sample, which is why no ``repeat(batch, ...)`` is needed)."""
        def build():
            w = self.weight[0] * self.scale
            if self.demodulate:
                w = w * torch.rsqrt(w.square().sum(dim=(1, 2, 3), keepdim=True) + 1e-8)
            return w.transpose(0, 1) if self.upsample else w
        # the filter does not depend on the style: built once per loss evaluation, shared by every call of the layer
        return memo(self.weight, "demod", build)

    def style_scale(self, style, batch):
        """the per-sample, per-input-channel scale s [N, Cin] of a non-spatial style (reference :278-283)"""
        s = self.modulation(style.reshape(batch, -1))
        if self.demodulate:
            s = s * torch.rsqrt(s.square().mean(dim=1, keepdim=True) + 1e-8)
        return s

    def per_sample_geom(self, input, style):
        """geometry object when the plain (no up / down sampling) convolution can run on per-sample filters (no modulated copy
        of the input), else None"""
        if self.upsample or self.downsample or style.dim() > 2 or not torch.is_floating_point(input):
            return None
        w = self.weight[0]
        return modulated_conv_ok(input, w, self.padding)

    def modulated_input(self, input, style):
        """input * (RMS-normalised) style — reference :269-284"""
        batch = input.shape[0]
        if style.dim() > 2:
            # spatially varying style (reference :269-276; evaluation-time only)
            if spatial_style_native():
                # the modulation affine commutes with bilinear interpolation (weights sum to 1): evaluate it at the code map's
                # resolution and let one kernel interpolate the Cin-channel result, normalise it per pixel and scale the input
                return modulate_spatial(input, self.modulation(style), self.demodulate)
            style = F.interpolate(style, size=input.shape[2:], mode='bilinear', align_corners=False)
            style = self.modulation(style)
            if self.demodulate:
                style = style * torch.rsqrt(style.square().mean(dim=1, keepdim=True) + 1e-8)
            return input * style
        return modulate(input, self.style_scale(style, batch))

    def forward(self, input, style):
        g = self.per_sample_geom(input, style)
        if g is not None:
            return modulated_conv2d(input, self.style_scale(style, input.shape[0]), self.filter(), g)
        input = self.modulated_input(input, style)
        w = self.filter()
        if self.upsample:
            out = conv_transpose2d(input, w, stride=2, padding=0)      # filter() already returns [Cin, Cout, k, k] here
            return self.blur(out)
        if self.downsample:
            return conv2d(self.blur(input), w, stride=2, padding=0)
        return conv2d(input, w, padding=self.padding)


class _ShapeOnly:
    """stand-in for a not-yet-computed conv output: NoiseInjection only needs its shape, dtype and device"""

    def __init__(self, shape, like):
        self.shape, self._like = shape, like

    def new_empty(self, *size):
        return self._like.new_empty(*size)


class NoiseInjection(nn.Module):
    """reference :328-351 — the class name and the ``image_size`` / ``fixed_noise`` attributes are load-bearing
    (base_network.py:41-54 looks modules up by the string "NoiseInjection")."""

    def __init__(self):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(1))
        self.fixed_noise = None
        self.image_size = None

    def resolve_noise(self, image, noise=None):
        if self.image_size is None:
            self.image_size = image.shape
        if self.fixed_noise is not None:
            noise = self.fixed_noise
            if noise.shape[2:] != image.shape[2:]:
                noise = F.interpolate(noise, image.shape[2:], mode="nearest")
        elif noise is None:
            b, _, h, w = image.shape
            noise = image.new_empty(b, 1, h, w).normal_()
        return noise

    def forward(self, image, noise=None):
        return image + self.weight * self.resolve_noise(image, noise)


class ConstantInput(nn.Module):
    """reference :354-364"""

    def __init__(self, channel, size=4):
        super().__init__()
        self.input = nn.Parameter(torch.randn(1, channel, size, size))

    def forward(self, input):
        return self.input.repeat(input.shape[0], 1, 1, 1)


class StyledConv(nn.Module):
    """ModulatedConv2d -> NoiseInjection -> FusedLeakyReLU (reference :367-405); the last two run as one kernel."""

    def __init__(self, in_channel, out_channel, kernel_size, style_dim, upsample=False, blur_kernel=[1, 3, 3, 1],
                 demodulate=True, use_noise=True, lr_mul=1.0):
        super().__init__()
        self.conv = ModulatedConv2d(in_channel, out_channel, kernel_size, style_dim, upsample=upsample,
                                    blur_kernel=blur_kernel, demodulate=demodulate)
        self.use_noise = use_noise
        self.noise = NoiseInjection()
        self.activate = FusedLeakyReLU(out_channel)

    def forward(self, input, style, noise=None, out_scale=1.0):
        """``out_scale`` (extension): extra factor on the activated output, folded into the activation gain (the
        generator's residual blocks pass 1/sqrt(2), see networks/generator.py)."""
        conv, act = self.conv, self.activate
        gain = act.scale * out_scale
        if not (conv.upsample or conv.downsample):
            g = conv.per_sample_geom(input, style)
            if g is not None:
                # style scale in the per-sample filters, noise + bias + activation in the epilogue: ONE kernel touches the
                # activation (no modulated copy of it exists in either direction)
                z = None
                if self.use_noise:
                    z = self.noise.resolve_noise(_ShapeOnly(torch.Size((input.shape[0], conv.out_channel, g.P, g.Q)), input), noise)
                if z is None or (z.shape[0] == input.shape[0] and z.shape[1] == 1 and tuple(z.shape[2:]) == (g.P, g.Q)):
                    return modulated_conv2d(input, conv.style_scale(style, input.shape[0]), conv.filter(), g, z, self.noise.weight,
                                            act.bias, act.negative_slope, gain)
            # plain 3x3: noise + bias + activation ride in the conv kernel's epilogue
            x = conv.modulated_input(input, style)
            w = conv.filter()
            if not self.use_noise:
                return conv2d_bias_act(x, w, act.bias, padding=conv.padding, negative_slope=act.negative_slope, scale=gain)
            shape = torch.Size((x.shape[0], conv.out_channel, x.shape[2], x.shape[3]))
            z = self.noise.resolve_noise(_ShapeOnly(shape, x), noise)
            if z.shape[0] == x.shape[0] and z.shape[1] == 1 and z.shape[2:] == x.shape[2:]:
                return conv2d_noise_bias_act(x, w, z, self.noise.weight, act.bias, padding=conv.padding,
                                             negative_slope=act.negative_slope, scale=gain)
            out = conv2d(x, w, padding=conv.padding)
            return fused_leaky_relu(out + self.noise.weight * z, act.bias, act.negative_slope, gain)   # broadcast noise: unfused
        if conv.upsample and not conv.blur.reflection and conv.out_channel % 4 == 0:
            # transposed conv, then blur + noise + bias + activation as ONE pass (no standalone blur launch, the blurred tensor
            # never reaches HBM)
            blur = conv.blur
            u = conv_transpose2d(conv.modulated_input(input, style), conv.filter(), stride=2, padding=0)
            k = blur.kernel.shape[0]
            oh, ow = u.shape[2] + blur.pad[0] + blur.pad[1] - k + 1, u.shape[3] + blur.pad[0] + blur.pad[1] - k + 1
            z = None
            if self.use_noise:
                z = self.noise.resolve_noise(_ShapeOnly(torch.Size((u.shape[0], conv.out_channel, oh, ow)), u), noise)
            if z is None or (z.shape[0] == u.shape[0] and z.shape[1] == 1 and tuple(z.shape[2:]) == (oh, ow)):
                return fir_noise_bias_act(u, FirSpec(blur.kernel, blur.pad, blur.taps, 1), z, self.noise.weight, act.bias,
                                          act.negative_slope, gain)
            out = blur(u)
            return fused_leaky_relu(out + self.noise.weight * z, act.bias, act.negative_slope, gain)   # broadcast noise: unfused
        out = conv(input, style)
        if not self.use_noise:
            return fused_leaky_relu(out, act.bias, act.negative_slope, gain)
        z = self.noise.resolve_noise(out, noise)
        if z.shape[0] != out.shape[0] or z.shape[1] != 1:
            return fused_leaky_relu(out + self.noise.weight * z, act.bias, act.negative_slope, gain)   # broadcast noise: unfused
        return fused_noise_bias_leaky_relu(out, z, self.noise.weight, act.bias, act.negative_slope, gain)


class ToRGB(nn.Module):
    """1x1 modulated conv without demodulation + bias (+ optional upsampled skip) (reference :408-427)."""

    def __init__(self, in_channel, style_dim, upsample=True, blur_kernel=[1, 3, 3, 1]):
        super().__init__()
        if upsample:
            self.upsample = Upsample(blur_kernel)
        self.conv = ModulatedConv2d(in_channel, 3, 1, style_dim, demodulate=False)
        self.bias = nn.Parameter(torch.zeros(1, 3, 1, 1))

    def forward(self, input, style, skip=None):
        conv = self.conv
        if (not conv.demodulate and conv.kernel_size == 1 and conv.out_channel == 3 and not (conv.upsample or conv.downsample)
                and input.shape[1] % 4 == 0 and input.shape[1] <= 1024 and (style.dim() <= 2 or spatial_style_native())):
            # one pass over the input: style scale, 1x1 conv to 3 channels and bias together (csrc/torgb.cu); no N = 3 GEMM and,
            # for a texture vector, no modulated copy of the generator's largest activation
            if style.dim() <= 2:
                s = conv.modulation(style.reshape(input.shape[0], -1))
            else:
                # code map: the per-pixel scale is applied first, the kernel then runs with a unit style
                input = conv.modulated_input(input, style)
                s = input.new_ones(input.shape[0], input.shape[1])
            out = torgb(input, s, conv.weight[0], self.bias, conv.scale)
        else:
            out = conv(input, style) + self.bias
        if skip is not None:
            out = out + self.upsample(skip)
        return out


class Generator(nn.Module):
    """The original StyleGAN2 synthesis network (reference :430-609).  Not used by the Swapping Autoencoder
    (its decoder is networks/generator.py) — kept so the operator surface is complete."""

    def __init__(self, size, style_dim, n_mlp, channel_multiplier=2, blur_kernel=[1, 3, 3, 1], lr_mlp=0.01):
        super().__init__()
        self.size = size
        self.style_dim = style_dim
        mlp = [PixelNorm()]
        mlp += [EqualLinear(style_dim, style_dim, lr_mul=lr_mlp, activation='fused_lrelu') for _ in range(n_mlp)]
        self.style = nn.Sequential(*mlp)
        cm = channel_multiplier
        self.channels = {4: 512, 8: 512, 16: 512, 32: 512, 64: 256 * cm, 128: 128 * cm, 256: 64 * cm,
                         512: 32 * cm, 1024: 16 * cm}
        self.input = ConstantInput(self.channels[4])
        self.conv1 = StyledConv(self.channels[4], self.channels[4], 3, style_dim, blur_kernel=blur_kernel)
        self.to_rgb1 = ToRGB(self.channels[4], style_dim, upsample=False)
        self.log_size = int(math.log(size, 2))
        self.num_layers = (self.log_size - 2) * 2 + 1
        self.convs = nn.ModuleList()
        self.upsamples = nn.ModuleList()
        self.to_rgbs = nn.ModuleList()
        self.noises = nn.Module()
        for layer_idx in range(self.num_layers):
            res = 2 ** ((layer_idx + 5) // 2)
            self.noises.register_buffer(f'noise_{layer_idx}', torch.randn(1, 1, res, res))
        ch = self.channels[4]
        for i in range(3, self.log_size + 1):
            nxt = self.channels[2 ** i]
            self.convs.append(StyledConv(ch, nxt, 3, style_dim, upsample=True, blur_kernel=blur_kernel))
            self.convs.append(StyledConv(nxt, nxt, 3, style_dim, blur_kernel=blur_kernel))
            self.to_rgbs.append(ToRGB(nxt, style_dim))
            ch = nxt
        self.n_latent = self.log_size * 2 - 2

    def make_noise(self):
        device = self.input.input.device
        noises = [torch.randn(1, 1, 4, 4, device=device)]
        for i in range(3, self.log_size + 1):
            noises += [torch.randn(1, 1, 2 ** i, 2 ** i, device=device) for _ in range(2)]
        return noises

    def mean_latent(self, n_latent):
        z = torch.randn(n_latent, self.style_dim, device=self.input.input.device)
        return self.style(z).mean(0, keepdim=True)

    def get_latent(self, input):
        return self.style(input)

    def forward(self, styles, return_latents=False, inject_index=None, truncation=1, truncation_latent=None,
                input_is_latent=False, noise=None, randomize_noise=True):
        if not input_is_latent:
            styles = [self.style(s) for s in styles]
        if noise is None:
            noise = ([None] * self.num_layers if randomize_noise
                     else [getattr(self.noises, f'noise_{i}') for i in range(self.num_layers)])
        if truncation < 1:
            styles = [truncation_latent + truncation * (s - truncation_latent) for s in styles]
        if len(styles) < 2:
            inject_index = self.n_latent
            latent = styles[0].unsqueeze(1).repeat(1, inject_index, 1) if styles[0].dim() < 3 else styles[0]
        else:
            if inject_index is None:
                inject_index = random.randint(1, self.n_latent - 1)
            latent = torch.cat([styles[0].unsqueeze(1).repeat(1, inject_index, 1),
                                styles[1].unsqueeze(1).repeat(1, self.n_latent - inject_index, 1)], 1)
        out = self.conv1(self.input(latent), latent[:, 0], noise=noise[0])
        skip = self.to_rgb1(out, latent[:, 1])
        i = 1
        for up, same, n1, n2, rgb in zip(self.convs[::2], self.convs[1::2], noise[1::2], noise[2::2], self.to_rgbs):
            out = same(up(out, latent[:, i], noise=n1), latent[:, i + 1], noise=n2)
            skip = rgb(out, latent[:, i + 2], skip)
            i += 2
        return (skip, latent) if return_latents else (skip, None)


def _is_pointwise_stride2(conv):
    return conv.weight.shape[2] == 1 and conv.weight.shape[3] == 1 and conv.stride == 2 and conv.padding == 0


class ConvLayer(nn.Sequential):
    """[Blur | RefPad] -> Conv -> [Act] with the reference's sub-module names (reference :612-668)."""

    def __init__(self, in_channel, out_channel, kernel_size, downsample=False, blur_kernel=[1, 3, 3, 1], bias=True,
                 activate=True, pad=None, reflection_pad=False):
        layers = []
        if downsample:
            if pad is None:
                pad = (len(blur_kernel) - 2) + (kernel_size - 1)
            layers.append(("Blur", Blur(blur_kernel, pad=_split_pad(pad), reflection_pad=reflection_pad)))
            stride, self.padding = 2, 0
        else:
            stride = 1
            self.padding = kernel_size // 2 if pad is None else pad
            if reflection_pad:
                layers.append(("RefPad", nn.ReflectionPad2d(self.padding)))
                self.padding = 0
        layers.append(("Conv", EqualConv2d(in_channel, out_channel, kernel_size, padding=self.padding, stride=stride,
                                           bias=bias and not activate)))
        if activate:
            layers.append(("Act", FusedLeakyReLU(out_channel) if bias else ScaledLeakyReLU(0.2)))
        super().__init__(OrderedDict(layers))

    def forward(self, x, out_scale=1.0):
        """``out_scale`` (extension): extra factor on the activated output, folded into the activation gain — the
        residual blocks pass 1/sqrt(2) so that their merge needs no scaling pass in either direction."""
        mods = self._modules
        conv, act = mods["Conv"], mods.get("Act")
        stride = conv.stride
        if "Blur" in mods:
            if _is_pointwise_stride2(conv):
                x, stride = mods["Blur"](x, down=2), 1       # the 1x1 stride-2 conv reads only the even blurred pixels
            else:
                x = mods["Blur"](x)
        if "RefPad" in mods:
            x = reflect_pad(x, mods["RefPad"].padding)
        if isinstance(act, FusedLeakyReLU) and conv.bias is None:
            # bias + leaky-ReLU applied in the conv kernel's epilogue
            return conv2d_bias_act(x, conv.weight, act.bias, stride=stride, padding=conv.padding,
                                   negative_slope=act.negative_slope, scale=act.scale * out_scale, wscale=conv.scale)
        x = conv2d(x, conv.weight, bias=conv.bias, stride=stride, padding=conv.padding, wscale=conv.scale)
        x = act(x) if act is not None else x
        return x if out_scale == 1.0 else x * out_scale


class ResBlock(nn.Module):
    """conv1 (3x3) -> conv2 (blur + 3x3 stride 2) plus 1x1 skip, summed and divided by sqrt(2) (reference :672-693)."""

    def __init__(self, in_channel, out_channel, blur_kernel=[1, 3, 3, 1], reflection_pad=False, pad=None,
                 downsample=True):
        super().__init__()
        self.conv1 = ConvLayer(in_channel, in_channel, 3, reflection_pad=reflection_pad, pad=pad)
        self.conv2 = ConvLayer(in_channel, out_channel, 3, downsample=downsample, blur_kernel=blur_kernel,
                               reflection_pad=reflection_pad, pad=pad)
        self.skip = ConvLayer(in_channel, out_channel, 1, downsample=downsample, blur_kernel=blur_kernel,
                              activate=False, bias=False)

    def _fused_spec(self):
        """ResBlockSpec when the block has the discriminators' standard shape (3x3 + act, blur + 3x3 stride 2 + act,
        blur + 1x1 stride 2 skip, zero padding) — then the whole block is ONE autograd node (stylegan2_op/blocks.py);
        None otherwise (reflection padding, no downsampling, exotic kernels)."""
        spec = self.__dict__.get("_spec", False)
        if spec is not False:
            return spec
        spec = None
        c1, c2, sk = self.conv1._modules, self.conv2._modules, self.skip._modules

        def plain_act(m):
            return isinstance(m.get("Act"), FusedLeakyReLU) and m["Conv"].bias is None and "RefPad" not in m

        if (plain_act(c1) and plain_act(c2) and "Blur" not in c1 and "Blur" in c2 and "Blur" in sk and "Act" not in sk
                and "RefPad" not in sk and sk["Conv"].bias is None and _is_pointwise_stride2(sk["Conv"])
                and not c2["Blur"].reflection and not sk["Blur"].reflection
                and tuple(c1["Conv"].weight.shape[2:]) == (3, 3) and c1["Conv"].stride == 1 and c1["Conv"].padding == 1
                and tuple(c2["Conv"].weight.shape[2:]) == (3, 3) and c2["Conv"].stride == 2 and c2["Conv"].padding == 0
                and c1["Act"].negative_slope == c2["Act"].negative_slope):
            b2, bs = c2["Blur"], sk["Blur"]
            spec = ResBlockSpec(c1["Conv"].scale, c2["Conv"].scale, sk["Conv"].scale / _SQRT2, c1["Act"].negative_slope,
                                c1["Act"].scale, c2["Act"].scale / _SQRT2,
                                FirSpec(b2.kernel, b2.pad, b2.taps, 1), FirSpec(bs.kernel, bs.pad, bs.taps, 2))
        self.__dict__["_spec"] = spec
        return spec

    def forward(self, input):
        spec = self._fused_spec() if (input.shape[1] % 4 == 0 and fused_blocks_enabled()) else None
        if spec is not None:
            # buffers may have moved (module.to(device)) since the spec was built
            spec.blur2.kernel, spec.blur_s.kernel = self.conv2._modules["Blur"].kernel, self.skip._modules["Blur"].kernel
            c1, c2, sk = self.conv1._modules, self.conv2._modules, self.skip._modules
            return resblock(input, c1["Conv"].weight, c1["Act"].bias, c2["Conv"].weight, c2["Act"].bias,
                            sk["Conv"].weight, spec)
        mods = self.skip._modules
        conv = mods["Conv"]
        if conv.bias is None and "Act" not in mods and "RefPad" not in mods:
            # skip branch: [Blur] -> 1x1 conv whose epilogue performs the residual merge.  The 1/sqrt(2) of the merge is
            # folded into conv2's activation gain and into the skip filter's scale, so the merge is a plain add: its
            # backward hands dy to both branches untouched (no scaling pass over the block output or its gradient).
            out = self.conv2(self.conv1(input), out_scale=1.0 / _SQRT2)
            stride = conv.stride
            if "Blur" in mods and _is_pointwise_stride2(conv):
                h, stride = mods["Blur"](input, down=2), 1    # blur evaluated only where the 1x1 stride-2 conv samples it
            else:
                h = mods["Blur"](input) if "Blur" in mods else input
            return conv2d_residual(h, conv.weight, out, 1.0, stride=stride, padding=conv.padding,
                                   wscale=conv.scale / _SQRT2)
        out = self.conv2(self.conv1(input))
        return add_scale(out, self.skip(input), 1.0 / _SQRT2)


class Discriminator(nn.Module):
    """StyleGAN2 residual discriminator without minibatch-stddev (reference :696-764)."""

    def __init__(self, size, channel_multiplier=2, blur_kernel=[1, 3, 3, 1]):
        super().__init__()
        cm = channel_multiplier
        channels = {4: 512, 8: 512, 16: min(512, int(512 * cm)), 32: min(512, int(512 * cm)), 64: int(256 * cm),
                    128: int(128 * cm), 256: int(64 * cm), 512: int(32 * cm), 1024: int(16 * cm)}
        original_size = size
        size = 2 ** int(round(math.log(size, 2)))
        log_size = int(math.log(size, 2))
        blocks = [('0', ConvLayer(3, channels[size], 1))]
        ch = channels[size]
        for i in range(log_size, 2, -1):
            nxt = channels[2 ** (i - 1)]
            name = str(9 - i) if i <= 8 else "%dx%d" % (2 ** i, 2 ** i)
            blocks.append((name, ResBlock(ch, nxt, blur_kernel)))
            ch = nxt
        self.convs = nn.Sequential(OrderedDict(blocks))
        self.final_conv = ConvLayer(ch, channels[4], 3)
        side = int(4 * original_size / size)
        self.final_linear = nn.Sequential(
            EqualLinear(channels[4] * side * side, channels[4], activation='fused_lrelu'),
            EqualLinear(channels[4], 1),
        )

    def get_features(self, input):
        return self.final_conv(self.convs(input))

    def forward(self, input):
        feat = self.get_features(input)
        # flatten in logical (C, H, W) order exactly like the reference's .view(batch, -1)
        return self.final_linear(feat.reshape(feat.shape[0], -1))

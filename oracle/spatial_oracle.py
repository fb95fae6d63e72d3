"""ORACLE — test infrastructure only.  The generator driven by a texture code MAP [B, C, h, w], restated as the reference
writes it (models/networks/generator.py:62-67, stylegan2_layers.py:269-276): the map is interpolated to each layer's resolution,
the modulation affine runs there per pixel, then the per-pixel RMS normalisation.  Independent of the product's commuted
formulation (affine at the map's resolution, then interpolation).  Vector codes go to ``sae_oracle`` unchanged."""
import math

import torch
import torch.nn.functional as F

from . import sae_oracle as O


def modulated_conv2d(P, name, x, style, kernel_size, demodulate=True, upsample=False, blur_taps=(1, 3, 3, 1)):
    """``sae_oracle.modulated_conv2d`` for a style that may be a code map (reference stylegan2_layers.py:269-276)"""
    if style.dim() <= 2:
        return O.modulated_conv2d(P, name, x, style, kernel_size, demodulate=demodulate, upsample=upsample, blur_taps=blur_taps)
    style = F.interpolate(style, size=(x.shape[2], x.shape[3]), mode="bilinear", align_corners=False)
    s = O.equal_linear(P, name + ".modulation", style)
    if demodulate:
        s = s * torch.rsqrt(s.pow(2).mean(dim=1, keepdim=True) + 1e-8)
    x = x * s
    w = P[name + ".weight"][0]
    w = w * (1.0 / math.sqrt(w.shape[1] * kernel_size ** 2))
    if demodulate:
        w = w * torch.rsqrt(w.pow(2).sum(dim=(1, 2, 3), keepdim=True) + 1e-8)
    if upsample:
        out = F.conv_transpose2d(x, w.transpose(0, 1), stride=2, padding=0)
        p = (len(blur_taps) - 2) - (kernel_size - 1)
        k = P.get(name + ".blur.kernel")
        if k is None:
            k = O.make_kernel(list(blur_taps), x.dtype) * 4
        return O.upfirdn2d(out, k.to(x), pad=((p + 1) // 2 + 1, p // 2 + 1))
    return F.conv2d(x, w, padding=kernel_size // 2)


def styled_conv(P, name, x, style, upsample=False, use_noise=True, noise=None, blur_taps=(1, 3, 3, 1)):
    """``sae_oracle.styled_conv`` for a style that may be a code map"""
    out = modulated_conv2d(P, name + ".conv", x, style, 3, upsample=upsample, blur_taps=blur_taps)
    if use_noise:
        if noise is None:
            noise = torch.randn(out.shape[0], 1, out.shape[2], out.shape[3], dtype=out.dtype).to(out.device)
        out = out + P[name + ".noise.weight"] * noise
    return O.fused_leaky_relu(out, P[name + ".activate.bias"])


def generator_forward(P, opt, sp, gl, noises=None):
    """``sae_oracle.generator_forward`` with gl a code map [B, C, h, w] (reference generator.py:62-67, 147-161)"""
    noises = noises or {}
    blur = (1, 3, 3, 1) if opt.use_antialias else (1,)
    sp, gl = O.normalize(sp), O.normalize(gl)
    g = F.interpolate(gl, size=(sp.shape[2], sp.shape[3]), mode="bilinear", align_corners=False)
    x = sp * O.equal_linear(P, "SpatialCodeModulation.scale", g) + O.equal_linear(P, "SpatialCodeModulation.bias", g)
    ch = opt.spatial_code_ch
    for i in range(opt.netG_num_base_resnet_layers):
        nxt = max(opt.spatial_code_ch, round((i + 1) / opt.netG_num_base_resnet_layers * O.generator_nf(opt, 0)))
        name = "HeadResnetBlock%d" % i
        skip = O.conv_layer(P, name + ".skip", x, 1, activate=False, bias=False) if ch != nxt else x
        r = styled_conv(P, name + ".conv1", x, gl, noise=noises.get(name + ".conv1"))
        r = styled_conv(P, name + ".conv2", r, gl, noise=noises.get(name + ".conv2"))
        x = (skip + r) / O.SQRT2
        ch = nxt
    for j in range(opt.netE_num_downsampling_sp):
        nxt = O.generator_nf(opt, j + 1)
        name = "UpsamplingResBlock%d" % (2 ** (4 + j))
        skip = O.conv_layer(P, name + ".skip", x, 1, activate=True, bias=True) if ch != nxt else x
        skip = F.interpolate(skip, scale_factor=2, mode="bilinear", align_corners=False)
        r = styled_conv(P, name + ".conv1", x, gl, upsample=True, use_noise=opt.netG_use_noise,
                        noise=noises.get(name + ".conv1"), blur_taps=blur)
        r = styled_conv(P, name + ".conv2", r, gl, use_noise=opt.netG_use_noise, noise=noises.get(name + ".conv2"))
        x = (skip + r) / O.SQRT2
        ch = nxt
    rgb = modulated_conv2d(P, "ToRGB.conv", x, gl, 1, demodulate=False)
    return rgb + P["ToRGB.bias"]

"""Drop-in for the reference package ``models.networks.stylegan2_op`` (reference __init__.py:1-2): same three
public names, backed by the sm_100a kernels behind include/sae_b200.h instead of the JIT-built extensions."""
from .fused_act import FusedLeakyReLU, fused_leaky_relu, fused_noise_bias_leaky_relu
from .upfirdn2d import upfirdn2d
from .conv import (add_scale, conv2d, conv2d_bias_act, conv2d_noise_bias_act, conv2d_residual, conv_transpose2d,
                   filter_reuse, linear, memo, modulate, modulate_spatial, modulated_conv2d, modulated_conv_ok, reflect_pad, spatial_style_native,
                   torgb, upsample2x_add_scale)

__all__ = ["FusedLeakyReLU", "fused_leaky_relu", "fused_noise_bias_leaky_relu", "upfirdn2d", "conv2d",
           "conv_transpose2d", "linear", "modulate", "add_scale", "conv2d_bias_act", "conv2d_noise_bias_act",
           "conv2d_residual", "upsample2x_add_scale", "reflect_pad", "filter_reuse", "memo", "torgb", "modulated_conv2d", "modulated_conv_ok",
           "modulate_spatial", "spatial_style_native"]

"""Dense convolution family with closed first- and second-order autograd on the sm_100a implicit-GEMM kernels.

Replaces the ``F.conv2d`` / ``F.conv_transpose2d`` / ``F.linear`` call sites of the reference operator surface
(models/networks/stylegan2_layers.py:136-142, :174-186, :299-323).  A convolution is bilinear in (input, weight),
so three primitives — fprop(x, w), dgrad(dy, w), wgrad(dy, x) — are closed under differentiation; each is an
``autograd.Function`` whose backward is written with the other two.  That is what lets
``SwappingAutoencoderModel.compute_R1_loss`` (reference swapping_autoencoder_model.py:138-185) take
``autograd.grad(..., create_graph=True)`` through D / Dpatch and back-propagate the penalty.

Weights enter in the reference's parameter layout ``[Cout, Cin, R, S]`` and are permuted to the kernels'
``[K, R, S, C]`` by a (differentiable) torch permute of the small filter tensor.
"""
import contextlib

import torch
import torch.nn.functional as F
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import backend
from ..backend import make_geom


_data_only = [False]


def set_data_gradients_only(flag):
    """see blocks.data_gradients_only; returns the previous value"""
    prev, _data_only[0] = _data_only[0], bool(flag)
    return prev


def data_gradients_only_active():
    return _data_only[0]


def _want_wgrad(ctx, idx):
    """weight gradient of a conv Function's backward: skipped when the backward is being recorded inside
    ``data_gradients_only()`` (R1's first backward needs the data gradient only; the weight gradient would be computed,
    recorded and thrown away — one forward-equivalent of tensor work per convolution)"""
    return ctx.needs_input_grad[idx] and not (_data_only[0] and torch.is_grad_enabled())


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _impl(g):
    """Kernel choice hint: linears (1x1 maps) have M = batch rows only — far below a 128-row tensor-core tile — and
    take unrounded inputs (style codes, pooled features), so they always use the generic kernel, which rounds its
    operands itself; everything else lets the library pick (None)."""
    return 1 if (g.H == 1 and g.W == 1 and g.P == 1 and g.Q == 1) else None


class _PrepFilter(Function):
    """[K,C,R,S] parameter * scale -> ([K,R,S,C], [C,R,S,K]) in the kernels' layouts, TF32-rounded, in ONE kernel
    (the reference spends a `weight * scale` pass per call, stylegan2_layers.py:138; the layouts and rounding would cost
    three more).  Linear, so its backward is the adjoint kernel and the pair is closed under differentiation.  The second
    output is an auxiliary copy for the dgrad kernel and carries no gradient."""

    @staticmethod
    def forward(ctx, w_oihw, scale):
        ctx.scale = scale
        krsc, crsk = backend.kernels().filter_prep(w_oihw.contiguous(), scale)
        ctx.mark_non_differentiable(crsk)
        return krsc, crsk

    @staticmethod
    def backward(ctx, d_krsc, _unused):
        return _UnprepFilter.apply(d_krsc, ctx.scale), None


class _UnprepFilter(Function):
    @staticmethod
    def forward(ctx, d_krsc, scale):
        ctx.scale = scale
        return backend.kernels().filter_unprep(d_krsc.contiguous(), scale)

    @staticmethod
    def backward(ctx, gg):
        return _PrepFilter.apply(gg, ctx.scale)[0], None


class _FilterMemo:
    """Per-loss-evaluation memo of derived filter tensors.  One loss command runs each network several times on the
    same parameters (D on real / rec / mix, Dpatch on three crop sets, G on rec / mix): the scaled, demodulated, padded and
    kernel-layout filters are functions of the parameters only, so inside ``filter_reuse()`` they are built once and the
    same autograd node feeds every use (its gradient is the sum over the uses — exactly what separate copies give)."""
    depth = 0
    store = {}


@contextlib.contextmanager
def filter_reuse():
    """Scope of one loss evaluation (model.SwappingAutoencoderModel.forward); nested scopes share the outermost memo."""
    _FilterMemo.depth += 1
    try:
        yield
    finally:
        _FilterMemo.depth -= 1
        if _FilterMemo.depth == 0:
            _FilterMemo.store.clear()


def memo(source, tag, build):
    """``build()`` once per (source tensor identity and version, tag, grad mode) inside ``filter_reuse()``; outside a scope it
    is always rebuilt.  The entry keeps ``source`` alive so its id cannot be recycled while the scope is open."""
    if _FilterMemo.depth == 0:
        return build()
    key = (id(source), source._version, tag, torch.is_grad_enabled(), source.requires_grad)
    hit = _FilterMemo.store.get(key)
    if hit is None:
        hit = (source, build())
        _FilterMemo.store[key] = hit
    return hit[1]


def prep_filter(weight, scale=1.0):
    """returns (w_krsc, w_crsk) for the conv Functions below"""
    scale = float(scale)
    return memo(weight, ("prep", scale), lambda: _PrepFilter.apply(weight, scale))


class _ConvFprop(Function):
    """y = conv(x, w)   x: logical NCHW, w: [K,R,S,C]; wt: the same filter as [C,R,S,K] (from prep_filter) or None"""

    @staticmethod
    def forward(ctx, x, w, wt, g):
        ctx.g = g
        ctx.save_for_backward(x, w, wt)
        return _nchw(backend.kernels().conv_fprop(_nhwc(x), w.contiguous(), g, impl=_impl(g), prepared=wt is not None))

    @staticmethod
    def backward(ctx, dy):
        x, w, wt = ctx.saved_tensors
        dx = _ConvDgrad.apply(dy, w, wt, ctx.g) if ctx.needs_input_grad[0] else None
        dw = _ConvWgrad.apply(dy, x, ctx.g) if _want_wgrad(ctx, 1) else None
        return dx, dw, None, None


class _ConvDgrad(Function):
    """dx = conv^T(dy, w)   (also the forward of a transposed convolution)"""

    @staticmethod
    def forward(ctx, dy, w, wt, g):
        ctx.g = g
        ctx.save_for_backward(dy, w, wt)
        return _nchw(backend.kernels().conv_dgrad(_nhwc(dy), w.contiguous(), g, impl=_impl(g), w_crsk=wt))

    @staticmethod
    def backward(ctx, ddx):
        dy, w, wt = ctx.saved_tensors
        d_dy = _ConvFprop.apply(ddx, w, wt, ctx.g) if ctx.needs_input_grad[0] else None
        d_w = _ConvWgrad.apply(dy, ddx, ctx.g) if ctx.needs_input_grad[1] else None
        return d_dy, d_w, None, None


class _ConvWgrad(Function):
    """dw[K,R,S,C] = sum_pixels dy (x) x_gathered"""

    @staticmethod
    def forward(ctx, dy, x, g):
        ctx.g = g
        ctx.save_for_backward(dy, x)
        return backend.kernels().conv_wgrad(_nhwc(dy), _nhwc(x), g, impl=_impl(g))

    @staticmethod
    def backward(ctx, ddw):
        dy, x = ctx.saved_tensors
        d_dy = _ConvFprop.apply(x, ddw, None, ctx.g) if ctx.needs_input_grad[0] else None
        d_x = _ConvDgrad.apply(dy, ddw, None, ctx.g) if ctx.needs_input_grad[1] else None
        return d_dy, d_x, None


class _ConvBiasAct(Function):
    """lrelu(conv(x, w) + b) * gain with the bias / activation applied in the conv kernel's epilogue (no separate
    pass over the output).  Backward = the differentiable masked-gradient Function of fused_act.py followed by
    dgrad / wgrad, so the discriminators' R1 double backward flows through it (EqualConv2d + FusedLeakyReLU,
    stylegan2_layers.py:136-142 + fused_act.py:89-96)."""

    @staticmethod
    def forward(ctx, x, w, wt, bias, g, negative_slope, gain):
        y = backend.kernels().conv_fprop(_nhwc(x), w.contiguous(), g, impl=_impl(g), prepared=wt is not None,
                                         bias=bias.contiguous(), act=3, alpha=negative_slope, gain=gain)
        out = _nchw(y)
        ctx.g, ctx.cfg, ctx.act_mask = g, (negative_slope, gain), backend.act_mask_of(y)
        ctx.save_for_backward(x, w, wt, out)
        return out

    @staticmethod
    def backward(ctx, dy):
        from .fused_act import FusedLeakyReLUFunctionBackward
        x, w, wt, out = ctx.saved_tensors
        # out.detach(): the mask is piecewise constant (the masked-gradient Function returns no gradient for it), but an
        # attached ``out`` would keep this node's own forward graph reachable from a recorded backward, and the engine
        # would then run a complete extra backward of the network on materialised zeros during R1's second backward
        gi, gb = FusedLeakyReLUFunctionBackward.apply(dy, out.detach(), *ctx.cfg, ctx.act_mask)
        dx = _ConvDgrad.apply(gi, w, wt, ctx.g) if ctx.needs_input_grad[0] else None
        dw = _ConvWgrad.apply(gi, x, ctx.g) if _want_wgrad(ctx, 1) else None
        return dx, dw, None, gb, None, None, None


class _ConvNoiseBiasAct(Function):
    """StyledConv tail fused into the conv epilogue: lrelu(conv(x, w) + nw * noise + b) * gain
    (stylegan2_layers.py:398-405).  Generator only, hence once-differentiable."""

    @staticmethod
    def forward(ctx, x, w, wt, noise, noise_weight, bias, g, negative_slope, gain):
        noise_flat = noise.reshape(-1).contiguous()
        y = backend.kernels().conv_fprop(_nhwc(x), w.contiguous(), g, prepared=wt is not None, bias=bias.contiguous(),
                                         act=3, alpha=negative_slope, gain=gain, noise=noise_flat,
                                         noise_weight=noise_weight.contiguous())
        out = _nchw(y)
        ctx.g, ctx.cfg, ctx.act_mask = g, (negative_slope, gain, tuple(noise.shape)), backend.act_mask_of(y)
        ctx.save_for_backward(x, w, wt, out, noise_flat, noise_weight)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        x, w, wt, out, noise_flat, noise_weight = ctx.saved_tensors
        negative_slope, gain, noise_shape = ctx.cfg
        k = backend.kernels()
        gi, gb, gnw = k.bias_act_backward(_nhwc(dy), _nhwc(out), negative_slope, gain, want_bias=True, noise=noise_flat,
                                          mask=ctx.act_mask)
        dx = _nchw(k.conv_dgrad(gi, w.contiguous(), ctx.g, w_crsk=wt)) if ctx.needs_input_grad[0] else None
        dw = k.conv_wgrad(gi, _nhwc(x), ctx.g) if ctx.needs_input_grad[1] else None
        g_noise = None
        if ctx.needs_input_grad[3]:
            g_noise = (gi.sum(dim=3) * noise_weight).reshape(noise_shape)
        return dx, dw, None, g_noise, gnw, gb, None, None, None


class _ConvResidual(Function):
    """(conv(x, w) + res) * scale — the ResBlock merge "(out + skip) / sqrt(2)" (stylegan2_layers.py:691) folded into
    the skip convolution's epilogue.  Linear in (x, res) and bilinear with w: backward reuses the differentiable
    primitives, so it is valid under double backward."""

    @staticmethod
    def forward(ctx, x, w, wt, res, g, scale):
        ctx.g, ctx.scale = g, scale
        ctx.save_for_backward(x, w, wt)
        return _nchw(backend.kernels().conv_fprop(_nhwc(x), w.contiguous(), g, prepared=wt is not None, residual=_nhwc(res),
                                                 res_scale=scale))

    @staticmethod
    def backward(ctx, dy):
        x, w, wt = ctx.saved_tensors
        gs = dy if ctx.scale == 1.0 else _AddScale.apply(dy, None, ctx.scale)
        dx = _ConvDgrad.apply(gs, w, wt, ctx.g) if ctx.needs_input_grad[0] else None
        dw = _ConvWgrad.apply(gs, x, ctx.g) if _want_wgrad(ctx, 1) else None
        return dx, dw, None, (gs if ctx.needs_input_grad[3] else None), None, None


class _PadChannels(Function):
    """[N, c, H, W] (any layout) -> channels zero-padded to ``c_out``, stored NHWC: one kernel for what would be an F.pad
    plus a layout copy of the 32-channel result.  Linear; its adjoint is a channel slice (a differentiable torch view),
    so R1's gradient with respect to the image passes through and can be differentiated again."""

    @staticmethod
    def forward(ctx, x, c_out):
        ctx.c_in = x.shape[1]
        return _nchw(backend.kernels().pad_channels(x, c_out))

    @staticmethod
    def backward(ctx, dy):
        return dy[:, :ctx.c_in], None


class _ViewAsPadded(Function):
    """[N, c, H, W] view of a channels-last buffer whose channels c..C-1 are known to be zero  ->  the [N, C, H, W] view of the
    same memory (no kernel, no copy).  Only for buffers a producer of this library marked ``_sae_zero_padded`` (the crop
    resampler, util._CropGather).  Adjoint = channel slice, as for _PadChannels."""

    @staticmethod
    def forward(ctx, x, c_out):
        n, c, h, w = x.shape
        ctx.c_in = c
        return torch.as_strided(x, (n, c_out, h, w), (h * w * c_out, 1, w * c_out, c_out), x.storage_offset())

    @staticmethod
    def backward(ctx, dy):
        return dy[:, :ctx.c_in], None


def _zero_padded_width(x):
    """C when ``x`` is the leading-channels view of a channels-last [N, H, W, C] buffer marked zero-padded by its producer"""
    base = x._base
    cp = getattr(base, "_sae_zero_padded", 0) if base is not None else 0
    if cp and x.dim() == 4:
        n, c, h, w = x.shape
        if c < cp and x.stride() == (h * w * cp, 1, w * cp, cp) and x.storage_offset() % cp == 0:
            return cp
    return 0


def _pad4(input, weight):
    """RGB tensors (3 channels) are zero-padded to 4 so rows are 16-byte aligned and the kernels keep their vector
    / TMA paths (the pad and the matching slice are differentiable torch ops on tiny tensors).  Returns
    (input, weight, original Cout or None)."""
    cin = input.shape[1]
    if cin % 4 != 0:
        # RGB inputs go to 32 channels: one 128-byte TMA row per pixel, so FromRGB / the first Dpatch conv and their
        # weight gradients run on the tensor-core kernels (the extra zero channels cost 1/4 of the 128-channel output)
        extra = (32 - cin) if cin < 32 else 4 - cin % 4
        if _zero_padded_width(input) == cin + extra:
            input = _ViewAsPadded.apply(input, cin + extra)        # the producer already wrote the padded layout
        else:
            input = _PadChannels.apply(input, cin + extra)
        weight = memo(weight, ("pad_cin", extra), lambda w=weight: F.pad(w, (0, 0, 0, 0, 0, extra)))
    cout = weight.shape[0]
    if cout % 4 != 0:
        weight = memo(weight, "pad_cout", lambda w=weight: F.pad(w, (0, 0, 0, 0, 0, 0, 0, 4 - cout % 4)))
        return input, weight, cout
    return input, weight, None


_PAD32_MIN = 40          # narrower layers stay as they are (their cost is bandwidth, not the tensor-core path)


def _round32(c):
    return c if (c % 32 == 0 or c < _PAD32_MIN) else c + 32 - c % 32


def _pad32(input, weight, transposed=False):
    """Wide layers whose channel counts are not multiples of 32 — the ffhq1024 option set's generator runs 409 / 204 / 102
    channels (netG_scale_capacity 0.8, experiments/ffhq1024_pretrained_launcher.py:23-27) — are zero-padded to the next
    multiple so that they run on the tcgen05 kernels (whose TMA rows are 32 channels) instead of the shape-complete mma.sync
    kernel: input through the channel-pad kernel, filter through a memoised F.pad, output through a channel slice; all three
    are differentiable, so gradients come back in the original shapes.  Returns (input, weight, Cout to slice back to or None).
    weight is [Cout, Cin, R, S], or [Cin, Cout, R, S] when ``transposed``."""
    ci_axis, co_axis = (0, 1) if transposed else (1, 0)
    cin, cout = weight.shape[ci_axis], weight.shape[co_axis]
    cin_p, cout_p = _round32(cin), _round32(cout)
    if cin_p == cin and cout_p == cout:
        return input, weight, None
    if cin_p != cin:
        input = _PadChannels.apply(input, cin_p)
    pads = [0, 0, 0, 0, 0, 0, 0, 0]                  # F.pad lists the last dimension first: (S, R, dim 1, dim 0)
    pads[5 if ci_axis == 1 else 7] = cin_p - cin
    pads[5 if co_axis == 1 else 7] = cout_p - cout
    weight = memo(weight, ("pad32", transposed), lambda w=weight: F.pad(w, tuple(pads)))
    return input, weight, (cout if cout_p != cout else None)


def _geom_for(input, weight, stride, padding):
    n, c, h, w_ = input.shape
    k, c2, r, s = weight.shape
    assert c == c2, "channel mismatch: input %d vs weight %d" % (c, c2)
    if (h + 2 * padding - r) < 0 or (w_ + 2 * padding - s) < 0:
        # same failure the reference hits at 64x64 with default options (SURVEY.md §0.5)
        raise RuntimeError("Kernel size can't be greater than actual input size")
    return make_geom(n, h, w_, c, k, r, s, stride, padding, padding)


def conv2d_bias_act(input, weight, bias, stride=1, padding=0, negative_slope=0.2, scale=2 ** 0.5, wscale=1.0):
    """fused_leaky_relu(F.conv2d(input, weight * wscale, stride=stride, padding=padding), bias) in one kernel"""
    input, weight, cout = _pad4(input, weight)
    if cout is None:
        input, weight, cout = _pad32(input, weight)
    if cout is not None:
        bias = F.pad(bias, (0, weight.shape[0] - cout))
    g = _geom_for(input, weight, stride, padding)
    w, wt = prep_filter(weight, wscale)
    out = _ConvBiasAct.apply(input, w, wt, bias, g, negative_slope, scale)
    return out if cout is None else out[:, :cout]


def conv2d_noise_bias_act(input, weight, noise, noise_weight, bias, padding=0, negative_slope=0.2, scale=2 ** 0.5,
                          wscale=1.0):
    """fused_leaky_relu(F.conv2d(input, weight * wscale, padding=padding) + noise_weight * noise, bias) in one kernel"""
    input, weight, cout = _pad32(input, weight)
    if cout is not None:
        bias = F.pad(bias, (0, weight.shape[0] - cout))
    g = _geom_for(input, weight, 1, padding)
    w, wt = prep_filter(weight, wscale)
    out = _ConvNoiseBiasAct.apply(input, w, wt, noise, noise_weight, bias, g, negative_slope, scale)
    return out if cout is None else out[:, :cout]


def conv2d_residual(input, weight, residual, scale, stride=1, padding=0, wscale=1.0):
    """(F.conv2d(input, weight * wscale, stride=stride, padding=padding) + residual) * scale in one kernel"""
    input, weight, cout = _pad32(input, weight)
    if cout is not None:
        residual = _PadChannels.apply(residual, weight.shape[0])
    g = _geom_for(input, weight, stride, padding)
    w, wt = prep_filter(weight, wscale)
    out = _ConvResidual.apply(input, w, wt, residual, g, scale)
    return out if cout is None else out[:, :cout]


def conv2d(input, weight, bias=None, stride=1, padding=0, wscale=1.0):
    """``F.conv2d(input, weight * wscale, bias, stride, padding)`` for NCHW-shaped input, [Cout,Cin,R,S] weight."""
    input, weight, cout = _pad4(input, weight)
    if cout is None:
        input, weight, cout = _pad32(input, weight)
    g = _geom_for(input, weight, stride, padding)
    w, wt = prep_filter(weight, wscale)
    out = _ConvFprop.apply(input, w, wt, g)
    if cout is not None:
        out = out[:, :cout]
    if bias is not None:
        out = out + bias.view(1, -1, 1, 1)
    return out


def conv_transpose2d(input, weight, stride=2, padding=0, wscale=1.0):
    """``F.conv_transpose2d(input, weight[Cin,Cout,R,S], stride, padding)`` — computed as the data-gradient of
    the strided convolution whose filter is ``weight`` read as [K=Cin, C=Cout, R, S]."""
    assert input.shape[1] == weight.shape[0]
    input, weight, cout_orig = _pad32(input, weight, transposed=True)
    n, cin, h, w_ = input.shape
    cin2, cout, r, s = weight.shape
    oh = (h - 1) * stride - 2 * padding + r
    ow = (w_ - 1) * stride - 2 * padding + s
    g = make_geom(n, oh, ow, cout, cin, r, s, stride, padding, padding, P=h, Q=w_)
    w, wt = prep_filter(weight, wscale)
    out = _ConvDgrad.apply(input, w, wt, g)
    return out if cout_orig is None else out[:, :cout_orig]


def linear(input, weight, bias=None, wscale=1.0):
    """``F.linear(input, weight * wscale)`` for [B, in] x [out, in]: a 1x1 convolution on a 1x1 map."""
    b, cin = input.shape
    cout = weight.shape[0]
    g = make_geom(b, 1, 1, cin, cout, 1, 1, 1, 0, 0)
    wscale = float(wscale)
    w, wt = memo(weight, ("linear", wscale), lambda: _PrepFilter.apply(weight.view(cout, cin, 1, 1), wscale))
    out = _ConvFprop.apply(input.reshape(b, cin, 1, 1), w, wt, g).reshape(b, cout)
    if bias is not None:
        out = out + bias
    return out


class _Modulate(Function):
    """x * s[:, :, None, None] (stylegan2_layers.py:284) with the style gradient reduced in the same pass.
    Only the generator modulates, and the generator is never differentiated twice (SURVEY.md §8 a16), so the
    backward is once-differentiable: a second-order request raises instead of silently detaching."""

    @staticmethod
    def forward(ctx, x, s):
        ctx.save_for_backward(x, s)
        return _nchw(backend.kernels().modulate(_nhwc(x), s.contiguous()))

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        x, s = ctx.saved_tensors
        dx, ds = backend.kernels().modulate_backward(_nhwc(dy), _nhwc(x), s.contiguous())
        return _nchw(dx), ds


def modulate(x, s):
    return _Modulate.apply(x, s)


class _ModulateSpatial(Function):
    """x * demod(bilinear(s_lo)) for a spatially varying style (stylegan2_layers.py:269-276) whose modulation affine was
    evaluated at the code map's own resolution: s_lo [Ns, C, hs, ws], Ns in {1, N}.  One pass over x; the style gradient
    is the interpolation's adjoint, reduced without atomics.  Generator only: once-differentiable."""

    @staticmethod
    def forward(ctx, x, s_lo, demodulate):
        xh, sh = _nhwc(x), _nhwc(s_lo)
        ctx.demodulate = demodulate
        ctx.save_for_backward(xh, sh)
        return _nchw(backend.kernels().modulate_spatial(xh, sh, demodulate))

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        xh, sh = ctx.saved_tensors
        dx, ds = backend.kernels().modulate_spatial_backward(_nhwc(dy), xh, sh, ctx.demodulate)
        return _nchw(dx), _nchw(ds), None


def spatial_style_native():
    """True when the active kernel set modulates with code maps natively (``modulate_spatial``).  False selects the reference's
    formulation — interpolate the map to each layer's resolution, then apply the modulation affine there — which
    ``SAE_SPATIAL_STYLE=glue`` asks of the CUDA kernels and which a kernel set declaring no ``spatial_style`` gets"""
    return getattr(backend.kernels(), "spatial_style", "glue") == "native"


def modulate_spatial(x, s_lo, demodulate):
    """``x * s`` with ``s = F.interpolate(s_lo, size=x.shape[2:], mode='bilinear', align_corners=False)``, RMS-normalised over
    channels per pixel when ``demodulate``; s_lo [Ns, C, hs, ws] with Ns == 1 (broadcast) or Ns == x.shape[0]"""
    n, c = x.shape[:2]
    if s_lo.dim() != 4 or s_lo.shape[1] != c or s_lo.shape[0] not in (1, n):
        raise ValueError("modulate_spatial: style map %s does not fit input %s" % (tuple(s_lo.shape), tuple(x.shape)))
    return _ModulateSpatial.apply(x, s_lo, bool(demodulate))


class _ModulatedConv(Function):
    """ModulatedConv2d's core (stylegan2_layers.py:284-323) WITHOUT a modulated copy of the activation: the style scale goes into
    per-sample filters W_n = W * s[n] that the tensor-core kernel selects per pixel tile (``sae_conv2d_fprop_per_sample``),
    optionally with the StyledConv tail (noise + bias + leaky-ReLU) in the same kernel's epilogue.  Backward: the data gradient
    with the transposed per-sample filters; the weight gradient takes x UNSCALED and forms  dW = sum_n s[n] G_n  and
    ds[n] = <W, G_n>  while draining its accumulators once per image (``sae_conv2d_wgrad_modulated``).
    Inputs: x [N,C,H,W], s [N,C] (already normalised), w [K,R,S,C] prepared (scaled, demodulated, rounded).
    Generator only, hence once-differentiable."""

    @staticmethod
    def forward(ctx, x, s, w, g, noise, noise_weight, bias, negative_slope, gain):
        k = backend.kernels()
        xh, sc = _nhwc(x), s.contiguous()
        w_n, _ = k.filter_modulate(w.contiguous(), sc, want_krsc=True, want_crsk=False)
        act = bias is not None
        epi = {}
        noise_flat = None
        if act:
            epi = dict(bias=bias.contiguous(), act=3, alpha=negative_slope, gain=gain)
            if noise is not None:
                noise_flat = noise.reshape(-1).contiguous()
                epi.update(noise=noise_flat, noise_weight=noise_weight.contiguous())
        out = k.conv_fprop_per_sample(xh, w_n, g, **epi)
        ctx.act_mask = backend.act_mask_of(out)
        ctx.g, ctx.cfg = g, (act, negative_slope, gain, tuple(noise.shape) if noise is not None else None)
        ctx.save_for_backward(xh, sc, w, out if act else None, noise_flat, noise_weight if noise is not None else None)
        return _nchw(out)

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        xh, sc, w, out, noise_flat, noise_weight = ctx.saved_tensors
        act, negative_slope, gain, noise_shape = ctx.cfg
        k = backend.kernels()
        gi, gb, gnw = _nhwc(dy), None, None
        if act:
            gi, gb, gnw = k.bias_act_backward(gi, out, negative_slope, gain, want_bias=True, noise=noise_flat, mask=ctx.act_mask)
        dx = None
        if ctx.needs_input_grad[0]:
            _, w_nt = k.filter_modulate(w.contiguous(), sc, want_krsc=False, want_crsk=True)
            dx = _nchw(k.conv_dgrad_per_sample(gi, w_nt, ctx.g))
        dw = ds = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dw, ds = k.conv_wgrad_modulated(gi, xh, sc, w.contiguous(), ctx.g)
        g_noise = None
        if noise_flat is not None and ctx.needs_input_grad[4]:
            g_noise = (gi.sum(dim=3) * noise_weight).reshape(noise_shape)
        return dx, ds, dw, None, g_noise, gnw, gb, None, None


def modulated_conv_ok(input, weight, padding):
    """does the per-sample-filter path take ``F.conv2d(input * s, weight, padding=padding)``?  Needs kernel support for the
    geometry AND a filter set much smaller than the activation (N |W| written + read  vs  |x| read + written by a scaling pass)"""
    n, c, h, w_ = input.shape
    k, c2, r, s_ = weight.shape
    if c != c2 or r != s_ or padding != r // 2 or c % 32 != 0 or k % 32 != 0:
        return None
    if 4 * k * r * s_ > h * w_:
        return None
    kern = backend.kernels()
    if not hasattr(kern, "conv_modulated_ok"):
        return None
    g = make_geom(n, h, w_, c, k, r, s_, 1, padding, padding)
    return g if kern.conv_modulated_ok(g) else None


def modulated_conv2d(input, s, weight, g, noise=None, noise_weight=None, bias=None, negative_slope=0.2, scale=2 ** 0.5, wscale=1.0):
    """``F.conv2d(input * s[:, :, None, None], weight * wscale, padding=k // 2)`` — optionally followed by
    ``fused_leaky_relu(. + noise_weight * noise, bias, negative_slope, scale)`` — on per-sample filters; ``g`` from
    ``modulated_conv_ok``"""
    w, _ = prep_filter(weight, wscale)
    return _ModulatedConv.apply(input, s, w, g, noise, noise_weight, bias, negative_slope, scale)


class _ToRGB(Function):
    """bias + conv1x1(x * s, w * wscale) with 3 output channels as ONE pass over x (csrc/torgb.cu) — the generator's ToRGB
    (stylegan2_layers.py:408-427: ModulatedConv2d(in, 3, 1, demodulate=False) + bias).  Backward is one more pass over x:
    dx and the per-sample outer products G[n] = sum_p dy (x) x, from which ds and dw follow on [N, 3, C] values.
    Generator only: once-differentiable."""

    @staticmethod
    def forward(ctx, x, s, w, bias, wscale):
        xh, sc, wc = _nhwc(x), s.contiguous(), w.reshape(3, -1).contiguous()
        y = backend.kernels().torgb_forward(xh, sc, wc, bias.reshape(-1).contiguous() if bias is not None else None, wscale)
        ctx.save_for_backward(xh, sc, wc)
        ctx.wscale, ctx.w_shape, ctx.bias_shape = wscale, tuple(w.shape), (tuple(bias.shape) if bias is not None else None)
        return _nchw(y)[:, :3]

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        xh, sc, wc = ctx.saved_tensors
        need = ctx.needs_input_grad
        dx, gw = backend.kernels().torgb_backward(dy, xh, sc, wc, ctx.wscale, want_dx=need[0], want_gw=need[1] or need[2])
        ds = dw = db = None
        if need[1]:
            ds = (gw * wc.unsqueeze(0)).sum(dim=1) * ctx.wscale
        if need[2]:
            dw = ((gw * sc.unsqueeze(1)).sum(dim=0) * ctx.wscale).reshape(ctx.w_shape)
        if need[3]:
            db = dy.sum(dim=(0, 2, 3)).reshape(ctx.bias_shape)
        return (_nchw(dx) if dx is not None else None), ds, dw, db, None


def torgb(x, s, w, bias, wscale):
    """``F.conv2d(x * s[:, :, None, None], w * wscale) + bias`` for a [3, C, 1, 1] filter (C % 4 == 0, C <= 1024)"""
    return _ToRGB.apply(x, s, w, bias, float(wscale))


class _AddScale(Function):
    """(a + b) * scale in one pass — the residual merges "(out + skip) / sqrt(2)" (stylegan2_layers.py:691,
    generator.py:36,53).  Linear, so its backward is the same kernel with b = None and stays differentiable."""

    @staticmethod
    def forward(ctx, a, b, scale):
        ctx.scale = scale
        k = backend.kernels()
        if a.dim() == 4:
            return _nchw(k.add_scale(_nhwc(a), _nhwc(b) if b is not None else None, scale))
        return k.add_scale(a.contiguous(), b.contiguous() if b is not None else None, scale)

    @staticmethod
    def backward(ctx, dy):
        g = _AddScale.apply(dy, None, ctx.scale)
        return g, (g if ctx.needs_input_grad[1] else None), None


def add_scale(a, b, scale):
    return _AddScale.apply(a, b, scale)


class _ReflectPad(Function):
    """nn.ReflectionPad2d on channels-last data in one pass.  Linear: its backward is the adjoint kernel, whose backward
    is the padding again — closed under differentiation like the FIR pair."""

    @staticmethod
    def forward(ctx, x, pads):
        ctx.pads = pads
        return _nchw(backend.kernels().reflect_pad(_nhwc(x), pads))

    @staticmethod
    def backward(ctx, dy):
        return _ReflectPadAdjoint.apply(dy, ctx.pads), None


class _ReflectPadAdjoint(Function):
    @staticmethod
    def forward(ctx, dy, pads):
        ctx.pads = pads
        return _nchw(backend.kernels().reflect_pad_backward(_nhwc(dy), pads))

    @staticmethod
    def backward(ctx, ddx):
        return _ReflectPad.apply(ddx, ctx.pads), None


def reflect_pad(x, pads):
    """pads = (left, right, top, bottom), the nn.ReflectionPad2d convention"""
    pads = tuple(int(p) for p in pads)
    if x.shape[1] % 4 != 0:
        return F.pad(x, pads, mode="reflect")
    return _ReflectPad.apply(x, pads)


class _Upsample2xAddScale(Function):
    """(bilinear_x2(skip) + res) * scale in one kernel — the generator's upsampling-block merge
    (generator.py:51-53).  Generator only: once-differentiable."""

    @staticmethod
    def forward(ctx, skip, res, scale):
        ctx.scale = scale
        return _nchw(backend.kernels().upsample2x_add_scale(_nhwc(skip), _nhwc(res), scale))

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        k = backend.kernels()
        g = _nhwc(dy)
        d_skip = _nchw(k.upsample2x_backward(g, ctx.scale)) if ctx.needs_input_grad[0] else None
        if ctx.scale == 1.0:
            d_res = dy if ctx.needs_input_grad[1] else None
        else:
            d_res = _nchw(k.add_scale(g, None, ctx.scale)) if ctx.needs_input_grad[1] else None
        return d_skip, d_res, None


def upsample2x_add_scale(skip, res, scale):
    return _Upsample2xAddScale.apply(skip, res, scale)

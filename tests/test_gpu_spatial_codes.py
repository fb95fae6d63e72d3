"""GPU (B200): texture code maps [N, C, h, w] through the CUDA kernels — ``sae_modulate_spatial`` and its backward against an fp64
torch formulation (F.interpolate -> demodulation -> multiply, and its autograd), the layers against the oracle, the generator against
the reference's own numbers (tests/golden/generator_spatial_code_tiny.npz), against the glue formulation and against the
vector-code decode, and its memory against the vector-code decode."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import sae_oracle as O, spatial_oracle as SO
from oracle.fixtures import load_golden, perturbed_state_dict, rel_err, rel_l2, rnd
from swapping_autoencoder_pytorch_b200 import backend, default_options, networks

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL_TF32 = 1e-3
TOL_NET = 3e-3
# Gradients behind a leaky-ReLU: the activation mask flips (slope 1 <-> 0.2) where a pre-activation lies within TF32 rounding of
# zero, about 1 element in 1000.  A style-map cell sums ~10^4 such products, ~10 of them flipped: sqrt(10) * 0.8 / sqrt(10^4)
# ~ 2.5 % in L2, the size seen for StyledConv and the generator (max-norm errors are larger and not meaningful there)
TOL_ACT_GRAD = 5e-2


def cuda(t):
    return t.float().to(DEV)


@contextlib.contextmanager
def _kernel_setting(name, value):
    k = backend.kernels()
    prev = getattr(k, name)
    setattr(k, name, value)
    try:
        yield
    finally:
        setattr(k, name, prev)


def _reference(x, s, demod, dy):
    """fp64: x [N,C,H,W], s [Ns,C,hs,ws] -> (y, dx, ds)"""
    x, s = x.double().requires_grad_(), s.double().requires_grad_()
    u = F.interpolate(s, size=x.shape[2:], mode="bilinear", align_corners=False)
    if demod:
        u = u * torch.rsqrt(u.square().mean(dim=1, keepdim=True) + 1e-8)
    y = x * u
    dx, ds = torch.autograd.grad(y, [x, s], dy.double())
    return y.detach(), dx, ds


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _nchw(t):
    return t.permute(0, 3, 1, 2)


RATIOS = {"up": ((4, 4), (256, 256)), "down": ((64, 64), (16, 16)), "equal": ((16, 16), (16, 16)), "fractional": ((3, 4), (6, 7))}


@pytest.mark.parametrize("ratio", sorted(RATIOS))
@pytest.mark.parametrize("c", [5, 8, 128, 512, 1024])
def test_modulate_spatial_kernel_against_fp64(c, ratio):
    (hs, ws), (h, w) = RATIOS[ratio]
    n = 2
    k = backend.kernels()
    gen = torch.Generator(device=DEV).manual_seed(c * 131 + h)
    x = torch.randn(n, c, h, w, device=DEV, generator=gen)
    dy = torch.randn(n, c, h, w, device=DEV, generator=gen)
    for ns in (1, n):
        s = torch.randn(ns, c, hs, ws, device=DEV, generator=gen) * 0.5 + 1.0
        for demod in (True, False):
            y_r, dx_r, ds_r = _reference(x, s, demod, dy)
            for rounding, tol in ((True, 5e-4), (False, 2e-6)):
                with _kernel_setting("round_tf32", rounding):
                    y = k.modulate_spatial(_nhwc(x), _nhwc(s), demod)
                    dx, ds = k.modulate_spatial_backward(_nhwc(dy), _nhwc(x), _nhwc(s), demod)
                errs = (rel_err(_nchw(y), y_r), rel_err(_nchw(dx), dx_r), rel_err(_nchw(ds), ds_r))
                # ds sums up to N (H / hs) (W / ws) products per cell in fp32; it is never rounded to TF32
                assert errs[0] < tol and errs[1] < tol and errs[2] < 2e-6, (ns, demod, rounding, errs)


def test_modulate_spatial_backward_is_deterministic():
    k = backend.kernels()
    gen = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(4, 128, 128, 128, device=DEV, generator=gen)
    dy = torch.randn(4, 128, 128, 128, device=DEV, generator=gen)
    for s in (torch.randn(1, 128, 7, 9, device=DEV, generator=gen), torch.randn(4, 128, 16, 16, device=DEV, generator=gen)):
        a = k.modulate_spatial_backward(_nhwc(dy), _nhwc(x), _nhwc(s), True)
        b = k.modulate_spatial_backward(_nhwc(dy), _nhwc(x), _nhwc(s), True)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_modulate_spatial_rejects_bad_maps():
    from swapping_autoencoder_pytorch_b200.stylegan2_op import modulate_spatial
    x = torch.randn(2, 8, 6, 6, device=DEV)
    for bad in (torch.randn(3, 8, 2, 2, device=DEV), torch.randn(2, 4, 2, 2, device=DEV)):
        with pytest.raises(ValueError):
            modulate_spatial(x, bad, True)


# ------------------------------------------------------------------------------------------------ layers vs the oracle
def _load(module, params):
    sd = module.state_dict()
    sd.update({k: v.float() for k, v in params.items()})
    module.load_state_dict(sd)
    return module.to(DEV)


def _grads(y, wgt, inputs):
    return torch.autograd.grad((y * wgt).sum(), inputs)


def _check(y, y_r, grads, grads_r, through_activation=False):
    """values max-norm at the per-op TF32 tolerance; gradients likewise, except behind a leaky-ReLU (TOL_ACT_GRAD)"""
    assert rel_err(y, y_r) < TOL_TF32, rel_err(y, y_r)
    for i, (g, g_r) in enumerate(zip(grads, grads_r)):
        if through_activation:
            assert rel_l2(g, g_r) < TOL_ACT_GRAD, (i, rel_l2(g, g_r), rel_err(g, g_r))
        else:
            assert rel_err(g, g_r) < (2 + i) * TOL_TF32, (i, rel_err(g, g_r))


@pytest.mark.parametrize("kind", ["plain", "upsample", "downsample"])
def test_modulated_conv_with_code_map(kind):
    from swapping_autoencoder_pytorch_b200 import stylegan2_layers as L
    cin, cout = 32, 64
    P = {"weight": rnd(1, 1, cout, cin, 3, 3), "modulation.weight": rnd(2, cin, 16), "modulation.bias": rnd(3, cin) * 0.1 + 1}
    m = _load(L.ModulatedConv2d(cin, cout, 3, 16, upsample=kind == "upsample", downsample=kind == "downsample"), P)
    x, s = rnd(4, 2, cin, 20, 18), rnd(5, 2, 16, 3, 4)
    xr, sr = x.clone().requires_grad_(), s.clone().requires_grad_()
    PO = {"m." + k: v for k, v in P.items()}
    if kind == "downsample":
        st = O.equal_linear(PO, "m.modulation", F.interpolate(sr, size=(20, 18), mode="bilinear", align_corners=False))
        xm = xr * st * torch.rsqrt(st.square().mean(dim=1, keepdim=True) + 1e-8)
        blur = O.make_kernel([1, 3, 3, 1], torch.float64)
        w = P["weight"][0] / math.sqrt(cin * 9)
        w = w * torch.rsqrt(w.square().sum(dim=(1, 2, 3), keepdim=True) + 1e-8)
        y_r = F.conv2d(O.upfirdn2d(xm, blur, pad=(2, 2)), w, stride=2)
    else:
        y_r = SO.modulated_conv2d(PO, "m", xr, sr, 3, upsample=kind == "upsample")
    wgt = rnd(6, *y_r.shape)
    xg, sg = cuda(x).requires_grad_(), cuda(s).requires_grad_()
    y = m(xg, sg)
    _check(y, y_r, _grads(y, cuda(wgt), [xg, sg]), _grads(y_r, wgt, [xr, sr]))


@pytest.mark.parametrize("upsample", [False, True])
def test_styled_conv_with_code_map(upsample):
    from swapping_autoencoder_pytorch_b200 import stylegan2_layers as L
    P = {"conv.weight": rnd(10, 1, 32, 32, 3, 3), "conv.modulation.weight": rnd(11, 32, 16), "conv.modulation.bias": rnd(12, 32) * 0.1 + 1,
         "noise.weight": torch.tensor([0.3], dtype=torch.float64), "activate.bias": rnd(13, 32) * 0.1}
    m = _load(L.StyledConv(32, 32, 3, 16, upsample=upsample), P)
    x, s = rnd(14, 2, 32, 16, 16), rnd(15, 2, 16, 5, 3)
    hw = 32 if upsample else 16
    nz = rnd(16, 2, 1, hw, hw)
    xr, sr = x.clone().requires_grad_(), s.clone().requires_grad_()
    y_r = SO.styled_conv({"s." + k: v for k, v in P.items()}, "s", xr, sr, upsample=upsample, noise=nz)
    wgt = rnd(17, *y_r.shape)
    xg, sg = cuda(x).requires_grad_(), cuda(s).requires_grad_()
    y = m(xg, sg, noise=cuda(nz))
    _check(y, y_r, _grads(y, cuda(wgt), [xg, sg]), _grads(y_r, wgt, [xr, sr]), through_activation=True)


def test_torgb_with_code_map():
    from swapping_autoencoder_pytorch_b200 import stylegan2_layers as L
    from swapping_autoencoder_pytorch_b200.stylegan2_op import conv as C
    P = {"conv.weight": rnd(20, 1, 3, 64, 1, 1), "conv.modulation.weight": rnd(21, 64, 16), "conv.modulation.bias": rnd(22, 64) * 0.1 + 1,
         "bias": rnd(23, 1, 3, 1, 1) * 0.1}
    m = _load(L.ToRGB(64, 16, upsample=False), P)
    x, s = rnd(24, 2, 64, 32, 32), rnd(25, 2, 16, 4, 4)
    xr, sr = x.clone().requires_grad_(), s.clone().requires_grad_()
    y_r = SO.modulated_conv2d({"t." + k: v for k, v in P.items()}, "t.conv", xr, sr, 1, demodulate=False) + P["bias"]
    wgt = rnd(26, *y_r.shape)
    xg, sg = cuda(x).requires_grad_(), cuda(s).requires_grad_()
    calls = []
    orig = C._ToRGB.forward
    C._ToRGB.forward = staticmethod(lambda *a: calls.append(1) or orig(*a))
    try:
        y = m(xg, sg)
    finally:
        C._ToRGB.forward = staticmethod(orig)
    assert calls, "a code map must take the ToRGB kernel wherever a texture vector does"
    _check(y, y_r, _grads(y, cuda(wgt), [xg, sg]), _grads(y_r, wgt, [xr, sr]))


def test_generator_modulation_with_code_map():
    from swapping_autoencoder_pytorch_b200.networks.generator import GeneratorModulation
    P = {"scale.weight": rnd(30, 8, 16), "scale.bias": rnd(31, 8) * 0.1, "bias.weight": rnd(32, 8, 16), "bias.bias": rnd(33, 8) * 0.1}
    m = _load(GeneratorModulation(16, 8), P)
    x, s = rnd(34, 2, 8, 16, 16), rnd(35, 2, 16, 3, 5)
    xr, sr = x.clone().requires_grad_(), s.clone().requires_grad_()
    st = F.interpolate(sr, size=(16, 16), mode="bilinear", align_corners=False)
    y_r = xr * O.equal_linear(P, "scale", st) + O.equal_linear(P, "bias", st)
    wgt = rnd(36, *y_r.shape)
    xg, sg = cuda(x).requires_grad_(), cuda(s).requires_grad_()
    y = m(xg, sg)
    _check(y, y_r, _grads(y, cuda(wgt), [xg, sg]), _grads(y_r, wgt, [xr, sr]))


# ------------------------------------------------------------------------------------------------ networks
def _generator(**over):
    opt = default_options(**dict(dict(num_gpus=1), **over))
    torch.manual_seed(0)
    return opt, networks.create_network(opt, opt.netG, "generator").to(DEV)


def test_tiny_generator_against_reference_code_map():
    meta, G = load_golden("generator_spatial_code_tiny")
    opt, g = _generator(**dict(meta["opt"], num_gpus=1))
    sd = perturbed_state_dict(default_options(**meta["opt"]))
    own = g.state_dict()
    own.update({k[2:]: v.float().to(DEV) for k, v in sd.items() if k.startswith("G.") and k[2:] in own})
    g.load_state_dict(own)
    sp = cuda(rnd(meta["sp_seed"], 1, opt.spatial_code_ch, 8, 8)).requires_grad_()
    code_map = cuda(rnd(meta["map_seed"], *meta["map_shape"])).requires_grad_()
    g(sp.detach(), code_map.detach())
    g.fix_and_gather_noise_parameters()
    mods = dict(g.named_modules())
    for i, (name, shape) in enumerate(zip(meta["noise_names"], meta["noise_shapes"])):
        mods[name].fixed_noise = torch.nn.Parameter(cuda(rnd(meta["noise_seed0"] + i, *shape)))
    weight = dict(g.named_parameters())[meta["weight_grad"][2:]]
    img = g(sp, code_map)
    g_map, g_sp, g_w = _grads(img, cuda(rnd(meta["weight_seed"], *img.shape)), [code_map, sp, weight])
    assert rel_err(img, G["img"]) < TOL_NET, rel_err(img, G["img"])
    errs = [rel_l2(a, G[k]) for a, k in ((g_map, "grad_map"), (g_sp, "grad_sp"), (g_w, "grad_weight"))]
    assert max(errs) < TOL_ACT_GRAD, errs


def _default_256(batch):
    opt, g = _generator()
    gen = torch.Generator(device=DEV).manual_seed(11)
    sp = torch.randn(batch, opt.spatial_code_ch, 16, 16, device=DEV, generator=gen)
    code = torch.randn(batch, opt.global_code_ch, device=DEV, generator=gen)
    with torch.no_grad():
        g(sp, code)
        g.fix_and_gather_noise_parameters()
    return opt, g, sp, code, gen


def test_default_256_native_matches_glue():
    opt, g, sp, _, gen = _default_256(4)
    code_map = torch.randn(4, opt.global_code_ch, 16, 16, device=DEV, generator=gen)
    with torch.no_grad():
        native = g(sp, code_map)
        with _kernel_setting("spatial_style", "glue"):
            glue = g(sp, code_map)
    assert rel_err(native, glue) < TOL_NET, rel_err(native, glue)


def test_default_256_constant_map_and_memory():
    _, g, sp, code, _ = _default_256(4)
    code_map = code[:, :, None, None].expand(-1, -1, 16, 16).contiguous()
    peaks = {}
    with torch.no_grad():
        for tag, c in (("vector", code), ("map", code_map)):
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            out = g(sp, c)
            torch.cuda.synchronize()
            peaks[tag] = (torch.cuda.max_memory_allocated() - base, out)
    assert rel_err(peaks["map"][1], peaks["vector"][1]) < TOL_NET, rel_err(peaks["map"][1], peaks["vector"][1])
    # the map decode may hold one more activation than the vector decode: the plain 3x3 StyledConv takes a modulated copy of its
    # input where a vector code rides in per-sample filters.  At most one copy of the largest one (4 x 128 x 256^2 fp32) —
    # nothing with global_code_ch channels at a layer's resolution
    largest = 4 * 128 * 256 * 256 * 4
    assert peaks["map"][0] <= peaks["vector"][0] + largest, (peaks["map"][0], peaks["vector"][0])


def test_ffhq1024_option_set_decodes_a_code_map():
    opt, g = _generator(crop_size=1024, batch_size=2, netG_scale_capacity=0.8, netE_num_downsampling_sp=5, netE_scale_capacity=0.4,
                        global_code_ch=1536, patch_size=256)
    gen = torch.Generator(device=DEV).manual_seed(12)
    sp = torch.randn(2, opt.spatial_code_ch, 32, 32, device=DEV, generator=gen)
    code_map = torch.randn(2, opt.global_code_ch, 8, 8, device=DEV, generator=gen)
    with torch.no_grad():
        img = g(sp, code_map)
    assert img.shape == (2, 3, 1024, 1024) and torch.isfinite(img).all()

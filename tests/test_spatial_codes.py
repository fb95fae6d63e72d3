"""CPU: texture code maps [N, C, h, w] (region-wise texture editing) through the generator — the oracle and the product on the
kernel emulation against the reference's own generator run with a code map (tests/golden/generator_spatial_code_tiny.npz, written
by oracle/make_golden_spatial.py), plus the invariants the commuted formulation must keep and ``decode_regions``."""
import pytest
import torch
import torch.nn.functional as F

from oracle import sae_oracle as O, spatial_oracle as SO
from oracle.fixtures import TINY, load_golden, perturbed_state_dict, rel_err, rnd
from swapping_autoencoder_pytorch_b200 import backend, default_options
from tests.cpu_emulation import EmulatedKernels

TOL = 1e-9


class SpatialEmulatedKernels(EmulatedKernels):
    """the CPU kernel emulation plus fp64 stand-ins for sae_modulate_spatial and its backward (F.interpolate formulation)"""
    spatial_style = "native"

    def modulate_spatial(self, x, s_lo, demodulate):
        n, h, w, c = x.shape
        u = F.interpolate(s_lo.permute(0, 3, 1, 2), size=(h, w), mode="bilinear", align_corners=False)
        if demodulate:
            u = u * torch.rsqrt(u.square().mean(dim=1, keepdim=True) + 1e-8)
        return x * u.permute(0, 2, 3, 1)

    def modulate_spatial_backward(self, dy, x, s_lo, demodulate):
        xs, ss = x.detach().requires_grad_(), s_lo.detach().requires_grad_()
        with torch.enable_grad():
            y = self.modulate_spatial(xs, ss, demodulate)
        return torch.autograd.grad(y, [xs, ss], dy.detach())


@pytest.fixture(autouse=True)
def spatial_kernels():
    prev = backend.set_kernels(SpatialEmulatedKernels())
    yield
    backend.set_kernels(prev)


def _inputs(meta):
    opt = default_options(**meta["opt"])
    sp = rnd(meta["sp_seed"], 1, opt.spatial_code_ch, 8, 8)
    code_map = rnd(meta["map_seed"], *meta["map_shape"])
    noises = {name: rnd(meta["noise_seed0"] + i, *shape) for i, (name, shape) in enumerate(zip(meta["noise_names"], meta["noise_shapes"]))}
    return opt, sp, code_map, noises


def _product_model(opt):
    from swapping_autoencoder_pytorch_b200.model import SwappingAutoencoderModel
    model = SwappingAutoencoderModel(opt)
    model.initialize()
    model.double()
    missing, unexpected = model.load_state_dict(perturbed_state_dict(opt), strict=False)
    assert not unexpected
    return model


def _pin_noise(G, noises):
    mods = dict(G.named_modules())
    for name, z in noises.items():
        mods[name].fixed_noise = torch.nn.Parameter(z.clone())


def test_oracle_matches_reference_code_map():
    meta, G = load_golden("generator_spatial_code_tiny")
    opt, sp, code_map, noises = _inputs(meta)
    P = O.OracleModel(opt, perturbed_state_dict(opt)).G
    w_key = meta["weight_grad"][len("G."):]
    P[w_key] = P[w_key].clone().requires_grad_()
    sp, code_map = sp.requires_grad_(), code_map.requires_grad_()
    img = SO.generator_forward(P, opt, sp, code_map, noises={k[:-len(".noise")]: v for k, v in noises.items()})
    g_map, g_sp, g_w = torch.autograd.grad((img * rnd(meta["weight_seed"], *img.shape)).sum(), [code_map, sp, P[w_key]])
    assert rel_err(img, G["img"]) < TOL
    assert rel_err(g_map, G["grad_map"]) < TOL and rel_err(g_sp, G["grad_sp"]) < TOL and rel_err(g_w, G["grad_weight"]) < TOL


def test_product_generator_matches_reference_code_map():
    meta, G = load_golden("generator_spatial_code_tiny")
    opt, sp, code_map, noises = _inputs(meta)
    model = _product_model(opt)
    _pin_noise(model.G, noises)
    weight = dict(model.named_parameters())[meta["weight_grad"]]
    sp, code_map = sp.requires_grad_(), code_map.requires_grad_()
    img = model.G(sp, code_map)
    g_map, g_sp, g_w = torch.autograd.grad((img * rnd(meta["weight_seed"], *img.shape)).sum(), [code_map, sp, weight])
    assert rel_err(img, G["img"]) < TOL
    assert rel_err(g_map, G["grad_map"]) < TOL and rel_err(g_sp, G["grad_sp"]) < TOL and rel_err(g_w, G["grad_weight"]) < TOL


def test_native_formulation_equals_glue():
    """the commuted formulation (affine at the map's resolution, one interpolation of its result) against the reference's
    (map interpolated to every layer, affine there), which a kernel set without native code maps runs"""
    meta, _ = load_golden("generator_spatial_code_tiny")
    opt, sp, code_map, noises = _inputs(meta)
    model = _product_model(opt)
    _pin_noise(model.G, noises)
    with torch.no_grad():
        native = model.G(sp, code_map)
        prev = backend.set_kernels(EmulatedKernels())
        try:
            glue = model.G(sp, code_map)
        finally:
            backend.set_kernels(prev)
    assert rel_err(native, glue) < 1e-12


def test_constant_map_equals_vector_code():
    meta, _ = load_golden("generator_spatial_code_tiny")
    opt, sp, _, noises = _inputs(meta)
    model = _product_model(opt)
    _pin_noise(model.G, noises)
    code = rnd(1200, 1, opt.global_code_ch)
    with torch.no_grad():
        a = model.G(sp, code)
        b = model.G(sp, code[:, :, None, None].expand(-1, -1, 3, 5))
    assert rel_err(b, a) < 1e-12


def test_batch_of_maps_is_per_sample():
    opt = default_options(**TINY)
    model = _product_model(opt)
    sp = rnd(1210, 2, opt.spatial_code_ch, 8, 8)
    code_map = rnd(1211, 2, opt.global_code_ch, 4, 3)
    model.G(sp, code_map)
    noise = {name: rnd(1220 + i, 2, 1, *m.image_size[2:]) for i, (name, m) in enumerate(model.G.named_modules())
             if type(m).__name__ == "NoiseInjection"}
    _pin_noise(model.G, noise)
    with torch.no_grad():
        both = model.G(sp, code_map)
        for i in range(2):
            _pin_noise(model.G, {k: v[i:i + 1] for k, v in noise.items()})
            assert rel_err(model.G(sp[i:i + 1], code_map[i:i + 1]), both[i:i + 1]) < 1e-12


def test_decode_regions():
    opt = default_options(**TINY)
    model = _product_model(opt)
    sp = rnd(1230, 2, opt.spatial_code_ch, 8, 8)
    codes = rnd(1231, 2, 3, opt.global_code_ch)
    model(sp, codes[:, 0], command="decode")
    model.G.fix_and_gather_noise_parameters()
    masks = torch.zeros(2, 3, 5, 4, dtype=torch.float64)
    masks[:, 1] = 1.0
    with torch.no_grad():
        ref = model(sp, codes[:, 1], command="decode")
        out = model(sp, codes, masks, command="decode_regions")
        assert rel_err(out, ref) < 1e-12
        # two regions: left half code 0, right half code 2
        masks.zero_()
        masks[:, 0, :, :2] = 1.0
        masks[:, 2, :, 2:] = 1.0
        assert torch.isfinite(model(sp, codes, masks, command="decode_regions")).all()
        with pytest.raises(ValueError):
            model(sp, codes, masks * 0.5, command="decode_regions")          # does not sum to 1
        bad = masks.clone()
        bad[:, 0], bad[:, 1] = bad[:, 0] + 0.5, bad[:, 1] - 0.5
        with pytest.raises(ValueError):
            model(sp, codes, bad, command="decode_regions")                  # negative weights
        with pytest.raises(ValueError):
            model(sp, codes, masks[:, :2], command="decode_regions")         # K differs between codes and masks

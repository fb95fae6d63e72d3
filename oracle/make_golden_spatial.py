"""ORACLE SUPPORT — writes tests/golden/generator_spatial_code_tiny.npz by running the REFERENCE ITSELF (native-PyTorch CPU path,
fp64) with a texture code map; the companion of oracle/make_golden.py, with the same requirements (a reference checkout, see
oracle/ref_import.py):
    python oracle/make_golden_spatial.py
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_import  # noqa: E402
from oracle.fixtures import TINY, rnd  # noqa: E402
from oracle.make_golden import build_ref_model, save  # noqa: E402
from swapping_autoencoder_pytorch_b200 import default_options  # noqa: E402


def gen_spatial_codes(R):
    """The reference's own StyleGAN2ResnetGenerator driven by a texture code MAP (generator.py:62-67, stylegan2_layers.py:269-276):
    TINY options, perturbed parameters, noise pinned as in gen_networks, batch 1 (the reference's spatial branch only survives
    batch 1), a 3 x 5 map (no integer ratio to any layer).  Output image and the gradients with respect to the map, the
    structure code and one modulation weight."""
    opt = default_options(**TINY)
    model, _ = build_ref_model(R, opt)
    G = model.G
    sp = rnd(1100, 1, opt.spatial_code_ch, 8, 8)
    code_map = rnd(1101, 1, opt.global_code_ch, 3, 5)
    G(sp, rnd(1102, 1, opt.global_code_ch))             # one pass so every NoiseInjection knows its map size
    G.fix_and_gather_noise_parameters()
    noises = {}
    idx = 0
    for name, m in G.named_modules():
        if type(m).__name__ == "NoiseInjection":
            z = rnd(1110 + idx, *m.fixed_noise.shape)
            m.fixed_noise = torch.nn.Parameter(z)
            noises[name] = z
            idx += 1
    sp_ = sp.clone().requires_grad_()
    map_ = code_map.clone().requires_grad_()
    w_name = "UpsamplingResBlock16.conv1.conv.modulation.weight"
    weight = dict(G.named_parameters())[w_name]
    img = G(sp_, map_)
    wt = rnd(1103, *img.shape)
    g_map, g_sp, g_w = torch.autograd.grad((img * wt).sum(), [map_, sp_, weight])
    save("generator_spatial_code_tiny", dict(opt=TINY, param_seed=7, bias_seed=11, sp_seed=1100, map_seed=1101, map_shape=list(code_map.shape),
                                             weight_seed=1103, noise_seed0=1110, noise_names=list(noises.keys()),
                                             noise_shapes=[list(v.shape) for v in noises.values()], weight_grad="G." + w_name),
         img=img, grad_map=g_map, grad_sp=g_sp, grad_weight=g_w)


def main():
    torch.set_default_dtype(torch.float32)
    gen_spatial_codes(ref_import.import_reference())


if __name__ == "__main__":
    main()

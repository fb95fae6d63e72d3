"""ORACLE SUPPORT — deterministic inputs shared by oracle/make_golden.py and tests/ (test infrastructure only)."""
import json
import os

import numpy as np
import torch

from . import sae_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# reduced-capacity option set of the golden network fixtures (same topology as the defaults, 64x64 images)
TINY = dict(num_gpus=0, crop_size=64, batch_size=2, netE_num_downsampling_sp=3, netE_scale_capacity=0.25,
            global_code_ch=128, netG_scale_capacity=0.125, netD_scale_capacity=0.125, netPatchD_scale_capacity=0.5,
            netPatchD_max_nc=32, patch_size=32, patch_num_crops=2)


def rnd(seed, *shape, dtype=torch.float64):
    """standard-normal tensor from NumPy's legacy generator (bit-stable across machines)"""
    return torch.from_numpy(np.random.RandomState(seed).standard_normal(shape)).to(dtype)


def perturbed_state_dict(opt, dtype=torch.float64, param_seed=7, bias_seed=11):
    """init_state_dict + non-zero biases and noise weights so that parity checks exercise every term"""
    sd = O.init_state_dict(opt, seed=param_seed, dtype=dtype)
    rs = np.random.RandomState(bias_seed)
    for k in sd:
        if k.endswith(".bias") and "modulation" not in k:
            sd[k] = sd[k] + torch.from_numpy(rs.standard_normal(tuple(sd[k].shape)) * 0.1).to(dtype)
        if k.endswith("noise.weight"):
            sd[k] = sd[k] + 0.05
    return sd


def surface_steps(make_model, make_trainer):
    """One D half-step with R1 (double backward) and one G half-step of the TINY nets at the perturbed parameters, seeded;
    returns the losses of both and a checksum of the updated parameters.  ``make_model(opt)`` returns a model wrapper,
    ``make_trainer(opt, wrapper)`` its training driver.  Run with fp64 as the default dtype."""
    import contextlib
    import io
    from swapping_autoencoder_pytorch_b200 import default_options
    opt = default_options(**dict(TINY, R1_once_every=1))
    sd = perturbed_state_dict(opt, dtype=torch.float64)
    real = rnd(900, 2, 3, 64, 64).clamp(-1, 1)
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        wrapper = make_model(opt)
    inner = wrapper.singlegpu_model
    missing, unexpected = inner.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    trainer = make_trainer(opt, wrapper)
    torch.manual_seed(1)
    out = {}
    for tag in ("D", "G"):
        losses = trainer.train_one_step({"real_A": real}, 0)
        out.update({tag + "/" + k: float(v) for k, v in losses.items()})
    with torch.no_grad():
        out["param_checksum"] = float(sum(p.double().abs().sum() for p in inner.parameters()))
    return out


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    arrays = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta"}
    return meta, arrays


def rel_err(a, b):
    """max|a-b| / max|b|  — the tolerance metric of BASELINE.json ("1e-3 rel"), SURVEY.md §9.5"""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def rel_l2(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))

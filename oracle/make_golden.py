"""ORACLE SUPPORT — generates tests/golden/*.npz by running the REFERENCE ITSELF (native-PyTorch CPU path, fp64).

Needs a checkout of the reference (``SAE_REFERENCE_ROOT``, see oracle/ref_import.py):
    python oracle/make_golden.py [ops layers networks surface contract ref_checkpoint ref_surface_steps]
The fixtures are small (inputs are seeded, parameters are re-derived from a seed by
``sae_oracle.init_state_dict``; only outputs / gradients are stored) and are committed, so a machine without the
reference checkout can still check the oracle and the CUDA path against the reference's numbers.
"""
import contextlib
import hashlib
import io
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_import, sae_oracle as O            # noqa: E402
from swapping_autoencoder_pytorch_b200 import default_options  # noqa: E402  (option Namespace only; no kernels)

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
DT = torch.float64

from oracle.fixtures import TINY, perturbed_state_dict, rnd  # noqa: E402


def save(name, meta, **arrays):
    os.makedirs(OUT, exist_ok=True)
    arrs = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), meta=json.dumps(meta), **arrs)
    print("wrote", name, {k: v.shape for k, v in arrs.items()})


FIR_CASES = [
    # (taps, gain, up, down, pad) — every configuration the hot path uses (SURVEY.md §8 a1) + the up/down=2 API modes
    ([1, 3, 3, 1], 1, 1, 1, (2, 2)), ([1, 3, 3, 1], 1, 1, 1, (1, 1)), ([1, 3, 3, 1], 4, 1, 1, (1, 1)),
    ([1, 2, 1], 1, 1, 1, (0, 0)), ([1, 2, 1], 1, 1, 1, (1, 0)), ([1], 1, 1, 1, (0, 0)),
    ([1, 3, 3, 1], 4, 2, 1, (2, 1)), ([1, 3, 3, 1], 1, 1, 2, (1, 1)), ([1, 3, 3, 1], 1, 1, 1, (0, -1)),
    ([1, 3, 3, 1], 1, 1, 1, (2, 1)), ([1, 2, 1], 1, 2, 2, (1, 1)),
]


def gen_ops(R):
    fir = {}
    meta = []
    for i, (taps, gain, up, down, pad) in enumerate(FIR_CASES):
        k = R.layers.make_kernel(taps).to(DT) * gain
        x = rnd(100 + i, 2, 3, 9, 10).requires_grad_()
        y = R.ops.upfirdn2d(x, k, up=up, down=down, pad=pad)
        w = rnd(200 + i, *y.shape)
        gx, = torch.autograd.grad((y * w).sum(), x, create_graph=True)
        # second order: d/dw of sum(gx * v)
        meta.append(dict(taps=taps, gain=gain, up=up, down=down, pad=list(pad)))
        fir["y%d" % i] = y
        fir["gx%d" % i] = gx
    save("ops_upfirdn2d", dict(cases=meta, x_seed0=100, w_seed0=200, shape=[2, 3, 9, 10]), **fir)

    act = {}
    for i, shape in enumerate([(2, 4, 5, 6), (3, 8)]):
        x = rnd(300 + i, *shape).requires_grad_()
        b = rnd(310 + i, shape[1]).requires_grad_()
        y = R.ops.fused_leaky_relu(x, b)
        w = rnd(320 + i, *shape)
        gx, gb = torch.autograd.grad((y * w).sum(), [x, b])
        act.update({"y%d" % i: y, "gx%d" % i: gx, "gb%d" % i: gb})
    save("ops_fused_leaky_relu", dict(shapes=[[2, 4, 5, 6], [3, 8]], x_seed0=300, b_seed0=310, w_seed0=320), **act)


def load_module(mod, params):
    mod.double()                       # convert first: loading into fp32 storage would round the fp64 values
    sd = mod.state_dict()
    for k in sd:
        if k in params:
            sd[k] = params[k].to(DT)
    mod.load_state_dict(sd)
    return mod


def gen_layers(R):
    L = R.layers
    out = {}
    meta = {}
    # ModulatedConv2d variants
    for i, (cin, cout, k, demod, up) in enumerate([(8, 12, 3, True, False), (8, 12, 3, True, True), (8, 3, 1, False, False)]):
        m = L.ModulatedConv2d(cin, cout, k, 16, demodulate=demod, upsample=up)
        P = {"weight": rnd(400 + i, 1, cout, cin, k, k), "modulation.weight": rnd(410 + i, cin, 16),
             "modulation.bias": rnd(420 + i, cin) * 0.1 + 1}
        load_module(m, P)
        x = rnd(430 + i, 2, cin, 6, 7).requires_grad_()
        s = rnd(440 + i, 2, 16).requires_grad_()
        y = m(x, s)
        w = rnd(450 + i, *y.shape)
        gx, gs, gw = torch.autograd.grad((y * w).sum(), [x, s, m.weight])
        out.update({"modconv%d_y" % i: y, "modconv%d_gx" % i: gx, "modconv%d_gs" % i: gs, "modconv%d_gw" % i: gw})
    meta["modconv"] = [[8, 12, 3, True, False], [8, 12, 3, True, True], [8, 3, 1, False, False]]
    # ConvLayer / ResBlock variants incl. reflection pad + [1,2,1] blur (encoder) and the discriminators' [1,3,3,1]
    for i, (cin, cout, blur, refl, down) in enumerate([(8, 16, [1, 3, 3, 1], False, True), (8, 16, [1, 2, 1], True, True),
                                                        (8, 16, [1, 3, 3, 1], False, False)]):
        m = L.ResBlock(cin, cout, blur, reflection_pad=refl, downsample=down)
        P = {"conv1.Conv.weight": rnd(500 + i, cin, cin, 3, 3), "conv1.Act.bias": rnd(510 + i, cin) * 0.1,
             "conv2.Conv.weight": rnd(520 + i, cout, cin, 3, 3), "conv2.Act.bias": rnd(530 + i, cout) * 0.1,
             "skip.Conv.weight": rnd(540 + i, cout, cin, 1, 1)}
        load_module(m, P)
        x = rnd(550 + i, 2, cin, 10, 10).requires_grad_()
        y = m(x)
        w = rnd(560 + i, *y.shape)
        gx, = torch.autograd.grad((y * w).sum(), x, create_graph=True)
        # R1-style second order: gradient of |gx|^2 w.r.t. the first conv weight
        gg, = torch.autograd.grad(gx.pow(2).sum(), m.conv1.Conv.weight)
        out.update({"resblock%d_y" % i: y, "resblock%d_gx" % i: gx, "resblock%d_gg" % i: gg})
    meta["resblock"] = [[8, 16, [1, 3, 3, 1], False, True], [8, 16, [1, 2, 1], True, True], [8, 16, [1, 3, 3, 1], False, False]]
    # StyledConv with explicit noise and non-zero noise weight
    for i, up in enumerate([False, True]):
        m = L.StyledConv(8, 8, 3, 16, upsample=up)
        P = {"conv.weight": rnd(600 + i, 1, 8, 8, 3, 3), "conv.modulation.weight": rnd(610 + i, 8, 16),
             "conv.modulation.bias": torch.ones(8, dtype=DT), "noise.weight": torch.tensor([0.3], dtype=DT),
             "activate.bias": rnd(620 + i, 8) * 0.1}
        load_module(m, P)
        x = rnd(630 + i, 2, 8, 5, 5)
        s = rnd(640 + i, 2, 16)
        hw = 10 if up else 5
        nz = rnd(650 + i, 2, 1, hw, hw)
        out["styled%d_y" % i] = m(x, s, noise=nz)
    # EqualLinear
    m = L.EqualLinear(16, 8, activation='fused_lrelu')
    load_module(m, {"weight": rnd(700, 8, 16), "bias": rnd(701, 8) * 0.1})
    out["linear_act_y"] = m(rnd(702, 3, 16))
    m = L.EqualLinear(16, 8, bias_init=1)
    load_module(m, {"weight": rnd(703, 8, 16), "bias": rnd(704, 8)})
    out["linear_y"] = m(rnd(705, 3, 16))
    save("layers", meta, **out)


def build_ref_model(R, opt):
    model = R.sae_model.SwappingAutoencoderModel(opt)
    with contextlib.redirect_stdout(io.StringIO()):
        model.initialize()
    sd = perturbed_state_dict(opt, dtype=DT, param_seed=7, bias_seed=11)
    model = model.double()
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all(k.endswith(".kernel") or k == "num_discriminator_iters" for k in missing), missing
    return model, sd


def gen_networks(R):
    opt = default_options(**TINY)
    model, sd = build_ref_model(R, opt)
    real = rnd(900, 2, 3, 64, 64).clamp(-1, 1)
    out = {}
    torch.manual_seed(5)
    sp, gl = model.E(real)
    out["sp"], out["gl"] = sp, gl
    # fix the generator noise so its output is deterministic
    torch.manual_seed(6)
    model.G(sp, gl)
    noise_params = model.G.fix_and_gather_noise_parameters()
    noises = {}
    idx = 0
    for name, m in model.G.named_modules():
        if type(m).__name__ == "NoiseInjection":
            z = rnd(950 + idx, *m.fixed_noise.shape)
            m.fixed_noise = torch.nn.Parameter(z)          # fp64 (the helper allocates fp32 noise)
            noises[name] = z
            idx += 1
    out["rec"] = model.G(sp, gl)
    out["d_real"] = model.D(real)
    crops = rnd(901, 2, 2, 3, 32, 32)
    f1 = model.Dpatch.extract_features(crops, aggregate=True)
    f2 = model.Dpatch.extract_features(rnd(902, 2, 2, 3, 32, 32))
    out["patch_feat_agg"], out["patch_feat"] = f1, f2
    out["patch_pred"] = model.Dpatch.discriminate_features(f1, f2)
    save("networks_tiny", dict(opt=TINY, param_seed=7, bias_seed=11, real_seed=900, noise_seed0=950,
                               noise_names=list(noises.keys()), noise_shapes=[list(v.shape) for v in noises.values()], crop_seeds=[901, 902]), **out)

    # loss graph with the generator noise re-randomised (weights small): fix RNG seed, compare losses + a few grads
    model.G.remove_noise_parameters(None)
    losses = {}
    # the reference builds its crop grids in the default dtype (util/util.py:326-335): run this part in fp64 defaults
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(21)
    dl, _, _, _ = model.compute_discriminator_losses(real)
    for k, v in dl.items():
        losses["D/" + k] = v
    torch.manual_seed(22)
    gl_, gm = model.compute_generator_losses(real, None, None)
    for k, v in gl_.items():
        losses["G/" + k] = v
    torch.manual_seed(23)
    r1 = model.compute_R1_loss(real.clone())
    losses["R1/D_R1"] = r1["D_R1"]
    # gradient of the R1 loss w.r.t. D's first ResBlock conv weight (double backward through conv/FIR/act/linear)
    w = model.D.stylegan2_D.convs[1].conv1.Conv.weight
    g, = torch.autograd.grad(r1["D_R1"].mean(), w)
    losses["R1/grad_D_convs1_conv1"] = g
    wp = model.Dpatch.convs[1].conv2.Conv.weight
    torch.manual_seed(23)
    r1b = model.compute_R1_loss(real.clone())
    gp, = torch.autograd.grad(r1b["D_R1"].mean(), wp)
    losses["R1/grad_Dpatch_convs1_conv2"] = gp
    torch.set_default_dtype(torch.float32)
    save("losses_tiny", dict(opt=TINY, param_seed=7, bias_seed=11, real_seed=900, seeds=dict(D=21, G=22, R1=23)), **losses)


def gen_surface_branches(R):
    """Branches of the operator surface that training does not exercise but evaluation / the original StyleGAN2 classes
    do (SURVEY.md §8 f4): Upsample / Downsample modules, ToRGB with an upsampled skip, ModulatedConv2d with a spatially
    varying style and with downsample=True, the original Generator class, encoder feature extraction."""
    L = R.layers
    out = {}
    x = rnd(1000, 2, 4, 7, 6).requires_grad_()
    for name, mod in (("upsample", L.Upsample([1, 3, 3, 1])), ("downsample", L.Downsample([1, 3, 3, 1]))):
        mod = mod.double()
        y = mod(x)
        w = rnd(1001, *y.shape)
        gx, = torch.autograd.grad((y * w).sum(), x)
        out[name + "_y"], out[name + "_gx"] = y, gx
    m = L.ToRGB(8, 16, upsample=True)
    load_module(m, {"conv.weight": rnd(1010, 1, 3, 8, 1, 1), "conv.modulation.weight": rnd(1011, 8, 16),
                    "conv.modulation.bias": rnd(1012, 8) * 0.1 + 1, "bias": rnd(1013, 1, 3, 1, 1) * 0.1})
    out["torgb_skip_y"] = m(rnd(1014, 2, 8, 10, 10), rnd(1015, 2, 16), skip=rnd(1016, 2, 3, 5, 5))
    m = L.ModulatedConv2d(8, 12, 3, 16)
    P = {"weight": rnd(1020, 1, 12, 8, 3, 3), "modulation.weight": rnd(1021, 8, 16), "modulation.bias": rnd(1022, 8) * 0.1 + 1}
    load_module(m, P)
    # spatially varying style, interpolated to the input size.  Batch 1: the reference's branch broadcasts
    # [B,C,H,W] * [B,1,C,H,W] into a 5-D tensor and only survives its own .view() when B == 1 (stylegan2_layers.py:269-276)
    xs = rnd(1023, 1, 8, 6, 7).requires_grad_()
    ss = rnd(1024, 1, 16, 3, 4).requires_grad_()
    y = m(xs, ss)
    w = rnd(1025, *y.shape)
    gx, gs = torch.autograd.grad((y * w).sum(), [xs, ss])
    out.update({"modconv_spatial_y": y, "modconv_spatial_gx": gx, "modconv_spatial_gs": gs})
    m = L.ModulatedConv2d(8, 12, 3, 16, downsample=True)
    load_module(m, P)
    out["modconv_down_y"] = m(rnd(1026, 2, 8, 8, 8), rnd(1027, 2, 16))
    # the original StyleGAN2 synthesis network at its smallest size, fixed noise buffers
    torch.manual_seed(31)
    g = L.Generator(8, 16, 2, channel_multiplier=1).double()
    sd = g.state_dict()
    rs = np.random.RandomState(1030)
    for k in sorted(sd):
        if sd[k].dtype.is_floating_point and not k.endswith(".kernel"):
            sd[k] = torch.from_numpy(rs.standard_normal(tuple(sd[k].shape))).to(DT) * (0.1 if k.endswith("bias") or "noise" in k else 1.0)
    g.load_state_dict(sd)
    img, _ = g([rnd(1031, 2, 16)], randomize_noise=False)
    out["generator8_img"] = img
    save("surface_branches", dict(state_seed=1030, keys=sorted(k for k in sd if sd[k].dtype.is_floating_point and not k.endswith(".kernel"))),
         **out)

    # encoder feature extraction (evaluation path, encoder.py:93-107) on the tiny networks of the other fixtures
    opt = default_options(**TINY)
    model, sd = build_ref_model(R, opt)
    real = rnd(900, 2, 3, 64, 64).clamp(-1, 1)
    sp, gl, feat = model.E(real, extract_features=True)
    save("encoder_features_tiny", dict(opt=TINY, param_seed=7, bias_seed=11, real_seed=900), sp=sp, gl=gl, feature=feat)


def gen_state_dict_contract(R):
    """names, shapes and dtypes of the reference model's state_dict (what its checkpoints contain) for the default 256x256
    option set and for the reduced one — the contract reference checkpoints are loaded by (SURVEY.md §8(b), f3)"""
    contract = {}
    for label, over in (("default256", dict(num_gpus=0)), ("tiny", TINY)):
        opt = default_options(**over)
        model = R.sae_model.SwappingAutoencoderModel(opt)
        with contextlib.redirect_stdout(io.StringIO()):
            model.initialize()
        contract[label] = {k: [list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in model.state_dict().items()}
        print("state_dict contract", label, len(contract[label]), "tensors")
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "state_dict_contract.json"), "w") as f:
        json.dump(contract, f, indent=0, sort_keys=True)


def tensor_sha256(t):
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


def gen_reference_checkpoint(R):
    """What the reference's own ``BaseModel.save`` (models/base_model.py:33-41) writes for the TINY model at the perturbed
    fp32 parameters: the directory layout (checkpoint file and ``latest`` symlink), the ordered keys with dtype, shape and
    SHA-256 of every tensor, the state_dict's ``_metadata``, the full values of the tensors that are not re-derived from the parameter seeds, and the
    reference encoder's outputs for the seeded image.  The file itself (80 MB) is not stored: the test rebuilds it."""
    opt = default_options(**TINY)
    sd = perturbed_state_dict(opt, dtype=torch.float32, param_seed=7, bias_seed=11)
    with tempfile.TemporaryDirectory() as tmp:
        opt.checkpoints_dir, opt.name = tmp, "written_by_reference"
        model = R.sae_model.SwappingAutoencoderModel(opt)
        with contextlib.redirect_stdout(io.StringIO()):
            model.initialize()
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected, unexpected
        d = os.path.join(tmp, opt.name)
        os.makedirs(d)
        model.save(7000)
        files = [[f, os.readlink(os.path.join(d, f)) if os.path.islink(os.path.join(d, f)) else None]
                 for f in sorted(os.listdir(d))]
        ckpt = torch.load(os.path.join(d, "7k_checkpoint.pth"), map_location="cpu")
    real = rnd(900, 2, 3, 64, 64).clamp(-1, 1).float()
    with torch.no_grad():
        sp, gl = model.E(real)
    tensors = [[k, str(v.dtype).replace("torch.", ""), list(v.shape), tensor_sha256(v)] for k, v in ckpt.items()]
    stored = {"stored." + k: v for k, v in ckpt.items() if k not in sd}
    metadata = [[k, v] for k, v in getattr(ckpt, "_metadata", {}).items()]      # the state_dict's per-module versions
    save("reference_checkpoint", dict(opt=TINY, param_seed=7, bias_seed=11, real_seed=900, total_steps=7000, files=files,
                                      tensors=tensors, metadata=metadata), enc_sp=sp, enc_gl=gl, **stored)


def gen_reference_surface_steps():
    """Losses and updated-parameter checksum of the reference's own model / optimizer / network files run over this
    operator surface (oracle/ref_surface_driver.py, a process of its own)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "oracle", "ref_surface_driver.py"), root,
                          ref_import.REFERENCE_ROOT], capture_output=True, text=True, check=True, cwd=root)
    out = json.loads(res.stdout.strip().splitlines()[-1])
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "reference_surface_steps.json"), "w") as f:
        json.dump({"reference_files": out["reference_files"]}, f, indent=1, sort_keys=True)
    print("wrote reference_surface_steps", out["reference_files"])


def main():
    torch.set_default_dtype(torch.float32)
    R = ref_import.import_reference()
    which = sys.argv[1:] or ["ops", "layers", "networks", "surface", "contract", "ref_checkpoint", "ref_surface_steps"]
    if "ops" in which:
        gen_ops(R)
    if "layers" in which:
        gen_layers(R)
    if "networks" in which:
        gen_networks(R)
    if "surface" in which:
        gen_surface_branches(R)
    if "contract" in which:
        gen_state_dict_contract(R)
    if "ref_checkpoint" in which:
        gen_reference_checkpoint(R)
    if "ref_surface_steps" in which:
        gen_reference_surface_steps()


if __name__ == "__main__":
    main()

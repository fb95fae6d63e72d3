"""CPU: north_star says the reference's ``swapping_autoencoder_model.py`` and ``swapping_autoencoder_optimizer.py``
"consume [the operator surface] unchanged".  ``oracle/ref_surface_driver.py`` imports the reference's own model / optimizer /
network files with ``models.networks.stylegan2_op`` and ``models.networks.stylegan2_layers`` aliased to this package
(INTEGRATION.md §1) and runs a D half-step with R1 (double backward) and a G half-step; its losses and updated-parameter
checksum are stored in ``tests/golden/reference_surface_steps.json`` (``oracle/make_golden.py ref_surface_steps``).  The
same steps through this repo's restated callers (model.py / optimizer.py) on the same parameters and seeds must give the
same losses and the same updated parameters."""
import json
import math
import os

from oracle.fixtures import GOLDEN_DIR, surface_steps


def test_reference_model_and_optimizer_run_on_this_surface(emulated_kernels, fp64_default):
    import swapping_autoencoder_pytorch_b200 as S
    ref = json.load(open(os.path.join(GOLDEN_DIR, "reference_surface_steps.json")))["reference_files"]
    ours = surface_steps(S.create_model, S.create_optimizer)
    for k in ("D/D_real", "D/D_rec", "D/D_mix", "D/PatchD_real", "D/PatchD_mix", "D/D_R1", "D/D_total",
              "G/G_L1", "G/G_GAN_rec", "G/G_GAN_mix", "G/G_mix", "G/L1_dist"):
        assert k in ref and math.isfinite(ref[k]), (k, ref)
    assert set(ref) == set(ours), set(ref) ^ set(ours)
    for k in ref:
        assert abs(ref[k] - ours[k]) <= 1e-9 * max(1.0, abs(ref[k])), (k, ref[k], ours[k])

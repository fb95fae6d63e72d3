"""ORACLE SUPPORT (CPU, needs the reference checkout).  Runs the REFERENCE'S OWN swapping_autoencoder_model.py,
swapping_autoencoder_optimizer.py and network files (encoder / generator / discriminator / patch_discriminator) over this
repo's operator surface — the sys.modules aliasing of INTEGRATION.md §1 — with the kernel interface emulated on the CPU,
and, on the same parameters and RNG seeds, this repo's restated callers.  Prints one JSON line, which
``oracle/make_golden.py ref_surface_steps`` stores for tests/test_reference_on_surface.py.  Own process because it
re-binds ``models.networks.stylegan2_*`` in sys.modules.
usage: python oracle/ref_surface_driver.py <repo root> <reference root>"""
import json
import sys

import torch

ROOT, REF = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
torch.set_default_dtype(torch.float64)

from swapping_autoencoder_pytorch_b200 import backend                      # noqa: E402
import swapping_autoencoder_pytorch_b200 as S                               # noqa: E402
import swapping_autoencoder_pytorch_b200.stylegan2_op as _op                # noqa: E402
import swapping_autoencoder_pytorch_b200.stylegan2_layers as _layers        # noqa: E402
from tests.cpu_emulation import EmulatedKernels                             # noqa: E402
from oracle.fixtures import surface_steps                                   # noqa: E402
from oracle.ref_import import install_stubs                                 # noqa: E402

backend.set_kernels(EmulatedKernels())
install_stubs()
sys.path.insert(0, REF)
# ---- INTEGRATION.md §1: the two aliases, BEFORE the reference's "models" package is imported
sys.modules["models.networks.stylegan2_op"] = _op
sys.modules["models.networks.stylegan2_layers"] = _layers
import models                                                               # noqa: E402  (the reference's package)
import models.swapping_autoencoder_model as ref_model_mod                   # noqa: E402
import optimizers.swapping_autoencoder_optimizer as ref_opt_mod            # noqa: E402
import models.networks.encoder as ref_enc                                   # noqa: E402

assert ref_model_mod.__file__.startswith(REF) and ref_opt_mod.__file__.startswith(REF) and ref_enc.__file__.startswith(REF)
assert ref_enc.ConvLayer is _layers.ConvLayer            # the reference's network files build from THIS repo's classes

ref = surface_steps(models.create_model, lambda opt, w: ref_opt_mod.SwappingAutoencoderOptimizer(w))
ours = surface_steps(S.create_model, S.create_optimizer)
print(json.dumps({"reference_files": ref, "restated_callers": ours}))

"""ORACLE SUPPORT — test infrastructure only.  Import the *reference itself* (a read-only checkout, ``SAE_REFERENCE_ROOT``)
on CPU with its native-PyTorch op path, to pin the oracle and to generate golden fixtures.  Nothing the tests, ``smoke()``
or bench.py run may call this: the committed fixtures stand in for the reference there.

Recipe (SURVEY.md §8(c)): stub the optional dependencies that ``util/__init__.py`` imports eagerly (``install_stubs``), and
force ``util.is_custom_kernel_supported`` to False *before* ``models.networks.stylegan2_op`` is imported so the
reference neither JIT-compiles its CUDA extension nor tries to use a GPU.
"""
import importlib.util
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("SAE_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "models", "networks"))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def install_stubs():
    """Stand-ins for the optional modules the reference's ``util`` package imports eagerly; none of them is on the training
    path (sklearn's PCA only colours feature visualisations, so it is stubbed only where sklearn is not installed)."""
    if "func_timeout" not in sys.modules:
        _stub("func_timeout", func_timeout=lambda *a, **k: None, FunctionTimedOut=type("FunctionTimedOut", (Exception,), {}))
    if "dominate" not in sys.modules:
        tags = _stub("dominate.tags", **{t: (lambda *a, **k: None) for t in ("meta", "h3", "table", "tr", "td", "p", "a", "img", "br")})
        _stub("dominate", document=lambda *a, **k: None, tags=tags)
    if "visdom" not in sys.modules:
        _stub("visdom", Visdom=lambda *a, **k: None)
    if "sklearn" not in sys.modules and importlib.util.find_spec("sklearn") is None:
        decomposition = _stub("sklearn.decomposition", PCA=lambda *a, **k: None)
        _stub("sklearn", decomposition=decomposition)


def import_reference():
    """Returns the reference's top-level packages as a namespace: .models, .networks, .layers, .ops, .util, .optimizers"""
    if not available():
        raise RuntimeError("reference checkout not found at %s" % REFERENCE_ROOT)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    install_stubs()
    import util.util as uu                      # noqa: E402  (reference's util package)
    uu.is_custom_kernel_supported = lambda: False
    import util as u
    u.is_custom_kernel_supported = lambda: False
    import models                               # noqa: E402
    import models.networks as networks
    import models.networks.stylegan2_layers as layers
    import models.networks.stylegan2_op as ops
    ops_fir = sys.modules["models.networks.stylegan2_op.upfirdn2d"]   # the package re-exports a same-named function
    ops_act = sys.modules["models.networks.stylegan2_op.fused_act"]
    import models.swapping_autoencoder_model as sae_model
    import optimizers.swapping_autoencoder_optimizer as sae_opt
    assert not ops_fir.use_custom_kernel and not ops_act.use_custom_kernel
    return types.SimpleNamespace(models=models, networks=networks, layers=layers, ops=ops, util=u,
                                 sae_model=sae_model, sae_opt=sae_opt, ops_fir=ops_fir)

"""ctypes binding of libsae_b200.so (the C ABI declared in include/sae_b200.h).

The library is built in-tree by ``make -C csrc`` (see ``build_library``) and loaded lazily.  There is
no fallback: if the shared object is missing or a tensor is not on a CUDA device the call raises.
"""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsae_b200.so")
CSRC_DIR = os.path.join(_HERE, "csrc")

SAE_ABI_VERSION = 14

c_float_p = ctypes.c_void_p   # raw device pointers travel as integers
c_stream = ctypes.c_void_p


class ConvGeom(ctypes.Structure):
    """Mirror of ``sae_conv_geom`` (include/sae_b200.h)."""
    _fields_ = [(n, ctypes.c_int32) for n in
                ("N", "H", "W", "C", "K", "R", "S", "P", "Q", "stride", "pad_t", "pad_l")]

    def key(self):
        return tuple(getattr(self, n) for n, _ in self._fields_)


class ConvEpilogue(ctypes.Structure):
    """Mirror of ``sae_conv_epilogue``."""
    _fields_ = [("bias", ctypes.c_void_p), ("noise", ctypes.c_void_p), ("noise_weight", ctypes.c_void_p),
                ("residual", ctypes.c_void_p), ("alpha", ctypes.c_float), ("gain", ctypes.c_float),
                ("res_scale", ctypes.c_float), ("act", ctypes.c_int32), ("round_tf32", ctypes.c_int32),
                ("act_mask", ctypes.c_void_p)]


# name -> (restype, argtypes); the test-suite checks that every one of these is exported.
SIGNATURES = {
    "sae_abi_version": (ctypes.c_int, []),
    "sae_last_error": (ctypes.c_char_p, []),
    "sae_launch_count": (ctypes.c_int64, []),
    "sae_tcgen05_available": (ctypes.c_int, []),
    "sae_upfirdn2d": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, c_stream]),
    "sae_upfirdn2d_separable": (ctypes.c_int, [c_float_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, ctypes.c_int64,
                                               ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_int, ctypes.c_int, c_stream]),
    "sae_fused_bias_act": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, ctypes.c_int64, ctypes.c_int64,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                          c_float_p, c_float_p, ctypes.c_int64, ctypes.c_int, c_stream]),
    "sae_bias_act_backward": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, ctypes.c_int64, ctypes.c_int,
                                             ctypes.c_float, ctypes.c_float, c_float_p, ctypes.c_int64, c_float_p,
                                             ctypes.c_int, ctypes.c_void_p, c_stream]),
    "sae_fir_act_backward": (ctypes.c_int, [c_float_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, c_float_p, c_float_p,
                                            ctypes.c_int64] + [ctypes.c_int] * 9 + [ctypes.c_float, ctypes.c_float,
                                                                                    ctypes.c_int, ctypes.c_void_p, c_stream]),
    "sae_fir_bias_act": (ctypes.c_int, [c_float_p, ctypes.c_void_p, ctypes.c_void_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                        ctypes.c_int64] + [ctypes.c_int] * 9 + [ctypes.c_float, ctypes.c_float, ctypes.c_int,
                                                                                ctypes.c_void_p, c_stream]),
    "sae_modulate": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int,
                                    ctypes.c_int, c_stream]),
    "sae_modulate_backward": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, ctypes.c_int,
                                             ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_stream]),
    "sae_modulate_spatial": (ctypes.c_int, [c_float_p] * 3 + [ctypes.c_int] * 9 + [c_stream]),
    "sae_modulate_spatial_backward": (ctypes.c_int, [c_float_p] * 6 + [ctypes.c_int] * 9 + [c_stream]),
    "sae_add_scale": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.c_int64, ctypes.c_float, ctypes.c_int,
                                     c_stream]),
    "sae_round_tf32": (ctypes.c_int, [c_float_p, c_float_p, ctypes.c_int64, c_stream]),
    "sae_upsample2x_add_scale": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_float, ctypes.c_int, c_stream]),
    "sae_upsample2x_backward": (ctypes.c_int, [c_float_p, c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_float, ctypes.c_int, c_stream]),
    "sae_filter_prep": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_float, ctypes.c_int, c_stream]),
    "sae_filter_unprep": (ctypes.c_int, [c_float_p, c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_float, c_stream]),
    "sae_reflect_pad": (ctypes.c_int, [c_float_p, c_float_p] + [ctypes.c_int] * 8 + [c_stream]),
    "sae_reflect_pad_backward": (ctypes.c_int, [c_float_p, c_float_p] + [ctypes.c_int] * 8 + [c_stream]),
    "sae_pad_channels": (ctypes.c_int, [c_float_p, c_float_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, c_stream]),
    "sae_conv2d_fprop": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.POINTER(ConvGeom),
                                        ctypes.POINTER(ConvEpilogue), ctypes.c_int, c_stream]),
    "sae_conv2d_dgrad": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.POINTER(ConvGeom),
                                        ctypes.POINTER(ConvEpilogue), ctypes.c_int, c_stream]),
    "sae_conv2d_wgrad": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.POINTER(ConvGeom), ctypes.c_int,
                                        c_stream]),
    "sae_conv2d_query_impl": (ctypes.c_int, [ctypes.POINTER(ConvGeom), ctypes.c_int]),
    "sae_bucket_pack": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, c_float_p,
                                       ctypes.c_int64, c_stream]),
    "sae_bucket_unpack": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, c_float_p,
                                         ctypes.c_int64, ctypes.c_float, c_stream]),
    "sae_filter_modulate": (ctypes.c_int, [c_float_p] * 4 + [ctypes.c_int] * 6 + [c_stream]),
    "sae_conv2d_query_modulated": (ctypes.c_int, [ctypes.POINTER(ConvGeom)]),
    "sae_conv2d_fprop_per_sample": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.POINTER(ConvGeom),
                                                   ctypes.POINTER(ConvEpilogue), c_stream]),
    "sae_conv2d_dgrad_per_sample": (ctypes.c_int, [c_float_p, c_float_p, c_float_p, ctypes.POINTER(ConvGeom),
                                                   ctypes.POINTER(ConvEpilogue), c_stream]),
    "sae_conv2d_wgrad_modulated": (ctypes.c_int, [c_float_p] * 6 + [ctypes.POINTER(ConvGeom), c_stream]),
    "sae_adam_step": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                     c_float_p, c_float_p, c_float_p] + [ctypes.c_float] * 5 + [c_stream]),
    "sae_crop_gather": (ctypes.c_int, [c_float_p] * 5 + [ctypes.c_int] * 7 + [ctypes.c_int64] * 4 + [ctypes.c_int, c_stream]),
    "sae_crop_gather_backward": (ctypes.c_int, [c_float_p] * 5 + [ctypes.c_int] * 6 + [ctypes.c_int64] * 4 + [c_stream]),
    "sae_torgb_forward": (ctypes.c_int, [c_float_p] * 5 + [ctypes.c_int] * 4 + [ctypes.c_float, ctypes.c_int, c_stream]),
    "sae_torgb_backward": (ctypes.c_int, [c_float_p] * 6 + [ctypes.c_int] * 4 + [ctypes.c_float] + [ctypes.c_int64] * 4
                           + [ctypes.c_int, c_stream]),
}

_lib = None
_lock = threading.Lock()


class SaeError(RuntimeError):
    """Raised when a C-ABI entry point returns a negative code (the reference raises RuntimeError from
    TORCH_CHECK in the same situations, upfirdn2d.cpp:15-16)."""


def build_library(verbose=False):
    """Compile csrc/*.cu for sm_100a into libsae_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j", str(os.cpu_count() or 4)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise RuntimeError("building libsae_b200.so failed")
    return LIB_PATH


def load():
    """Return the ctypes handle, loading (never building) the shared object on first use."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SaeError(
                "libsae_b200.so not found at %s — build it with __graft_entry__.build() or "
                "`make -C swapping_autoencoder_pytorch_b200/csrc`; there is no CPU / PyTorch fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError here means header and library diverged
            fn.restype = res
            fn.argtypes = args
        if lib.sae_abi_version() != SAE_ABI_VERSION:
            raise SaeError("libsae_b200.so ABI %d != expected %d — rebuild" % (lib.sae_abi_version(), SAE_ABI_VERSION))
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().sae_last_error()
        raise SaeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def launch_count():
    return int(load().sae_launch_count())

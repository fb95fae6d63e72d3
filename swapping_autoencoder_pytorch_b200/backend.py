"""Tensor-level entry points of the hot path: thin wrappers that allocate outputs with torch and pass raw
device pointers + the current CUDA stream to the C ABI (include/sae_b200.h).

All activations here are *physical* NHWC: contiguous ``[N, H, W, C]`` (or ``[B, C]``) fp32 CUDA tensors.
The autograd layer in ``stylegan2_op`` converts from / to the logical NCHW shapes the reference's modules
expose.  ``set_kernels`` lets the CPU test-suite swap in an emulation built on the oracle so the host-side
autograd logic can be grad-checked without a GPU; the product never does that — ``CudaKernels`` raises if
the shared library is missing or a tensor lives on the CPU.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import ConvEpilogue, ConvGeom, check


def make_geom(N, H, W, C, K, R, S, stride, pad_t, pad_l, P=None, Q=None):
    """Geometry of y[n,p,q,k] = sum x[n, p*stride - pad_t + r, q*stride - pad_l + s, c] w[k,r,s,c].
    P/Q default to the F.conv2d rule with symmetric padding (pad_t on both sides)."""
    if P is None:
        P = (H + 2 * pad_t - R) // stride + 1
    if Q is None:
        Q = (W + 2 * pad_l - S) // stride + 1
    return ConvGeom(N, H, W, C, K, R, S, P, Q, stride, pad_t, pad_l)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts, strided=False):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.SaeError("sae_b200 kernels need CUDA tensors (got a %s tensor); there is no CPU fallback"
                                % t.device.type)
        if t.dtype != torch.float32:
            raise _lib.SaeError("sae_b200 kernels are fp32-only (got %s)" % t.dtype)
        if not strided and not t.is_contiguous():
            raise _lib.SaeError("sae_b200 kernels need contiguous NHWC storage")


class PointerTables:
    """Device copies of host address lists (tuples of ``data_ptr()``), cached by content.  The pinned staging rows are
    allocated up front — a miss costs a device allocation and an async copy, so a miss inside a CUDA-graph capture is legal:
    the copy becomes a memcpy node that re-reads its pinned row on every replay.  Rows filled during a capture are therefore
    permanent; rows filled in eager execution (where the caching allocator may hand the gradients new addresses now and
    then) are recycled round-robin, each guarded by an event so a row is never rewritten before its copy has run."""

    def __init__(self, n, device, eager_rows=24, capture_rows=24):
        self.n, self.device = n, device
        self.eager_rows, self.capture_rows = eager_rows, capture_rows
        cuda = device.type == "cuda"
        self.pinned = torch.zeros(eager_rows + capture_rows, max(n, 1), dtype=torch.int64).pin_memory() if cuda else None
        self.eager, self.captured = {}, {}
        self.row_key, self.row_event = [None] * eager_rows, [None] * eager_rows
        self.next_row, self.next_capture = 0, 0

    def _upload(self, row, key):
        row[:len(key)].copy_(torch.tensor(key, dtype=torch.int64))
        dev = torch.empty(len(key), dtype=torch.int64, device=self.device)
        dev.copy_(row[:len(key)], non_blocking=True)
        return dev

    def get(self, key):
        hit = self.captured.get(key)
        if hit is None:
            hit = self.eager.get(key)
        if hit is not None:
            return hit
        if self.pinned is None:
            hit = torch.tensor(key, dtype=torch.int64)
            self.eager[key] = hit
            return hit
        if torch.cuda.is_current_stream_capturing():
            if self.next_capture >= self.capture_rows:
                raise _lib.SaeError("PointerTables: more than %d address lists captured into CUDA graphs" % self.capture_rows)
            hit = self._upload(self.pinned[self.eager_rows + self.next_capture], key)
            self.next_capture += 1
            self.captured[key] = hit
            return hit
        r = self.next_row
        self.next_row = (r + 1) % self.eager_rows
        if self.row_key[r] is not None:
            self.eager.pop(self.row_key[r], None)
            self.row_event[r].synchronize()
        hit = self._upload(self.pinned[r], key)
        ev = torch.cuda.Event()
        ev.record()
        self.row_key[r], self.row_event[r] = key, ev
        self.eager[key] = hit
        return hit


class CudaKernels:
    """The product path: every method is one (or two) launches of hand-written sm_100a kernels."""
    name = "cuda"

    def __init__(self):
        self.lib = _lib.load()
        self.conv_impl = 0       # 0 auto, 1 force generic (mma.sync), 2 force tcgen05
        # Every activation / gradient / filter this library writes is rounded to the nearest TF32 value (still stored
        # as fp32): the tensor cores ignore the low 13 mantissa bits of their operands, so rounding in the producer
        # makes that truncation exact and unbiased.  Set False for bit-exact fp32 results from the pointwise kernels.
        self.round_tf32 = True
        self.fused_fir_act = os.environ.get("SAE_FUSED_FIR_ACT", "1") != "0"
        # activation bit masks next to the tensor-core convs' / the FIR + activation kernel's outputs (A/B: SAE_ACT_MASK=0)
        self.act_masks = os.environ.get("SAE_ACT_MASK", "1") != "0"
        # texture code maps [N, C, h, w]: "native" modulates with the affine evaluated at the map's resolution
        # (sae_modulate_spatial); "glue" interpolates the map to every layer's resolution first (A/B: SAE_SPATIAL_STYLE=glue)
        self.spatial_style = os.environ.get("SAE_SPATIAL_STYLE", "native")
        if self.spatial_style not in ("native", "glue"):
            raise ValueError("SAE_SPATIAL_STYLE must be 'native' or 'glue', not %r" % self.spatial_style)

    # ------------------------------------------------------------------ FIR
    def upfirdn2d(self, x, kernel, up_x, up_y, down_x, down_y, pad_x0, pad_x1, pad_y0, pad_y1, taps=None):
        """taps: optional host-side 1-D factors (taps_y, taps_x) with kernel == outer(taps_y, taps_x); supplied by
        the Blur modules, which build their kernels from 1-D tap lists — selects the separable fast path."""
        _need_cuda(x, kernel)
        n, h, w, c = x.shape
        kh, kw = kernel.shape
        oh = (h * up_y + pad_y0 + pad_y1 - kh) // down_y + 1
        ow = (w * up_x + pad_x0 + pad_x1 - kw) // down_x + 1
        out = torch.empty((n, oh, ow, c), device=x.device, dtype=x.dtype)
        ud = (up_x, down_x)
        if up_x == up_y and down_x == down_y and ud in ((1, 1), (1, 2), (2, 1)) and c % 4 == 0 \
                and n * oh * ow * (c // 4) < 2 ** 32 and x.data_ptr() % 16 == 0 and n > 0:
            if taps is not None and len(taps[0]) == kh and len(taps[1]) == kw and kh == kw and kh <= 4:
                ty = (ctypes.c_float * kh)(*taps[0])
                tx = (ctypes.c_float * kw)(*taps[1])
                with torch.cuda.device(x.device):
                    check(self.lib.sae_upfirdn2d_separable(_ptr(x), ty, tx, _ptr(out), n, h, w, c, kh, kw, up_x, down_x, pad_x0,
                                                           pad_x1, pad_y0, pad_y1, int(self.round_tf32), _stream()),
                          "sae_upfirdn2d_separable")
                return out
        with torch.cuda.device(x.device):
            check(self.lib.sae_upfirdn2d(_ptr(x), _ptr(kernel), _ptr(out), n, h, w, c, kh, kw, up_x, up_y,
                                         down_x, down_y, pad_x0, pad_x1, pad_y0, pad_y1, int(self.round_tf32), _stream()),
                  "sae_upfirdn2d")
        return out

    # ------------------------------------------------------------- bias/act
    def bias_act(self, x, bias, ref, act, grad, alpha, scale, noise=None, noise_weight=None):
        """x: [..., C] channels innermost.  noise: one value per pixel (numel = x.numel() / C)."""
        _need_cuda(x, bias, ref, noise, noise_weight)
        out = torch.empty_like(x)
        c = x.shape[-1]
        with torch.cuda.device(x.device):
            check(self.lib.sae_fused_bias_act(_ptr(x), _ptr(bias), _ptr(ref), _ptr(out), x.numel(), 1,
                                              bias.numel() if bias is not None else 1, act, grad, alpha, scale,
                                              _ptr(noise), _ptr(noise_weight), c, int(self.round_tf32), _stream()),
                  "sae_fused_bias_act")
        return out

    def bias_act_backward(self, grad_out, out, alpha, scale, want_bias=True, noise=None, mask=None):
        """mask: the activation bit mask a forward kernel wrote for ``out`` (``act_mask_of(out)``) — read instead of ``out``"""
        _need_cuda(grad_out, out, noise)
        c = out.shape[-1]
        gi = torch.empty_like(out)
        gb = torch.zeros(c, device=out.device, dtype=out.dtype) if want_bias else None
        gnw = torch.zeros(1, device=out.device, dtype=out.dtype) if noise is not None else None
        with torch.cuda.device(out.device):
            check(self.lib.sae_bias_act_backward(_ptr(grad_out), _ptr(out), _ptr(gi), _ptr(gb), out.numel(), c,
                                                 alpha, scale, _ptr(noise), c, _ptr(gnw), int(self.round_tf32), _ptr(mask), _stream()),
                  "sae_bias_act_backward")
        return gi, gb, gnw

    def fir_act_backward(self, grad, taps, act_out, pad, alpha, scale, want_bias=True, mask=None):
        """(FIR(grad) masked by the activation saved in ``act_out``, bias gradient) in one pass, or None when the shape is
        outside the fused kernel's configuration (the caller then runs upfirdn2d + bias_act_backward).
        grad [N,h,w,C]; act_out [N,oh,ow,C]; taps = (taps_y, taps_x) host factors; pad = (x0, x1, y0, y1)."""
        _need_cuda(grad, act_out)
        n, h, w, c = grad.shape
        kh, kw = len(taps[0]), len(taps[1])
        px0, px1, py0, py1 = pad
        oh, ow = h + py0 + py1 - kh + 1, w + px0 + px1 - kw + 1
        if (c % 32 != 0 or kh != kw or kh not in (3, 4) or oh < 8 or ow < 8 or n == 0 or grad.data_ptr() % 16 != 0
                or tuple(act_out.shape) != (n, oh, ow, c) or not self.fused_fir_act):
            return None
        gi = torch.empty_like(act_out)
        gb = torch.zeros(c, device=grad.device, dtype=grad.dtype) if want_bias else None
        ty = (ctypes.c_float * kh)(*taps[0])
        tx = (ctypes.c_float * kw)(*taps[1])
        with torch.cuda.device(grad.device):
            rc = self.lib.sae_fir_act_backward(_ptr(grad), ty, tx, _ptr(act_out), _ptr(gi), _ptr(gb), n, h, w, c, kh, kw,
                                               px0, px1, py0, py1, alpha, scale, int(self.round_tf32), _ptr(mask), _stream())
        if rc == -3:            # SAE_E_UNSUPPORTED: e.g. no TMA on this device
            return None
        check(rc, "sae_fir_act_backward")
        return gi, gb

    def fir_bias_act(self, x, taps, pad, bias, noise, noise_weight, alpha, scale):
        """lrelu(FIR(x) + noise_weight * noise + bias) * scale in one pass, or None when the shape is outside the fused kernel's
        configuration (the caller then runs upfirdn2d + bias_act).  x [N,h,w,C]; taps = (taps_y, taps_x) host factors;
        pad = (x0, x1, y0, y1); noise: one value per output pixel or None."""
        _need_cuda(x, bias, noise, noise_weight)
        n, h, w, c = x.shape
        kh, kw = len(taps[0]), len(taps[1])
        px0, px1, py0, py1 = pad
        oh, ow = h + py0 + py1 - kh + 1, w + px0 + px1 - kw + 1
        if c % 32 != 0 or kh != kw or kh not in (3, 4) or oh < 8 or ow < 8 or n == 0 or x.data_ptr() % 16 != 0:
            return None
        out = torch.empty((n, oh, ow, c), device=x.device, dtype=x.dtype)
        mask = self._new_act_mask(out, 3, True)
        ty = (ctypes.c_float * kh)(*taps[0])
        tx = (ctypes.c_float * kw)(*taps[1])
        with torch.cuda.device(x.device):
            rc = self.lib.sae_fir_bias_act(_ptr(x), ty, tx, _ptr(bias), _ptr(noise), _ptr(noise_weight), _ptr(out), n, h, w, c,
                                           kh, kw, px0, px1, py0, py1, alpha, scale, int(self.round_tf32), _ptr(mask), _stream())
        if rc == -3:
            return None
        check(rc, "sae_fir_bias_act")
        if mask is not None:
            out._sae_act_mask = mask
        return out

    # ------------------------------------------------------------- modulate
    def modulate(self, x, s):
        _need_cuda(x, s)
        n, h, w, c = x.shape
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            check(self.lib.sae_modulate(_ptr(x), _ptr(s), _ptr(out), n, h * w, c, int(self.round_tf32), _stream()),
                  "sae_modulate")
        return out

    def modulate_backward(self, dy, x, s):
        _need_cuda(dy, x, s)
        n, h, w, c = x.shape
        dx = torch.empty_like(x)
        ds = torch.zeros_like(s)
        with torch.cuda.device(x.device):
            check(self.lib.sae_modulate_backward(_ptr(dy), _ptr(x), _ptr(s), _ptr(dx), _ptr(ds), n, h * w, c,
                                                 int(self.round_tf32), _stream()), "sae_modulate_backward")
        return dx, ds

    def modulate_spatial(self, x, s_lo, demodulate):
        """x [N,H,W,C] * demod(bilinear(s_lo)) with s_lo [Ns,hs,ws,C], Ns in {1, N} (include/sae_b200.h sae_modulate_spatial)"""
        _need_cuda(x, s_lo)
        n, h, w, c = x.shape
        ns, hs, ws, _ = s_lo.shape
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            check(self.lib.sae_modulate_spatial(_ptr(x), _ptr(s_lo), _ptr(out), n, h, w, c, ns, hs, ws, int(demodulate),
                                                int(self.round_tf32), _stream()), "sae_modulate_spatial")
        return out

    def modulate_spatial_backward(self, dy, x, s_lo, demodulate):
        """-> (dx [N,H,W,C], ds_lo [Ns,hs,ws,C])"""
        _need_cuda(dy, x, s_lo)
        n, h, w, c = x.shape
        ns, hs, ws, _ = s_lo.shape
        dx = torch.empty_like(x)
        ds = torch.empty_like(s_lo)
        work = torch.empty((n * h * ws * c + 3) // 4 * 4 + 2 * n * h * w, device=x.device, dtype=x.dtype)
        with torch.cuda.device(x.device):
            check(self.lib.sae_modulate_spatial_backward(_ptr(dy), _ptr(x), _ptr(s_lo), _ptr(dx), _ptr(ds), _ptr(work), n, h, w, c, ns,
                                                         hs, ws, int(demodulate), int(self.round_tf32), _stream()),
                  "sae_modulate_spatial_backward")
        return dx, ds

    # ------------------------------------------------------- residual merge
    def add_scale(self, a, b, scale):
        """(a + b) * scale, or a * scale when b is None; any shape, a and b contiguous with identical layout"""
        _need_cuda(a, b)
        out = torch.empty_like(a)
        with torch.cuda.device(a.device):
            check(self.lib.sae_add_scale(_ptr(a), _ptr(b), _ptr(out), a.numel(), scale, int(self.round_tf32), _stream()),
                  "sae_add_scale")
        return out

    def upsample2x_add_scale(self, skip, res, scale):
        """(bilinear_x2(skip) + res) * scale;  skip [N,h,w,C], res [N,2h,2w,C]"""
        _need_cuda(skip, res)
        n, h, w, c = skip.shape
        assert tuple(res.shape) == (n, 2 * h, 2 * w, c)
        out = torch.empty_like(res)
        with torch.cuda.device(res.device):
            check(self.lib.sae_upsample2x_add_scale(_ptr(skip), _ptr(res), _ptr(out), n, h, w, c, scale,
                                                    int(self.round_tf32), _stream()), "sae_upsample2x_add_scale")
        return out

    def upsample2x_backward(self, dy, scale):
        """adjoint of the x2 bilinear interpolation times scale: dy [N,2h,2w,C] -> [N,h,w,C]"""
        _need_cuda(dy)
        n, oh, ow, c = dy.shape
        out = torch.empty((n, oh // 2, ow // 2, c), device=dy.device, dtype=dy.dtype)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_upsample2x_backward(_ptr(dy), _ptr(out), n, oh // 2, ow // 2, c, scale,
                                                   int(self.round_tf32), _stream()), "sae_upsample2x_backward")
        return out

    def pad_channels(self, x, c_out):
        """x: logical [N, c_in, H, W] with any (n, c) strides and a flattenable pixel plane -> NHWC [N, H, W, c_out],
        channels c_in.. zero (one kernel instead of F.pad + a layout copy)"""
        _need_cuda(x, strided=True)          # the kernel addresses x through (n, c, pixel) element strides
        n, c, h, w = x.shape
        if h > 1 and x.stride(2) != w * x.stride(3):
            x = x.contiguous()
        out = torch.empty((n, h, w, c_out), device=x.device, dtype=x.dtype)
        with torch.cuda.device(x.device):
            check(self.lib.sae_pad_channels(_ptr(x), _ptr(out), n, h * w, c, c_out, x.stride(0), x.stride(1), x.stride(3),
                                            int(self.round_tf32), _stream()), "sae_pad_channels")
        return out

    def reflect_pad(self, x, pads):
        """x [N,H,W,C] -> [N, H+pt+pb, W+pl+pr, C]; pads = (left, right, top, bottom)"""
        _need_cuda(x)
        n, h, w, c = x.shape
        pl, pr, pt, pb = pads
        out = torch.empty((n, h + pt + pb, w + pl + pr, c), device=x.device, dtype=x.dtype)
        with torch.cuda.device(x.device):
            check(self.lib.sae_reflect_pad(_ptr(x), _ptr(out), n, h, w, c, pl, pr, pt, pb, _stream()), "sae_reflect_pad")
        return out

    def reflect_pad_backward(self, dy, pads):
        _need_cuda(dy)
        n, oh, ow, c = dy.shape
        pl, pr, pt, pb = pads
        dx = torch.empty((n, oh - pt - pb, ow - pl - pr, c), device=dy.device, dtype=dy.dtype)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_reflect_pad_backward(_ptr(dy), _ptr(dx), n, oh - pt - pb, ow - pl - pr, c, pl, pr, pt, pb,
                                                    _stream()), "sae_reflect_pad_backward")
        return dx

    def filter_prep(self, w_oihw, scale, want_crsk=True):
        """[K,C,R,S] parameter -> ([K,R,S,C], [C,R,S,K] or None), scaled and TF32-rounded, in one kernel"""
        _need_cuda(w_oihw)
        k, c, r, s = w_oihw.shape
        krsc = torch.empty((k, r, s, c), device=w_oihw.device, dtype=w_oihw.dtype)
        crsk = torch.empty((c, r, s, k), device=w_oihw.device, dtype=w_oihw.dtype) if want_crsk else None
        with torch.cuda.device(w_oihw.device):
            check(self.lib.sae_filter_prep(_ptr(w_oihw), _ptr(krsc), _ptr(crsk), k, c, r, s, scale, int(self.round_tf32),
                                           _stream()), "sae_filter_prep")
        return krsc, crsk

    def filter_unprep(self, d_krsc, scale):
        """adjoint of filter_prep: [K,R,S,C] gradient -> [K,C,R,S] * scale"""
        _need_cuda(d_krsc)
        k, r, s, c = d_krsc.shape
        out = torch.empty((k, c, r, s), device=d_krsc.device, dtype=d_krsc.dtype)
        with torch.cuda.device(d_krsc.device):
            check(self.lib.sae_filter_unprep(_ptr(d_krsc), _ptr(out), k, c, r, s, scale, _stream()), "sae_filter_unprep")
        return out

    def _filter(self, w):
        """contiguous copy of a (small) filter tensor, rounded to TF32 when the policy says so"""
        w = w.contiguous()
        if not self.round_tf32:
            return w
        out = torch.empty_like(w)
        with torch.cuda.device(w.device):
            check(self.lib.sae_round_tf32(_ptr(w), _ptr(out), w.numel(), _stream()), "sae_round_tf32")
        return out

    # ----------------------------------------------------------------- conv
    def _new_act_mask(self, y, act, tensor_core_kernel):
        """1 bit per element of an activation output ``y`` [..., C] (C % 32 == 0), written by the kernel that produces y and read
        by the activation's backward instead of y itself (sae_conv_epilogue.act_mask); None where no kernel would write it"""
        if act != 3 or not tensor_core_kernel or not self.act_masks or y.shape[-1] % 32 != 0 or y.numel() == 0:
            return None
        return torch.empty(y.numel() // 32, device=y.device, dtype=torch.int32)

    def _epi(self, bias=None, act=1, alpha=0.2, gain=1.0, noise=None, noise_weight=None, residual=None,
             res_scale=1.0, round_tf32=None, act_mask=None):
        _need_cuda(bias, noise, noise_weight, residual)
        e = ConvEpilogue()
        e.bias = bias.data_ptr() if bias is not None else None
        e.noise = noise.data_ptr() if noise is not None else None
        e.noise_weight = noise_weight.data_ptr() if noise_weight is not None else None
        e.residual = residual.data_ptr() if residual is not None else None
        e.alpha, e.gain, e.res_scale, e.act = alpha, gain, res_scale, act
        e.round_tf32 = int(self.round_tf32 if round_tf32 is None else round_tf32)
        e.act_mask = act_mask.data_ptr() if act_mask is not None else None
        return e

    def conv_fprop(self, x, w_krsc, g, impl=None, prepared=False, **epi):
        """x [N,H,W,C], w [K,R,S,C] -> y [N,P,Q,K].  prepared: w is already contiguous and TF32-rounded (filter_prep)"""
        _need_cuda(x, w_krsc if prepared else None)
        if not prepared:
            w_krsc = self._filter(w_krsc)
        assert tuple(x.shape) == (g.N, g.H, g.W, g.C) and tuple(w_krsc.shape) == (g.K, g.R, g.S, g.C), \
            (tuple(x.shape), tuple(w_krsc.shape), g.key())
        y = torch.empty((g.N, g.P, g.Q, g.K), device=x.device, dtype=x.dtype)
        impl = self.conv_impl if impl is None else impl
        mask = None
        if epi.get("act", 1) == 3 and self.act_masks:
            mask = self._new_act_mask(y, 3, impl == 2 or (impl == 0 and self.conv_impl_for(g, 0) == 2))
        e = self._epi(act_mask=mask, **epi)
        with torch.cuda.device(x.device):
            check(self.lib.sae_conv2d_fprop(_ptr(x), _ptr(w_krsc), _ptr(y), ctypes.byref(g), ctypes.byref(e), impl, _stream()),
                  "sae_conv2d_fprop")
        if mask is not None:
            y._sae_act_mask = mask
        return y

    def conv_dgrad(self, dy, w_krsc, g, impl=None, w_crsk=None, **epi):
        """dy [N,P,Q,K], w [K,R,S,C] -> dx [N,H,W,C] (also the forward of the transposed convolution).
        w_crsk: the same filter already transposed to [C,R,S,K] and rounded (filter_prep), if the caller has it."""
        _need_cuda(dy)
        assert tuple(dy.shape) == (g.N, g.P, g.Q, g.K) and tuple(w_krsc.shape) == (g.K, g.R, g.S, g.C), \
            (tuple(dy.shape), tuple(w_krsc.shape), g.key())
        wt = w_crsk if w_crsk is not None else self._filter(w_krsc.permute(3, 1, 2, 0))     # [C,R,S,K]
        dx = torch.empty((g.N, g.H, g.W, g.C), device=dy.device, dtype=dy.dtype)
        e = self._epi(**epi)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_conv2d_dgrad(_ptr(dy), _ptr(wt), _ptr(dx), ctypes.byref(g), ctypes.byref(e),
                                            self.conv_impl if impl is None else impl, _stream()), "sae_conv2d_dgrad")
        return dx

    def conv_wgrad(self, dy, x, g, impl=None):
        """dy [N,P,Q,K], x [N,H,W,C] -> dw [K,R,S,C]"""
        _need_cuda(dy, x)
        assert tuple(dy.shape) == (g.N, g.P, g.Q, g.K) and tuple(x.shape) == (g.N, g.H, g.W, g.C), \
            (tuple(dy.shape), tuple(x.shape), g.key())
        dw = torch.zeros((g.K, g.R, g.S, g.C), device=dy.device, dtype=dy.dtype)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_conv2d_wgrad(_ptr(dy), _ptr(x), _ptr(dw), ctypes.byref(g),
                                            self.conv_impl if impl is None else impl, _stream()), "sae_conv2d_wgrad")
        return dw

    # ------------------------------------------------ style-modulated conv, per-sample filters
    def conv_modulated_ok(self, g):
        """True when the per-sample-filter kernels (fprop, dgrad, modulated wgrad) all take this geometry"""
        return bool(self.lib.sae_conv2d_query_modulated(ctypes.byref(g)))

    def filter_modulate(self, w_krsc, s, want_krsc=True, want_crsk=False):
        """prepared filter [K,R,S,C] x per-sample scale [N,C] -> ([N,K,R,S,C] or None, [N,C,R,S,K] or None)"""
        _need_cuda(w_krsc, s)
        k, r, s_, c = w_krsc.shape
        n = s.shape[0]
        a = torch.empty((n, k, r, s_, c), device=s.device, dtype=s.dtype) if want_krsc else None
        b = torch.empty((n, c, r, s_, k), device=s.device, dtype=s.dtype) if want_crsk else None
        with torch.cuda.device(s.device):
            check(self.lib.sae_filter_modulate(_ptr(w_krsc), _ptr(s), _ptr(a), _ptr(b), n, k, c, r, s_, int(self.round_tf32),
                                               _stream()), "sae_filter_modulate")
        return a, b

    def conv_fprop_per_sample(self, x, w_nkrsc, g, **epi):
        """x [N,H,W,C], per-sample filters [N,K,R,S,C] -> y [N,P,Q,K]"""
        _need_cuda(x, w_nkrsc)
        y = torch.empty((g.N, g.P, g.Q, g.K), device=x.device, dtype=x.dtype)
        mask = self._new_act_mask(y, epi.get("act", 1), True)          # only the tcgen05 kernel implements per-sample filters
        e = self._epi(act_mask=mask, **epi)
        with torch.cuda.device(x.device):
            check(self.lib.sae_conv2d_fprop_per_sample(_ptr(x), _ptr(w_nkrsc), _ptr(y), ctypes.byref(g), ctypes.byref(e), _stream()),
                  "sae_conv2d_fprop_per_sample")
        if mask is not None:
            y._sae_act_mask = mask
        return y

    def conv_dgrad_per_sample(self, dy, w_ncrsk, g, **epi):
        """dy [N,P,Q,K], per-sample transposed filters [N,C,R,S,K] -> dx [N,H,W,C]"""
        _need_cuda(dy, w_ncrsk)
        dx = torch.empty((g.N, g.H, g.W, g.C), device=dy.device, dtype=dy.dtype)
        e = self._epi(**epi)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_conv2d_dgrad_per_sample(_ptr(dy), _ptr(w_ncrsk), _ptr(dx), ctypes.byref(g), ctypes.byref(e), _stream()),
                  "sae_conv2d_dgrad_per_sample")
        return dx

    def conv_wgrad_modulated(self, dy, x, s, w_krsc, g):
        """dy [N,P,Q,K], UNSCALED x [N,H,W,C], s [N,C], forward filter [K,R,S,C] -> (dw [K,R,S,C], ds [N,C])"""
        _need_cuda(dy, x, s, w_krsc)
        dw = torch.zeros((g.K, g.R, g.S, g.C), device=dy.device, dtype=dy.dtype)
        ds = torch.zeros((g.N, g.C), device=dy.device, dtype=dy.dtype)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_conv2d_wgrad_modulated(_ptr(dy), _ptr(x), _ptr(s), _ptr(w_krsc), _ptr(dw), _ptr(ds), ctypes.byref(g),
                                                      _stream()), "sae_conv2d_wgrad_modulated")
        return dw, ds

    def conv_impl_for(self, g, direction):
        return int(self.lib.sae_conv2d_query_impl(ctypes.byref(g), direction))

    # --------------------------------------------------------------- bucket
    def bucket_pack(self, ptrs, offsets, sizes, n, bucket):
        with torch.cuda.device(bucket.device):
            check(self.lib.sae_bucket_pack(_ptr(ptrs), _ptr(offsets), _ptr(sizes), n, _ptr(bucket), bucket.numel(),
                                           _stream()), "sae_bucket_pack")

    def bucket_unpack(self, ptrs, offsets, sizes, n, bucket, scale):
        with torch.cuda.device(bucket.device):
            check(self.lib.sae_bucket_unpack(_ptr(ptrs), _ptr(offsets), _ptr(sizes), n, _ptr(bucket), bucket.numel(),
                                             scale, _stream()), "sae_bucket_unpack")


    # ----------------------------------------------------------------- Adam
    def adam_step(self, params, grads, offsets, sizes, exp_avg, exp_avg_sq, steps, lr, beta1, beta2, eps, grad_scale, cache):
        """One multi-tensor Adam update (torch.optim.Adam semantics) of ``params`` (list of tensors).  grads: list aligned with
        params — a tensor (the parameter's own gradient, or a view into the flat all-reduce bucket) or None (parameter
        skipped, its step count untouched).  offsets / sizes: device int64 tensors locating each parameter's moments in
        the flat ``exp_avg`` / ``exp_avg_sq``; steps: device float tensor, one count per parameter.  cache: the caller's
        ``PointerTables`` (device copies of the address lists)."""
        dev = exp_avg.device
        p_tab = cache.get(tuple(p.data_ptr() for p in params))
        g_tab = cache.get(tuple(0 if g is None else g.data_ptr() for g in grads))
        for g in grads:
            if g is not None and (not g.is_cuda or g.dtype != torch.float32 or not g.is_contiguous()):
                raise _lib.SaeError("adam_step: gradients must be contiguous fp32 CUDA tensors")
        with torch.cuda.device(dev):
            check(self.lib.sae_adam_step(_ptr(p_tab), _ptr(g_tab), _ptr(offsets), _ptr(sizes), len(params), _ptr(exp_avg),
                                         _ptr(exp_avg_sq), _ptr(steps), lr, beta1, beta2, eps, grad_scale, _stream()),
                  "sae_adam_step")

    # ----------------------------------------------------------------- ToRGB
    def torgb_forward(self, x, s, w, bias, wscale):
        """x [N,H,W,C], s [N,C], w [3,C], bias [3] or None -> y [N,H,W,4] (channel 3 zero)"""
        _need_cuda(x, s, w, bias)
        n, h, wd, c = x.shape
        y = torch.empty((n, h, wd, 4), device=x.device, dtype=x.dtype)
        with torch.cuda.device(x.device):
            check(self.lib.sae_torgb_forward(_ptr(x), _ptr(s), _ptr(w), _ptr(bias), _ptr(y), n, h, wd, c, wscale,
                                             int(self.round_tf32), _stream()), "sae_torgb_forward")
        return y

    def torgb_backward(self, dy, x, s, w, wscale, want_dx=True, want_gw=True):
        """dy: logical [N,3,H,W] (any strides) -> (dx [N,H,W,C] or None, gw [N,3,C] = sum_p dy (x) x or None)"""
        _need_cuda(x, s, w)
        _need_cuda(dy, strided=True)
        n, h, wd, c = x.shape
        dx = torch.empty_like(x) if want_dx else None
        gw = torch.zeros((n, 3, c), device=x.device, dtype=x.dtype) if want_gw else None
        with torch.cuda.device(x.device):
            check(self.lib.sae_torgb_backward(_ptr(dy), _ptr(x), _ptr(s), _ptr(w), _ptr(dx), _ptr(gw), n, h, wd, c, wscale,
                                              dy.stride(0), dy.stride(1), dy.stride(2), dy.stride(3), int(self.round_tf32),
                                              _stream()), "sae_torgb_backward")
        return dx, gw

    # ----------------------------------------------------------------- crops
    def crop_gather(self, x, flip, scale, offset, num_crops, size, c_pad, out=None):
        """x: logical [B, C, H, W] (any strides); flip [Q], scale / offset [Q, 2] -> NHWC [Q, size, size, c_pad], channels
        C.. zero.  out: optional destination (a [Q, size, size, c_pad] slice of a larger batch buffer)"""
        _need_cuda(x, flip, scale, offset, strided=True)
        b, c, h, w = x.shape
        q = flip.numel()
        if out is None:
            out = torch.empty((q, size, size, c_pad), device=x.device, dtype=x.dtype)
        assert tuple(out.shape) == (q, size, size, c_pad) and out.is_contiguous()
        with torch.cuda.device(x.device):
            check(self.lib.sae_crop_gather(_ptr(x), _ptr(flip), _ptr(scale), _ptr(offset), _ptr(out), q, num_crops, c, h, w, size,
                                           c_pad, x.stride(0), x.stride(1), x.stride(2), x.stride(3), int(self.round_tf32),
                                           _stream()), "sae_crop_gather")
        return out

    def crop_gather_backward(self, dy, flip, scale, offset, num_crops, c, h, w):
        """dy: logical [Q, C', S, S] (any strides, C' >= c) -> dx [Q / num_crops, c, h, w] contiguous"""
        _need_cuda(dy, flip, scale, offset, strided=True)
        q, s = dy.shape[0], dy.shape[2]
        dx = torch.empty((q // num_crops, c, h, w), device=dy.device, dtype=dy.dtype)
        with torch.cuda.device(dy.device):
            check(self.lib.sae_crop_gather_backward(_ptr(dy), _ptr(flip), _ptr(scale), _ptr(offset), _ptr(dx), q, num_crops, c, h, w,
                                                    s, dy.stride(0), dy.stride(1), dy.stride(2), dy.stride(3), _stream()),
                  "sae_crop_gather_backward")
        return dx


_kernels = None


def act_mask_of(t):
    """the activation bit mask the producing kernel left next to ``t`` (None: the backward reads ``t`` itself).  The mask is a
    Python attribute of the tensor object the kernel wrapper returned: callers that hand ``t`` to autograd (outputs of a
    Function come back as new objects) read it right after the forward call and keep it in their ctx."""
    return getattr(t, "_sae_act_mask", None) if t is not None else None


def kernels():
    """The active kernel set; instantiates ``CudaKernels`` (loading the .so) on first use."""
    global _kernels
    if _kernels is None:
        _kernels = CudaKernels()
    return _kernels


def set_kernels(k):
    """Test hook (tests/ only): install an object with the ``CudaKernels`` interface."""
    global _kernels
    prev = _kernels
    _kernels = k
    return prev

"""Drop-in replacements for the reference's transform wrappers (xumx_slicq_v2/transforms.py).

Same names, call signatures, attributes and ragged per-bucket output layout, so the CDAE model,
separator, inference and export code of xumx-sliCQ-V2 run on the B200 kernels unchanged:

    make_filterbanks(nsgt_base, sample_rate=44100.0) -> (NSGT_SL, INSGT_SL)      transforms.py:11-18
    NSGTBase(scale, fbins, fmin, fmax=22050.0, fgamma=15.0, fs=44100.0, device)   transforms.py:21-94
    NSGT_SL(nsgt).forward(x[..., T])  -> list of [..., F_b, S, M_b, 2] float32    transforms.py:97-131
    INSGT_SL(nsgt).forward(X_list, length) -> [..., length] float32               transforms.py:134-178
    ComplexNorm().forward(list | Tensor)                                          transforms.py:181-208

Differences that are deliberate (DESIGN.md): outputs are contiguous per bucket (the reference
returns permuted views of [S,N,F,M] storage), INSGT_SL does not modify its input in place, and
there is no CPU execution path -- CPU inputs handed to a CUDA-resident module (the reference's
`predict_input_size` does that, transforms.py:83-89) are moved to the module's device.
"""
from __future__ import annotations

from typing import List

import torch
import torch.nn as nn
from torch import Tensor

from .nsgt import NSGT_sliced
from .plan import make_scale


def make_filterbanks(nsgt_base, sample_rate=44100.0):
    if sample_rate != 44100.0:
        raise ValueError("i was lazy and harcoded a lot of 44100.0, forgive me")  # transforms.py:12-13
    return NSGT_SL(nsgt_base), INSGT_SL(nsgt_base)


class NSGTBase(nn.Module):
    def __init__(self, scale, fbins, fmin, fmax=22050.0, fgamma=15.0, fs=44100.0, device="cuda"):
        super().__init__()
        self.fbins = fbins
        self.fmin = fmin
        self.fmax = fmax
        self.scl = make_scale(scale, self.fmin, self.fmax, self.fbins, fgamma)
        self.sllen, self.trlen = self.scl.suggested_sllen_trlen(fs)
        scale_to_print = scale if scale != "vqlog" else f"vqlog (gamma={fgamma})"
        print(f"scale={scale_to_print}, fbins={fbins}, fmin={fmin:.2f}, fmax={fmax:.2f}, "
              f"sllen={self.sllen}, trlen={self.trlen}")
        self.nsgt = NSGT_sliced(self.scl, self.sllen, self.trlen, fs, real=True, multichannel=True, device=device)
        self.M = self.nsgt.ncoefs
        self.fs = fs
        self.fbins_actual = self.nsgt.fbins_actual

    def max_bins(self, bandwidth):  # convert hz bandwidth into bins (transforms.py:73-78)
        if bandwidth is None or bandwidth < 0:
            return None
        freqs, _ = self.scl()
        freqs = torch.from_numpy(freqs)
        max_bin = min(torch.argwhere(freqs > bandwidth))[0]
        return max_bin + 1

    def predict_input_size(self, batch_size, nb_channels, seq_dur_s):
        fwd = NSGT_SL(self)
        x = torch.rand((batch_size, nb_channels, int(seq_dur_s * self.fs)), dtype=torch.float32)
        return fwd(x), x

    def _apply(self, fn, *a, **k):
        self.nsgt._apply(fn)
        return self


def _module_device(nsgt_base) -> torch.device:
    return nsgt_base.nsgt.device


class NSGT_SL(nn.Module):
    def __init__(self, nsgt):
        super().__init__()
        self.nsgt = nsgt

    def _apply(self, fn, *a, **k):
        self.nsgt._apply(fn)
        return self

    def forward(self, x: Tensor) -> List[Tensor]:
        """x [..., T] -> list over buckets of [..., F_b, S, M_b, 2] (last axis re, im)."""
        shape = x.size()
        dev = _module_device(self.nsgt)
        if x.device != dev and x.device.type == "cpu":
            x = x.to(dev)
        if torch.is_grad_enabled() and x.requires_grad:
            return list(_ForwardFn.apply(self, x))
        x = x.contiguous().view(-1, shape[-1])
        return self.nsgt.nsgt.forward_rows(x, lead=tuple(shape[:-1]), as_real=True)

    def forward_with_norm(self, x: Tensor):
        """(X, |X|) in one pass: ``X`` exactly as :meth:`forward`, ``|X|`` what ``ComplexNorm()(X)`` returns
        (list of [..., F_b, S, M_b]); the magnitude is written by the epilogue of the analysis kernels
        instead of a separate pass over the coefficients (reference call sites: separator.py:338,346,
        model.py via abs_of_real_complex phase.py:116-118).  Extra entry point: :meth:`forward` is unchanged."""
        shape = x.size()
        dev = _module_device(self.nsgt)
        if x.device != dev and x.device.type == "cpu":
            x = x.to(dev)
        x = x.contiguous().view(-1, shape[-1])
        return self.nsgt.nsgt.forward_rows(x, lead=tuple(shape[:-1]), as_real=True, with_norm=True)


class _ForwardFn(torch.autograd.Function):
    """Differentiable analysis: forward = NSGT kernels, backward = their exact adjoint on the synthesis kernels
    (third plan, SLICQ_PLAN_ADJOINT_OF_ANALYSIS).  The reference gets this gradient from torch autograd over
    nsgt/slicing.py + nsgt/nsgtf.py (training.py:77-95 when the input requires grad)."""

    @staticmethod
    def forward(ctx, module, x):
        ctx.module = module
        ctx.xshape = tuple(x.shape)
        with torch.no_grad():
            X = module.forward(x.detach())
        ctx.S = X[0].shape[-3]
        return tuple(X)

    @staticmethod
    def backward(ctx, *gX):
        module = ctx.module
        nsg = module.nsgt.nsgt
        dev = _module_device(module.nsgt)
        rows = 1
        for d in ctx.xshape[:-1]:
            rows *= d
        views, keep = [], []
        for g, (_, nb, M) in zip(gX, nsg.tables.buckets):
            if g is None:
                g = torch.zeros(ctx.xshape[:-1] + (nb, ctx.S, M, 2), dtype=torch.float32, device=dev)
            g = g.to(torch.float32).contiguous()
            keep.append(g)
            views.append((g.data_ptr(), nb * ctx.S * M, ctx.S * M, M))
        gx = nsg.analysis_adjoint_views(views, rows, ctx.S, dev, ctx.xshape[-1])
        del keep
        return None, gx.view(ctx.xshape)


class _InverseFn(torch.autograd.Function):
    """Differentiable synthesis: forward = INSGT kernels, backward = their exact adjoint on the
    analysis kernels (the transform is linear, so no activations are saved).  The reference gets
    this gradient from torch autograd over nsgt/nsigtf.py + nsgt/unslicing.py, which its README
    reports as a 5-25x slower epoch (SURVEY.md section 6.1); here it costs one analysis pass."""

    @staticmethod
    def forward(ctx, module, length, *X_list):
        ctx.module = module
        ctx.shapes = [tuple(X.shape) for X in X_list]
        with torch.no_grad():
            return module._forward_impl(list(X_list), length)

    @staticmethod
    def backward(ctx, gy):
        module = ctx.module
        nsg = module.nsgt.nsgt
        shp = ctx.shapes[0]
        lead, S = tuple(shp[:-4]), shp[-3]
        g = gy.contiguous().view(-1, gy.shape[-1])
        grads = nsg.synthesis_adjoint_rows(g, S, as_real=True, lead=lead)
        return (None, None) + tuple(grads)


class INSGT_SL(nn.Module):
    """Inverse wrapper.  X_list: per bucket [B, C, F_b, S, M_b, 2] or [T, B, C, F_b, S, M_b, 2]."""

    def __init__(self, nsgt):
        super().__init__()
        self.nsgt = nsgt

    def _apply(self, fn, *a, **k):
        self.nsgt._apply(fn)
        return self

    def forward(self, X_list, length: int, out: Tensor = None) -> Tensor:
        """transforms.py:154-178.  ``out`` (extension, optional): a contiguous float32 tensor of the result's shape
        to write into (staging buffers of a copy pipeline: saves one device copy); contiguous float32 inputs only."""
        if torch.is_grad_enabled() and any(X.requires_grad for X in X_list):
            return _InverseFn.apply(self, length, *X_list)
        return self._forward_impl(X_list, length, out)

    def _forward_impl(self, X_list, length: int, out: Tensor = None) -> Tensor:
        dev = _module_device(self.nsgt)
        nsg = self.nsgt.nsgt
        buckets = nsg.tables.buckets
        if len(X_list) == len(buckets) and all(
                X.is_contiguous() and X.dtype == torch.float32 and X.device == dev for X in X_list):
            # fast path (model outputs, forward outputs): bucket views straight from the real tensors,
            # no per-bucket view_as_complex / reshape on the host
            X0 = X_list[0]
            lead = tuple(X0.shape[:-4])
            S = X0.shape[-3]
            rows = 1
            for d in lead:
                rows *= d
            views = []
            for X, (_, nb, M) in zip(X_list, buckets):
                if tuple(X.shape) != lead + (nb, S, M, 2):
                    raise ValueError(f"bucket shape {tuple(X.shape)} != {lead + (nb, S, M, 2)}")
                views.append((X.data_ptr(), nb * S * M, S * M, M))
            nsg._BACKEND_check(X0)
            o2 = None
            if out is not None:
                if not out.is_contiguous() or tuple(out.shape[:-1]) != lead:
                    raise ValueError("out must be contiguous with the leading dimensions of the coefficients")
                o2 = out.view(rows, -1)
            y = nsg.backward_views(views, rows, S, dev, length, out=o2)
            return y.view(*lead, -1)
        if out is not None:
            raise ValueError("out= needs contiguous float32 coefficient tensors on the transform's device")
        cs = []
        lead = None
        for X in X_list:
            if X.device != dev and X.device.type == "cpu":
                X = X.to(dev)
            if X.dtype != torch.float32:
                X = X.to(torch.float32)
            if X.stride(-1) != 1 or X.stride(-2) != 2:
                X = X.contiguous()
            Xc = torch.view_as_complex(X)            # [*lead, F, S, M]
            lead = tuple(Xc.shape[:-3])
            try:
                Xc = Xc.view((-1,) + tuple(Xc.shape[-3:]))
            except RuntimeError:                      # leading dims not collapsible: make it so
                Xc = Xc.contiguous().view((-1,) + tuple(Xc.shape[-3:]))
            cs.append(Xc)
        y = nsg.backward_rows(cs, length)
        return y.view(*lead, -1)

    def forward_masked(self, X_list, mask_list, length: int) -> Tensor:
        """Fused realtime-model synthesis (not in the reference API; SURVEY.md section 8 row A10):
        X_list per bucket [B, C, F, S, M, 2] (the mixture sliCQT), mask_list per bucket
        [targets, B, C, F, S, M] (the CDAE sigmoid masks, model.py:231-234).  Returns
        [targets, B, C, length] == self.forward([m.unsqueeze(-1) * X for ...], length).
        Differentiable with respect to the masks and X (:class:`_MaskedInverseFn`)."""
        if torch.is_grad_enabled() and any(t.requires_grad for t in list(X_list) + list(mask_list)):
            return _MaskedInverseFn.apply(self, length, len(X_list), *X_list, *mask_list)
        return self._forward_masked_impl(X_list, mask_list, length)

    def _masked_inputs(self, X_list, mask_list):
        """(mixture per bucket complex [N, F, S, M], masks per bucket [targets, N, F, S, M], lead dims of X)."""
        dev = _module_device(self.nsgt)
        xs, ms = [], []
        lead = None
        for X, Mk in zip(X_list, mask_list):
            if X.device != dev and X.device.type == "cpu":
                X, Mk = X.to(dev), Mk.to(dev)
            if X.dtype != torch.float32:
                X = X.to(torch.float32)
            if X.stride(-1) != 1 or X.stride(-2) != 2:
                X = X.contiguous()
            Xc = torch.view_as_complex(X)
            lead = tuple(Xc.shape[:-3])
            xs.append(Xc.reshape((-1,) + tuple(Xc.shape[-3:])))
            ms.append(Mk.reshape((Mk.shape[0], -1) + tuple(Mk.shape[-3:])))
        return xs, ms, lead

    def _forward_masked_impl(self, X_list, mask_list, length: int) -> Tensor:
        xs, ms, lead = self._masked_inputs(X_list, mask_list)
        y = self.nsgt.nsgt.backward_rows_masked(xs, ms, length)
        return y.view(ms[0].shape[0], *lead, -1)


class _MaskedInverseFn(torch.autograd.Function):
    """Differentiable fused masked synthesis.  Output row r = t * N + n is y_r = S(m_r * X_n), so with g_r = dL/dy_r
        dL/dm_r = Re(conj(X_n) * S^T g_r),        dL/dX_n = sum_t m_{t,n} * S^T g_{t*N+n}.
    When only masks need a gradient, one call of the adjoint-of-synthesis analysis kernels takes the product with the
    mixture in their epilogue (NSGT_sliced.mask_grad_rows): S^T g is never stored.  When X needs one, S^T g is computed
    once (synthesis_adjoint_rows) and both products are taken in torch."""

    @staticmethod
    def forward(ctx, module, length, n, *tensors):
        ctx.module, ctx.length, ctx.n = module, length, n
        ctx.save_for_backward(*tensors)
        with torch.no_grad():
            return module._forward_masked_impl(list(tensors[:n]), list(tensors[n:]), length)

    @staticmethod
    def backward(ctx, gy):
        module, n = ctx.module, ctx.n
        nsg = module.nsgt.nsgt
        saved = ctx.saved_tensors
        X_list, mask_list = saved[:n], saved[n:]
        need_x, need_m = ctx.needs_input_grad[3:3 + n], ctx.needs_input_grad[3 + n:]
        xs, ms, lead = module._masked_inputs(X_list, mask_list)
        Tn, N = ms[0].shape[0], xs[0].shape[0]
        S = xs[0].shape[2]
        g = gy.reshape(Tn * N, gy.shape[-1])
        gx, gm = [None] * n, [None] * n
        if any(need_x):
            cadj = nsg.synthesis_adjoint_rows(g, S)                  # per bucket complex [T * N, F, S, M]
            for i, (c, x, m) in enumerate(zip(cadj, xs, ms)):
                c = c.view((Tn, N) + tuple(c.shape[1:]))
                if need_x[i]:
                    d = (c * m.to(torch.float32)).sum(0)
                    gx[i] = torch.view_as_real(d).reshape(X_list[i].shape).to(X_list[i].dtype)
                if need_m[i]:
                    gm[i] = torch.real(x.conj() * c)
        elif any(need_m):
            gm = nsg.mask_grad_rows(g, xs, Tn)
        for i in range(n):
            if not need_m[i]:
                gm[i] = None
            elif gm[i] is not None:
                gm[i] = gm[i].reshape(mask_list[i].shape).to(device=mask_list[i].device, dtype=mask_list[i].dtype)
            if gx[i] is not None:
                gx[i] = gx[i].to(device=X_list[i].device)
        return (None, None, None) + tuple(gx) + tuple(gm)


class ComplexNorm(nn.Module):
    """Magnitude of a ragged sliCQT list or a single tensor (transforms.py:181-208)."""

    def forward(self, spec):
        if isinstance(spec, list):
            return [torch.abs(torch.view_as_complex(c)) for c in spec]
        elif isinstance(spec, Tensor):
            return self.forward([spec])[0]
        else:
            raise ValueError(f"unsupported type for 'spec': {type(spec)}")

"""`NSGT_sliced` -- host-side mirror of the reference's sliced transform driver
(xumx_slicq_v2/nsgt/slicq.py:70-243) on top of the sm_100a kernels in libslicq.so.

Same constructor arguments, attributes (``sl_len, tr_area, fs, frqs, q, g, gd, M, rfbas, wins,
nn, sl, fbins_actual, ncoefs``) and methods (``forward((sig,))``, ``backward(cseq, length)``,
``coef_factor``, ``coef_factors()``) as the reference for the configuration its wrappers use
(``real=True, multichannel=True, reducedform=0, recwnd=False``; transforms.py:60-68).  The
computation itself is one call into the C-ABI (include/slicq.h); there is no torch.fft, no CPU
path and no fallback -- tensors must live on a CUDA device.

Coefficient layout: all buckets of one call share ONE allocation; bucket b is the contiguous
block ``[N, F_b, S, M_b]`` complex64 (the layout the CDAE model consumes).  ``forward`` returns
the reference's ``[S, N, F_b, M_b]`` axis order as permuted views of that block.
"""
from __future__ import annotations

import copy
from math import ceil
from typing import List, Sequence

import numpy as np
import torch

from . import _cabi
from . import plan as _plan


class _CudaBackend:
    """The only backend of the product: libslicq.so on a CUDA device."""

    name = "cuda"

    def lib(self):
        return _cabi.load()

    def check(self, t: torch.Tensor):
        if not t.is_cuda:
            raise RuntimeError(
                "xumx_slicq_b200 runs on CUDA devices only (hand-written sm_100a kernels, no CPU fallback); "
                f"got a tensor on '{t.device}'")

    def stream(self, device: torch.device) -> int:
        return torch.cuda.current_stream(device).cuda_stream

    def device_guard(self, device: torch.device):
        return torch.cuda.device(device)


_BACKEND = _CudaBackend()


class _AdjointTables:
    """Tables of the plan whose ANALYSIS entry is the adjoint of the normal plan's SYNTHESIS
    (include/slicq.h: SLICQ_PLAN_ADJOINT_OF_SYNTHESIS): no slicing window, dual windows * M^2."""

    def __init__(self, t):
        self.sllen, self.n_bins = t.sllen, t.n_bins
        self.bin_M, self.bin_pos = t.bin_M, t.bin_pos
        m2 = np.concatenate([np.full(int(m), float(m) * float(m), dtype=np.float64) for m in t.bin_M])
        self.win_fwd = (t.win_inv.astype(np.float64) * m2).astype(np.float32)
        self.win_inv = t.win_inv
        self.tukey = np.ones(t.sllen, dtype=np.float32)
        self.flags = 1


class _AdjointAnalysisTables:
    """Tables of the plan whose SYNTHESIS entry is the adjoint of the normal plan's ANALYSIS
    (include/slicq.h: SLICQ_PLAN_ADJOINT_OF_ANALYSIS): analysis windows g * L / (2 M^2) in place of the duals."""

    def __init__(self, t):
        self.sllen, self.n_bins = t.sllen, t.n_bins
        self.bin_M, self.bin_pos = t.bin_M, t.bin_pos
        s = np.concatenate([np.full(int(m), float(t.sllen) / (2.0 * float(m) * float(m)), dtype=np.float64) for m in t.bin_M])
        self.win_fwd = t.win_fwd
        self.win_inv = (t.win_fwd.astype(np.float64) * s).astype(np.float32)
        self.tukey = t.tukey
        self.flags = 2


class _PlanCache:
    """Per-device `slicq_plan` handles, created lazily; never copied (ctypes handles)."""

    def __init__(self):
        self.plans = {}

    def __deepcopy__(self, memo):
        return _PlanCache()

    def get(self, tables, device: torch.device) -> _cabi.Plan:
        key = (device.type, device.index)
        p = self.plans.get(key)
        if p is None:
            with _BACKEND.device_guard(device):
                p = _cabi.Plan(tables, _BACKEND.lib())
            self.plans[key] = p
        return p


class NSGT_sliced(torch.nn.Module):
    def __init__(self, scale, sl_len, tr_area, fs, min_win=16, Qvar=1, real=False, recwnd=False,
                 reducedform=0, multichannel=False, dtype=torch.float32, device="cpu"):
        # argument checks of slicq.py:86-94
        assert fs > 0
        assert sl_len > 0
        assert tr_area >= 0
        assert sl_len > tr_area * 2
        assert min_win > 0
        assert 0 <= reducedform <= 2
        assert sl_len % 4 == 0
        assert tr_area % 2 == 0
        super().__init__()
        if not real or not multichannel or reducedform != 0 or recwnd or dtype != torch.float32:
            raise NotImplementedError(
                "the B200 path implements the configuration the xumx-sliCQ wrappers use: "
                "real=True, multichannel=True, reducedform=0, recwnd=False, float32")
        self.device = torch.device(device)
        self.sl_len, self.tr_area, self.fs = int(sl_len), int(tr_area), fs
        self.real, self.userecwnd, self.reducedform, self.multichannel = real, recwnd, reducedform, multichannel
        self.scale = scale
        self.tables = _plan.design(scale, fs, self.sl_len, self.tr_area, min_win=min_win, qvar=Qvar)
        t = self.tables
        self.frqs, self.q = torch.from_numpy(t.frqs), torch.from_numpy(t.q)
        self.M = torch.from_numpy(t.M_all.copy())
        self.rfbas = torch.from_numpy(t.rfbas_all.copy())
        self.sl = slice(0, t.n_bins)
        self.fbins_actual = t.n_bins
        self.ncoefs = t.ncoefs
        self.nn = self.sl_len
        self._cache = _PlanCache()
        self._adj_cache = _PlanCache()
        self._adj_tables = None
        self._adja_cache = _PlanCache()
        self._adja_tables = None
        self._anchor = torch.zeros(1, device=self.device)
        self.device = self._anchor.device        # "cuda" -> "cuda:<current>": comparable with tensor.device

    # -- reference-visible window tables (host copies, for inspection / visualisation) -----
    def _split(self, flat: np.ndarray) -> List[torch.Tensor]:
        out, o = [], 0
        for m in self.tables.bin_M:
            out.append(torch.from_numpy(flat[o:o + int(m)].copy()))
            o += int(m)
        return out

    @property
    def g(self) -> List[torch.Tensor]:
        return self._split(self.tables.win_fwd)

    @property
    def gd(self) -> List[torch.Tensor]:
        return self._split(self.tables.win_inv)

    @property
    def wins(self) -> List[torch.Tensor]:
        out = []
        for m, c in zip(self.tables.bin_M, self.tables.bin_pos):
            out.append(torch.from_numpy((np.arange(-(int(m) // 2), int(m) - int(m) // 2) + int(c)) % self.nn))
        return out

    # -- device plumbing (nn.Module.to / .cuda / .cpu), slicq.py:175-180 -------------------
    def _apply(self, fn, *a, **k):
        self._anchor = fn(self._anchor)
        self.device = self._anchor.device
        return self

    def plan(self, device: torch.device | None = None) -> _cabi.Plan:
        return self._cache.get(self.tables, device or self.device)

    # -- layout helpers ---------------------------------------------------------------------
    def n_slices(self, n_samples: int) -> int:
        return self.tables.num_slices(int(n_samples))

    def alloc_coefficients(self, n_rows: int, n_slices: int, device, lead=None, as_real: bool = False) -> tuple:
        """One slab for all buckets (canonical packed layout of include/slicq.h).  Returns
        (slab, [bucket tensors]); buckets are complex64 [N,F,S,M] or, with ``as_real``, float32
        [*lead,F,S,M,2] views -- ONE as_strided per bucket (host overhead matters at small batch)."""
        t = self.tables
        slab = torch.empty(n_rows * n_slices * t.sum_M * 2, dtype=torch.float32, device=device)
        out, o = [], 0
        lead = tuple(lead) if lead is not None else (n_rows,)
        for (_, nb, M) in t.buckets:
            n = n_rows * nb * n_slices * M * 2
            inner = (nb * n_slices * M * 2, n_slices * M * 2, M * 2, 2, 1)           # strides of [N,F,S,M,2]
            if as_real:
                st, acc = [], nb * n_slices * M * 2
                for d in reversed(lead):
                    st.append(acc)
                    acc *= d
                out.append(slab.as_strided(lead + (nb, n_slices, M, 2), tuple(reversed(st)) + inner[1:], o))
            else:
                out.append(torch.view_as_complex(slab.as_strided((n_rows, nb, n_slices, M, 2), inner, o)))
            o += n
        return slab, out

    def alloc_norms(self, n_rows: int, n_slices: int, device, lead=None) -> tuple:
        """One float32 slab for the magnitudes of all buckets, same bucket order / packing as the
        coefficients.  Returns (slab, [bucket tensors [*lead, F, S, M]])."""
        t = self.tables
        slab = torch.empty(n_rows * n_slices * t.sum_M, dtype=torch.float32, device=device)
        out, o = [], 0
        lead = tuple(lead) if lead is not None else (n_rows,)
        for (_, nb, M) in t.buckets:
            inner = (n_slices * M, M, 1)                       # strides of [F,S,M]
            st, acc = [], nb * n_slices * M
            for d in reversed(lead):
                st.append(acc)
                acc *= d
            out.append(slab.as_strided(lead + (nb, n_slices, M), tuple(reversed(st)) + inner, o))
            o += n_rows * nb * n_slices * M
        return slab, out

    @staticmethod
    def _view_of(c: torch.Tensor) -> tuple:
        """(ptr, s_row, s_bin, s_slice) of a complex [N,F,S,M] tensor with contiguous M."""
        return (c.data_ptr(), c.stride(0), c.stride(1), c.stride(2))

    # -- analysis ---------------------------------------------------------------------------
    def forward_rows(self, x: torch.Tensor, k0: int = 0, n_slices: int | None = None, t0: int = 0,
                     lead=None, as_real: bool = False, with_norm: bool = False):
        """x [N, T] float32 -> list of contiguous [N, F_b, S, M_b] complex64 (canonical layout).

        ``with_norm``: also return the magnitudes |c| (list of float32 [*lead, F_b, S, M_b]) written by
        the same kernels (fused ComplexNorm, transforms.py:181-208): returns (coefficients, norms).

        ``k0 / n_slices / t0`` select a slice range of a longer signal (shard of a long track):
        local slice i is global slice k0+i and x[:, 0] is global sample t0."""
        _BACKEND.check(x)
        if x.dim() != 2:
            raise ValueError("expected [rows, samples]")
        if x.dtype != torch.float32:
            x = x.to(torch.float32)  # the reference computes in float32 regardless of input dtype
        if x.stride(1) != 1:
            x = x.contiguous()
        N, T = x.shape
        S = self.n_slices(T) if n_slices is None else int(n_slices)
        plan = self.plan(x.device)
        with _BACKEND.device_guard(x.device):
            slab, out = self.alloc_coefficients(N, S, x.device, lead=lead, as_real=as_real)
            nbytes = plan.scratch_bytes(N, S, False)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            if with_norm:
                nslab, norms = self.alloc_norms(N, S, x.device, lead=lead)
                plan.forward_packed_norm(x.data_ptr(), N, x.stride(0), T, int(t0), int(k0), S, slab.data_ptr(),
                                         nslab.data_ptr(), scratch.data_ptr(), nbytes, _BACKEND.stream(x.device))
                return out, norms
            plan.forward_packed(x.data_ptr(), N, x.stride(0), T, int(t0), int(k0), S, slab.data_ptr(),
                                scratch.data_ptr(), nbytes, _BACKEND.stream(x.device))
        return out

    def forward_rows_into(self, ctx: dict, x: torch.Tensor, k0: int = 0, n_slices: int | None = None, t0: int = 0):
        """``forward_rows`` into buffers kept in ``ctx`` (coefficient slab, bucket tensors, scratch): repeated calls of
        one shape allocate nothing and rebuild no views.  The returned tensors are overwritten by the next call."""
        _BACKEND.check(x)
        N, T = x.shape
        S = self.n_slices(T) if n_slices is None else int(n_slices)
        plan = self.plan(x.device)
        key = (N, S, x.device)
        with _BACKEND.device_guard(x.device):
            if ctx.get("fwd_key") != key:
                ctx["slab"], ctx["coefs"] = self.alloc_coefficients(N, S, x.device)
                ctx["fwd_bytes"] = plan.scratch_bytes(N, S, False)
                ctx["fwd_scratch"] = torch.empty(ctx["fwd_bytes"], dtype=torch.uint8, device=x.device)
                ctx["fwd_key"] = key
            plan.forward_packed(x.data_ptr(), N, x.stride(0), T, int(t0), int(k0), S, ctx["slab"].data_ptr(),
                                ctx["fwd_scratch"].data_ptr(), ctx["fwd_bytes"], _BACKEND.stream(x.device))
        return ctx["coefs"]

    def forward(self, sig: Sequence[torch.Tensor]) -> List[torch.Tensor]:
        """slicq.py:182-196: ``sig`` is a 1-tuple holding [N, T]; returns list of [S, N, F_b, M_b]."""
        (x,) = sig
        return [c.permute(2, 0, 1, 3) for c in self.forward_rows(x)]

    # -- synthesis --------------------------------------------------------------------------
    def backward_rows(self, coefs: Sequence[torch.Tensor], length: int, k0: int = 0, t0: int = 0,
                      halo_out: torch.Tensor | None = None, ctx: dict | None = None) -> torch.Tensor:
        """list of complex [N, F_b, S, M_b] (any strides, M contiguous) -> [N, length] float32.
        ``ctx`` (a dict the caller keeps, keyed by the input tensors): bucket views, scratch and the output tensor
        are built once and reused by later calls on the same tensors."""
        t = self.tables
        if ctx is not None and "inv_views" in ctx:
            plan = self.plan(coefs[0].device)
            y = ctx["y"]
            with _BACKEND.device_guard(coefs[0].device):
                plan.inverse(ctx["inv_views"], ctx["inv_N"], ctx["inv_S"], int(k0), y.data_ptr(), y.stride(0) if y.shape[1] else 1,
                             y.shape[1], int(t0), halo_out.data_ptr() if halo_out is not None else 0,
                             ctx["inv_scratch"].data_ptr(), ctx["inv_bytes"], _BACKEND.stream(coefs[0].device))
            return y
        if len(coefs) != len(t.buckets):
            raise ValueError(f"expected {len(t.buckets)} coefficient buckets, got {len(coefs)}")
        c0 = coefs[0]
        _BACKEND.check(c0)
        N, S = c0.shape[0], c0.shape[2]
        views = []
        keep = []
        for c, (_, nb, M) in zip(coefs, t.buckets):
            if c.dtype != torch.complex64:
                c = c.to(torch.complex64)
            if tuple(c.shape) != (N, nb, S, M):
                raise ValueError(f"bucket shape {tuple(c.shape)} != {(N, nb, S, M)}")
            if c.stride(3) != 1 and M > 1:
                c = c.contiguous()
            keep.append(c)
            views.append(self._view_of(c))
        length = int(length)
        avail = (int(k0) + S) * t.hop - int(t0)
        out_len = max(0, min(length, avail))  # reblock(fulllast=False): at most the samples that exist
        plan = self.plan(c0.device)
        with _BACKEND.device_guard(c0.device):
            y = torch.empty((N, out_len), dtype=torch.float32, device=c0.device)
            nbytes = plan.scratch_bytes(N, S, True)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=c0.device)
            plan.inverse(views, N, S, int(k0), y.data_ptr(), y.stride(0) if out_len else 1, out_len, int(t0),
                         halo_out.data_ptr() if halo_out is not None else 0,
                         scratch.data_ptr(), nbytes, _BACKEND.stream(c0.device))
        if ctx is not None:
            ctx.update(inv_views=plan.make_views(views), inv_N=N, inv_S=S, y=y, inv_scratch=scratch, inv_bytes=nbytes, keep=keep)
        del keep
        return y

    def backward_rows_masked(self, mix: Sequence[torch.Tensor], masks: Sequence[torch.Tensor], length: int,
                             k0: int = 0, t0: int = 0, halo_out: torch.Tensor | None = None,
                             ctx: dict | None = None) -> torch.Tensor:
        """Synthesis fused with mask * mixture (realtime model, phase.py:96-113 / model.py:258-265).

        mix: per bucket complex [N, F_b, S, M_b]; masks: per bucket float32 [T, N, F_b, S, M_b].
        Returns [T * N, length] (row t * N + n) = inverse of masks[t, n] * mix[n], bitwise equal to
        ``backward_rows([ (m * x).flatten(0, 1) ])`` without materialising the T coefficient sets."""
        t = self.tables
        if ctx is not None and "m_views" in ctx:
            plan = self.plan(mix[0].device)
            y = ctx["y"]
            with _BACKEND.device_guard(mix[0].device):
                plan.inverse_masked(ctx["x_views"], ctx["m_views"], ctx["inv_T"], ctx["inv_N"], ctx["inv_S"], int(k0), y.data_ptr(),
                                    y.stride(0) if y.shape[1] else 1, y.shape[1], int(t0),
                                    halo_out.data_ptr() if halo_out is not None else 0,
                                    ctx["inv_scratch"].data_ptr(), ctx["inv_bytes"], _BACKEND.stream(mix[0].device))
            return y
        if len(mix) != len(t.buckets) or len(masks) != len(t.buckets):
            raise ValueError(f"expected {len(t.buckets)} buckets")
        c0 = mix[0]
        _BACKEND.check(c0)
        N, S = c0.shape[0], c0.shape[2]
        Tn = masks[0].shape[0]
        vx, vm, keep = [], [], []
        for c, m, (_, nb, M) in zip(mix, masks, t.buckets):
            if c.dtype != torch.complex64:
                c = c.to(torch.complex64)
            if tuple(c.shape) != (N, nb, S, M) or tuple(m.shape) != (Tn, N, nb, S, M):
                raise ValueError(f"bucket shapes {tuple(c.shape)}, {tuple(m.shape)} != {(N, nb, S, M)}, {(Tn, N, nb, S, M)}")
            if c.stride(3) != 1:
                c = c.contiguous()
            m = m.to(torch.float32).reshape(Tn * N, nb, S, M)
            if m.stride(3) != 1:
                m = m.contiguous()
            keep += [c, m]
            vx.append(self._view_of(c))
            vm.append(self._view_of(m))
        length = int(length)
        out_len = max(0, min(length, (int(k0) + S) * t.hop - int(t0)))
        plan = self.plan(c0.device)
        with _BACKEND.device_guard(c0.device):
            y = torch.empty((Tn * N, out_len), dtype=torch.float32, device=c0.device)
            nbytes = plan.scratch_bytes(Tn * N, S, True)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=c0.device)
            plan.inverse_masked(vx, vm, Tn, N, S, int(k0), y.data_ptr(), y.stride(0) if out_len else 1, out_len,
                                int(t0), halo_out.data_ptr() if halo_out is not None else 0,
                                scratch.data_ptr(), nbytes, _BACKEND.stream(c0.device))
        if ctx is not None:
            ctx.update(x_views=plan.make_views(vx), m_views=plan.make_views(vm), inv_T=Tn, inv_N=N, inv_S=S, y=y,
                       inv_scratch=scratch, inv_bytes=nbytes, keep=keep)
        del keep
        return y

    @staticmethod
    def _BACKEND_check(t: torch.Tensor):
        _BACKEND.check(t)

    def backward_views(self, views, n_rows: int, n_slices: int, device, length: int, k0: int = 0, t0: int = 0,
                       halo_out: torch.Tensor | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
        """Synthesis from precomputed (ptr, s_row, s_bin, s_slice) bucket views (complex64 element
        strides); the caller keeps the tensors alive and guarantees shapes / 16-byte alignment.
        ``out``: optional float32 [n_rows, out_len] tensor (unit stride along samples) to write into."""
        t = self.tables
        length = int(length)
        out_len = max(0, min(length, (int(k0) + n_slices) * t.hop - int(t0)))
        plan = self.plan(device)
        with _BACKEND.device_guard(device):
            if out is not None:
                if tuple(out.shape) != (n_rows, out_len) or out.dtype != torch.float32 or out.device != device or \
                        (out_len > 1 and out.stride(1) != 1):
                    raise ValueError(f"out must be a float32 [{n_rows}, {out_len}] tensor on {device}")
                y = out
            else:
                y = torch.empty((n_rows, out_len), dtype=torch.float32, device=device)
            nbytes = plan.scratch_bytes(n_rows, n_slices, True)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=device)
            plan.inverse(views, n_rows, n_slices, int(k0), y.data_ptr(), y.stride(0) if out_len else 1, out_len,
                         int(t0), halo_out.data_ptr() if halo_out is not None else 0,
                         scratch.data_ptr(), nbytes, _BACKEND.stream(device))
        return y

    # -- adjoint of the synthesis (autograd through the inverse transform) ----------------------
    def synthesis_adjoint_rows(self, g: torch.Tensor, n_slices: int, as_real: bool = False, lead=None) -> List[torch.Tensor]:
        """g [N, length] (gradient w.r.t. the synthesis output) -> per bucket [N, F_b, S, M_b] complex:
        the transpose of ``backward_rows`` with respect to the real inner product
        <y, g> = sum y*g, <c, d> = sum Re(c) Re(d) + Im(c) Im(d).  Runs on the analysis kernels
        with a second plan (no slicing window, dual windows, zero instead of mirrored margins, and the transpose of the
        mirrored-bin pass for bins that reach below DC)."""
        _BACKEND.check(g)
        if self._adj_tables is None:
            self._adj_tables = _AdjointTables(self.tables)
        if g.dtype != torch.float32:
            g = g.to(torch.float32)
        if g.stride(1) != 1:
            g = g.contiguous()
        N, T = g.shape
        plan = self._adj_cache.get(self._adj_tables, g.device)
        with _BACKEND.device_guard(g.device):
            slab, out = self.alloc_coefficients(N, n_slices, g.device, lead=lead, as_real=as_real)
            nbytes = plan.scratch_bytes(N, n_slices, False)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=g.device)
            plan.forward_packed(g.data_ptr(), N, g.stride(0), T, 0, 0, n_slices, slab.data_ptr(),
                                scratch.data_ptr(), nbytes, _BACKEND.stream(g.device))
        return out

    def mask_grad_rows(self, g: torch.Tensor, mix: Sequence[torch.Tensor], n_targets: int,
                       lead=None) -> List[torch.Tensor]:
        """Gradient of ``backward_rows_masked`` with respect to its masks.  g [T * N, length] (gradient w.r.t. that
        call's output, row t * N + n), mix: the per-bucket complex [N, F_b, S, M_b] mixture it read (any strides, M
        contiguous).  Returns per bucket float32 [T * N, F_b, S, M_b] (or [*lead, F_b, S, M_b]), one slab as
        ``alloc_norms``: Re(conj(mix[n]) * (S^T g)[t * N + n]).  The adjoint of the synthesis runs on the analysis
        kernels of the ``synthesis_adjoint_rows`` plan, whose epilogue takes the product with the mixture: S^T g is never
        stored."""
        _BACKEND.check(g)
        t = self.tables
        if len(mix) != len(t.buckets):
            raise ValueError(f"expected {len(t.buckets)} buckets")
        if self._adj_tables is None:
            self._adj_tables = _AdjointTables(self.tables)
        if g.dtype != torch.float32:
            g = g.to(torch.float32)
        if g.stride(1) != 1:
            g = g.contiguous()
        Tn = int(n_targets)
        N, S = mix[0].shape[0], mix[0].shape[2]
        if g.shape[0] != Tn * N:
            raise ValueError(f"expected {Tn * N} gradient rows, got {g.shape[0]}")
        vx, keep = [], []
        for c, (_, nb, M) in zip(mix, t.buckets):
            if c.dtype != torch.complex64:
                c = c.to(torch.complex64)
            if tuple(c.shape) != (N, nb, S, M):
                raise ValueError(f"bucket shape {tuple(c.shape)} != {(N, nb, S, M)}")
            if c.stride(3) != 1:
                c = c.contiguous()
            keep.append(c)
            vx.append(self._view_of(c))
        plan = self._adj_cache.get(self._adj_tables, g.device)
        with _BACKEND.device_guard(g.device):
            slab, out = self.alloc_norms(Tn * N, S, g.device, lead=lead)
            vg = [(o.data_ptr(), nb * S * M, S * M, M) for o, (_, nb, M) in zip(out, t.buckets)]
            nbytes = plan.scratch_bytes(Tn * N, S, False)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=g.device)
            plan.forward_mask_grad(g.data_ptr(), Tn, N, g.stride(0), g.shape[1], 0, 0, S, vx, vg,
                                   scratch.data_ptr(), nbytes, _BACKEND.stream(g.device))
        del keep
        return out

    def analysis_adjoint_views(self, views, n_rows: int, n_slices: int, device, length: int) -> torch.Tensor:
        """Gradient of the analysis: per-bucket views of d [N, F_b, S, M_b] complex (gradient w.r.t. the coefficients) ->
        [N, length] float32 = A^T d, the transpose of ``forward_rows`` with respect to the real inner products
        <c, d> = sum Re(c) Re(d) + Im(c) Im(d), <x, g> = sum x g.  Runs on the SYNTHESIS kernels with a third plan
        (analysis windows instead of duals, out-of-band bin parts folded back, slicing window before the overlap-add)."""
        if self._adja_tables is None:
            self._adja_tables = _AdjointAnalysisTables(self.tables)
        plan = self._adja_cache.get(self._adja_tables, device)
        length = int(length)
        with _BACKEND.device_guard(device):
            # the analysis zero-extends the signal: slices reach past `length`, their gradient there is dropped
            y = torch.empty((n_rows, length), dtype=torch.float32, device=device)
            nbytes = plan.scratch_bytes(n_rows, n_slices, True)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=device)
            plan.inverse(views, n_rows, n_slices, 0, y.data_ptr(), y.stride(0) if length else 1, length, 0, 0,
                         scratch.data_ptr(), nbytes, _BACKEND.stream(device))
        return y

    def backward(self, cseq: Sequence[torch.Tensor], length: int) -> torch.Tensor:
        """slicq.py:198-230: list of [S, N, F_b, M_b] complex -> [N, length].
        Unlike the reference this does not modify ``cseq`` in place."""
        return self.backward_rows([c.permute(1, 2, 0, 3) for c in cseq], length)

    # -- bookkeeping ------------------------------------------------------------------------
    @property
    def coef_factor(self) -> float:  # slicq.py:232-234
        return float(self.ncoefs) / self.sl_len

    def coef_factors(self) -> List[float]:  # slicq.py:236-243
        return [float(int(ceil(float(m) / m)) * m) / self.sl_len for m in map(int, self.tables.bin_M)]

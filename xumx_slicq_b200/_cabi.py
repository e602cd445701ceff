"""ctypes binding of the C-ABI in include/slicq.h (libslicq.so, hand-written sm_100a kernels).

There is no fallback: if the shared library is missing or a call fails this module raises.
PyTorch is used by the callers for device memory and streams only; no torch type crosses the ABI.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libslicq.so"

SLICQ_OK = 0
SLICQ_E_INVALID = -1
SLICQ_E_UNSUPPORTED = -2
SLICQ_E_CUDA = -3
SLICQ_E_SCRATCH = -4

EXPORTS = (
    "slicq_abi_version", "slicq_build_kind", "slicq_last_error", "slicq_plan_create", "slicq_plan_destroy",
    "slicq_plan_n_buckets", "slicq_plan_bucket_info", "slicq_plan_num_slices",
    "slicq_scratch_bytes", "slicq_forward", "slicq_forward_packed", "slicq_forward_norm", "slicq_forward_packed_norm", "slicq_inverse", "slicq_inverse_masked", "slicq_forward_mask_grad",
    "slicq_launch_count",
    "slicq_profile_enable", "slicq_profile_read",
)
KERNEL_NAMES = ("slice_fft_fwd", "bins_fwd", "bins_inv", "slice_fft_inv")


class SlicqTablesC(C.Structure):
    _fields_ = [
        ("sl_len", C.c_int32),
        ("n_bins", C.c_int32),
        ("bin_M", C.POINTER(C.c_int32)),
        ("bin_pos", C.POINTER(C.c_int32)),
        ("win_fwd", C.POINTER(C.c_float)),
        ("win_inv", C.POINTER(C.c_float)),
        ("tukey", C.POINTER(C.c_float)),
        ("flags", C.c_int32),
    ]


class BucketViewC(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("s_row", C.c_int64), ("s_bin", C.c_int64), ("s_slice", C.c_int64)]


class SlicqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libslicq error {code}: {msg}")
        self.code = code


def _declare(lib: C.CDLL) -> C.CDLL:
    lib.slicq_abi_version.restype = C.c_int
    lib.slicq_build_kind.restype = C.c_int
    lib.slicq_last_error.restype = C.c_char_p
    lib.slicq_plan_create.argtypes = [C.POINTER(SlicqTablesC), C.POINTER(C.c_void_p)]
    lib.slicq_plan_create.restype = C.c_int
    lib.slicq_plan_destroy.argtypes = [C.c_void_p]
    lib.slicq_plan_destroy.restype = None
    lib.slicq_plan_n_buckets.argtypes = [C.c_void_p]
    lib.slicq_plan_n_buckets.restype = C.c_int
    lib.slicq_plan_bucket_info.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                           C.POINTER(C.c_int32)]
    lib.slicq_plan_bucket_info.restype = C.c_int
    lib.slicq_plan_num_slices.argtypes = [C.c_void_p, C.c_int64]
    lib.slicq_plan_num_slices.restype = C.c_int64
    lib.slicq_scratch_bytes.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int]
    lib.slicq_scratch_bytes.restype = C.c_size_t
    lib.slicq_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                  C.c_int64, C.POINTER(BucketViewC), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.slicq_forward.restype = C.c_int
    lib.slicq_forward_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.slicq_forward_packed.restype = C.c_int
    lib.slicq_forward_norm.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                       C.c_int64, C.POINTER(BucketViewC), C.POINTER(BucketViewC), C.c_void_p, C.c_size_t,
                                       C.c_void_p]
    lib.slicq_forward_norm.restype = C.c_int
    lib.slicq_forward_packed_norm.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                              C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                              C.c_void_p]
    lib.slicq_forward_packed_norm.restype = C.c_int
    lib.slicq_inverse.argtypes = [C.c_void_p, C.POINTER(BucketViewC), C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                  C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.slicq_inverse.restype = C.c_int
    lib.slicq_inverse_masked.argtypes = [C.c_void_p, C.POINTER(BucketViewC), C.POINTER(BucketViewC), C.c_int64, C.c_int64,
                                         C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                         C.c_void_p, C.c_size_t, C.c_void_p]
    lib.slicq_inverse_masked.restype = C.c_int
    lib.slicq_forward_mask_grad.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                            C.c_int64, C.c_int64, C.POINTER(BucketViewC), C.POINTER(BucketViewC),
                                            C.c_void_p, C.c_size_t, C.c_void_p]
    lib.slicq_forward_mask_grad.restype = C.c_int
    lib.slicq_launch_count.restype = C.c_int64
    lib.slicq_profile_enable.argtypes = [C.c_int]
    lib.slicq_profile_enable.restype = C.c_int
    lib.slicq_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    lib.slicq_profile_read.restype = C.c_int
    return lib


def profile_enable(on: bool, lib: C.CDLL | None = None) -> None:
    (lib or load()).slicq_profile_enable(int(bool(on)))


def profile_read(lib: C.CDLL | None = None) -> dict:
    """{kernel name: (total ms, launches)} since the last read (synchronises the recorded events)."""
    ms = (C.c_double * 8)()
    n = (C.c_int64 * 8)()
    (lib or load()).slicq_profile_read(ms, n)
    return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(KERNEL_NAMES)}


def library_path() -> str:
    return os.path.join(_HERE, LIB_NAME)


_lib = None


def load(path: str | None = None) -> C.CDLL:
    """Load libslicq.so (built by ``__graft_entry__.build()`` / ``python -m xumx_slicq_b200.build``)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or library_path()
    if not os.path.exists(p):
        raise ImportError(
            f"{p} not found: the CUDA extension is required (no CPU fallback). "
            "Build it with `python -m xumx_slicq_b200.build`.")
    lib = _declare(C.CDLL(p))
    if lib.slicq_abi_version() != 1:
        raise ImportError(f"{p}: ABI version {lib.slicq_abi_version()} != 1")
    if path is None:
        # the product loader only takes CUDA builds: the host emulation library of the test tier (tests/emu) exports
        # the same C ABI and must never stand in for the GPU
        if lib.slicq_build_kind() != 0:
            raise ImportError(f"{p} is not a CUDA build of libslicq (host emulation libraries are test infrastructure)")
        _lib = lib
    return lib


def _check(lib: C.CDLL, rc: int) -> None:
    if rc != SLICQ_OK:
        msg = lib.slicq_last_error().decode("utf-8", "replace")
        if rc in (SLICQ_E_INVALID, SLICQ_E_UNSUPPORTED):
            raise ValueError(f"libslicq: {msg}")
        raise SlicqError(rc, msg)


class Plan:
    """Owns a ``slicq_plan*``; device tables are uploaded to the current CUDA device."""

    def __init__(self, tables, lib: C.CDLL | None = None):
        self.lib = lib or load()
        self._keep = [np.ascontiguousarray(tables.bin_M, dtype=np.int32),
                      np.ascontiguousarray(tables.bin_pos, dtype=np.int32),
                      np.ascontiguousarray(tables.win_fwd, dtype=np.float32),
                      np.ascontiguousarray(tables.win_inv, dtype=np.float32),
                      np.ascontiguousarray(tables.tukey, dtype=np.float32)]
        t = SlicqTablesC(
            int(tables.sllen), int(tables.n_bins),
            self._keep[0].ctypes.data_as(C.POINTER(C.c_int32)),
            self._keep[1].ctypes.data_as(C.POINTER(C.c_int32)),
            self._keep[2].ctypes.data_as(C.POINTER(C.c_float)),
            self._keep[3].ctypes.data_as(C.POINTER(C.c_float)),
            self._keep[4].ctypes.data_as(C.POINTER(C.c_float)),
            int(getattr(tables, "flags", 0)))
        h = C.c_void_p()
        _check(self.lib, self.lib.slicq_plan_create(C.byref(t), C.byref(h)))
        self.handle = h
        nb = self.lib.slicq_plan_n_buckets(h)
        self.buckets = []
        for b in range(nb):
            fb, n, m = C.c_int32(), C.c_int32(), C.c_int32()
            _check(self.lib, self.lib.slicq_plan_bucket_info(h, b, C.byref(fb), C.byref(n), C.byref(m)))
            self.buckets.append((fb.value, n.value, m.value))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.slicq_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def num_slices(self, n_samples: int) -> int:
        return int(self.lib.slicq_plan_num_slices(self.handle, int(n_samples)))

    def scratch_bytes(self, n_rows: int, n_slices: int, inverse: bool) -> int:
        return int(self.lib.slicq_scratch_bytes(self.handle, int(n_rows), int(n_slices), int(bool(inverse))))

    def _views(self, views):
        """ctypes array of bucket views; an array built earlier (``make_views``) passes through, so callers that
        repeat a call on the same buffers pay for the 70 struct fills once."""
        if isinstance(views, C.Array):
            return views
        arr = (BucketViewC * len(views))()
        for i, (ptr, s_row, s_bin, s_slice) in enumerate(views):
            arr[i] = BucketViewC(ptr, s_row, s_bin, s_slice)
        return arr

    def make_views(self, views: Sequence[tuple]):
        return self._views(views)

    def forward(self, x_ptr: int, n_rows: int, x_row_stride: int, n_samples: int, t0: int, k0: int,
                n_slices: int, views: Sequence[tuple], scratch_ptr: int, scratch_bytes: int, stream: int):
        _check(self.lib, self.lib.slicq_forward(
            self.handle, C.c_void_p(x_ptr), n_rows, x_row_stride, n_samples, t0, k0, n_slices,
            self._views(views), C.c_void_p(scratch_ptr), scratch_bytes, C.c_void_p(stream)))

    def forward_packed(self, x_ptr: int, n_rows: int, x_row_stride: int, n_samples: int, t0: int, k0: int,
                       n_slices: int, coefs_ptr: int, scratch_ptr: int, scratch_bytes: int, stream: int):
        _check(self.lib, self.lib.slicq_forward_packed(
            self.handle, C.c_void_p(x_ptr), n_rows, x_row_stride, n_samples, t0, k0, n_slices,
            C.c_void_p(coefs_ptr), C.c_void_p(scratch_ptr), scratch_bytes, C.c_void_p(stream)))

    def forward_packed_norm(self, x_ptr: int, n_rows: int, x_row_stride: int, n_samples: int, t0: int, k0: int,
                            n_slices: int, coefs_ptr: int, norms_ptr: int, scratch_ptr: int, scratch_bytes: int,
                            stream: int):
        _check(self.lib, self.lib.slicq_forward_packed_norm(
            self.handle, C.c_void_p(x_ptr), n_rows, x_row_stride, n_samples, t0, k0, n_slices,
            C.c_void_p(coefs_ptr), C.c_void_p(norms_ptr), C.c_void_p(scratch_ptr), scratch_bytes, C.c_void_p(stream)))

    def forward_norm(self, x_ptr: int, n_rows: int, x_row_stride: int, n_samples: int, t0: int, k0: int,
                     n_slices: int, views: Sequence[tuple], norm_views: Sequence[tuple], scratch_ptr: int,
                     scratch_bytes: int, stream: int):
        _check(self.lib, self.lib.slicq_forward_norm(
            self.handle, C.c_void_p(x_ptr), n_rows, x_row_stride, n_samples, t0, k0, n_slices,
            self._views(views), self._views(norm_views), C.c_void_p(scratch_ptr), scratch_bytes, C.c_void_p(stream)))

    def inverse(self, views: Sequence[tuple], n_rows: int, n_slices: int, k0: int, y_ptr: int, y_row_stride: int,
                length: int, t0: int, halo_ptr: int, scratch_ptr: int, scratch_bytes: int, stream: int):
        _check(self.lib, self.lib.slicq_inverse(
            self.handle, self._views(views), n_rows, n_slices, k0, C.c_void_p(y_ptr), y_row_stride, length, t0,
            C.c_void_p(halo_ptr) if halo_ptr else None, C.c_void_p(scratch_ptr), scratch_bytes,
            C.c_void_p(stream)))

    def inverse_masked(self, mix_views: Sequence[tuple], mask_views: Sequence[tuple], n_targets: int, n_rows: int,
                       n_slices: int, k0: int, y_ptr: int, y_row_stride: int, length: int, t0: int, halo_ptr: int,
                       scratch_ptr: int, scratch_bytes: int, stream: int):
        _check(self.lib, self.lib.slicq_inverse_masked(
            self.handle, self._views(mix_views), self._views(mask_views), n_targets, n_rows, n_slices, k0,
            C.c_void_p(y_ptr), y_row_stride, length, t0, C.c_void_p(halo_ptr) if halo_ptr else None,
            C.c_void_p(scratch_ptr), scratch_bytes, C.c_void_p(stream)))

    def forward_mask_grad(self, g_ptr: int, n_targets: int, n_rows: int, g_row_stride: int, n_samples: int, t0: int,
                          k0: int, n_slices: int, mix_views: Sequence[tuple], grad_views: Sequence[tuple],
                          scratch_ptr: int, scratch_bytes: int, stream: int):
        _check(self.lib, self.lib.slicq_forward_mask_grad(
            self.handle, C.c_void_p(g_ptr), n_targets, n_rows, g_row_stride, n_samples, t0, k0, n_slices,
            self._views(mix_views), self._views(grad_views), C.c_void_p(scratch_ptr), scratch_bytes, C.c_void_p(stream)))

    def launch_count(self) -> int:
        return int(self.lib.slicq_launch_count())

"""The seven call entries of the C ABI (slicq_forward, _forward_norm, _forward_packed, _forward_packed_norm,
_forward_mask_grad, _inverse, _inverse_masked), called directly on the host emulation (tests/emu).  Checked: the error
code and message of each single-fault call, and that splitting a call into two row groups (SLICQ_SPLIT_UNITS) or into
chunks (SLICQ_CHUNK_MB) leaves every output bitwise unchanged, where a shared mixture allows or forbids the split.
CPU tier only."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest

from xumx_slicq_b200 import _cabi
from xumx_slicq_b200.nsgt import _AdjointTables

INVALID, SCRATCH = _cabi.SLICQ_E_INVALID, _cabi.SLICQ_E_SCRATCH
CFG = ("mel", 32, 115.5)      # generic slice kernels, L = 2016; bin 1 reaches below DC (mirrored-bin passes)
ENTRIES = ("forward", "forward_norm", "forward_packed", "forward_packed_norm", "forward_mask_grad", "inverse",
           "inverse_masked")


@pytest.fixture(scope="module")
def lib():
    from tests.emu.emu_backend import EmuBackend
    return EmuBackend().lib()


@pytest.fixture(scope="module")
def tables():
    from xumx_slicq_b200.plan import design, make_scale
    with contextlib.redirect_stdout(io.StringIO()):
        scl = make_scale(CFG[0], CFG[2], 22050.0, CFG[1])
    sl, tr = scl.suggested_sllen_trlen(44100.0)
    return design(scl, 44100.0, sl, tr)


def _plans(lib, tables, monkeypatch, split_units=None, chunk_mb=None):
    """The normal and the adjoint-of-synthesis plan, created under the given SLICQ_SPLIT_UNITS / SLICQ_CHUNK_MB."""
    with monkeypatch.context() as m:
        for k, v in (("SLICQ_SPLIT_UNITS", split_units), ("SLICQ_CHUNK_MB", chunk_mb)):
            if v is None:
                m.delenv(k, raising=False)
            else:
                m.setenv(k, str(v))
        return _cabi.Plan(tables, lib), _cabi.Plan(_AdjointTables(tables), lib)


class Call:
    """Buffers and arguments of one valid call of `entry` with `n_rows` output rows (n_targets x mix_rows where a
    mixture is shared); `args(**faults)` gives its argument list with the named arguments replaced."""

    def __init__(self, entry, plan, adj_plan, hop, n_rows, n_slices, T, mix_rows=None, seed=0):
        rng = np.random.default_rng(seed)
        self.entry, self.plan = entry, adj_plan if entry == "forward_mask_grad" else plan
        self.n_rows, self.n_slices, self.T = n_rows, n_slices, T
        self.mix_rows = mix_rows or n_rows
        self.n_targets = n_rows // self.mix_rows
        self.inverse = entry.startswith("inverse")
        buckets = self.plan.buckets
        shared = entry in ("forward_mask_grad", "inverse_masked")
        coef_rows = self.mix_rows if shared else n_rows

        def cplx(rows, F, M):
            return (rng.standard_normal((rows, F, n_slices, M)) + 1j * rng.standard_normal((rows, F, n_slices, M))
                    ).astype(np.complex64)
        if self.inverse or entry == "forward_mask_grad":
            self.coefs = [cplx(coef_rows, F, M) for (_, F, M) in buckets]
        else:
            self.coefs = [np.zeros((n_rows, F, n_slices, M), np.complex64) for (_, F, M) in buckets]
        self.aux = None
        if entry in ("forward_norm", "forward_packed_norm", "forward_mask_grad"):
            self.aux = [np.zeros((n_rows, F, n_slices, M), np.float32) for (_, F, M) in buckets]
        elif entry == "inverse_masked":
            self.aux = [rng.random((n_rows, F, n_slices, M), dtype=np.float32) for (_, F, M) in buckets]
        if entry.startswith("forward_packed"):     # one allocation, the buckets one after the other
            self.coefs = [np.zeros(sum(c.size for c in self.coefs), np.complex64)]
            if self.aux is not None:
                self.aux = [np.zeros(sum(a.size for a in self.aux), np.float32)]
        self.x = (rng.standard_normal((n_rows, T)) if not self.inverse else np.zeros((n_rows, T))).astype(np.float32)
        self.halo = np.zeros((n_rows, hop), np.float32)
        self.scratch_bytes = self.plan.scratch_bytes(n_rows, n_slices, self.inverse)
        self._scratch = np.zeros(self.scratch_bytes + 64, np.uint8)
        base = self._scratch.ctypes.data
        self.scratch = base + (-base) % 16

    def outputs(self):
        if self.inverse:
            return [self.x, self.halo]
        return self.coefs + (self.aux or []) if self.entry != "forward_mask_grad" else self.aux

    @staticmethod
    def _views(arrs, null_bucket=None):
        v = (_cabi.BucketViewC * len(arrs))()
        for i, a in enumerate(arrs):
            s = [st // a.itemsize for st in a.strides]
            v[i] = _cabi.BucketViewC(None if i == null_bucket else a.ctypes.data, s[0], s[1], s[2])
        return v

    def args(self, **f):
        g = {"plan": self.plan.handle, "x": self.x.ctypes.data, "n_rows": self.n_rows, "n_targets": self.n_targets,
             "mix_rows": self.mix_rows, "n_slices": self.n_slices, "length": self.T, "t0": 0,
             "k0": 2 if self.inverse else 0,       # synthesis: local slice 0 is not the first, so the halo is written
             "halo": self.halo.ctypes.data if self.inverse else None,
             "scratch": self.scratch, "scratch_bytes": self.scratch_bytes}
        if self.entry.startswith("forward_packed"):
            g["coefs"] = self.coefs[0].ctypes.data
            g["aux"] = self.aux[0].ctypes.data if self.aux else None
        else:
            g["coefs"] = self._views(self.coefs, f.pop("null_coef_bucket", None))
            g["aux"] = self._views(self.aux, f.pop("null_aux_bucket", None)) if self.aux else None
        g.update(f)
        stride = self.T
        if self.entry == "forward_mask_grad":
            return [g["plan"], g["x"], g["n_targets"], g["mix_rows"], stride, g["length"], g["t0"], g["k0"],
                    g["n_slices"], g["coefs"], g["aux"], g["scratch"], g["scratch_bytes"], None]
        if self.entry == "inverse_masked":
            return [g["plan"], g["coefs"], g["aux"], g["n_targets"], g["mix_rows"], g["n_slices"], g["k0"], g["x"],
                    stride, g["length"], g["t0"], g["halo"], g["scratch"], g["scratch_bytes"], None]
        if self.entry == "inverse":
            return [g["plan"], g["coefs"], g["n_rows"], g["n_slices"], g["k0"], g["x"], stride, g["length"], g["t0"],
                    g["halo"], g["scratch"], g["scratch_bytes"], None]
        head = [g["plan"], g["x"], g["n_rows"], stride, g["length"], g["t0"], g["k0"], g["n_slices"], g["coefs"]]
        if self.entry in ("forward_norm", "forward_packed_norm"):
            head.append(g["aux"])
        return head + [g["scratch"], g["scratch_bytes"], None]

    def run(self, lib, **faults):
        rc = getattr(lib, "slicq_" + self.entry)(*self.args(**faults))
        return rc, lib.slicq_last_error().decode()


NULL = "null argument"
BAD_SHAPE = "bad shape"
TOO_SMALL = "scratch buffer too small (see slicq_scratch_bytes)"


def _faults(entry):
    """(fault name, argument overrides, expected code, expected message) for the single-fault calls of `entry`."""
    mg = entry == "forward_mask_grad"
    im = entry == "inverse_masked"
    views = not entry.startswith("forward_packed")
    f = [("plan", {"plan": None}, INVALID, "null argument or bad shape" if mg else NULL),
         ("signal", {"x": None}, INVALID, NULL),
         ("coefs", {"coefs": None}, INVALID, NULL),
         ("n_slices", {"n_slices": 0}, INVALID, BAD_SHAPE),
         ("n_slices<0", {"n_slices": -3}, INVALID, BAD_SHAPE),
         ("length<0", {"length": -1}, INVALID, BAD_SHAPE),
         ("units", {"n_slices": 2 ** 31}, INVALID, "too many (row,slice) units"),
         ("scratch_small", {"scratch_bytes": 16}, SCRATCH, TOO_SMALL),
         ("scratch_null", {"scratch": None}, SCRATCH, TOO_SMALL),
         ("scratch_misaligned", "misaligned", SCRATCH, "scratch buffer must be 16-byte aligned")]
    if mg or im:
        f += [("n_rows", {"mix_rows": 0}, INVALID, "null argument or bad shape" if mg else BAD_SHAPE),
              ("n_targets", {"n_targets": 0}, INVALID, "null argument or bad shape" if mg else "masks / n_targets missing"),
              ("aux", {"aux": None}, INVALID, "null argument or bad shape" if mg else "masks / n_targets missing")]
    else:
        f += [("n_rows", {"n_rows": 0}, INVALID, BAD_SHAPE), ("n_rows<0", {"n_rows": -2}, INVALID, BAD_SHAPE)]
    if entry == "forward_norm":
        f.append(("aux", {"aux": None}, INVALID, "norms missing"))
    if entry == "forward_packed_norm":
        f.append(("aux", {"aux": None}, INVALID, NULL))
    if views:
        f.append(("coef_bucket", {"null_coef_bucket": 2}, INVALID, "null bucket pointer"))
        if entry in ("forward_norm", "forward_mask_grad", "inverse_masked"):
            f.append(("aux_bucket", {"null_aux_bucket": 1}, INVALID, "null mask pointer" if im else "null bucket pointer"))
    return f


@pytest.mark.parametrize("entry", ENTRIES)
def test_argument_errors(lib, tables, monkeypatch, entry):
    plan, adj = _plans(lib, tables, monkeypatch)
    T = 1500
    S = plan.num_slices(T)
    c = Call(entry, plan, adj, tables.sllen // 2, 4, S, T, mix_rows=2)
    assert c.run(lib)[0] == 0
    for name, over, code, msg in _faults(entry):
        if over == "misaligned":
            over = {"scratch": c.scratch + 8, "scratch_bytes": c.scratch_bytes + 8}
        rc, err = c.run(lib, **over)
        assert (rc, err) == (code, msg), (entry, name)
    if entry == "forward_mask_grad":          # a plan that does not compute the adjoint of the synthesis
        rc, err = c.run(lib, plan=plan.handle)
        assert (rc, err) == (INVALID, "the mask gradient needs a plan created with SLICQ_PLAN_ADJOINT_OF_SYNTHESIS")
    if c.inverse:                             # no output samples: the output may be null, the halo is still produced
        c.halo[:] = 0
        assert c.run(lib, x=None, length=0)[0] == 0
        assert np.abs(c.halo).max() > 0


def _run(lib, entry, plans, hop, n_targets, mix_rows, S, T):
    c = Call(entry, *plans, hop, n_targets * mix_rows, S, T, mix_rows=mix_rows, seed=7)
    n0 = lib.slicq_launch_count()
    assert c.run(lib)[0] == 0
    return [o.copy() for o in c.outputs()], lib.slicq_launch_count() - n0


SHARED = ("forward_mask_grad", "inverse_masked")


@pytest.mark.parametrize("entry, n_targets", [(e, 2) for e in ENTRIES] + [(e, 3) for e in SHARED])
def test_split_and_chunks_leave_results_unchanged(lib, tables, monkeypatch, entry, n_targets):
    """2 targets x 2 mixture rows split at row 2; 3 x 2 would split at row 3, not a multiple of the 2 mixture rows, and
    stays whole.  Entries without a shared mixture run 4 rows.  SLICQ_CHUNK_MB=1 gives several chunks."""
    mix_rows = 2 if entry in SHARED else 1
    n_targets = n_targets if entry in SHARED else 4
    T, hop = 32000, tables.sllen // 2
    plain = _plans(lib, tables, monkeypatch)
    S = plain[0].num_slices(T)
    ref, n_plain = _run(lib, entry, plain, hop, n_targets, mix_rows, S, T)
    assert all(np.abs(o).max() > 0 for o in ref)
    split_ok = entry not in SHARED or n_targets == 2
    out, n_split = _run(lib, entry, _plans(lib, tables, monkeypatch, split_units=8), hop, n_targets, mix_rows, S, T)
    assert n_split == (2 * n_plain if split_ok else n_plain)
    assert all(np.array_equal(a, b) for a, b in zip(out, ref))
    out, n_chunk = _run(lib, entry, _plans(lib, tables, monkeypatch, chunk_mb=1), hop, n_targets, mix_rows, S, T)
    assert n_chunk >= 2 * n_plain
    assert all(np.array_equal(a, b) for a, b in zip(out, ref))

"""Drop-in proof (CPU tier, host-emulated kernels).

The reference Separator + Unmix call the transforms only through NSGT_SL -> ComplexNorm -> (model) ->
INSGT_SL, so the drop-in holds when those wrappers return what the reference's do:
* always: the wrappers on the inputs of tests/golden/small_fwdinv.npz against the vectors the UNMODIFIED
  reference produced for them (tests/golden/make_golden.py): coefficients, magnitudes, and the synthesis of
  the reference's own and of perturbed ("masked") coefficients, targets-first as Separator passes them;
* where the reference package is installed (``__graft_entry__.build()`` puts it in baseline/_ref, or
  $SLICQ_REFERENCE names a checkout): the reference Separator + Unmix (seeded random weights -- the shipped
  .pth files are Git-LFS pointers) run once on the reference's transforms and once on these wrappers, and
  the separated stems must agree."""
import contextlib
import io
import os
import sys

import numpy as np
import pytest
import torch

import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SLICQ_REFERENCE", "/root/reference")
if not os.path.isdir(os.path.join(REF, "xumx_slicq_v2")):
    REF = os.path.join(ROOT, "baseline", "_ref")
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "xumx_slicq_v2")),
                                     reason="reference package not installed")


@pytest.fixture(scope="module")
def emu():
    from tests.emu.emu_backend import EmuBackend
    import xumx_slicq_b200.nsgt as nsgt_mod
    old = nsgt_mod._BACKEND
    nsgt_mod._BACKEND = EmuBackend()
    yield
    nsgt_mod._BACKEND = old


def test_dropin_wrappers_match_reference_golden(emu, golden_dir):
    from xumx_slicq_b200 import NSGTBase, make_filterbanks, ComplexNorm
    gold = np.load(os.path.join(golden_dir, "small_fwdinv.npz"))
    buckets = [tuple(int(v) for v in b) for b in gold["buckets"]]
    ref = common.unpack(gold["coefs"], buckets)                      # reference NSGT_sliced: [S, N, F, M] complex64
    with contextlib.redirect_stdout(io.StringIO()):
        base = NSGTBase("bark", 262, 32.9, device="cpu")
    nsgt, insgt = make_filterbanks(base)
    T = common.SMALL_T
    X = nsgt(torch.from_numpy(common.small_input()).view(1, 2, T))   # [1, 2, F, S, M, 2] per bucket
    mags = ComplexNorm()(X)
    assert len(X) == len(mags) == len(ref)
    for Xb, mb, r in zip(X, mags, ref):
        rw = r.transpose(1, 2, 0, 3)[None]                            # the reference wrapper's layout [1, 2, F, S, M]
        scale = np.abs(rw).max()
        assert np.abs(torch.view_as_complex(Xb).numpy() - rw).max() <= 1e-5 * scale
        assert np.abs(mb.numpy() - np.abs(rw)).max() <= 1e-5 * scale
    # targets first, as Separator hands the masked estimates to INSGT_SL: [targets, 1, 2, F, S, M, 2]
    wrap = lambda cs: [torch.view_as_real(torch.from_numpy(np.ascontiguousarray(c.transpose(1, 2, 0, 3))))[None] for c in cs]
    Y = [torch.stack([p, r]) for p, r in zip(wrap(common.perturb(ref)), wrap(ref))]
    y = insgt(Y, T)
    assert y.shape == (2, 1, 2, T)
    np.testing.assert_allclose(y[0, 0].numpy(), gold["y_perturbed"], atol=5e-6)
    np.testing.assert_allclose(y[1, 0].numpy(), gold["y_roundtrip"], atol=5e-6)


@needs_reference
def test_reference_separator_runs_on_the_dropin_transforms(emu):
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            from xumx_slicq_v2.transforms import NSGTBase as RefBase, make_filterbanks as ref_filterbanks, ComplexNorm as RefNorm
            from xumx_slicq_v2.model import Unmix
            from xumx_slicq_v2.separator import Separator
            from xumx_slicq_b200 import NSGTBase, make_filterbanks, ComplexNorm
            rbase = RefBase("bark", 262, 32.9, device="cpu")
            rn, ri = ref_filterbanks(rbase)
            base = NSGTBase("bark", 262, 32.9, device="cpu")
            n, i = make_filterbanks(base)
            torch.manual_seed(0)
            sample = RefNorm()(rbase.predict_input_size(1, 2, 2.0)[0])
            model = Unmix(sample, realtime=True)
            model.freeze()
    finally:
        sys.path.remove(REF)
    sep_ref = Separator(xumx_model=model, encoder=(rn, ri, RefNorm()), device="cpu", quiet=True)
    sep_new = Separator(xumx_model=model, encoder=(n, i, ComplexNorm()), device="cpu", quiet=True)
    torch.manual_seed(1)
    audio = torch.rand(1, 2, 30000) * 2 - 1
    with torch.no_grad():
        out_ref = sep_ref(audio)
        out_new = sep_new(audio)
    assert out_new.shape == out_ref.shape == (4, 1, 2, 30000)
    scale = float(out_ref.abs().max())
    assert float((out_new - out_ref).abs().max()) <= 2e-5 * scale
    # the same shapes come out of the shape probe the reference uses to build the model
    Xs, _ = base.predict_input_size(1, 2, 0.5)
    Xr, _ = rbase.predict_input_size(1, 2, 0.5)
    assert [tuple(a.shape) for a in Xs] == [tuple(b.shape) for b in Xr]

"""Configurations whose bins reach below DC (pos_j < M_j / 2 for a bin j >= 1): the reference's mirrored-bin pass
(nsigtf.py:63-80) adds a conjugated copy of those bins into the kept half spectrum.  Checked here: the synthesis against
the float64 oracle (two such bins that overlap at the same positions), the exact adjoints behind the gradients of
INSGT_SL (transpose of the mirrored-bin pass) and NSGT_SL (overflow below DC folded back), and, on the GPU, that repeated
runs are bitwise equal.  CPU tier: the real kernel sources on the host emulation (tests/emu); GPU tier: -m gpu."""
import numpy as np
import pytest
import torch

import common
from oracle.slicq_oracle import SlicqOracle

CONFIGS = {
    "bark64_30": ("bark", 64, 30.0),     # bins 1 and 2 below DC; bin 2 overlaps bin 0 there (overflow entries below DC)
    "bark20_60": ("bark", 20, 60.0),     # bins 1 and 2 below DC, slice length 1328
    "mel48_30": ("mel", 48, 30.0),       # bins 1 and 2 below DC
    "tinymel": ("mel", 32, 115.5),       # one bin below DC
    "bark30_150": ("bark", 30, 150.0),   # one bin below DC
}
ORACLE_CONFIGS = ["bark64_30", "bark20_60"]      # the oracle restates the Bark scale
TOL_IDENTITY = 2e-5
TOL_DIRECTIONAL = 2e-4


def _below_dc(nsg):
    """Per bucket: bool [F_b], True for the bins j >= 1 (below Nyquist) whose window reaches below DC."""
    t = nsg.tables
    out = []
    for (first, nb, M) in t.buckets:
        js = np.arange(first, first + nb)
        out.append(torch.from_numpy((js >= 1) & (js <= t.n_bins - 2) & (t.bin_pos[js] < M // 2)))
    return out


def _on_bins(X, sel):
    """Zero every bin of the wrapper tensors [..., F, S, M, 2] except the selected ones."""
    return [Xb * s.to(Xb.device, Xb.dtype).view(-1, 1, 1, 1) for Xb, s in zip(X, sel)]


def _inner(a, b):
    return float(sum((x.double() * y.double()).sum() for x, y in zip(a, b)))


def _check(lhs, rhs, tol):
    assert abs(lhs - rhs) <= tol * max(abs(lhs), 1.0), (lhs, rhs, abs(lhs - rhs) / max(abs(lhs), 1e-300))


def inverse_adjoint(base, dev, T, seed=0):
    """INSGT_SL: <S c, g> == <c, S^T g> (a) for all coefficients and (b) with c non-zero only on the bins below DC,
    a directional derivative, and an SDR-style loss that decreases along the negative gradient.  Returns the gradients."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, insgt = make_filterbanks(base)
    sel = _below_dc(base.nsgt)
    assert any(bool(s.any()) for s in sel)
    gen = torch.Generator().manual_seed(seed)
    x = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    g = torch.randn(1, 2, T, generator=gen).to(dev)
    X = nsgt(x)
    R = _on_bins([torch.randn(Xb.shape, generator=gen).to(dev) for Xb in X], sel)
    grads = []
    for C0 in (X, R):
        C = [c.detach().clone().requires_grad_(True) for c in C0]
        y = insgt(C, T)
        assert y.requires_grad
        (y * g).sum().backward()
        _check(_inner([y.detach()], [g]), _inner([c.detach() for c in C], [c.grad for c in C]), TOL_IDENTITY)
        grads.append([c.grad for c in C])
    # directional derivative along a random direction d: d/de <S(c + e d), g> = <d, S^T g>
    d = [torch.randn(Xb.shape, generator=gen).to(dev) for Xb in X]
    with torch.no_grad():
        fd = (_inner([insgt([a + 0.5 * b for a, b in zip(X, d)], T)], [g]) - _inner([insgt(X, T)], [g])) / 0.5
    _check(fd, _inner(d, grads[0]), TOL_DIRECTIONAL)
    # an SDR-style loss decreases along the negative gradient, also when only the bins below DC move; the loss is
    # quadratic, so the step that minimises it along -G is |G|^2 / (2 mean((S G)^2))
    target = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    C = [c.detach().clone().requires_grad_(True) for c in X]
    loss0 = ((insgt(C, T) - target) ** 2).mean()
    loss0.backward()
    for G in ([c.grad for c in C], _on_bins([c.grad for c in C], sel)):
        with torch.no_grad():
            step = _inner(G, G) / (2.0 * float((insgt(G, T) ** 2).mean()))
            loss1 = ((insgt([c - step * gc for c, gc in zip(C, G)], T) - target) ** 2).mean()
        assert float(loss1) < float(loss0.detach()), (float(loss0.detach()), float(loss1))
    return grads


def forward_adjoint(base, dev, T, seed=1):
    """NSGT_SL: <A x, d> == <x, A^T d> (a) for all coefficients and (b) with d non-zero only on the bins below DC, and
    a directional derivative.  Returns the gradients."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, _ = make_filterbanks(base)
    sel = _below_dc(base.nsgt)
    gen = torch.Generator().manual_seed(seed)
    x0 = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    with torch.no_grad():
        shapes = [Xb.shape for Xb in nsgt(x0)]
    D = [torch.randn(s, generator=gen).to(dev) for s in shapes]
    grads = []
    for d in (D, _on_bins(D, sel)):
        x = x0.clone().requires_grad_(True)
        X = nsgt(x)
        assert all(Xb.requires_grad for Xb in X)
        sum((Xb * db).sum() for Xb, db in zip(X, d)).backward()
        _check(_inner([Xb.detach() for Xb in X], d), _inner([x.detach()], [x.grad]), TOL_IDENTITY)
        grads.append(x.grad)
    e = torch.randn(x0.shape, generator=gen).to(dev)
    with torch.no_grad():
        fd = (_inner(nsgt(x0 + 0.25 * e), D) - _inner(nsgt(x0), D)) / 0.25
    _check(fd, _inner([e], [grads[0]]), TOL_DIRECTIONAL)
    return grads


def synthesis_vs_oracle(base, orc, dev, T, seed=3):
    """Synthesis of perturbed (model-output-like) coefficients, plain and fused with masks, against the float64 oracle.
    Returns the two outputs."""
    nsg = base.nsgt
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    P = common.perturb([o.astype(np.complex64) for o in orc.forward(x.astype(np.float64))])      # [S, N, F, M]
    C = [torch.from_numpy(np.ascontiguousarray(p.transpose(1, 2, 0, 3))).to(dev) for p in P]   # [N, F, S, M]
    y_ref = orc.backward([p.astype(np.complex128) for p in P], T)
    y = nsg.backward_rows(C, T)
    assert np.abs(y.cpu().numpy() - y_ref).max() < 5e-6, float(np.abs(y.cpu().numpy() - y_ref).max())
    rs = np.random.RandomState(seed + 1)
    masks = [rs.rand(2, *c.shape).astype(np.float32) for c in C]                                # [targets, N, F, S, M]
    ym = nsg.backward_rows_masked(C, [torch.from_numpy(m).to(dev) for m in masks], T)
    Y = [np.concatenate([p * m[t].transpose(2, 0, 1, 3) for t in range(2)], axis=1) for p, m in zip(P, masks)]
    ym_ref = orc.backward([v.astype(np.complex128) for v in Y], T)
    assert ym.shape == ym_ref.shape == (4, T)
    assert np.abs(ym.cpu().numpy() - ym_ref).max() < 5e-6, float(np.abs(ym.cpu().numpy() - ym_ref).max())
    return y, ym


def _base(cfg, dev):
    from xumx_slicq_b200 import NSGTBase
    name, fbins, fmin = CONFIGS[cfg]
    return NSGTBase(name, fbins, fmin, device=dev)


def _oracle(cfg):
    _, fbins, fmin = CONFIGS[cfg]
    return SlicqOracle(scale="bark", fbins=fbins, fmin=fmin)


# ------------------------------------------------------------------------------------------------ CPU tier (emulation)
@pytest.fixture
def emu():
    """The emulation backend for one test (the GPU tests of this module run on the product backend)."""
    from tests.emu.emu_backend import EmuBackend
    import xumx_slicq_b200.nsgt as nsgt_mod
    old = nsgt_mod._BACKEND
    nsgt_mod._BACKEND = EmuBackend()
    yield nsgt_mod._BACKEND
    nsgt_mod._BACKEND = old


@pytest.fixture(scope="module")
def emu_bases():
    cache = {}

    def get(cfg):
        if cfg not in cache:
            cache[cfg] = _base(cfg, "cpu")
        return cache[cfg]
    return get


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_inverse_adjoint_emu(emu, emu_bases, cfg):
    b = emu_bases(cfg)
    inverse_adjoint(b, torch.device("cpu"), 2 * b.sllen + 123)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_forward_adjoint_emu(emu, emu_bases, cfg):
    b = emu_bases(cfg)
    forward_adjoint(b, torch.device("cpu"), 2 * b.sllen + 123)


@pytest.mark.parametrize("cfg", ORACLE_CONFIGS)
def test_synthesis_vs_oracle_emu(emu, emu_bases, cfg):
    b = emu_bases(cfg)
    synthesis_vs_oracle(b, _oracle(cfg), torch.device("cpu"), 3 * b.sllen + 77)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tier needs CUDA"
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_adjoints_gpu_bitwise_repeatable(dev, cfg):
    b = _base(cfg, dev)
    T = 6 * b.sllen + 123
    gi1, gi2 = inverse_adjoint(b, dev, T), inverse_adjoint(b, dev, T)
    gf1, gf2 = forward_adjoint(b, dev, T), forward_adjoint(b, dev, T)
    for a, c in zip(gi1, gi2):
        assert all(torch.equal(u, v) for u, v in zip(a, c))
    assert all(torch.equal(u, v) for u, v in zip(gf1, gf2))


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ORACLE_CONFIGS)
def test_synthesis_vs_oracle_gpu_bitwise_repeatable(dev, cfg):
    """The mirrored-bin pass adds two bins at the same plane-0 positions here: a lost update would show against the
    oracle, and a nondeterministic order between two runs."""
    b = _base(cfg, dev)
    orc = _oracle(cfg)
    T = 40 * b.sllen + 77
    y1, ym1 = synthesis_vs_oracle(b, orc, dev, T)
    y2, ym2 = synthesis_vs_oracle(b, orc, dev, T)
    assert torch.equal(y1, y2) and torch.equal(ym1, ym2)


@pytest.mark.gpu
def test_bark64_30s_stereo_gpu(dev):
    """A 30 s stereo signal on Bark(64, 30 Hz): coefficients and synthesis against the oracle, both adjoints."""
    b = _base("bark64_30", dev)
    orc = _oracle("bark64_30")
    T = 1323000
    x = np.random.RandomState(0).rand(2, T).astype(np.float32) * 2 - 1
    C = b.nsgt.forward_rows(torch.from_numpy(x).to(dev))
    O = orc.forward(x.astype(np.float64))
    worst = max(float(np.abs(c.permute(2, 0, 1, 3).cpu().numpy() - o).max() / np.abs(o).max()) for c, o in zip(C, O))
    assert worst < 1e-5, worst
    del C, O
    synthesis_vs_oracle(b, orc, dev, T)
    inverse_adjoint(b, dev, T)
    forward_adjoint(b, dev, T)

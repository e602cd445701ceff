"""Gradients through the fused masked synthesis INSGT_SL.forward_masked (realtime model: output row t * N + n is
y = S(m_{t,n} * X_n)).  dL/dm = Re(conj(X) * S^T g) comes from the epilogue of the adjoint-of-synthesis analysis kernels
(and of the mirrored-bin adjoint for bins that reach below DC); dL/dX = sum_t m_t * S^T g.  Checked: adjoint identities
for masks and mixture, the fused mask gradient against Re(conj(X) * synthesis_adjoint_rows(g)), inputs and layouts, an
SGD step, and on the GPU bitwise repeatability and the row-group split of large calls.
CPU tier: the real kernel sources on the host emulation (tests/emu); GPU tier: -m gpu."""
import numpy as np
import pytest
import torch

CONFIGS = {
    "bark262": ("bark", 262, 32.9),      # tuned L = 18060 slice kernels; all three per-bin transform families
    "bark100_50": ("bark", 100, 50.0),   # generic slice kernels, L = 6884 = 4 * 1721
    "bark64_30": ("bark", 64, 30.0),     # bins 1 and 2 below DC
    "tinymel": ("mel", 32, 115.5),       # bin 1 below DC
}
BELOW_DC = ["bark64_30", "tinymel"]
TOL_IDENTITY = 2e-5


def _base(cfg, dev):
    from xumx_slicq_b200 import NSGTBase
    name, fbins, fmin = CONFIGS[cfg]
    return NSGTBase(name, fbins, fmin, device=dev)


def _below_dc(nsg):
    """Per bucket: bool [F_b], True for the bins j >= 1 (below Nyquist) whose window reaches below DC."""
    t = nsg.tables
    out = []
    for (first, nb, M) in t.buckets:
        js = np.arange(first, first + nb)
        out.append(torch.from_numpy((js >= 1) & (js <= t.n_bins - 2) & (t.bin_pos[js] < M // 2)))
    return out


def _inner(a, b):
    return float(sum((x.double() * y.double()).sum() for x, y in zip(a, b)))


def _check(lhs, rhs, tol):
    assert abs(lhs - rhs) <= tol * max(abs(lhs), 1.0), (lhs, rhs, abs(lhs - rhs) / max(abs(lhs), 1e-300))


def _problem(base, dev, T, n_targets=2, batch=1, seed=0):
    """Mixture transform X (list of [B, C, F, S, M, 2]), masks [targets, B, C, F, S, M] in (0, 1), output gradient g."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, insgt = make_filterbanks(base)
    gen = torch.Generator().manual_seed(seed)
    x = (torch.rand(batch, 2, T, generator=gen) * 2 - 1).to(dev)
    with torch.no_grad():
        X = nsgt(x)
    masks = [torch.rand((n_targets,) + tuple(Xb.shape[:-1]), generator=gen).to(dev) for Xb in X]
    g = torch.randn(n_targets, batch, 2, T, generator=gen).to(dev)
    return insgt, X, masks, g, gen


def _grads(insgt, X, masks, g, T, x_grad=False, m_grad=True):
    Xg = [Xb.detach().clone().requires_grad_(x_grad) for Xb in X]
    Mg = [m.detach().clone().requires_grad_(m_grad) for m in masks]
    y = insgt.forward_masked(Xg, Mg, T)
    assert y.requires_grad
    (y * g).sum().backward()
    return y.detach(), [Xb.grad for Xb in Xg], [m.grad for m in Mg]


def mask_identity(base, dev, T, below_dc_only=False, n_targets=2, seed=0):
    """<S((m + dM) X) - S(m X), g> == sum dM * dL/dm, dM optionally non-zero only on the bins below DC."""
    insgt, X, masks, g, gen = _problem(base, dev, T, n_targets=n_targets, seed=seed)
    _, _, gm = _grads(insgt, X, masks, g, T)
    assert all(a.shape == m.shape and a.dtype == m.dtype for a, m in zip(gm, masks))
    dM = [torch.randn(m.shape, generator=gen).to(dev) for m in masks]
    if below_dc_only:
        sel = _below_dc(base.nsgt)
        assert any(bool(s.any()) for s in sel)
        dM = [d * s.to(dev, d.dtype).view(-1, 1, 1) for d, s in zip(dM, sel)]
    with torch.no_grad():
        y1 = insgt.forward_masked(X, [m + d for m, d in zip(masks, dM)], T)
        y0 = insgt.forward_masked(X, masks, T)
    _check(_inner([y1 - y0], [g]), _inner(dM, gm), TOL_IDENTITY)
    return gm


def fused_vs_unfused(base, dev, T, n_targets=2, batch=1, seed=2):
    """The fused mask gradient == Re(conj(X) * synthesis_adjoint_rows(g)) within 1e-6 of each bucket's maximum, and
    the fused path never materialises S^T g."""
    from xumx_slicq_b200.nsgt import NSGT_sliced
    insgt, X, masks, g, _ = _problem(base, dev, T, n_targets=n_targets, batch=batch, seed=seed)
    nsg = base.nsgt
    calls = []
    orig = NSGT_sliced.synthesis_adjoint_rows

    def spy(self, *a, **k):
        calls.append(1)
        return orig(self, *a, **k)
    NSGT_sliced.synthesis_adjoint_rows = spy
    try:
        _, _, gm = _grads(insgt, X, masks, g, T)
        assert not calls, "masks-only backward must not compute the complex adjoint"
    finally:
        NSGT_sliced.synthesis_adjoint_rows = orig
    rows = n_targets * batch * 2
    S = X[0].shape[-3]
    cadj = nsg.synthesis_adjoint_rows(g.reshape(rows, T), S)
    for a, c, Xb in zip(gm, cadj, X):
        xc = torch.view_as_complex(Xb.contiguous()).reshape((-1,) + tuple(Xb.shape[-4:-1]))
        ref = torch.real(xc.conj() * c.view((n_targets, -1) + tuple(c.shape[1:]))).reshape(a.shape)
        assert float((a - ref).abs().max()) <= 1e-6 * float(ref.abs().max()), float((a - ref).abs().max())
    return gm


def x_identity(base, dev, T, seed=4):
    """<S(m X), g> == <X, dL/dX> (X alone, and X with the masks, where also == <m, dL/dm>); inputs unchanged."""
    insgt, X, masks, g, _ = _problem(base, dev, T, seed=seed)
    X0, M0 = [Xb.clone() for Xb in X], [m.clone() for m in masks]
    for m_grad in (False, True):
        y, gx, gm = _grads(insgt, X, masks, g, T, x_grad=True, m_grad=m_grad)
        assert all(a.shape == Xb.shape and a.dtype == Xb.dtype for a, Xb in zip(gx, X))
        lhs = _inner([y], [g])
        _check(lhs, _inner(X, gx), TOL_IDENTITY)
        if m_grad:
            _check(lhs, _inner(masks, gm), TOL_IDENTITY)
        else:
            assert all(a is None for a in gm)
    assert all(torch.equal(a, b) for a, b in zip(X, X0)) and all(torch.equal(a, b) for a, b in zip(masks, M0))


# ------------------------------------------------------------------------------------------------ CPU tier (emulation)
@pytest.fixture(scope="module")
def emu(request):
    from tests.emu.emu_backend import EmuBackend
    import xumx_slicq_b200.nsgt as nsgt_mod
    old = nsgt_mod._BACKEND
    nsgt_mod._BACKEND = EmuBackend()
    yield nsgt_mod._BACKEND
    nsgt_mod._BACKEND = old


@pytest.fixture(scope="module")
def emu_bases(emu):
    cache = {}

    def get(cfg):
        if cfg not in cache:
            cache[cfg] = _base(cfg, "cpu")
        return cache[cfg]
    return get


def _emu_T(b):
    return b.sllen + b.sllen // 2 + 123


CPU = torch.device("cpu")


def test_forward_masked_tracks_gradients(emu_bases):
    b = emu_bases("tinymel")
    T = _emu_T(b)
    insgt, X, masks, g, _ = _problem(b, CPU, T)
    y_ref = insgt.forward_masked(X, masks, T)
    assert not y_ref.requires_grad
    for x_grad, m_grad in ((False, True), (True, False), (True, True)):
        Xg = [Xb.clone().requires_grad_(x_grad) for Xb in X]
        Mg = [m.clone().requires_grad_(m_grad) for m in masks]
        y = insgt.forward_masked(Xg, Mg, T)
        assert y.requires_grad and torch.equal(y.detach(), y_ref)
        with torch.no_grad():
            assert not insgt.forward_masked(Xg, Mg, T).requires_grad


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_mask_identity_emu(emu_bases, cfg):
    b = emu_bases(cfg)
    mask_identity(b, CPU, _emu_T(b))


@pytest.mark.parametrize("cfg", BELOW_DC)
def test_mask_identity_bins_below_dc_emu(emu_bases, cfg):
    """Only the bins below DC move: their gradient includes the transpose of the mirrored-bin pass."""
    b = emu_bases(cfg)
    mask_identity(b, CPU, _emu_T(b), below_dc_only=True)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_fused_vs_unfused_emu(emu_bases, cfg):
    b = emu_bases(cfg)
    fused_vs_unfused(b, CPU, _emu_T(b))


@pytest.mark.parametrize("cfg", ["bark262", "tinymel"])
def test_x_identity_emu(emu_bases, cfg):
    b = emu_bases(cfg)
    x_identity(b, CPU, _emu_T(b))


@pytest.mark.parametrize("n_targets", [1, 4])
def test_targets_and_permuted_layouts_emu(emu_bases, n_targets):
    """1 and 4 targets; reference-style permuted (non-contiguous) X and masks give the same gradients."""
    b = emu_bases("bark64_30")
    T = _emu_T(b)
    insgt, X, masks, g, _ = _problem(b, CPU, T, n_targets=n_targets, seed=6)
    _, gx, gm = _grads(insgt, X, masks, g, T, x_grad=True)
    Xp = [Xb.permute(0, 1, 3, 2, 4, 5).contiguous().permute(0, 1, 3, 2, 4, 5) for Xb in X]
    Mp = [m.permute(0, 1, 2, 4, 3, 5).contiguous().permute(0, 1, 2, 4, 3, 5) for m in masks]
    assert not Xp[1].is_contiguous() and not Mp[1].is_contiguous()
    _, gxp, gmp = _grads(insgt, Xp, Mp, g, T, x_grad=True)
    assert all(torch.equal(a, c) for a, c in zip(gx, gxp))
    # with X requiring grad the mask gradient is a torch product, whose rounding may depend on the layout
    for a, c in zip(gmp, gm):
        assert float((a - c).abs().max()) <= 1e-6 * float(c.abs().max())
    _, _, gf = _grads(insgt, X, masks, g, T)                      # masks only: the fused path
    _, _, gfp = _grads(insgt, Xp, Mp, g, T)
    assert all(torch.equal(a, c) for a, c in zip(gf, gfp))
    for a, c in zip(gf, gm):
        assert float((a - c).abs().max()) <= 1e-6 * float(c.abs().max())


def test_bf16_masks_emu(emu_bases):
    """Masks in bf16 (autocast): the gradient comes back in bf16, equal to the fp32 gradient at the same mask values."""
    b = emu_bases("tinymel")
    T = _emu_T(b)
    insgt, X, masks, g, _ = _problem(b, CPU, T, seed=8)
    mb = [m.to(torch.bfloat16) for m in masks]
    _, _, gb = _grads(insgt, X, mb, g, T)
    _, _, gf = _grads(insgt, X, [m.float() for m in mb], g, T)
    assert all(a.dtype == torch.bfloat16 and a.shape == m.shape for a, m in zip(gb, mb))
    assert all(torch.equal(a, c.to(torch.bfloat16)) for a, c in zip(gb, gf))


def test_sgd_step_lowers_sdr_loss_emu(emu_bases):
    """Masks as nn.Parameter under an SDR-style loss through forward_masked: one SGD step lowers the loss."""
    b = emu_bases("bark64_30")
    T = _emu_T(b)
    insgt, X, masks, _, _ = _problem(b, CPU, T, seed=10)
    with torch.no_grad():
        target = insgt.forward_masked(X, masks, T)
    params = [torch.nn.Parameter(torch.full_like(m, 0.5)) for m in masks]

    def loss_fn():
        y = insgt.forward_masked(X, list(params), T)
        num = (target ** 2).sum(-1)
        den = ((target - y) ** 2).sum(-1)
        return -(10.0 * torch.log10(num / den)).mean()
    loss0 = loss_fn()
    loss0.backward()
    gmax = max(float(p.grad.abs().max()) for p in params)
    assert gmax > 0
    opt = torch.optim.SGD(params, lr=1e-2 / gmax)
    opt.step()
    with torch.no_grad():
        loss1 = loss_fn()
    assert float(loss1) < float(loss0.detach()), (float(loss0), float(loss1))


def split_check(base, dev, T, n_targets, batch, split, lib):
    """Fused mask gradient of a call that does (or, when a group boundary is not a multiple of the mixture rows, does
    not) split into two row groups, against the unfused path; the split shows in the launch count."""
    insgt, X, masks, g, _ = _problem(base, dev, T, n_targets=n_targets, batch=batch, seed=12)
    nsg = base.nsgt
    rows = n_targets * batch * 2
    S = X[0].shape[-3]
    xs, _, _ = insgt._masked_inputs(X, masks)
    g2 = g.reshape(rows, T)
    nsg.mask_grad_rows(g2, xs, n_targets)                       # plan creation and first-call set-up
    n0 = lib.slicq_launch_count()
    gm = nsg.mask_grad_rows(g2, xs, n_targets)
    launches = lib.slicq_launch_count() - n0
    per_group = 3 if any(bool(s.any()) for s in _below_dc(nsg)) else 2     # slice, bins [, mirrored-bin adjoint]
    assert launches == (2 * per_group if split else per_group), launches
    cadj = nsg.synthesis_adjoint_rows(g2, S)
    for a, c, x in zip(gm, cadj, xs):
        ref = torch.real(x.conj() * c.view((n_targets, -1) + tuple(c.shape[1:]))).reshape(a.shape)
        assert float((a - ref).abs().max()) <= 1e-6 * float(ref.abs().max())


@pytest.mark.parametrize("n_targets, batch, split", [(2, 1, True), (3, 1, False)])
def test_row_group_split_emu(monkeypatch, emu, n_targets, batch, split):
    """2 targets x 2 rows split at row 2; 3 targets x 2 rows would split at row 3, not a multiple of the 2 mixture rows,
    and stays whole.  The split threshold is lowered for the small emulated sizes."""
    monkeypatch.setenv("SLICQ_SPLIT_UNITS", "8")       # read when the (adjoint) plan is created
    b = _base("tinymel", "cpu")
    split_check(b, CPU, _emu_T(b), n_targets, batch, split, emu.lib())


def test_mask_grad_needs_the_adjoint_plan(emu_bases):
    """slicq_forward_mask_grad refuses a plan that does not compute the adjoint of the synthesis."""
    b = emu_bases("tinymel")
    nsg = b.nsgt
    plan = nsg.plan(torch.device("cpu"))
    T = _emu_T(b)
    S = nsg.n_slices(T)
    g = torch.zeros(2, T)
    xs = nsg.alloc_coefficients(1, S, "cpu")[1]
    gs = nsg.alloc_norms(2, S, "cpu")[1]
    nbytes = plan.scratch_bytes(2, S, False)
    scratch = torch.empty(nbytes, dtype=torch.uint8)
    with pytest.raises(ValueError, match="ADJOINT_OF_SYNTHESIS"):
        plan.forward_mask_grad(g.data_ptr(), 2, 1, T, T, 0, 0, S, [nsg._view_of(c) for c in xs],
                               [(o.data_ptr(), o.stride(0), o.stride(1), o.stride(2)) for o in gs],
                               scratch.data_ptr(), nbytes, 0)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tier needs CUDA"
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_mask_and_x_gradients_gpu(dev, cfg):
    b = _base(cfg, dev)
    T = 6 * b.sllen + 123
    mask_identity(b, dev, T)
    if cfg in BELOW_DC:
        mask_identity(b, dev, T, below_dc_only=True)
    fused_vs_unfused(b, dev, T)
    x_identity(b, dev, T)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["bark262", "bark64_30"])
def test_backward_gpu_bitwise_repeatable(dev, cfg):
    b = _base(cfg, dev)
    T = 6 * b.sllen + 123
    insgt, X, masks, g, _ = _problem(b, dev, T, n_targets=4)
    for x_grad in (False, True):
        _, gx1, gm1 = _grads(insgt, X, masks, g, T, x_grad=x_grad)
        _, gx2, gm2 = _grads(insgt, X, masks, g, T, x_grad=x_grad)
        assert all(torch.equal(a, c) for a, c in zip(gm1, gm2))
        if x_grad:
            assert all(torch.equal(a, c) for a, c in zip(gx1, gx2))


@pytest.mark.gpu
@pytest.mark.parametrize("n_targets, batch, split", [(4, 1, True), (3, 2, False)])
def test_30s_row_group_split_gpu(dev, n_targets, batch, split):
    """Bark-262, 30 s stereo: 4 targets x 2 rows = 1184 units split into two row groups; 3 targets x 4 rows has its
    halfway boundary at row 6, not a multiple of the 4 mixture rows, and stays whole.  Both agree with the unfused path."""
    from xumx_slicq_b200 import _cabi
    split_check(_base("bark262", dev), dev, 1323000, n_targets, batch, split, _cabi.load())

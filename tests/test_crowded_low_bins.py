"""Bark and mel filterbanks whose lowest bins crowd together near DC: the lowest bins all get the minimum window length
and sit only a few positions apart, so bins share a position, five or more windows overlap at one position, or a bin of
a two-pass / prime transform sends more than its first run of outputs to its overflow slot.  Checked here: which
configurations slicq_plan_create accepts, that every configuration accepted before gets the same synthesis layout,
and the transforms, their adjoints and the masked synthesis on one configuration of each kind, against the float64
oracle.  CPU tier: the real kernel sources on the host emulation (tests/emu); GPU tier: -m gpu."""
import contextlib
import ctypes as C
import io
import os
import sys

import numpy as np
import pytest
import torch

import common
import oracle.slicq_oracle as slicq_oracle
from oracle.slicq_oracle import SlicqOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "xumx_slicq_b200", "csrc"))
from gen_codelets import choose_split   # noqa: E402

CONFIGS = {
    "bark20_30": ("bark", 20, 30.0),     # bins 0 and 1 share position 0; five windows overlap near DC
    "bark24_329": ("bark", 24, 32.9),    # bins 0-4 at 0, 2, 6, 10, 14: five windows over positions 6 and 7
    "bark9_100": ("bark", 9, 100.0),     # overflow over several runs of a two-pass / prime transform
    "mel40_10": ("mel", 40, 10.0),       # bins share a position
}
TOL_IDENTITY = 2e-5
FS = 44100.0

# the grid of the acceptance sweep: Bark and mel, fbins 6 .. 63 and 64 .. 388 in steps of 12, 17 values of fmin
FBINS = list(range(6, 64)) + list(range(64, 400, 12))
FMINS = (10., 12., 15., 20., 25., 30., 32.9, 40., 50., 60., 70., 80., 100., 115.5, 130., 150., 200.)


def _design(scale, fbins, fmin):
    from xumx_slicq_b200.plan import design, make_scale
    with contextlib.redirect_stdout(io.StringIO()):
        scl = make_scale(scale, fmin, FS / 2, fbins)
    sl, tr = scl.suggested_sllen_trlen(FS)
    return design(scl, FS, sl, tr)


def _first_run(M):
    k, a, b = choose_split(int(M))
    return M if k == 1 else (a if k == 2 else b)


# ------------------------------------------------------------------------------------------------ layout rules
def overflow_counts(M, pos):
    """ov_j: the leading positions of bin j that an earlier bin of its plane (j mod 2) reaches, clamped to [0, M_j]."""
    ov, end = [0] * len(M), [None, None]
    for j in range(len(M)):
        lo = int(pos[j]) - int(M[j]) // 2
        e = end[j & 1]
        ov[j] = 0 if e is None else min(int(M[j]), max(0, e - lo))
        end[j & 1] = lo + int(M[j]) if e is None else max(e, lo + int(M[j]))
    return ov


def overflow_slots(M, pos, N2, fold):
    """Per target position, the overflow slots (bin, m) in bin order: direct ones, and (fold) those below DC / above
    Nyquist folded back."""
    ov = overflow_counts(M, pos)
    direct, folded = {}, {}
    for j in range(len(M)):
        for m in range(ov[j]):
            f = int(pos[j]) - int(M[j]) // 2 + m
            out = f < 0 or f > N2
            if out and not fold:
                continue
            f = -f if f < 0 else (2 * N2 - f if f > N2 else f)
            (folded if out else direct).setdefault(f, []).append((j, m))
    return ov, direct, folded


def parent_layout(M, pos, N2, fold):
    """The layout rules before bins could crowd (at most 4 bins per position, overflow against bin j - 2 only, at most
    two entries per position): ov and the entries {f, slot0, slot1 or -1, fold}, or None where those rules reject."""
    J = len(M)
    ov = [0] * J
    for j in range(J):
        lo = int(pos[j]) - int(M[j]) // 2
        if j and pos[j] <= pos[j - 1]:
            return None
        if j >= 2:
            ov[j] = max(0, int(pos[j - 2]) + int(M[j - 2]) // 2 - lo)
        if ov[j] > M[j] or ov[j] & 1:
            return None
        if j >= 4 and int(pos[j - 4]) + int(M[j - 4]) // 2 > lo:
            return None
        if _first_run(M[j]) < M[j] and ov[j] > _first_run(M[j]):
            return None
    _, direct, folded = overflow_slots(M, pos, N2, fold)
    if any(len(v) > 2 for v in list(direct.values()) + list(folded.values())):
        return None
    return ov, direct, folded


class _Layout:
    """slicq_plan_create's overflow layout, read through the emulation build's test hook."""

    def __init__(self, tables, flags=0):
        from tests.emu.emu_backend import EmuBackend
        from xumx_slicq_b200 import _cabi
        from xumx_slicq_b200.nsgt import _AdjointAnalysisTables
        lib = EmuBackend().lib()
        t = _AdjointAnalysisTables(tables) if flags == 2 else tables
        self.plan = _cabi.Plan(t, lib)
        ov, ex = C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)()
        n_ex, rounds, multi = C.c_int(), C.c_int(), C.c_int()
        fn = lib.slicq_emu_plan_layout
        fn.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        assert fn(self.plan.handle, C.byref(ov), C.byref(ex), C.byref(n_ex), C.byref(rounds), C.byref(multi)) == 0
        J = int(tables.n_bins)
        self.ov = [ov[j] for j in range(J)]
        self.ex = [tuple(ex[4 * i + c] for c in range(4)) for i in range(n_ex.value)]
        self.rounds, self.multi_run = rounds.value, bool(multi.value)


def _ovoff(M, ov):
    """Offset of bin j's overflow slot relative to the overflow area (slots in bin order)."""
    return np.concatenate([[0], np.cumsum(ov)[:-1]]).astype(int)


def _expected_entries(M, ov, direct, folded):
    """Entries {f, slot0, slot1 or -1, fold | round << 1} with slots relative to the overflow area, ordered by
    (fold, round, f); the r-th pair of slots of a position is round r."""
    off = _ovoff(M, ov)
    out = []
    for w, slots in ((0, direct), (1, folded)):
        rounds = max([(len(v) + 1) // 2 for v in slots.values()] + [0])
        for r in range(rounds):
            for f in sorted(slots):
                s = [int(off[j] + m) for j, m in slots[f]]
                if len(s) > 2 * r:
                    out.append((f, s[2 * r], s[2 * r + 1] if len(s) > 2 * r + 1 else -1, w | (r << 1)))
    return out


def _relative(ex, base):
    return [(f, a - base, b - base if b >= 0 else -1, w) for f, a, b, w in ex]


def _ovf_base(t):
    """2 * pl_len: start of the overflow area in a row of T (slicq_plan_create)."""
    M, pos = np.asarray(t.bin_M), np.asarray(t.bin_pos)
    pad_l = max(max(0, int(m) // 2 - int(p)) for m, p in zip(M, pos))
    pad_r = max(max(0, int(p) + int(m) // 2 - 1 - t.sllen // 2) for m, p in zip(M, pos))
    pad_l, pad_r = (pad_l + 1) & ~1, (pad_r + 1) & ~1
    return 2 * ((pad_l + t.sllen // 2 + 2 + max(pad_r, 2) + 1) & ~1)


# ------------------------------------------------------------------------------------------------ plan tests (CPU)
@pytest.fixture(scope="module")
def grid_tables():
    return {(s, fb, fm): _design(s, fb, fm) for s in ("bark", "mel") for fb in FBINS for fm in FMINS}


def test_acceptance_sweep(grid_tables):
    """Every Bark / mel configuration of the grid plans, except the six- and seven-bin filterbanks whose bins reach too
    far beyond DC / Nyquist."""
    from tests.emu.emu_backend import EmuBackend
    from xumx_slicq_b200 import _cabi
    lib = EmuBackend().lib()
    refused, wrong = [], []
    for key, t in grid_tables.items():
        try:
            _cabi.Plan(t, lib).close()
        except ValueError as e:
            refused.append(key)
            if "too far beyond DC / Nyquist" not in str(e) or key[1] > 7:
                wrong.append((key, str(e)))
    assert not wrong, wrong[:10]
    assert len(grid_tables) - len(refused) >= 2882, len(refused)


@pytest.mark.parametrize("key", [("bark", 262, 32.9), ("bark", 64, 30.0)])
def test_existing_configurations_still_plan(key):
    lay = _Layout(_design(*key))
    assert lay.rounds <= 1 and not lay.multi_run


@pytest.mark.parametrize("flags", [0, 2])
def test_layout_unchanged_where_parent_rules_accept(grid_tables, flags):
    """Where the earlier rules accepted a configuration, the plan derives the same ov, the same entries in the same
    order and a single round (flags 2: the adjoint-of-analysis plan, whose entries below DC / above Nyquist fold back)."""
    n = 0
    for key, t in grid_tables.items():
        M, pos, N2 = np.asarray(t.bin_M), np.asarray(t.bin_pos), t.sllen // 2
        old = parent_layout(M, pos, N2, flags == 2)
        pad = max(max(0, int(m) // 2 - int(p)) for m, p in zip(M, pos))
        if old is None or (pad + 1) // 2 * 2 > N2 // 2:
            continue
        ov, direct, folded = old
        lay = _Layout(t, flags)
        assert lay.ov == ov, key
        assert lay.rounds <= 1 and not lay.multi_run, key
        # the parent's entries: {f, slot0, slot1 or -1, fold}, direct by f, then folded by f
        off = _ovoff(M, ov)
        want = []
        for w, slots in ((0, direct), (1, folded)):
            for f in sorted(slots):
                s = [int(off[j] + m) for j, m in slots[f]]
                want.append((f, s[0], s[1] if len(s) > 1 else -1, w))
        assert _relative(lay.ex, _ovf_base(t)) == want, key
        n += 1
    assert n >= 2000, n


@pytest.mark.parametrize("cfg", list(CONFIGS))
@pytest.mark.parametrize("flags", [0, 2])
def test_crowded_layout(cfg, flags):
    """The plan's ov and entries equal the rules restated here; the configurations need what they are chosen for."""
    t = _design(*CONFIGS[cfg])
    M, pos, N2 = np.asarray(t.bin_M), np.asarray(t.bin_pos), t.sllen // 2
    ov, direct, folded = overflow_slots(M, pos, N2, flags == 2)
    lay = _Layout(t, flags)
    assert lay.ov == ov
    assert _relative(lay.ex, _ovf_base(t)) == _expected_entries(M, ov, direct, folded)
    multi = any(_first_run(m) < m and o > _first_run(m) for m, o in zip(M, ov))
    assert lay.multi_run == multi
    if cfg in ("bark20_30", "mel40_10"):
        assert (np.diff(pos) == 0).any()
    if cfg in ("bark20_30", "bark24_329") and flags == 0:
        assert lay.rounds == 2
    if cfg == "bark9_100":
        assert multi


def test_tuned_slice_length_refuses_a_second_round():
    """The tuned L = 18060 slice kernels add the entries in one round: a plan of that length that needs two is refused."""
    from tests.emu.emu_backend import EmuBackend
    from xumx_slicq_b200 import _cabi

    class Crowded:
        pass
    t, u = _design("bark", 262, 32.9), Crowded()
    assert t.sllen == 18060 and (np.asarray(t.bin_M[1:7]) == 16).all() and t.bin_pos[7] >= 8
    u.sllen, u.n_bins, u.bin_M, u.win_fwd, u.win_inv, u.tukey, u.flags = (
        t.sllen, t.n_bins, t.bin_M, t.win_fwd, t.win_inv, t.tukey, 0)
    u.bin_pos = np.array(t.bin_pos, copy=True)
    u.bin_pos[1:7] = t.bin_pos[7]   # bins 1-7 at one position: four overflow entries there
    with pytest.raises(ValueError, match="tuned slice kernels"):
        _cabi.Plan(u, EmuBackend().lib())


# ------------------------------------------------------------------------------------------------ transforms
def crowded_bins(nsg):
    """Per bucket: bool [F_b], True for the bins that take part in a crowded spot: an overflow slot at a position with
    more than two of them, a position shared with a neighbour, or an overflow over several transform runs."""
    t = nsg.tables
    M, pos, N2 = np.asarray(t.bin_M), np.asarray(t.bin_pos), t.sllen // 2
    ov, direct, _ = overflow_slots(M, pos, N2, False)
    sel = np.zeros(len(M), bool)
    for slots in direct.values():
        if len(slots) > 2:
            for j, _m in slots:
                sel[j] = True
    same = np.diff(pos) == 0
    sel[1:] |= same
    sel[:-1] |= same
    sel |= np.array([_first_run(m) < m and o > _first_run(m) for m, o in zip(M, ov)])
    assert sel.any()
    return [torch.from_numpy(sel[first:first + nb].copy()) for (first, nb, _M) in t.buckets]


def _on_bins(X, sel):
    """Zero every bin of the wrapper tensors [..., F, S, M, 2] except the selected ones."""
    return [Xb * s.to(Xb.device, Xb.dtype).view(-1, 1, 1, 1) for Xb, s in zip(X, sel)]


def _inner(a, b):
    return float(sum((x.double() * y.double()).sum() for x, y in zip(a, b)))


def _check(lhs, rhs, tol):
    assert abs(lhs - rhs) <= tol * max(abs(lhs), 1.0), (lhs, rhs, abs(lhs - rhs) / max(abs(lhs), 1e-300))


def _oracle(cfg):
    """The float64 oracle.  It restates the Bark scale; for mel its scale is replaced by the product's mel scale
    (plan.MelScale: frequencies and Q factors only), and the oracle's own float64 windows, duals and transforms run on it."""
    scale, fbins, fmin = CONFIGS.get(cfg, ("mel", 160, 10.0))
    if scale == "bark":
        return SlicqOracle(scale="bark", fbins=fbins, fmin=fmin)
    from xumx_slicq_b200.plan import make_scale
    bark = slicq_oracle.BarkScale

    def mel(fmin_, fmax_, bnds):
        with contextlib.redirect_stdout(io.StringIO()):
            return make_scale("mel", fmin_, fmax_, bnds)
    slicq_oracle.BarkScale = mel
    try:
        return SlicqOracle(scale="bark", fbins=fbins, fmin=fmin)
    finally:
        slicq_oracle.BarkScale = bark


def forward_vs_oracle(base, orc, dev, T, seed=0):
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    C = base.nsgt.forward_rows(torch.from_numpy(x).to(dev))
    O = orc.forward(x.astype(np.float64))
    worst = max(float(np.abs(c.permute(2, 0, 1, 3).cpu().numpy() - o).max() / np.abs(o).max()) for c, o in zip(C, O))
    assert worst < 1e-5, worst


def synthesis_vs_oracle(base, orc, dev, T, seed=3):
    """Synthesis of perturbed coefficients, all bins and the crowded bins alone, plain and masked, against the oracle.
    Returns the outputs."""
    nsg = base.nsgt
    sel = [s.numpy() for s in crowded_bins(nsg)]
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    P = common.perturb([o.astype(np.complex64) for o in orc.forward(x.astype(np.float64))])      # [S, N, F, M]
    outs = []
    for only in (False, True):
        Q = [p * s.reshape(1, 1, -1, 1) for p, s in zip(P, sel)] if only else P
        C = [torch.from_numpy(np.ascontiguousarray(q.transpose(1, 2, 0, 3))).to(dev) for q in Q]   # [N, F, S, M]
        y_ref = orc.backward([q.astype(np.complex128) for q in Q], T)
        y = nsg.backward_rows(C, T)
        err = float(np.abs(y.cpu().numpy() - y_ref).max())
        assert err < 5e-6, err
        rs = np.random.RandomState(seed + 1)
        masks = [rs.rand(2, *c.shape).astype(np.float32) for c in C]                            # [targets, N, F, S, M]
        ym = nsg.backward_rows_masked(C, [torch.from_numpy(m).to(dev) for m in masks], T)
        Y = [np.concatenate([q * m[t].transpose(2, 0, 1, 3) for t in range(2)], axis=1) for q, m in zip(Q, masks)]
        ym_ref = orc.backward([v.astype(np.complex128) for v in Y], T)
        assert np.abs(ym.cpu().numpy() - ym_ref).max() < 5e-6, float(np.abs(ym.cpu().numpy() - ym_ref).max())
        outs += [y, ym]
    return outs


def inverse_adjoint(base, dev, T, seed=0):
    """INSGT_SL: <S c, g> == <c, S^T g> for all coefficients and with c non-zero only on the crowded bins."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, insgt = make_filterbanks(base)
    sel = crowded_bins(base.nsgt)
    gen = torch.Generator().manual_seed(seed)
    x = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    g = torch.randn(1, 2, T, generator=gen).to(dev)
    X = nsgt(x)
    R = _on_bins([torch.randn(Xb.shape, generator=gen).to(dev) for Xb in X], sel)
    grads = []
    for C0 in (X, R):
        Cg = [c.detach().clone().requires_grad_(True) for c in C0]
        y = insgt(Cg, T)
        (y * g).sum().backward()
        _check(_inner([y.detach()], [g]), _inner([c.detach() for c in Cg], [c.grad for c in Cg]), TOL_IDENTITY)
        grads.append([c.grad for c in Cg])
    return grads


def forward_adjoint(base, dev, T, seed=1):
    """NSGT_SL: <A x, d> == <x, A^T d> for all coefficients and with d non-zero only on the crowded bins (A^T is the
    synthesis of the adjoint-of-analysis plan, whose overflow below DC folds back)."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, _ = make_filterbanks(base)
    sel = crowded_bins(base.nsgt)
    gen = torch.Generator().manual_seed(seed)
    x0 = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    with torch.no_grad():
        shapes = [Xb.shape for Xb in nsgt(x0)]
    D = [torch.randn(s, generator=gen).to(dev) for s in shapes]
    grads = []
    for d in (D, _on_bins(D, sel)):
        x = x0.clone().requires_grad_(True)
        X = nsgt(x)
        sum((Xb * db).sum() for Xb, db in zip(X, d)).backward()
        _check(_inner([Xb.detach() for Xb in X], d), _inner([x.detach()], [x.grad]), TOL_IDENTITY)
        grads.append(x.grad)
    return grads


def masked(base, dev, T, n_targets=2, seed=5):
    """forward_masked == the synthesis of the materialised product, and the mask-gradient identity
    <S((m + dM) X) - S(m X), g> == sum dM * dL/dm, dM over all bins and on the crowded bins alone."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, insgt = make_filterbanks(base)
    gen = torch.Generator().manual_seed(seed)
    x = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    with torch.no_grad():
        X = nsgt(x)
        masks = [torch.rand((n_targets,) + tuple(Xb.shape[:-1]), generator=gen).to(dev) for Xb in X]
        y = insgt.forward_masked(X, masks, T)
        for t in range(n_targets):
            yt = insgt([Xb * m[t].unsqueeze(-1) for Xb, m in zip(X, masks)], T)
            assert float((y[t] - yt).abs().max()) <= 1e-6 * max(1.0, float(yt.abs().max())), float((y[t] - yt).abs().max())
    g = torch.randn(tuple(y.shape), generator=gen).to(dev)
    Mg = [m.clone().requires_grad_(True) for m in masks]
    yg = insgt.forward_masked(X, Mg, T)
    (yg * g).sum().backward()
    gm = [m.grad for m in Mg]
    sel = crowded_bins(base.nsgt)
    dM = [torch.randn(m.shape, generator=gen).to(dev) for m in masks]
    for d in (dM, [a * s.to(dev, a.dtype).view(-1, 1, 1) for a, s in zip(dM, sel)]):
        with torch.no_grad():
            y1 = insgt.forward_masked(X, [m + a for m, a in zip(masks, d)], T)
        _check(_inner([y1 - y], [g]), _inner(d, gm), TOL_IDENTITY)
    return y, gm


def round_trip(base, orc, dev, T, seed=7):
    """Round-trip SNR within 0.1 dB of the oracle's."""
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    y = base.nsgt.backward_rows(base.nsgt.forward_rows(torch.from_numpy(x).to(dev)), T).cpu().numpy()
    yo = orc.backward(orc.forward(x.astype(np.float64)), T)

    def snr(a):
        return 10 * np.log10((x.astype(np.float64) ** 2).sum() / ((a - x) ** 2).sum())
    print(f"round trip SNR {snr(y):.2f} dB, oracle {snr(yo):.2f} dB")
    assert abs(snr(y) - snr(yo)) < 0.1, (snr(y), snr(yo))


def _base(cfg, dev):
    from xumx_slicq_b200 import NSGTBase
    name, fbins, fmin = CONFIGS.get(cfg, ("mel", 160, 10.0))
    return NSGTBase(name, fbins, fmin, device=dev)


# ------------------------------------------------------------------------------------------------ CPU tier (emulation)
@pytest.fixture
def emu():
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
            cache[cfg] = (_base(cfg, "cpu"), _oracle(cfg))
        return cache[cfg]
    return get


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_forward_and_round_trip_emu(emu, emu_bases, cfg):
    b, orc = emu_bases(cfg)
    forward_vs_oracle(b, orc, torch.device("cpu"), 2 * b.sllen + 51)
    round_trip(b, orc, torch.device("cpu"), 2 * b.sllen + 51)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_synthesis_vs_oracle_emu(emu, emu_bases, cfg):
    b, orc = emu_bases(cfg)
    synthesis_vs_oracle(b, orc, torch.device("cpu"), 3 * b.sllen + 77)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_adjoints_emu(emu, emu_bases, cfg):
    b, _ = emu_bases(cfg)
    inverse_adjoint(b, torch.device("cpu"), 2 * b.sllen + 123)
    forward_adjoint(b, torch.device("cpu"), 2 * b.sllen + 123)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_masked_synthesis_emu(emu, emu_bases, cfg):
    b, _ = emu_bases(cfg)
    masked(b, torch.device("cpu"), 2 * b.sllen + 123)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tier needs CUDA"
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_crowded_gpu(dev, cfg):
    """All checks on the GPU, and bitwise-equal repeated runs of the synthesis and of both gradients."""
    b, orc = _base(cfg, dev), _oracle(cfg)
    T = 12 * b.sllen + 77
    forward_vs_oracle(b, orc, dev, T)
    round_trip(b, orc, dev, T)
    s1, s2 = synthesis_vs_oracle(b, orc, dev, T), synthesis_vs_oracle(b, orc, dev, T)
    assert all(torch.equal(u, v) for u, v in zip(s1, s2))
    gi1, gi2 = inverse_adjoint(b, dev, T), inverse_adjoint(b, dev, T)
    for a, c in zip(gi1, gi2):
        assert all(torch.equal(u, v) for u, v in zip(a, c))
    gf1, gf2 = forward_adjoint(b, dev, T), forward_adjoint(b, dev, T)
    assert all(torch.equal(u, v) for u, v in zip(gf1, gf2))
    (y1, gm1), (y2, gm2) = masked(b, dev, T), masked(b, dev, T)
    assert torch.equal(y1, y2) and all(torch.equal(u, v) for u, v in zip(gm1, gm2))


@pytest.mark.gpu
def test_mel160_30s_stereo_gpu(dev):
    """mel(160, 10 Hz) on a 30 s stereo signal: coefficients, synthesis and round trip against the oracle, both
    adjoints, the masked synthesis and its mask gradient."""
    b, orc = _base("mel160_10", dev), _oracle("mel160_10")
    T = 1323000
    forward_vs_oracle(b, orc, dev, T)
    synthesis_vs_oracle(b, orc, dev, T)
    round_trip(b, orc, dev, T)
    inverse_adjoint(b, dev, T)
    forward_adjoint(b, dev, T)
    masked(b, dev, T)

"""Band-limited filterbanks (NSGTBase(..., fmax < fs / 2)): the Nyquist bin gets a plateau window as wide as the band
between fmax and fs / 2, so it is far longer than the bins kernels' codelets (M > 292).  The plan makes it a bucket of its
own that the long-bin kernels transform (k_slice_generic.cu).  Checked here: which configurations plan, that long interior
bins (cqlog / vqlog) are still refused, the integer tables against the float64 oracle, the transforms against the oracle,
both adjoints, the masked synthesis and its mask gradient, the fused magnitudes, split / chunked / sharded calls, with all
coefficients and with only the long bin non-zero.  CPU tier: the real kernel sources on the host emulation (tests/emu);
GPU tier: -m gpu."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

import common
from oracle.slicq_oracle import SlicqOracle

FS = 44100.0
# adjoint identities <u, v> == <u', v'>: the error relative to the Cauchy-Schwarz bound |u| |v| (float32 rounding scales
# with it; a missing or wrong long bin moves the inner product by about |u| |v| / sqrt(samples), ~1e-3 of it here)
TOL_IDENTITY = 1e-6
# (scale, fbins, fmin, fmax): Nyquist bin length, its factors
PARITY = {
    "bark100_20k": ("bark", 100, 50.0, 20000.0),      # M_N = 656 = 2^4 * 41: the double path of the engine
    "bark100_16750": ("bark", 100, 50.0, 16750.0),    # M_N = 1772 = 4 * 443
    "bark64_18k": ("bark", 64, 30.0, 18000.0),        # M_N = 840, factors <= 7; bins 1, 2 below DC (mirrored-bin pass)
}
IDENTITY = dict(PARITY, mel48_14k=("mel", 48, 30.0, 14000.0), linear100_16k=("linear", 100, 100.0, 16000.0))
BARK262_16K = ("bark", 262, 32.9, 16000.0)            # M_N = 5360 = 2^4 * 5 * 67, 27 % of the coefficients

# the acceptance grid: bark / mel / linear x fmax x fbins x fmin (588 configurations)
GRID_FMAX = (11025.0, 12000.0, 14000.0, 16000.0, 18000.0, 20000.0, 21000.0)
GRID_FBINS = (24, 48, 100, 160, 262, 300, 388)
GRID_FMIN = (20.0, 32.9, 50.0, 100.0)
# outcome counts: planned (with a long Nyquist bin / with all bins <= 292) and the refusals.  Only the first two refusals
# involve the Nyquist bin (fmax below about fs / 4); the last two are limits of the other bins: the last interior bin of
# some Bark(24) filterbanks at fmax >= 20 kHz reaches beyond Nyquist (the reference's mirrored-bin pass above Nyquist), and
# the linear filterbanks with 160 or more bins have more bins of one length than one CTA of the bins kernels takes.
GRID_OUTCOMES = {"long": 357, "short": 68, "too far beyond DC / Nyquist": 14, "slice kernels' shared memory": 37,
                 "a bin below Nyquist reaches beyond it": 28, "bucket has too many bins for one CTA": 84}


def _design(scale, fbins, fmin, fmax):
    from xumx_slicq_b200.plan import design, make_scale
    with contextlib.redirect_stdout(io.StringIO()):
        scl = make_scale(scale, fmin, fmax, fbins)
    sl, tr = scl.suggested_sllen_trlen(FS)
    return design(scl, FS, sl, tr)


def _base(cfg, dev):
    from xumx_slicq_b200 import NSGTBase
    scale, fbins, fmin, fmax = cfg
    with contextlib.redirect_stdout(io.StringIO()):
        return NSGTBase(scale, fbins, fmin, fmax=fmax, device=dev)


def _oracle(cfg, dtype=np.float64):
    scale, fbins, fmin, fmax = cfg
    assert scale == "bark"
    return SlicqOracle(scale="bark", fbins=fbins, fmin=fmin, fmax=fmax, dtype=dtype)


def _emu_lib():
    from tests.emu.emu_backend import EmuBackend
    return EmuBackend().lib()


# ------------------------------------------------------------------------------------------------ plan tests (CPU)
def test_acceptance_sweep():
    """Every configuration of the grid plans, except those refused for one of the reasons of GRID_OUTCOMES; the count of
    each outcome is recorded there."""
    from xumx_slicq_b200 import _cabi
    lib = _emu_lib()
    seen, wrong = {k: 0 for k in GRID_OUTCOMES}, []
    for scale in ("bark", "mel", "linear"):
        for fmax in GRID_FMAX:
            for fbins in GRID_FBINS:
                for fmin in GRID_FMIN:
                    t = _design(scale, fbins, fmin, fmax)
                    assert (np.asarray(t.bin_M[:-1]) <= 292).all()
                    try:
                        _cabi.Plan(t, lib).close()
                    except ValueError as e:
                        why = [k for k in GRID_OUTCOMES if k in str(e)]
                        if len(why) != 1:
                            wrong.append(((scale, fbins, fmin, fmax), str(e)))
                        else:
                            seen[why[0]] += 1
                        continue
                    seen["long" if int(t.bin_M[-1]) > 292 else "short"] += 1
    assert not wrong, wrong[:10]
    assert seen == GRID_OUTCOMES, seen


@pytest.mark.parametrize("cfg", [("cqlog", 48, 100.0, 22050.0), ("cqlog", 24, 60.0, 22050.0), ("vqlog", 40, 80.0, 22050.0)])
def test_long_interior_bins_still_refused(cfg):
    from xumx_slicq_b200 import _cabi
    t = _design(*cfg)
    assert (np.asarray(t.bin_M[:-1]) > 292).any()
    with pytest.raises(ValueError, match="bin length M must be a multiple of 4 in"):
        _cabi.Plan(t, _emu_lib())


@pytest.mark.parametrize("cfg", list(PARITY.values()) + [BARK262_16K])
def test_tables_match_oracle(cfg):
    """The integer tables (M, rfbas) and the windows of plan.design against the float64 oracle's nsgfwin.  The reference
    itself is not available to the tests, so these tables are pinned against the oracle only."""
    t, orc = _design(*cfg), _oracle(cfg)
    J = t.n_bins
    assert t.sllen == orc.sl_len and J == orc.nbins
    assert np.array_equal(t.bin_M, np.asarray(orc.M[:J])) and np.array_equal(t.bin_pos, np.asarray(orc.rfbas[:J]))
    assert int(t.bin_M[-1]) > 292
    g = np.concatenate([np.asarray(orc.g[j], np.float64) for j in range(J)])
    assert np.abs(t.win_fwd.astype(np.float64) - g).max() <= 1e-6


# ------------------------------------------------------------------------------------------------ transforms
def long_only(nsg):
    """Per bucket: bool [F_b], True only for the long Nyquist bin (the last bucket)."""
    t = nsg.tables
    assert t.buckets[-1][1] == 1 and t.buckets[-1][2] > 292
    return [torch.from_numpy(np.full(nb, i == len(t.buckets) - 1)) for i, (_, nb, _M) in enumerate(t.buckets)]


def _on_bins(X, sel):
    return [Xb * s.to(Xb.device, Xb.dtype).view(-1, 1, 1, 1) for Xb, s in zip(X, sel)]


def _inner(a, b):
    return float(sum((x.double() * y.double()).sum() for x, y in zip(a, b)))


def _norm(a):
    return _inner(a, a) ** 0.5


def _check(lhs, rhs, bound, tol=TOL_IDENTITY):
    """|lhs - rhs| <= tol * bound, bound = |u| |v| of lhs = <u, v>."""
    assert abs(lhs - rhs) <= tol * bound, (lhs, rhs, abs(lhs - rhs) / bound)


def forward_vs_oracle(base, orc, dev, T, seed=0):
    """Per bucket, the long one included, max |c - c_oracle| / max |c_oracle| <= 1e-5."""
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    C = base.nsgt.forward_rows(torch.from_numpy(x).to(dev))
    O = orc.forward(x.astype(np.float64))
    errs = [float(np.abs(c.permute(2, 0, 1, 3).cpu().numpy() - o).max() / np.abs(o).max()) for c, o in zip(C, O)]
    assert max(errs) <= 1e-5, (max(errs), errs[-1])
    return C


def synthesis_vs_oracle(base, orc, dev, T, seed=3):
    """Synthesis of perturbed coefficients, all bins and the long bin alone, within 5e-6 of the oracle."""
    nsg = base.nsgt
    sel = [s.numpy() for s in long_only(nsg)]
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    P = common.perturb([o.astype(np.complex64) for o in orc.forward(x.astype(np.float64))])      # [S, N, F, M]
    outs = []
    for only in (False, True):
        Q = [p * s.reshape(1, 1, -1, 1) for p, s in zip(P, sel)] if only else P
        C = [torch.from_numpy(np.ascontiguousarray(q.transpose(1, 2, 0, 3))).to(dev) for q in Q]   # [N, F, S, M]
        y = nsg.backward_rows(C, T)
        err = float(np.abs(y.cpu().numpy() - orc.backward([q.astype(np.complex128) for q in Q], T)).max())
        assert err <= 5e-6, (only, err)
        outs.append(y)
    return outs


def round_trip(base, cfg, dev, T, seed=7):
    """Round-trip SNR no more than 0.1 dB below that of the oracle run in float32 on the same input (the oracle in
    float32 stands in for the reference's float32 result)."""
    x = np.random.RandomState(seed).rand(2, T).astype(np.float32) * 2 - 1
    y = base.nsgt.backward_rows(base.nsgt.forward_rows(torch.from_numpy(x).to(dev)), T).cpu().numpy()
    o32 = _oracle(cfg, np.float32)
    yo = o32.backward(o32.forward(x), T)

    def snr(a):
        return 10 * np.log10((x.astype(np.float64) ** 2).sum() / ((a.astype(np.float64) - x) ** 2).sum())
    print(f"round trip SNR {snr(y):.2f} dB, float32 oracle {snr(yo):.2f} dB")
    assert snr(y) >= snr(yo) - 0.1, (snr(y), snr(yo))


def inverse_adjoint(base, dev, T, seed=0):
    """INSGT_SL: <S c, g> == <c, S^T g> for all coefficients and with only the long bin non-zero."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, insgt = make_filterbanks(base)
    gen = torch.Generator().manual_seed(seed)
    x = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    g = torch.randn(1, 2, T, generator=gen).to(dev)
    X = nsgt(x)
    R = _on_bins([torch.randn(Xb.shape, generator=gen).to(dev) for Xb in X], long_only(base.nsgt))
    grads = []
    for C0 in (X, R):
        Cg = [c.detach().clone().requires_grad_(True) for c in C0]
        y = insgt(Cg, T)
        (y * g).sum().backward()
        _check(_inner([y.detach()], [g]), _inner([c.detach() for c in Cg], [c.grad for c in Cg]), _norm([y.detach()]) * _norm([g]))
        grads.append([c.grad for c in Cg])
    assert float(grads[1][-1].abs().max()) > 0
    return grads


def forward_adjoint(base, dev, T, seed=1):
    """NSGT_SL: <A x, d> == <x, A^T d> for all coefficients and with d non-zero only on the long bin (A^T is the
    synthesis of the adjoint-of-analysis plan: the part of the long bin above Nyquist folds back)."""
    from xumx_slicq_b200 import make_filterbanks
    nsgt, _ = make_filterbanks(base)
    gen = torch.Generator().manual_seed(seed)
    x0 = (torch.rand(1, 2, T, generator=gen) * 2 - 1).to(dev)
    with torch.no_grad():
        shapes = [Xb.shape for Xb in nsgt(x0)]
    D = [torch.randn(s, generator=gen).to(dev) for s in shapes]
    grads = []
    for d in (D, _on_bins(D, long_only(base.nsgt))):
        x = x0.clone().requires_grad_(True)
        X = nsgt(x)
        sum((Xb * db).sum() for Xb, db in zip(X, d)).backward()
        _check(_inner([Xb.detach() for Xb in X], d), _inner([x.detach()], [x.grad]), _norm([Xb.detach() for Xb in X]) * _norm(d))
        grads.append(x.grad)
    return grads


def masked(base, dev, T, n_targets=2, seed=5):
    """forward_masked == the synthesis of the materialised product; the mask identity
    <S((m + dM) X) - S(m X), g> == sum dM * dL/dm (dM everywhere and on the long bin alone); the mixture identity
    <S(m X), g> == <X, dL/dX>; the fused mask gradient == Re(conj(X) S^T g) of the unfused adjoint."""
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
    dM = [torch.randn(m.shape, generator=gen).to(dev) for m in masks]
    for d in (dM, [a * s.to(dev, a.dtype).view(-1, 1, 1) for a, s in zip(dM, long_only(base.nsgt))]):
        with torch.no_grad():
            y1 = insgt.forward_masked(X, [m + a for m, a in zip(masks, d)], T)
        _check(_inner([y1 - y], [g]), _inner(d, gm), _norm([y1 - y]) * _norm([g]))
    # mixture identity
    Xg = [Xb.clone().requires_grad_(True) for Xb in X]
    yx = insgt.forward_masked(Xg, masks, T)
    (yx * g).sum().backward()
    _check(_inner([yx.detach()], [g]), _inner(X, [a.grad for a in Xg]), _norm([yx.detach()]) * _norm([g]))
    # fused == unfused mask gradient
    rows = n_targets * 2
    cadj = base.nsgt.synthesis_adjoint_rows(g.reshape(rows, T), X[0].shape[-3])
    for a, c, Xb in zip(gm, cadj, X):
        xc = torch.view_as_complex(Xb.contiguous()).reshape((-1,) + tuple(Xb.shape[-4:-1]))
        ref = torch.real(xc.conj() * c.view((n_targets, -1) + tuple(c.shape[1:]))).reshape(a.shape)
        assert float((a - ref).abs().max()) <= 1e-6 * float(ref.abs().max()), float((a - ref).abs().max())
    return y, gm


def norms(base, dev, T, seed=6):
    """forward_with_norm: the coefficients of the plain call, and |X| == ComplexNorm()(X)."""
    from xumx_slicq_b200 import make_filterbanks, ComplexNorm
    nsgt, _ = make_filterbanks(base)
    x = (torch.rand(1, 2, T, generator=torch.Generator().manual_seed(seed)) * 2 - 1).to(dev)
    X_ref = nsgt(x)
    X, Xmag = nsgt.forward_with_norm(x)
    for a, a_ref, m, m_ref in zip(X, X_ref, Xmag, ComplexNorm()(X_ref)):
        assert torch.equal(a, a_ref)
        assert m.shape == m_ref.shape and float((m - m_ref).abs().max()) <= 1e-6 * float(m_ref.max())


def shards_bitwise(base, dev, T, worlds=(2, 3)):
    """Slice ranges with one half-slice halo per boundary == the unsharded transform, bitwise."""
    nsg = base.nsgt
    hop = nsg.sl_len // 2
    x = (torch.rand(2, T, generator=torch.Generator().manual_seed(9)) * 2 - 1).to(dev)
    S = nsg.n_slices(T)
    full = nsg.forward_rows(x)
    y_full = nsg.backward_rows(full, T)
    for world in worlds:
        cuts = [round(i * S / world) for i in range(world + 1)]
        ys, halos = [], []
        for a, b in zip(cuts[:-1], cuts[1:]):
            lo, hi = max(0, (a - 1) * hop), min(T, b * hop)
            part = nsg.forward_rows(x[:, lo:hi].contiguous(), k0=a, n_slices=b - a, t0=lo)
            assert all(torch.equal(pc, fc[:, :, a:b]) for pc, fc in zip(part, full))
            halo = torch.zeros(2, hop, device=dev)
            ys.append(nsg.backward_rows(part, min(T, b * hop) - a * hop, k0=a, t0=a * hop, halo_out=halo))
            halos.append(halo)
        for i in range(world - 1):
            ys[i][:, -hop:] += halos[i + 1]
        assert torch.equal(torch.cat(ys, dim=1), y_full), world


# ------------------------------------------------------------------------------------------------ CPU tier (emulation)
@pytest.fixture(scope="module")
def emu():
    from tests.emu.emu_backend import EmuBackend
    import xumx_slicq_b200.nsgt as nsgt_mod
    old = nsgt_mod._BACKEND
    nsgt_mod._BACKEND = EmuBackend()
    yield nsgt_mod._BACKEND
    nsgt_mod._BACKEND = old


@pytest.fixture(scope="module")
def emu_bases(emu):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = _base(IDENTITY[name], "cpu")
        return cache[name]
    return get


CPU = torch.device("cpu")


def _emu_T(b):
    return 2 * b.sllen + 51


@pytest.mark.parametrize("name", list(PARITY))
def test_parity_emu(emu_bases, name):
    b = emu_bases(name)
    orc = _oracle(PARITY[name])
    forward_vs_oracle(b, orc, CPU, _emu_T(b))
    synthesis_vs_oracle(b, orc, CPU, _emu_T(b) + b.sllen // 3)
    round_trip(b, PARITY[name], CPU, _emu_T(b))


@pytest.mark.parametrize("name", list(IDENTITY))
def test_adjoints_emu(emu_bases, name):
    b = emu_bases(name)
    inverse_adjoint(b, CPU, _emu_T(b) + 72)
    forward_adjoint(b, CPU, _emu_T(b) + 72)


@pytest.mark.parametrize("name", list(IDENTITY))
def test_masked_and_norms_emu(emu_bases, name):
    b = emu_bases(name)
    masked(b, CPU, _emu_T(b) + 72)
    norms(b, CPU, _emu_T(b))


def test_shards_emu(emu_bases):
    b = emu_bases("bark100_20k")
    shards_bitwise(b, CPU, 5 * b.sllen + 333)


def test_split_and_chunks_emu(emu, monkeypatch):
    """Calls split into two row groups (SLICQ_SPLIT_UNITS) or into chunks (SLICQ_CHUNK_MB) give bitwise the results of
    whole calls, for the analysis, its magnitudes, the synthesis and the masked synthesis.  The launch count shows the
    long-bin kernel once per chunk: the analysis runs slice, bins and long-bin kernel per chunk."""
    cfg = IDENTITY["bark100_20k"]
    lib = emu.lib()
    t = _design(*cfg)
    M, pos, N2 = np.asarray(t.bin_M), np.asarray(t.bin_pos), t.sllen // 2
    assert not ((pos[1:-1] < M[1:-1] // 2).any())           # no mirrored-bin pass: three analysis launches per chunk
    T = 4 * t.sllen + 99
    gen = torch.Generator().manual_seed(11)
    x = torch.rand(4, T, generator=gen) * 2 - 1

    def run(**env):
        with monkeypatch.context() as m:
            for k in ("SLICQ_SPLIT_UNITS", "SLICQ_CHUNK_MB"):
                m.delenv(k, raising=False)
            for k, v in env.items():
                m.setenv(k, v)
            nsg = _base(cfg, "cpu").nsgt
            nsg.plan(CPU)                                    # the plan reads the environment when it is created
        n0 = lib.slicq_launch_count()
        C = nsg.forward_rows(x)
        n_fwd = lib.slicq_launch_count() - n0
        masks = [torch.rand((2,) + tuple(c.shape), generator=torch.Generator().manual_seed(12)) for c in C]
        y = nsg.backward_rows(C, T)
        ym = nsg.backward_rows_masked(C, masks, T)
        return [*C, y, ym], n_fwd

    ref, n_whole = run()
    assert n_whole == 3
    out, n_split = run(SLICQ_SPLIT_UNITS="8")
    assert n_split == 6 and all(torch.equal(a, b) for a, b in zip(out, ref))
    out, n_chunk = run(SLICQ_CHUNK_MB="1")
    pad_l = max(0, int(max(M // 2 - pos)))
    pad_r = max(0, int(max(pos + M // 2 - 1 - N2)))
    pad_l, pad_r = (pad_l + 1) & ~1, (pad_r + 1) & ~1
    per_unit = ((pad_l + N2 + 1 + pad_r + 1) & ~1) * 8
    chunks = -(-4 * t.num_slices(T) // ((1 << 20) // per_unit))
    assert chunks >= 2 and n_chunk == 3 * chunks, (n_chunk, chunks)
    assert all(torch.equal(a, b) for a, b in zip(out, ref))


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tier needs CUDA"
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(IDENTITY))
def test_long_bin_gpu(dev, name):
    """All checks on the GPU; repeated runs of the synthesis, both gradients and the masked synthesis are bitwise equal."""
    b = _base(IDENTITY[name], dev)
    T = 12 * b.sllen + 77
    if name in PARITY:
        orc = _oracle(PARITY[name])
        forward_vs_oracle(b, orc, dev, T)
        s1, s2 = synthesis_vs_oracle(b, orc, dev, T), synthesis_vs_oracle(b, orc, dev, T)
        assert all(torch.equal(u, v) for u, v in zip(s1, s2))
        round_trip(b, PARITY[name], dev, T)
    gi1, gi2 = inverse_adjoint(b, dev, T), inverse_adjoint(b, dev, T)
    for a, c in zip(gi1, gi2):
        assert all(torch.equal(u, v) for u, v in zip(a, c))
    gf1, gf2 = forward_adjoint(b, dev, T), forward_adjoint(b, dev, T)
    assert all(torch.equal(u, v) for u, v in zip(gf1, gf2))
    (y1, gm1), (y2, gm2) = masked(b, dev, T), masked(b, dev, T)
    assert torch.equal(y1, y2) and all(torch.equal(u, v) for u, v in zip(gm1, gm2))
    norms(b, dev, T)
    shards_bitwise(b, dev, T, worlds=(2, 4, 8))


@pytest.mark.gpu
def test_bark262_16k_30s_stereo_gpu(dev):
    """Bark(262, 32.9 Hz, fmax 16 kHz) on a 30 s stereo signal: the Nyquist bin holds 27 % of the coefficients.
    Coefficients, synthesis and round trip against the oracle, both adjoints, the masked synthesis and its gradient."""
    b = _base(BARK262_16K, dev)
    assert int(b.nsgt.tables.bin_M[-1]) == 5360
    orc = _oracle(BARK262_16K)
    T = 1323000
    forward_vs_oracle(b, orc, dev, T)
    synthesis_vs_oracle(b, orc, dev, T)
    round_trip(b, BARK262_16K, dev, T)
    inverse_adjoint(b, dev, T)
    forward_adjoint(b, dev, T)
    masked(b, dev, T)

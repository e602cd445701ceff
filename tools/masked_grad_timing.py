"""Time the mask gradient of INSGT_SL.forward_masked at the realtime demix shape: fused vs unfused.

    python tools/masked_grad_timing.py [--targets 4] [--batch 8] [--seconds 30] [--reps 10] [--out result.json]

Bark(262, 32.9 Hz), `targets` masks requiring grad over a batch of stereo mixtures.  Two paths compute
dL/dm = Re(conj(X) * S^T g) for the same output gradient g:
  fused    NSGT_sliced.mask_grad_rows: the adjoint analysis takes the product with the mixture in its epilogue
           (what forward_masked's backward runs when only the masks require grad)
  unfused  NSGT_sliced.synthesis_adjoint_rows (complex S^T g stored) + torch elementwise Re(conj(X) * .)
plus `autograd`: torch.autograd.grad through forward_masked (the fused path with the wrapper's reshapes).
Each pass is timed with CUDA events on the current stream; a 512 MB buffer is overwritten between passes so that no pass
starts with its inputs in L2.  The paths alternate within one run.  Prints the card, its power limit, per-path times
(median, min) and the largest difference between the fused and unfused gradients relative to each bucket's maximum.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card_info() -> dict:
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl, clk = [v.strip() for v in out.split(",")]
        info.update(name=name, power_limit_w=float(pl), max_sm_clock_mhz=float(clk))
    except Exception as e:  # the query is informational; the timing does not depend on it
        info["query_error"] = str(e)
    return info


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--targets", type=int, default=4)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the result as JSON here")
    a = ap.parse_args()

    import torch
    from xumx_slicq_b200 import NSGTBase, make_filterbanks

    if not torch.cuda.is_available():
        raise SystemExit("masked_grad_timing needs a CUDA device")
    dev = torch.device("cuda:0")
    base = NSGTBase("bark", 262, 32.9, device=dev)
    nsgt, insgt = make_filterbanks(base)
    nsg = base.nsgt
    T = int(a.seconds * 44100)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(a.batch, 2, T, device=dev, generator=gen) * 2 - 1
    with torch.no_grad():
        X = nsgt(x)
    masks = [torch.rand((a.targets,) + tuple(Xb.shape[:-1]), device=dev, generator=gen).requires_grad_(True) for Xb in X]
    g = torch.randn(a.targets, a.batch, 2, T, device=dev, generator=gen)
    rows, N, S = a.targets * a.batch * 2, a.batch * 2, X[0].shape[-3]
    xs, _, _ = insgt._masked_inputs(X, masks)
    g2 = g.view(rows, T)
    y = insgt.forward_masked(X, masks, T)

    def fused():
        return nsg.mask_grad_rows(g2, xs, a.targets)

    def unfused():
        c = nsg.synthesis_adjoint_rows(g2, S)
        return [torch.real(x.conj() * cb.view((a.targets, N) + tuple(cb.shape[1:]))) for x, cb in zip(xs, c)]

    def autograd():
        return torch.autograd.grad(y, masks, g, retain_graph=True)

    paths = {"fused": fused, "unfused": unfused, "autograd": autograd}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    for fn in paths.values():          # warm-up: modules, plans, allocator
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in paths}
    for _ in range(a.reps):
        for k, fn in paths.items():
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
            del out
    gf, gu = fused(), unfused()
    worst = max(float((f.reshape(u.shape) - u).abs().max() / u.abs().max()) for f, u in zip(gf, gu))
    coefs = rows * S * nsg.tables.sum_M
    res = {
        "card": card_info(),
        "shape": {"targets": a.targets, "batch": a.batch, "channels": 2, "samples": T, "slices": S,
                  "mask_coefficients": coefs},
        "ms": {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "all": v} for k, v in times.items()},
        "max_rel_diff_fused_vs_unfused": worst,
    }
    res["speedup_fused_vs_unfused"] = res["ms"]["unfused"]["median"] / res["ms"]["fused"]["median"]
    c = res["card"]
    print(f"card: {c['name']}, power limit {c.get('power_limit_w')} W")
    print(f"shape: {a.targets} targets x {a.batch} x 2 x {T} samples, {S} slices, {coefs / 1e6:.1f} M mask coefficients")
    for k, v in res["ms"].items():
        print(f"{k:9s} median {v['median']:8.3f} ms   min {v['min']:8.3f} ms")
    print(f"fused vs unfused: {res['speedup_fused_vs_unfused']:.2f}x, max |diff| / bucket max {worst:.3g}")
    print(json.dumps({k: v for k, v in res.items() if k != "ms"} | {"ms": {k: v["median"] for k, v in res["ms"].items()}}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

"""Time forward + masked inverse on band-limited filterbanks, whose Nyquist bin runs on the long-bin kernels.

    python tools/long_bin_timing.py [--targets 4] [--batch 8] [--seconds 30] [--reps 10] [--out result.json]

For each configuration: NSGT_SL forward of a batch of stereo mixtures, then INSGT_SL.forward_masked with `targets` masks
(the realtime demix pair), without grad.  Bark(262, 32.9 Hz) at fmax 22 050 Hz (the pretrained configuration, no long
bin) is timed alongside at fmax 20 000 and 16 000 Hz; mel(160, 10 Hz, 16 kHz) and Bark(100, 50 Hz, 16 750 Hz) (Nyquist
bin 4 * 443) complete the set.  Each pass is timed with CUDA events on the current stream; a 512 MB buffer is overwritten
between passes so that no pass starts with its inputs in L2.  The configurations alternate within one run.  A separate
torch.profiler run (CUDA activities) then sums the device time per kernel name over `--prof-reps` passes of each
configuration and reports the long-bin kernels' share, next to the Nyquist bin's share of the coefficients.  Prints the
card, its power limit and per-configuration times (median, min).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

CONFIGS = {"bark262_22050": ("bark", 262, 32.9, 22050.0), "bark262_20000": ("bark", 262, 32.9, 20000.0),
           "bark262_16000": ("bark", 262, 32.9, 16000.0), "mel160_16000": ("mel", 160, 10.0, 16000.0),
           "bark100_16750": ("bark", 100, 50.0, 16750.0)}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--targets", type=int, default=4)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--prof-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the result as JSON here")
    a = ap.parse_args()

    import torch
    from masked_grad_timing import card_info
    from xumx_slicq_b200 import NSGTBase, make_filterbanks

    if not torch.cuda.is_available():
        raise SystemExit("long_bin_timing needs a CUDA device")
    dev = torch.device("cuda:0")
    T = int(a.seconds * 44100)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(a.batch, 2, T, device=dev, generator=gen) * 2 - 1
    runs, shapes = {}, {}
    for name, (scale, fbins, fmin, fmax) in CONFIGS.items():
        base = NSGTBase(scale, fbins, fmin, fmax=fmax, device=dev)
        nsgt, insgt = make_filterbanks(base)
        with torch.no_grad():
            X = nsgt(x)
        masks = [torch.rand((a.targets,) + tuple(Xb.shape[:-1]), device=dev, generator=gen) for Xb in X]
        M = base.nsgt.tables.bin_M
        shapes[name] = {"sllen": base.sllen, "bins": base.nsgt.tables.n_bins, "slices": X[0].shape[-3],
                        "nyquist_M": int(M[-1]), "nyquist_share": float(M[-1]) / float(M.sum())}

        def step(nsgt=nsgt, insgt=insgt, masks=masks):
            with torch.no_grad():
                return insgt.forward_masked(nsgt(x), masks, T)
        runs[name] = step
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    for fn in runs.values():           # warm-up: modules, plans, allocator
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(a.reps):
        for k, fn in runs.items():
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
            del out

    # device time per kernel name, per configuration
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for k, fn in runs.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.prof_reps):
                fn()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if t > 0:
                per[ev.key] = per.get(ev.key, 0.0) + t / 1000.0 / a.prof_reps     # ms per pass
        total = sum(per.values())
        long_ms = sum(v for n, v in per.items() if "long_bin" in n)
        kernels[k] = {"device_ms": total, "long_bin_ms": long_ms, "long_bin_share": long_ms / total if total else 0.0,
                      "per_kernel_ms": dict(sorted(per.items(), key=lambda kv: -kv[1]))}

    res = {"card": card_info(),
           "shape": {"targets": a.targets, "batch": a.batch, "channels": 2, "samples": T},
           "configs": shapes,
           "ms": {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "all": v} for k, v in times.items()},
           "profile": kernels}
    c = res["card"]
    print(f"card: {c['name']}, power limit {c.get('power_limit_w')} W")
    print(f"forward + {a.targets}-target masked inverse, batch {a.batch} x 2 x {T} samples")
    for k, v in res["ms"].items():
        s, p = shapes[k], kernels[k]
        print(f"{k:14s} sllen {s['sllen']:6d} Nyquist M {s['nyquist_M']:5d} ({100 * s['nyquist_share']:4.1f} % of the "
              f"coefficients)   median {v['median']:8.3f} ms   min {v['min']:8.3f} ms   device {p['device_ms']:8.3f} ms, "
              f"long-bin kernels {p['long_bin_ms']:7.3f} ms ({100 * p['long_bin_share']:4.1f} %)")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

"""Time forward + masked inverse on filterbanks whose lowest bins crowd together near DC, next to Bark-262.

    python tools/crowded_timing.py [--targets 4] [--batch 8] [--seconds 30] [--reps 10] [--out result.json]

For each configuration: NSGT_SL forward of a batch of stereo mixtures, then INSGT_SL.forward_masked with `targets` masks
(the realtime demix pair), without grad.  Bark(24, 32.9 Hz) needs two rounds of overflow entries in the generic slice
kernel; mel(160, 10 Hz) shares positions between its lowest bins.  Bark(262, 32.9 Hz), the pretrained configuration on
the tuned kernels, is timed alongside for scale.  Each pass is timed with CUDA events on the current stream; a 512 MB
buffer is overwritten between passes so that no pass starts with its inputs in L2.  The configurations alternate within
one run.  Prints the card, its power limit and per-configuration times (median, min).
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

CONFIGS = {"bark24_32.9": ("bark", 24, 32.9), "mel160_10": ("mel", 160, 10.0), "bark262_32.9": ("bark", 262, 32.9)}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--targets", type=int, default=4)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the result as JSON here")
    a = ap.parse_args()

    import torch
    from masked_grad_timing import card_info
    from xumx_slicq_b200 import NSGTBase, make_filterbanks

    if not torch.cuda.is_available():
        raise SystemExit("crowded_timing needs a CUDA device")
    dev = torch.device("cuda:0")
    T = int(a.seconds * 44100)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(a.batch, 2, T, device=dev, generator=gen) * 2 - 1
    runs, shapes = {}, {}
    for name, (scale, fbins, fmin) in CONFIGS.items():
        base = NSGTBase(scale, fbins, fmin, device=dev)
        nsgt, insgt = make_filterbanks(base)
        with torch.no_grad():
            X = nsgt(x)
        masks = [torch.rand((a.targets,) + tuple(Xb.shape[:-1]), device=dev, generator=gen) for Xb in X]
        shapes[name] = {"sllen": base.sllen, "bins": base.nsgt.tables.n_bins, "slices": X[0].shape[-3]}

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
    res = {"card": card_info(),
           "shape": {"targets": a.targets, "batch": a.batch, "channels": 2, "samples": T},
           "configs": shapes,
           "ms": {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "all": v} for k, v in times.items()}}
    c = res["card"]
    print(f"card: {c['name']}, power limit {c.get('power_limit_w')} W")
    print(f"forward + {a.targets}-target masked inverse, batch {a.batch} x 2 x {T} samples")
    for k, v in res["ms"].items():
        print(f"{k:13s} sllen {shapes[k]['sllen']:6d} bins {shapes[k]['bins']:4d}   median {v['median']:8.3f} ms   "
              f"min {v['min']:8.3f} ms")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

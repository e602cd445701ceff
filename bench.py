#!/usr/bin/env python3
"""Benchmark of the sliCQT hot path (BASELINE.json metric: fwd+inv audio-seconds per second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[1]: the sliCQT path of a realtime-model demix of one synthetic 30 s
44.1 kHz stereo mixture -- ONE forward (2 rows x 148 slices) and ONE inverse of the 4 target
estimates (8 rows x 148 slices).  The 4 target coefficient sets stand in for the model output
(mixture coefficients times per-target gains, generated before the timed region; the CDAE model
is out of scope, SURVEY.md section 8).  One step = one such pass per GPU (weak scaling: every rank
owns its own mixture, tracks are independent, no data-path collective).

Printed JSON line (rank 0): see the keys documented in DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

FS = 44100
SECONDS = 30.0
T = int(SECONDS * FS)            # 1 323 000 samples
N_TARGETS = 4
GAINS = (0.9, 0.6, 0.4, 0.2)     # stand-in "soft masks" of the four targets
SCALE = dict(scale="bark", fbins=262, fmin=32.9)
# algorithmic HBM bytes (SURVEY.md section 8(d)): per (row, slice) and direction
B_IN = 9030 * 4                  # new input / output samples of one hop
B_COEF = 18640 * 8               # complex64 coefficients
B_UNIT = B_IN + B_COEF           # 185 240


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons during the timed region (pynvml, nvidia-smi fallback)."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _reasons(self, mask: int):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        return {k for k, bit in names.items() if mask & bit}

    def run(self):
        if self.h is None:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.reasons |= self._reasons(int(mask))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
def _import_reference():
    """The UNMODIFIED reference package (xumx_slicq_v2): baseline/_ref (pip --target install, DESIGN.md),
    then $SLICQ_REFERENCE, then /root/reference.  Returns (module transforms, where) or (None, why)."""
    import importlib
    cands = [os.path.join(ROOT, "baseline", "_ref"), os.environ.get("SLICQ_REFERENCE", ""), "/root/reference"]
    why = "not found"
    for c in cands:
        if not c or not os.path.isdir(os.path.join(c, "xumx_slicq_v2")):
            continue
        sys.path.insert(0, c)
        try:
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                mod = importlib.import_module("xumx_slicq_v2.transforms")
            return mod, c
        except Exception as e:          # missing optional dependency of the reference package
            why = f"{c}: {type(e).__name__}: {e}"
            sys.path.remove(c)
    return None, why


def cpu_reference_arm(steps: int, warmup: int, sample_seconds: float):
    """The reference's own CPU implementation of the path on the host cores, all threads: the unmodified
    xumx_slicq_v2 NSGT_SL / INSGT_SL (torch, device="cpu") when the package can be imported (kind "reference"),
    else the NumPy/pocketfft port in oracle/ (kind "port").  One step = a bounded sample of the workload:
    a `sample_seconds` stereo mixture, 1 forward + inverse of 4 targets.
    Returns (audio-s/s, seconds per step, cores, sample description, kind)."""
    cores = os.cpu_count() or 1
    Ts = int(sample_seconds * FS)
    rs = np.random.RandomState(0)
    x = (rs.rand(2, Ts).astype(np.float32) * 2 - 1)
    sample = f"{sample_seconds:g} s stereo mixture: 1 forward (2 rows) + inverse of 4 targets (8 rows)"
    ref, where = _import_reference()
    if ref is not None:
        import io, contextlib, warnings
        import torch
        torch.set_num_threads(cores)
        with contextlib.redirect_stdout(io.StringIO()):
            base = ref.NSGTBase(SCALE["scale"], SCALE["fbins"], SCALE["fmin"], device="cpu")
        nsgt, insgt = ref.make_filterbanks(base)
        xt = torch.from_numpy(x).view(1, 2, Ts)
        gains = torch.tensor(GAINS).view(4, 1, 1, 1, 1, 1, 1)

        def step():
            with torch.no_grad(), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                X = nsgt(xt)
                # model-output stand-in (contiguous like Unmix outputs; the reference's backward mutates it: fresh every step)
                Y = [(Xb.unsqueeze(0) * gains).contiguous() for Xb in X]
                return insgt(Y, Ts)
        kind = "reference"
        sample += f"; unmodified xumx_slicq_v2 torch CPU path from {os.path.relpath(where, ROOT) if where.startswith(ROOT) else where}, {cores} threads"
    else:
        from oracle.slicq_oracle import SlicqOracle
        orc = SlicqOracle(**SCALE, dtype=np.float32, workers=cores)

        def step():
            C = orc.forward(x)
            Y = [np.concatenate([c * np.float32(g) for g in GAINS], axis=1) for c in C]   # [S, 4*2, F, M]
            return orc.backward(Y, Ts)
        kind = "port"
        sample += f"; NumPy port (reference package not importable: {where})"

    for _ in range(max(1, warmup)):
        step()
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t = time.perf_counter()
        step()
        times.append(time.perf_counter() - t)
        if time.perf_counter() - t_start > 150.0:      # keep the arm within a few minutes on slow hosts
            break
    dt = float(np.mean(times))
    return sample_seconds / dt, dt, cores, sample, kind, len(times)


def slice_sharding_run(nsg, dev, rank, world, steps: int, warmup: int):
    """BASELINE.json configs[3]: ONE synthetic 3-min stereo track (881 slices), 1 forward + 4-target synthesis fused with
    mask * mixture; slices split into contiguous ranges over the ranks, one [rows, 9030] fp32 halo message per boundary
    and direction over NCCL.  Every rank also runs the unsharded track on its own GPU (the 1-GPU time of the same work)
    and checks its shard against it bit for bit.  Returns a dict on every rank (max over ranks where it matters)."""
    import torch
    import torch.distributed as dist
    from xumx_slicq_b200.sharding import SliceShardedSliCQT
    Ttrack = 180 * FS
    distributed = world > 1
    gen = torch.Generator(device=dev).manual_seed(7)
    x = torch.rand(2, Ttrack, device=dev, generator=gen) * 2 - 1
    stream = torch.cuda.current_stream(dev)

    def timed(step):
        for _ in range(warmup):
            step()
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(steps):
            y = step()
        b.record(stream)
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t = torch.tensor([a.elapsed_time(b) / steps], device=dev, dtype=torch.float64)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), y

    # unsharded (what one GPU does alone), same buffers reused every step
    ctx1, ctx1i = {}, {}
    C1 = nsg.forward_rows_into(ctx1, x)
    masks1 = [torch.stack([torch.full(tuple(c.shape), g, dtype=torch.float32, device=dev) for g in GAINS]) for c in C1]

    def step1():
        C = nsg.forward_rows_into(ctx1, x)
        return nsg.backward_rows_masked(C, masks1, Ttrack, ctx=ctx1i)
    ms1, y1 = timed(step1)
    out = {"ms_per_step_1gpu": ms1, "n_gpus": world}
    if not distributed:
        out.update(ms_per_step=ms1, speedup_vs_1=1.0, bitwise_equal=True,
                   max_abs_err_target0=float((y1[:2] - GAINS[0] * x).abs().max()))
        return out
    sh = SliceShardedSliCQT(nsg, Ttrack, persistent=True)
    x_local = sh.local_input(x)
    masks = [m[:, :, :, sh.k0:sh.k1].contiguous() for m in masks1]

    def stepn():
        C = sh.forward(x_local)
        return sh.inverse_masked(C, masks)
    msn, yn = timed(stepn)
    Cn = sh.forward(x_local)
    ok = all(torch.equal(pc, fc[:, :, sh.k0:sh.k1]) for pc, fc in zip(Cn, C1)) and torch.equal(yn, y1[:, sh.lo:sh.hi])
    flag = torch.tensor([int(ok)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out.update(ms_per_step=msn, speedup_vs_1=ms1 / msn, bitwise_equal=bool(int(flag.item())),
               slices_per_rank=sh.k1 - sh.k0, halo_bytes_per_boundary_and_direction=[2 * sh.hop * 4, 8 * sh.hop * 4],
               max_abs_err_target0=float((yn[:2] - GAINS[0] * x_local).abs().max()))
    return out


def bench_sweep(args, nsg, dev, rank, world, distributed):
    """BASELINE.json configs[4]: throughput sweep over `--tracks` synthetic 3-min stereo tracks, dealt round-robin to the
    ranks (sharding.shard_tracks, no data-path communication).  Every track is generated ON THE DEVICE from its own seed,
    analysed (2 rows x 881 slices) and resynthesised for 4 targets (mask * mixture fused into the synthesis); wall clock
    between two barriers, all tracks."""
    import torch
    import torch.distributed as dist
    from xumx_slicq_b200.sharding import shard_tracks
    Ttrack = 180 * FS
    mine = shard_tracks(args.tracks, rank, world)
    ctx, ctxi = {}, {}
    gen = torch.Generator(device=dev)
    x = torch.empty(2, Ttrack, device=dev)
    C = nsg.forward_rows_into(ctx, x)
    masks = [torch.stack([torch.full(tuple(c.shape), g, dtype=torch.float32, device=dev) for g in GAINS]) for c in C]
    worst = 0.0

    def one(track_id, check=False):
        gen.manual_seed(track_id)
        x.uniform_(-1.0, 1.0, generator=gen)
        Cc = nsg.forward_rows_into(ctx, x)
        y = nsg.backward_rows_masked(Cc, masks, Ttrack, ctx=ctxi)
        return float((y[:2] - GAINS[0] * x).abs().max()) if check else 0.0
    for t in mine[:2]:
        worst = max(worst, one(t, check=True))
    if distributed:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for t in mine:
        one(t)
    torch.cuda.synchronize(dev)
    if distributed:
        dist.barrier()
    wall = time.perf_counter() - t0
    tw = torch.tensor([wall], device=dev, dtype=torch.float64)
    if distributed:
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
    wall = float(tw.item())
    if rank == 0:
        emit(({
            "metric": "sliCQT fwd+inv audio-sec/sec", "value": args.tracks * 180.0 / wall, "unit": "audio-s/s",
            "n_gpus": world, "steps": args.tracks, "warmup": 2, "ms_per_step": wall / max(1, len(mine)) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"configs[4]: {args.tracks} synthetic 3-min 44.1 kHz stereo tracks (generated on the device per "
                                   "track seed), 1 forward + 4-target synthesis each, dealt round-robin to the GPUs",
                       "parallelism": f"tracks x{world}", "tracks_per_gpu": len(mine)},
            "wall_s": wall, "max_abs_err_target0": worst,
        }))
    if distributed:
        dist.destroy_process_group()


def bench_slices(args, nsg, dev, rank, world, distributed):
    """`--mode slices`: the configs[3] line on its own (strong scaling)."""
    import torch.distributed as dist
    r = slice_sharding_run(nsg, dev, rank, world, args.steps, args.warmup)
    if rank == 0:
        emit(({
            "metric": "sliCQT fwd+inv audio-sec/sec", "value": 180.0 / (r["ms_per_step"] * 1e-3), "unit": "audio-s/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[3]: one synthetic 3-min stereo track (881 slices), 1 forward + 4-target "
                                   "inverse, slices sharded in contiguous ranges, one [rows, 9030] fp32 halo message "
                                   "per boundary and direction over NCCL; the 4 targets are mask * mixture fused into the synthesis "
                                   "(constant masks as the model stand-in)",
                       "parallelism": f"slices x{world}"},
            "slice_sharding": r, "max_abs_err_target0": r["max_abs_err_target0"],
        }))
    if distributed:
        dist.destroy_process_group()


def bind_rank_to_cores(local_rank: int, local_world: int):
    """Pin this rank to its own share of the host cores near its GPU (NVML cpu affinity of the device, split evenly
    between the ranks that share it), BEFORE pinned buffers are allocated: page-locked staging memory is then
    first-touched on the GPU's NUMA node and the copy-submitting threads of the ranks do not migrate over each other.
    Returns a description for the bench line."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1 and w * 64 + b < ncpu]
        try:
            numa = [w * 64 + b for w, m in enumerate(pynvml.nvmlDeviceGetMemoryAffinity(h, 4, 0)) for b in range(64) if (m >> b) & 1]
        except Exception:
            numa = None
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0))) or sorted(os.sched_getaffinity(0))
        # ranks whose GPUs share this affinity mask split it evenly
        per = max(1, len(allowed) // max(1, local_world))
        mine = allowed[(local_rank % max(1, local_world)) * per:(local_rank % max(1, local_world) + 1) * per] or allowed
        os.sched_setaffinity(0, mine)
        info = {"bound": True, "cores": f"{mine[0]}-{mine[-1]}", "n_cores": len(mine), "gpu_numa_nodes": numa,
                "gpu_cpu_affinity": f"{cpus[0]}-{cpus[-1]}" if cpus else None}
    except Exception as e:                      # binding is an optimisation: report and carry on
        info["error"] = f"{type(e).__name__}: {e}"[:160]
    return info


DUMP_COEFS = 3 << 20             # complex coefficients kept by --dump-outputs (24 MiB as float32 pairs)
DUMP_SAMPLES = 6 << 20           # waveform samples kept by --dump-outputs (24 MiB)


def _sample(flat, n: int, seed: int):
    """A fixed sample of a flat device tensor: up to n distinct positions (all of them if it has no more), drawn from
    a seeded CPU generator and sorted, so that every run with the same arguments picks the same elements."""
    N = flat.numel()
    if N <= n:
        return flat
    import torch
    idx = torch.unique(torch.randint(N, (n,), generator=torch.Generator().manual_seed(seed)))   # sorted
    return flat[idx.to(flat.device)]


def dump_outputs(out_dir: str, coefs, y) -> dict:
    """Write what one step of the timed path returned: the forward coefficients (every bucket [rows, F_b, S, M_b]
    complex64, flattened in bucket order and sampled, stored as float32 [n, 2] real / imaginary pairs) and the inverse
    output (4 target waveforms, [targets * rows, T] float32, flattened and sampled).  Returns {name: shape}."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat_c = torch.cat([c.reshape(-1) for c in coefs])
    out = {"forward_coefficients": torch.view_as_real(_sample(flat_c, DUMP_COEFS, 0)),
           "inverse_waveforms": _sample(y.reshape(-1), DUMP_SAMPLES, 1)}
    shapes = {}
    for name, t in out.items():
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        shapes[name] = list(a.shape)
    return shapes


_JSON_FD = None


def _claim_stdout() -> None:
    """stdout carries exactly ONE JSON line: everything else a library prints to file descriptor 1 (the NCCL
    version banner, build chatter) is redirected to stderr; emit() writes to the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj) -> None:
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50,
                    help="timed steps of the headline measurement (value, ms_per_step; --mode slices and --impl "
                         "reference too); the secondary blocks of the default line use fixed counts: e2e "
                         "min(steps, 20) with at least 3, single_mixture and fused_step 20, slice_sharding 20, "
                         "cpu_baseline 5")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="30 s mixtures per GPU per step (Separator.forward takes a batch)")
    ap.add_argument("--mode", default="tracks", choices=["tracks", "slices", "sweep"],
                    help="tracks: every rank demixes its own batch of 30 s mixtures (weak scaling, configs[1]); "
                         "slices: ONE 3-min stereo track sharded by slice range with NCCL halo exchange (strong, configs[3]); "
                         "sweep: --tracks synthetic 3-min stereo tracks dealt round-robin to the GPUs (configs[4])")
    ap.add_argument("--tracks", type=int, default=1024, help="--mode sweep: number of 3-min tracks")
    ap.add_argument("--cpu-sample-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (a fixed sample of the coefficients "
                         "and waveforms, at most 48 MiB) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "tracks"):
        ap.error("--dump-outputs applies to the default workload (--impl b200 --mode tracks)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    binding = bind_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))) if args.impl != "reference" else None
    base_cfg = {"workload": "configs[1]: sliCQT path of a realtime demix of synthetic 30 s 44.1 kHz stereo mixtures "
                            "(per mixture: 1 forward of 2 rows x 148 slices + inverse of 4 targets = 8 rows x 148 slices), "
                            "Bark(262, 32.9 Hz), sllen 18060; one step = one batch of mixtures per GPU, as "
                            "Separator.forward(audio[B,2,T]) processes them",
                "mixtures_per_gpu_per_step": args.batch, "parallelism": f"tracks x{max(world, args.gpus)}",
                "l2": "inputs+outputs of one step (>= 330 MB) exceed the 126 MB L2 and an extra 256 MB buffer is "
                      "written between timed steps"}

    if args.impl == "reference":
        if rank != 0:
            return
        val, dt, cores, sample, kind, done = cpu_reference_arm(args.steps, args.warmup, args.cpu_sample_seconds)
        emit(({
            "impl": "reference", "metric": "sliCQT fwd+inv audio-sec/sec", "value": val, "unit": "audio-s/s",
            "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_cfg,
            "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }))
        return

    if not os.path.exists(os.path.join(ROOT, "xumx_slicq_b200", "libslicq.so")) and rank == 0:
        import __graft_entry__
        __graft_entry__.build()          # fresh checkout: compile the sm_100a library first (nvcc is in the image)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL banners go to stderr: stdout carries ONE JSON line
    import torch
    import torch.distributed as dist
    from xumx_slicq_b200 import NSGTBase, make_filterbanks, _cabi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import io, contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        base = NSGTBase(SCALE["scale"], SCALE["fbins"], SCALE["fmin"], device=dev)
    nsg = base.nsgt
    nsgt, insgt = make_filterbanks(base)
    if args.mode == "slices":
        return bench_slices(args, nsg, dev, rank, world, distributed)
    if args.mode == "sweep":
        return bench_sweep(args, nsg, dev, rank, world, distributed)
    B = args.batch
    S = nsg.n_slices(T)
    rows_f, rows_i = 2 * B, 2 * B * N_TARGETS

    # ---- synthetic inputs, resident in HBM before the timed region
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    x = torch.rand(rows_f, T, device=dev, generator=gen) * 2 - 1
    Cmix = nsg.forward_rows(x)
    # model-output stand-in: [targets*rows, F, S, M] per bucket (targets-major like separator.py:174)
    Y = [torch.cat([c * g for g in GAINS], dim=0).contiguous() for c in Cmix]
    del Cmix
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    plan = nsg.plan(dev)
    stream = torch.cuda.current_stream(dev)

    # preallocated outputs + scratch so that the timed region is kernels only
    slab, Cout = nsg.alloc_coefficients(rows_f, S, dev)
    views_f = [nsg._view_of(c) for c in Cout]
    views_i = [nsg._view_of(c) for c in Y]
    sb_f, sb_i = plan.scratch_bytes(rows_f, S, False), plan.scratch_bytes(rows_i, S, True)
    scratch = torch.empty(max(sb_f, sb_i), dtype=torch.uint8, device=dev)
    yout = torch.empty(rows_i, T, device=dev)

    def step_device():
        plan.forward(x.data_ptr(), rows_f, x.stride(0), T, 0, 0, S, views_f, scratch.data_ptr(), sb_f,
                     stream.cuda_stream)
        plan.inverse(views_i, rows_i, S, 0, yout.data_ptr(), yout.stride(0), T, 0, 0, scratch.data_ptr(), sb_i,
                     stream.cuda_stream)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step_device()
    barrier()

    # ---- timed region: K steps, CUDA events per step on the launching stream, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = plan.launch_count()
    barrier()
    for a, b in ev:
        flush.fill_(1)
        a.record(stream)
        step_device()
        b.record(stream)
    barrier()
    launches = plan.launch_count() - launches0
    clocks = sampler.stop()
    # the passes below reuse Cout and yout: take the timed path's outputs first
    dumped = dump_outputs(args.dump_outputs, Cout, yout) if args.dump_outputs and rank == 0 else None
    step_ms = np.asarray([a.elapsed_time(b) for a, b in ev], dtype=np.float64)
    ms_per_step = float(step_ms.mean())
    t = torch.tensor([ms_per_step], device=dev, dtype=torch.float64)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item())
    n_gpus = world
    audio_s = SECONDS * B * n_gpus
    value = audio_s / (ms_per_step * 1e-3)

    # ---- per-kernel CUDA-event timing (separate pass; event records between kernels are not free).
    #      A second plan without the two-stream row split runs the same step on ONE stream, so that a
    #      kernel's events bracket that kernel alone (with the split the halves overlap and the per-kernel
    #      sums exceed the step).
    os.environ["SLICQ_SPLIT_UNITS"] = "0"
    with contextlib.redirect_stdout(io.StringIO()):
        base1 = NSGTBase(SCALE["scale"], SCALE["fbins"], SCALE["fmin"], device=dev)
    plan1 = base1.nsgt.plan(dev)          # the library reads SLICQ_SPLIT_UNITS when the plan is created
    os.environ.pop("SLICQ_SPLIT_UNITS", None)
    sb1_f, sb1_i = plan1.scratch_bytes(rows_f, S, False), plan1.scratch_bytes(rows_i, S, True)
    scratch1 = torch.empty(max(sb1_f, sb1_i), dtype=torch.uint8, device=dev)

    def step_single_stream():
        plan1.forward(x.data_ptr(), rows_f, x.stride(0), T, 0, 0, S, views_f, scratch1.data_ptr(), sb1_f,
                      stream.cuda_stream)
        plan1.inverse(views_i, rows_i, S, 0, yout.data_ptr(), yout.stride(0), T, 0, 0, scratch1.data_ptr(), sb1_i,
                      stream.cuda_stream)

    step_single_stream()
    torch.cuda.synchronize(dev)
    _cabi.profile_enable(True)
    nprof = 5
    for _ in range(nprof):
        flush.fill_(1)
        step_single_stream()
    torch.cuda.synchronize(dev)
    prof = _cabi.profile_read()
    _cabi.profile_enable(False)
    del scratch1
    units_f, units_i = rows_f * S, rows_i * S
    kern = {}
    alg = {"slice_fft_fwd": B_IN * units_f, "bins_fwd": B_COEF * units_f, "bins_inv": B_COEF * units_i,
           "slice_fft_inv": B_IN * units_i}
    tot_ms = 0.0
    for k, (ms, n) in prof.items():
        per_step = ms / nprof
        tot_ms += per_step
        kern[k] = {"ms_per_step": round(per_step, 4), "launches_per_step": n // nprof,
                   "hbm_bytes_per_step": alg[k]}
    peak, peak_src = load_peaks()
    alg_step = B_UNIT * (units_f + units_i)
    dom = max(kern, key=lambda k: kern[k]["ms_per_step"])
    achieved = alg_step / (ms_per_step * 1e-3) / 1e9
    # DRAM bytes per (row, slice) unit measured by ncu for this build (dram__bytes_read.sum + dram__bytes_write.sum of every
    # launch of one step: profiles/r2_launches.csv -> profiles/r2_dram_traffic.json, regenerated with tools/r2_capture.sh)
    traffic_step, traffic_src = None, "profiles/r2_dram_traffic.json not found"
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")) as f:
            tr = json.load(f)
        traffic_step = int(tr["analysis_dram_bytes_per_unit"] * units_f + tr["synthesis_dram_bytes_per_unit"] * units_i)
        traffic_src = tr["source"]
    except (OSError, KeyError, ValueError):
        pass
    roofline = {
        "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
        "frac": round(achieved / peak, 4), "traffic": traffic_step,
        "traffic_note": "DRAM bytes of one step, per-unit figures of the committed ncu launch list scaled to this step's units "
                        "(the intermediate spectra H / T make a round trip through HBM at the default chunk size); " + traffic_src,
        "scope": "whole path: algorithmic bytes of one step (185 240 B per (row,slice) and direction) / "
                 "CUDA-event time of the step (all five kernels)",
        "peak_source": peak_src, "algorithmic_bytes_per_step": alg_step,
        "dominant_kernel": dom, "kernel_share": {k: round(v["ms_per_step"] / max(tot_ms, 1e-9), 3) for k, v in kern.items()},
        "kernels": kern,
        "kernels_note": "per-kernel times: same step on one stream (no row split), CUDA events around every launch",
    }
    # the dominant kernel alone: its own algorithmic bytes per launch / its average launch duration
    dk = kern[dom]
    dl = max(dk["launches_per_step"], 1)
    d_ach = alg[dom] / (dk["ms_per_step"] * 1e-3) / 1e9
    roofline["dominant"] = {"kernel": dom, "algorithmic_bytes_per_launch": alg[dom] // dl,
                            "avg_launch_ms": round(dk["ms_per_step"] / dl, 4), "achieved": round(d_ach, 1),
                            "frac": round(d_ach / peak, 4)}

    # ---- end to end through the public wrappers with HOST buffers (pinned), every step:
    #      H2D of the mixture, NSGT_SL, target stand-in, INSGT_SL, D2H of the 4 target waveforms
    xh = torch.empty(B, 2, T, dtype=torch.float32).pin_memory()
    xh.copy_(x.view(B, 2, T).cpu())
    yh = torch.empty(N_TARGETS, B, 2, T, dtype=torch.float32).pin_memory()
    gains = torch.tensor(GAINS, device=dev).view(4, 1, 1, 1, 1, 1, 1)

    def step_e2e():
        xd = xh.to(dev, non_blocking=True)
        X = nsgt(xd)
        Yl = [Xb.unsqueeze(0) * gains for Xb in X]          # [4,B,2,F,S,M,2] stand-in for Unmix output
        y = insgt(Yl, T)
        yh.copy_(y, non_blocking=True)

    for _ in range(3):
        step_e2e()
    barrier()
    e_steps = max(3, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(e_steps):
        step_e2e()
    torch.cuda.synchronize(dev)
    seq_ms = (time.perf_counter() - t0) / e_steps * 1e3
    # the same work through TransformStream: H2D(i+1) / kernels(i) / D2H(i-1) on three streams
    from xumx_slicq_b200.pipeline import TransformStream
    ts = TransformStream(base, lambda X: [Xb.unsqueeze(0) * gains for Xb in X], dev)
    for _ in ts.process(xh for _ in range(3)):
        pass
    barrier()
    t0 = time.perf_counter()
    n_out = 0
    for yo in ts.process(xh for _ in range(e_steps)):
        n_out += 1
    torch.cuda.synchronize(dev)
    barrier()
    e_ms = (time.perf_counter() - t0) / e_steps * 1e3
    assert n_out == e_steps
    e2e_err = float((yo[0].to(dev) - GAINS[0] * x.view(B, 2, T)).abs().max())
    te = torch.tensor([e_ms], device=dev, dtype=torch.float64)
    if distributed:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e_ms = float(te.item())
    # ---- what the host side of this box allows: the same bytes per step as plain pinned copies (H2D and D2H on two
    #      streams, no kernels), all ranks at once -- the ceiling of any end-to-end number at this N
    yd_c = torch.empty(N_TARGETS, B, 2, T, dtype=torch.float32, device=dev)
    s_h2d, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def copies_only():
        with torch.cuda.stream(s_h2d):
            xh.to(dev, non_blocking=True)
        with torch.cuda.stream(s_d2h):
            yh.copy_(yd_c, non_blocking=True)
    for _ in range(3):
        copies_only()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e_steps):
        copies_only()
    torch.cuda.synchronize(dev)
    barrier()
    c_ms = (time.perf_counter() - t0) / e_steps * 1e3
    tc = torch.tensor([c_ms], device=dev, dtype=torch.float64)
    if distributed:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    c_ms = float(tc.item())
    del yd_c
    e2e = {"value": audio_s / (e_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": e_ms,
           "host_copy_ceiling": {"value": audio_s / (c_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": c_ms,
                                 "what": "pinned H2D + D2H of the same byte counts on two streams, no kernels, all ranks concurrently",
                                 "gbytes_per_s_per_gpu": round((xh.numel() + yh.numel()) * 4 / (c_ms * 1e-3) / 1e9, 1)},
           "frac_of_host_copy_ceiling": round(c_ms / e_ms, 3), "host_binding": binding,
           "h2d_bytes_per_step": int(xh.numel() * 4), "d2h_bytes_per_step": int(yh.numel() * 4),
           "includes": "every step: pinned H2D of the mixtures, NSGT_SL, 4-target gain stand-in (torch), INSGT_SL, "
                       "pinned D2H of the 4 target waveforms; xumx_slicq_b200.pipeline.TransformStream overlaps the "
                       "copies of neighbouring steps with the kernels (wall clock over all steps)",
           "sequential_ms_per_step": seq_ms, "max_abs_err_target0": e2e_err}

    # ---- quality guard: the timed path really reconstructs (gain g of target t times the mixture)
    err = float((yout[:rows_f] - GAINS[0] * x).abs().max())

    # ---- the same path for ONE mixture per step (latency view of configs[1]; launch-bound)
    single = None
    if world == 1 and B != 1:
        x1 = x[:2]
        Y1 = [torch.cat([c[2 * B * t: 2 * B * t + 2] for t in range(N_TARGETS)], 0).contiguous() for c in Y]
        slab1, C1 = nsg.alloc_coefficients(2, S, dev)
        vf1, vi1 = [nsg._view_of(c) for c in C1], [nsg._view_of(c) for c in Y1]
        s1f, s1i = plan.scratch_bytes(2, S, False), plan.scratch_bytes(2 * N_TARGETS, S, True)
        y1 = torch.empty(2 * N_TARGETS, T, device=dev)

        def step1():
            plan.forward(x1.data_ptr(), 2, x1.stride(0), T, 0, 0, S, vf1, scratch.data_ptr(), s1f, stream.cuda_stream)
            plan.inverse(vi1, 2 * N_TARGETS, S, 0, y1.data_ptr(), y1.stride(0), T, 0, 0, scratch.data_ptr(), s1i,
                         stream.cuda_stream)
        for _ in range(3):
            step1()
        torch.cuda.synchronize(dev)
        n1 = 20
        ev1 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n1)]
        for a, b in ev1:
            flush.fill_(1)
            a.record(stream); step1(); b.record(stream)
        torch.cuda.synchronize(dev)
        ms1 = float(np.mean([a.elapsed_time(b) for a, b in ev1]))
        single = {"mixtures_per_step": 1, "ms_per_step": ms1, "value": SECONDS / (ms1 * 1e-3), "unit": "audio-s/s",
                  "roofline_frac": round(B_UNIT * (2 + 2 * N_TARGETS) * S / (ms1 * 1e-3) / 1e9 / peak, 4)}
        # the same step captured once into a CUDA graph (kernels + the fork/join of the two internal streams) and replayed
        try:
            gs = torch.cuda.Stream(device=dev)
            gs.wait_stream(stream)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=gs):
                cs = torch.cuda.current_stream(dev).cuda_stream
                plan.forward(x1.data_ptr(), 2, x1.stride(0), T, 0, 0, S, vf1, scratch.data_ptr(), s1f, cs)
                plan.inverse(vi1, 2 * N_TARGETS, S, 0, y1.data_ptr(), y1.stride(0), T, 0, 0, scratch.data_ptr(), s1i, cs)
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize(dev)
            evg = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n1)]
            for a, b in evg:
                flush.fill_(1)
                a.record(stream); graph.replay(); b.record(stream)
            torch.cuda.synchronize(dev)
            single["graph_ms_per_step"] = float(np.mean([a.elapsed_time(b) for a, b in evg]))
        except Exception as e:                      # informational only
            single["graph_error"] = str(e)[:200]

    # ---- the fused variant of the same step (SURVEY 8f N1 / row A10): forward that also writes |X|, inverse that
    #      reads the mixture coefficients + 4 fp32 masks instead of 4 materialised target coefficient sets
    fused = None
    if world == 1:
        del Y
        torch.cuda.empty_cache()
        nslab, Nout = nsg.alloc_norms(rows_f, S, dev)
        masks = [torch.full((rows_i,) + tuple(c.shape[1:]), 1.0, device=dev) for c in Cout]
        for m in masks:                              # mask of target t = its gain: same waveforms as the plain step
            for t_, g_ in enumerate(GAINS):
                m[t_ * rows_f:(t_ + 1) * rows_f] = g_
        views_m = [(m.data_ptr(), m.stride(0), m.stride(1), m.stride(2)) for m in masks]
        sbm = plan.scratch_bytes(rows_i, S, True)
        scr_m = scratch if sbm <= scratch.numel() else torch.empty(sbm, dtype=torch.uint8, device=dev)

        def step_fused():
            plan.forward_packed_norm(x.data_ptr(), rows_f, x.stride(0), T, 0, 0, S, slab.data_ptr(), nslab.data_ptr(),
                                     scr_m.data_ptr(), sb_f, stream.cuda_stream)
            plan.inverse_masked(views_f, views_m, N_TARGETS, rows_f, S, 0, yout.data_ptr(), yout.stride(0), T, 0, 0,
                                scr_m.data_ptr(), sbm, stream.cuda_stream)
        for _ in range(3):
            step_fused()
        torch.cuda.synchronize(dev)
        nfu = 20
        evf = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nfu)]
        for a, b in evf:
            flush.fill_(1)
            a.record(stream); step_fused(); b.record(stream)
        torch.cuda.synchronize(dev)
        msf = float(np.mean([a.elapsed_time(b) for a, b in evf]))
        ferr = float((yout[:rows_f] - GAINS[0] * x).abs().max())
        # algorithmic bytes of the fused step (SURVEY 8d): fwd 185 240 + 4 * 18 640 (|X|), inverse 18 640 * (8 + 4*4) + 4 * 36 120
        fb = (B_UNIT + 4 * 18640) * units_f + (18640 * (8 + 4 * N_TARGETS) + N_TARGETS * B_IN) * units_f
        fused = {"ms_per_step": msf, "value": audio_s / (msf * 1e-3), "unit": "audio-s/s",
                 "what": "forward_with_norm (coefficients + |X|) + inverse_masked (mixture + 4 fp32 masks -> 4 target waveforms)",
                 "algorithmic_bytes_per_step": int(fb), "roofline_frac": round(fb / (msf * 1e-3) / 1e9 / peak, 4),
                 "max_abs_err_target0": ferr}
        del masks, nslab

    # ---- configs[3] beside the headline when there is more than one GPU: one 3-min track sharded by slice range over NCCL
    shard = None
    if distributed:
        del Y, Cout, slab, scratch, yout
        torch.cuda.empty_cache()
        shard = slice_sharding_run(nsg, dev, rank, world, 20, 3)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, cores, sample, kind, _ = cpu_reference_arm(5, 1, args.cpu_sample_seconds)
        cpu = {"value": v, "unit": "audio-s/s", "cores": cores, "kind": kind, "sample": sample,
               "ms_per_sample": dt * 1e3}

    if rank == 0:
        line = {
            "metric": "sliCQT fwd+inv audio-sec/sec", "value": value, "unit": "audio-s/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": base_cfg,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "single_mixture": single, "fused_step": fused,
            "slice_sharding": shard,
            "gpu_launches": int(launches),
            "clocks": clocks, "max_abs_err_target0": err,
        }
        if dumped is not None:
            line["dumped_outputs"] = {"dir": args.dump_outputs, "shapes": dumped}
        emit(line)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

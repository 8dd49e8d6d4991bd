#!/usr/bin/env python
"""Inference throughput on a file set of mixed lengths: the per-file loop against ragged batches.

    python tools/bench_ragged.py [--files 240] [--rounds 3] [--seed 0] [--out profiles] [--tag r3_ragged]

Workload: a seeded synthetic set of ``--files`` clips whose lengths are drawn uniformly from 2.1 - 9.8 s (the range of the reference's 25
AudioSamples), 16 kHz, already in GPU memory (no wav I/O is timed).  TSCNet has seeded random weights (the weights do not change the work).
Paths, all eager as a user calls them, tf32 mode:
  per_file       signal.enhance on every clip (B = 1 forward passes: what evaluation() did per file)
  ragged_b{N}    signal.plan_ragged(max_batch = N) + signal.enhance_ragged per batch, N = 4, 8, 16, 32
Every path is warmed up once over the whole set; then ``--rounds`` rounds time the paths alternately, each pass from a device synchronise
to a device synchronise.  Reported per path: files/s and audio-seconds/s (median over rounds), the fraction of padded frames, and from a
separate instrumented pass the mean host time until a call returns and the mean wall time until its GPU work is done (the host cost per
call).  The GPU name and power limit are read in the same run.  Writes <out>/<tag>.json and <out>/<tag>.md.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SR = 16000
BATCHES = (4, 8, 16, 32)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        pl, mhz = [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(mhz)
    except Exception as e:          # the numbers are still reported, without the power limit
        info["error"] = str(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=240)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--tag", default="r3_ragged_inference")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged.py measures the GPU path and needs a CUDA device")

    import cmgan_b200
    from cmgan_b200 import ops, signal
    ops.set_precision("tf32")
    dev = torch.device("cuda", 0)
    torch.manual_seed(args.seed)
    model = cmgan_b200.TSCNet(64, 201).to(dev).eval()
    rng = np.random.default_rng(args.seed)
    lengths = [int(v) for v in rng.integers(int(2.1 * SR), int(9.8 * SR) + 1, size=args.files)]
    waves = [torch.from_numpy((rng.standard_normal(n) * 0.05).astype(np.float32)).to(dev) for n in lengths]
    audio_s = sum(lengths) / SR

    plans = {f"ragged_b{n}": signal.plan_ragged(lengths, max_batch=n)[0] for n in BATCHES}

    def padded_fraction(batches):
        valid = sum(signal.clip_frames(lengths[i]) for b in batches for i in b)
        total = sum(len(b) * max(signal.clip_frames(lengths[i]) for i in b) for b in batches)
        return 1.0 - valid / total

    def run_per_file():
        return [signal.enhance(model, w[None]) for w in waves]

    def make_ragged(batches):
        def run():
            return [signal.enhance_ragged(model, [waves[i] for i in b]) for b in batches]
        return run

    paths = {"per_file": run_per_file}
    paths.update({k: make_ragged(v) for k, v in plans.items()})
    calls = {"per_file": len(waves), **{k: len(v) for k, v in plans.items()}}

    with torch.no_grad():
        for fn in paths.values():              # warm-up: every shape, the weight cache, the allocator
            fn()
        torch.cuda.synchronize()
        times = {k: [] for k in paths}
        for _ in range(args.rounds):
            for k, fn in paths.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                times[k].append(time.perf_counter() - t0)
        # instrumented pass: host time until each call returns vs wall time until its GPU work is done
        host = {}
        for k in paths:
            units = [[i] for i in range(len(waves))] if k == "per_file" else plans[k]
            h, w = [], []
            for b in units:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if k == "per_file":
                    signal.enhance(model, waves[b[0]][None])
                else:
                    signal.enhance_ragged(model, [waves[i] for i in b])
                t1 = time.perf_counter()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                h.append(t1 - t0)
                w.append(t2 - t0)
            host[k] = (1e3 * statistics.mean(h), 1e3 * statistics.mean(w))
    info = gpu_info()

    res = {"gpu": info, "precision": "tf32", "files": len(waves), "audio_seconds": audio_s, "seed": args.seed, "rounds": args.rounds,
           "length_range_s": [min(lengths) / SR, max(lengths) / SR], "paths": {}}
    base = None
    for k in paths:
        med = statistics.median(times[k])
        d = {"seconds_median": med, "seconds_all": times[k], "files_per_s": len(waves) / med, "audio_s_per_s": audio_s / med,
             "calls": calls[k], "host_ms_per_call": host[k][0], "wall_ms_per_call": host[k][1],
             "padded_frame_fraction": 0.0 if k == "per_file" else padded_fraction(plans[k])}
        if base is None:
            base = med
        d["speedup_vs_per_file"] = base / med
        res["paths"][k] = d
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, args.tag + ".json"), "w") as fh:
        json.dump(res, fh, indent=1)
    lines = [f"# Ragged-batch inference vs the per-file loop ({info['name']}, power limit {info['power_limit_w']} W)", "",
             f"{len(waves)} synthetic clips, {min(lengths) / SR:.1f} - {max(lengths) / SR:.1f} s (seed {args.seed}), {audio_s:.0f} s of audio, "
             f"tf32, eager; median of {args.rounds} alternated rounds, each from a device synchronise to a device synchronise. "
             "Host ms / wall ms per call: mean time until the call returns / until its GPU work is done (separate pass).", "",
             "| path | files/s | audio s/s | vs per-file | padded frames | calls | host ms/call | wall ms/call |",
             "|---|---|---|---|---|---|---|---|"]
    for k, d in res["paths"].items():
        lines.append(f"| {k} | {d['files_per_s']:.1f} | {d['audio_s_per_s']:.0f} | {d['speedup_vs_per_file']:.2f}x | "
                     f"{100 * d['padded_frame_fraction']:.1f} % | {d['calls']} | {d['host_ms_per_call']:.1f} | {d['wall_ms_per_call']:.1f} |")
    with open(os.path.join(args.out, args.tag + ".md"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()

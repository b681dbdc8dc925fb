"""Tracking many sequences: ope_pose_tracker_step_batch against the serial loop of ope_pose_estimate_final_device.

S sequences x F frames (synth.make_sequence, distinct scenes, rendered before any timing). Every step is one batched call over the
S trackers; the serial loop runs the same frames of the first --serial sequences one tracker call at a time. Reports frames/s of
both, how many trackers re-ran SAC-IA or tracked at each step, and the commit kernel's algorithmic bytes (3 reads + 2 writes of
16 B per point and tracker) over its device time (torch.profiler, a separate pass) against 7.7 TB/s, with the card's name and
power limit read in the same run. Usage: python tools/bench_track_batch.py [--sizes 256 1024] [--frames 4] [--out file.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from multiprocessing import Pool

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ope_pkg  # noqa: E402

ope_pkg.load()
from ope_b200 import cuda_lib, synth  # noqa: E402

_MODEL = None


def _seq(args):
    s, frames = args
    return [f[0] for f in synth.make_sequence(_MODEL, 1000 + s, frames)]


def _init(model):
    global _MODEL
    _MODEL = model


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers are still reported, marked as unattributed
        return "unknown (%s)" % e, "unknown"


def run_batch(ctx, model, seqs, frames):
    trackers = [cuda_lib.PoseTracker(ctx) for _ in seqs]
    sources = [ctx.upload(model) for _ in seqs]
    split, times = [], []
    for k in range(frames):
        ctx.synchronize()
        t0 = time.perf_counter()
        res, st = ctx.pose_track_batch(trackers, sources, [s[k] for s in seqs])
        ctx.synchronize()
        times.append(time.perf_counter() - t0)
        split.append({"recoarse": int(sum(r.ran_coarse for r in res)), "track": int(sum(1 - r.ran_coarse for r in res)),
                      "failed": int((st != 0).sum())})
    return trackers, sources, split, times


def commit_share(ctx, model, seqs):
    import torch
    from torch.profiler import ProfilerActivity, profile
    trackers = [cuda_lib.PoseTracker(ctx) for _ in seqs]
    sources = [ctx.upload(model) for _ in seqs]
    ctx.pose_track_batch(trackers, sources, [s[0] for s in seqs])
    ctx.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.pose_track_batch(trackers, sources, [s[1] for s in seqs])
        ctx.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "track_commit_kernel" in e.key)
    byts = 5 * 16 * len(model) * len(seqs)
    for t in trackers:
        t.close()
    torch.cuda.synchronize()
    return byts, us * 1e-6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--serial", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    model = synth.make_model()
    S = max(a.sizes)
    with Pool(min(os.cpu_count() or 1, 32), initializer=_init, initargs=(model,)) as pool:
        seqs = pool.map(_seq, [(s, a.frames) for s in range(S)])
    ctx = cuda_lib.Context()
    name, power = card()
    out = {"card": name, "power_limit": power, "frames_per_sequence": a.frames, "sizes": {}}
    run_batch(ctx, model, seqs[:32], 2)   # warm-up: module loads, worker contexts, pools
    for n in a.sizes:
        _, _, split, times = run_batch(ctx, model, seqs[:n], a.frames)
        out["sizes"][str(n)] = {"frames_per_s": n * a.frames / sum(times), "step_s": times, "split": split}
    # the serial loop on the first sequences of the same set
    trackers = [cuda_lib.PoseTracker(ctx) for _ in range(a.serial)]
    sources = [ctx.upload(model) for _ in range(a.serial)]
    t0 = time.perf_counter()
    for k in range(a.frames):
        for i in range(a.serial):
            tg = ctx.upload(seqs[i][k])
            trackers[i].estimate_final_device(sources[i], tg)
            tg.free()
    ctx.synchronize()
    out["serial_frames_per_s"] = a.serial * a.frames / (time.perf_counter() - t0)
    for n in a.sizes:
        out["sizes"][str(n)]["speedup_vs_serial"] = out["sizes"][str(n)]["frames_per_s"] / out["serial_frames_per_s"]
    byts, sec = commit_share(ctx, model, seqs[:min(S, 256)])
    out["commit_kernel"] = {"trackers": min(S, 256), "bytes": byts, "device_s": sec,
                            "tb_per_s": byts / sec / 1e12 if sec > 0 else None,
                            "share_of_7_7_tb_s": byts / sec / 7.7e12 if sec > 0 else None}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

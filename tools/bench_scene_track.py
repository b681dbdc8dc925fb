"""Many cameras, each giving a depth image per tick: ope_scene_track_step (scene batch -> cluster choice -> tracker step in one call)
against the host-side composition of the calls it replaces.

N cameras x F frames (synth.make_scene_sequence with two distractors; every 8th object jumps 12 cm at frame 2; --distinct
sequences rendered before any timing and tiled over the cameras), the depth stack of each tick resident on the device. Per tick:
ope_scene_batch_create, then ope_scene_track_step (--accept-fitness / --accept-strength: the reference's 1e-4 / 0.4 by default). Reports ms per tick for the scene, the
centroids + gate, each round and the commit (host wall time of phases that each end synchronised), frames/s, the histogram of
modes and tries, the centroid_chain_kernel's device time (torch.profiler, a separate pass) and the wall time of ope_cloud_centroid
on the 157 825-point model, and the same frames through the host-side composition (download every frame's cropped cloud and
labels, centroids and gate in numpy, cut on the host, one ope_pose_tracker_step_batch per round with host targets), with the card's
name and power limit read in the same run. Usage: python tools/bench_scene_track.py [--sizes 256 1024] [--frames 4] [--out f.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time
from collections import Counter
from multiprocessing import Pool

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ope_pkg  # noqa: E402

ope_pkg.load()
from ope_b200 import cuda_lib, synth  # noqa: E402

T = cuda_lib.T
_MODEL = None
GATE = np.float32(0.05)


def _seq(args):
    s, frames = args
    d, _ = synth.make_scene_sequence(_MODEL, 2000 + s, frames, jump_at=2 if s % 8 == 7 else None)
    return d


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


def _sync(ctx):
    import torch
    ctx.synchronize()
    torch.cuda.synchronize()


def run_one_call(ctx, model, ticks, n, tp):
    """ticks: per frame a device tensor (n, 480, 640). Returns per tick the phase times and the choices."""
    trackers = [cuda_lib.PoseTracker(ctx) for _ in range(n)]
    sources = [ctx.upload(model) for _ in range(n)]
    rows = []
    for d in ticks:
        _sync(ctx)
        t0 = time.perf_counter()
        sb = ctx.scene_batch(d)
        t1 = time.perf_counter()
        _, ch, st = sb.track(trackers, sources, **tp)
        t2 = time.perf_counter()
        ph = ctx.track_phase_ms()
        rows.append({"scene_ms": (t1 - t0) * 1e3, "track_ms": (t2 - t1) * 1e3, "gate_ms": ph["gate"], "rounds_ms": ph["rounds"],
                     "commit_ms": ph["commit"], "modes": dict(Counter(T.TRACK_MODES[c.mode] for c in ch)),
                     "tries": dict(Counter(str(c.tries) for c in ch)), "failed": int((st != 0).sum())})
        sb.close()
    for t in trackers:
        t.close()
    return rows


def _centroid(p):
    return np.array([np.cumsum(p[:, a], dtype=np.float32)[-1] / np.float32(len(p)) for a in range(3)], np.float32)


def run_composition(ctx, model, ticks, n, tp):
    """the same frames through the calls the one call replaces; returns per tick the wall ms"""
    trackers = [cuda_lib.PoseTracker(ctx) for _ in range(n)]
    sources = [ctx.upload(model) for _ in range(n)]
    found = [False] * n
    out = []
    for d in ticks:
        _sync(ctx)
        t0 = time.perf_counter()
        sb = ctx.scene_batch(d)
        frames = [sb.frame(f) for f in range(n)]                                  # download: cropped cloud + labels
        cut = [lambda r, f=f: frames[f][0] if sb.info[f].n_clusters < 0 else frames[f][0][frames[f][1] == r] for f in range(n)]
        K = [0 if sb.status[f] != 0 else (1 if sb.info[f].n_clusters < 0 else sb.info[f].n_clusters) for f in range(n)]
        chosen, search = {}, {}
        for i in range(n):
            if found[i]:
                m = _centroid(sources[i].download())
                for k in range(K[i]):
                    c = _centroid(cut[i](k))
                    dx, dy, dz = (np.float32(c[a]) - m[a] for a in range(3))
                    if np.sqrt(np.float32((dx * dx + dy * dy) + dz * dz)) < GATE:
                        chosen[i] = k
                        break
                if i in chosen:
                    continue
            if K[i]:
                search[i] = K[i]
        r = 0
        while True:
            ent = [(i, None, trackers[i], sources[i], cut[i](chosen[i])) for i in range(n) if r == 0 and i in chosen]
            ent += [(i, r, cuda_lib.PoseTracker(ctx), ctx.upload(model), cut[i](r)) for i in range(n) if i in search]
            ent.sort(key=lambda e: e[0])
            if not ent:
                break
            res, st = ctx.pose_track_batch([e[2] for e in ent], [e[3] for e in ent], [e[4] for e in ent])
            for (i, rank, t, s, _), o, c in zip(ent, res, st):
                if rank is None:
                    sources[i] = s
                elif c == 0 and (o.fitness < tp["accept_fitness"] or o.align_strength > tp["accept_strength"]):
                    trackers[i].close()
                    trackers[i], sources[i], found[i] = t, s, True
                    del search[i]
                else:
                    t.close()
                    if rank + 1 >= search[i]:
                        del search[i]
            r += 1
        for i in chosen:
            found[i] = True
        _sync(ctx)
        out.append((time.perf_counter() - t0) * 1e3)
        sb.close()
    for t in trackers:
        t.close()
    return out


def centroid_kernel(ctx, model, ticks, n, tp):
    """device time of centroid_chain_kernel in one steady-state call, and the wall time of ope_cloud_centroid on the model"""
    from torch.profiler import ProfilerActivity, profile
    trackers = [cuda_lib.PoseTracker(ctx) for _ in range(n)]
    sources = [ctx.upload(model) for _ in range(n)]
    sb = ctx.scene_batch(ticks[0])
    sb.track(trackers, sources, **tp)
    sb.close()
    sb = ctx.scene_batch(ticks[1])
    _sync(ctx)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sb.track(trackers, sources, **tp)
        _sync(ctx)
    ev = [e for e in prof.key_averages() if "centroid_chain_kernel" in e.key]
    sb.close()
    src = ctx.upload(model)
    walls = []
    for _ in range(21):
        t0 = time.perf_counter()
        ctx.centroid(src)
        walls.append((time.perf_counter() - t0) * 1e3)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.centroid(src)
        _sync(ctx)
    one = [e for e in prof.key_averages() if "centroid_chain_kernel" in e.key]
    for t in trackers:
        t.close()
    return {"cameras": n, "launches_in_call": int(sum(e.count for e in ev)), "device_ms_in_call": sum(e.device_time_total for e in ev) * 1e-3,
            "model_points": len(model), "model_device_ms": sum(e.device_time_total for e in one) * 1e-3,
            "model_call_wall_ms_median": float(np.median(walls))}


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--distinct", type=int, default=128)
    ap.add_argument("--accept-fitness", type=float, default=1e-4)
    ap.add_argument("--accept-strength", type=float, default=0.4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    tp = {"accept_fitness": a.accept_fitness, "accept_strength": a.accept_strength}
    model = synth.make_model()
    with Pool(min(os.cpu_count() or 1, 32), initializer=_init, initargs=(model,)) as pool:
        seqs = pool.map(_seq, [(s, a.frames) for s in range(a.distinct)])
    ctx = cuda_lib.Context()
    name, power = card()
    out = {"card": name, "power_limit": power, "frames_per_camera": a.frames, "distinct_sequences": a.distinct, "track_params": tp, "sizes": {}}
    libc = ctypes.CDLL(None)

    def ticks_for(n):
        return [torch.from_numpy(np.stack([seqs[c % a.distinct][k] for c in range(n)]).astype(np.int16)).cuda().contiguous()
                for k in range(a.frames)]

    run_one_call(ctx, model, ticks_for(16), 16, tp)   # warm-up: module loads, worker contexts, pools
    for n in a.sizes:
        ticks = ticks_for(n)
        libc.srand(1)
        rows = run_one_call(ctx, model, ticks, n, tp)
        libc.srand(1)
        comp = run_composition(ctx, model, ticks, n, tp)
        one = sum(r["scene_ms"] + r["track_ms"] for r in rows)
        out["sizes"][str(n)] = {"frames_per_s": n * a.frames / one * 1e3, "ticks": rows, "composition_tick_ms": comp,
                                "composition_frames_per_s": n * a.frames / sum(comp) * 1e3, "speedup_vs_composition": sum(comp) / one}
        del ticks
        torch.cuda.empty_cache()
    out["centroid_kernel"] = centroid_kernel(ctx, model, ticks_for(min(a.sizes)), min(a.sizes), tp)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Depth images -> segmented scenes -> poses, many frames per call (ope_scene_batch_create + ope_scene_pose_batch).

    python tools/bench_depth_pose.py [--out FILE.json] [--unique 64]

The full record goes to --out when given (profiles/r03_a_depth_pose.json is one); without it, to stdout. A summary line is
printed either way.

Frames are 640x480 uint16 depth images of synth.make_frame scenes (depth = rint(z * 1000), as tests/test_gpu_parity.py::_depth_mm);
`--unique` distinct scenes are rendered and tiled to 256 and 1024 frames (rendering is host work). Measured with CUDA events:
  * scene preparation from device-resident depth, ms per frame, at 256 and 1024 frames;
  * the same frames through the single-frame calls (ope_depth_to_cloud -> ope_pass_through -> ope_segment_objects_on_plane);
  * end to end from host uint16 (614 KB H2D per frame) through ope_scene_pose_batch on cluster 0, frames/s;
  * per full-frame launch (torch.profiler, a run of its own): algorithmic bytes over kernel time, share of 7.7 TB/s;
  * the sizes of the clusters handed on (and how many exceed the pose batch's 1 cm capacity); parity with the single-frame path
    on every frame and with the oracle on a sample.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
LIMITS = (-0.5, 0.5, -0.5, 0.3, 0.5, 1.6)
HBM_BYTES_PER_S = 7.7e12


def depth_mm(cloud):
    return np.rint(np.nan_to_num(cloud[..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown (nvidia-smi failed)"


def timed(torch, stream, fn, reps):
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = fn()
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
        if hasattr(out, "close"):
            out.close()
    return float(np.median(ms)), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the full JSON record here (default: print it)")
    ap.add_argument("--unique", type=int, default=64)
    ap.add_argument("--sizes", default="256,1024")
    a = ap.parse_args()
    import torch
    import ope_pkg
    ope_pkg.load()
    from ope_b200 import cuda_lib, synth
    import orc_py
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = cuda_lib.Context(0, stream.cuda_stream)
    model = synth.make_model(157825)
    t0 = time.perf_counter()
    base = np.stack([depth_mm(synth.make_frame(model, 5000 + f)[1]) for f in range(a.unique)])
    render_s = time.perf_counter() - t0
    sizes = [int(s) for s in a.sizes.split(",")]
    out = {"card": card(), "workload": "640x480 uint16 depth of synth.make_frame scenes 5000..%d, tiled to %s frames" % (5000 + a.unique - 1, sizes),
           "render_s": render_s, "scene_preparation": {}, "end_to_end": {}}

    # ---- scene preparation from device-resident depth ----
    for n in sizes:
        stack = np.ascontiguousarray(base[np.arange(n) % a.unique])
        dev = torch.from_numpy(stack.astype(np.int16)).cuda().contiguous()
        torch.cuda.synchronize()
        ctx.scene_batch(dev).close()                                    # warm-up: pools, module load
        t, all_ms = timed(torch, stream, lambda: ctx.scene_batch(dev), 3)
        out["scene_preparation"][str(n)] = {"ms_per_frame": t / n, "frames_per_sec": 1e3 * n / t, "call_ms": all_ms}
        # end to end from host uint16: H2D + scene preparation + the pose batch on cluster 0
        sb = ctx.scene_batch(stack)
        sb.pose(model)
        sb.close()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        h0 = time.perf_counter()
        sb = ctx.scene_batch(stack)
        e_mid = torch.cuda.Event(enable_timing=True)
        e_mid.record(stream)
        res, st = sb.pose(model)
        e1.record(stream)
        e1.synchronize()
        wall = time.perf_counter() - h0
        sizes0 = np.array([r.n_tgt_coarse for r in res])
        out["end_to_end"][str(n)] = {"ms": e0.elapsed_time(e1), "frames_per_sec": 1e3 * n / e0.elapsed_time(e1), "host_wall_s": wall,
                                     "scene_ms": e0.elapsed_time(e_mid), "pose_ms": e_mid.elapsed_time(e1), "status_ok": int((st == 0).sum()),
                                     # frames beyond the frame-spanning launches' 1 cm capacity: they take the per-frame path
                                     "frames_over_2048_at_1cm": int((sizes0 > 2048).sum())}
        if n == sizes[-1]:
            cl = np.array([sb.info[f].n_clusters for f in range(n)])
            c0 = np.array([(sb.frame(f)[1] == 0).sum() if cl[f] > 0 else 0 for f in range(a.unique)])
            out["clusters"] = {"n_clusters_histogram": {str(k): int((cl == k).sum()) for k in np.unique(cl)},
                               "cluster0_points_percentiles_5_50_95": [float(np.percentile(c0, q)) for q in (5, 50, 95)],
                               "cluster0_points_mean": float(c0.mean()),
                               "target_1cm_sample_points_percentiles_5_50_95": [float(np.percentile(sizes0, q)) for q in (5, 50, 95)]}
        sb.close()
        del dev

    # ---- the same frames through the single-frame calls ----
    def single(d):
        c = ctx.depth_to_cloud(d)
        f = ctx.pass_through(c, LIMITS)
        r = ctx.segment_objects_on_plane(f)
        return c, f, r
    single(base[0])
    t, _ = timed(torch, stream, lambda: [single(base[f]) for f in range(a.unique)], 2)
    out["single_frame_calls"] = {"ms_per_frame": t / a.unique, "frames": a.unique}
    out["speedup_at_%d" % sizes[-1]] = out["single_frame_calls"]["ms_per_frame"] / out["scene_preparation"][str(sizes[-1])]["ms_per_frame"]

    # ---- parity: every unique frame vs the single-frame path, a sample vs the oracle ----
    sb = ctx.scene_batch(base)
    same = 0
    for f in range(a.unique):
        c, filt, (labels, k, p1, p2, it) = single(base[f])
        xyz, bl = sb.frame(f)
        i = sb.info[f]
        same += int(i.n_points == len(c) and np.array_equal(xyz, filt.download()) and np.array_equal(bl, labels) and i.n_clusters == k
                    and np.array_equal(np.array(list(i.plane1), np.float32), p1) and np.array_equal(np.array(list(i.plane2), np.float32), p2)
                    and (i.iterations[0], i.iterations[1]) == tuple(it))
    oracle_same = 0
    sample = list(range(0, a.unique, max(1, a.unique // 4)))[:4]
    for f in sample:
        pts = orc_py.depth_to_cloud(base[f])
        keep = np.arange(len(pts), dtype=np.int32)
        for field, lo, hi in ((2, LIMITS[4], LIMITS[5]), (1, LIMITS[2], LIMITS[3]), (0, LIMITS[0], LIMITS[1])):
            keep = keep[orc_py.pass_through(pts[keep], field, lo, hi)]
        ol, ok, op1, op2, oit = orc_py.segment_objects_on_plane(pts[keep])
        xyz, bl = sb.frame(f)
        oracle_same += int(np.array_equal(xyz, pts[keep]) and np.array_equal(bl, ol) and sb.info[f].n_clusters == ok)
    out["parity"] = {"frames_equal_to_single_frame_path": same, "frames": a.unique, "oracle_sample": sample, "oracle_equal": oracle_same,
                     "ok": same == a.unique and oracle_same == len(sample)}
    n_cropped = np.array([sb.info[f].n_cropped for f in range(a.unique)])
    n_points = np.array([sb.info[f].n_points for f in range(a.unique)])
    n_prism = np.array([(sb.frame(f)[1] != -3).sum() if sb.info[f].n_clusters >= 0 else 0 for f in range(a.unique)])
    sb.close()

    # ---- per full-frame launch: torch.profiler over one call at the largest size (a run of its own) ----
    n = sizes[-1]
    idx = np.arange(n) % a.unique
    dev = torch.from_numpy(np.ascontiguousarray(base[idx]).astype(np.int16)).cuda().contiguous()
    torch.cuda.synchronize()
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.scene_batch(dev).close()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            k = kern.setdefault(e.name, [0, 0.0])
            k[0] += 1
            k[1] += e.time_range.elapsed_us() / 1e3
    px = n * 480 * 640
    pts, crop, prism = int(n_points[idx].sum()), int(n_cropped[idx].sum()), int(n_prism[idx].sum())
    algorithmic = {   # bytes the kernel has to move at least: its inputs read once, its outputs written once
        "depth_fused_kernel": 2 * px + 16 * pts,
        "pass_flag_kernel": 16 * pts + 4 * pts,
        "plane_count_kernel": 16 * crop + 16 * prism,     # two launches: the table plane over the crop, the second over the prism
        "prism_flag_kernel": 16 * crop + 4 * crop,
    }
    launches = {}
    for name, b in algorithmic.items():
        hit = [(k, v) for k, v in kern.items() if name in k]
        if not hit:
            continue
        cnt = sum(v[0] for _, v in hit)
        ms = sum(v[1] for _, v in hit)
        launches[name] = {"launches": cnt, "kernel_ms": ms, "algorithmic_bytes": b, "algorithmic_GB_per_s": b / (ms * 1e-3) / 1e9,
                          "share_of_7_7_TB_per_s": b / (ms * 1e-3) / HBM_BYTES_PER_S}
    total_ms = sum(v[1] for v in kern.values())
    out["full_frame_launches_%d_frames" % n] = {"note": "algorithmic figures: bytes the launch must move over its kernel time (torch.profiler)",
                                                "kernels": launches}
    out["kernel_time_by_name_ms_%d_frames" % n] = {k: round(v[1], 4) for k, v in sorted(kern.items(), key=lambda kv: -kv[1][1])[:16]}
    out["kernel_time_total_ms_%d_frames" % n] = total_ms
    out["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    else:
        print(json.dumps(out))
    print(json.dumps({k: out[k] for k in ("card", "scene_preparation", "single_frame_calls", "end_to_end", "parity")}))
    ctx.close()


if __name__ == "__main__":
    main()

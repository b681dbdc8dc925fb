"""Normal estimation beyond 32 neighbours: ope_normals_radius at r = 1 cm and 3 cm, and ope_normals_knn at k = 64 and 256 beside the
k = 30 reference point, on the 157 825-point model and on a 640 x 480 C3 scene (synth.make_frame, 307 200 points). Each
configuration reports the median wall time of the call on a resident device cloud (the call ends in a stream synchronise; it
includes the n x 16 B download of the normals), the neighbours visited per second (the radius sets' total size, or n_finite x k),
the device scratch bytes the call allocates beyond the cloud and its normals, and the CPU reference on one core for the same cloud
(the oracle's orc_normals_knn, tests/orc_radius.py for radius normals), with the card's name and power limit read in the same run.
Usage: python tools/bench_normals.py [--reps 5] [--out f.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import ope_pkg  # noqa: E402

ope_pkg.load()
from ope_b200 import cuda_lib, synth  # noqa: E402
import orc_py  # noqa: E402
import orc_radius  # noqa: E402

SMEM_KEYS = 8192                 # features.cu kRadSmemKeys: longer lists take global scratch
DEFAULT_BUDGET = 256 << 20       # OPE_RADIUS_NORMALS_SCRATCH_BYTES default


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers are still reported, marked as unattributed
        return "unknown (%s)" % e, "unknown"


def radius_scratch_bytes(counts, budget=DEFAULT_BUDGET):
    """what normals_radius_device allocates: the counts, and for lists above SMEM_KEYS their offsets and the largest tile"""
    n = len(counts)
    big = np.where(counts > SMEM_KEYS, counts, 0).astype(np.int64)
    if not big.any():
        return 4 * n
    off = np.concatenate([[0], np.cumsum(big)])
    keys, q0 = 0, 0
    per = budget // 8
    while q0 < n:
        q1 = q0 + 1
        while q1 < n and off[q1 + 1] - off[q0] <= per:
            q1 += 1
        keys = max(keys, int(off[q1] - off[q0]))
        q0 = q1
    return 4 * n + 8 * (n + 1) + 8 * keys


def timed(fn, reps):
    fn()   # warm-up: grids, module load
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts)), [1e3 * t for t in ts]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    model = synth.make_model(157825)
    scene = synth.make_frame(model, 940)[1]
    scene = np.ascontiguousarray(scene.reshape(-1, scene.shape[-1])[:, :3], np.float32)
    ctx = cuda_lib.Context(0)
    name, power = card()
    out = {"card": name, "power_limit": power, "reps": a.reps, "runs": []}
    for cname, pts in (("model_157825", model), ("scene_307200", scene)):
        cl = ctx.upload(pts)
        n_fin = int(np.isfinite(pts[:, :3]).all(1).sum())
        for kind, v in (("knn", 30), ("knn", 64), ("knn", 256), ("radius", 0.01), ("radius", 0.03)):
            if kind == "knn":
                ms, all_ms = timed(lambda: ctx.normals_knn(cl, v), a.reps)
                visited, scratch = n_fin * min(v, n_fin), 0
                t0 = time.perf_counter(); orc_py.normals_knn(pts, v); orc_s = time.perf_counter() - t0
                extra = {}
            else:
                ms, all_ms = timed(lambda: ctx.normals_radius(cl, v), a.reps)
                off, _, _ = ctx.radius(cl, cl, v)
                counts = np.diff(off)
                visited, scratch = int(counts.sum()), radius_scratch_bytes(counts)
                t0 = time.perf_counter(); orc_radius.normals_radius(pts, v); orc_s = time.perf_counter() - t0
                extra = {"neighbours_median": float(np.median(counts[counts > 0])) if counts.any() else 0,
                         "neighbours_max": int(counts.max()), "lists_above_smem": int((counts > SMEM_KEYS).sum())}
            rec = {"cloud": cname, "n": len(pts), "n_finite": n_fin, "kind": kind, "param": v, "ms": ms, "ms_all": all_ms,
                   "neighbours": visited, "neighbours_per_s": visited / (ms * 1e-3), "scratch_bytes": scratch, "oracle_one_core_s": orc_s,
                   "speedup_vs_oracle": orc_s / (ms * 1e-3)}
            rec.update(extra)
            print(json.dumps(rec), flush=True)
            out["runs"].append(rec)
        cl.free()
    ctx.close()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

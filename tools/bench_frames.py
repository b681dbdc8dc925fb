#!/usr/bin/env python
"""C5 (BASELINE.json configs[4]): batched localisation of independent synthetic 640x480 frames (SAC-IA hypothesis pool + ICP,
the full first-frame estimateFinalPose path) sharded frame f -> rank f mod N over the GPUs of one box. No data-path collective:
the per-rank device times are max-reduced and the frame counts summed only to print one line.

  python tools/bench_frames.py [--frames 1024]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29513 tools/bench_frames.py

Scenes are generated once (64 distinct frames, cycled) outside the timed region; every frame starts a fresh tracker, so
SAC-IA runs on every frame (the expensive first-frame path of the reference)."""
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # ope_pose_batch: one hardware queue per lane stream (before CUDA starts)
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np


def main():
    import torch
    import ctypes
    import ope_pkg
    ope_pkg.load()
    from ope_b200 import cuda_lib, parallel, synth
    n = 1024
    if "--frames" in sys.argv:
        n = int(sys.argv[sys.argv.index("--frames") + 1])
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()       # a real handle: the legacy default stream (0) would make the ctx create its own
    torch.cuda.set_stream(stream)      # torch work (L2 flush, events) and the library's kernels share ONE stream
    ctx = cuda_lib.Context(local, stream.cuda_stream)
    model = synth.make_model()
    distinct = 64
    frames = [synth.make_frame(model, 5000 + f)[0] for f in range(distinct)]
    libc = ctypes.CDLL(None)
    mine = parallel.shard_units(n, rank, world)
    model_cloud = ctx.upload(model)
    targets = [ctx.upload(c) for c in frames]

    def run(host):
        for f in mine:
            tr = cuda_lib.PoseTracker(ctx)
            libc.srand(1)
            if host:
                src = model.copy()
                tr.estimate_final(src, frames[f % distinct])
            else:
                src = ctx.transform(model_cloud, np.eye(4, dtype=np.float32))
                tr.estimate_final_device(src, targets[f % distinct])
                src.free()
            tr.close()

    workers = int(sys.argv[sys.argv.index("--workers") + 1]) if "--workers" in sys.argv else 16

    def run_batch(host):
        # ope_pose_batch: lanes with their own streams, model side cached (SURVEY 8f-3); the decision tables are drawn
        # from libc rand() in frame order inside the call
        libc.srand(1)
        inputs = [frames[f % distinct] if host else targets[f % distinct] for f in mine]
        prm = None
        if os.environ.get("OPE_BENCH_ICP_ITERS"):      # experiment knob: how much of the frame time is the ICP loop
            prm = cuda_lib.pose_params()
            prm.icp.max_iterations = int(os.environ["OPE_BENCH_ICP_ITERS"])
        res, status = ctx.pose_batch(model, inputs, prm=prm, workers=workers)
        assert (status == 0).all()
        return res

    if "--serial" not in sys.argv:
        run = run_batch
        run_batch(False)
    for f in mine[:3]:
        run(False) if f == mine[0] else None
    out = {}
    for host in (False, True):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run(host)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        out["e2e_frames_per_s" if host else "frames_per_s"] = n / (float(ms.item()) / 1e3)
    if rank == 0:
        print(json.dumps({"metric": "frames_per_sec_fpfh_sacia_icp_640x480", "n_gpus": world, "frames": n, "scaling": "strong",
                          "value": out["frames_per_s"], "e2e": out["e2e_frames_per_s"], "unit": "frames/s",
                          "config": {"workload": "C5: %d independent frames, full first-frame path, frame f -> rank f mod N" % n,
                                     "mode": "serial trackers" if "--serial" in sys.argv else "ope_pose_batch, one call per GPU",
                                     "host_cores": os.cpu_count()}}))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

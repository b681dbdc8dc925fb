#!/usr/bin/env python
"""bench.py — headline benchmark of the registration hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline (BASELINE.json metric "frames/sec FPFH+SAC-IA+ICP @640x480 scene", configs[4] "C5"): batched localisation of 1 024
independent synthetic 640x480 frames — the model the reference ships (157 825 points) under a random pose at 0.6-1.6 m, table,
wall, depth noise; the segmented cluster of every frame goes through the full first-frame path of estimateFinalPose
(UniformSampling 1 cm / 8 mm, normals k = 30, FPFH r = 3 cm, SAC-IA 400 x 5 drawn from libc rand() INSIDE the timed region,
ICP-with-normals <= 100 iterations, fitness, dense SVD) via ope_pose_batch. A step = one pass over the 1 024 frames.
STRONG scaling: frame f goes to rank f mod N, no data-path collective (SURVEY 8e); value = frames of all ranks / max-over-ranks
device time.

  value     clusters already resident in HBM (device clouds); CUDA-event time around the synchronous batch call; L2 flushed
            between steps
  e2e       the same call with HOST buffers: H2D of every cluster and D2H of every result inside the timed region
  roofline  the dominant kernel of a frame (the ICP loop): algorithmic bytes / its CUDA-event duration
  cpu_baseline  the CPU oracle (restatement of the PCL path, pinned to the reference's vendored sources by tests/test_ref.py)
                on ONE host core on a bounded sample of the same frames, with a parity record (GPU vs oracle, same frames)
  icp       (N=1) BASELINE's second metric, configs[1] "C2": ICP iterations/s at 50k points, with its own roofline, its CPU
            baseline and the parity of the timed pair
  feature_gemm / depth_to_cloud  (N=1) the tcgen05 feature-distance GEMM (tensor roofline) and the HBM-bound stage

--impl reference times the CPU oracle on all host cores on the same frames (one frame per core at a time, full iteration
budget: the same configuration), a bounded sample per step.

--dump-outputs DIR writes what the headline's last timed step returned (see dump_outputs) for comparing two builds: with the same
arguments every run feeds the same frames and the same libc rand() stream.
"""
import argparse
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # ope_pose_batch: one hardware queue per worker stream (before CUDA starts)
import json
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

N_FRAMES = 1024
FRAME0 = 1000                # frame seeds 1000 .. 2023 (the agreement scenes of tools/pose_agreement.py)
METRIC = "frames_per_sec_fpfh_sacia_icp_640x480"
UNIT = "frames/s"
WORKLOAD = ("C5: batched localisation of 1024 independent synthetic 640x480 frames (bundled 157825-point model vs segmented cluster; "
            "UniformSampling 1 cm / 8 mm, normals k=30, FPFH r=0.03, SAC-IA 400x5, ICP-with-normals <=100 it, dense SVD)")
WORKERS = 16
N_PTS = 50000
ICP_ITERS = 50
MAX_CORR = 0.05
ICP_WORKLOAD = "C2: ICP-only point-to-point, 50k-point source vs 50k-point target, 50 iterations, max-corr-distance 0.05"


def icp_kwargs():
    return dict(max_iterations=ICP_ITERS, max_correspondence_distance=MAX_CORR, transformation_epsilon=1e-8,
                euclidean_fitness_epsilon=1e-8, force_all_iterations=1)


# DRAM bytes of ONE launch from ncu --set full captures of these exact workloads (committed under profiles/): what the kernels really
# moved, to set beside the algorithmic bytes. icp_kernel: the 1.6 MB pair is read once and then lives in L2 (80 MB algorithmic over 50
# iterations, 5.2 MB from DRAM); depth_fused_kernel: DRAM traffic equals the algorithmic bytes.
NCU_ICP_DRAM_BYTES = 4826624 + 816128
NCU_DEPTH_DRAM_BYTES = 629331712 + 4976560000
NCU_ICP_BATCH_DRAM_BYTES = 24792832 + 121856      # icp_small_batch_kernel over 296 frames (profiles/r02_f_batch_kernels_full.txt)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """samples SM clock and throttle reasons through NVML while the timed region runs"""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------ frames ----
_GEN = {}


def _gen_init():
    import ope_pkg
    ope_pkg.load()
    from ope_b200 import synth
    _GEN["synth"], _GEN["model"] = synth, synth.bundled_model()


def _gen_frame(f):
    return _GEN["synth"].make_frame(_GEN["model"], FRAME0 + f)[0]


def make_clusters(indices):
    """the segmented clusters of the given frames, rendered on the host cores (fork pool: call before CUDA is initialised)"""
    import multiprocessing as mp
    procs = max(1, min(os.cpu_count() or 1, 32, len(indices)) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1"))))
    with mp.get_context("fork").Pool(procs, initializer=_gen_init) as pool:
        return pool.map(_gen_frame, list(indices), chunksize=4)


# ------------------------------------------------------------------------------------------ reference arm ----
_REF = {}


def _ref_init():
    import orc_py
    _gen_init()
    _REF["orc"] = orc_py
    orc_py.lib()


def _ref_frame(f):
    """one frame through the oracle's estimateFinalPose: fresh PoseEstimator, SAC-IA drawing from libc rand(), full budget"""
    orc_py = _REF["orc"]
    if ("cl", f) not in _REF:
        _REF[("cl", f)] = _gen_frame(f)
    src = _GEN["model"].copy()
    p = orc_py.PoseEstimator().estimate_final(src, _REF[("cl", f)])
    return p.icp_iterations


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_step = 2 * cores          # bounded sample: two frames per host core per step, the first frames of the same 1024
    with mp.get_context("fork").Pool(cores, initializer=_ref_init) as pool:
        for _ in range(max(args.warmup, 1)):
            pool.map(_ref_frame, range(per_step), chunksize=1)     # also renders and caches the frames in the workers
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_ref_frame, range(per_step), chunksize=1)
        wall = time.perf_counter() - t0
    value = per_step * args.steps / wall
    sample = ("per step: the first %d of the 1024 frames (two per host core), full estimateFinalPose each with the full iteration "
              "budget, one frame per core at a time" % per_step)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "same_config": True,
                       "note": "CPU restatement of the PCL path (PCL itself unavailable; pinned to the reference's vendored "
                               "registration sources by tests/test_ref.py), all host cores"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ our arm ----
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # this rank's frames, rendered on the host BEFORE CUDA starts (fork pool)
    mine = [f for f in range(N_FRAMES) if f % world == rank]
    clusters = make_clusters(mine)

    import torch
    import ope_pkg
    ope_pkg.load()
    from ope_b200 import cuda_lib, synth
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        # NCCL's version banner and logs go to stderr — stdout carries exactly one JSON line. (NCCL honours NCCL_DEBUG_FILE only
        # above the VERSION level.)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # concurrent chunk lanes of ope_pose_batch: the library's own default (one per host core this rank can count on, 2..8), pinned
    # here so that the line can say what ran
    cores = max(1, len(os.sched_getaffinity(0)) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1"))))
    lanes = int(os.environ.setdefault("OPE_BATCH_LANES", str(min(8, max(2, cores - 1)))))
    stream = torch.cuda.Stream()       # a real handle: the legacy default stream (0) would make the ctx create its own
    torch.cuda.set_stream(stream)      # torch work (L2 flush, events) and the library's calls share ONE stream
    ctx = cuda_lib.Context(local, stream.cuda_stream)
    model = synth.bundled_model()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    targets = [ctx.upload(c) for c in clusters]
    import ctypes
    libc = ctypes.CDLL(None)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step(inputs):
        # tables=None: every frame's SAC-IA decision table (400 x 5 samples + picks) is drawn here, from libc rand(), in frame order
        res, status = ctx.pose_batch(model, inputs, tables=None, workers=WORKERS)
        assert (status == 0).all(), status
        return res

    libc.srand(1)
    barrier()   # the first collective builds NCCL's communicator (threads, peer mappings): before the warm-up, not inside the timing
    for _ in range(max(args.warmup, 3)):   # full steps: the chunking (and with it the memory pool's shape) depends on the batch size
        step(targets)

    def timed(inputs, steps=None):
        steps = args.steps if steps is None else steps
        sampler = ClockSampler(local)
        barrier()
        sampler.start()
        l0 = ctx.launches
        ms = []
        last = None
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            last = step(inputs)
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        barrier()
        clocks = sampler.stop()
        t = torch.tensor([float(np.sum(ms))], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), ctx.launches - l0, clocks, last

    if os.environ.get("OPE_BENCH_DEBUG_ARMS"):   # diagnosis: both arms, alternating, per-rank ms per step on stderr
        for name, inp in (("resident", targets), ("host", clusters), ("resident", targets), ("host", clusters)):
            step(inp)
            ms, _, _, _ = timed(inp)
            sys.stderr.write("[arms] rank %d %s %.2f ms/step\n" % (rank, name, ms / args.steps))
    # (untimed dress rehearsal of the timed region itself — barrier, clock sampler, events: at N > 1 the first pass through it was
    # measured 60 % slower than every later one)
    timed(targets, 2)
    # ---- value: clusters resident in HBM ----
    total_ms, launches, clocks, outputs = timed(targets)
    value = N_FRAMES * args.steps / (total_ms / 1e3)
    # ---- e2e: host buffers in (H2D of every cluster), results out (D2H of every ope_pose_result) ----
    step(clusters)   # untimed: the pinned staging buffers of the host path grow to this batch
    e2e_ms, _, _, last = timed(clusters)
    e2e_value = N_FRAMES * args.steps / (e2e_ms / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, mine, outputs, cuda_lib.T, dist)
    h2d = int(sum(len(c) for c in clusters)) * 16 + len(model) * 12
    d2h = len(clusters) * ctypes.sizeof(cuda_lib.T.PoseResult)
    if dist is not None:
        t = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        h2d, d2h = int(t[0].item()), int(t[1].item())

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step": N_FRAMES, "l2": "flushed between steps (256 MiB write)",
                       "sharding": "frame f -> rank f mod N, no collective", "api": "ope_pose_batch", "workers_per_rank": WORKERS, "chunk_lanes_per_rank": lanes, "untimed_rehearsal_steps": 2,
                       "host_cores_per_rank": cores,
                       "sacia_tables": "drawn from libc rand() inside the timed region (ope_sacia_draw)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clocks}
    try:
        line["roofline"] = frame_roofline(ctx, cuda_lib, synth, model, clusters, stream, torch)
    except Exception as e:
        line["roofline"] = {"error": repr(e)}

    if world > 1:
        try:
            line["sharded_sacia"] = sharded_sacia_numbers(ctx, cuda_lib, model, clusters, stream, torch, dist, rank, world)
        except Exception as e:
            line["sharded_sacia"] = {"error": repr(e)}
    if rank == 0 and world == 1:
        line["cpu_baseline"] = frames_cpu_baseline(ctx, cuda_lib, synth, model, clusters)
        for key, fn in (("icp", lambda: icp_numbers(ctx, cuda_lib, synth, model, stream, torch, flush, args)),
                        ("feature_gemm", lambda: feature_gemm_numbers(ctx)),
                        ("depth_to_cloud", lambda: depth_numbers(ctx, synth, model, stream, torch)),
                        ("scene_preparation", lambda: scene_numbers(ctx, cuda_lib, synth, model, stream, torch)),
                        ("single_frame", lambda: single_frame_numbers(ctx, cuda_lib, synth, model, clusters, stream, torch))):
            try:
                line[key] = fn()
            except Exception as e:  # the headline line must survive a failure of a secondary workload
                line[key] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def dump_outputs(out_dir, frames, results, T, dist):
    """the ope_pose_result of every frame as DIR/<field>.npy, row f = frame f of the 1024: the poses as float32 (N, 16) in the
    ABI's column-major order, every other field as float64 (N,); ranks send their frames to rank 0, which writes"""
    import ctypes
    cols = {}
    for name, ctype in T.PoseResult._fields_:
        if name == "reserved":
            continue
        if issubclass(ctype, ctypes.Array):
            cols[name] = np.array([list(getattr(r, name)) for r in results], np.float32)
        else:
            cols[name] = np.array([getattr(r, name) for r in results], np.float64)
    order = np.asarray(frames)
    if dist is not None:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, (order, cols))
        if dist.get_rank() != 0:
            return
        order = np.concatenate([p[0] for p in parts])
        cols = {k: np.concatenate([p[1][k] for p in parts]) for k in cols}
    perm = np.argsort(order)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in cols.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[perm])


def sharded_sacia_numbers(ctx, cuda_lib, model, clusters, stream, torch, dist, rank, world, pool=131072):
    """the path's ONE collective (SURVEY 8e row 2), inside the library: a SAC-IA pool of `pool` hypotheses of one alignment sharded
    over the ranks — ope_sacia_align_sharded: ncclAllReduce(MIN) of the packed (error, index) key + ncclBroadcast of the 4x4 on the
    context's stream. Device time (CUDA events, max over ranks) beside one GPU evaluating the whole pool; same winner required."""
    import ctypes
    cm, cc = ctx.upload(model), ctx.upload(clusters[0] if rank == 0 else clusters[0])
    # every rank needs the SAME pair: rank 0's first cluster
    box = [clusters[0] if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    cc = ctx.upload(box[0])
    sp_c, tp_c = ctx.uniform_sample_cloud(cm, 0.01), ctx.uniform_sample_cloud(cc, 0.01)
    ctx.normals_knn(sp_c, 30); ctx.normals_knn(tp_c, 30)
    sf, tf = ctx.fpfh(sp_c, 0.03), ctx.fpfh(tp_c, 0.03)
    kw = dict(max_iterations=pool, nr_samples=5, k_correspondences=5, min_sample_distance=0.01, max_correspondence_distance=0.05)
    ctypes.CDLL(None).srand(1)      # every rank draws the same table from libc rand()
    table = cuda_lib.rng_table(*cuda_lib.sacia_draw(sp_c.download(), pool, 5, 5, 0.01))
    uid = [cuda_lib.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    comm = cuda_lib.Comm(ctx, uid[0], world, rank)
    prm = cuda_lib.sacia_params(**kw)

    def timed(fn):
        fn()                                        # warm-up (NCCL connects lazily)
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return r, float(t.item())

    one, one_ms = timed(lambda: ctx.sacia(sp_c, sf, tp_c, tf, prm, table))
    sh, sh_ms = timed(lambda: comm.sacia(sp_c, sf, tp_c, tf, prm, table))
    same = (sh.best_iteration == one.best_iteration and np.float32(sh.best_error) == np.float32(one.best_error)
            and np.array_equal(np.array(list(sh.T), np.float32), np.array(list(one.T), np.float32)))
    ok = torch.tensor([1.0 if same else 0.0], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    comm.close()
    if ok.item() != 1.0:
        raise AssertionError("the sharded pool's winner differs from the single-GPU winner")
    return {"workload": "one alignment, SAC-IA pool of %d hypotheses x %d source points vs %d target points" % (pool, len(sp_c), len(tp_c)),
            "api": "ope_sacia_align_sharded (ncclAllReduce MIN of a 64-bit key + ncclBroadcast of 16 floats, in the library)",
            "one_gpu_ms": one_ms, "sharded_ms": sh_ms, "speedup": one_ms / sh_ms, "ranks": world, "same_winner_on_every_rank": True,
            "nccl_version": int(cuda_lib.lib().ope_comm_nccl_version())}


def frame_roofline(ctx, cuda_lib, synth, model, clusters, stream, torch, n=8):
    """the dominant kernel of the headline is the frame-spanning ICP launch (icp_small_batch_kernel; SURVEY 8d, K8): algorithmic bytes
    = sum over the frames of iterations x (32 N_s + 32 N_t + 64) (points + normals on both sides) over its CUDA-event duration
    (ope_pose_batch_stage_ms, events on the library's stream), measured on one more pass over this rank's frames"""
    import ctypes
    peak, peak_src = peaks()
    ctx.batch_stage_ms(1)       # timing on: one lane, chunks of <= 296 frames — a different shape from the headline's small chunks,
    for _ in range(2):          # so one pass first lets the memory pool grow to it
        ctypes.CDLL(None).srand(1)
        ctx.batch_stage_ms(1)
        res, status = ctx.pose_batch(model, clusters, tables=None, workers=WORKERS)
    st = ctx.batch_stage_ms(0)
    total = sum(st.values())
    bytes_ = sum(r.icp_iterations * (32.0 * r.n_src_fine + 32.0 * r.n_tgt_fine + 64.0) for r in res)
    k_ms = st["icp"]
    a = bytes_ / (k_ms * 1e-3) / 1e9
    return {"kernel": "icp_small_batch_kernel (timed on one lane: one launch per chunk of <= 296 frames, nothing else on the device)", "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s",
            "frac": a / peak, "traffic": NCU_ICP_BATCH_DRAM_BYTES, "traffic_source": "ncu --set full of one launch over 296 frames "
            "(profiles/r02_f_batch_kernels_full.txt): dram__bytes_read.sum + dram__bytes_write.sum", "peak_source": peak_src,
            "kernel_ms_per_frame": k_ms / len(clusters), "kernel_share_of_step": k_ms / total,
            "stage_ms_per_frame": {k: round(v / len(clusters), 5) for k, v in st.items()},
            "note": "a frame's fine clouds are ~1.7k + ~1.1k points and live in shared memory for the whole alignment: the launch is "
                    "issue/latency-bound (ncu: 39 % issue-active, 44 % of the stall samples on barriers, DRAM 0.008 %), not HBM-bound "
                    "(SURVEY 8d); frac is reported against HBM as the contract asks. Timed on one lane (nothing else on the device); "
                    "in the headline run eight lanes overlap the launches' tails. The HBM-bound stage is depth_to_cloud (below)."}


def frames_cpu_baseline(ctx, cuda_lib, synth, model, clusters, n=24, seed=7):
    """the oracle on ONE host core on the first n frames (a fresh PoseEstimator per frame, SAC-IA drawing from libc rand() in
    frame order after srand(seed)), and the parity of the GPU batch on the same frames consuming the same rand() stream"""
    import ctypes
    import orc_py
    T = cuda_lib.T
    n = min(n, len(clusters))
    orc_py.srand(seed)
    t0 = time.perf_counter()
    oracle = [orc_py.PoseEstimator().estimate_final(model.copy(), clusters[f]) for f in range(n)]
    dt = time.perf_counter() - t0
    ctypes.CDLL(None).srand(seed)
    got, status = ctx.pose_batch(model, clusters[:n], tables=None, workers=WORKERS)
    agree, rot, trans, fit = 0, 0.0, 0.0, 0.0
    for g, o in zip(got, oracle):
        r, t = synth.pose_error(T.mat4(g.final_pose), T.mat4(o.final_pose))
        ok = (r < 1e-4 and t < 1e-5 and abs(g.fitness - o.fitness) < 1e-5 and
              (g.icp_state, g.icp_converged, g.icp_iterations, g.sacia_best_iteration) ==
              (o.icp_state, o.icp_converged, o.icp_iterations, o.sacia_best_iteration))
        agree += ok
        if ok:
            rot, trans, fit = max(rot, r), max(trans, t), max(fit, abs(g.fitness - o.fitness))
    # the north star's bar: >= 95 % of the scenes within 1e-4 rad / 1e-5 m with the same convergence state (an ICP that never
    # converges amplifies the 1e-16 summation-order noise of its double-precision moments once in ~1 000 frames, DESIGN.md section 7)
    parity = {"frames": n, "agreeing_frames": int(agree), "agreement": agree / n, "max_rot_rad": rot, "max_trans_m": trans,
              "max_fitness_diff": fit, "bar": "1e-4 rad, 1e-5 m, fitness 1e-5, same ICP state / iterations / SAC-IA winner",
              "ok": bool(agree / n >= 0.95 and (status == 0).all())}
    if not parity["ok"]:
        raise AssertionError("GPU frames differ from the oracle: %r" % parity)
    return {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "the first %d of the 1024 frames, full estimateFinalPose each, %.1f s" % (n, dt), "parity": parity}


def icp_numbers(ctx, cuda_lib, synth, model, stream, torch, flush, args):
    """BASELINE's second metric (configs[1], C2): ICP iterations/s, 50k-point source vs 50k-point target, exactly 50 iterations
    (convergence tests evaluated but not acted on), max-corr-distance 0.05; a step = one align() = target index build + the fused
    loop. Device-resident and end to end, the roofline of icp_kernel, the oracle on one core on the SAME pair, and their parity."""
    T = cuda_lib.T
    src, tgt, _ = synth.icp_pair(N_PTS, seed=0, model=model)
    prm = cuda_lib.icp_params(**icp_kwargs())
    cs, ct = ctx.upload(src), ctx.upload(tgt)

    def step_device():
        ctx.invalidate(ct)            # the reference rebuilds its kd-tree per align(); so do we
        return ctx.icp(cs, ct, prm)

    for _ in range(3):
        res = step_device()
    step_ms, kern_ms = [], []
    steps = max(5, min(args.steps, 20))
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        res = step_device()
        e1.record(stream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        kern_ms.append(ctx.last_kernel_ms(0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        a, b = ctx.upload(src), ctx.upload(tgt)
        r, aligned = ctx.icp(a, b, prm, want_aligned=True)
        aligned.download()
        a.free(); b.free(); aligned.free()
    e1.record(stream)
    torch.cuda.synchronize()
    peak, peak_src = peaks()
    k_ms = float(np.mean(kern_ms))
    alg = ICP_ITERS * (16 * len(src) + 16 * len(tgt) + 64)
    cpu = cpu_baseline(src, tgt)
    o = cpu.pop("_result")
    rot, trans = synth.pose_error(T.mat4(res.T), T.mat4(o.T))
    parity = {"rot_rad": rot, "trans_m": trans, "same_state": bool((res.state, res.converged, res.iterations, res.n_correspondences) ==
                                                                   (o.state, o.converged, o.iterations, o.n_correspondences))}
    parity["ok"] = bool(parity["same_state"] and rot < 1e-4 and trans < 1e-5)
    if not parity["ok"]:
        raise AssertionError("the timed 50k pair differs from the oracle: %r" % parity)
    return {"metric": "icp_iterations_per_sec_50k", "workload": ICP_WORKLOAD, "value": ICP_ITERS * steps / (float(np.sum(step_ms)) / 1e3),
            "e2e": ICP_ITERS * steps / (e0.elapsed_time(e1) / 1e3), "unit": "iterations/s", "ms_per_align": float(np.mean(step_ms)),
            "roofline": {"kernel": "icp_kernel", "bound": "hbm", "achieved": alg / (k_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (k_ms / 1e3) / 1e9 / peak, "traffic": NCU_ICP_DRAM_BYTES,
                         "traffic_source": "ncu --set full of one icp_kernel launch on this workload (profiles/)", "peak_source": peak_src,
                         "kernel_ms": k_ms, "kernel_share_of_step": k_ms / float(np.mean(step_ms)),
                         "note": "one C2 alignment is 1.6 MB and stays in L2: search-latency / grid-barrier bound, not HBM bound"},
            "cpu_baseline": cpu, "parity": parity}


def cpu_baseline(src, tgt):
    """the oracle (CPU restatement of the PCL path) on one host core, same pair, all 50 iterations"""
    import orc_py
    t0 = time.perf_counter()
    res = orc_py.icp(src, tgt, orc_py.icp_params(**icp_kwargs()))
    dt = time.perf_counter() - t0
    return {"value": res.iterations / dt, "unit": "iterations/s", "cores": 1, "kind": "port", "_result": res,
            "sample": "one full alignment of the same 50k/50k pair (%d iterations, kd-tree build included), %.1f s" % (res.iterations, dt)}


def feature_gemm_numbers(ctx, nq=18944, nt=307200):
    """K6 at C3 scale (FPFH-space 5-NN of nq source descriptors in a 307 200-descriptor scene): the tcgen05/TMA distance GEMM with
    fused candidate selection, timed by its own CUDA events; tensor roofline against the measured bf16 peak."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(p))["bf16_tflops"]) if os.path.exists(p) else 1590.0
    rng = np.random.default_rng(0)
    ft = rng.gamma(0.6, 8.0, size=(nt, 33)).astype(np.float32)
    ft = (100.0 * ft / ft.reshape(nt, 3, 11).sum(2).repeat(11, 1)).astype(np.float32)
    fq = ft[rng.integers(0, nt, nq)] + rng.normal(0, 0.5, size=(nq, 33)).astype(np.float32)
    os.environ["OPE_FEATURE_KNN"] = "gemm"
    ms = []
    for _ in range(4):
        ctx.feature_knn(ft, fq, 5)
        ms.append(ctx.last_kernel_ms(2))
    os.environ.pop("OPE_FEATURE_KNN", None)
    k_ms = float(np.median(ms[1:]))
    g, f = ctx.feature_knn_stats()
    alg = 2.0 * 33 * nq * nt / (k_ms * 1e-3) / 1e12
    issued = 2.0 * 128 * nq * nt / (k_ms * 1e-3) / 1e12
    return {"workload": "C3-scale feature k-NN: %d x %d FPFH descriptors, k = 5" % (nq, nt), "kernel": "featgemm_kernel", "kernel_ms": k_ms,
            "roofline": {"bound": "tensor", "achieved": alg, "peak": peak, "unit": "TFLOP/s", "frac": alg / peak, "traffic": None,
                         "note": "achieved = 2*33*Nq*Nt algorithmic flops; the kernel issues K = 128 (3-way bf16 split + norm columns), "
                                 "i.e. %.0f TFLOP/s of tensor work; ncu sm__pipe_tensor_cycles_active in profiles/" % issued},
            "exact_fallback_queries": f, "gemm_queries": g}


def depth_numbers(ctx, synth, model, stream, torch, frames=1024):
    """The one stage whose inputs exceed the 126 MB L2 (SURVEY 8d: only such launches say anything about HBM): depth image -> cloud
    for a batch of Kinect frames resident in HBM (8f-1), one launch of depth_fused_kernel; roofline against the measured copy peak."""
    base = []
    for f in range(8):
        _, cloud, _ = synth.make_frame(model, 700 + f)
        base.append(np.rint(np.nan_to_num(cloud[..., 2], nan=0.0).astype(np.float64) * 1000.0).astype(np.uint16))
    depth = torch.from_numpy(np.stack(base).astype(np.int16)).cuda().repeat(frames // 8, 1, 1).contiguous()
    B, R, Cc = depth.shape
    out = torch.empty((B * R * Cc, 4), dtype=torch.float32, device="cuda")
    col = torch.empty(B * Cc + 1, dtype=torch.int32, device="cuda")
    ms = []
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.depth_to_cloud_batch(depth.data_ptr(), B, R, Cc, out.data_ptr(), col.data_ptr())
        e1.record(stream)
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    kept = int(col[-1].item())
    t = float(np.median(ms[2:])) * 1e-3
    peak, peak_src = peaks()
    npx = B * R * Cc
    alg = (2 * npx + 16 * kept) / t / 1e9
    del depth, out, col
    torch.cuda.empty_cache()
    return {"workload": "depth image -> cloud, %d frames of %dx%d resident in HBM (%.0f MB in, %.0f MB out), one launch" % (B, Cc, R, 2 * npx / 1e6, 16 * kept / 1e6),
            "kernel": "depth_fused_kernel", "ms": t * 1e3, "frames_per_sec": B / t,
            "roofline": {"bound": "hbm", "achieved": alg, "peak": peak, "unit": "GB/s", "frac": alg / peak,
                         "traffic": NCU_DEPTH_DRAM_BYTES if frames == 1024 else None,
                         "traffic_source": "ncu --set full, profiles/r01_e_depth_fused_full.txt", "peak_source": peak_src,
                         "note": "algorithmic = 2 B per pixel in + 16 B per kept pixel out; ncu dram__bytes of the launch equal it (profiles/)"}}


def scene_numbers(ctx, cuda_lib, synth, model, stream, torch, frames=(21, 22, 23)):
    """Scene preparation (SURVEY 8f-2, D&L/src/objectsegmentationplane.cpp): pass-through crop + getSegmentedObjectsOnPlane (table
    plane RANSAC, polygonal prism, second plane, Euclidean clusters) on full 640x480 frames resident in HBM, device time per frame;
    the oracle on one host core on the same frames; per-point labels, plane equations and RANSAC iteration counts must be equal."""
    import orc_py
    limits = (-0.5, 0.5, -0.5, 0.3, 0.5, 1.6)      # ObjectSegmentationPlane::getFiltered, D&L/src/objectsegmentationplane.cpp:17-18
    clouds = [synth.make_frame(model, f)[1].reshape(-1, 3) for f in frames]
    dev = [ctx.upload(c) for c in clouds]

    def gpu(c):
        filt = ctx.pass_through(c, limits)
        return filt, ctx.segment_objects_on_plane(filt)

    for c in dev:
        gpu(c)
    ms = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        got = [gpu(c) for c in dev]
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / len(dev))
    t0 = time.perf_counter()
    same, kept = True, 0
    for pts, (filt, g) in zip(clouds, got):
        keep = np.arange(len(pts), dtype=np.int32)
        for field, lo, hi in ((2, limits[4], limits[5]), (1, limits[2], limits[3]), (0, limits[0], limits[1])):   # z, y, x
            keep = keep[orc_py.pass_through(pts[keep], field, lo, hi)]
        o = orc_py.segment_objects_on_plane(pts[keep])
        kept += len(keep)
        same &= bool(np.array_equal(filt.download(), pts[keep]) and np.array_equal(g[0], o[0]) and g[1] == o[1] and
                     np.array_equal(g[2], o[2]) and np.array_equal(g[3], o[3]) and tuple(g[4]) == tuple(o[4]))
    cpu_s = (time.perf_counter() - t0) / len(dev)
    t = float(np.median(ms))
    return {"workload": "pass-through + getSegmentedObjectsOnPlane on %d full 640x480 frames resident in HBM (%d of 307200 points survive "
                        "the crop on average)" % (len(dev), kept // len(dev)),
            "api": "ope_pass_through + ope_segment_objects_on_plane", "ms_per_frame": t, "frames_per_sec": 1e3 / t,
            "cpu_baseline": {"value": 1.0 / cpu_s, "unit": "frames/s", "cores": 1, "kind": "port",
                             "sample": "the same %d frames, %.2f s each" % (len(dev), cpu_s)},
            "parity": {"labels_planes_iterations_equal": same, "ok": same}}


def single_frame_numbers(ctx, cuda_lib, synth, model, clusters, stream, torch, n=12):
    """C1: one frame at a time through ope_pose_tracker (a fresh tracker per frame: the first-frame path, SAC-IA drawn from libc
    rand()): latency view of the same pipeline, per-stage device time, and what the model-side cache (8f-3) saves"""
    out = {}
    for cache in ("0", "1"):
        os.environ["OPE_MODEL_CACHE"] = cache
        stage = np.zeros(8)
        for f in range(3):
            tr = cuda_lib.PoseTracker(ctx); tr.estimate_final(model.copy(), clusters[f]); tr.close()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for f in range(n):
            tr = cuda_lib.PoseTracker(ctx)
            tr.estimate_final(model.copy(), clusters[f % len(clusters)])
            stage += np.array(tr.stage_ms())
            tr.close()
        e1.record(stream)
        torch.cuda.synchronize()
        key = "model_cache_on" if cache == "1" else "model_cache_off"
        out[key] = {"e2e_frames_per_sec": n / (e0.elapsed_time(e1) / 1e3), "stage_ms_per_frame": (stage / n).round(4).tolist()}
    os.environ.pop("OPE_MODEL_CACHE", None)
    out["stage_names"] = ["downsample", "normals", "fpfh", "sacia", "icp", "fitness", "umeyama+transforms", "total"]
    out["workload"] = "C1: estimateFinalPose, one frame at a time, host buffers in / aligned cloud out"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computes")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

"""Per-object point clouds of a batch of frames in one pass (clouds.object_clouds_frames) against one object_clouds call
per frame.

  frames        F = 1 / 8 / 30 frames of 640x480, 1-2 or 8 objects per frame: one object_clouds_frames call against F
                object_clouds calls.  Device time: CUDA events around the step, L2 overwritten before each; host time:
                host clock around the enqueue of the step (no synchronise inside).  Variants alternated.
  single_frame  the stage workloads of object_clouds_bench.py (640x480 and 1280x720, 8 / 32 / 64 / 256 objects):
                object_clouds and backproject_instances with this tree's library against --before-lib (a build of the
                parent commit's libgenpose_b200.so), alternated in the same process.  Skipped without --before-lib.
  tracking      a 30-video tracking step: one 640x480 frame of one object per video, each video with its own camera,
                50 hypotheses, step_control="object", keyed, T0 = 0.25 with warm starts, graphed.  Frames in (host depth
                + labels) to poses out, host clock with a synchronise at the end, and CUDA events around the device
                part; the clouds made by one object_clouds_frames call or by 30 object_clouds calls.  Alternated.

The GPU's name and power limit are read in the same run.

    python profiles/frames_clouds_bench.py [--reps 20] [--before-lib PATH] [--out profiles/frames_clouds_b200.json]
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from genpose2_b200 import _lib, clouds, synthetic  # noqa: E402
from genpose2_b200.pipeline import PosePipeline  # noqa: E402
from step_control_bench import L2_FLUSH_BYTES, gpu_info  # noqa: E402

N = 1024
REPEAT = 50


def stats(ts):
    return {"median": float(np.median(ts)), "min": float(min(ts)), "max": float(max(ts))}


def alternate(variants, reps, flush):
    """variants: name -> fn.  Per rep and variant: L2 overwritten, CUDA events around fn, host clock around its
    enqueue.  -> name -> {"device_ms": ..., "host_enqueue_ms": ...}"""
    for fn in variants.values():
        fn()
    torch.cuda.synchronize()
    dev = {n: [] for n in variants}
    host = {n: [] for n in variants}
    for _ in range(reps):
        for name, fn in variants.items():
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            t0 = time.perf_counter()
            fn()
            host[name].append((time.perf_counter() - t0) * 1e3)
            e.record()
            torch.cuda.synchronize()
            dev[name].append(s.elapsed_time(e))
    return {n: {"device_ms": stats(dev[n]), "host_enqueue_ms": stats(host[n])} for n in variants}


def pattern(F, per):
    return [1 + f % 2 for f in range(F)] if per == "1-2" else [8] * F


def frames(args, flush, result):
    H, W = 480, 640
    for F in (1, 8, 30):
        for per in ("1-2", "8"):
            counts = pattern(F, per)
            depth, labels, intr = synthetic.make_instance_frames(H, W, counts, seed=F, bad_depth=0.01)
            d, lab = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda()
            B = sum(counts)
            keys = torch.arange(B, dtype=torch.int64, device="cuda")
            intr_t = torch.from_numpy(intr).float().cuda()
            offs_t = torch.from_numpy(np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)).cuda()
            base = np.concatenate([[0], np.cumsum(counts)])
            split = [(f, n, keys[base[f]:base[f] + n]) for f, n in enumerate(counts)]
            host_intr = [tuple(float(v) for v in r) for r in intr]

            def per_frame():
                return [clouds.object_clouds(d[f], lab[f], host_intr[f], k, N) for f, n, k in split]

            variants = {"frames_host_forms": lambda: clouds.object_clouds_frames(d, lab, intr, counts, keys, N),
                        "frames_cuda_forms": lambda: clouds.object_clouds_frames(d, lab, intr_t, offs_t, keys, N),
                        "per_frame_calls": per_frame}
            want = per_frame()
            got = variants["frames_host_forms"]()
            for n in ("pts", "pts_center", "counts"):   # the variants compute the same clouds
                assert torch.equal(got[n], torch.cat([w[n] for w in want])), n
            entry = {"frame": f"{W}x{H}", "frames": F, "objects_per_frame": per, "objects": B}
            entry.update(alternate(variants, args.reps, flush))
            print(json.dumps(entry), flush=True)
            result["frames"].append(entry)


def load_before(path):
    lib = ctypes.CDLL(os.path.abspath(path))
    for name, (res, argt) in _lib.SIGNATURES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, argt
    return lib


def single_frame(args, flush, result):
    after = _lib.load()
    before = load_before(args.before_lib)

    def with_lib(lib, fn):
        def run():
            _lib._lib = lib
            try:
                return fn()
            finally:
                _lib._lib = after
        return run

    for H, W in ((480, 640), (720, 1280)):
        for B in (8, 32, 64, 256):
            depth, labels = synthetic.make_instance_frame(H, W, B, seed=B, bad_depth=0.01)
            d, lab = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda()
            keys = torch.arange(B, dtype=torch.int64, device="cuda")
            intr = (600.0, 600.0, W / 2.0, H / 2.0)
            oc_ = lambda: clouds.object_clouds(d, lab, intr, keys, N)
            bp = lambda: clouds.backproject_instances(d, lab, intr, B)
            a, b = with_lib(after, oc_)(), with_lib(before, oc_)()
            for n in ("pts", "pts_center", "counts"):   # the parent's library computes the same clouds
                assert torch.equal(a[n], b[n]), n
            variants = {"object_clouds_before": with_lib(before, oc_), "object_clouds_after": with_lib(after, oc_),
                        "stage_a_before": with_lib(before, bp), "stage_a_after": with_lib(after, bp)}
            entry = {"frame": f"{W}x{H}", "objects": B}
            entry.update({n: v["device_ms"] for n, v in alternate(variants, args.reps, flush).items()})
            print(json.dumps(entry), flush=True)
            result["single_frame"].append(entry)


def tracking(args, flush, result):
    H, W, F = 480, 640, 30
    pipe = PosePipeline(device="cuda", use_graph=True, step_control="object").load_synthetic_weights()
    R0 = synthetic._random_rotations(np.random.default_rng(0), F)
    init = torch.zeros(F, 9)
    init[:, :3] = torch.from_numpy(R0[:, :, 0]).float()
    init[:, 3:6] = torch.from_numpy(R0[:, :, 1]).float()
    init = init.cuda()
    steps = [synthetic.make_instance_frames(H, W, [1] * F, seed=s) for s in (200, 300)]
    keys = torch.arange(F, dtype=torch.int64, device="cuda")
    pinned = {"depth": torch.empty((F, H, W), dtype=torch.float32, pin_memory=True),
              "labels": torch.empty((F, H, W), dtype=torch.int32, pin_memory=True)}
    k = [0]

    def upload():
        k[0] += 1
        depth, labels, intr = steps[k[0] % len(steps)]
        pinned["depth"].copy_(torch.from_numpy(depth))
        pinned["labels"].copy_(torch.from_numpy(labels))
        return (pinned["depth"].to("cuda", non_blocking=True), pinned["labels"].to("cuda", non_blocking=True),
                [tuple(float(v) for v in r) for r in intr])

    def frames_variant():
        d, lab, intr = upload()
        data = clouds.object_clouds_frames(d, lab, intr, [1] * F, keys, N)
        return pipe(data, repeat_num=REPEAT, T0=0.25, init_x=init, noise_keys=keys)

    def per_frame_variant():
        d, lab, intr = upload()
        outs = [clouds.object_clouds(d[f], lab[f], intr[f], keys[f:f + 1], N) for f in range(F)]
        data = {n: torch.cat([o[n] for o in outs]) for n in ("pts", "pts_center", "counts")}
        return pipe(data, repeat_num=REPEAT, T0=0.25, init_x=init, noise_keys=keys)

    variants = {"frames_call": frames_variant, "per_frame_calls": per_frame_variant}
    for fn in variants.values():   # warm-up: captures the graph, loads every kernel
        fn()
    torch.cuda.synchronize()
    k[0] = 0
    a = frames_variant()
    k[0] = 0
    b = per_frame_variant()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])   # the same poses either way
    host = {n: [] for n in variants}
    for _ in range(args.reps):
        for name, fn in variants.items():
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            host[name].append((time.perf_counter() - t0) * 1e3)
    dev = alternate(variants, args.reps, flush)
    entry = {"videos": F, "frame": f"{W}x{H}", "objects_per_video": 1, "hypotheses": REPEAT, "T0": 0.25,
             "warm_start": True, "step_control": "object", "graphed": True, "keyed": True,
             "frame_to_poses_host_clock_ms": {n: stats(t) for n, t in host.items()},
             "device_event_ms": {n: v["device_ms"] for n, v in dev.items()},
             "host_enqueue_ms": {n: v["host_enqueue_ms"] for n, v in dev.items()},
             "host_cpu": os.cpu_count()}
    print(json.dumps(entry), flush=True)
    result["tracking"] = entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--before-lib", default=None, help="the parent commit's libgenpose_b200.so, for single_frame")
    ap.add_argument("--out", default=os.path.join(HERE, "frames_clouds_b200.json"))
    args = ap.parse_args()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "reps": args.reps, "num_points": N,
              "timing": "device: median CUDA-event ms, L2 overwritten before each timed call; host_enqueue: host clock "
                        "around the enqueue; tracking: host clock around frame in -> poses out with a synchronise at "
                        "the end; variants alternated",
              "frames": [], "single_frame": [], "tracking": None}
    frames(args, flush, result)
    if args.before_lib:
        single_frame(args, flush, result)
    tracking(args, flush, result)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()

"""Per-object point clouds built on the device (genpose2_b200.clouds) against the host preparation they replace.

  stages        CUDA-event device time of Stage A (backproject_instances: depth + labels -> ragged clouds) and Stage B
                (sample_points: ragged clouds -> [B,1024,3] + centres), 640x480 and 1280x720 frames, 8 / 32 / 64 / 256
                objects.  Median over --reps, L2 overwritten before every timed call.
  tracking      a C4-like tracking frame: 32 objects x 50 hypotheses, keyed, step_control="object", graphed, T0 = 0.25
                with warm starts.  Frame in (host depth + labels) to poses out, host clock around the whole step with a
                synchronise at its end, for three ways of making the clouds:
                  device      upload depth + labels, object_clouds on the GPU
                  host_loop   numpy, one mask test per object (as the reference's datasets do), upload pts / pts_center
                  host_sort   numpy, one stable label sort per frame, then slices per object, upload pts / pts_center
                The host variants draw the random choice from numpy's generator, as the datasets do.

The GPU's name and power limit are read in the same run.

    python profiles/object_clouds_bench.py [--reps 20] [--out profiles/object_clouds_b200.json]
"""
import argparse
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

from genpose2_b200 import clouds, synthetic  # noqa: E402
from genpose2_b200.pipeline import PosePipeline  # noqa: E402
from step_control_bench import L2_FLUSH_BYTES, ev_time, gpu_info  # noqa: E402

N = 1024
REPEAT = 50


def intrinsics(H, W):
    return (600.0, 600.0, W / 2.0, H / 2.0)


def host_loop(depth, labels, B, intr, rng):
    """The datasets' preparation: per object a mask test, back-projection and sample_points
    (datasets_omni6dpose.py:459-473)."""
    fx, fy, cx, cy = intr
    H, W = depth.shape
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float32)
    pts = np.zeros((B, N, 3), np.float32)
    for b in range(B):
        m = (labels == b + 1) & (depth > 0)
        pts[b] = _sample(_points(depth[m], xs[m], ys[m], fx, fy, cx, cy), rng)
    return pts, pts.mean(1)


def host_sort(depth, labels, B, intr, rng):
    """One stable label sort per frame, then a slice per object."""
    fx, fy, cx, cy = intr
    H, W = depth.shape
    v, u = np.divmod(np.arange(H * W), W)
    z, lab = depth.reshape(-1), labels.reshape(-1)
    keep = np.nonzero((lab >= 1) & (lab <= B) & (z > 0) & np.isfinite(z))[0]
    keep = keep[np.argsort(lab[keep], kind="stable")]
    bounds = np.searchsorted(lab[keep], np.arange(1, B + 2))
    p_all = _points(z[keep], u[keep].astype(np.float32), v[keep].astype(np.float32), fx, fy, cx, cy)
    pts = np.zeros((B, N, 3), np.float32)
    for b in range(B):
        pts[b] = _sample(p_all[bounds[b]:bounds[b + 1]], rng)
    return pts, pts.mean(1)


def _points(z, x_pix, y_pix, fx, fy, cx, cy):
    return np.stack([(x_pix - cx) * z / fx, (y_pix - cy) * z / fy, z], -1)


def _sample(p, rng):
    K = len(p)
    if K < N:
        return np.concatenate([np.tile(p, (N // K, 1)), p[rng.permutation(K)[:N % K]]])
    if K > N:
        return p[rng.permutation(K)[:N]]
    return p


def stage_times(args, flush, result):
    for H, W in ((480, 640), (720, 1280)):
        for B in (8, 32, 64, 256):
            depth, labels = synthetic.make_instance_frame(H, W, B, seed=B, bad_depth=0.01)
            d, lab = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda()
            keys = torch.arange(B, dtype=torch.int64, device="cuda")
            intr = intrinsics(H, W)
            xyz, off = clouds.backproject_instances(d, lab, intr, B)
            a = ev_time(lambda: clouds.backproject_instances(d, lab, intr, B), args.reps, flush)
            b = ev_time(lambda: clouds.sample_points(xyz, off, N, keys=keys), args.reps, flush)
            both = ev_time(lambda: clouds.object_clouds(d, lab, intr, keys, N), args.reps, flush)
            points = int(off[-1])
            entry = {"frame": f"{W}x{H}", "objects": B, "kept_points": points,
                     "stage_a_ms": dict(zip(("median", "min", "max"), a)),
                     "stage_b_ms": dict(zip(("median", "min", "max"), b)),
                     "object_clouds_ms": dict(zip(("median", "min", "max"), both)),
                     "stage_a_bytes": H * W * 8 + points * 12}
            print(json.dumps(entry), flush=True)
            result["stages"].append(entry)


def tracking(args, flush, result):
    H, W, B = 480, 640, 32
    intr = intrinsics(H, W)
    pipe = PosePipeline(device="cuda", use_graph=True, step_control="object").load_synthetic_weights()
    R0 = synthetic._random_rotations(np.random.default_rng(0), B)
    init = torch.zeros(B, 9)
    init[:, :3] = torch.from_numpy(R0[:, :, 0]).float()
    init[:, 3:6] = torch.from_numpy(R0[:, :, 1]).float()
    init = init.cuda()
    frames = [synthetic.make_instance_frame(H, W, B, seed=s) for s in (105, 107, 124, 139)]   # no object fully covered
    rng = np.random.default_rng(0)
    keys = torch.arange(B, dtype=torch.int64, device="cuda")
    pinned = {"depth": torch.empty((H, W), dtype=torch.float32, pin_memory=True),
              "labels": torch.empty((H, W), dtype=torch.int32, pin_memory=True),
              "pts": torch.empty((B, N, 3), dtype=torch.float32, pin_memory=True),
              "center": torch.empty((B, 3), dtype=torch.float32, pin_memory=True)}
    k = [0]

    def next_frame():
        k[0] += 1
        return frames[k[0] % len(frames)]

    def device_variant():
        depth, labels = next_frame()
        pinned["depth"].copy_(torch.from_numpy(depth))
        pinned["labels"].copy_(torch.from_numpy(labels))
        d = pinned["depth"].to("cuda", non_blocking=True)
        lab = pinned["labels"].to("cuda", non_blocking=True)
        data = clouds.object_clouds(d, lab, intr, keys, N)
        return pipe(data, repeat_num=REPEAT, T0=0.25, init_x=init, noise_keys=keys)

    def host_variant(prep):
        def run():
            depth, labels = next_frame()
            pts, center = prep(depth, labels, B, intr, rng)
            pinned["pts"].copy_(torch.from_numpy(pts))
            pinned["center"].copy_(torch.from_numpy(center))
            data = {"pts": pinned["pts"].to("cuda", non_blocking=True),
                    "pts_center": pinned["center"].to("cuda", non_blocking=True)}
            return pipe(data, repeat_num=REPEAT, T0=0.25, init_x=init, noise_keys=keys)
        return run

    variants = {"device": device_variant, "host_loop": host_variant(host_loop), "host_sort": host_variant(host_sort)}
    for name, fn in variants.items():   # warm-up: captures the graph, loads every kernel
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name in variants}
    prep_ms = {name: [] for name in ("host_loop", "host_sort")}
    for _ in range(args.reps):
        for name, fn in variants.items():   # alternated, so that drift of the shared host affects all alike
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
        for name, prep in (("host_loop", host_loop), ("host_sort", host_sort)):
            depth, labels = next_frame()
            t0 = time.perf_counter()
            prep(depth, labels, B, intr, rng)
            prep_ms[name].append((time.perf_counter() - t0) * 1e3)
    depth, labels = frames[0]
    d, lab = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda()
    dev_step = ev_time(lambda: pipe(clouds.object_clouds(d, lab, intr, keys, N), repeat_num=REPEAT, T0=0.25,
                                    init_x=init, noise_keys=keys), args.reps, flush)
    dev_clouds = ev_time(lambda: clouds.object_clouds(d, lab, intr, keys, N), args.reps, flush)
    entry = {"frame": f"{W}x{H}", "objects": B, "hypotheses": REPEAT, "T0": 0.25, "step_control": "object",
             "graphed": True, "keyed": True,
             "frame_to_poses_host_clock_ms": {n: dict(zip(("median", "min", "max"),
                                                          (float(np.median(t)), float(min(t)), float(max(t)))))
                                              for n, t in times.items()},
             "host_preparation_ms": {n: float(np.median(t)) for n, t in prep_ms.items()},
             "device_object_clouds_plus_step_event_ms": dict(zip(("median", "min", "max"), dev_step)),
             "device_object_clouds_event_ms": dict(zip(("median", "min", "max"), dev_clouds)),
             "host_cpu": os.cpu_count()}
    print(json.dumps(entry), flush=True)
    result["tracking"] = entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(HERE, "object_clouds_b200.json"))
    args = ap.parse_args()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "reps": args.reps, "num_points": N,
              "timing": "device: median CUDA-event ms, L2 overwritten before each timed call; tracking: host clock "
                        "around frame in -> poses out with a synchronise at the end, variants alternated",
              "stages": [], "tracking": None}
    stage_times(args, flush, result)
    tracking(args, flush, result)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()

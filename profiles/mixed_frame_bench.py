"""Per-object start times and keyed per-object noise (PosePipeline(..., T0=[B], noise_keys=[B])) on the workloads of a
tracker:

  mixed frame   32 objects x 50 hypotheses: k in {1, 8, 16} new objects (T0 = 0.55, no warm start), the others
                tracked (T0 = 0.25, init_x).  One graphed mixed step (step_control="object", keys) against the two
                graphed steps needed without per-object T0 (new objects, then tracked objects), in each step control.
  noise cost    C2 (64 objects, T0 = 0.55) and the 1024-object shard, both step controls: a graphed step with the prior
                drawn on the CPU (global generator + pinned upload) against keyed noise generated inside the graph.
                Device ms per step (CUDA events) and host ms per step (host clock around the call, no synchronise).

Device times are medians of CUDA-event timings with the L2 overwritten before every timed step.  The GPU's name and
power limit are read in the same run.

    python profiles/mixed_frame_bench.py [--reps 10] [--out profiles/mixed_frame_b200.json]
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

from genpose2_b200 import samplers, synthetic  # noqa: E402
from genpose2_b200.pipeline import PosePipeline  # noqa: E402
from step_control_bench import L2_FLUSH_BYTES, ev_time, gpu_info  # noqa: E402

REPEAT = 50


def tracking_frame(B, n_new, seed):
    pts, center = synthetic.make_point_clouds(B, 1024, seed=seed)
    R0 = synthetic._random_rotations(np.random.default_rng(seed), B)
    init = torch.zeros(B, 9)
    init[:, :3] = torch.from_numpy(R0[:, :, 0]).float()
    init[:, 3:6] = torch.from_numpy(R0[:, :, 1]).float()
    init[:n_new] = 0.0   # new objects: no warm start
    T = np.full(B, 0.25)
    T[:n_new] = 0.55
    keys = torch.arange(B, dtype=torch.int64) + 1000 * seed
    return {"pts": pts.cuda(), "pts_center": center.cuda()}, init.cuda(), T, keys


def host_ms(fn, reps):
    """host clock around each call (no synchronise inside the window): the host work of a step"""
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
        torch.cuda.synchronize()
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(HERE, "mixed_frame_b200.json"))
    args = ap.parse_args()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "mlp_mode": "fp32", "hypotheses": REPEAT, "reps": args.reps,
              "timing": "median CUDA-event ms, L2 overwritten before each timed step; host ms: host clock around the "
                        "call without a synchronise", "mixed_frame": [], "noise_cost": []}
    pipes = {sc: PosePipeline(device="cuda", use_graph=True, step_control=sc).load_synthetic_weights()
             for sc in samplers.STEP_CONTROLS}
    torch.manual_seed(0)

    B = 32
    for n_new in (1, 8, 16):
        data, init, T, keys = tracking_frame(B, n_new, seed=n_new)
        new, old = slice(0, n_new), slice(n_new, B)
        obj = pipes["object"]
        entry = {"objects": B, "new": n_new, "tracked": B - n_new}
        mixed = lambda: obj(dict(data), repeat_num=REPEAT, T0=T, init_x=init, noise_keys=keys)
        med, lo, hi = ev_time(mixed, args.reps, flush)
        entry["one_mixed_step_object_keyed"] = {"ms_median": med, "ms_min": lo, "ms_max": hi}
        med, lo, hi = ev_time(lambda: obj(dict(data), repeat_num=REPEAT, T0=T, init_x=init), args.reps, flush)
        entry["one_mixed_step_object_cpu_noise"] = {"ms_median": med, "ms_min": lo, "ms_max": hi}
        for sc, pipe in pipes.items():
            def two_steps(pipe=pipe):
                pipe({"pts": data["pts"][new], "pts_center": data["pts_center"][new]}, repeat_num=REPEAT, T0=0.55)
                pipe({"pts": data["pts"][old], "pts_center": data["pts_center"][old]}, repeat_num=REPEAT, T0=0.25,
                     init_x=init[old])
            med, lo, hi = ev_time(two_steps, args.reps, flush)
            entry[f"two_steps_{sc}"] = {"ms_median": med, "ms_min": lo, "ms_max": hi}
        entry["graphs_object_pipeline"] = len(obj._graphs)
        print(json.dumps(entry), flush=True)
        result["mixed_frame"].append(entry)

    for name, B in (("C2", 64), ("C5 shard", 1024)):
        pts, center = synthetic.make_point_clouds(B, 1024, seed=B)
        data = {"pts": pts.cuda(), "pts_center": center.cuda()}
        keys = torch.arange(B, dtype=torch.int64)
        for sc, pipe in pipes.items():
            for noise in ("cpu", "keyed"):
                kw = {"noise_keys": keys} if noise == "keyed" else {}
                fn = lambda: pipe(dict(data), repeat_num=REPEAT, T0=0.55, **kw)
                dmed, dlo, dhi = ev_time(fn, args.reps, flush)
                hmed, hlo, hhi = host_ms(fn, args.reps)
                entry = {"config": name, "objects": B, "T0": 0.55, "step_control": sc, "noise": noise,
                         "device_ms_median": dmed, "device_ms_min": dlo, "device_ms_max": dhi,
                         "host_ms_median": hmed, "host_ms_min": hlo, "host_ms_max": hhi}
                print(json.dumps(entry), flush=True)
                result["noise_cost"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()

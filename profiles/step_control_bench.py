"""Cost of per-object RK45 step control (cond_ode_sampler(..., step_control="object")) against the shared batch
controller, on the workloads users run:

  C2        64 objects x 50 hypotheses, T0 = 0.55, full PosePipeline step replayed as one CUDA graph
  C4        32 objects x 50 hypotheses, T0 = 0.25 with init_x (tracking), full graphed step
  C5 shard  1024 objects x 50 hypotheses, T0 = 0.55, full graphed step (one GPU's shard of a large batch)

For each: ms/step (median of CUDA-event timings, L2 overwritten before every timed step), the batch controller's nfev
and the per-object nfev min / median / max.  The sampler alone is also timed for each tensor-core evaluator shape
(cluster per object, one CTA per object) on both sides of the 32-object threshold of the automatic choice.  The GPU's
name and power limit are read in the same run.

    python profiles/step_control_bench.py [--reps 10] [--out profiles/step_control_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from genpose2_b200 import samplers, synthetic  # noqa: E402
from genpose2_b200.pipeline import PosePipeline  # noqa: E402
from oracle import pose_oracle as po  # noqa: E402

REPEAT = 50
CONFIGS = [("C2", 64, 0.55, False), ("C4", 32, 0.25, True), ("C5 shard", 1024, 0.55, False)]
L2_FLUSH_BYTES = 256 << 20   # twice the 126 MB L2


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + q,
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")] if out.count(",") == 2 else (out, "?", "?")
    return {"name": name or torch.cuda.get_device_name(), "power_limit": power, "max_sm_clock": clock}


def ev_time(fn, reps, flush):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def workload(B, T0, tracking, seed):
    pts, center = synthetic.make_point_clouds(B, 1024, seed=seed)
    init = None
    if tracking:
        R0 = synthetic._random_rotations(np.random.default_rng(seed), B)
        init = torch.zeros(B, 9)
        init[:, :3] = torch.from_numpy(R0[:, :, 0]).float()
        init[:, 3:6] = torch.from_numpy(R0[:, :, 1]).float()
        init = init.cuda()
    noise = po.ve_prior((B * REPEAT, 9), T=T0).float()
    return {"pts": pts.cuda(), "pts_center": center.cuda()}, init, noise


def nfev_summary(st):
    if "obj_nfev" not in st:
        return {"nfev": st["nfev"], "accepted": st["accepted"], "rejected": st["rejected"]}
    n = st["obj_nfev"]
    return {"nfev_max": int(n.max()), "nfev_min": int(n.min()), "nfev_median": float(np.median(n)),
            "nfev_mean": float(n.mean()), "accepted_median": float(np.median(st["obj_accepted"])),
            "rejected_total": int(st["rejected"])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "step_control_b200.json"))
    args = ap.parse_args()
    dev = torch.device("cuda")
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    result = {"gpu": gpu_info(), "mlp_mode": "fp32", "hypotheses": REPEAT, "reps": args.reps,
              "timing": "median CUDA-event ms, L2 overwritten before each timed run", "configs": []}
    pipes = {sc: PosePipeline(device="cuda", use_graph=True, step_control=sc).load_synthetic_weights()
             for sc in samplers.STEP_CONTROLS}
    for name, B, T0, tracking in CONFIGS:
        data, init, noise = workload(B, T0, tracking, seed=B)
        entry = {"config": name, "objects": B, "T0": T0, "init_x": tracking, "step": {}, "sampler_only": {}}
        for sc, pipe in pipes.items():
            pipe.score_agent.net.prior_fn = lambda shape, T=1.0: noise.clone()
            med, lo, hi = ev_time(lambda: pipe(dict(data), repeat_num=REPEAT, T0=T0, init_x=init), args.reps, flush)
            st = samplers.ode_stats()
            assert st["status"] == 0, st
            entry["step"][sc] = {"ms_median": med, "ms_min": lo, "ms_max": hi, **nfev_summary(st)}
            print(f"{name} step [{sc}]: {med:.2f} ms ({lo:.2f}..{hi:.2f}) {nfev_summary(st)}", flush=True)
        # the sampler alone, per evaluator shape: features of the step's encoder, same noise
        net = pipes["batch"].score_agent.net
        feat = net(data, mode="pts_feature")
        sdata = {"pts": torch.zeros(B * REPEAT, 1, 3),
                 "pts_center": data["pts_center"].repeat_interleave(REPEAT, 0).contiguous(),
                 "_gp_pts_feat_obj": feat, "_gp_rows_per_object": REPEAT}
        rinit = None if init is None else init.repeat_interleave(REPEAT, 0)
        runs = [("batch", "auto"), ("object", "auto"), ("object", "solo")] + ([("object", "cluster")] if B <= 64 else [])
        for sc, shape in runs:
            net.pose_score_net.eval_shape = shape
            fn = lambda: samplers.cond_ode_sampler(net, dict(sdata), lambda s, T: noise.clone(), net.sde_fn, device="cuda",
                                                   T=T0, pose_mode="rot_matrix", init_x=rinit, return_trajectory=False,
                                                   step_control=sc)
            med, lo, hi = ev_time(fn, args.reps, flush)
            st = samplers.ode_stats()
            entry["sampler_only"][f"{sc}/{shape}"] = {"ms_median": med, "ms_min": lo, "ms_max": hi, **nfev_summary(st)}
            print(f"{name} sampler [{sc}/{shape}]: {med:.2f} ms", flush=True)
        net.pose_score_net.eval_shape = "auto"
        result["configs"].append(entry)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()

"""Trunk arithmetic "tf32" (tf32 operands on the tensor cores, 2 MMAs per 16 k) against "fp32" (split-bf16 x3, 3 MMAs
per 16 k) and "bf16" (1 MMA per 16 k) on the workloads users run:

  C2        64 objects x 50 hypotheses, T0 = 0.55: the sampler alone and the full PosePipeline step as one CUDA graph
  C4        32 objects x 50 hypotheses, T0 = 0.25 with init_x (tracking): the sampler alone and the full graphed step
  C5 shard  1024 objects x 50 hypotheses, T0 = 0.55: the sampler alone and the full graphed step (one GPU's shard)

The three modes are timed alternately inside every repetition (fp32, tf32, bf16, fp32, ...), so that clock and
neighbour drift hit them alike; ms are medians of CUDA-event timings with the L2 overwritten before every timed run.
All modes see the same features (the fp32 pipeline's encoder) and the same prior noise.  Recorded per mode: nfev /
accepted / rejected of the batch controller, and for tf32 and bf16 the largest per-hypothesis rotation (rad) and
translation difference against fp32 on the same inputs.  The GPU's name, power limit and SM clocks are read in the
same run.

    python profiles/tf32_bench.py [--reps 10] [--out profiles/tf32_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from genpose2_b200 import samplers  # noqa: E402
from genpose2_b200.pipeline import PosePipeline  # noqa: E402
from step_control_bench import L2_FLUSH_BYTES, workload  # noqa: E402
from tests.util import pose_errors  # noqa: E402

REPEAT = 50
MODES = ["fp32", "tf32", "bf16"]
CONFIGS = [("C2", 64, 0.55, False), ("C4", 32, 0.25, True), ("C5 shard", 1024, 0.55, False)]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + q,
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    f = [s.strip() for s in out.split(",")]
    if len(f) != 4:
        f = [torch.cuda.get_device_name(), "?", "?", "?"]
    return {"name": f[0], "power_limit": f[1], "sm_clock": f[2], "max_sm_clock": f[3]}


def alternating(fns, reps, flush):
    """{mode: fn} -> {mode: (median, min, max) ms}; every repetition times each mode once, in turn"""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    ts = {m: [] for m in fns}
    for _ in range(reps):
        for m, fn in fns.items():
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts[m].append(s.elapsed_time(e))
    return {m: {"ms_median": float(np.median(v)), "ms_min": float(min(v)), "ms_max": float(max(v))} for m, v in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(HERE, "tf32_b200.json"))
    args = ap.parse_args()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "hypotheses": REPEAT, "reps": args.reps,
              "timing": "median CUDA-event ms over reps, modes alternated within each rep, L2 overwritten before "
                        "each timed run", "configs": []}
    pipes = {m: PosePipeline(device="cuda", use_graph=True, mlp_mode=m).load_synthetic_weights() for m in MODES}
    for name, B, T0, tracking in CONFIGS:
        data, init, noise = workload(B, T0, tracking, seed=B)
        entry = {"config": name, "objects": B, "T0": T0, "init_x": tracking}
        # the sampler alone: same features, same noise, every mode
        feat = pipes["fp32"].score_agent.net(data, mode="pts_feature")
        sdata = {"pts": torch.zeros(B * REPEAT, 1, 3),
                 "pts_center": data["pts_center"].repeat_interleave(REPEAT, 0).contiguous(),
                 "_gp_pts_feat_obj": feat, "_gp_rows_per_object": REPEAT}
        rinit = None if init is None else init.repeat_interleave(REPEAT, 0)
        out = {}

        def sampler(m):
            net = pipes[m].score_agent.net

            def fn():
                _, x = samplers.cond_ode_sampler(net, dict(sdata), lambda s, T: noise.clone(), net.sde_fn,
                                                 device="cuda", T=T0, pose_mode="rot_matrix", init_x=rinit,
                                                 return_trajectory=False)
                out[m] = x
            return fn

        entry["sampler_only"] = alternating({m: sampler(m) for m in MODES}, args.reps, flush)
        for m in MODES:   # one more run per mode for its statistics and poses
            sampler(m)()
            st = samplers.ode_stats()
            assert st["status"] == 0, (m, st)
            entry["sampler_only"][m].update(nfev=st["nfev"], accepted=st["accepted"], rejected=st["rejected"])
            if m != "fp32":
                rot, trans = pose_errors(out[m].cpu().numpy(), out["fp32"].cpu().numpy())
                entry["sampler_only"][m].update(max_rot_vs_fp32=rot, max_trans_vs_fp32=trans)
        for pipe in pipes.values():
            pipe.score_agent.net.prior_fn = lambda shape, T=1.0: noise.clone()
        entry["step"] = alternating({m: (lambda p=p: p(dict(data), repeat_num=REPEAT, T0=T0, init_x=init))
                                     for m, p in pipes.items()}, args.reps, flush)
        for m in MODES:
            entry["step"][m]["graphs"] = len(pipes[m]._graphs)
        print(json.dumps(entry), flush=True)
        result["configs"].append(entry)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()

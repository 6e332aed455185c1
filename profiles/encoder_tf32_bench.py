"""Encoder operand precision "tf32" (npass = 2: tf32 operands, tcgen05 kind::tf32, 8 MMAs per 64 k) against the split
mode "bf16x3" (npass = 3, 12 MMAs per 64 k) of the set-abstraction GEMMs, on the workloads users run:

  encoder   Pointnet2ClsMSG alone at 64 (C2) and 1024 objects (one GPU's C5 shard): the whole pass, the pass split by
            level (CUDA events around each set-abstraction module), and -- in a separate torch.profiler run -- the device
            time of every tensor-core kernel launch of a pass, in launch order
  step      the full PosePipeline step as one CUDA graph at C2 (64 objects) and the C5 shard (1024 objects), 50
            hypotheses, T0 = 0.55, for (mlp_mode, encoder_mode) = (fp32, auto), (fp32, tf32), (tf32, auto), (tf32, tf32)

The variants of a measurement are timed alternately inside every repetition, so that clock and neighbour drift hit them
alike; ms are medians of CUDA-event timings with the L2 overwritten before every timed run.  Recorded beside the times:
the encoder's feature difference against the split mode (max over the scale of the split mode's features) and, per
step variant, nfev and the largest per-hypothesis rotation (rad) / translation difference against (fp32, auto) on the
same inputs and noise.  The GPU's name, power limit and SM clocks are read in the same run.

    python profiles/encoder_tf32_bench.py [--reps 10] [--out profiles/encoder_tf32_b200.json]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from genpose2_b200 import samplers, synthetic  # noqa: E402
from genpose2_b200.pipeline import PosePipeline  # noqa: E402
from genpose2_b200.pointnet2 import Pointnet2ClsMSG  # noqa: E402
from step_control_bench import L2_FLUSH_BYTES, workload  # noqa: E402
from tests.util import pose_errors  # noqa: E402
from tf32_bench import alternating, gpu_info  # noqa: E402

REPEAT = 50
ENC_MODES = ["bf16x3", "tf32"]
ENC_SIZES = [64, 1024]
STEP_VARIANTS = [("fp32", "auto"), ("fp32", "tf32"), ("tf32", "auto"), ("tf32", "tf32")]
STEP_CONFIGS = [("C2", 64), ("C5 shard", 1024)]


def encoder(sd, mode):
    enc = Pointnet2ClsMSG(0).cuda().eval().set_gemm_mode(mode)
    enc.load_state_dict(sd)
    return enc


def per_level(enc, pts, reps, flush):
    """median ms of each set-abstraction module (level) inside a whole pass"""
    evs = []
    originals = []
    for sa in enc.SA_modules:
        orig = sa.forward_cl

        def timed(*a, _orig=orig, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = _orig(*a, **kw)
            e.record()
            evs.append((s, e))
            return r
        originals.append(orig)
        sa.forward_cl = timed
    ts = [[] for _ in enc.SA_modules]
    try:
        with torch.no_grad():
            for _ in range(reps):
                flush.zero_()
                evs.clear()
                enc(pts)
                torch.cuda.synchronize()
                for k, (s, e) in enumerate(evs):
                    ts[k].append(s.elapsed_time(e))
    finally:
        for sa in enc.SA_modules:
            del sa.forward_cl
    return [float(np.median(t)) for t in ts]


def kernel_launches(enc, pts):
    """device time (us) of the tensor-core kernels of one pass, in launch order (torch.profiler, separate run)"""
    from torch.profiler import ProfilerActivity, profile
    with torch.no_grad():
        enc(pts)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            enc(pts)
            torch.cuda.synchronize()
    out = []
    for ev in prof.events():
        if "sa_mlp2_kernel" in ev.name or "gemm_bias_relu_kernel" in ev.name:
            out.append((ev.time_range.start, ev.name.split("(")[0].replace("void gp::", ""), ev.time_range.elapsed_us()))
    out.sort()
    return [{"kernel": n, "us": round(float(t), 1)} for _, n, t in out]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(HERE, "encoder_tf32_b200.json"))
    args = ap.parse_args()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "hypotheses": REPEAT, "reps": args.reps,
              "timing": "median CUDA-event ms over reps, variants alternated within each rep, L2 overwritten before "
                        "each timed run", "encoder": [], "step": []}
    sd = synthetic.random_encoder_state_dict(100, prefix="")
    encs = {m: encoder(sd, m) for m in ENC_MODES}
    for B in ENC_SIZES:
        pts, _ = synthetic.make_point_clouds(B, 1024, seed=B, dup_fraction=0.25)
        pts = pts.cuda()
        entry = {"objects": B}
        feats = {}

        def run(m):
            def fn():
                with torch.no_grad():
                    feats[m] = encs[m](pts)
            return fn
        entry["pass"] = alternating({m: run(m) for m in ENC_MODES}, args.reps, flush)
        entry["feature_err_vs_bf16x3"] = float((feats["tf32"] - feats["bf16x3"]).abs().max() / feats["bf16x3"].abs().max())
        entry["levels_ms"] = {m: per_level(encs[m], pts, args.reps, flush) for m in ENC_MODES}
        entry["launches"] = {m: kernel_launches(encs[m], pts) for m in ENC_MODES}
        print(json.dumps({k: v for k, v in entry.items() if k != "launches"}), flush=True)
        result["encoder"].append(entry)
    del encs
    pipes = {f"{m}/{e}": PosePipeline(device="cuda", use_graph=True, mlp_mode=m, encoder_mode=e).load_synthetic_weights()
             for m, e in STEP_VARIANTS}
    for name, B in STEP_CONFIGS:
        data, init, noise = workload(B, 0.55, False, seed=B)
        for pipe in pipes.values():
            pipe.score_agent.net.prior_fn = lambda shape, T=1.0: noise.clone()
        entry = {"config": name, "objects": B, "T0": 0.55}
        entry["step"] = alternating({k: (lambda p=p: p(dict(data), repeat_num=REPEAT, T0=0.55)) for k, p in pipes.items()},
                                    args.reps, flush)
        poses = {}
        for k, p in pipes.items():   # one eager run per variant for its statistics and poses
            poses[k] = p(dict(data), repeat_num=REPEAT, T0=0.55, return_all=True)["pred_pose"].cpu().numpy()
            st = samplers.ode_stats()
            assert st["status"] == 0, (k, st)
            entry["step"][k].update(nfev=st["nfev"], graphs=len(p._graphs))
        for k in pipes:
            if k != "fp32/auto":
                rot, trans = pose_errors(poses[k], poses["fp32/auto"])
                entry["step"][k].update(max_rot_vs_fp32_auto=rot, max_trans_vs_fp32_auto=trans)
        print(json.dumps(entry), flush=True)
        result["step"].append(entry)
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()

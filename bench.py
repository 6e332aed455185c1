#!/usr/bin/env python
"""bench.py -- objects/s of the per-object pose-generation hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (libgenpose_b200.so)
    python bench.py --impl reference --gpus N ...             # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                    # also writes the last timed step's outputs as DIR/*.npy

A "step" is one pass of the full path (PointNet++ encoder x2 -> RK45 ScoreNet sampling, 50 hypotheses/object ->
EnergyNet scoring -> aggregation -> ScaleNet) over one batch of synthetic objects.

Headline workload = BASELINE.json configs[1] (C2): 64 objects x 50 hypotheses per GPU, T0 = 0.55
(scripts/eval_single.sh), random-init weights, synthetic clouds.  Multi-GPU: objects are sharded by rank, no
collective on the data path, weak scaling (64 objects per GPU).

`value`   : objects/s with the clouds already resident in HBM (CUDA events, max over ranks).
`e2e`     : objects/s through the same public call with HOST (pinned) clouds: H2D copy of the clouds and D2H read of
            the poses + lengths inside the timed region.
`roofline`: the dominant kernel of this library (the fused ScoreNet / RK45 integrator), algorithmic FLOPs (SURVEY.md
            8(d), hoisted figure) / CUDA-event duration, against MEASURED_PEAKS.json (burst AND sustained).
`cpu_baseline`: the reference's own CPU path (oracle/_ref/refpkg: the unmodified reference modules; its CUDA-only
            encoder through the oracle port) timed on this box's host cores on a bounded sample of the workload.
`other_configs`: the other BASELINE.json configs, measured in the same run after the timed region:
            c5 (8192 objects x 50 sharded by object over the N ranks, STRONG scaling, the one gather in the timed
            region, fp32 and bf16), and at N = 1: c1 (1 object latency, sampler only, T0 = 1), c3 (FPS / ball query /
            grouping sweep 1024..16384 points x 256 objects, beside the reference's own CUDA ext), c4 (tracking,
            32 objects / frame over a 100-frame synthetic sequence).
`reference_gpu`: the UNMODIFIED reference on this GPU (torch + host scipy loop + sklearn, its own CUDA ext): the
            denominator of north_star's ">= 100x the reference's 1-GPU torch+scipy sampling throughput".
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "objects_per_sec_50hyp"
UNIT = "objects/s"
OBJECTS_PER_GPU = 64
REPEAT = 50
T0 = 0.55
NUM_POINTS = 1024
L2_FLUSH_BYTES = 256 << 20
C5_OBJECTS = 8192

# dram__bytes_read.sum + dram__bytes_write.sum of the integrator kernel per launch at C2.  A CONSTANT taken from the
# `ncu --set full` captures summarised in profiles/README.md (not a per-run counter: ncu cannot run inside the bench).
NCU_DRAM_BYTES_PER_LAUNCH = {"fp32_ffma": 2270464 + 22784, "bf16": 1686784 + 58368, "fp32": 2249472 + 72960}
NCU_DRAM_SOURCE = "constant from the ncu --set full capture in profiles/README.md (C2, cluster evaluator), not a per-run counter"

# algorithmic work of the ScoreNet RHS after hoisting (SURVEY.md 8(d)), in FLOP
ROW_EVAL_FLOP = 2 * 266752
STAGE_SHARED_FLOP = 2 * 114688
OBJECT_ONCE_FLOP = 2 * 786432


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps, all of which run (after the warm-up), in either arm")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--objects", type=int, default=OBJECTS_PER_GPU, help="objects per GPU per step")
    ap.add_argument("--mlp_mode", type=str, default="fp32", choices=["fp32", "fp32_ffma", "bf16"])
    ap.add_argument("--cpu_sample_objects", type=int, default=8, help="cpu_baseline sample of the B200 arm")
    ap.add_argument("--ref_objects", type=int, default=OBJECTS_PER_GPU, help="objects per step of --impl reference")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--single_mode", action="store_true", help="skip the measurement of the other mlp_mode")
    ap.add_argument("--no_extras", action="store_true", help="skip other_configs and reference_gpu")
    ap.add_argument("--c5_objects", type=int, default=C5_OBJECTS)
    ap.add_argument("--graph", type=str, default="on", choices=["on", "off"],
                    help="replay the step as one CUDA graph (PosePipeline(use_graph=True)); falls back to eager launches if the capture fails")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (aggregated_pose [B,4,4], "
                         "length [B,3], all ranks' objects in order) as DIR/<name>.npy in float32, in either arm")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


_SAMPLER_CODE = r"""
import sys, time
idx = int(sys.argv[1])
try:
    import pynvml as n
    n.nvmlInit()
    h = n.nvmlDeviceGetHandleByIndex(idx)
    get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
    mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
    print("ready nvml", flush=True)
    while True:
        print(time.time(), n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), mx, int(get(h)), flush=True)
        time.sleep(0.004)
except Exception as e:
    import subprocess
    print("ready nvidia-smi", flush=True)
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while True:
        t = time.time()
        out = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout
        p = [x.strip() for x in out.strip().split(",")]
        if len(p) >= 6:
            bits = sum(b for b, v in zip((0x8, 0x40, 0x20, 0x4), p[2:6]) if v.lower().startswith("active"))
            print(t, p[0], p[1], bits, flush=True)
"""


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region by a helper process (NVML every ~4 ms, or
    `nvidia-smi` when NVML cannot be initialised): a thread in this process would have to fight the step loop for
    the GIL.  The helper is started at construction (before the warm-up); only its samples with a wall-clock stamp
    inside [start(), stop()] are kept."""
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        phys = index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:  # torch's index counts visible devices
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                phys = int(ids[index])
        self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_CODE, str(phys)], stdout=subprocess.PIPE, text=True)
        self.source = (self.proc.stdout.readline().split() + ["?", "?"])[1]
        self.t0 = self.t1 = None

    def start(self):
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        time.sleep(0.02)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], 0.0, set()
        for line in out.splitlines():
            p = line.split()
            if len(p) != 4:
                continue
            try:
                t, clk, mxc, bits = float(p[0]), float(p[1]), float(p[2]), int(p[3])
            except ValueError:
                continue
            if not (self.t0 <= t <= self.t1):
                continue
            sm.append(clk)
            mx = max(mx, mxc)
            reasons.update(name for name, b in self.BITS if bits & b)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "source": self.source}


def synthetic_weights():
    from genpose2_b200 import synthetic
    return (synthetic.random_gfobjectpose_state_dict(100), synthetic.random_gfobjectpose_state_dict(200),
            synthetic.random_scalenet_state_dict(300))


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU path on the host cores
# --------------------------------------------------------------------------------------------------
class CpuReference:
    """One step = `n` objects x 50 hypotheses through the reference's CPU path: pred_func (scipy RK45 host loop) ->
    get_energy -> aggregation block (sklearn DBSCAN) -> pred_scale_func, all the UNMODIFIED reference modules
    (oracle/_ref/refpkg; kind "reference").  The reference's encoder is a CUDA-only extension, so the two encoder
    passes of a step are the oracle port's (oracle/pose_oracle.py:pointnet2_encoder: C restatement of FPS / ball query /
    grouping + torch-CPU conv / BN / max-pool, pinned to the reference on the GPU box by tests/test_gpu_reference.py),
    timed inside the step, their features injected.  Without oracle/_ref/refpkg the whole step is the oracle port
    (kind "port")."""

    def __init__(self, n_max):
        import torch
        from genpose2_b200 import synthetic
        from oracle import ref_shim
        torch.set_num_threads(os.cpu_count() or 1)
        self.pts, self.center = synthetic.make_point_clouds(max(n_max, 1), NUM_POINTS, seed=0)
        self.sds = synthetic_weights()
        self.kind = "port"
        self.agents = None
        if ref_shim.available():
            try:
                from oracle.ref_runner import ReferenceAgents
                self.agents = ReferenceAgents(*self.sds, device="cpu", inject_features=True)
                self.kind = "reference"
            except Exception as e:  # noqa: BLE001
                print("reference modules not loadable, timing the oracle port instead:", e, file=sys.stderr)

    def step(self, n):
        """-> (seconds, seconds spent in the two encoder passes, (aggregated_pose, length))"""
        import torch
        from oracle import pose_oracle as po
        pts, center = self.pts[:n], self.center[:n]
        t0 = time.perf_counter()
        if self.agents is None:
            torch.manual_seed(1)
            noise = po.ve_prior((n * REPEAT, 9), T=T0)
            out = po.full_pipeline(self.sds[0], self.sds[1], self.sds[2], pts, center, noise, repeat_num=REPEAT, T0=T0,
                                   integrator="scipy")
            return time.perf_counter() - t0, None, (out["aggregated_pose"], out["length"])
        with torch.no_grad():
            sfeat = po.pointnet2_encoder(self.sds[0], pts)
            efeat = po.pointnet2_encoder(self.sds[1], pts)
        t_enc = time.perf_counter() - t0
        out = self.agents.full(pts, center, REPEAT, T0, noise_seed=1, score_feat=sfeat, energy_feat=efeat)
        return time.perf_counter() - t0, t_enc, (out["aggregated_pose"], out["length"])

    def describe(self, n, steps, enc_share):
        what = ("reference modules (oracle/_ref/refpkg): torch-CPU nets + scipy RK45 + sklearn DBSCAN; the CUDA-only "
                "encoder through the oracle port" if self.kind == "reference"
                else "oracle port: torch-CPU nets + scipy RK45 + sklearn DBSCAN")
        s = f"{n} objects x {REPEAT} hypotheses per step, full path incl. both encoders, {steps} step(s) ({what})"
        if enc_share is not None:
            s += f"; encoders = {100 * enc_share:.0f}% of the step"
        return s


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU reference; other ranks exit without work
    import torch
    n = args.ref_objects
    ref = CpuReference(n)
    ref.step(min(n, 4))  # warm-up (thread pools, imports) on a few objects: a full-size step takes seconds on the host
    times, encs = [], []
    for _ in range(args.steps):
        dt, enc, outputs = ref.step(n)
        times.append(dt)
        encs.append(enc)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *outputs, rank)
    total = sum(times)
    value = n * len(times) / total
    cores = torch.get_num_threads()
    enc_share = None if encs[0] is None else sum(encs) / total
    sample = ref.describe(n, len(times), enc_share)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "steps_timed": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C2: {OBJECTS_PER_GPU} objects x {REPEAT} hypotheses, full path, T0={T0}",
                   "objects_per_step": n, "same_config": n == OBJECTS_PER_GPU},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": ref.kind, "sample": sample,
                         "os_cpu_count": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# helpers of the B200 arm
# --------------------------------------------------------------------------------------------------
def ev_time(fn, reps, flush=None):
    """median CUDA-event milliseconds of fn() over `reps` runs (after one untimed run)"""
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts.sort()
    return ts[len(ts) // 2]


def load_ref_ext():
    """The reference's own CUDA extension (oracle/_ref/pointnet2_cuda.so), or None."""
    d = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(d, "pointnet2_cuda.so")):
        return None
    if d not in sys.path:
        sys.path.insert(0, d)
    try:
        import pointnet2_cuda
        return pointnet2_cuda
    except Exception:  # noqa: BLE001
        return None


def dump_outputs(out_dir, pose, length, rank):
    """--dump-outputs: the last timed step's results, gathered over the ranks in object order, as float32 .npy files.
    The clouds, weights and prior noise depend on the arguments alone, so two builds can be compared output for output."""
    import numpy as np
    from genpose2_b200.pipeline import gather_results
    pose, length = gather_results(pose, length)
    if rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("aggregated_pose", pose), ("length", length)):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def sampler_inputs(net, feat, center_d, B, T, seed=99):
    import torch
    N = B * REPEAT
    sdata = {"pts": torch.empty(N, 0), "pts_center": center_d.unsqueeze(1).expand(B, REPEAT, 3).reshape(N, 3).contiguous(),
             "_gp_pts_feat_obj": feat, "_gp_rows_per_object": REPEAT}
    torch.manual_seed(seed)
    noise = net.prior_fn((N, 9), T=T)
    return sdata, noise


def sampler_roofline(net, sdata, noise, B, T, peaks, mlp_mode, dev, flush, reps, kernel_name):
    """Roofline of the integrator kernel alone: algorithmic FLOPs / CUDA-event time (projection kernel included)."""
    from genpose2_b200 import samplers
    prior = lambda shape, T=1.0: noise  # noqa: E731

    def sampler_only():
        return samplers.cond_ode_sampler(net, sdata, prior, net.sde_fn, device=dev, eps=1e-5, T=T,
                                         pose_mode="rot_matrix", return_trajectory=False)

    k_med = ev_time(sampler_only, reps, flush)
    st = samplers.ode_stats()
    N = B * REPEAT
    nfev_total = st["nfev"] + 1  # + the denoise evaluation
    flop = N * nfev_total * ROW_EVAL_FLOP + nfev_total * STAGE_SHARED_FLOP + B * OBJECT_ONCE_FLOP
    achieved = flop / (k_med * 1e-3) / 1e12
    ffma_peak = 148 * 128 * 2 * 1.965e9 / 1e12  # 148 SMs x 128 FP32 lanes x 2 FLOP x max SM clock
    return {
        "bound": "tensor", "kernel": kernel_name, "achieved": achieved, "unit": "TFLOP/s",
        # the kernel is timed alone (a few ms): the burst figure is the honest denominator; the sustained one beside it
        "peak": peaks["bf16_tflops"], "frac": achieved / peaks["bf16_tflops"],
        "peak_sustained": peaks["bf16_tflops_sustained"], "frac_of_sustained": achieved / peaks["bf16_tflops_sustained"],
        "peak_source": f"{peaks['source']} bf16 dense (MEASURED_PEAKS.json): burst; sustained beside it",
        "mlp_mode": mlp_mode, "kernel_ms": k_med, "nfev": nfev_total, "accepted": st["accepted"], "rejected": st["rejected"],
        "algorithmic_flop_per_launch": flop, "hyp_evals_per_s": N * nfev_total / (k_med * 1e-3),
        "issued_over_algorithmic": {"fp32": 3.0, "bf16": 1.0, "fp32_ffma": 1.0}[mlp_mode],
        "note": {"fp32_ffma": "MLPs on FP32 FFMA (no tensor cores): also quoted against the FP32 FFMA peak",
                 "fp32": "split-bf16 x3 on tcgen05 (3 MMAs per product, fp32-class accuracy); achieved counts the "
                         "algorithmic FLOPs once, so the tensor pipe does 3x that",
                 "bf16": "bf16 operands on tcgen05, fp32 accumulation in TMEM"}[mlp_mode],
        "ffma_peak_tflops": ffma_peak, "frac_of_ffma_peak": achieved / ffma_peak,
    }


# --------------------------------------------------------------------------------------------------
# other BASELINE configs (after the headline's timed region)
# --------------------------------------------------------------------------------------------------
def bench_c5(args, world, rank, dev, peaks, barrier):
    """C5: `c5_objects` objects x 50 hypotheses sharded by object over the ranks (contiguous shards, SURVEY 8(e)): strong
    scaling.  Per step: the full path on this rank's shard (encoders in passes of <= 1024 objects; ONE RK45 sampler
    call over the whole shard -- the step controller is shared per shard, like the reference run once per shard) and
    the single gather of [B,4,4] + [B,3] (NCCL all_gather) INSIDE the timed region."""
    import torch
    import torch.distributed as dist
    from genpose2_b200 import samplers, synthetic
    from genpose2_b200.pipeline import PosePipeline, gather_results, shard_range
    total = args.c5_objects
    lo, hi = shard_range(total, rank, world)
    Bl = hi - lo
    # the clouds of the 8192 objects: 512 distinct synthetic clouds repeated (generation cost only; every object is processed)
    base_pts, base_center = synthetic.make_point_clouds(512, NUM_POINTS, seed=5)
    idx = torch.arange(lo, hi) % 512
    pts_d, center_d = base_pts[idx].to(dev), base_center[idx].to(dev)
    out = {"objects_total": total, "objects_this_rank": Bl, "scaling": "strong",
           "gather": ("NCCL all_gather of [B,4,4]+[B,3] inside the timed region" if world > 1 else "single rank: nothing to gather"),
           "note": "encoders run in passes of <= 1024 objects; one RK45 sampler call per shard (shared step controller per shard)"}
    steps = 3
    for mode in ("fp32", "bf16"):
        pipe = PosePipeline(device=str(dev), mlp_mode=mode).load_synthetic_weights((100, 200, 300))

        def step():
            pose, length = pipe({"pts": pts_d, "pts_center": center_d}, repeat_num=REPEAT, T0=T0)
            return gather_results(pose, length)

        torch.manual_seed(4321 + rank)
        step()
        torch.cuda.synchronize()
        barrier()
        evs = []
        for _ in range(steps):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            pose, length = step()
            e.record()
            evs.append((s, e))
        torch.cuda.synchronize()
        barrier()
        ms = sum(s.elapsed_time(e) for s, e in evs)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        st = samplers.ode_stats()
        ok = bool(torch.isfinite(pose).all()) and pose.shape[0] == total
        res = {"value": total * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
               "nfev_this_shard": st["nfev"] + 1, "status": st["status"], "gathered_ok": ok,
               "hyp_evals_per_s": total * REPEAT * (st["nfev"] + 1) * steps / (ms * 1e-3)}
        # roofline of the sampler kernel on this rank's shard (one-CTA-per-tile evaluator at this size)
        net = pipe.score_agent.net
        feat = pipe._encode(pipe.score_agent, pts_d)[0]
        sdata, noise = sampler_inputs(net, feat, center_d, Bl, T0)
        res["roofline"] = sampler_roofline(
            net, sdata, noise.to(dev), Bl, T0, peaks, mode, dev, None, 3,
            "ode_rk45_kernel<TcSolo<%d>> (one CTA per 128-row tile)" % (3 if mode == "fp32" else 1)
            if Bl * REPEAT > 32 * 128 else "ode_rk45_kernel<TcEval> (4-CTA clusters)")
        out[mode] = res
        del pipe
        torch.cuda.empty_cache()
    return out


def bench_c1(dev, flush):
    """C1: 1 object x 50 hypotheses, ScoreNet ODE sampling only, T0 = 1.0 (BASELINE.json configs[0]): latency."""
    import torch
    from genpose2_b200 import samplers
    from genpose2_b200.pipeline import PosePipeline
    out = {"workload": "1 object x 50 hypotheses, cond_ode_sampler only, T0 = 1.0, rtol = atol = 1e-5"}
    g = torch.Generator().manual_seed(11)
    feat = torch.relu(torch.randn(1, 1024, generator=g))
    center = torch.randn(1, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 0.8])
    for mode in ("fp32", "bf16"):
        pipe = PosePipeline(device=str(dev), mlp_mode=mode).load_synthetic_weights((100, 200, 300))
        net = pipe.score_agent.net
        sdata, noise = sampler_inputs(net, feat.to(dev), center.to(dev), 1, 1.0, seed=1)
        noise = noise.to(dev)
        ms = ev_time(lambda: samplers.cond_ode_sampler(net, sdata, lambda s, T=1.0: noise, net.sde_fn, device=dev, T=1.0,
                                                       pose_mode="rot_matrix", return_trajectory=False), 10, flush)
        st = samplers.ode_stats()
        out[mode] = {"latency_ms": ms, "nfev": st["nfev"] + 1, "objects_per_s": 1e3 / ms}
    return out, feat, center


def bench_c3(dev):
    """C3: FPS / ball query / grouping at 1024..16384 points x 256 objects, ours beside the reference's own CUDA ext
    (sampling_gpu.cu:93-253, ball_query_gpu.cu:9-45, group_points_gpu.cu:47-66) on the same clouds, CUDA events."""
    import torch
    from genpose2_b200 import pointnet2_utils as pu, synthetic
    ext = load_ref_ext()
    B = 256
    rows = []
    for N in (1024, 2048, 4096, 8192, 16384):
        pts, _ = synthetic.make_point_clouds(32, N, seed=N)
        xyz = pts.repeat(B // 32, 1, 1).contiguous().to(dev)
        M = N // 2
        scale = (1024.0 / N) ** 0.5   # keeps the expected neighbour count of the level-1 radii
        radii, ns = (0.01 * scale, 0.02 * scale), (16, 32)
        row = {"points": N, "objects": B}
        idx, new_xyz = pu.furthest_point_sample_gather(xyz, M)
        t = ev_time(lambda: pu.furthest_point_sample_gather(xyz, M), 3)
        row["fps"] = {"us": 1e3 * t, "dist_updates_per_s": B * N * (M - 1) / (t * 1e-3),
                      "GBps_algorithmic": B * (12 * N + 16 * M) / (t * 1e-3) / 1e9}
        bq = pu.ball_query2(radii, ns, xyz, new_xyz)
        t = ev_time(lambda: pu.ball_query2(radii, ns, xyz, new_xyz), 5)
        row["ball_query_2radii"] = {"us": 1e3 * t, "GBps_algorithmic": B * (12 * N + 12 * M + 4 * M * (ns[0] + ns[1])) / (t * 1e-3) / 1e9}
        t = ev_time(lambda: pu.query_group(xyz, new_xyz, None, bq[1]), 5)
        row["query_group_C3"] = {"us": 1e3 * t, "GBps_algorithmic": B * (12 * N + 12 * M + 4 * M * ns[1] + 12 * M * ns[1]) / (t * 1e-3) / 1e9}
        feat = None
        if N <= 2048:
            feat = torch.randn(B, 96, N, device=dev)
            t = ev_time(lambda: pu.grouping_operation(feat, bq[1]), 3)
            row["group_C96"] = {"us": 1e3 * t, "GBps_algorithmic": B * (4 * 96 * N + 4 * M * ns[1] + 4 * 96 * M * ns[1]) / (t * 1e-3) / 1e9}
        if ext is not None:
            temp = torch.empty((B, N), dtype=torch.float32, device=dev)
            ridx = torch.empty((B, M), dtype=torch.int32, device=dev)

            def ref_fps():
                temp.fill_(1e10)
                ext.furthest_point_sampling_wrapper(B, N, M, xyz, temp, ridx)

            row["fps"]["reference_ext_us"] = 1e3 * ev_time(ref_fps, 2)
            row["fps"]["bit_exact"] = bool(torch.equal(ridx, idx))
            r0 = torch.zeros((B, M, ns[0]), dtype=torch.int32, device=dev)
            r1 = torch.zeros((B, M, ns[1]), dtype=torch.int32, device=dev)

            def ref_bq():
                ext.ball_query_wrapper(B, N, M, radii[0], ns[0], new_xyz, xyz, r0)
                ext.ball_query_wrapper(B, N, M, radii[1], ns[1], new_xyz, xyz, r1)

            row["ball_query_2radii"]["reference_ext_us"] = 1e3 * ev_time(ref_bq, 3)
            row["ball_query_2radii"]["bit_exact"] = bool(torch.equal(r0, bq[0]) and torch.equal(r1, bq[1]))
            xyz_t = xyz.transpose(1, 2).contiguous()
            gout = torch.empty((B, 3, M, ns[1]), dtype=torch.float32, device=dev)
            row["query_group_C3"]["reference_ext_group_only_us"] = 1e3 * ev_time(
                lambda: ext.group_points_wrapper(B, 3, N, M, ns[1], xyz_t, r1, gout), 3)
            if feat is not None:
                gout = torch.empty((B, 96, M, ns[1]), dtype=torch.float32, device=dev)
                row["group_C96"]["reference_ext_us"] = 1e3 * ev_time(
                    lambda: ext.group_points_wrapper(B, 96, N, M, ns[1], feat, r1, gout), 3)
        del feat
        rows.append(row)
        torch.cuda.empty_cache()
    return {"reference_ext_loaded": ext is not None, "sweep": rows}


def bench_c4(dev):
    """C4: tracking mode (evaluation_tracking.py:110-216): 32 objects per frame, T0 = 0.25, the aggregated pose of frame f
    fed back as init_x of frame f + 1, over a 100-frame synthetic sequence; clouds uploaded from pinned host memory
    every frame, the pose read back every frame."""
    import torch
    from genpose2_b200 import synthetic
    from genpose2_b200.pipeline import PosePipeline
    B, F, T = 32, 100, 0.25
    pipe = PosePipeline(device=str(dev), mlp_mode="fp32", use_graph=True).load_synthetic_weights((100, 200, 300))
    frames = []
    base, base_c = synthetic.make_point_clouds(B, NUM_POINTS, seed=900)
    gen = torch.Generator().manual_seed(901)
    drift = torch.zeros(B, 1, 3)
    for f in range(F):   # a smooth random walk of <= 1 cm per frame plus fresh 1 mm noise
        drift = drift + torch.randn(B, 1, 3, generator=gen) * 0.003
        p = (base + drift + torch.randn(base.shape, generator=gen) * 0.001).contiguous().pin_memory()
        frames.append((p, p.mean(dim=1).contiguous().pin_memory()))
    R0 = synthetic._random_rotations(__import__("numpy").random.default_rng(902), B)
    prev = torch.zeros(B, 9)
    prev[:, :3] = torch.from_numpy(R0[:, :, 0]).float()
    prev[:, 3:6] = torch.from_numpy(R0[:, :, 1]).float()
    prev[:, 6:] = frames[0][1]
    out_h = torch.empty((B, 4, 4), dtype=torch.float32).pin_memory()

    def run(n):
        pv = prev.to(dev)
        for f in range(n):
            p = frames[f][0].to(dev, non_blocking=True)
            c = frames[f][1].to(dev, non_blocking=True)
            init = pv.clone()
            init[:, 6:] -= c                                  # evaluation_tracking.py:117-118
            agg, length = pipe({"pts": p, "pts_center": c}, repeat_num=REPEAT, T0=T, init_x=init)
            pv = PosePipeline.next_init_x(agg)                # :210-214
            out_h.copy_(agg, non_blocking=True)
        return pv

    torch.manual_seed(7)
    run(5)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    run(F)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e)
    return {"workload": f"{B} objects/frame x {REPEAT} hypotheses, T0 = {T}, {F} frames, pose feedback, host clouds in / pose out per frame",
            "ms_per_frame": ms / F, "frames_per_s": F / (ms * 1e-3), "objects_per_s": B * F / (ms * 1e-3), "mlp_mode": "fp32",
            "cuda_graph": "one graph replay per frame (PosePipeline(use_graph=True))"}


def bench_reference_gpu(dev, c1_feat, c1_center):
    """The UNMODIFIED reference on this GPU (oracle/_ref/refpkg + its own CUDA ext): the C2 batch through
    pred_func -> get_energy -> aggregation -> pred_scale_func, per stage, and the C1 sampler (GPU and CPU)."""
    import torch
    from genpose2_b200 import synthetic
    from oracle import ref_shim
    if not (ref_shim.available() and ref_shim.has_cuda_ext()):
        return {"unavailable": "oracle/_ref/refpkg or oracle/_ref/pointnet2_cuda.so missing"}
    from oracle.ref_runner import ReferenceAgents
    tf32 = torch.backends.cudnn.allow_tf32
    out = {"what": "reference modules unmodified: torch fp32 nets on the GPU (cuDNN TF32 at its default: %s), scipy solve_ivp "
                   "on the host with a device round trip per RHS evaluation (samplers.py:204-234), sklearn DBSCAN per object" % tf32}
    ref = ReferenceAgents(*synthetic_weights(), device="cuda")
    pts, center = synthetic.make_point_clouds(OBJECTS_PER_GPU, NUM_POINTS, seed=0)
    runs = []
    for it in range(4):
        st = {}
        t0 = time.perf_counter()
        res = ref.full(pts, center, REPEAT, T0, noise_seed=1, stages=st)
        torch.cuda.synchronize()
        runs.append((time.perf_counter() - t0, st, res["nfev"]))
    dt, st, nfev = sorted(runs[1:], key=lambda r: r[0])[1]
    out["c2_full_path"] = {"objects": OBJECTS_PER_GPU, "ms_per_step": 1e3 * dt, "objects_per_s": OBJECTS_PER_GPU / dt,
                           "nfev": nfev, "stages_ms": {k: 1e3 * v for k, v in st.items()},
                           "sampling_objects_per_s": OBJECTS_PER_GPU / st["pred_func"],
                           "note": "median of 3 after 1 warm-up; pred_func = encoder + ODE sampling"}
    # C1: the reference's cond_ode_sampler alone, features injected, on the GPU and on the CPU
    for device in ("cuda", "cpu"):
        agents = ReferenceAgents(*synthetic_weights(), device=device, inject_features=True)
        net = agents.score_agent.net
        R = REPEAT
        rep = lambda a: a.unsqueeze(1).repeat(1, R, 1).view(R, -1)  # noqa: E731
        data = {"pts": torch.zeros(R, 4, 3, device=device), "pts_feat": rep(c1_feat).to(device), "pts_center": rep(c1_center).to(device)}
        ts = []
        for it in range(3):
            torch.manual_seed(1)
            if device == "cuda":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.no_grad():
                ref_ns = agents.ns
                ref_ns.samplers.cond_ode_sampler(score_model=net, data=dict(data), prior=net.prior_fn, sde_coeff=net.sde_fn,
                                                 atol=1e-5, rtol=1e-5, device=device, eps=net.sampling_eps, T=1.0,
                                                 num_steps=None, pose_mode="rot_matrix", denoise=True, init_x=None)
            if device == "cuda":
                torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        out["c1_sampler_%s_ms" % device] = 1e3 * sorted(ts)[1]
    out["cpu_threads"] = torch.get_num_threads()
    return out


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from genpose2_b200 import _lib, synthetic
    from genpose2_b200.pipeline import PosePipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (B200 arm) needs a GPU; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    B = args.objects
    # every rank owns its own contiguous slice of the global object list (weak scaling)
    pts_all, center_all = synthetic.make_point_clouds(B * world, NUM_POINTS, seed=0)
    pts_h = pts_all[rank * B:(rank + 1) * B].contiguous().pin_memory()
    center_h = center_all[rank * B:(rank + 1) * B].contiguous().pin_memory()
    pts_d, center_d = pts_h.to(dev), center_h.to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    out_pose_h = torch.empty((B, 4, 4), dtype=torch.float32).pin_memory()
    out_len_h = torch.empty((B, 3), dtype=torch.float32).pin_memory()
    peaks = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sampler=None):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        if sampler:
            sampler.start()
        for s, e in evs:
            flush.zero_()  # L2 flush between timed iterations (inputs are far smaller than the 126 MB L2)
            s.record()
            out = fn()
            e.record()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        barrier()
        per_step = [s.elapsed_time(e) for s, e in evs]
        total_ms = sum(per_step)
        if world > 1:
            t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        timed.last_spread = {"min": min(per_step), "median": sorted(per_step)[len(per_step) // 2], "max": max(per_step)}
        timed.last_out = out
        return total_ms, clocks

    def measure(mlp_mode, with_e2e, with_clocks):
        pipe = PosePipeline(device=f"cuda:{local_rank}", mlp_mode=mlp_mode, use_graph=args.graph == "on").load_synthetic_weights((100, 200, 300))
        graph_note = "off"
        if pipe.use_graph:
            try:
                torch.manual_seed(1)
                pipe({"pts": pts_d, "pts_center": center_d}, repeat_num=REPEAT, T0=T0)
                torch.cuda.synchronize()
                graph_note = "one CUDA graph per step (%d kernels of this library per replay)" % pipe.graph_launches
            except Exception as e:  # noqa: BLE001  (bench-level fallback: eager launches of the same kernels)
                print("CUDA graph capture failed, measuring eager launches:", repr(e)[:300], file=sys.stderr)
                pipe = PosePipeline(device=f"cuda:{local_rank}", mlp_mode=mlp_mode).load_synthetic_weights((100, 200, 300))
                graph_note = "capture failed: eager launches"

        def step_resident():
            return pipe({"pts": pts_d, "pts_center": center_d}, repeat_num=REPEAT, T0=T0)

        def step_e2e():
            # the call a user of the reference makes, with the reference-API defaults (pred_pose_q_wxyz included)
            p = pts_h.to(dev, non_blocking=True)
            c = center_h.to(dev, non_blocking=True)
            pose, length = pipe({"pts": p, "pts_center": c}, repeat_num=REPEAT, T0=T0)
            out_pose_h.copy_(pose, non_blocking=True)
            out_len_h.copy_(length, non_blocking=True)
            return pose, length

        torch.manual_seed(1234 + rank)
        sampler = ClockSampler(local_rank) if with_clocks else None   # helper process: up and sampling before the timed region
        for _ in range(max(args.warmup, 3)):
            step_resident()
        torch.cuda.synchronize()
        _lib.reset_launch_count()
        total_ms, clocks = timed(step_resident, args.steps, sampler)
        from genpose2_b200 import samplers as _s
        launches = pipe.graph_launches * args.steps if pipe.use_graph else _lib.launch_count()
        res = {"launches": launches, "graph": graph_note, "total_ms": total_ms, "clocks": clocks, "outputs": timed.last_out,
               "value": world * B * args.steps / (total_ms * 1e-3), "step_ms_spread": timed.last_spread,
               "last_step_ode": {k: v for k, v in _s.ode_stats().items() if k in ("nfev", "accepted", "rejected", "status")}}
        if with_e2e:
            for _ in range(2):
                step_e2e()
            e2e_ms, _ = timed(step_e2e, args.steps)
            res["e2e_ms"] = e2e_ms
            res["e2e_value"] = world * B * args.steps / (e2e_ms * 1e-3)

        # ---- roofline of the dominant kernel of this library: the fused ScoreNet / RK45 integrator ----
        score_net = pipe.score_agent.net
        feat = score_net(dict(pts=pts_d, pts_center=center_d), mode="pts_feature")
        sdata, noise = sampler_inputs(score_net, feat, center_d, B, T0)
        ntiles = (B * REPEAT + 127) // 128
        kname = ("ode_rk45_kernel<%s> (fused ScoreNet RHS + Dormand-Prince controller)"
                 % {"bf16": "TcEval<1>: tcgen05 bf16, 4-CTA cluster per tile" if ntiles <= 32 else "TcSolo<1>: tcgen05 bf16, one CTA per tile",
                    "fp32": "TcEval<3>: tcgen05 split-bf16 x3, 4-CTA cluster per tile" if ntiles <= 32 else "TcSolo<3>: tcgen05 split-bf16 x3, one CTA per tile",
                    "fp32_ffma": "SimtEval: FFMA fp32"}[mlp_mode])
        rf = sampler_roofline(score_net, sdata, noise, B, T0, peaks, mlp_mode, dev, flush, max(5, min(args.steps, 20)), kname)
        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel: weights and state are L2-resident, not HBM bound
        rf["traffic"] = NCU_DRAM_BYTES_PER_LAUNCH[mlp_mode] if B == OBJECTS_PER_GPU else None
        rf["traffic_source"] = NCU_DRAM_SOURCE
        res["roofline"] = rf
        return res

    main_res = measure(args.mlp_mode, True, True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *main_res["outputs"], rank)
    other_mode = "bf16" if args.mlp_mode != "bf16" else "fp32"
    other_res = measure(other_mode, False, False) if not args.single_mode else None
    value, total_ms, clocks, launches = main_res["value"], main_res["total_ms"], main_res["clocks"], main_res["launches"]
    e2e_value, e2e_ms, roofline = main_res["e2e_value"], main_res["e2e_ms"], main_res["roofline"]
    h2d = pts_h.numel() * 4 + center_h.numel() * 4
    d2h = out_pose_h.numel() * 4 + out_len_h.numel() * 4

    other_configs, reference_gpu = {}, None
    if not args.no_extras:
        try:
            other_configs["c5"] = bench_c5(args, world, rank, dev, peaks, barrier)
        except Exception as e:  # noqa: BLE001  (an extra must never lose the headline line)
            other_configs["c5"] = {"error": repr(e)}
        if world == 1:
            c1_feat = c1_center = None
            for name, fn in (("c1", lambda: bench_c1(dev, flush)), ("c3", lambda: bench_c3(dev)), ("c4", lambda: bench_c4(dev))):
                try:
                    r = fn()
                    if name == "c1":
                        r, c1_feat, c1_center = r
                    other_configs[name] = r
                except Exception as e:  # noqa: BLE001
                    other_configs[name] = {"error": repr(e)}
                torch.cuda.empty_cache()
            try:
                reference_gpu = bench_reference_gpu(dev, c1_feat, c1_center)
                if "c1_sampler_cpu_ms" in reference_gpu and "c1" in other_configs and "fp32" in other_configs["c1"]:
                    other_configs["c1"]["reference_cpu_ms"] = reference_gpu["c1_sampler_cpu_ms"]
                    other_configs["c1"]["reference_gpu_ms"] = reference_gpu["c1_sampler_cuda_ms"]
            except Exception as e:  # noqa: BLE001
                reference_gpu = {"error": repr(e)}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = args.cpu_sample_objects
        ref = CpuReference(n)
        ref.step(min(n, 2))  # warm-up
        reps = [ref.step(n) for _ in range(3)]
        med, enc, _ = sorted(reps, key=lambda r: r[0])[1]
        cpu_baseline = {"value": n / med, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
                        "sample": ref.describe(n, 3, None if enc is None else enc / med) + ", median",
                        "os_cpu_count": os.cpu_count()}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.mlp_mode == "bf16" else ("f32 (split-bf16 x3 tensor-core products, fp32 accumulation)" if args.mlp_mode == "fp32" else "f32"), "data": "synthetic",
            "config": {"workload": f"C2: {B} objects x {REPEAT} hypotheses per GPU, full path "
                                   f"(encoder x2 + RK45 ScoreNet sampling + EnergyNet + aggregation + ScaleNet), "
                                   f"T0={T0}, rtol=atol=1e-5, {NUM_POINTS} pts/object, random-init weights",
                       "objects_per_gpu": B, "hypotheses": REPEAT, "T0": T0, "l2": "flushed between timed steps "
                       f"({L2_FLUSH_BYTES >> 20} MiB memset)", "parallelism": f"object-sharded x{world}, no collective on the data path",
                       "streams": "the energy encoder runs on a second stream beside the cooperative sampler launch",
                       "cuda_graph": main_res["graph"]},
            "clocks": clocks, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                      "ms_per_step": e2e_ms / args.steps,
                                      "api": "PosePipeline -> PoseNet.pred_func (reference defaults, pred_pose_q_wxyz computed) -> "
                                             "get_energy -> aggregate_pose -> pred_scale_func"},
            "gpu_launches": launches, "step_ms_spread": main_res["step_ms_spread"], "last_step_ode": main_res["last_step_ode"],
            "roofline": roofline, "cpu_baseline": cpu_baseline,
        }
        if other_res is not None:
            line["other_mode"] = {"mlp_mode": other_mode, "value": other_res["value"], "unit": UNIT,
                                  "ms_per_step": other_res["total_ms"] / args.steps, "step_ms_spread": other_res["step_ms_spread"],
                                  "last_step_ode": other_res["last_step_ode"], "roofline": other_res["roofline"]}
        if other_configs:
            line["other_configs"] = other_configs
        if reference_gpu is not None:
            line["reference_gpu"] = reference_gpu
            try:
                line["reference_gpu"]["speedup_e2e_vs_reference_gpu_full_path"] = e2e_value / reference_gpu["c2_full_path"]["objects_per_s"]
            except Exception:  # noqa: BLE001
                pass
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

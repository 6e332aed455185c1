"""The per-object pose-generation path end to end, in the order the reference runners execute it
(runners/evaluation_single.py:404-420, runners/evaluation_tracking.py:110-216):

    score_agent.pred_func  ->  energy_agent.get_energy(T=1e-5)  ->  aggregate_pose  ->  scale_agent.pred_scale_func

plus the object sharding used for multi-GPU runs: objects are split into contiguous ranges, one
process per GPU, no collective inside the path, one gather of [B,4,4] + [B,3] at the end
(SURVEY.md section 8(e)).
"""
import copy

import torch
import torch.distributed as dist

from . import _lib, synthetic
from .aggregation import aggregate_pose
from .config import get_config
from .posenet_agent import PoseNet
from .rotation import matrix_to_rotation_6d_cols


def shard_range(num_objects, rank, world_size):
    """Contiguous object range [lo, hi) of `rank` (SURVEY.md 8(e)): the first `num_objects %
    world_size` ranks get one extra object."""
    base, rem = divmod(num_objects, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_results(pose, length, group=None):
    """All ranks contribute their [b_local,4,4] / [b_local,3] shard; rank 0 gets the concatenation
    (ragged shards allowed).  Works with NCCL (device tensors) and gloo (CPU tensors)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return pose, length
    world = dist.get_world_size(group)
    flat = torch.cat([pose.reshape(pose.shape[0], 16), length.reshape(length.shape[0], 3)], dim=1).contiguous()
    counts = [torch.zeros(1, dtype=torch.int64, device=flat.device) for _ in range(world)]
    dist.all_gather(counts, torch.tensor([flat.shape[0]], dtype=torch.int64, device=flat.device), group=group)
    counts = [int(c.item()) for c in counts]
    mx = max(counts)
    padded = torch.zeros((mx, 19), dtype=flat.dtype, device=flat.device)
    padded[: flat.shape[0]] = flat
    bufs = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(bufs, padded, group=group)
    full = torch.cat([b[:c] for b, c in zip(bufs, counts)], dim=0)
    return full[:, :16].reshape(-1, 4, 4), full[:, 16:]


class PosePipeline:
    """score + energy + scale agents wired together; every stage runs on libgenpose_b200.so."""

    def __init__(self, cfg=None, device="cuda", mlp_mode="fp32", use_graph=False, step_control="batch", encoder_mode="auto"):
        """use_graph: replay the whole step as ONE CUDA graph per input signature (batch size, points, hypotheses, T0 --
        or "per-object T0", whatever the values --, warm start and noise keys present or not):
        ~80 kernel launches, the two-stream fork / join and the cooperative sampler launch become one graph launch; the
        only host work left per step is drawing the prior noise with the CPU generator (exactly like the reference,
        sde.py:34) and one pinned upload.  The captured graph bakes in the packed weights: load_state_dicts() drops it.
        step_control: "batch" (the reference's RK45 controller over the whole batch) or "object" (every object integrated
        as if it were alone: its poses do not depend on the other objects of the step), see samplers.STEP_CONTROLS.
        encoder_mode: operand precision of both point-cloud encoders' SharedMLP GEMMs, "auto" (follows mlp_mode),
        "bf16x3", "tf32" or "bf16", see posenet.ENCODER_MODES."""
        from .samplers import check_step_control
        check_step_control(step_control)
        cfg = copy.copy(cfg) if cfg is not None else get_config()
        cfg.device = device
        cfg.mlp_mode = mlp_mode
        cfg.step_control = step_control
        cfg.encoder_mode = encoder_mode
        if not getattr(cfg, "sampler_mode", None):
            cfg.sampler_mode = ["ode"]
        self.cfg = cfg
        c = copy.copy(cfg); c.agent_type = "score"
        self.score_agent = PoseNet(c)
        c = copy.copy(cfg); c.agent_type = "energy"
        self.energy_agent = PoseNet(c)
        c = copy.copy(cfg); c.agent_type = "scale"
        self.scale_agent = PoseNet(c)
        self._side = None   # second stream: the energy encoder overlaps the sampler
        self.use_graph = bool(use_graph)
        self._graphs = {}
        self.graph_launches = 0

    def load_state_dicts(self, score_sd, energy_sd, scale_sd):
        self.score_agent.net.load_state_dict(score_sd)
        self.energy_agent.net.load_state_dict(energy_sd)
        self.scale_agent.net.load_state_dict(scale_sd)
        self._graphs.clear()
        return self

    def load_synthetic_weights(self, seeds=(100, 200, 300)):
        return self.load_state_dicts(synthetic.random_gfobjectpose_state_dict(seeds[0]),
                                     synthetic.random_gfobjectpose_state_dict(seeds[1]),
                                     synthetic.random_scalenet_state_dict(seeds[2]))

    ENCODER_CHUNK = 1024   # objects per encoder pass (bounds the level buffers; objects are independent)

    def _encode(self, agent, pts, geometries=None, keep_geometry=False):
        """Encoder features of all objects, at most ENCODER_CHUNK objects per pass (bit-identical to one pass: every
        encoder kernel works per object).  Returns (features [B,1024], per-chunk geometry list or None)."""
        B = pts.shape[0]
        feats, geos = [], []
        for k, lo in enumerate(range(0, B, self.ENCODER_CHUNK)):
            chunk = {"pts": pts[lo:lo + self.ENCODER_CHUNK]}
            if geometries is not None:
                f = agent.net(chunk, mode="pts_feature", geometry=geometries[k])
            elif keep_geometry:
                f, g = agent.net(chunk, mode="pts_feature", return_geometry=True)
                geos.append(g)
            else:
                f = agent.net(chunk, mode="pts_feature")
            feats.append(f)
        return (feats[0] if len(feats) == 1 else torch.cat(feats, dim=0)), (geos if keep_geometry else None)

    @torch.no_grad()
    def __call__(self, data, repeat_num=None, T0=None, init_x=None, return_all=False, *, noise_keys=None):
        """data{'pts' [B,N,3] f32 cuda, 'pts_center' [B,3]} -> (aggregated_pose [B,4,4] f32, length [B,3] f32).

        T0: one start time for the step, or one per object (1-D host values; step_control="object" only), so that a
        tracking frame of new objects (T0 = 0.55, no warm start) and tracked ones (T0 = 0.25 with their previous pose)
        is one call.  init_x [B,9]: warm start added to the prior noise; a zero row means "no warm start" for that
        object (0 + noise == noise).  noise_keys: int64 [B] (CPU or device), object b's prior noise drawn by
        gp_object_noise from noise_keys[b] instead of the global CPU generator.  With step_control="object" and keys,
        an object's aggregated pose and length depend only on its cloud, its key, its T0 and its warm start (for
        results computed on the same evaluator shape, DESIGN.md section 6)."""
        from . import samplers
        cfg = self.cfg
        R = cfg.eval_repeat_num if repeat_num is None else repeat_num
        T0 = cfg.T0 if T0 is None else T0
        B = data["pts"].shape[0]
        T_obj = samplers.object_start_times(T0, B, cfg.step_control, self.score_agent.sampling_eps)
        noise_keys = samplers.check_noise_keys(noise_keys, B)
        if T_obj is not None:
            T0 = T_obj
        if self.use_graph and not return_all:
            return self._graph_step(data, R, float(T0) if T_obj is None else T0, init_x, noise_keys)
        return self._step(data, R, T0, init_x, return_all, noise_keys)

    def _graph_key(self, pts, R, T0, init_x, noise_keys=None):
        """One captured graph per input signature and sampler step control.  Per-object start times and noise keys
        live in static buffers refilled before every replay: the key records that they are used, not their values."""
        per_object = isinstance(T0, (list, tuple)) or getattr(T0, "ndim", 0) > 0
        return (pts.shape[0], pts.shape[1], R, "per-object" if per_object else T0, init_x is not None,
                pts.device.index, noise_keys is not None, self.score_agent.cfg.step_control)

    def _fill_object_inputs(self, st, T0, noise_keys, B):
        """Per-object start times, grids, sigmas and keys -> the graph's static buffers (pinned staging, asynchronous
        uploads).  Returns the host sigmas."""
        from . import samplers
        T_obj = T0 if "T" in st else None
        sig = samplers.object_sigmas(T_obj, T0, B)
        uploads = [("sigma", sig)]
        if T_obj is not None:
            uploads.append(("T", torch.from_numpy(T_obj)))
            if "t_eval" in st:
                grids = samplers.object_grids(T_obj, self.score_agent.sampling_eps, st["t_eval"].shape[1])
                uploads.append(("t_eval", torch.from_numpy(grids)))
        if noise_keys is not None:
            if noise_keys.is_cuda:
                st["keys"].copy_(noise_keys, non_blocking=True)
            else:
                uploads.append(("keys", noise_keys))
        for name, host in uploads:
            st[name + "_host"].copy_(host)
            st[name].copy_(st[name + "_host"], non_blocking=True)
        return sig

    def _graph_step(self, data, R, T0, init_x, noise_keys=None):
        """The step as a CUDA graph: copy the inputs into the graph's static buffers, draw + upload the prior noise
        (or, with noise_keys, upload the keys: the noise is generated inside the graph), replay.  Returns clones of the
        two small results (the static ones are overwritten by the next replay)."""
        from . import samplers
        pts, center = data["pts"], data["pts_center"]
        B, N = pts.shape[0], pts.shape[1]
        key = self._graph_key(pts, R, T0, init_x, noise_keys)
        per_object, keyed = key[3] == "per-object", noise_keys is not None
        ent = self._graphs.get(key)
        net = self.score_agent.net
        real_prior = net.prior_fn
        if ent is None:
            dev = pts.device
            st = dict(pts=torch.empty_like(pts), center=torch.empty_like(center, dtype=torch.float32),
                      init=None if init_x is None else torch.empty_like(init_x),
                      noise=torch.empty((B * R, 9), dtype=torch.float32, device=dev),
                      noise_host=torch.empty((B * R, 9), dtype=torch.float32, pin_memory=True))
            if per_object or keyed:
                bufs = {"sigma": ((B,), torch.float32)}
                if per_object:
                    bufs["T"] = ((B,), torch.float64)
                    if self.cfg.sampling_steps is not None:
                        bufs["t_eval"] = ((B, int(self.cfg.sampling_steps)), torch.float64)
                if keyed:
                    bufs["keys"] = ((B,), torch.int64)
                for name, (shape, dtype) in bufs.items():
                    st[name] = torch.empty(shape, dtype=dtype, device=dev)
                    st[name + "_host"] = torch.empty(shape, dtype=dtype, pin_memory=True)
                self._fill_object_inputs(st, T0, noise_keys, B)   # no draw: the global generator is not touched
            st["pts"].copy_(pts); st["center"].copy_(center)
            if init_x is not None:
                st["init"].copy_(init_x)
            # warm-up / capture noise from a private generator: building the graph must not consume the global CPU
            # generator (the first graphed step has to see the same draw as an eager step would)
            st["noise"].copy_(torch.randn((B * R, 9), generator=torch.Generator().manual_seed(0)))
            sdata = {"pts": st["pts"], "pts_center": st["center"]}
            net.prior_fn = lambda shape, T=1.0: st["noise"]    # device tensor: no host work inside the capture
            if per_object or keyed:   # the sampler takes T, sigma, keys and the noise from the static buffers
                net.static_object_inputs = {k: st.get(k) for k in ("noise", "sigma", "T", "t_eval", "keys")}
            try:
                warm = torch.cuda.Stream(device=dev)
                warm.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(warm):
                    for _ in range(2):   # packs weights, sets kernel attributes, sizes the allocator pools
                        self._step(sdata, R, T0, st["init"], False, st.get("keys"))
                torch.cuda.current_stream(dev).wait_stream(warm)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                n0 = _lib.launch_count()
                with torch.cuda.graph(graph):
                    out = self._step(sdata, R, T0, st["init"], False, st.get("keys"))
                self.graph_launches = _lib.launch_count() - n0   # kernels of this library inside one replay
                stats = {k: v for k, v in samplers.last_ode_stats.items() if k in ("device_stats", "device_obj_stats")}
            finally:
                net.prior_fn = real_prior
                net.static_object_inputs = None
            ent = self._graphs[key] = (graph, st, out, stats)
        graph, st, out, stats = ent
        if pts.data_ptr() != st["pts"].data_ptr():
            st["pts"].copy_(pts, non_blocking=True)
        st["center"].copy_(center, non_blocking=True)
        if init_x is not None:
            st["init"].copy_(init_x, non_blocking=True)
        ev = st.get("noise_event")
        if ev is not None:
            ev.synchronize()     # the previous uploads out of the pinned buffers (long finished in practice)
        sig = self._fill_object_inputs(st, T0, noise_keys, B) if (per_object or keyed) else None
        if not keyed:
            # prior noise: drawn on the CPU from the global generator in the reference's call order (samplers.py:197-201)
            st["noise_host"].copy_(real_prior((B * R, 9), T=T0) if not per_object
                                   else samplers.object_prior_noise(sig, R))
            st["noise"].copy_(st["noise_host"], non_blocking=True)
        st["noise_event"] = torch.cuda.Event()
        st["noise_event"].record()
        graph.replay()
        if stats:
            samplers.last_ode_stats.clear()
            samplers.last_ode_stats.update(stats)
        return out[0].clone(), out[1].clone()

    def _step(self, data, R, T0, init_x, return_all, noise_keys=None):
        cfg = self.cfg
        capturing = torch.cuda.is_current_stream_capturing()
        # The sampler of a small batch is a cooperative launch of at most 33 four-CTA clusters (100 SMs at 64 x 50): the
        # energy encoder, which only needs the cloud and the shared FPS / ball-query geometry, runs beside it on a second
        # stream and fills the remaining SMs.  The sampler is enqueued first so that it gets its SMs first.
        main = torch.cuda.current_stream()
        score_feat, geometry = self._encode(self.score_agent, data["pts"], keep_geometry=True)
        fork = torch.cuda.Event()
        fork.record(main)
        pred_pose, pred_q = self.score_agent.pred_func(
            data=data, repeat_num=R, T0=T0, init_x=init_x, save_path=None, pts_feat=score_feat, noise_keys=noise_keys)
        if self._side is None:
            self._side = torch.cuda.Stream(device=score_feat.device)
        self._side.wait_event(fork)
        with torch.cuda.stream(self._side):
            energy_feat, _ = self._encode(self.energy_agent, data["pts"], geometries=geometry)
            # everything of the energy evaluation that does not need the sampled poses, still beside the sampler
            energy_pre = self.energy_agent.energy_prepare(energy_feat, data["pts_center"], R, 1e-5)
            if not capturing:
                for t in (energy_feat,) + tuple(energy_pre):
                    t.record_stream(main)
        main.wait_stream(self._side)
        energy = self.energy_agent.get_energy(data={"pts_feat": energy_feat, "pts_center": data["pts_center"],
                                                    "_gp_energy_pre": energy_pre},
                                              pose_samples=pred_pose, T=1e-5, mode="test", extract_feature=False)
        agg = aggregate_pose(pred_pose, energy, eval_repeat_num=R, retain_ratio=cfg.retain_ratio,
                             clustering=cfg.clustering, clustering_eps=cfg.clustering_eps,
                             clustering_minpts=cfg.clustering_minpts)
        _, length = self.scale_agent.pred_scale_func({"pts_feat": score_feat, "rgb_feat": None,
                                                      "axes": agg[:, :3, :3]})
        if return_all:
            return dict(pred_pose=pred_pose, pred_pose_q_wxyz=pred_q, energy=energy, aggregated_pose=agg,
                        length=length, pts_feat=score_feat)
        return agg, length

    @staticmethod
    def next_init_x(aggregated_pose):
        """Tracking feedback (evaluation_tracking.py:210-214): aggregated pose re-encoded as 6D + t."""
        return torch.cat([matrix_to_rotation_6d_cols(aggregated_pose[:, :3, :3]), aggregated_pose[:, :3, 3]], dim=-1)

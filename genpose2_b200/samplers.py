"""Drop-ins for `cond_ode_sampler` and `cond_pc_sampler`
(networks/gf_algorithms/samplers.py:180-258, 113-177): same signatures, same returned shapes and
dtypes (the ODE sampler returns float64 like scipy's state), same consumption of the global CPU
generator for the initial noise (`prior` is called exactly as the reference calls it).

What changes: the scipy `solve_ivp` host loop with a host<->device round trip per RHS evaluation
(samplers.py:204-234) is one persistent device kernel (gp_scorenet_ode); the 500-step PC loop is
one persistent kernel (gp_scorenet_pc).
"""
import threading

import numpy as np
import torch

from . import _lib
from .scorenet import _object_features
from .sde import prior_std

POSE_DIM = 9  # get_pose_dim("rot_matrix"), utils/genpose_utils.py:34-35
MAX_TRAJ = 512  # accepted-step slots recorded when the trajectory is requested (upper bound)
TRAJ_BYTES_BUDGET = 2 << 30   # the recording buffer [slots, N, 9] f64 is capped at this size (never below 64 slots)


def _traj_slots(batch_size):
    """Slots of the trajectory buffer: MAX_TRAJ for small batches, fewer when [slots, N, 9] f64 would exceed
    TRAJ_BYTES_BUDGET (the evaluation settings accept 9 - 62 steps; a longer trajectory raises)."""
    per_slot = max(1, batch_size) * POSE_DIM * 8
    return int(max(64, min(MAX_TRAJ, TRAJ_BYTES_BUDGET // per_slot)))

last_ode_stats = {}  # statistics of the most recent cond_ode_sampler call (nfev, accepted, ...)

# RK45 step-size control of cond_ode_sampler (not in the reference):
#   "batch"  one step size and one RMS error norm over the whole flattened batch, as scipy's solve_ivp on the
#            reference's [N*9] state does (the default);
#   "object" every object integrated as if the sampler had been called with that object alone, so that its poses
#            depend only on its own features, noise and the weights (gp_scorenet_ode_objects).
STEP_CONTROLS = ("batch", "object")
MAX_ROWS_PER_OBJECT = 128   # "object": an object's hypotheses must fit one 128-row tile of the integrator


def check_step_control(step_control, sampler="ode", rows_per_object=1, num_steps=None, return_trajectory=False):
    """Raises for an unknown mode and for what "object" does not support, before any device work."""
    if step_control not in STEP_CONTROLS:
        raise ValueError(f"step_control must be one of {STEP_CONTROLS}, got {step_control!r}")
    if step_control == "batch":
        return
    if sampler == "pc":
        raise NotImplementedError("step_control='object' is implemented for the ODE sampler only")
    if rows_per_object > MAX_ROWS_PER_OBJECT:
        raise NotImplementedError(f"step_control='object' supports up to {MAX_ROWS_PER_OBJECT} hypotheses per object, "
                                  f"got {rows_per_object}")
    if return_trajectory and num_steps is None:
        raise NotImplementedError("step_control='object' records no trajectory of accepted steps (objects accept "
                                  "different numbers of steps): pass num_steps for dense output on a common grid, or "
                                  "return_trajectory=False")


def object_start_times(T, num_objects, step_control, eps):
    """Per-object start times of the ODE sampler.  A scalar T (a number, or a 0-d array / tensor) -> None: one start
    time for the call, as before.  A 1-D host sequence, ndarray or CPU tensor of `num_objects` values -> float64
    ndarray [B] (a float32 tensor's values are read as they are stored).  Raises, before any sampler work, for:
    a CUDA tensor (reading it would hide a device synchronisation), step_control other than "object" (the batch
    controller has one t for the whole batch), the wrong length, and a value that is not finite or not > eps."""
    if isinstance(T, torch.Tensor):
        if T.dim() == 0:
            return None
        if T.is_cuda:
            raise TypeError("a per-object T must be a host sequence, ndarray or CPU tensor: reading a CUDA tensor "
                            "would synchronise the device")
        vals = T.detach().to(torch.float64).numpy()
    elif isinstance(T, np.ndarray):
        if T.ndim == 0:
            return None
        vals = T.astype(np.float64)
    elif isinstance(T, (list, tuple)):
        vals = np.asarray(T, dtype=np.float64)
    else:
        return None
    if vals.ndim != 1:
        raise ValueError(f"a per-object T must be 1-D, got shape {tuple(vals.shape)}")
    if step_control != "object":
        raise NotImplementedError("a per-object T needs step_control='object' (the batch controller integrates the "
                                  "whole batch from one start time)")
    if vals.shape[0] != num_objects:
        raise ValueError(f"a per-object T needs one value per object: {num_objects} objects, got {vals.shape[0]} values")
    if not np.isfinite(vals).all() or (vals <= eps).any():
        raise ValueError(f"every per-object T must be finite and > eps={eps}, got {vals.tolist()}")
    return np.ascontiguousarray(vals)


def check_noise_keys(noise_keys, num_objects):
    """noise_keys: int64 [B] (CPU or CUDA tensor, or ndarray) -> tensor; None -> None.  Raises for another dtype or
    shape."""
    if noise_keys is None:
        return None
    if isinstance(noise_keys, np.ndarray):
        noise_keys = torch.from_numpy(noise_keys)
    if not isinstance(noise_keys, torch.Tensor):
        raise TypeError(f"noise_keys must be an int64 tensor of shape [{num_objects}], got {type(noise_keys).__name__}")
    if noise_keys.dtype != torch.int64:
        raise TypeError(f"noise_keys must be int64, got {noise_keys.dtype}")
    if tuple(noise_keys.shape) != (num_objects,):
        raise ValueError(f"noise_keys must have shape [{num_objects}] (one key per object), got {tuple(noise_keys.shape)}")
    return noise_keys


def object_sigmas(T_obj, T, num_objects):
    """float32 [B] standard deviation of each object's prior noise: float32(sigma(T_b)), sigma as ve_marginal_prob
    computes it (the factor ve_prior applies to its float32 normals)."""
    times = T_obj if T_obj is not None else [float(T)] * num_objects
    return torch.tensor([prior_std(float(t)) for t in times], dtype=torch.float32)


def object_prior_noise(sigmas, rows_per_object):
    """Unkeyed per-object prior: the draw ve_prior makes (torch.randn((N, 9)) from the global CPU generator), with the
    rows of object b scaled by sigmas[b] in float32.  A vector of equal sigmas gives ve_prior's result bit for bit."""
    z = torch.randn((sigmas.shape[0] * rows_per_object, POSE_DIM))
    return z * sigmas.repeat_interleave(rows_per_object).unsqueeze(1)


def object_grids(T_obj, eps, num_steps):
    """Dense-output grids of per-object start times: float64 [B, num_steps], row b = linspace(T_obj[b], eps)."""
    return np.stack([np.linspace(t, eps, int(num_steps)) for t in T_obj])


def keyed_noise(keys, sigmas, rows_per_object, out=None):
    """gp_object_noise: [B*R, 9] float32 noise on the keys' device, object b's block a function of keys[b] and
    sigmas[b] only (both device tensors)."""
    B = keys.shape[0]
    keys = _lib.check_cuda(keys.contiguous(), "noise_keys", torch.int64)
    sigmas = _lib.check_cuda(sigmas.contiguous(), "sigmas", torch.float32)
    if out is None:
        out = torch.empty((B * rows_per_object, POSE_DIM), dtype=torch.float32, device=keys.device)
    _lib.call("gp_object_noise", _lib.ptr(keys), _lib.ptr(sigmas), B, rows_per_object, _lib.ptr(out), device=out.device)
    return out


# Failure of the device integrator (status -1: step size underflow, -2: attempt cap) must not pass silently, and
# checking it must not stall the stream: every call copies its statistics to pinned host memory asynchronously; the
# copies that have landed are inspected at the next sampler call / ode_stats() and a failed integration raises there.
# (In band, the kernel also turns x_out of a failed integration into NaN.)
_pending_stats = []


def _watch(stats):
    if torch.cuda.is_current_stream_capturing():
        return   # no host allocations / events inside a graph capture; the graph's owner watches the static stats
    host = torch.empty(stats.shape, dtype=stats.dtype, pin_memory=True)
    host.copy_(stats, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(stats.device))
    _pending_stats.append((ev, host))
    if len(_pending_stats) > 64:
        _pending_stats.pop(0)[0].synchronize()


def check_pending(wait=False):
    """Raise if an earlier device integration failed (only looks at statistics that have already reached the host
    unless wait=True)."""
    if torch.cuda.is_current_stream_capturing():
        return
    while _pending_stats and (wait or _pending_stats[0][0].query()):
        ev, host = _pending_stats.pop(0)
        ev.synchronize()
        status = int(host[_lib.STAT_STATUS])
        if status != 0:
            raise RuntimeError(f"device RK45 integration failed with status {status} "
                               "(-1: step size underflow, -2: attempt cap); its poses are NaN")


def _score_net(score_model):
    net = getattr(score_model, "pose_score_net", score_model)
    if not hasattr(net, "packed"):
        raise TypeError("score_model must be a genpose2_b200 GFObjectPose / PoseScoreNet (no fallback path)")
    if hasattr(net, "mode_arg"):
        net.mode_arg()   # an unsupported mlp_mode / eval_shape pair raises before the prior draw
    return net


def _mlp_mode(score_model):
    return _score_net(score_model).mode_arg()


_staging = {}
_staging_lock = threading.Lock()


def _to_device_async(t, device):
    """Host tensor -> device without blocking the host: a pageable copy is synchronous AND ordered behind everything
    already enqueued on the stream, so the prior draw (made on the CPU with the CPU generator, like the reference)
    would stall the host until the encoder has finished.  Staged through a cached pinned buffer instead."""
    if t.is_cuda:
        return t.to(device)
    # one staging buffer per (device, host thread, shape, dtype): two threads / devices never share one, so a buffer
    # is only reused after the event of ITS previous copy; the cache is bounded (least recently created entry goes)
    key = (str(device), threading.get_ident(), tuple(t.shape), t.dtype)
    with _staging_lock:
        ent = _staging.get(key)
        if ent is None:
            if len(_staging) >= 16:
                _staging.pop(next(iter(_staging)))
            ent = _staging[key] = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True), None]
    buf, ev = ent
    if ev is not None:
        ev.synchronize()   # the previous copy out of this buffer (long finished in practice)
    buf.copy_(t)
    out = buf.to(device, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(out.device))
    ent[1] = ev
    return out


def cond_ode_sampler(score_model, data, prior, sde_coeff, atol=1e-5, rtol=1e-5, device="cuda", eps=1e-5,
                     T=1.0, num_steps=None, pose_mode="quat_wxyz", denoise=True, init_x=None,
                     return_trajectory=True, *, step_control="batch", noise_keys=None):
    """-> (xs [N, S, 9] f64, x [N, 9] f64).  num_steps=None: xs holds every accepted step (scipy's res.y);
    num_steps=n: scipy's dense output on t_eval = linspace(T, eps, n) (samplers.py:222-235).
    `return_trajectory=False` (not in the reference) skips recording and returns xs = x[:, None].
    `step_control` (not in the reference): "batch" or "object", see STEP_CONTROLS.  "object" needs
    num_steps or return_trajectory=False, and at most MAX_ROWS_PER_OBJECT rows per object.
    Not in the reference either:
      T           may be one start time per object (1-D host values, B = N / R; step_control="object" only, see
                  object_start_times): object b is integrated from T[b], its prior noise is scaled by sigma(T[b]) and
                  its dense grid is linspace(T[b], eps, num_steps).  Without keys the noise is object_prior_noise
                  (the `prior` callable is not used).
      noise_keys  int64 [B] (CPU or device): the prior draw is replaced by gp_object_noise, so that object b's noise
                  depends on noise_keys[b] and its T only; the global CPU generator is not touched."""
    if pose_mode != "rot_matrix":
        raise NotImplementedError("accelerated sampler supports pose_mode='rot_matrix' only")
    net = _score_net(score_model)
    batch_size = data["pts"].shape[0]
    feat, rpo = _object_features(data, batch_size)
    check_step_control(step_control, "ode", rpo, num_steps, return_trajectory)
    B = batch_size // rpo
    T_obj = object_start_times(T, B, step_control, eps)
    keys = check_noise_keys(noise_keys, B)
    check_pending()
    # PosePipeline's graph capture hands in device buffers it refills before every replay
    static = getattr(score_model, "static_object_inputs", None)
    if keys is None and T_obj is None:
        noise = _to_device_async(prior((batch_size, POSE_DIM), T=T), device)  # CPU generator, like samplers.py:197-201
    elif static is not None:
        noise = static["noise"]
        if keys is not None:
            keyed_noise(static["keys"], static["sigma"], rpo, out=noise)
    else:
        sig = object_sigmas(T_obj, T, B)
        if keys is not None:
            kdev = keys.to(device) if keys.is_cuda else _to_device_async(keys, device)
            noise = keyed_noise(kdev, _to_device_async(sig, kdev.device), rpo)
        else:
            noise = _to_device_async(object_prior_noise(sig, rpo), device)
    x0 = noise if init_x is None else init_x + noise
    dev = x0.device
    x0 = x0.to(torch.float64).contiguous()  # scipy casts y0 to float64
    proj = net.project(feat.to(dev))
    center = _lib.check_cuda(data["pts_center"].to(torch.float32).contiguous(), "pts_center", torch.float32)
    if T_obj is not None:
        if static is not None:
            T_dev, grids = static["T"], static.get("t_eval")
        else:
            T_dev = _to_device_async(torch.from_numpy(T_obj), dev)
            grids = None if num_steps is None else _to_device_async(torch.from_numpy(object_grids(T_obj, eps, num_steps)), dev)
        return _ode_objects(net, score_model, proj, x0, center, batch_size, rpo, T, eps, rtol, atol, denoise, num_steps,
                            T_obj=T_dev, t_eval=grids)
    if step_control == "object":
        return _ode_objects(net, score_model, proj, x0, center, batch_size, rpo, T, eps, rtol, atol, denoise, num_steps)

    x_out = torch.empty((batch_size, POSE_DIM), dtype=torch.float64, device=dev)
    stats = torch.zeros(_lib.GP_STAT_COUNT, dtype=torch.float64, device=dev)
    ws_bytes = _lib.load().gp_scorenet_ode_workspace_bytes(batch_size)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    if num_steps is not None:
        import numpy as np
        t_eval = torch.from_numpy(np.linspace(T, eps, int(num_steps))).to(dev)   # float64, as solve_ivp receives it
        dense = torch.empty((int(num_steps), batch_size, POSE_DIM), dtype=torch.float64, device=dev)
        _lib.call("gp_scorenet_ode_dense", _lib.ptr(net.packed()), _lib.ptr(proj), _lib.ptr(x0), _lib.ptr(center),
                  batch_size, rpo, float(T), float(eps), float(rtol), float(atol), 1 if denoise else 0,
                  _lib.ptr(x_out), _lib.ptr(t_eval), int(num_steps), _lib.ptr(dense), _lib.ptr(stats),
                  _lib.ptr(ws), ws_bytes, _mlp_mode(score_model), device=dev)
        xs = torch.empty((batch_size, int(num_steps), POSE_DIM), dtype=torch.float64, device=dev)
        _lib.call("gp_traj_finalize", _lib.ptr(dense), _lib.ptr(center), int(num_steps), batch_size, _lib.ptr(xs), device=dev)
        last_ode_stats.clear()
        last_ode_stats["device_stats"] = stats
        _watch(stats)
        return xs, x_out
    traj = None
    slots = _traj_slots(batch_size)
    if return_trajectory:
        traj = torch.empty((slots, batch_size, POSE_DIM), dtype=torch.float64, device=dev)
    _lib.call("gp_scorenet_ode", _lib.ptr(net.packed()), _lib.ptr(proj), _lib.ptr(x0), _lib.ptr(center),
              batch_size, rpo, float(T), float(eps), float(rtol), float(atol), 1 if denoise else 0,
              _lib.ptr(x_out), _lib.ptr(traj), slots if traj is not None else 0, _lib.ptr(stats),
              _lib.ptr(ws), ws_bytes, _mlp_mode(score_model), device=dev)
    if return_trajectory:
        st = stats.cpu()
        S = int(st[_lib.STAT_ACCEPTED].item()) + 1
        if S > slots:
            raise RuntimeError(f"trajectory of {S} accepted steps does not fit the {slots} recorded slots "
                               "(raise samplers.TRAJ_BYTES_BUDGET, or pass return_trajectory=False)")
        xs = torch.empty((batch_size, S, POSE_DIM), dtype=torch.float64, device=dev)
        _lib.call("gp_traj_finalize", _lib.ptr(traj), _lib.ptr(center), S, batch_size, _lib.ptr(xs), device=dev)
        _record_stats(st)
    else:
        xs = x_out.unsqueeze(1)
        last_ode_stats.clear()
        last_ode_stats["device_stats"] = stats
        _watch(stats)
    return xs, x_out


def _ode_objects(net, score_model, proj, x0, center, batch_size, rpo, T, eps, rtol, atol, denoise, num_steps,
                 T_obj=None, t_eval=None):
    """step_control="object": gp_scorenet_ode_objects / gp_scorenet_ode_dense_objects; with per-object start times
    (T_obj [B] f64 device, t_eval [B, num_steps] f64 device or None) gp_scorenet_ode_objects_t0."""
    dev = x0.device
    B = batch_size // rpo
    x_out = torch.empty((batch_size, POSE_DIM), dtype=torch.float64, device=dev)
    stats = torch.zeros(_lib.GP_STAT_COUNT, dtype=torch.float64, device=dev)
    obj_stats = torch.zeros((B, _lib.GP_STAT_COUNT), dtype=torch.float64, device=dev)
    ws_bytes = _lib.load().gp_scorenet_ode_objects_workspace_bytes(B, rpo)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    if T_obj is not None:
        n_eval = 0 if num_steps is None else int(num_steps)
        dense = None if num_steps is None else torch.empty((n_eval, batch_size, POSE_DIM), dtype=torch.float64, device=dev)
        _lib.call("gp_scorenet_ode_objects_t0", _lib.ptr(net.packed()), _lib.ptr(proj), _lib.ptr(x0), _lib.ptr(center),
                  batch_size, rpo, _lib.ptr(T_obj), float(eps), float(rtol), float(atol), 1 if denoise else 0,
                  _lib.ptr(x_out), _lib.ptr(t_eval if dense is not None else None), n_eval, _lib.ptr(dense),
                  _lib.ptr(stats), _lib.ptr(obj_stats), _lib.ptr(ws), ws_bytes, _mlp_mode(score_model), device=dev)
        if dense is not None:
            xs = torch.empty((batch_size, n_eval, POSE_DIM), dtype=torch.float64, device=dev)
            _lib.call("gp_traj_finalize", _lib.ptr(dense), _lib.ptr(center), n_eval, batch_size, _lib.ptr(xs), device=dev)
        else:
            xs = x_out.unsqueeze(1)
        last_ode_stats.clear()
        last_ode_stats["device_stats"] = stats
        last_ode_stats["device_obj_stats"] = obj_stats
        _watch(stats)
        return xs, x_out
    args = (_lib.ptr(net.packed()), _lib.ptr(proj), _lib.ptr(x0), _lib.ptr(center), batch_size, rpo, float(T),
            float(eps), float(rtol), float(atol), 1 if denoise else 0, _lib.ptr(x_out))
    if num_steps is not None:
        t_eval = torch.from_numpy(np.linspace(T, eps, int(num_steps))).to(dev)
        dense = torch.empty((int(num_steps), batch_size, POSE_DIM), dtype=torch.float64, device=dev)
        _lib.call("gp_scorenet_ode_dense_objects", *args, _lib.ptr(t_eval), int(num_steps), _lib.ptr(dense),
                  _lib.ptr(stats), _lib.ptr(obj_stats), _lib.ptr(ws), ws_bytes, _mlp_mode(score_model), device=dev)
        xs = torch.empty((batch_size, int(num_steps), POSE_DIM), dtype=torch.float64, device=dev)
        _lib.call("gp_traj_finalize", _lib.ptr(dense), _lib.ptr(center), int(num_steps), batch_size, _lib.ptr(xs),
                  device=dev)
    else:
        _lib.call("gp_scorenet_ode_objects", *args, _lib.ptr(stats), _lib.ptr(obj_stats), _lib.ptr(ws), ws_bytes,
                  _mlp_mode(score_model), device=dev)
        xs = x_out.unsqueeze(1)
    last_ode_stats.clear()
    last_ode_stats["device_stats"] = stats
    last_ode_stats["device_obj_stats"] = obj_stats
    _watch(stats)
    return xs, x_out


def _record_stats(st, obj=None):
    last_ode_stats.clear()
    last_ode_stats.update(
        nfev=int(st[_lib.STAT_NFEV]), accepted=int(st[_lib.STAT_ACCEPTED]), rejected=int(st[_lib.STAT_REJECTED]),
        status=int(st[_lib.STAT_STATUS]), t_final=float(st[_lib.STAT_T_FINAL]),
        h_initial=float(st[_lib.STAT_H_INITIAL]), h_last=float(st[_lib.STAT_H_LAST]))
    if obj is not None:   # step_control="object": per-object arrays [B] beside the summary (nfev max, sums, first status)
        for key, col in (("obj_nfev", _lib.STAT_NFEV), ("obj_accepted", _lib.STAT_ACCEPTED),
                         ("obj_rejected", _lib.STAT_REJECTED), ("obj_status", _lib.STAT_STATUS)):
            last_ode_stats[key] = obj[:, col].astype(np.int64)
    if last_ode_stats["status"] != 0:
        # the reference ignores solve_ivp's status (samplers.py:226-236); here a failed integration is an error
        raise RuntimeError(f"device RK45 integration failed with status {last_ode_stats['status']} "
                           "(-1: step size underflow, -2: attempt cap); its poses are NaN")


def ode_stats():
    """Statistics of the last cond_ode_sampler call as a dict (synchronises if still on device)."""
    if "device_stats" in last_ode_stats:
        st = last_ode_stats["device_stats"].cpu()
        obj = last_ode_stats.get("device_obj_stats")
        obj = None if obj is None else obj.cpu().numpy()
        _pending_stats.clear()   # the call being read is the newest one; older ones were checked when it was issued
        _record_stats(st, obj)
    return dict(last_ode_stats)


def cond_pc_sampler(score_model, data, prior, sde_coeff, num_steps=500, snr=0.16, device="cuda", eps=1e-5,
                    pose_mode="quat_wxyz", init_x=None, noise=None, *, step_control="batch", noise_keys=None):
    """-> (xs [N, num_steps, 9] f32, mean_x [N, 9] f32).  `noise` (not in the reference):
    [num_steps, 2, N, 9] tensor replacing the per-step `torch.randn_like` draws; by default they are
    drawn with torch on `device` in the reference's call order.  `step_control`: "batch" only (the
    Langevin step size is one batch-wide reduction); "object" raises NotImplementedError.  `noise_keys`: keyed
    per-object noise is offered by the ODE sampler only; anything but None raises NotImplementedError."""
    if pose_mode != "rot_matrix":
        raise NotImplementedError("accelerated sampler supports pose_mode='rot_matrix' only")
    if noise_keys is not None:
        raise NotImplementedError("noise_keys (keyed per-object noise) is implemented for the ODE sampler only")
    check_step_control(step_control, "pc")
    net = _score_net(score_model)
    batch_size = data["pts"].shape[0]
    x0 = _to_device_async(prior((batch_size, POSE_DIM)), device) if init_x is None else init_x
    dev = x0.device
    x0 = x0.to(torch.float32).contiguous()
    time_steps = torch.linspace(1.0, eps, num_steps, device=dev)
    if noise is None:
        noise = torch.stack([torch.stack([torch.randn_like(x0), torch.randn_like(x0)]) for _ in range(num_steps)])
    noise = _lib.check_cuda(noise.to(dev, torch.float32).contiguous(), "noise", torch.float32)
    feat, rpo = _object_features(data, batch_size)
    proj = net.project(feat.to(dev))
    center = _lib.check_cuda(data["pts_center"].to(torch.float32).contiguous(), "pts_center", torch.float32)
    xs = torch.empty((batch_size, num_steps, POSE_DIM), dtype=torch.float32, device=dev)
    mean_x = torch.empty((batch_size, POSE_DIM), dtype=torch.float32, device=dev)
    ws_bytes = _lib.load().gp_scorenet_pc_workspace_bytes(batch_size)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.call("gp_scorenet_pc", _lib.ptr(net.packed()), _lib.ptr(proj), _lib.ptr(x0), _lib.ptr(noise),
              _lib.ptr(center), _lib.ptr(time_steps), batch_size, rpo, int(num_steps), float(snr), _lib.ptr(xs),
              _lib.ptr(mean_x), _lib.ptr(ws), ws_bytes, _mlp_mode(score_model), device=dev)
    return xs, mean_x

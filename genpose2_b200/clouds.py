"""Per-object point clouds built on the device from a depth frame and an instance-label image (DESIGN.md section 4.13).

The pipeline takes `pts [B,1024,3]` and `pts_center [B,3]`; the reference's datasets build them on the host, one object
at a time (back-project the object's pixels, `sample_points` to 1024 points, take the mean:
datasets/datasets_omni6dpose.py:459-473).  Here both stages run on libgenpose_b200.so:

  backproject_instances   depth + labels -> ragged per-object clouds (xyz, offsets)         gp_backproject_instances
  sample_points           ragged clouds -> fixed-size clouds with a keyed random choice     gp_sample_points
  object_clouds           both: the data dict PosePipeline(...)(data, ...) takes
  backproject_frames      stage A over F frames of one size in one pass, objects numbered frame-major
                                                                                    gp_backproject_frames
  object_clouds_frames    both stages over F frames

Object b's sampled cloud depends only on its pixels (or its K points) and keys[b]; the permutation uses the key's
Philox stream with counter word 2 = 1, apart from the prior noise of gp_object_noise, so one key per object can feed
both `object_clouds` and the pipeline's `noise_keys`.  All validation happens before any device work and nothing reads
device memory on the host: every function can be captured in a CUDA graph.
"""
import numpy as np
import torch

from . import _lib
from .samplers import check_noise_keys

MAX_OBJECTS = 1024   # GP_MAX_FRAME_OBJECTS: objects per frame of backproject_instances / object_clouds
MAX_PIXELS = 1 << 30   # GP_MAX_FRAME_PIXELS: pixels per frame (per call of backproject_frames / object_clouds_frames)
MAX_FRAMES = 1024   # GP_MAX_FRAMES: frames per call of backproject_frames / object_clouds_frames


def _device_tensor(t, name, dtype, ndim):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (genpose2_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if t.dim() != ndim:
        raise ValueError(f"{name} must be {ndim}-D, got shape {tuple(t.shape)}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")
    return t


def _same_device(ref, **tensors):
    for name, t in tensors.items():
        if t.device != ref.device:
            raise ValueError(f"{name} is on {t.device}, expected {ref.device}")


def _check_frame(depth, labels, intrinsics, num_objects):
    """-> (H, W, B, (fx, fy, cx, cy) as float32 values)"""
    _device_tensor(depth, "depth", torch.float32, 2)
    _device_tensor(labels, "labels", torch.int32, 2)
    if tuple(labels.shape) != tuple(depth.shape):
        raise ValueError(f"labels {tuple(labels.shape)} and depth {tuple(depth.shape)} must have the same shape")
    _same_device(depth, labels=labels)
    H, W = depth.shape
    if H * W == 0:
        raise ValueError("depth must have at least one pixel")
    if H * W > MAX_PIXELS:
        raise NotImplementedError(f"frames of at most 2^30 pixels are supported, got {H} x {W}")
    if isinstance(intrinsics, torch.Tensor) and intrinsics.is_cuda:
        raise TypeError("intrinsics must be host values (reading a CUDA tensor would synchronise)")
    try:
        vals = np.asarray(intrinsics, dtype=np.float64)
    except (TypeError, ValueError):
        raise TypeError(f"intrinsics must be four numbers (fx, fy, cx, cy), got {intrinsics!r}") from None
    if vals.shape != (4,):
        raise ValueError(f"intrinsics must be four numbers (fx, fy, cx, cy), got shape {vals.shape}")
    with np.errstate(over="ignore"):
        f32 = vals.astype(np.float32)
    if not np.isfinite(f32).all() or f32[0] == 0 or f32[1] == 0:
        raise ValueError(f"intrinsics must be finite float32 values with fx, fy != 0, got {vals.tolist()}")
    if isinstance(num_objects, bool) or not isinstance(num_objects, (int, np.integer)):
        raise TypeError(f"num_objects must be an int, got {type(num_objects).__name__}")
    B = int(num_objects)
    if B < 1:
        raise ValueError(f"num_objects must be >= 1, got {B}")
    if B > MAX_OBJECTS:
        raise NotImplementedError(f"at most {MAX_OBJECTS} objects per frame are supported, got {B}")
    return H, W, B, tuple(float(v) for v in f32)


def _check_num_points(num_points):
    if isinstance(num_points, bool) or not isinstance(num_points, (int, np.integer)):
        raise TypeError(f"num_points must be an int, got {type(num_points).__name__}")
    if not 1 <= int(num_points) <= 2 ** 31 - 1:
        raise ValueError(f"num_points must be >= 1, got {num_points}")
    return int(num_points)


def _check_keys(keys, B, ref):
    keys = check_noise_keys(keys, B)
    if keys is None:
        raise TypeError("keys must be an int64 tensor of one key per object, got None")
    _device_tensor(keys, "keys", torch.int64, 1)
    _same_device(ref, keys=keys)
    return keys


def _backproject(depth, labels, H, W, B, intr):
    dev = depth.device
    xyz = torch.empty((H * W, 3), dtype=torch.float32, device=dev)
    offsets = torch.empty((B + 1,), dtype=torch.int32, device=dev)
    lib = _lib.load()
    ws_bytes = lib.gp_backproject_instances_workspace_bytes(H, W, B)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    _lib.call("gp_backproject_instances", _lib.ptr(depth), _lib.ptr(labels), H, W, *intr, B, _lib.ptr(xyz),
              _lib.ptr(offsets), _lib.ptr(ws), ws_bytes, device=dev)
    return xyz, offsets


def _sample(xyz, offsets, keys, N):
    B, dev = keys.shape[0], xyz.device
    pts = torch.empty((B, N, 3), dtype=torch.float32, device=dev)
    center = torch.empty((B, 3), dtype=torch.float32, device=dev)
    counts = torch.empty((B,), dtype=torch.int32, device=dev)
    _lib.call("gp_sample_points", _lib.ptr(xyz) if xyz.numel() else None, xyz.shape[0], _lib.ptr(offsets),
              _lib.ptr(keys), B, N, _lib.ptr(pts), _lib.ptr(center), _lib.ptr(counts), device=dev)
    return pts, center, counts


def backproject_instances(depth, labels, intrinsics, num_objects):
    """Stage A.  depth float32 [H,W] (metres), labels int32 [H,W] (b + 1 = object b, anything outside 1..B is
    background), intrinsics (fx, fy, cx, cy) host numbers (used as float32), num_objects B <= MAX_OBJECTS.

    Pixel (u = column, v = row) is kept iff its label is in 1..B and its depth z is > 0 and finite; its point is
    (((float)u - cx) * z / fx, ((float)v - cy) * z / fy, z) in IEEE float32, no pixel-centre offset.
    Returns (xyz float32 [H*W, 3], offsets int32 [B+1]), both on the device: object b's points are the rows
    offsets[b] .. offsets[b+1]-1 of xyz in row-major pixel order (numpy's xyz[labels == b + 1]); xyz is sized for the
    whole frame so that no host synchronisation is needed, rows from offsets[B] on are unspecified."""
    H, W, B, intr = _check_frame(depth, labels, intrinsics, num_objects)
    return _backproject(depth, labels, H, W, B, intr)


def sample_points(xyz, offsets, num_points=1024, *, keys):
    """Stage B: sample_points (datasets_omni6dpose.py:459-473) with a keyed random choice.  xyz float32 [rows, 3],
    offsets int32 [B+1] (clamped into [0, rows] on the device), keys int64 [B] (device) -> (pts float32 [B,N,3],
    pts_center float32 [B,3], counts int32 [B]), N = num_points.

    With K = offsets[b+1] - offsets[b] points: K < N tiles the cloud N // K times and fills the last N % K rows with
    points pi_b(0..N%K-1); K == N copies it; K > N takes points pi_b(0..N-1); K == 0 gives zero rows, a zero centre
    and counts[b] = 0 (drop such objects before the pipeline).  pi_b is the keyed Feistel permutation of
    include/genpose_b200.h.  pts_center is the float64 mean of the N rows rounded to float32, within 1 float32 ulp
    of the float64 mean of pts (pts.double().mean(1)).  counts[b] = K."""
    _device_tensor(xyz, "xyz", torch.float32, 2)
    if xyz.shape[1] != 3:
        raise ValueError(f"xyz must be [rows, 3], got {tuple(xyz.shape)}")
    _device_tensor(offsets, "offsets", torch.int32, 1)
    B = offsets.shape[0] - 1
    if B < 1:
        raise ValueError(f"offsets must have B + 1 >= 2 entries, got {offsets.shape[0]}")
    _same_device(xyz, offsets=offsets)
    N = _check_num_points(num_points)
    keys = _check_keys(keys, B, xyz)
    return _sample(xyz, offsets, keys, N)


def object_clouds(depth, labels, intrinsics, keys, num_points=1024):
    """Both stages: a depth frame and its instance labels -> {"pts" [B,N,3], "pts_center" [B,3], "counts" [B]} on the
    device, B = len(keys) objects (label b + 1 is object b, keyed by keys[b]).  The dict can be passed straight to
    PosePipeline(...)(data, ...); objects with counts == 0 (no valid pixel) have zero clouds and should be dropped."""
    if not isinstance(keys, torch.Tensor) or keys.dim() != 1:
        raise TypeError("keys must be a 1-D int64 tensor, one key per object")
    H, W, B, intr = _check_frame(depth, labels, intrinsics, keys.shape[0])
    N = _check_num_points(num_points)
    keys = _check_keys(keys, B, depth)
    xyz, offsets = _backproject(depth, labels, H, W, B, intr)
    pts, center, counts = _sample(xyz, offsets, keys, N)
    return {"pts": pts, "pts_center": center, "counts": counts}


def _check_frames(depth, labels, intrinsics, objects_per_frame, num_objects):
    """-> (F, H, W, B, intrinsics, frame offsets): each either a CUDA tensor given by the caller or a host array to
    upload (float32 [F,4], int32 [F+1])."""
    _device_tensor(depth, "depth", torch.float32, 3)
    _device_tensor(labels, "labels", torch.int32, 3)
    if tuple(labels.shape) != tuple(depth.shape):
        raise ValueError(f"labels {tuple(labels.shape)} and depth {tuple(depth.shape)} must have the same shape")
    _same_device(depth, labels=labels)
    F, H, W = depth.shape
    if F * H * W == 0:
        raise ValueError(f"depth must hold at least one frame of at least one pixel, got {tuple(depth.shape)}")
    if F * H * W > MAX_PIXELS:
        raise NotImplementedError(f"at most 2^30 pixels per call are supported, got {F} frames of {H} x {W}")
    if F > MAX_FRAMES:
        raise NotImplementedError(f"at most {MAX_FRAMES} frames per call are supported, got {F}")
    capturing = torch.cuda.is_initialized() and torch.cuda.is_current_stream_capturing()
    if isinstance(intrinsics, torch.Tensor) and intrinsics.is_cuda:
        _device_tensor(intrinsics, "intrinsics", torch.float32, 2)
        if tuple(intrinsics.shape) != (F, 4):
            raise ValueError(f"intrinsics must be [F, 4] = [{F}, 4], got {tuple(intrinsics.shape)}")
        _same_device(depth, intrinsics=intrinsics)
        intr = intrinsics
    else:
        if capturing:
            raise RuntimeError("host intrinsics cannot be used in a CUDA graph capture: pass a CUDA float32 [F, 4] "
                               "tensor")
        try:
            vals = np.asarray(intrinsics, dtype=np.float64)
        except (TypeError, ValueError):
            raise TypeError(f"intrinsics must be F rows of four numbers (fx, fy, cx, cy), got {intrinsics!r}") from None
        if vals.shape != (F, 4):
            raise ValueError(f"intrinsics must be F rows of four numbers (fx, fy, cx, cy): [{F}, 4], got shape "
                             f"{vals.shape}")
        with np.errstate(over="ignore"):
            intr = vals.astype(np.float32)
        bad = ~np.isfinite(intr).all(1) | (intr[:, 0] == 0) | (intr[:, 1] == 0)
        if bad.any():
            f = int(np.nonzero(bad)[0][0])
            raise ValueError(f"intrinsics must be finite float32 values with fx, fy != 0, got {vals[f].tolist()} "
                             f"for frame {f}")
    if num_objects is not None:
        if isinstance(num_objects, bool) or not isinstance(num_objects, (int, np.integer)):
            raise TypeError(f"num_objects must be an int, got {type(num_objects).__name__}")
        num_objects = int(num_objects)
    if isinstance(objects_per_frame, torch.Tensor) and objects_per_frame.is_cuda:
        _device_tensor(objects_per_frame, "objects_per_frame", torch.int32, 1)
        if objects_per_frame.shape[0] != F + 1:
            raise ValueError(f"objects_per_frame as a CUDA tensor holds the frame offsets [F + 1] = [{F + 1}], got "
                             f"{tuple(objects_per_frame.shape)}")
        _same_device(depth, objects_per_frame=objects_per_frame)
        if num_objects is None:
            raise TypeError("the number of objects must be given with CUDA frame offsets (they are not read on the "
                            "host)")
        B, offsets = num_objects, objects_per_frame
    else:
        if capturing:
            raise RuntimeError("host objects_per_frame cannot be used in a CUDA graph capture: pass the frame offsets "
                               "as a CUDA int32 [F + 1] tensor")
        if isinstance(objects_per_frame, torch.Tensor):
            objects_per_frame = objects_per_frame.tolist()
        try:
            counts = list(objects_per_frame)
        except TypeError:
            raise TypeError(f"objects_per_frame must be a sequence of F ints, got {objects_per_frame!r}") from None
        if len(counts) != F:
            raise ValueError(f"objects_per_frame must hold one count per frame: {F} frames, got {len(counts)}")
        for n in counts:
            if isinstance(n, bool) or not isinstance(n, (int, np.integer)):
                raise TypeError(f"objects_per_frame must hold ints, got {n!r}")
            if n < 0:
                raise ValueError(f"objects_per_frame must hold counts >= 0, got {counts}")
        B = int(sum(int(n) for n in counts))
        if num_objects is not None and num_objects != B:
            raise ValueError(f"objects_per_frame sums to {B} objects, expected {num_objects}")
        offsets = counts
    if B < 1:
        raise ValueError(f"the frames must hold at least one object, got {B}")
    if B > MAX_OBJECTS:
        raise NotImplementedError(f"at most {MAX_OBJECTS} objects per call are supported, got {B}")
    if not isinstance(offsets, torch.Tensor):
        offsets = np.concatenate([[0], np.cumsum(offsets)]).astype(np.int32)
    return F, H, W, B, intr, offsets


def _upload(a, dev):
    """Host array -> device through pinned staging, without a synchronisation (torch's pinned-memory cache reuses the
    staging block only after the copy's event)."""
    if isinstance(a, torch.Tensor):
        return a
    return torch.from_numpy(a).pin_memory().to(dev, non_blocking=True)


def _backproject_frames(depth, labels, F, H, W, B, intr, frame_offsets):
    dev = depth.device
    intr, frame_offsets = _upload(intr, dev), _upload(frame_offsets, dev)
    xyz = torch.empty((F * H * W, 3), dtype=torch.float32, device=dev)
    offsets = torch.empty((B + 1,), dtype=torch.int32, device=dev)
    ws_bytes = _lib.load().gp_backproject_frames_workspace_bytes(F, H, W, B)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    _lib.call("gp_backproject_frames", _lib.ptr(depth), _lib.ptr(labels), F, H, W, _lib.ptr(intr),
              _lib.ptr(frame_offsets), B, _lib.ptr(xyz), _lib.ptr(offsets), _lib.ptr(ws), ws_bytes, device=dev)
    return xyz, offsets


def backproject_frames(depth, labels, intrinsics, objects_per_frame, *, num_objects=None):
    """Stage A over F frames of one size in one pass (one frame per tracked video, or per camera of a rig).
    depth float32 [F,H,W], labels int32 [F,H,W], intrinsics one (fx, fy, cx, cy) per frame: host values [F][4] or a
    CUDA float32 [F,4] tensor.  objects_per_frame: the host counts n_f of the F frames, or a CUDA int32 [F+1] tensor of
    frame offsets (0, n_0, n_0 + n_1, ..., B), which needs num_objects = B.  At most MAX_FRAMES frames, MAX_OBJECTS
    objects and MAX_PIXELS pixels in all.

    Objects are numbered frame-major: label l with 1 <= l <= n_f in frame f is object n_0 + ... + n_(f-1) + l - 1, any
    other label (one above n_f too) is background; each frame is back-projected with its own intrinsics by the rules of
    backproject_instances.  Returns (xyz float32 [F*H*W, 3], offsets int32 [B+1]): bit for bit the concatenation, in
    frame order, of backproject_instances on each frame.  Host forms are validated (finite, fx, fy != 0, counts >= 0)
    and uploaded without a synchronisation; CUDA forms are not read on the host, so a graph captured with them replays
    new intrinsics and new per-frame counts (same F, H, W and B).  Malformed CUDA offsets are clamped on the device
    (include/genpose_b200.h, gp_backproject_frames): wrong clouds, never an out-of-bounds access."""
    F, H, W, B, intr, offs = _check_frames(depth, labels, intrinsics, objects_per_frame, num_objects)
    return _backproject_frames(depth, labels, F, H, W, B, intr, offs)


def object_clouds_frames(depth, labels, intrinsics, objects_per_frame, keys, num_points=1024):
    """Both stages over F frames: backproject_frames, then sample_points with keys[b] for object b (B = len(keys),
    objects numbered frame-major) -> {"pts" [B,N,3], "pts_center" [B,3], "counts" [B]}, bit for bit the per-frame
    object_clouds results concatenated.  Host counts must sum to len(keys)."""
    if not isinstance(keys, torch.Tensor) or keys.dim() != 1:
        raise TypeError("keys must be a 1-D int64 tensor, one key per object")
    F, H, W, B, intr, offs = _check_frames(depth, labels, intrinsics, objects_per_frame, keys.shape[0])
    N = _check_num_points(num_points)
    keys = _check_keys(keys, B, depth)
    xyz, offsets = _backproject_frames(depth, labels, F, H, W, B, intr, offs)
    pts, center, counts = _sample(xyz, offsets, keys, N)
    return {"pts": pts, "pts_center": center, "counts": counts}

"""Synthetic inputs for the pose-generation hot path (SURVEY.md section 8(d)).

There is no dataset and no checkpoint offline, so every test / bench input is generated
here under a fixed seed: camera-frame point clouds with the duplicate-tiling the
reference's `sample_points` produces (datasets/datasets_omni6dpose.py:459-473), and
random state dicts with exactly the reference's key layout (SURVEY.md section 5,
"Checkpoint / resume") -- including re-initialised output layers, because the reference
zero-initialises them (`zero_module`, scorenet.py:15-21) which would make the ODE trivial.
"""
import math

import numpy as np
import torch

# ClsMSG_CFG_Light (networks/pts_encoder/pointnet2.py:77-89) with input_channels = 0
SA_NPOINTS = [512, 256, 128, 64, None]
SA_RADII = [[0.01, 0.02], [0.02, 0.04], [0.04, 0.08], [0.08, 0.16], [None, None]]
SA_NSAMPLES = [[16, 32], [16, 32], [16, 32], [16, 32], [None, None]]
SA_MLPS = [
    [[3, 16, 16, 32], [3, 32, 32, 64]],
    [[99, 64, 64, 128], [99, 64, 96, 128]],
    [[259, 128, 196, 256], [259, 128, 196, 256]],
    [[515, 256, 256, 512], [515, 256, 384, 512]],
    [[1027, 512, 512], [1027, 512, 512]],
]


def _linear(gen, out_f, in_f, scale=1.0):
    bound = scale / math.sqrt(in_f)
    w = (torch.rand(out_f, in_f, generator=gen) * 2 - 1) * bound
    b = (torch.rand(out_f, generator=gen) * 2 - 1) * bound
    return w, b


def random_trunk_state_dict(seed, prefix="pose_score_net.", head_std=0.05, bias_std=0.01):
    """PoseScoreNet / PoseEnergyNet parameters (scorenet.py:130-208, energynet.py:60-120)
    for regression_head=Rx_Ry_and_T, pose_mode=rot_matrix, dino=none."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    w, b = _linear(g, 256, 9)
    sd[prefix + "pose_encoder.0.weight"], sd[prefix + "pose_encoder.0.bias"] = w, b
    w, b = _linear(g, 256, 256)
    sd[prefix + "pose_encoder.2.weight"], sd[prefix + "pose_encoder.2.bias"] = w, b
    sd[prefix + "t_encoder.0.W"] = torch.randn(64, generator=g) * 30.0
    w, b = _linear(g, 128, 128)
    sd[prefix + "t_encoder.1.weight"], sd[prefix + "t_encoder.1.bias"] = w, b
    for head in ("rot_x", "rot_y", "trans"):
        w, b = _linear(g, 256, 1408)
        sd[prefix + f"fusion_tail_{head}.0.weight"] = w
        sd[prefix + f"fusion_tail_{head}.0.bias"] = b
        sd[prefix + f"fusion_tail_{head}.2.weight"] = torch.randn(3, 256, generator=g) * head_std
        sd[prefix + f"fusion_tail_{head}.2.bias"] = torch.randn(3, generator=g) * bias_std
    return sd


def random_encoder_state_dict(seed, prefix="pts_encoder.", perturb_bn=True):
    """Pointnet2ClsMSG(0) parameters: conv1x1 (no bias) + BatchNorm2d per layer
    (pytorch_utils.py:5-33, 168-202)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, scales in enumerate(SA_MLPS):
        for i, spec in enumerate(scales):
            for j in range(len(spec) - 1):
                cin, cout = spec[j], spec[j + 1]
                base = f"{prefix}SA_modules.{k}.mlps.{i}.layer{j}."
                std = math.sqrt(2.0 / cin)  # kaiming_normal_, the reference's conv init
                sd[base + "conv.weight"] = torch.randn(cout, cin, 1, 1, generator=g) * std
                if perturb_bn:
                    sd[base + "bn.bn.weight"] = torch.rand(cout, generator=g) * 0.5 + 0.75
                    sd[base + "bn.bn.bias"] = (torch.rand(cout, generator=g) - 0.5) * 0.2
                    sd[base + "bn.bn.running_mean"] = (torch.rand(cout, generator=g) - 0.5) * 0.2
                    sd[base + "bn.bn.running_var"] = torch.rand(cout, generator=g) + 0.5
                else:
                    sd[base + "bn.bn.weight"] = torch.ones(cout)
                    sd[base + "bn.bn.bias"] = torch.zeros(cout)
                    sd[base + "bn.bn.running_mean"] = torch.zeros(cout)
                    sd[base + "bn.bn.running_var"] = torch.ones(cout)
                sd[base + "bn.bn.num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    return sd


def random_gfobjectpose_state_dict(seed):
    """Full GFObjectPose state dict (encoder + trunk), score or energy agent."""
    sd = random_encoder_state_dict(seed)
    sd.update(random_trunk_state_dict(seed + 1))
    return sd


def random_scalenet_state_dict(seed, head_std=0.05, bias_std=0.01):
    """ScaleNet parameters (networks/scalenet.py:12-31)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    w, b = _linear(g, 256, 180)
    sd["axes_encoder.0.weight"], sd["axes_encoder.0.bias"] = w, b
    w, b = _linear(g, 256, 256)
    sd["axes_encoder.2.weight"], sd["axes_encoder.2.bias"] = w, b
    w, b = _linear(g, 256, 1280)
    sd["fusion_tail_length.0.weight"], sd["fusion_tail_length.0.bias"] = w, b
    sd["fusion_tail_length.2.weight"] = torch.randn(3, 256, generator=g) * head_std
    sd["fusion_tail_length.2.bias"] = torch.randn(3, generator=g) * bias_std
    return sd


def _random_rotations(rng, n):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    R = np.stack(
        [
            1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
            2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
            2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y),
        ],
        axis=1,
    ).reshape(n, 3, 3)
    return R


def make_point_clouds(num_objects, num_points=1024, seed=0, dup_fraction=0.1, scale=1.0):
    """Camera-frame clouds: points on the camera-facing faces of a posed box, 1 mm noise.

    `dup_fraction` of the objects are built from K ~ U{300..900} unique points tiled to
    `num_points` the way `sample_points` tiles short clouds, so that exact duplicates (FPS
    and ball-query ties) are exercised.  `scale` stretches the box (encoder sweeps).
    Returns (pts [B,N,3] f32, pts_center [B,3] f32).
    """
    rng = np.random.default_rng(seed)
    B, N = num_objects, num_points
    half = rng.uniform(0.03, 0.12, size=(B, 3)) * scale
    R = _random_rotations(rng, B)
    t = np.stack(
        [rng.uniform(-0.2, 0.2, B), rng.uniform(-0.2, 0.2, B), rng.uniform(0.5, 1.2, B)], axis=1
    )
    pts = np.empty((B, N, 3), dtype=np.float32)
    for b in range(B):
        # sample on the box surface, keep the faces whose outward normal looks at the camera
        face = rng.integers(0, 6, size=4 * N)
        u = rng.uniform(-1, 1, size=(4 * N, 3))
        axis = face // 2
        sign = (face % 2) * 2.0 - 1.0
        u[np.arange(4 * N), axis] = sign
        normal = np.zeros((4 * N, 3))
        normal[np.arange(4 * N), axis] = sign
        p_cam = (u * half[b]) @ R[b].T + t[b]
        n_cam = normal @ R[b].T
        vis = np.einsum("ij,ij->i", n_cam, p_cam) < 0
        p = p_cam[vis]
        if len(p) < N:
            p = p_cam
        p = p[:N] + rng.normal(0.0, 1e-3, size=(N, 3))
        if rng.uniform() < dup_fraction:
            K = int(rng.integers(max(1, (3 * N) // 10), max(2, (9 * N) // 10) + 1)) if N < 1000 else int(rng.integers(300, 901))
            # sample_points: ids = concat(tile(arange(K), N // K), choice(K, N % K))
            ids = np.concatenate(
                [np.tile(np.arange(K), N // K), rng.choice(K, N % K, replace=False)]
            )
            p = p[ids]
        pts[b] = p.astype(np.float32)
    pts_t = torch.from_numpy(pts)
    return pts_t, pts_t.mean(dim=1)


def make_cluster_quaternion_poses(num_objects, repeat_num=50, seed=0, outlier_fraction=0.3,
                                  jitter_deg=2.0):
    """Pose hypotheses [B,R,9] (6D rotation + translation, f64) whose rotations form one tight
    cluster plus a second smaller mode and outliers, so the DBSCAN branch of the aggregation block
    (evaluation_single.py:190-209) is exercised (random-weight sampling yields no clusters,
    SURVEY 8(c) trap 5)."""
    rng = np.random.default_rng(seed)
    B, Rn = num_objects, repeat_num
    out = np.empty((B, Rn, 9), dtype=np.float64)
    for b in range(B):
        base = _random_rotations(rng, 2)
        for r in range(Rn):
            u = rng.uniform()
            if u < outlier_fraction * 0.5:
                Rm = _random_rotations(rng, 1)[0]
            else:
                which = 0 if u < 0.75 else 1
                ax = rng.normal(size=3)
                ax /= np.linalg.norm(ax)
                ang = np.deg2rad(jitter_deg) * rng.normal()
                Kx = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
                dR = np.eye(3) + math.sin(ang) * Kx + (1 - math.cos(ang)) * Kx @ Kx
                Rm = dR @ base[which]
            out[b, r, :3] = Rm[:, 0]
            out[b, r, 3:6] = Rm[:, 1]
            out[b, r, 6:] = rng.normal(0, 0.01, 3) + np.array([0.0, 0.0, 0.8])
    return torch.from_numpy(out)


def make_instance_frame(H, W, num_objects, seed=0, bad_depth=0.0, stray_labels=0.0):
    """A depth frame and its instance-label image (the input of clouds.object_clouds): a slanted background 1.5-2.5 m
    away and B rectangles (labels 1..B, drawn in order, so a later one may cover an earlier one) 0.4-1.2 m away, 1 mm
    depth noise.  Rectangle sides scale with sqrt(H * W / B).  `bad_depth` of the pixels get a depth of 0, -0.5, NaN,
    +inf or -inf; `stray_labels` of them a label outside 1..B (0, -1, B + 1, 2^30).
    Returns (depth float32 [H,W], labels int32 [H,W]) as numpy arrays."""
    rng = np.random.default_rng(seed)
    B = num_objects
    v, u = np.mgrid[0:H, 0:W]
    depth = 1.5 + u / W * 0.5 + v / H * 0.5
    labels = np.zeros((H, W), dtype=np.int32)
    side = np.sqrt(H * W / B)
    for b in range(B):
        h = int(np.clip(side * rng.uniform(0.3, 1.5), 1, H))
        w = int(np.clip(side * rng.uniform(0.3, 1.5), 1, W))
        v0, u0 = int(rng.integers(0, H - h + 1)), int(rng.integers(0, W - w + 1))
        labels[v0:v0 + h, u0:u0 + w] = b + 1
        depth[v0:v0 + h, u0:u0 + w] = rng.uniform(0.4, 1.2) + 0.1 * (u[v0:v0 + h, u0:u0 + w] - u0) / max(w, 1)
    depth = (depth + rng.normal(0.0, 1e-3, size=(H, W))).astype(np.float32)
    pick = rng.random((H, W))
    bad = pick < bad_depth
    depth[bad] = rng.choice(np.array([0.0, -0.5, np.nan, np.inf, -np.inf], dtype=np.float32), int(bad.sum()))
    stray = rng.random((H, W)) < stray_labels
    labels[stray] = rng.choice(np.array([0, -1, B + 1, 1 << 30], dtype=np.int32), int(stray.sum()))
    return depth, labels


def make_instance_frames(H, W, objects_per_frame, seed=0, bad_depth=0.0, stray_labels=0.0):
    """F frames of make_instance_frame (the input of clouds.object_clouds_frames), frame f with objects_per_frame[f]
    objects and seed + f; a frame of 0 objects is a 1-object frame whose labels are all background (label 1 is above
    its count).  Each frame gets its own camera: focal lengths 0.9-1.1 x 600 * W / 640, the principal point within a
    few pixels of the centre.  Returns (depth float32 [F,H,W], labels int32 [F,H,W], intrinsics float64 [F,4])."""
    depth, labels = zip(*(make_instance_frame(H, W, max(n, 1), seed=seed + f, bad_depth=bad_depth,
                                              stray_labels=stray_labels) for f, n in enumerate(objects_per_frame)))
    rng = np.random.default_rng(seed)
    F = len(objects_per_frame)
    focal = 600.0 * W / 640 * rng.uniform(0.9, 1.1, size=(F, 2))
    centre = np.array([W / 2.0, H / 2.0]) + rng.uniform(-4.0, 4.0, size=(F, 2))
    return np.stack(depth), np.stack(labels), np.concatenate([focal, centre], axis=1)

"""GPU: per-object point clouds from a batch of frames (genpose2_b200.clouds.backproject_frames / object_clouds_frames)
against per-frame backproject_instances / object_clouds calls and the CPU restatements (oracle/object_clouds.py,
oracle/object_clouds_frames.py), bit for bit.  Frames of 640x480 and 1280x720, F = 1, 2, 8 and 30 with ragged per-frame counts (empty frames, up to 1024
objects), frame permutation, a graph captured with the CUDA forms replaying new frames and new per-frame counts, and 30
one-object frames through PosePipeline against 30 single-frame steps.  Only well-formed frame offsets reach the device:
the clamp of malformed ones is checked on the CPU."""
import functools

import numpy as np
import pytest
import torch

from genpose2_b200 import clouds, synthetic
from oracle import object_clouds as oc
from oracle import object_clouds_frames as ocf

pytestmark = pytest.mark.gpu

FRAMES = [(480, 640), (720, 1280)]
COUNTS = {
    1: [64],
    2: [0, 37],
    8: [3, 0, 1, 120, 7, 0, 64, 12],
    30: [0, 1, 2, 0, 5, 8, 13, 21, 34, 55, 89, 144, 0, 1, 1, 3, 7, 16, 33, 64, 100, 120, 90, 60, 40, 30, 20, 10, 4, 53],
}
assert sum(COUNTS[30]) == clouds.MAX_OBJECTS


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def ulps(a, b):
    return np.abs(bits(a).astype(np.int64) - bits(b).astype(np.int64))


def offsets_of(counts):
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)


@functools.lru_cache(maxsize=None)
def case(H, W, F):
    counts = COUNTS[F]
    depth, labels, intr = synthetic.make_instance_frames(H, W, counts, seed=F + H, bad_depth=0.03, stray_labels=0.02)
    # labels of the next frame's objects (above this frame's count) are background
    for f in range(F - 1):
        labels[f, :4, :64] = counts[f] + 1 + np.arange(64) % 3
    keys = np.random.default_rng(F + W).integers(-(1 << 62), 1 << 62, size=sum(counts), dtype=np.int64)
    return counts, depth, labels, intr, keys


def per_frame_calls(counts, d, l, intr, keys, N=1024):
    """Each non-empty frame through backproject_instances and object_clouds, concatenated in frame order."""
    xs, offs, outs, base = [], [0], [], 0
    for f, n in enumerate(counts):
        if n == 0:
            continue
        xyz, off = clouds.backproject_instances(d[f], l[f], tuple(intr[f]), n)
        off = off.cpu().numpy()
        xs.append(xyz[:int(off[-1])].cpu().numpy())
        offs += [offs[-1] + int(o) for o in off[1:]]
        outs.append(clouds.object_clouds(d[f], l[f], tuple(intr[f]), keys[base:base + n], N))
        base += n
    cat = {k: torch.cat([o[k] for o in outs]).cpu().numpy() for k in ("pts", "pts_center", "counts")}
    return np.concatenate(xs), np.asarray(offs, np.int32), cat


@pytest.mark.parametrize("H,W", FRAMES)
@pytest.mark.parametrize("F", sorted(COUNTS))
def test_frames_equal_per_frame_calls_and_oracle(H, W, F):
    counts, depth, labels, intr, keys = case(H, W, F)
    B = sum(counts)
    d, l, k = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(keys).cuda()
    xyz, off = clouds.backproject_frames(d, l, intr, counts)
    assert xyz.shape == (F * H * W, 3) and off.shape == (B + 1,)
    out = clouds.object_clouds_frames(d, l, intr, counts, k)
    got_off = off.cpu().numpy()
    total = int(got_off[-1])
    got_xyz = xyz[:total].cpu().numpy()
    got = {n: out[n].cpu().numpy() for n in ("pts", "pts_center", "counts")}

    want_xyz, want_off, want = per_frame_calls(counts, d, l, intr, k)
    assert np.array_equal(got_off, want_off)
    assert np.array_equal(bits(got_xyz), bits(want_xyz))
    for n in ("pts", "pts_center", "counts"):
        assert np.array_equal(got[n].view(np.int32), want[n].view(np.int32)), n

    o_xyz, o_off = ocf.backproject_frames(depth, labels, intr, offsets_of(counts), B)
    assert np.array_equal(got_off, o_off) and np.array_equal(bits(got_xyz), bits(o_xyz))
    o_pts, o_ctr, o_cnt = oc.sample_points(o_xyz, o_off, keys, 1024)
    assert np.array_equal(bits(got["pts"]), bits(o_pts)) and np.array_equal(got["counts"], o_cnt)
    assert ulps(got["pts_center"], o_ctr).max() <= 1
    print(f"{H}x{W} F={F} B={B}: {total} points, {int((o_cnt == 0).sum())} empty objects")


def test_one_frame_equals_object_clouds():
    H, W = 480, 640
    depth, labels = synthetic.make_instance_frame(H, W, 16, seed=12, bad_depth=0.02, stray_labels=0.02)
    intr = (600.0, 610.0, 319.5, 240.25)
    keys = torch.arange(16, dtype=torch.int64, device="cuda") * 7919
    d, l = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda()
    want = clouds.object_clouds(d, l, intr, keys)
    want_xyz, want_off = clouds.backproject_instances(d, l, intr, 16)
    for form in ("host", "cuda"):
        i = [intr] if form == "host" else torch.tensor([intr], dtype=torch.float32, device="cuda")
        c = [16] if form == "host" else torch.tensor([0, 16], dtype=torch.int32, device="cuda")
        got = clouds.object_clouds_frames(d[None], l[None], i, c, keys)
        xyz, off = clouds.backproject_frames(d[None], l[None], i, c, num_objects=16)
        for n in ("pts", "pts_center", "counts"):
            assert torch.equal(got[n], want[n]), (form, n)
        total = int(want_off[-1])
        assert torch.equal(off, want_off) and torch.equal(xyz[:total], want_xyz[:total]), form


def test_permuting_the_frames_permutes_the_objects():
    H, W = 480, 640
    counts, depth, labels, intr, keys = case(H, W, 8)
    perm = np.random.default_rng(3).permutation(len(counts))
    offs = offsets_of(counts)
    obj = np.concatenate([np.arange(offs[f], offs[f + 1]) for f in perm])
    run = lambda dp, lb, it, ct, ks: clouds.object_clouds_frames(torch.from_numpy(np.ascontiguousarray(dp)).cuda(),
                                                                 torch.from_numpy(np.ascontiguousarray(lb)).cuda(),
                                                                 it, ct, torch.from_numpy(ks).cuda())
    a = run(depth, labels, intr, counts, keys)
    b = run(depth[perm], labels[perm], intr[perm], [counts[f] for f in perm], keys[obj])
    for n in ("pts", "pts_center", "counts"):
        assert torch.equal(b[n], a[n][torch.from_numpy(obj).cuda()]), n


def test_graph_with_cuda_forms_replays_new_frames_and_counts():
    H, W, F, N = 480, 640, 6, 1024
    count_sets = [[4, 0, 9, 2, 1, 8], [0, 12, 3, 3, 6, 0], [24, 0, 0, 0, 0, 0]]
    B = 24
    frames = [synthetic.make_instance_frames(H, W, c, seed=50 + i, bad_depth=0.02, stray_labels=0.01)
              for i, c in enumerate(count_sets)]
    keys = [torch.randint(-(1 << 62), 1 << 62, (B,), generator=torch.Generator().manual_seed(s)) for s in (50, 51, 52)]
    s_depth = torch.from_numpy(frames[0][0]).cuda()
    s_labels = torch.from_numpy(frames[0][1]).cuda()
    s_intr = torch.from_numpy(frames[0][2]).float().cuda()
    s_offs = torch.from_numpy(offsets_of(count_sets[0])).cuda()
    s_keys = keys[0].cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        clouds.object_clouds_frames(s_depth, s_labels, s_intr, s_offs, s_keys, N)   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = clouds.object_clouds_frames(s_depth, s_labels, s_intr, s_offs, s_keys, N)
        with pytest.raises(RuntimeError, match="graph capture"):   # host forms are refused before any device work
            clouds.object_clouds_frames(s_depth, s_labels, frames[0][2], s_offs, s_keys, N)
    for i in (2, 1, 0):
        depth, labels, intr = frames[i]
        s_depth.copy_(torch.from_numpy(depth))
        s_labels.copy_(torch.from_numpy(labels))
        s_intr.copy_(torch.from_numpy(intr).float())
        s_offs.copy_(torch.from_numpy(offsets_of(count_sets[i])))
        s_keys.copy_(keys[i])
        graph.replay()
        want = clouds.object_clouds_frames(torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda(), intr,
                                           count_sets[i], keys[i].cuda(), N)
        for n in ("pts", "pts_center", "counts"):
            assert torch.equal(out[n], want[n]), (i, n)


def test_thirty_videos_to_poses_equal_thirty_single_frame_steps():
    """30 one-object frames (one per tracked video, each with its own camera): one object_clouds_frames call and one
    step give every object the aggregated pose and length of its own object_clouds call and one-object step.  Both
    sides run the score and energy nets in the cluster shape."""
    from genpose2_b200.pipeline import PosePipeline
    H, W, F, R = 480, 640, 30, 50
    depth, labels, intr = synthetic.make_instance_frames(H, W, [1] * F, seed=90, bad_depth=0.01)
    keys = torch.randint(-(1 << 62), 1 << 62, (F,), generator=torch.Generator().manual_seed(90))
    pipe = PosePipeline(device="cuda", step_control="object").load_synthetic_weights()
    for agent in (pipe.score_agent, pipe.energy_agent):
        agent.net.pose_score_net.eval_shape = "cluster"
    d, l = torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda()
    data = clouds.object_clouds_frames(d, l, intr, [1] * F, keys.cuda())
    assert (data["counts"] > 0).all()
    pose, length = pipe(dict(data), repeat_num=R, T0=0.55, noise_keys=keys)
    assert torch.isfinite(pose).all() and torch.isfinite(length).all()
    for f in range(F):
        one = clouds.object_clouds(d[f], l[f], tuple(intr[f]), keys[f:f + 1].cuda())
        p1, l1 = pipe(dict(one), repeat_num=R, T0=0.55, noise_keys=keys[f:f + 1])
        assert torch.equal(p1[0], pose[f]) and torch.equal(l1[0], length[f]), f

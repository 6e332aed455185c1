"""GPU: per-object point clouds from a depth frame (genpose2_b200.clouds) against the CPU restatement
(oracle/object_clouds.py).  Stage A bit for bit (xyz rows and offsets), Stage B bit for bit on the rows and within
1 float32 ulp on the centre, an object's cloud independent of the other objects, the keyed choice uniform, a captured
graph equal to eager calls, and the frame -> clouds -> PosePipeline path against the pipeline fed the oracle's clouds."""
import functools

import numpy as np
import pytest
import torch
from scipy import stats

from genpose2_b200 import clouds, synthetic
from oracle import object_clouds as oc
from tests.util import geodesic_mats

pytestmark = pytest.mark.gpu


def intrinsics(H, W):
    return (600.0, 600.0, W / 2.0, H / 2.0) if W <= 640 else (910.0, 910.0, W / 2.0 - 0.5, H / 2.0 + 0.25)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def ulps(a, b):
    return np.abs(bits(a).astype(np.int64) - bits(b).astype(np.int64))


@functools.lru_cache(maxsize=None)
def frame_case(H, W, B, kind):
    if kind == "whole":   # one object covering the whole frame, every depth valid
        depth, _ = synthetic.make_instance_frame(H, W, 1, seed=H + W)
        labels = np.ones((H, W), dtype=np.int32)
    else:                 # bad depths, stray labels and (for B > 1) one object whose pixels are all removed
        depth, labels = synthetic.make_instance_frame(H, W, B, seed=B + H, bad_depth=0.03, stray_labels=0.02)
        if B > 1:
            labels[labels == B // 2 + 1] = 0
    return depth, labels


FRAMES = [(480, 640), (720, 1280)]
CASES = [(B, "mixed") for B in (1, 8, 64, clouds.MAX_OBJECTS)] + [(1, "whole")]


@pytest.mark.parametrize("H,W", FRAMES)
@pytest.mark.parametrize("B,kind", CASES)
def test_backprojection_matches_oracle_bit_for_bit(H, W, B, kind):
    depth, labels = frame_case(H, W, B, kind)
    fx, fy, cx, cy = intrinsics(H, W)
    xyz, off = clouds.backproject_instances(torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda(),
                                            (fx, fy, cx, cy), B)
    want_xyz, want_off = oc.backproject_instances(depth, labels, fx, fy, cx, cy, B)
    got_off = off.cpu().numpy()
    assert np.array_equal(got_off, want_off)
    total = int(want_off[-1])
    assert np.array_equal(bits(xyz[:total].cpu().numpy()), bits(want_xyz))
    if kind == "whole":
        assert total == H * W
    elif B > 1:
        assert want_off[B // 2 + 1] == want_off[B // 2]   # the empty object
    print(f"{H}x{W} B={B} {kind}: {total} points, {int((np.diff(want_off) == 0).sum())} empty objects")


K_VALUES = [1, 2, 3, 511, 1023, 1024, 1025, 4096, 300000]


def ragged(Ks, seed):
    """xyz with the point's index inside its object in x (exact in float32), random y / z; offsets; keys"""
    rng = np.random.default_rng(seed)
    xyz = np.concatenate([np.stack([np.arange(K), rng.normal(0, 0.1, K), rng.uniform(0.4, 1.5, K)], 1)
                          for K in Ks] or [np.zeros((0, 3))]).astype(np.float32)
    offsets = np.concatenate([[0], np.cumsum(Ks)]).astype(np.int32)
    keys = rng.integers(-(1 << 62), 1 << 62, size=len(Ks), dtype=np.int64)
    return xyz, offsets, keys


def run_sample(xyz, offsets, keys, N):
    pts, ctr, cnt = clouds.sample_points(torch.from_numpy(xyz).cuda(), torch.from_numpy(offsets).cuda(), N,
                                         keys=torch.from_numpy(keys).cuda())
    return pts.cpu().numpy(), ctr.cpu().numpy(), cnt.cpu().numpy()


@pytest.mark.parametrize("N", [1024, 4096])
def test_sampling_matches_oracle(N):
    Ks = K_VALUES + [0]
    xyz, offsets, keys = ragged(Ks, seed=N)
    pts, ctr, cnt = run_sample(xyz, offsets, keys, N)
    want_pts, want_ctr, want_cnt = oc.sample_points(xyz, offsets, keys, N)
    assert np.array_equal(bits(pts), bits(want_pts))
    assert np.array_equal(cnt, want_cnt) and cnt.tolist() == Ks
    assert ulps(ctr, want_ctr).max() <= 1
    # against numpy's own float64 mean (pairwise summation, another order) rounded to float32
    assert ulps(ctr, pts.mean(1, dtype=np.float64).astype(np.float32)).max() <= 1
    for b, K in enumerate(Ks):
        ids = pts[b, :, 0].astype(np.int64)
        if K == 0:
            assert not pts[b].any() and not ctr[b].any()
        elif K >= N:
            assert len(np.unique(ids)) == N, K             # no repeated point
        else:
            c = np.bincount(ids, minlength=K)
            assert c.min() == N // K and c.max() == N // K + (N % K > 0) and (c > N // K).sum() == N % K, K


def test_offsets_are_clamped_on_the_device():
    xyz, _, keys = ragged([10, 20], seed=3)
    bad = np.array([-5, 12, 99], dtype=np.int32)          # -> [0, 12), [12, 30)
    pts, ctr, cnt = run_sample(xyz, bad, keys, 64)
    want = oc.sample_points(xyz, bad, keys, 64)
    assert cnt.tolist() == [12, 18] and np.array_equal(bits(pts), bits(want[0]))
    crossed = np.array([20, 5, 30], dtype=np.int32)       # object 0 has K = 0
    pts, ctr, cnt = run_sample(xyz, crossed, keys, 64)
    assert cnt.tolist() == [0, 25] and not pts[0].any() and not ctr[0].any()


def test_an_object_cloud_depends_on_its_points_and_key_only():
    rng = np.random.default_rng(5)
    Ks = [1, 700, 1024, 5000, 0, 3, 20000, 1500]
    xyz, offsets, keys = ragged(Ks, seed=6)
    N = 1024
    pts, ctr, cnt = run_sample(xyz, offsets, keys, N)
    for b, K in enumerate(Ks):   # alone
        sub = xyz[offsets[b]:offsets[b + 1]]
        p1, c1, n1 = run_sample(sub, np.array([0, K], np.int32), keys[b:b + 1], N)
        assert np.array_equal(bits(p1[0]), bits(pts[b])) and np.array_equal(bits(c1[0]), bits(ctr[b])), b
    perm = rng.permutation(len(Ks))   # permuted
    pk = [Ks[i] for i in perm]
    pxyz = np.concatenate([xyz[offsets[i]:offsets[i + 1]] for i in perm])
    pp, pc, _ = run_sample(pxyz, np.concatenate([[0], np.cumsum(pk)]).astype(np.int32), keys[perm], N)
    assert np.array_equal(bits(pp), bits(pts[perm])) and np.array_equal(bits(pc), bits(ctr[perm]))
    # embedded among 8192 objects
    M = 8192
    others = rng.integers(0, 2000, size=M).tolist()
    at = np.sort(rng.choice(M, len(Ks), replace=False))
    big_K = list(others)
    for i, a in enumerate(at):
        big_K[a] = Ks[i]
    bxyz, boff, bkeys = ragged(big_K, seed=7)
    for i, a in enumerate(at):
        bxyz[boff[a]:boff[a + 1]] = xyz[offsets[i]:offsets[i + 1]]
        bkeys[a] = keys[i]
    bp, bc, bn = run_sample(bxyz, boff, bkeys, N)
    assert np.array_equal(bits(bp[at]), bits(pts)) and np.array_equal(bits(bc[at]), bits(ctr))
    assert np.array_equal(bn[at], cnt)


@pytest.mark.parametrize("K,N", [(50, 20), (50, 70), (1000, 600)])
def test_keyed_choice_is_uniform(K, N):
    """Over 20000 keys (fixed seed): how often each point is chosen (all rows of the keyed part) and which point row 0
    of the keyed part holds both pass a chi-square test against uniform."""
    M = 20000
    xyz = np.stack([np.tile(np.arange(K), M), np.zeros(K * M), np.ones(K * M)], 1).astype(np.float32)
    offsets = (np.arange(M + 1) * K).astype(np.int32)
    keys = np.random.default_rng(K + N).integers(-(1 << 62), 1 << 62, size=M, dtype=np.int64)
    pts, _, _ = run_sample(xyz, offsets, keys, N)
    tiled = (N // K) * K if K < N else 0
    ids = pts[:, tiled:, 0].astype(np.int64)
    n_keyed = ids.shape[1]
    freq = np.bincount(ids.reshape(-1), minlength=K)
    assert freq.sum() == M * n_keyed
    p_freq = stats.chisquare(freq).pvalue
    p_first = stats.chisquare(np.bincount(ids[:, 0], minlength=K)).pvalue
    print(f"K={K} N={N}: chi-square p = {p_freq:.3g} (selection), {p_first:.3g} (first keyed row)")
    assert p_freq > 1e-3 and p_first > 1e-3
    assert all(len(np.unique(r)) == n_keyed for r in ids[:200])   # without replacement


def test_object_clouds_in_a_cuda_graph_equals_eager():
    H, W, B, N = 480, 640, 16, 1024
    intr = intrinsics(H, W)
    frames = [synthetic.make_instance_frame(H, W, B, seed=s, bad_depth=0.02, stray_labels=0.01) for s in (40, 41, 42)]
    keys = [torch.randint(-(1 << 62), 1 << 62, (B,), generator=torch.Generator().manual_seed(s)) for s in (40, 41, 42)]
    s_depth = torch.from_numpy(frames[0][0]).cuda()
    s_labels = torch.from_numpy(frames[0][1]).cuda()
    s_keys = keys[0].cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        clouds.object_clouds(s_depth, s_labels, intr, s_keys, N)   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = clouds.object_clouds(s_depth, s_labels, intr, s_keys, N)
    for (depth, labels), k in zip(frames[::-1], keys[::-1]):
        s_depth.copy_(torch.from_numpy(depth))
        s_labels.copy_(torch.from_numpy(labels))
        s_keys.copy_(k)
        graph.replay()
        want = clouds.object_clouds(torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda(), intr, k.cuda(), N)
        for name in ("pts", "pts_center", "counts"):
            assert torch.equal(out[name], want[name]), name


def end_to_end_frame(B=16, seed=3):
    """seeds 3 and 6: every object keeps pixels, some fewer than 1024, some more"""
    H, W = 480, 640
    depth, labels = synthetic.make_instance_frame(H, W, B, seed=seed, bad_depth=0.01)
    keys = torch.randint(-(1 << 62), 1 << 62, (B,), generator=torch.Generator().manual_seed(seed))
    return depth, labels, intrinsics(H, W), keys


def test_frame_to_poses_end_to_end():
    from genpose2_b200.pipeline import PosePipeline
    B, R = 16, 50
    depth, labels, intr, keys = end_to_end_frame(B)
    data = clouds.object_clouds(torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda(), intr, keys.cuda())
    xyz, off = oc.backproject_instances(depth, labels, *intr, B)
    want_pts, want_ctr, want_cnt = oc.sample_points(xyz, off, keys.numpy(), 1024)
    assert (want_cnt > 0).all() and (want_cnt < 1024).any() and (want_cnt > 1024).any()
    assert np.array_equal(bits(data["pts"].cpu().numpy()), bits(want_pts))
    assert ulps(data["pts_center"].cpu().numpy(), want_ctr).max() <= 1
    assert np.array_equal(data["counts"].cpu().numpy(), want_cnt)

    eager = PosePipeline(device="cuda", step_control="object").load_synthetic_weights()
    pose, length = eager(data, repeat_num=R, T0=0.55, noise_keys=keys)
    ref_pose, ref_length = eager({"pts": torch.from_numpy(want_pts).cuda(), "pts_center": torch.from_numpy(want_ctr).cuda()},
                                 repeat_num=R, T0=0.55, noise_keys=keys)
    pose, ref_pose = pose.cpu().numpy().astype(np.float64), ref_pose.cpu().numpy().astype(np.float64)
    geo = geodesic_mats(pose[:, :3, :3], ref_pose[:, :3, :3]).max()
    trans = np.linalg.norm(pose[:, :3, 3] - ref_pose[:, :3, 3], axis=1).max()
    assert np.isfinite(pose).all() and geo <= 1e-3 and trans <= 1e-4, (geo, trans)
    assert torch.allclose(length, ref_length, rtol=0, atol=1e-4)

    graphed = PosePipeline(device="cuda", use_graph=True, step_control="object").load_synthetic_weights()
    for seed in (3, 6):   # the second frame replays the graph captured for the first
        depth, labels, intr, keys = end_to_end_frame(B, seed)
        data = clouds.object_clouds(torch.from_numpy(depth).cuda(), torch.from_numpy(labels).cuda(), intr, keys.cuda())
        a = eager(dict(data), repeat_num=R, T0=0.55, noise_keys=keys)
        g = graphed(dict(data), repeat_num=R, T0=0.55, noise_keys=keys.cuda())
        assert torch.equal(a[0], g[0]) and torch.equal(a[1], g[1]), seed
    assert len(graphed._graphs) == 1

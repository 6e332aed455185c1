"""CPU: the float64 restatements that tests/test_gpu_aggregate_scale.py compares the aggregation and ScaleNet kernels
against are pinned to the float32 restatements they extend (po.scalenet_forward, po.aggregate_pose, which are pinned to
the reference): po.scalenet_f64 equal to float32 rounding relative to its absolute chain S, and po.aggregate_pose's
float64 / stable-sort option equal to the default path (labels exactly, the pose to one float32 rounding)."""
import numpy as np
import torch

from genpose2_b200 import synthetic
from oracle import pose_oracle as po

# An eighth of one float32 rounding relative to S (the worst case of the float32 chains is ~90 roundings; their errors
# are random-signed and S adds absolute values).
TOL = 2.0 ** -27


def _ratio(got, want, S):
    return float(((got.double() - want).abs() / S).max())


def test_scalenet_f64_matches_float32_restatement():
    sd = synthetic.random_scalenet_state_dict(301, head_std=0.5)
    B = 300
    g = torch.Generator().manual_seed(4)
    feat = torch.relu(torch.randn(B, 1024, generator=g))
    axes = torch.from_numpy(synthetic._random_rotations(np.random.default_rng(4), B)).float()
    want, S, R = po.scalenet_f64(sd, axes, feat, rss=True)
    assert want.dtype == torch.float64 and want.shape == (B, 3)
    assert bool((S >= want.abs()).all()) and bool((R <= S * (1 + 1e-12)).all()) and bool((R > 0).all())
    ref32 = po.scalenet_forward(sd, axes, feat)
    r, rr = _ratio(ref32, want, S), _ratio(ref32, want, 2.0 ** -24 * R)
    print(f"scalenet: max |f32 - f64| / S = {r:.2e} (tol {TOL:.2e}), / (2^-24 R) = {rr:.3g}")
    assert r <= TOL, r
    # the GPU kernel's random-signed bound (tests/test_gpu_aggregate_scale.py: 60 u R) holds for float32 torch too
    assert rr <= 60, rr
    want2, S2 = po.scalenet_f64(sd, torch.zeros(B, 4, 4)[:, :3, :3].copy_(axes), feat)   # a strided [B,4,4] view
    assert torch.equal(want2, want) and torch.equal(S2, S)
    # a NaN axis turns into a NaN length (torch.relu passes NaN), and only for that object
    bad = axes.clone()
    bad[7, 1, 2] = float("nan")
    wb, _ = po.scalenet_f64(sd, bad, feat)
    assert bool(wb[7].isnan().all()) and torch.equal(wb[torch.arange(B) != 7], want[torch.arange(B) != 7])


def _energy(B, R, seed):
    return torch.randn(B, R, 2, generator=torch.Generator().manual_seed(seed))


def test_aggregate_f64_matches_default_path():
    poses = torch.cat([synthetic.make_cluster_quaternion_poses(10, 50, seed=s, jitter_deg=j)
                       for s, j in ((1, 1.0), (2, 4.0), (3, 12.0))])
    energy = _energy(30, 50, 5)                  # continuous: no ties, so the stable sort changes nothing
    for clustering in (True, False):
        want, wl = po.aggregate_pose(poses, energy, clustering=clustering)
        got, gl, info = po.aggregate_pose(poses, energy, clustering=clustering, stable=True, float64=True)
        assert got.dtype == torch.float64 and np.array_equal(gl, wl)
        err = float((got.float() - want).abs().max())
        print(f"clustering={clustering}: max |f64 path - f32 path| = {err:.2e}")
        assert err <= 2.0 ** -23, err
        np.testing.assert_array_equal(got[:, :3, 3].float().numpy(), want[:, :3, 3].numpy())
        A, evals = info["A"], info["evals"]
        # A is the unweighted sum of v v^T over the averaged members: trace = member count, eigh's eigenvalues
        members = np.array([(l == np.argmax(np.bincount(l[l >= 0]))).sum() if clustering and (l >= 0).any() else 20
                            for l in gl])
        np.testing.assert_allclose(torch.diagonal(A, dim1=1, dim2=2).sum(1).numpy(), members, rtol=1e-12)
        np.testing.assert_allclose(evals.numpy(), torch.linalg.eigvalsh(A).numpy(), rtol=0, atol=1e-12)
        assert bool((evals[:, 3] - evals[:, 2] > 0).all())
        assert np.isinf(info["margin"]).all() != clustering


def test_aggregate_stable_sort_and_nan():
    """stable=True ranks like torch.sort(descending=True, stable=True): NaN first, ties in index order; a NaN pose in
    the retained set gives NaN rotation and translation rows and labels -1, and changes no other object"""
    poses = synthetic.make_cluster_quaternion_poses(4, 50, seed=9, jitter_deg=2.0)
    energy = torch.round(_energy(4, 50, 9) * 2) / 2            # many ties
    energy[1, [3, 17, 40], 0] = float("nan")
    sp = po._sorted_stable(poses, energy)
    idx = [i for i in (3, 17, 40)] + sorted((i for i in range(50) if i not in (3, 17, 40)),
                                             key=lambda i: -float(energy[1, i, 0]))
    assert torch.equal(sp[1, :, :6], poses[1, idx, :6])
    want, wl, _ = po.aggregate_pose(poses, energy, stable=True, float64=True)
    assert bool(torch.isfinite(want).all())
    bad_p, bad_e = poses.clone(), energy.clone()
    bad_p[2, 5] = float("nan")
    bad_e[2, 5] = float("nan")
    got, gl, info = po.aggregate_pose(bad_p, bad_e, stable=True, float64=True)
    assert bool(got[2, :3].isnan().all()) and got[2, 3].tolist() == [0, 0, 0, 1] and (gl[2] == -1).all()
    assert bool(info["evals"][2].isnan().all())
    keep = [0, 1, 3]
    assert torch.equal(got[keep], want[keep]) and np.array_equal(gl[keep], wl[keep])

"""CPU: the float64 trunk restatement (oracle/pose_oracle.py:trunk_f64) that the GPU trunk tests compare against is
itself pinned to the float32 restatement po.Trunk (which is pinned to the reference): score and energy equal to float32
rounding relative to the absolute chain S, with the projection hoisted per object, a partial last object, per-row t and
several row chunks."""
import pytest
import torch

from genpose2_b200 import synthetic
from oracle import pose_oracle as po

# An eighth of one float32 rounding relative to S.  The worst case of po.Trunk's chains (9 + 256 + 1408 + 256 sums) is
# ~2000 roundings, but their errors are random-signed and S adds absolute values: observed ~1.1e-9.  Dividing by std
# instead of std + 1e-7 moves the score by ~2e-8 S at these inputs, so the pin sees a float32 step that differs.
TOL = 2.0 ** -27


def _inputs(B, rpo, last, seed):
    g = torch.Generator().manual_seed(seed)
    N = (B - 1) * rpo + last
    feat = torch.relu(torch.randn(B, 1024, generator=g))
    t = torch.rand(N, generator=g) * (1 - 1e-5) + 1e-5
    t[:7] = torch.tensor([1e-5, 1.0, 0.55, 0.55, 0.55, 0.3, 1e-5])   # a few repeated times, both ends
    x = torch.randn(N, 9, generator=g) * po.ve_marginal_std(t)[:, None]
    obj = torch.arange(N) // rpo
    return feat, t, x, obj


def _ratio(got, want, S):
    return float(((got.double() - want).abs() / S).max())


@pytest.mark.parametrize("last", [50, 17])
def test_trunk_f64_score_matches_float32_restatement(last):
    sd = synthetic.random_trunk_state_dict(101)
    trunk = po.Trunk(sd)
    feat, t, x, obj = _inputs(4, 50, last, seed=1)
    want, S = po.trunk_f64(sd, feat, 50, x, t, chunk=64)          # chunk < N: rows in several chunks
    assert want.dtype == torch.float64 and want.shape == (x.shape[0], 9) and S.shape == want.shape
    assert bool((S >= want.abs()).all())
    ref32 = trunk.score(feat[obj], x, t[:, None])
    r = _ratio(ref32, want, S)
    print(f"score: max |f32 - f64| / S = {r:.2e} (tol {TOL:.2e})")
    assert r <= TOL, r
    # the root-sum-square scale: at most S, and float32 po.Trunk within the FFMA evaluator's bound on it
    # (tests/test_gpu_trunk_scale.py: 160 u R)
    _, _, R = po.trunk_f64(sd, feat, 50, x, t, chunk=64, rss=True)
    assert bool((R <= S * (1 + 1e-12)).all())
    rr = _ratio(ref32, want, 2.0 ** -24 * R)
    print(f"score: max |f32 - f64| / (2^-24 R) = {rr:.3g}")
    assert rr <= 160, rr
    # chunking and the per-object projection do not change the result
    want1, S1 = po.trunk_f64(sd, feat[obj], 1, x, t, chunk=1 << 20)
    assert _ratio(want1, want, S) <= 1e-12 and _ratio(S1, S, S) <= 1e-12


def test_trunk_f64_energy_matches_float32_restatement():
    sd = synthetic.random_trunk_state_dict(202)
    trunk = po.Trunk(sd)
    feat, t, x, obj = _inputs(3, 50, 23, seed=2)
    g = torch.Generator().manual_seed(3)
    centre = (torch.randn(3, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 0.8]))[obj]
    poses = x.double()
    poses[:, 6:] += centre.double()
    want, S = po.trunk_f64(sd, feat, 50, poses, t, energy=centre, chunk=40)
    assert want.shape == (x.shape[0], 2)
    sp = poses.float()
    sp[:, 6:] -= centre                                   # posenet_agent: type_as(f32), then - pts_center
    ref32 = trunk.energy(feat[obj], sp, t[:, None])
    r = _ratio(ref32, want, S)
    print(f"energy: max |f32 - f64| / S = {r:.2e} (tol {TOL:.2e})")
    assert r <= TOL, r

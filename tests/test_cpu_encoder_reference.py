"""CPU: the float64 encoder restatement (oracle/pose_oracle.py:pointnet2_encoder_f64) that the GPU encoder tests
compare against is itself pinned to the float32 restatement pointnet2_encoder (which is pinned to the reference):
same FPS and ball-query indices, features equal to float32 rounding."""
import torch

from genpose2_b200 import synthetic
from oracle import pose_oracle as po


def test_float64_encoder_restatement_matches_float32_restatement():
    sd = {"pts_encoder." + k: v for k, v in synthetic.random_encoder_state_dict(7, prefix="").items()}
    pts, _ = synthetic.make_point_clouds(3, 1024, seed=9, dup_fraction=0.5)
    want, trace32 = po.pointnet2_encoder(sd, pts, return_indices=True)
    levels, trace64 = [], []
    got = po.pointnet2_encoder_f64(sd, pts, chunk=2, levels=levels, trace=trace64)   # chunk < B: the chunking too
    assert got.dtype == torch.float64 and got.shape == (3, 1024)
    idx32 = [t for t in trace32 if t[0] in ("fps", "bq")]
    assert [t[:-1] for t in idx32] == [t[:-1] for t in trace64]
    for a, b in zip(idx32, trace64):
        assert torch.equal(a[-1].to(torch.int32), b[-1].to(torch.int32)), a[:-1]
    feats32 = [t[2] for t in trace32 if t[0] == "feat"]
    for k in range(5):
        w32 = feats32[k].squeeze(-1).transpose(1, 2) if k < 4 else feats32[k].transpose(1, 2)   # -> [B, M, C]
        f64 = levels[k][1]
        assert f64.shape == w32.shape, (k, f64.shape, w32.shape)
        rel = float((f64 - w32.double()).abs().max() / f64.abs().max())
        assert rel < 2e-6, (k, rel)      # float32 convs / BatchNorm over <= 1027 channels
    rel = float((got - want.double()).abs().max() / got.abs().max())
    assert rel < 2e-6, rel

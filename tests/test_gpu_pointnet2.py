"""GPU: FPS / ball query / gather / grouping through the C ABI vs (i) the C restatement in oracle/
and (ii) the reference's own CUDA extension (oracle/_ref) -- indices must be bit-exact."""
import numpy as np
import pytest
import torch

from genpose2_b200 import synthetic
from oracle import pointnet2_oracle as po
from tests.util import ref_ext

pytestmark = pytest.mark.gpu


def clouds(B, N, seed, dup_fraction=0.5):
    pts, _ = synthetic.make_point_clouds(B, N, seed=seed, dup_fraction=dup_fraction)
    return pts.cuda().contiguous()


def ref_fps(ext, xyz, m):
    B, N, _ = xyz.shape
    out = torch.empty((B, m), dtype=torch.int32, device="cuda")
    temp = torch.full((B, N), 1e10, dtype=torch.float32, device="cuda")
    ext.furthest_point_sampling_wrapper(B, N, m, xyz, temp, out)
    return out


def ref_bq(ext, radius, ns, xyz, new_xyz):
    B, N, _ = xyz.shape
    M = new_xyz.shape[1]
    idx = torch.zeros((B, M, ns), dtype=torch.int32, device="cuda")
    ext.ball_query_wrapper(B, N, M, radius, ns, new_xyz, xyz, idx)
    return idx


@pytest.mark.parametrize("N", [1, 2, 5, 33, 64, 128, 256, 512, 1000, 1024, 1500, 2048, 4096, 8192, 16384])
def test_fps_bit_exact_vs_oracle(N):
    from genpose2_b200 import pointnet2_utils as pu
    B = 6 if N <= 1024 else 2
    xyz = clouds(B, N, seed=N) if N >= 300 else torch.randn(B, N, 3, device="cuda")
    if N >= 8:
        xyz[0, N // 2:] = xyz[0, : N - N // 2].clone()  # exact duplicates: ties everywhere
        xyz[1] = xyz[1, 0]  # all points identical
    m = max(1, N // 2)
    got = pu.furthest_point_sample(xyz, m).cpu().numpy()
    want = po.furthest_point_sample(xyz.cpu().numpy(), m)
    np.testing.assert_array_equal(got, want)
    idx2, new_xyz = pu.furthest_point_sample_gather(xyz, m)
    np.testing.assert_array_equal(idx2.cpu().numpy(), want)
    np.testing.assert_array_equal(new_xyz.cpu().numpy(), np.take_along_axis(xyz.cpu().numpy(), want[..., None].astype(np.int64), 1))


@pytest.mark.parametrize("N,B", [(1024, 64), (1000, 8), (2048, 32), (4096, 16), (8192, 8), (16384, 4)])
def test_fps_bit_exact_vs_reference_ext(N, B):
    ext = ref_ext()
    if ext is None:
        pytest.skip("reference extension (oracle/_ref) not loadable")
    from genpose2_b200 import pointnet2_utils as pu
    xyz = clouds(B, N, seed=100 + N)
    m = N // 2
    got = pu.furthest_point_sample(xyz, m)
    want = ref_fps(ext, xyz, m)
    assert torch.equal(got, want)


def test_fps_encoder_levels_vs_reference_ext():
    """the four FPS levels of the encoder (1024->512->256->128->64), each on the previous level's output"""
    ext = ref_ext()
    from genpose2_b200 import pointnet2_utils as pu
    xyz = clouds(64, 1024, seed=7)
    for m in (512, 256, 128, 64):
        idx, new_xyz = pu.furthest_point_sample_gather(xyz, m)
        want = po.furthest_point_sample(xyz.cpu().numpy(), m) if ext is None else ref_fps(ext, xyz, m).cpu().numpy()
        np.testing.assert_array_equal(idx.cpu().numpy(), want)
        xyz = new_xyz


def _chain_case(kind, B, N):
    if kind == "clouds":  # half the objects are tiled from 300..900 unique points (exact duplicates)
        return clouds(B, N, seed=11)
    if kind == "lattice":  # integer lattice: different locations tie exactly all the time
        g = torch.stack(torch.meshgrid(*[torch.arange(16.0)] * 3, indexing="ij"), -1).reshape(-1, 3)
        return torch.stack([g[torch.randperm(g.shape[0], generator=torch.Generator().manual_seed(b))[:N]] for b in range(B)]).cuda().contiguous()
    if kind == "few":  # 40 distinct locations: the cloud is exhausted long before the first level ends
        base = torch.randn(B, 40, 3)
        return base[:, torch.arange(N) % 40].cuda().contiguous()
    xyz = torch.randn(B, N, 3)
    xyz[:] = xyz[:, :1]  # every point identical
    return xyz.cuda().contiguous()


@pytest.mark.parametrize("kind", ["clouds", "lattice", "few", "same"])
@pytest.mark.parametrize("N", [1024, 1000, 300])
def test_fps_chain_equals_level_by_level_sampling(kind, N):
    """gp_fps_chain over the encoder's cascade (N -> N/2 -> N/4 -> ...): bit-exact with sampling every level (oracle),
    whether or not the prefix shortcut applies."""
    from genpose2_b200 import pointnet2_utils as pu
    B = 16
    xyz = _chain_case(kind, B, N)
    tie, skipped = None, 0
    for level, m in enumerate((N // 2, N // 4, N // 8, N // 16)):
        idx, new_xyz, tie_next = pu.furthest_point_sample_chain(xyz, m, tie)
        want = po.furthest_point_sample(xyz.cpu().numpy(), m)
        np.testing.assert_array_equal(idx.cpu().numpy(), want, err_msg=f"{kind} level {level}")
        np.testing.assert_array_equal(new_xyz.cpu().numpy(),
                                      np.take_along_axis(xyz.cpu().numpy(), want[..., None].astype(np.int64), 1))
        if tie is not None:
            skipped += int((tie >= m).sum())
        assert int(tie_next.max()) <= max(m - 1, int(tie.max()) if tie is not None else 0)
        xyz, tie = new_xyz, tie_next
    if kind == "clouds":  # the shortcut must actually be taken on ordinary clouds (tiled ones included)
        assert skipped >= 3 * B * 3 // 4, skipped
    if kind == "same":  # nothing to vouch for: every step ties
        assert skipped == 0, skipped


def test_fps_chain_without_history_is_plain_fps():
    from genpose2_b200 import pointnet2_utils as pu
    xyz = clouds(8, 512, seed=5)
    idx, new_xyz, tie = pu.furthest_point_sample_chain(xyz, 128, None)
    assert torch.equal(idx, pu.furthest_point_sample(xyz, 128))
    # a history that does not vouch for enough steps is ignored
    short = torch.full((8,), 100, dtype=torch.int32, device="cuda")
    idx2, _, _ = pu.furthest_point_sample_chain(xyz, 128, short)
    assert torch.equal(idx2, idx)


@pytest.mark.parametrize("N,M,radius,ns", [(1024, 512, 0.01, 16), (1024, 512, 0.02, 32), (512, 256, 0.04, 32),
                                           (128, 64, 0.16, 32), (1000, 77, 0.03, 5), (5000, 300, 0.02, 16),
                                           (64, 64, 1e-6, 8)])
def test_ball_query_bit_exact(N, M, radius, ns):
    from genpose2_b200 import pointnet2_utils as pu
    ext = ref_ext()
    B = 5
    xyz = clouds(B, N, seed=N + M)
    idx = pu.furthest_point_sample(xyz, M)
    new_xyz = torch.gather(xyz, 1, idx.long().unsqueeze(-1).expand(-1, -1, 3)).contiguous()
    new_xyz[0, 0] += 10.0  # an empty ball -> all zeros
    got = pu.ball_query(radius, ns, xyz, new_xyz)
    want = po.ball_query(radius, ns, xyz.cpu().numpy(), new_xyz.cpu().numpy())
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    assert (got[0, 0] == 0).all()
    if ext is not None:
        assert torch.equal(got, ref_bq(ext, radius, ns, xyz, new_xyz))
    g0, g1 = pu.ball_query2([radius, radius * 2], [ns, ns * 2], xyz, new_xyz)
    assert torch.equal(g0, got)
    np.testing.assert_array_equal(g1.cpu().numpy(), po.ball_query(radius * 2, ns * 2, xyz.cpu().numpy(), new_xyz.cpu().numpy()))


def test_gather_group_match_oracle_and_reference():
    from genpose2_b200 import pointnet2_utils as pu
    ext = ref_ext()
    B, C, N, M, ns = 3, 37, 513, 100, 12
    feats = torch.randn(B, C, N, device="cuda")
    idx = torch.randint(0, N, (B, M), dtype=torch.int32, device="cuda")
    g = pu.gather_operation(feats, idx)
    np.testing.assert_array_equal(g.cpu().numpy(), po.gather_operation(feats.cpu().numpy(), idx.cpu().numpy()))
    gi = torch.randint(0, N, (B, M, ns), dtype=torch.int32, device="cuda")
    out = pu.grouping_operation(feats, gi)
    np.testing.assert_array_equal(out.cpu().numpy(), po.grouping_operation(feats.cpu().numpy(), gi.cpu().numpy()))
    gi5 = torch.randint(0, N, (B, M, 5), dtype=torch.int32, device="cuda")  # scalar fallback (ns % 4 != 0)
    out5 = pu.grouping_operation(feats, gi5)
    np.testing.assert_array_equal(out5.cpu().numpy(), po.grouping_operation(feats.cpu().numpy(), gi5.cpu().numpy()))
    if ext is not None:
        ref = torch.empty_like(out)
        ext.group_points_wrapper(B, C, N, M, ns, feats, gi, ref)
        assert torch.equal(out, ref)


@pytest.mark.parametrize("C", [0, 96])
def test_query_group_matches_reference_composition(C):
    """QueryAndGroup.forward (pointnet2_utils.py:279-296) composed from the oracle pieces."""
    from genpose2_b200 import pointnet2_utils as pu
    B, N, M, ns = 4, 512, 256, 16
    xyz = clouds(B, N, seed=3)
    idx, new_xyz = pu.furthest_point_sample_gather(xyz, M)
    feats = torch.randn(B, C, N, device="cuda") if C else None
    bq = pu.ball_query(0.03, ns, xyz, new_xyz)
    got = pu.QueryAndGroup(0.03, ns)(xyz, new_xyz, feats).cpu()
    gx = torch.from_numpy(po.grouping_operation(xyz.cpu().transpose(1, 2).contiguous().numpy(), bq.cpu().numpy()))
    gx = gx - new_xyz.cpu().transpose(1, 2).unsqueeze(-1)
    want = gx if not C else torch.cat([gx, torch.from_numpy(po.grouping_operation(feats.cpu().numpy(), bq.cpu().numpy()))], 1)
    assert torch.equal(got, want)


def test_full_size_properties_c3_sweep():
    """BASELINE config 3 sizes (256 objects, N up to 16384): size-independent FPS / ball-query
    properties, plus bit-exactness vs the reference ext when it is present."""
    from genpose2_b200 import pointnet2_utils as pu
    ext = ref_ext()
    for N, B in ((1024, 256), (4096, 256), (16384, 64)):
        xyz = clouds(B, N, seed=N + 1, dup_fraction=0.0) * 1.0
        m = N // 2
        idx, new_xyz = pu.furthest_point_sample_gather(xyz, m)
        assert (idx[:, 0] == 0).all() and int(idx.min()) >= 0 and int(idx.max()) < N
        srt = torch.sort(idx.long(), dim=1)[0]
        assert (srt[:, 1:] != srt[:, :-1]).all(), "FPS must not repeat a point while distinct points remain"
        # farthest-point property on a prefix: the distance of pick j to the earlier picks is non-increasing
        p = new_xyz[:, :64]
        d = (p[:, :, None].double() - p[:, None].double()).norm(dim=-1)
        mins = torch.stack([d[:, j, :j].min(dim=1)[0] for j in range(1, 64)], dim=1)
        assert (mins[:, 1:] <= mins[:, :-1] + 1e-6).all()
        r, ns = 0.02 * (1024 / N) ** 0.5, 16
        bq = pu.ball_query(r, ns, xyz, new_xyz[:, :512].contiguous())
        g = torch.gather(xyz, 1, bq.long().reshape(B, -1, 1).expand(-1, -1, 3)).reshape(B, 512, ns, 3)
        dist = (g - new_xyz[:, :512, None]).norm(dim=-1)
        assert (dist < r * 1.0001).all()  # every returned index is inside the ball (centres are cloud points)
        assert (bq[:, :, 1:] >= bq[:, :, :1]).all()  # ordered scan with first-hit back-fill
        if ext is not None:
            assert torch.equal(idx, ref_fps(ext, xyz, m))
            assert torch.equal(bq, ref_bq(ext, r, ns, xyz, new_xyz[:, :512].contiguous()))


def test_edge_cases_and_errors():
    from genpose2_b200 import pointnet2_utils as pu
    xyz = torch.randn(2, 16, 3, device="cuda")
    assert pu.furthest_point_sample(xyz, 1).tolist() == [[0], [0]]
    assert pu.furthest_point_sample(torch.randn(0, 16, 3, device="cuda"), 4).shape == (0, 4)
    with pytest.raises(RuntimeError):
        pu.furthest_point_sample(torch.randn(1, 20000, 3, device="cuda"), 4)  # documented limit
    with pytest.raises(RuntimeError):
        pu.furthest_point_sample(torch.randn(2, 16, 3), 4)  # CPU tensor: no fallback
    with pytest.raises(TypeError):
        pu.gather_operation(torch.randn(1, 3, 8, device="cuda"), torch.zeros(1, 4, dtype=torch.int64, device="cuda"))


def test_group_rows_and_maxpool_rows():
    """channels-last gather / max-pool vs the reference-layout ops"""
    from genpose2_b200 import pointnet2_utils as pu
    B, N, M, ns = 3, 512, 128, 16
    xyz = clouds(B, N, seed=11)
    idx, new_xyz = pu.furthest_point_sample_gather(xyz, M)
    bq = pu.ball_query(0.05, ns, xyz, new_xyz)
    for C in (0, 7, 96):
        feats = torch.randn(B, C, N, device="cuda") if C else None
        want = pu.query_group(xyz, new_xyz, feats, bq)  # [B, 3+C, M, ns]
        got = pu.group_rows(xyz, new_xyz, None if feats is None else feats.transpose(1, 2).contiguous(), bq)
        assert torch.equal(got.view(B, M, ns, 3 + C).permute(0, 3, 1, 2), want)
        h = torch.randn(B * M * ns, 40, device="cuda")
        out = torch.zeros(B * M, 100, device="cuda")
        pu.maxpool_rows(h, B * M, ns, out=out[:, 20:60])
        assert torch.equal(out[:, 20:60], h.view(B * M, ns, 40).amax(1)) and (out[:, :20] == 0).all() and (out[:, 60:] == 0).all()
        h3 = torch.randn(B * M * ns, 3, device="cuda")  # scalar path
        assert torch.equal(pu.maxpool_rows(h3, B * M, ns), h3.view(B * M, ns, 3).amax(1))


@pytest.mark.parametrize("absolute", [False, True])
def test_ball_query2_tails_equals_ball_query2_plus_torch(absolute):
    """the per-centre by-products of gp_ball_query2_tails (centres relative to the per-object shift, [x y z 0] tail
    rows) are exactly what the torch subtraction / pad they replace produce; the indices are gp_ball_query2's"""
    from genpose2_b200 import pointnet2_utils as pu
    xyz = clouds(5, 1000, 23)
    _, new_xyz = pu.furthest_point_sample_gather(xyz, 300)
    shift = xyz[:, 0:1, :].contiguous()
    (i0, i1), rel, tail = pu.ball_query2_tails((0.02, 0.05), (16, 32), xyz, new_xyz, shift, absolute)
    j0, j1 = pu.ball_query2((0.02, 0.05), (16, 32), xyz, new_xyz)
    assert torch.equal(i0, j0) and torch.equal(i1, j1)
    assert torch.equal(rel, new_xyz - shift)
    assert torch.equal(tail, torch.nn.functional.pad(new_xyz if absolute else new_xyz - shift, (0, 1)))


def test_level_buffer_tails_written_by_the_level_kernels():
    """every level buffer [feat | xyz | 0] of the encoder ends with the centres' tail rows (written by the level-1
    kernel / the centre-term kernel, not by a separate copy)"""
    from genpose2_b200.pointnet2 import Pointnet2ClsMSG
    enc = Pointnet2ClsMSG(0).cuda().eval()
    enc.load_state_dict(synthetic.random_encoder_state_dict(3, prefix=""))
    pts = clouds(4, 1024, 5)
    geo = enc.compute_geometry(pts)
    with torch.no_grad():
        xyz, feat, rows = pts, None, None
        for k, sa in enumerate(enc.SA_modules[:4]):
            xyz, feat, _, rows = sa.forward_cl(xyz, feat, geo[k], pts_rows=rows, return_rows=True)
            C = feat.shape[-1]
            assert rows.shape[1] == C + 4
            assert torch.equal(rows[:, C:], geo[k][3].reshape(-1, 4))
            assert torch.equal(rows[:, :C], feat.reshape(-1, C))

"""GPU: the tcgen05 SharedMLP-layer GEMM (gp_gemm_bias_relu) vs a float64 torch reference, and the
encoder in both operand precisions vs the CPU restatement."""
import numpy as np
import pytest
import torch

from genpose2_b200 import synthetic
from oracle import pose_oracle as po

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("R,K,N,ldx", [(128, 64, 256, 64), (1000, 99, 64, 100), (4096, 259, 196, 260),
                                       (2048, 515, 384, 516), (640, 1027, 512, 1028), (300, 3, 16, 4),
                                       (256, 32, 96, 32),
                                       # grids of >= 2 x SMs CTAs: the `wide` configuration (fewer stages, two CTAs
                                       # per SM).  The GroupAll merged first layer of the 1024-object pass, pooled
                                       # over 64 below, and a 99-wide level-2 shape with a partial last tile.
                                       (65536, 1027, 1024, 1028), (40000, 99, 64, 100)])
@pytest.mark.parametrize("npass", [3, 1])
def test_gemm_bias_relu_matches_float64(R, K, N, ldx, npass):
    """y = relu(x W^T + b) against float64 (on the GPU): the max error over the max value, and per element
    |y - want| <= kappa u S with S = |x| |W|^T + |b| (u = 2^-16 split-bf16, 2^-8 bf16; kappa 16 / 8 as in
    tests/test_gpu_encoder_scale.py); pooled into a column slice between NaN sentinel columns"""
    from genpose2_b200 import pointnet2_utils as pu
    g = torch.Generator().manual_seed(R + K + N)
    x = torch.zeros(R, ldx)
    x[:, :K] = torch.randn(R, K, generator=g)
    x[:, K:] = 7.0  # padding columns must only ever meet zero weights
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g) * 0.1
    x, w, b = x.cuda(), w.cuda(), b.cuda()
    xd, wd, bd = x[:, :K].double(), w.double(), b.double()
    want = torch.relu(xd @ wd.t() + bd)
    S = xd.abs() @ wd.abs().t() + bd.abs()
    del xd
    packed = pu.gemm_pack(w, npass)
    y = pu.gemm_bias_relu(x, packed, b, N, K, npass)
    assert y.shape == (R, (N + 31) // 32 * 32)
    assert (y[:, N:] == 0).all()
    err = float((y[:, :N].double() - want).abs().max() / want.abs().max())
    tol = 5e-5 if npass == 3 else 2e-2
    assert err < tol, err
    u, kappa = (2.0 ** -16, 16.0) if npass == 3 else (2.0 ** -8, 8.0)
    ratio = float(((y[:, :N].double() - want).abs() / (u * S)).max())
    ctas = -(-R // 128) * -(-N // 256)
    print(f"gemm_bias_relu R={R} K={K} N={N} npass={npass}: {ctas} CTAs, max err / (u S) {ratio:.3f}")
    assert ratio <= kappa, ratio
    for ns in (16, 32, 64):
        if R % ns:
            continue
        out = torch.full((R // ns, N + 8), float("nan"), device="cuda")
        out[:, 4:4 + N] = 0      # the pooled GEMM takes its max into a zero-initialised output
        pu.gemm_bias_relu(x, packed, b, N, K, npass, pool_ns=ns, pooled_out=out[:, 4:4 + N])
        assert torch.equal(out[:, 4:4 + N], y[:, :N].view(R // ns, ns, N).amax(1)), ns
        assert out[:, :4].isnan().all() and out[:, 4 + N:].isnan().all()


@pytest.mark.parametrize("mode,tol", [("bf16x3", 1e-4), ("bf16", 3e-2)])
def test_encoder_gemm_engines_vs_cpu_restatement(mode, tol):
    from genpose2_b200.pointnet2 import Pointnet2ClsMSG
    sd = synthetic.random_encoder_state_dict(7, prefix="")
    enc = Pointnet2ClsMSG(0).cuda().eval().set_gemm_mode(mode)
    enc.load_state_dict(sd)
    pts, _ = synthetic.make_point_clouds(3, 1024, seed=9, dup_fraction=0.5)
    with torch.no_grad():
        got = enc(pts.cuda())
    want = po.pointnet2_encoder({"pts_encoder." + k: v for k, v in sd.items()}, pts)
    err = float((got.cpu() - want).abs().max() / want.abs().max())
    print(f"encoder {mode}: max rel err {err:.3e}")
    assert err < tol, err


@pytest.mark.parametrize("npass,tol", [(3, 5e-5), (1, 3e-2)])
@pytest.mark.parametrize("spec,ns,M", [((64, 96, 128), 16, 128),     # fused layers 2+3 (gp_sa_mlp2_fused), level-2 widths
                                        ((128, 196, 256), 32, 100),   # fused, level-3 widths, partial last tile
                                        ((64, 64, 128), 8, 128),      # fused, pool over 8
                                        ((256, 256, 512), 16, 64),    # fused, level-4 widths (two output n-tiles)
                                        ((256, 384, 512), 16, 64),    # hidden width > 256: accumulator passes of 128 columns in split mode
                                        ((64, 64, 128), 32, 200),     # two CTAs per SM shape, partial last tile
                                        ((128, 130, 250), 8, 96)])    # widths that are not multiples of 16 / 64
def test_hoisted_scale_matches_direct_scale(npass, tol, spec, ns, M):
    """the hoisted first layer + gather loader (+ fused layers 2, 3 and max-pool where the widths allow) vs the
    direct (gather rows, 3 GEMMs, max) evaluation in float64"""
    from genpose2_b200 import pointnet2_utils as pu
    from genpose2_b200.pointnet2 import SharedMLP
    B, N, C = 3, 256, 96
    assert pu.sa_mlp2_fused_fits(*spec, npass, ns)    # every encoder shape is fused (H in tensor memory), both modes
    g = torch.Generator().manual_seed(4)
    pts, _ = synthetic.make_point_clouds(B, N, seed=21)
    xyz = pts.cuda()
    idx, new_xyz = pu.furthest_point_sample_gather(xyz, M)
    bq = pu.ball_query(0.05, ns, xyz, new_xyz)
    feat_cl = torch.randn(B, N, C, generator=g).cuda()
    mlp = SharedMLP([C + 3, *spec]).cuda().eval()
    gw = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for name, prm in mlp.named_parameters():
            if prm.dim() > 1:
                prm.copy_(torch.randn(prm.shape, generator=gw) * (1.5 / prm.shape[1] ** 0.5))
            elif name.endswith("weight"):
                prm.copy_(torch.rand(prm.shape, generator=gw) + 0.5)
            else:
                prm.copy_(torch.randn(prm.shape, generator=gw) * 0.1)
        for name, buf in mlp.named_buffers():
            if name.endswith("running_var"):
                buf.copy_(torch.rand(buf.shape, generator=gw) + 0.5)
            elif name.endswith("running_mean"):
                buf.copy_(torch.randn(buf.shape, generator=gw) * 0.1)
    rows = pu.group_rows(xyz, new_xyz, feat_cl, bq).double()
    h = rows
    for w, b in mlp._folded_layers():
        h = torch.relu(h @ w.double().t() + b.double())
    want = h.view(B * M, ns, -1).amax(1)
    out = torch.full((B * M, spec[2]), -1.0, device="cuda")
    pts_rows = torch.cat([feat_cl, xyz, torch.zeros(B, N, 1, device="cuda")], -1).reshape(B * N, -1)
    mlp.forward_hoisted(pts_rows, N, new_xyz, bq, out, "bf16x3" if npass == 3 else "bf16")
    err = float((out.double() - want).abs().max() / want.abs().max())
    print("hoisted scale rel err", npass, err)
    assert err < tol, err


@pytest.mark.parametrize("spec,ns", [((16, 16, 32), 16), ((32, 32, 64), 32), ((32, 32, 64), 16)])
def test_first_level_scale_kernels_match_float64_and_each_other(spec, ns):
    """gp_sa_small_mlp (weights staged in shared memory) and gp_sa_small_mlp_hostw (weights as constant operands
    through the launch's parameter space): same operation order, so bit-identical; both against float64."""
    from genpose2_b200 import pointnet2_utils as pu
    from genpose2_b200.pointnet2 import SharedMLP
    B, N, M = 5, 1024, 512
    pts, _ = synthetic.make_point_clouds(B, N, seed=33)
    xyz = pts.cuda()
    idx, new_xyz = pu.furthest_point_sample_gather(xyz, M)
    bq = pu.ball_query(0.02, ns, xyz, new_xyz)
    mlp = SharedMLP([3, *spec]).cuda().eval()
    gw = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for name, prm in mlp.named_parameters():
            prm.copy_(torch.randn(prm.shape, generator=gw) * (1.5 / prm.shape[1] ** 0.5) if prm.dim() > 1
                      else torch.rand(prm.shape, generator=gw) + 0.5 if name.endswith("weight")
                      else torch.randn(prm.shape, generator=gw) * 0.1)
    rows = pu.group_rows(xyz, new_xyz, None, bq).double()[:, :3]
    h = rows
    for w, b in mlp._folded_layers():
        h = torch.relu(h @ w.double().t() + b.double())
    want = h.view(B * M, ns, -1).amax(1)
    a = torch.full((B * M, spec[2] + 4), -1.0, device="cuda")
    b_ = torch.full((B * M, spec[2] + 4), -1.0, device="cuda")
    pu.sa_small_mlp(xyz, new_xyz, bq, mlp._folded_layers(), a[:, : spec[2]])
    pu.sa_small_mlp_hostw(xyz, new_xyz, bq, mlp._folded_layers_host(), b_[:, : spec[2]])
    assert torch.equal(a, b_)
    assert (a[:, spec[2]:] == -1).all()  # the column slice only
    err = float((a[:, : spec[2]].double() - want).abs().max() / want.abs().max())
    assert err < 1e-5, err


@pytest.mark.parametrize("npass,tol", [(3, 1e-4), (1, 3e-2)])
@pytest.mark.parametrize("spec,ns", [((32, 32, 64), 32), ((16, 16, 32), 16), ((32, 32, 64), 16)])
def test_first_level_on_the_fused_kernel_matches_the_fp32_kernel(npass, tol, spec, ns):
    """gp_sa_mlp2_fused_xyz (first layer K = 3 in the operand loader, layers 2 / 3 + max-pool on tcgen05) vs the FP32
    level-1 kernel gp_sa_small_mlp_hostw on the same ball-query groups, incl. a partial last tile and empty balls"""
    from genpose2_b200 import pointnet2_utils as pu
    from genpose2_b200.pointnet2 import SharedMLP
    B, N, M = 3, 1000, 200 if ns == 32 else 203
    pts, _ = synthetic.make_point_clouds(B, N, seed=31)
    xyz = pts.cuda()
    _, new_xyz = pu.furthest_point_sample_gather(xyz, M)
    idx = pu.ball_query(0.02, ns, xyz, new_xyz)
    mlp = SharedMLP([3, *spec]).cuda().eval()
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for p in mlp.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * 0.3)
        for i in range(3):
            bn = getattr(mlp, f"layer{i}").bn.bn
            bn.running_mean.copy_(torch.randn(bn.running_mean.shape, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(bn.running_var.shape, generator=g) + 0.5)
    ref = torch.empty((B * M, spec[2]), dtype=torch.float32, device="cuda")
    pu.sa_small_mlp_hostw(xyz, new_xyz, idx, mlp._folded_layers_host(), ref)
    t = mlp._tc_hoisted(npass)
    w0, b0 = mlp._folded_layers_host()[0]
    got = torch.empty((B * M, spec[2] + 4), dtype=torch.float32, device="cuda")   # a column slice of a wider buffer
    pu.sa_mlp2_fused_xyz(xyz, new_xyz, idx, w0, b0, t["p1"], t["b1"], t["c1"], t["c2"], t["p2"], t["b2"], t["c3"], npass,
                         got[:, :spec[2]])
    err = (got[:, :spec[2]] - ref).abs().max().item() / ref.abs().max().item()
    assert err < tol, err


def test_centre_term_tail_and_zero_fill():
    """gp_centre_term_tail = gp_centre_term + the tail rows copied into a 4-column slice of a wider buffer; gp_zero is a
    stream-ordered zero fill"""
    from genpose2_b200 import pointnet2_utils as pu
    g = torch.Generator().manual_seed(12)
    rows, c1, ldq = 300, 64, 128
    xyz = torch.randn(rows, 3, generator=g).cuda()
    w0t = torch.randn(3, c1, generator=g).cuda()
    b0 = torch.randn(c1, generator=g).cuda()
    tail = torch.randn(rows, 4, generator=g).cuda()
    buf = torch.full((rows, 260), 7.0, device="cuda")
    q_ref = pu.centre_term(xyz, w0t, b0, ldq)
    q = pu.centre_term(xyz, w0t, b0, ldq, tail=tail, tail_dst=buf[:, 256:260])
    assert torch.equal(q, q_ref)
    assert torch.equal(buf[:, 256:], tail) and bool((buf[:, :256] == 7.0).all())
    want = xyz.double() @ w0t.double() - b0.double()
    assert (q[:, :c1].double() - want).abs().max().item() < 1e-5 and bool((q[:, c1:] == 0).all())
    z = pu.zeros((5, 1, 1024), xyz.device)
    assert z.shape == (5, 1, 1024) and bool((z == 0).all())

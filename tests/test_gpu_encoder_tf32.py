"""GPU: encoder_mode "tf32" -- the set-abstraction GEMMs with tf32 operands (npass = 2: both operands rounded to nearest
tf32, tcgen05 kind::tf32, fp32 accumulation).

- The packed weight images hold the tf32 rounding of W at their swizzled places.
- Rounding, not truncation: against float64 on tf32-rounded operands the only error left is the fp32 accumulation.
- Every kernel case of test_gpu_encoder_scale.py at npass = 2, per element |got - want| <= kappa u S with u = 2^-11
  (tf32's unit roundoff) and kappa = 8, bf16's kappa: each operand is rounded once, as in bf16 mode.
- The whole encoder against the float64 restatement at 64 objects and its batch invariance at 1024 objects.
- The pipeline with tf32 encoders against the default pipeline at bf16's stated bounds (tf32 features move the poses
  past the north-star 1e-3 rad / 1e-4 at T0 = 0.55: a speed mode, as bf16 is), and its graphed step against the eager
  step."""
import numpy as np
import pytest
import torch

from genpose2_b200 import _lib, samplers, synthetic
from genpose2_b200 import pointnet2_utils as pu
from oracle.tf32 import tf32_round
from tests.test_gpu_encoder_scale import (EDGE, GATHER, LEVEL_SCALES, LINEAR, NAN, XYZ_CASES, ClsMSG_CFG_Light,  # noqa: F401
                                          _check_sentinels, _compare_levels, _edge_case, _encoder, _f64_reference,
                                          _fused_schedule, _gather_ref_rows, _layers, _nan_slice, _ref_tail, _report_tiles,
                                          _run_fused, _straddle_geometry, _tables, c2_clouds, c2_reference, c5_clouds,
                                          enc_sd, levels, ref_fused, sms)
from tests.test_gpu_sampler import BF16_ROT_TOL, BF16_TRANS_TOL
from tests.test_gpu_tf32 import unswizzle
from tests.util import geodesic_mats, pose_errors

pytestmark = pytest.mark.gpu

U_TF32 = 2.0 ** -11
KAPPA_TF32 = 8.0
NPASS = 2
ENC_TOL_TF32 = 4e-3     # bf16's 3e-2 scaled by its 2^-3 smaller u


def _check(got, want, S, label, u=U_TF32, kappa=KAPPA_TF32):
    assert bool(torch.isfinite(got).all()), f"{label}: non-finite outputs (a tile or row was skipped)"
    ratio = float(((got.double() - want).abs() / (u * S)).max())
    print(f"{label}: max |got - want| / (u S) = {ratio:.3f} (u 2^{np.log2(u):.0f}, kappa {kappa:g})")
    assert ratio <= kappa, (label, ratio)
    return ratio


def _tiles(label, R, c1, c2, c3, sms):
    # the tf32 images take the places of the split mode's hi and lo images: the same schedule as npass = 3
    _report_tiles(label, R, c1, c2, c3, 3, sms)


def _r(t):
    return torch.from_numpy(tf32_round(t.cpu().numpy())).to(t.device)


# ------------------------------------------------------------------------------------------------------------------
# packing and rounding
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("N,K", [(196, 128), (128, 259), (512, 516), (32, 32)])
def test_pack_layout(N, K):
    """gp_gemm_pack(W, 2): per 256-column n-tile and 64-k chunk, two [bn][32 k] images (k 0..31, k 32..63) holding
    tf32_round(W) at their SWIZZLE_128B places, zeros beyond N and K; the same size as npass = 3"""
    g = torch.Generator().manual_seed(N + K)
    w = torch.randn(N, K, generator=g) * 3.7
    packed = pu.gemm_pack(w.cuda(), NPASS).cpu().numpy().view(np.float32)
    assert packed.nbytes == pu.gemm_pack(w.cuda(), 3).numel()
    wr = np.zeros((N + 255, (K + 63) // 64 * 64), dtype=np.float32)
    wr[:N, :K] = tf32_round(w.numpy())
    off = 0
    for j in range(-(-N // 256)):
        bn = (min(256, N - 256 * j) + 15) // 16 * 16
        for c in range((K + 63) // 64):
            for half in range(2):
                img = packed[off:off + bn * 32]
                off += bn * 32
                want = wr[256 * j:256 * j + bn, 64 * c + 32 * half:64 * c + 32 * half + 32]
                assert np.array_equal(unswizzle(img, bn), want), (j, c, half)
    assert off == packed.size


@pytest.mark.parametrize("K,N,R", [(100, 128, 65536), (260, 256, 32768), (516, 512, 16384)])
def test_rounding_is_to_nearest(sms, K, N, R):
    """gp_gemm_linear and gp_gemm_bias_relu at npass = 2 against float64 on tf32_round(X), tf32_round(W): what is left is
    the fp32 accumulation, within 2 * 2^-16 S.  This also checks the loader's one-add rounding (tf32_rna_bits), which
    relies on the MMA ignoring an operand's 13 low bits.  Non-negative X (activations after a ReLU) and W make a conversion that
    truncated instead of rounding biased by about 2^-11 S: an order of magnitude over this gate.  Against plain float64
    on the unrounded operands: u = 2^-11."""
    g = torch.Generator().manual_seed(K + N)
    x = torch.relu(torch.randn(R, K, generator=g)).cuda()
    w = (torch.randn(N, K, generator=g).abs() / K ** 0.5).cuda()
    b = (torch.randn(N, generator=g) * 0.1).cuda()
    packed = pu.gemm_pack(w, NPASS)
    xr, wr = _r(x).double(), _r(w).double()
    S = x.double().abs() @ w.double().abs().t()
    ldy = (N + 31) // 32 * 32
    y = torch.full((R, ldy), NAN, device="cuda")
    _lib.call("gp_gemm_linear", _lib.ptr(x), R, K, _lib.ptr(packed), N, K, NPASS, _lib.ptr(y), ldy, device=x.device)
    label = f"gemm_linear K={K} N={N} R={R} npass=2"
    _check(y[:, :N], xr @ wr.t(), S, label + " vs rounded operands", u=2.0 ** -16, kappa=2.0)
    _check(y[:, :N], x.double() @ w.double().t(), S, label + " vs float64")
    yb = pu.gemm_bias_relu(x, packed, b, N, K, NPASS)
    label = f"gemm_bias_relu K={K} N={N} R={R} npass=2"
    Sb = S + b.double().abs()
    _check(yb[:, :N], torch.relu(xr @ wr.t() + b.double()), Sb, label + " vs rounded operands", u=2.0 ** -16, kappa=2.0)
    _check(yb[:, :N], torch.relu(x.double() @ w.double().t() + b.double()), Sb, label + " vs float64")


# ------------------------------------------------------------------------------------------------------------------
# the kernel cases of test_gpu_encoder_scale.py at npass = 2
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("k,i,spec,B", LEVEL_SCALES, ids=[f"L{k + 1}s{i}" for k, i, _, _ in LEVEL_SCALES])
def test_fused_scale_at_level_geometry(levels, sms, k, i, spec, B):
    c1 = spec[0]
    lv = levels[k]
    n_src, M = lv["src"].shape[1], lv["centres"].shape[1]
    ns = ClsMSG_CFG_Light["NSAMPLE"][k][i]
    idx = lv["bq"][i][:B].contiguous()
    ldp = (2 * c1 + 31) // 32 * 32
    P, Q = _tables(B, n_src, M, ldp, seed=100 + 10 * k + i)
    col = i * c1
    Ps, Qs = P[:, col:col + c1], Q[:, col:col + c1]
    lay = _layers(*spec, seed=200 + 10 * k + i)
    label = f"fused L{k + 1} scale {i} {spec} ns={ns} B={B} npass=2"
    _tiles(label, B * M * ns, *spec, sms)
    got = _run_fused(Ps, n_src, idx, Qs, lay, spec, NPASS, ns)
    want, S = ref_fused(Ps, n_src, idx, Qs, *lay)
    _check(got, want, S, label)


@pytest.mark.parametrize("name", EDGE)
def test_fused_edge_cases(levels, sms, name):
    n_src, idx, spec = _edge_case(levels, name)
    B, M, ns = idx.shape
    c1 = spec[0]
    P, Q = _tables(B, n_src, M, 2 * c1, seed=300 + EDGE.index(name))
    Ps, Qs = P[:, c1:], Q[:, c1:]
    lay = _layers(*spec, seed=400 + EDGE.index(name))
    label = f"fused {name} {spec} ns={ns} B={B} M={M} npass=2"
    _tiles(label, B * M * ns, *spec, sms)
    got = _run_fused(Ps, n_src, idx, Qs, lay, spec, NPASS, ns)
    want, S = ref_fused(Ps, n_src, idx, Qs, *lay)
    _check(got, want, S, label)


@pytest.mark.parametrize("spec,ns,B", XYZ_CASES)
def test_fused_first_level_at_level_geometry(levels, sms, spec, ns, B):
    """gp_sa_mlp2_fused_xyz at npass = 2: K = c1 <= 32, so GEMM 1 multiplies (and streams) the first tf32 image only"""
    c1, c2, c3 = spec
    lv = levels[0]
    xyz, centres = lv["src"][:B].contiguous(), lv["centres"][:B].contiguous()
    idx = lv["bq"][0 if ns == 16 else 1][:B].contiguous()
    M = idx.shape[1]
    g = torch.Generator().manual_seed(500 + c3 + ns + B)
    w0 = torch.randn(c1, 3, generator=g) * 50.0
    b0 = torch.randn(c1, generator=g) * 0.3
    w1, b1, w2, b2 = _layers(c1, c2, c3, seed=600 + c3 + ns)
    ntiles = -(-B * M * ns // 128)
    label = f"fused_xyz {spec} ns={ns} B={B} npass=2"
    _tiles(label, B * M * ns, c1, c2, c3, sms)
    if B == 61:
        assert ntiles % _fused_schedule(c1, c2, c3, 3, ntiles, sms)[1] != 0
    buf, out = _nan_slice(B * M, c3)
    pu.sa_mlp2_fused_xyz(xyz, centres, idx, w0, b0, pu.gemm_pack(w1, NPASS), b1, c1, c2, pu.gemm_pack(w2, NPASS), b2, c3,
                         NPASS, out)
    _check_sentinels(buf, c3)
    w0d, b0d = w0.double().cuda(), b0.double().cuda()
    wants, Ss = [], []
    for c0 in range(0, B, 16):
        cb = min(B, c0 + 16)
        gi = idx[c0:cb].long().reshape(cb - c0, -1, 1).expand(-1, -1, 3)
        d = xyz[c0:cb].double().gather(1, gi).view(cb - c0, M, ns, 3) - centres[c0:cb].double().unsqueeze(2)
        pre = d @ w0d.t() + b0d
        want, _ = _ref_tail(pre, torch.zeros(cb - c0, M, c1, dtype=torch.float64, device="cuda"), w1, b1, w2, b2, ns)
        s = (d.abs() @ w0d.abs().t() + b0d.abs()) @ w1.double().abs().t() + b1.double().abs()
        S = (s @ w2.double().abs().t() + b2.double().abs()).amax(2)
        wants.append(want.reshape(-1, c3))
        Ss.append(S.reshape(-1, c3))
    _check(out, torch.cat(wants), torch.cat(Ss), label)


@pytest.mark.parametrize("objects", [64, 1024])
@pytest.mark.parametrize("K,ldx,N,n_src", LINEAR)
def test_gemm_linear_matches_float64(sms, objects, K, ldx, N, n_src):
    R = objects * n_src
    g = torch.Generator().manual_seed(K + N + objects)
    x = torch.full((R, ldx), 7.0)
    x[:, :K] = torch.randn(R, K, generator=g)
    x = x.cuda()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    ldy = (N + 31) // 32 * 32
    y = torch.full((R, ldy), NAN, device="cuda")
    packed = pu.gemm_pack(w, NPASS)
    _lib.call("gp_gemm_linear", _lib.ptr(x), R, ldx, _lib.ptr(packed), N, K, NPASS, _lib.ptr(y), ldy, device=x.device)
    ctas = -(-R // 128) * -(-N // 256)
    label = f"gemm_linear K={K} N={N} R={R} npass=2: {ctas} CTAs, {'wide' if ctas >= 2 * sms else 'narrow'}"
    if objects == 1024:
        assert ctas >= 2 * sms, label
    assert bool((y[:, N:] == 0).all()), "padding columns N..ldy must be zero"
    xd, wd = x[:, :K].double(), w.double()
    _check(y[:, :N], xd @ wd.t(), xd.abs() @ wd.abs().t(), label)


@pytest.mark.parametrize("case", GATHER)
def test_gemm_gather_bias_relu_matches_float64_and_the_fused_kernel(levels, sms, case):
    if case == "one_tile":
        lv = levels[1]
        n_src, idx, spec = lv["src"].shape[1], lv["bq"][1][:1, :4].contiguous(), (64, 96, 128)
    elif case == "many_tiles":
        lv = levels[2]
        n_src, idx, spec = lv["src"].shape[1], lv["bq"][1][:64].contiguous(), (128, 196, 256)
    else:
        n_src, idx = _straddle_geometry(levels, 48, 203, 16)
        spec = (128, 196, 256)
    c1, c2, c3 = spec
    B, M, ns = idx.shape
    R = B * M * ns
    P, Q = _tables(B, n_src, M, 2 * c1, seed=700 + GATHER.index(case))
    Ps, Qs = P[:, c1:], Q[:, c1:]
    lay = _layers(*spec, seed=800 + GATHER.index(case))
    w1, b1, w2, b2 = lay
    p1, p2 = pu.gemm_pack(w1, NPASS), pu.gemm_pack(w2, NPASS)
    gidx = idx.reshape(-1).contiguous()
    ctas = -(-R // 128) * -(-c2 // 256)
    label = f"gemm_gather {case} {spec} ns={ns} B={B} npass=2: {ctas} CTAs"
    if case == "many_tiles":
        assert ctas >= 2 * sms
    want, S = _gather_ref_rows(Ps, n_src, idx, Qs, w1, b1)
    ldy = (c2 + 31) // 32 * 32
    h2 = torch.full((R, ldy), NAN, device="cuda")
    _lib.call("gp_gemm_gather_bias_relu", _lib.ptr(Ps), n_src, int(Ps.stride(0)), _lib.ptr(gidx), R, M * ns, _lib.ptr(Qs),
              int(Qs.stride(0)), ns, _lib.ptr(p1), _lib.ptr(b1), c2, c1, NPASS, _lib.ptr(h2), ldy, 0, None, 0,
              device=Ps.device)
    assert bool((h2[:, c2:] == 0).all())
    _check(h2[:, :c2], want, S, label + " unpooled")
    buf, pooled = _nan_slice(B * M, c2)
    pu.gemm_gather_bias_relu(Ps, n_src, gidx, M * ns, Qs, ns, p1, b1, c2, c1, NPASS, pool_ns=ns, pooled_out=pooled)
    _check_sentinels(buf, c2)
    _check(pooled, want.view(B * M, ns, -1).amax(1), S.view(B * M, ns, -1).amax(1), label + " pooled")
    assert torch.equal(pooled, h2[:, :c2].reshape(B * M, ns, -1).amax(1))
    buf3, chain = _nan_slice(B * M, c3)
    chain.zero_()
    pu.gemm_bias_relu(h2, p2, b2, c3, c2, NPASS, pool_ns=ns, pooled_out=chain)
    _check_sentinels(buf3, c3)
    fused = _run_fused(Ps, n_src, idx, Qs, lay, spec, NPASS, ns)
    want3, S3 = ref_fused(Ps, n_src, idx, Qs, *lay)
    _check(chain, want3, S3, label + " unfused tail")
    _check(fused, want3, S3, label + " fused tail")
    ratio = float(((chain.double() - fused.double()).abs() / (U_TF32 * S3)).max())
    print(f"{label}: unfused vs fused {ratio:.3f} u S")
    assert ratio <= 2 * KAPPA_TF32


# ------------------------------------------------------------------------------------------------------------------
# the whole encoder
# ------------------------------------------------------------------------------------------------------------------

def test_encoder_at_c2_matches_float64(enc_sd, c2_clouds, c2_reference):
    enc = _encoder(enc_sd, "tf32")
    lv = []
    with torch.no_grad():
        got, geo = enc(c2_clouds.cuda(), return_geometry=True, levels=lv)
    _compare_levels("encoder C2 [tf32]", got, lv, c2_reference, ENC_TOL_TF32, geo=geo)


def test_encoder_batch_invariance_at_1024_objects(enc_sd, c5_clouds):
    enc = _encoder(enc_sd, "tf32")
    pts = c5_clouds.cuda()
    lv = []
    with torch.no_grad():
        full = enc(pts, levels=lv)
        sel = torch.tensor([0, 1, 127, 511, 512, 700, 1022, 1023])
        small = enc(pts[sel.cuda()].contiguous())
        perm = torch.randperm(1024, generator=torch.Generator().manual_seed(3))
        permuted = enc(pts[perm.cuda()].contiguous())
    assert full.shape == (1024, 1024)
    assert torch.equal(small, full[sel.cuda()]), "batch of 8 differs from the 1024-object pass"
    assert torch.equal(permuted, full[perm.cuda()]), "permuted batch differs from the 1024-object pass"
    sub = torch.arange(5, 1024, 16)
    ref = _f64_reference(enc_sd, c5_clouds[sub])
    lv_sub = [(None if x is None else x[sub.cuda()], f[sub.cuda()]) for x, f in lv]
    _compare_levels("encoder 1024-object pass, 64-object subset [tf32]", full[sub.cuda()], lv_sub, ref, ENC_TOL_TF32)


# ------------------------------------------------------------------------------------------------------------------
# the pipeline
# ------------------------------------------------------------------------------------------------------------------

def _init_x(B, seed):
    R0 = synthetic._random_rotations(np.random.default_rng(seed), B)
    init = torch.zeros(B, 9)
    init[:, :3] = torch.from_numpy(R0[:, :, 0]).float()
    init[:, 3:6] = torch.from_numpy(R0[:, :, 1]).float()
    init[:, 6:] = torch.randn(B, 3, generator=torch.Generator().manual_seed(seed)) * 0.02
    return init.cuda()


@pytest.mark.parametrize("T0,track", [(0.55, False), (0.25, True)])
def test_pipeline_matches_the_default_pipeline(T0, track):
    """8 camera-frame clouds, the same weights and noise: poses and aggregated poses within bf16's stated bounds
    (BF16_ROT_TOL rad / BF16_TRANS_TOL) of the default (split-bf16 encoder) pipeline with the same number of score
    evaluations, lengths (metres, like the translation) within BF16_TRANS_TOL.  Measured on a B200: 1.3e-3 rad / 2.2e-4
    and lengths 1.0e-3 at T0 = 0.55, 2.5e-5 rad / 1.3e-5 and 2.0e-4 in tracking -- outside the north-star 1e-3 / 1e-4."""
    from genpose2_b200.pipeline import PosePipeline
    B, R = 8, 50
    base = PosePipeline(device="cuda").load_synthetic_weights()
    tf = PosePipeline(device="cuda", encoder_mode="tf32").load_synthetic_weights()
    pts, center = synthetic.make_point_clouds(B, 1024, seed=61, dup_fraction=0.25)
    data = {"pts": pts.cuda(), "pts_center": center.cuda()}
    init = _init_x(B, 5) if track else None
    outs, nfev = [], []
    for pipe in (base, tf):
        torch.manual_seed(21)
        outs.append(pipe(dict(data), repeat_num=R, T0=T0, init_x=init, return_all=True))
        nfev.append(samplers.ode_stats()["nfev"])
    a, b = outs
    feat = float((a["pts_feat"] - b["pts_feat"]).abs().max() / a["pts_feat"].abs().max())
    rot, trans = pose_errors(a["pred_pose"].cpu().numpy(), b["pred_pose"].cpu().numpy())
    qa, qb = a["aggregated_pose"].double().cpu().numpy(), b["aggregated_pose"].double().cpu().numpy()
    arot = float(geodesic_mats(qa[:, :3, :3], qb[:, :3, :3]).max())
    atrans = float(np.abs(qa[:, :3, 3] - qb[:, :3, 3]).max())
    dlen = float((a["length"] - b["length"]).abs().max())
    print(f"T0={T0} track={track}: features {feat:.2e} of scale; worst hypothesis {rot:.2e} rad / {trans:.2e}; "
          f"aggregated {arot:.2e} rad / {atrans:.2e}; length {dlen:.2e}; nfev {nfev}")
    assert nfev[0] == nfev[1], nfev
    assert rot <= BF16_ROT_TOL and trans <= BF16_TRANS_TOL, (rot, trans)
    assert arot <= BF16_ROT_TOL and atrans <= BF16_TRANS_TOL, (arot, atrans)
    assert dlen <= BF16_TRANS_TOL, dlen


def test_cuda_graph_step_equals_eager_step():
    from genpose2_b200.pipeline import PosePipeline
    eager = PosePipeline(device="cuda", encoder_mode="tf32").load_synthetic_weights()
    graph = PosePipeline(device="cuda", encoder_mode="tf32", use_graph=True).load_synthetic_weights()
    for B, seed, T0, track in ((8, 0, 0.55, False), (8, 1, 0.55, False), (4, 2, 0.25, True)):
        pts, center = synthetic.make_point_clouds(B, 1024, seed=70 + seed)
        data = {"pts": pts.cuda(), "pts_center": center.cuda()}
        init = _init_x(B, seed) if track else None
        torch.manual_seed(seed)
        a_pose, a_len = eager(dict(data), repeat_num=50, T0=T0, init_x=init)
        torch.manual_seed(seed)
        g_pose, g_len = graph(dict(data), repeat_num=50, T0=T0, init_x=init)
        assert torch.equal(a_pose, g_pose) and torch.equal(a_len, g_len), (B, seed)
    assert len(graph._graphs) == 2

"""GPU: the encoder's tensor-core set-abstraction kernels against float64 at production batch sizes.

At 3 objects every CTA of the persistent fused kernel (gp_sa_mlp2_fused, csrc/sa_fused.cu) runs one tile, and no GEMM
grid is large enough for the `wide` configuration of csrc/gemm_tc.cu.  The cases here run what C2 (64 objects) and
the 1024-object pass run: many tiles per CTA (the weight ring running ahead across tiles, the next tile's indices
requested early and gathered in parts under GEMM 2, mbarrier parities carried from tile to tile), tiles that
straddle two objects, the 8-worker-warp loaders, and the wide GEMM grids.

Per-kernel bound, per element: |got - want| <= kappa * u * S, where want is the same operation in float64 from the
same float32 inputs and S is that chain evaluated in float64 on absolute values (|input|, |W|, |b|, same gather, same
max-pool: |max a - max b| <= max |a - b|).  u = 2^-8 (bf16 operands) or 2^-16 (split-bf16).  Each case prints its
observed max |got - want| / (u S) and its tile schedule.  Every output goes into a column slice of a wider buffer
pre-filled with NaN: every pooled value must be finite (no tile skipped) and the sentinel columns untouched.
"""
import math

import pytest
import torch

from genpose2_b200 import _lib, synthetic
from genpose2_b200 import pointnet2_utils as pu
from genpose2_b200.pointnet2 import Pointnet2ClsMSG, ClsMSG_CFG_Light
from oracle import pose_oracle as po

pytestmark = pytest.mark.gpu

U = {3: 2.0 ** -16, 1: 2.0 ** -8}
KAPPA = {3: 16.0, 1: 8.0}
NAN = float("nan")
SENT = 4          # sentinel columns on each side of an output slice


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def levels():
    """Level geometry of 96 camera-frame clouds (a quarter of them tiled, so ball queries back-fill duplicates): per
    level k < 4 the source points [B, n_src, 3], the centres [B, M, 3] and both ball-query index sets, chained
    through FPS exactly as the encoder computes them."""
    pts, _ = synthetic.make_point_clouds(96, 1024, seed=5, dup_fraction=0.25)
    src = pts.cuda()
    out = []
    for k in range(4):
        _, new_xyz = pu.furthest_point_sample_gather(src, ClsMSG_CFG_Light["NPOINTS"][k])
        bq = pu.ball_query2(ClsMSG_CFG_Light["RADIUS"][k], ClsMSG_CFG_Light["NSAMPLE"][k], src, new_xyz)
        out.append(dict(src=src, centres=new_xyz, bq=bq))
        src = new_xyz
    return out


def _layers(c1, c2, c3, seed):
    """Folded-layer weights scaled like the other encoder tests; every 7th hidden and every 5th output bias is -20,
    so whole H columns and whole pre-pool columns are negative: the ReLU and the pool see zeros."""
    g = torch.Generator().manual_seed(seed)
    w1 = torch.randn(c2, c1, generator=g) * (1.5 / c1 ** 0.5)
    b1 = torch.randn(c2, generator=g) * 0.1
    w2 = torch.randn(c3, c2, generator=g) * (1.5 / c2 ** 0.5)
    b2 = torch.randn(c3, generator=g) * 0.1
    b1[3::7] = -20.0
    b2[2::5] = -20.0
    return [t.cuda() for t in (w1, b1, w2, b2)]


def _nan_slice(rows, cols):
    buf = torch.full((rows, cols + 2 * SENT), NAN, device="cuda")
    return buf, buf[:, SENT:SENT + cols]


def _check_sentinels(buf, cols):
    assert bool(buf[:, :SENT].isnan().all()) and bool(buf[:, SENT + cols:].isnan().all()), "sentinel columns written"


def _check(got, want, S, npass, label):
    assert bool(torch.isfinite(got).all()), f"{label}: non-finite outputs (a tile or row was skipped)"
    ratio = float(((got.double() - want).abs() / (U[npass] * S)).max())
    print(f"{label}: max |got - want| / (u S) = {ratio:.3f} (kappa {KAPPA[npass]:g})")
    assert ratio <= KAPPA[npass], (label, ratio)
    return ratio


def _round16(n):
    return (n + 15) // 16 * 16


def _fused_schedule(c1, c2, c3, npass, ntiles, sms):
    """(two CTAs per SM, grid) of gp_sa_mlp2_fused: the plan() / launch() of csrc/sa_fused.cu restated."""
    im = 2 if npass == 3 else 1
    k1, k2 = -(-c1 // 64), -(-c2 // 64)
    avail = 256 - k2 * 32 * im
    dn = 256 if avail >= 256 else 128
    fits = avail >= 128 and any(im * k1 * 16384 + bias + 512 + 1024 + 2 * 16384 * im <= 113 * 1024 for bias in (3584, 0))
    two = fits and _round16(c2) <= dn and _round16(c3) <= dn
    return two, min(ntiles, 2 * sms if two else sms)


def _report_tiles(label, R, c1, c2, c3, npass, sms):
    ntiles = -(-R // 128)
    two, grid = _fused_schedule(c1, c2, c3, npass, ntiles, sms)
    print(f"{label}: {ntiles} tiles, {'2' if two else '1'} CTA/SM ({4 if two else 8} worker warps), grid {grid}, "
          f"{ntiles // grid}-{-(-ntiles // grid)} tiles per CTA")
    # every CTA runs several tiles: the code that only runs from a CTA's second tile on is covered
    assert ntiles > 4 * sms, (label, ntiles)


def _ref_tail(Pg, Qr, w1, b1, w2, b2, ns):
    """float64 layers 2, 3 and the max-pool, and the same chain on absolute values, for gathered first-layer inputs
    Pg [n, M, ns, c1] and Qr [n, M, c1] (A = relu(Pg - Q))."""
    w1, b1, w2, b2 = (t.double() for t in (w1, b1, w2, b2))
    a = torch.relu(Pg - Qr.unsqueeze(2))
    h = torch.relu(a @ w1.t() + b1)
    want = torch.relu(h @ w2.t() + b2).amax(2)
    s = (Pg.abs() + Qr.abs().unsqueeze(2)) @ w1.abs().t() + b1.abs()
    S = (s @ w2.abs().t() + b2.abs()).amax(2)
    return want, S


def ref_fused(P, n_src, idx, Q, w1, b1, w2, b2, chunk=16):
    """float64 gp_sa_mlp2_fused: P [B*n_src, c1] and Q [B*M, c1] (column slices allowed), idx [B, M, ns]."""
    B, M, ns = idx.shape
    c1 = P.shape[1]
    P3, Q3 = P.reshape(B, n_src, c1), Q.reshape(B, M, c1)
    wants, Ss = [], []
    for b0 in range(0, B, chunk):
        b1_ = min(B, b0 + chunk)
        gi = idx[b0:b1_].long().reshape(b1_ - b0, -1, 1).expand(-1, -1, c1)
        Pg = P3[b0:b1_].double().gather(1, gi).view(b1_ - b0, M, ns, c1)
        want, S = _ref_tail(Pg, Q3[b0:b1_].double(), w1, b1, w2, b2, ns)
        wants.append(want.reshape(-1, want.shape[-1]))
        Ss.append(S.reshape(-1, S.shape[-1]))
    return torch.cat(wants), torch.cat(Ss)


def _tables(B, n_src, M, ldp, seed):
    """Merged per-point / per-centre tables with the encoder's layout ([rows, ldp], one column slice per scale):
    relu(P[idx] - Q) is about half zeros."""
    g = torch.Generator().manual_seed(seed)
    P = torch.randn(B * n_src, ldp, generator=g).cuda()
    Q = (torch.randn(B * M, ldp, generator=g) * 0.5).cuda()
    return P, Q


def _run_fused(P, n_src, idx, Q, lay, spec, npass, ns):
    c1, c2, c3 = spec
    w1, b1, w2, b2 = lay
    B, M, _ = idx.shape
    buf, out = _nan_slice(B * M, c3)
    pu.sa_mlp2_fused(P, n_src, idx.reshape(-1).contiguous(), M * ns, Q, ns, pu.gemm_pack(w1, npass), b1, c1, c2,
                     pu.gemm_pack(w2, npass), b2, c3, npass, ns, out)
    _check_sentinels(buf, c3)
    return out


# (level k, scale i, (c1, c2, c3), objects): the six scales of levels 2-4 with the level's geometry.  The level-4
# 16-sample scale has 512 tiles at 64 objects (3-4 per CTA); it runs at 96 so that every case has > 4 x SMs tiles.
LEVEL_SCALES = [(1, 0, (64, 64, 128), 64), (1, 1, (64, 96, 128), 64),
                (2, 0, (128, 196, 256), 64), (2, 1, (128, 196, 256), 64),
                (3, 0, (256, 256, 512), 96), (3, 1, (256, 384, 512), 64)]


@pytest.mark.parametrize("npass", [3, 1])
@pytest.mark.parametrize("k,i,spec,B", LEVEL_SCALES, ids=[f"L{k + 1}s{i}" for k, i, _, _ in LEVEL_SCALES])
def test_fused_scale_at_level_geometry(levels, sms, npass, k, i, spec, B):
    """gp_sa_mlp2_fused on column slices (offset 0 / c1) of a merged first-layer table, level-k geometry"""
    c1 = spec[0]
    lv = levels[k]
    n_src, M = lv["src"].shape[1], lv["centres"].shape[1]
    ns = ClsMSG_CFG_Light["NSAMPLE"][k][i]
    idx = lv["bq"][i][:B].contiguous()
    ldp = (2 * c1 + 31) // 32 * 32        # _merged_first_layer: two scales of c1 columns each
    P, Q = _tables(B, n_src, M, ldp, seed=100 + 10 * k + i)
    col = i * c1
    Ps, Qs = P[:, col:col + c1], Q[:, col:col + c1]
    lay = _layers(*spec, seed=200 + 10 * k + i)
    label = f"fused L{k + 1} scale {i} {spec} ns={ns} B={B} npass={npass}"
    _report_tiles(label, B * M * ns, *spec, npass, sms)
    got = _run_fused(Ps, n_src, idx, Qs, lay, spec, npass, ns)
    want, S = ref_fused(Ps, n_src, idx, Qs, *lay)
    _check(got, want, S, npass, label)


def _straddle_geometry(levels, B, M, ns):
    """M centres per object of the level-3 sources (256 points): M * ns rows per object is not a multiple of the
    128-row tile, so tiles straddle two objects"""
    src = levels[2]["src"][:B].contiguous()
    _, centres = pu.furthest_point_sample_gather(src, M)
    return src.shape[1], pu.ball_query(0.08, ns, src, centres)


def _edge_case(levels, name):
    """(n_src, idx [B, M, ns], spec) of the edge cases"""
    if name.startswith("straddle"):
        n_src, idx = _straddle_geometry(levels, 48, 203, 16)
        return n_src, idx, (128, 196, 256) if name == "straddle_atoms" else (64, 96, 128)
    lv = levels[1]
    if name == "row8_64_64_256":
        return lv["src"].shape[1], lv["bq"][0][:64].contiguous(), (64, 64, 256)
    if name == "row8_64_384_512":
        return lv["src"].shape[1], lv["bq"][1][:64].contiguous(), (64, 384, 512)
    if name == "pool8":
        return lv["src"].shape[1], pu.ball_query(0.04, 8, lv["src"][:64].contiguous(), lv["centres"][:64].contiguous()), \
            (64, 64, 128)
    assert name == "random_idx_last_row"
    lv = levels[3]
    n_src, M = lv["src"].shape[1], lv["centres"].shape[1]
    g = torch.Generator().manual_seed(17)
    idx = torch.randint(0, n_src, (64, M, 32), generator=g, dtype=torch.int32)
    idx[:, :, 5] = n_src - 1            # the last row of every object's P block
    return n_src, idx.cuda(), (256, 384, 512)


EDGE = ["straddle_atoms", "straddle_rows", "row8_64_64_256", "row8_64_384_512", "pool8", "random_idx_last_row"]


@pytest.mark.parametrize("npass", [3, 1])
@pytest.mark.parametrize("name", EDGE)
def test_fused_edge_cases(levels, sms, npass, name):
    """tiles straddling objects (M = 203, ns = 16: 3248 rows per object) in the per-atom and the one-row-per-thread
    loaders; the 8-worker-warp one-row-per-thread loader (c1 = 64 with a wide output); pool_ns = 8; random indices
    that read the last row of every object's P block"""
    n_src, idx, spec = _edge_case(levels, name)
    B, M, ns = idx.shape
    c1 = spec[0]
    P, Q = _tables(B, n_src, M, 2 * c1, seed=300 + EDGE.index(name))
    Ps, Qs = P[:, c1:], Q[:, c1:]        # the second scale's slice
    lay = _layers(*spec, seed=400 + EDGE.index(name))
    label = f"fused {name} {spec} ns={ns} B={B} M={M} npass={npass}"
    _report_tiles(label, B * M * ns, *spec, npass, sms)
    if name.startswith("straddle"):
        assert (M * ns) % 128 != 0
    got = _run_fused(Ps, n_src, idx, Qs, lay, spec, npass, ns)
    want, S = ref_fused(Ps, n_src, idx, Qs, *lay)
    _check(got, want, S, npass, label)


XYZ_CASES = [((32, 32, 64), 32, 64), ((32, 32, 64), 32, 61), ((32, 32, 256), 32, 64), ((32, 32, 256), 16, 61),
             ((16, 16, 32), 16, 64), ((16, 16, 32), 16, 61)]


@pytest.mark.parametrize("npass", [3, 1])
@pytest.mark.parametrize("spec,ns,B", XYZ_CASES)
def test_fused_first_level_at_level_geometry(levels, sms, npass, spec, ns, B):
    """gp_sa_mlp2_fused_xyz (the K = 3 first layer in the operand loader) on camera-frame clouds (|xyz| ~ 1 m), level-1
    geometry; 61 objects: a tile count that is not a multiple of the grid; (32, 32, 256): the 8-worker-warp loader"""
    c1, c2, c3 = spec
    lv = levels[0]
    xyz, centres = lv["src"][:B].contiguous(), lv["centres"][:B].contiguous()
    idx = lv["bq"][0 if ns == 16 else 1][:B].contiguous()
    M = idx.shape[1]
    g = torch.Generator().manual_seed(500 + c3 + ns + B)
    w0 = torch.randn(c1, 3, generator=g) * 50.0      # W0 . (xyz - centre) ~ 0.5 over the ball radius
    b0 = torch.randn(c1, generator=g) * 0.3
    lay = _layers(c1, c2, c3, seed=600 + c3 + ns)
    w1, b1, w2, b2 = lay
    ntiles = -(-B * M * ns // 128)
    label = f"fused_xyz {spec} ns={ns} B={B} npass={npass}"
    _report_tiles(label, B * M * ns, c1, c2, c3, npass, sms)
    two, grid = _fused_schedule(c1, c2, c3, npass, ntiles, sms)
    if B == 61:
        assert ntiles % grid != 0
    buf, out = _nan_slice(B * M, c3)
    pu.sa_mlp2_fused_xyz(xyz, centres, idx, w0, b0, pu.gemm_pack(w1, npass), b1, c1, c2, pu.gemm_pack(w2, npass), b2,
                         c3, npass, out)
    _check_sentinels(buf, c3)
    w0d, b0d = w0.double().cuda(), b0.double().cuda()
    wants, Ss = [], []
    for c0 in range(0, B, 16):
        cb = min(B, c0 + 16)
        gi = idx[c0:cb].long().reshape(cb - c0, -1, 1).expand(-1, -1, 3)
        d = xyz[c0:cb].double().gather(1, gi).view(cb - c0, M, ns, 3) - centres[c0:cb].double().unsqueeze(2)
        # the first layer as P = W0 . d + b0 with Q = 0; its absolute chain is |W0| . |d| + |b0|
        pre = d @ w0d.t() + b0d
        want, _ = _ref_tail(pre, torch.zeros(cb - c0, M, c1, dtype=torch.float64, device="cuda"), w1, b1, w2, b2, ns)
        s = (d.abs() @ w0d.abs().t() + b0d.abs()) @ w1.double().abs().t() + b1.double().abs()
        S = (s @ w2.double().abs().t() + b2.double().abs()).amax(2)
        wants.append(want.reshape(-1, c3))
        Ss.append(S.reshape(-1, c3))
    _check(out, torch.cat(wants), torch.cat(Ss), npass, label)


# merged first-layer shapes of levels 2-4 (K, ldx, N) at the row counts of 64 (C2) and 1024 objects; the last shape has
# padding columns N..ldy
LINEAR = [(99, 100, 128, 512), (259, 260, 256, 256), (515, 516, 512, 128), (259, 260, 196, 256)]


@pytest.mark.parametrize("npass", [3, 1])
@pytest.mark.parametrize("objects", [64, 1024])
@pytest.mark.parametrize("K,ldx,N,n_src", LINEAR)
def test_gemm_linear_matches_float64(sms, npass, objects, K, ldx, N, n_src):
    """gp_gemm_linear (the per-point table P of every hoisted level); at 1024 objects the wide configuration"""
    R = objects * n_src
    g = torch.Generator().manual_seed(K + N + objects)
    x = torch.full((R, ldx), 7.0)       # padding columns must only ever meet zero weights
    x[:, :K] = torch.randn(R, K, generator=g)
    x = x.cuda()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    ldy = (N + 31) // 32 * 32
    y = torch.full((R, ldy), NAN, device="cuda")
    packed = pu.gemm_pack(w, npass)
    _lib.call("gp_gemm_linear", _lib.ptr(x), R, ldx, _lib.ptr(packed), N, K, npass, _lib.ptr(y), ldy, device=x.device)
    ctas = -(-R // 128) * -(-N // 256)
    label = f"gemm_linear K={K} N={N} R={R} npass={npass}: {ctas} CTAs, {'wide' if ctas >= 2 * sms else 'narrow'}"
    if objects == 1024:
        assert ctas >= 2 * sms, label
    assert bool((y[:, N:] == 0).all()), "padding columns N..ldy must be zero"
    xd, wd = x[:, :K].double(), w.double()
    _check(y[:, :N], xd @ wd.t(), xd.abs() @ wd.abs().t(), npass, label)


def _gather_ref_rows(P, n_src, idx, Q, w, b):
    """float64 rows of gp_gemm_gather_bias_relu (unpooled) and their absolute chain"""
    B, M, ns = idx.shape
    c1 = P.shape[1]
    gi = idx.long().reshape(B, -1, 1).expand(-1, -1, c1)
    Pg = P.reshape(B, n_src, c1).double().gather(1, gi).view(B, M, ns, c1)
    Qr = Q.reshape(B, M, c1).double().unsqueeze(2)
    wd, bd = w.double(), b.double()
    want = torch.relu(torch.relu(Pg - Qr) @ wd.t() + bd)
    S = (Pg.abs() + Qr.abs()) @ wd.abs().t() + bd.abs()
    return want.reshape(B * M * ns, -1), S.reshape(B * M * ns, -1)


GATHER = ["one_tile", "many_tiles", "straddle"]


@pytest.mark.parametrize("npass", [3, 1])
@pytest.mark.parametrize("case", GATHER)
def test_gemm_gather_bias_relu_matches_float64_and_the_fused_kernel(levels, sms, npass, case):
    """gp_gemm_gather_bias_relu (the hoisted_tail path for widths the fused kernel does not take), pooled and unpooled,
    against float64; its unpooled output fed through the pooled gp_gemm_bias_relu (layer 3 + max) against
    gp_sa_mlp2_fused on the same inputs -- the two paths hoisted_tail chooses between"""
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
    p1, p2 = pu.gemm_pack(w1, npass), pu.gemm_pack(w2, npass)
    gidx = idx.reshape(-1).contiguous()
    ctas = -(-R // 128) * -(-c2 // 256)
    label = f"gemm_gather {case} {spec} ns={ns} B={B} npass={npass}: {ctas} CTAs"
    if case == "many_tiles":
        assert ctas >= 2 * sms
    want, S = _gather_ref_rows(Ps, n_src, idx, Qs, w1, b1)
    # unpooled (layer 2)
    ldy = (c2 + 31) // 32 * 32
    h2 = torch.full((R, ldy), NAN, device="cuda")
    _lib.call("gp_gemm_gather_bias_relu", _lib.ptr(Ps), n_src, int(Ps.stride(0)), _lib.ptr(gidx), R, M * ns, _lib.ptr(Qs),
              int(Qs.stride(0)), ns, _lib.ptr(p1), _lib.ptr(b1), c2, c1, npass, _lib.ptr(h2), ldy, 0, None, 0,
              device=Ps.device)
    assert bool((h2[:, c2:] == 0).all())
    _check(h2[:, :c2], want, S, npass, label + " unpooled")
    # pooled (layer 2 + max)
    buf, pooled = _nan_slice(B * M, c2)
    pu.gemm_gather_bias_relu(Ps, n_src, gidx, M * ns, Qs, ns, p1, b1, c2, c1, npass, pool_ns=ns, pooled_out=pooled)
    _check_sentinels(buf, c2)
    _check(pooled, want.view(B * M, ns, -1).amax(1), S.view(B * M, ns, -1).amax(1), npass, label + " pooled")
    assert torch.equal(pooled, h2[:, :c2].reshape(B * M, ns, -1).amax(1))
    # layers 2 + 3 + max: the unfused path against the fused kernel, both against float64
    buf3, chain = _nan_slice(B * M, c3)
    chain.zero_()          # the pooled GEMM takes its max into a zero-initialised output
    pu.gemm_bias_relu(h2, p2, b2, c3, c2, npass, pool_ns=ns, pooled_out=chain)
    _check_sentinels(buf3, c3)
    fused = _run_fused(Ps, n_src, idx, Qs, lay, spec, npass, ns)
    want3, S3 = ref_fused(Ps, n_src, idx, Qs, *lay)
    _check(chain, want3, S3, npass, label + " unfused tail")
    _check(fused, want3, S3, npass, label + " fused tail")
    ratio = float(((chain.double() - fused.double()).abs() / (U[npass] * S3)).max())
    print(f"{label}: unfused vs fused {ratio:.3f} u S")
    assert ratio <= 2 * KAPPA[npass]


@pytest.mark.parametrize("spec,ns,off", [((16, 16, 32), 16, 0), ((32, 32, 64), 32, 32)])
def test_small_mlp_hostw_tail_matches_hostw(levels, spec, ns, off):
    """gp_sa_small_mlp_hostw_tail (the production level-1 narrow scale, which also writes the level buffer's tail):
    feature columns bit-identical to gp_sa_small_mlp_hostw, the four tail columns equal to `tail`, nothing else
    of the level buffer touched"""
    from genpose2_b200.pointnet2 import SharedMLP
    lv = levels[0]
    B = 64
    xyz, centres = lv["src"][:B].contiguous(), lv["centres"][:B].contiguous()
    idx = lv["bq"][0 if ns == 16 else 1][:B].contiguous()
    M = idx.shape[1]
    mlp = SharedMLP([3, *spec]).eval()
    g = torch.Generator().manual_seed(900 + ns)
    with torch.no_grad():
        for name, prm in mlp.named_parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * (1.5 / prm.shape[1] ** 0.5) if prm.dim() > 1
                      else torch.rand(prm.shape, generator=g) + 0.5 if name.endswith("weight")
                      else torch.randn(prm.shape, generator=g) * 0.1)
    host = mlp._folded_layers_host()
    C = 96                                               # both level-1 scales; the tail follows at column C
    tail = torch.randn(B, M, 4, generator=g).cuda()
    ref = torch.full((B * M, C + 4 + SENT), NAN, device="cuda")
    got = torch.full((B * M, C + 4 + SENT), NAN, device="cuda")
    pu.sa_small_mlp_hostw(xyz, centres, idx, host, ref[:, off:off + spec[2]])
    pu.sa_small_mlp_hostw(xyz, centres, idx, host, got[:, off:off + spec[2]], tail=tail, tail_col=C - off)
    assert torch.equal(got[:, off:off + spec[2]], ref[:, off:off + spec[2]])
    assert bool(torch.isfinite(got[:, off:off + spec[2]]).all())
    assert torch.equal(got[:, C:C + 4], tail.view(-1, 4))
    untouched = torch.ones(C + 4 + SENT, dtype=torch.bool)
    untouched[off:off + spec[2]] = False
    untouched[C:C + 4] = False
    assert bool(got[:, untouched.cuda()].isnan().all())


# ------------------------------------------------------------------------------------------------------------------
# the whole encoder against the float64 restatement, and batch invariance at the 1024-object pass
# ------------------------------------------------------------------------------------------------------------------

# the gates of test_encoder_levels_match_reference: each level's max error over its feature scale
ENC_TOL = {"bf16x3": 1e-4, "bf16": 3e-2}


@pytest.fixture(scope="module")
def enc_sd():
    return synthetic.random_encoder_state_dict(7, prefix="")


def _encoder(sd, mode):
    enc = Pointnet2ClsMSG(0).cuda().eval().set_gemm_mode(mode)
    enc.load_state_dict(sd)
    return enc


def _f64_reference(sd, pts):
    lv, trace = [], []
    out = po.pointnet2_encoder_f64({"pts_encoder." + k: v for k, v in sd.items()}, pts, device="cuda", levels=lv,
                                   trace=trace)
    return out, lv, trace


def _compare_levels(label, got, levels_got, ref, tol, geo=None):
    out64, lv64, trace = ref
    errs = []
    for k in range(5):
        ours, want = levels_got[k][1], lv64[k][1]
        assert ours.shape == want.shape, (k, ours.shape, want.shape)
        if k < 4:
            assert torch.equal(levels_got[k][0].cpu(), lv64[k][0]), f"level {k}: centres differ"
        errs.append(float((ours.double() - want).abs().max() / want.abs().max()))
    final = float((got.double() - out64).abs().max() / out64.abs().max())
    if geo is not None:
        fps = [t for t in trace if t[0] == "fps"]
        bqs = [t for t in trace if t[0] == "bq"]
        for k in range(4):
            assert torch.equal(geo[k][0].cpu(), fps[k][2].to(torch.int32)), f"level {k}: FPS indices"
            for i in range(2):
                assert torch.equal(geo[k][2][i].cpu(), bqs[2 * k + i][3].to(torch.int32)), f"level {k} scale {i}: ball query"
    print(f"{label}: per-level max err / scale {['%.2e' % e for e in errs]} final {final:.2e}")
    assert max(errs) <= tol and final <= tol, (label, errs, final)


@pytest.fixture(scope="module")
def c2_clouds():
    pts, _ = synthetic.make_point_clouds(64, 1024, seed=9, dup_fraction=0.25)
    return pts


@pytest.fixture(scope="module")
def c2_reference(enc_sd, c2_clouds):
    return _f64_reference(enc_sd, c2_clouds)


@pytest.mark.parametrize("mode", ["bf16x3", "bf16"])
def test_encoder_at_c2_matches_float64(enc_sd, c2_clouds, c2_reference, mode):
    """Pointnet2ClsMSG at 64 objects, every level and the output, against the float64 restatement (BatchNorm applied
    from the state dict, not folded); FPS and ball-query indices identical to the C restatement's"""
    enc = _encoder(enc_sd, mode)
    lv = []
    with torch.no_grad():
        got, geo = enc(c2_clouds.cuda(), return_geometry=True, levels=lv)
    _compare_levels(f"encoder C2 [{mode}]", got, lv, c2_reference, ENC_TOL[mode], geo=geo)


@pytest.fixture(scope="module")
def c5_clouds():
    pts, _ = synthetic.make_point_clouds(1024, 1024, seed=13, dup_fraction=0.25)
    return pts


@pytest.mark.parametrize("mode", ["bf16x3", "bf16"])
def test_encoder_batch_invariance_at_1024_objects(enc_sd, c5_clouds, mode):
    """An object's features do not depend on its position, on the batch size or on the other objects: 1024 clouds in
    one pass (the wide GEMM grids, tens to hundreds of tiles per fused-kernel CTA) against the same objects in a
    batch of 8 and in a permuted batch of 1024, bit for bit; a 64-object subset against float64"""
    enc = _encoder(enc_sd, mode)
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
    _compare_levels(f"encoder 1024-object pass, 64-object subset [{mode}]", full[sub.cuda()], lv_sub, ref, ENC_TOL[mode])

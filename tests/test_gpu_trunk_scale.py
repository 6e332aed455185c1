"""GPU: the score / energy trunk against float64 at production batch sizes, in every evaluator shape and operand mode;
and the multi-tile sampler kernels' tile loops checked bit for bit by tile replication.

The direct trunk checks elsewhere run 250-350 rows (2-3 tiles of 128) against po.Trunk (float32) with a tolerance
relative to the batch maximum.  Here the trunk runs what C2 (3200 rows, 25 tiles), the 32 / 33-tile shape switch,
a 1024-object shard (51 200 rows, 400 tiles) and C5 (409 600 rows, 3200 tiles) run, against the float64 restatement
po.trunk_f64, per element.

Per-element bound: |got - want| <= kappa * u * S, S the float64 chain on absolute values (trunk_f64).  u is the unit
roundoff of the operands: 2^-8 bf16, 2^-11 tf32, 2^-16 split-bf16, 2^-24 fp32 FFMA.  First-order error coefficients,
counted in u relative to S along the longest path (the ReLUs and the absolute chain carry a coefficient unchanged):

* Tensor-core layers (pose_encoder.0 9 -> 256 with x itself rounded, pose_encoder.2 256 -> 256, the heads' 256 pose
  columns -> 768).  bf16 and tf32 round both operands of every product once: 2u per layer, 6u for the three.  Split
  bf16 holds each operand as hi + lo (|w - hi - lo| <= 2^-16 |w|) and drops lo*lo (<= 2^-16 |a||b|): 3u per layer,
  9u for the three.
* fp32 parts common to every mode, in fp32 roundings (2^-24): the projection (project_kernel: 32 FMAs per lane, a
  5-level shuffle tree, the bias: 38); the t-branch (sincosf within 2 ulp; t_feat 64 FMAs + a shuffle + the bias, then
  128 FMAs: 196); the head pre-activation adds proj + tq to the accumulator (1); the head output layer (256 -> 3; the
  FFMA evaluator's chain is 4 FMAs, 5 shuffles, the two column halves, the bias: 11); the division by std + 1e-7 (1);
  energy's division by std, product and 6-term sum (7).  The tensor cores accumulate in fp32: at most 9 + 256 + 256
  sequential roundings for the three layers.
* FFMA (SimtEval): layer 1 is 9 FMAs, layer 2 256, the head 256 + 1: 522 along the pose path (the projection's 38 and
  the t-branch's 196 join at the head and are shorter), + 11 output layer + 7 energy = 540.  kappa = 560.
* bf16: 6 + (540 + 521) * 2^-16 = 6.02; tf32: 6 + 1061 * 2^-13 = 6.13.  kappa = 8 (the encoder's bf16 value).
* split: 9 + 1061 * 2^-8 = 13.1.  kappa = 16 (the encoder's split value).
* gp_trunk_project alone (FFMA, u = 2^-24): 38.  kappa = 40.

The worst case is far from what happens: S adds absolute values through four layers and is 1e3 - 1e4 times the
outputs, so this bound cannot see a wrong projection row or a missing split pass.  Every check therefore also applies
|got - want| <= kappa_R * u * R, R the root-sum-square scale of trunk_f64(rss=True): every sum y = sum_k t_k has
R_y^2 = sum_k (t_k^2 + R_tk^2), R zero for x, sin / cos and feat, masked by the float64 ReLUs.  Model: every rounding
is an independent error of mean 0 and variance <= eps^2 / 3 for |error| <= eps (uniform at worst).

* Tensor-core modes.  A product w a with both operands rounded carries w a (d_w + d_a): variance <= (2/3) u^2 (w a)^2;
  split adds the dropped lo*lo (<= u |w a|, variance <= u^2 / 9).  A layer's error is then
  sum_j w_j (a_j (d_wj + d_aj) + e_aj), and by induction over the layers Var(e) <= c u^2 R^2 with c = 2/3 (bf16,
  tf32) or 7/9 (split): std <= 0.82 u R and 0.88 u R.  The fp32 parts (projection, t-branch, output layer, the
  tensor cores' accumulation) add at most sqrt(260) * 2^-24 / u R: 0.06 u R in split mode, nothing in the others.
* FFMA.  A sequential chain acc_k = acc_(k-1) + t_k rounds every partial sum s_k: variance (u^2 / 3) sum_k s_k^2, and
  E[s_k^2] <= s_0^2 + sum_i t_i^2 for random-signed terms, so a chain of n adds a variance <= (n / 3) u^2 R_local^2.
  Summed over the chains (layer 1: 9, layer 2: 256, head: 257, output layer: 11, projection: 38, t-branch: 66 and
  128, sincosf: 2 ulp, energy: 7), c <= 260: std <= 16 u R.
* Tail factor 10 (a Gaussian needs 6 over the ~1e8 elements checked; rows where a few terms dominate a sum, as in
  the 9-input first layer, have heavier tails): kappa_R = 8 (bf16, tf32), 9 (split), 160 (FFMA); gp_trunk_project
  alone (chain 38: std 3.6 u R) 36.  An emulation of the roundings in float64 (bf16 / tf32 / split operands, the FFMA
  chains in float32 order) on 2000 rows gave max 2.0, 1.9, 0.8 and 13.2 u R.

Every case prints the evaluator, mode, rows, tiles, objects per tile and both ratios against their kappa.
Every output lands in the middle of a NaN-filled buffer: all outputs finite (no row or tile skipped), the spare
rows untouched.  test_negative_controls_against_the_bound asserts that the R bound rejects a wrong projection row and
a wrong t in every mode, and the bf16 output held to the split bound.

Tile replication (no float64 reference is affordable for a whole batch ODE at C5): 64 objects x 50 hypotheses = 25
tiles, repeated to 1024 and 8192 objects.  With batch step control every row sees the same h, so every tile equals its
copy in the first period bit for bit; period 25 is coprime to the 148-CTA grid stride, so copies run on different CTAs
after different predecessor tiles (a stale projection table, a skipped tile, a weight-ring or mbarrier-parity slip
would show).
"""
import zlib

import pytest
import torch

from genpose2_b200 import _lib, samplers, synthetic
from genpose2_b200.scorenet import EVAL_SHAPES, MLP_MODES, PoseScoreNet
from oracle import pose_oracle as po
from tests.util import pose_errors

pytestmark = pytest.mark.gpu

U = {"bf16": 2.0 ** -8, "tf32": 2.0 ** -11, "split": 2.0 ** -16, "ffma": 2.0 ** -24}
KAPPA = {"bf16": 8.0, "tf32": 8.0, "split": 16.0, "ffma": 560.0}          # worst case, in units of u S
KAPPA_R = {"bf16": 8.0, "tf32": 8.0, "split": 9.0, "ffma": 160.0}        # random-signed rounding, in units of u R
KAPPA_PROJECT, KAPPA_R_PROJECT = 40.0, 36.0
MLP = {"ffma": "fp32_ffma", "bf16": "bf16", "split": "fp32", "tf32": "tf32"}   # scorenet.MLP_MODES names
NPASS = {"bf16": 1, "tf32": 2, "split": 3}
# every (shape, mode) pair of with_evaluator's table (csrc/trunk.cu); FFMA has no shapes
EVALUATORS = [("cluster", "bf16"), ("cluster", "split"), ("cluster", "tf32"), ("solo", "bf16"), ("solo", "split"),
              ("solo", "tf32"), ("solo_smem_a", "bf16"), ("solo_smem_a", "split"), ("auto", "ffma")]
RT = 128          # rows of a tensor-core tile
RPO = 50          # hypotheses per object in production
SPARE = 5         # NaN rows on each side of an output
NAN = float("nan")
SEED = 100


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def sd():
    return synthetic.random_trunk_state_dict(SEED)


def _module(sd, mode, shape="auto"):
    net = PoseScoreNet(None, 0, pose_mode="rot_matrix", regression_head="Rx_Ry_and_T")
    net.load_state_dict({k[len("pose_score_net."):]: v for k, v in sd.items()})
    net = net.cuda().eval()
    net.mlp_mode, net.eval_shape = MLP[mode], shape
    return net


@pytest.fixture(scope="module")
def blobs(sd):
    net = _module(sd, "split")
    plain = net.packed().clone()
    net.mlp_mode = "tf32"
    return {"ffma": plain, "bf16": plain, "split": plain, "tf32": net.packed().clone()}


@pytest.fixture(scope="module")
def feats():
    g = torch.Generator().manual_seed(7)
    return torch.relu(torch.randn(8192, 1024, generator=g)).cuda()


@pytest.fixture(scope="module")
def proj(blobs, feats):
    """gp_trunk_project of all 8192 objects (the projection columns are fp32 in both blobs)"""
    out = torch.empty((feats.shape[0], 768), device="cuda")
    _lib.call("gp_trunk_project", _lib.ptr(blobs["split"]), _lib.ptr(feats), feats.shape[0], _lib.ptr(out))
    return out


def _ratio(got, want, scale, mode):
    return float(((got.double() - want).abs() / (U[mode] * scale)).max())


def _check(got, ref, mode, label, kappa=None, kappa_r=None):
    """both bounds: |got - want| <= kappa u S (worst case) and <= kappa_r u R (random-signed rounding); returns the
    ratio against R"""
    want, S, R = ref
    kappa = KAPPA[mode] if kappa is None else kappa
    kappa_r = KAPPA_R[mode] if kappa_r is None else kappa_r
    assert bool(torch.isfinite(got).all()), f"{label}: non-finite outputs (a row or tile was skipped)"
    rs, rr = _ratio(got, want, S, mode), _ratio(got, want, R, mode)
    print(f"{label}: max |got - want| / (u S) = {rs:.3g} (kappa {kappa:g}), / (u R) = {rr:.3g} (kappa_R {kappa_r:g})")
    assert rs <= kappa, (label, rs)
    assert rr <= kappa_r, (label, rr)
    return rr


def _nan_rows(n, cols):
    buf = torch.full((n + 2 * SPARE, cols), NAN, device="cuda")
    return buf, buf[SPARE:SPARE + n]


def _check_spare(buf, n):
    assert bool(buf[:SPARE].isnan().all()) and bool(buf[SPARE + n:].isnan().all()), "spare rows written"


# ------------------------------------------------------------------------------------------------------------------
# inputs, the float64 reference (cached per case: it does not depend on the evaluator) and the C ABI calls
# ------------------------------------------------------------------------------------------------------------------

def _poses(t, g):
    """[N,9] f32 at the magnitude the sampler feeds at t: a random rotation's 6D and a translation, + sigma(t) N(0,1)"""
    N = t.shape[0]
    q = torch.randn(N, 4, generator=g, device="cuda")
    R = po.quaternion_to_matrix(q / q.norm(dim=1, keepdim=True))
    clean = torch.cat([R[:, :, 0], R[:, :, 1], torch.randn(N, 3, generator=g, device="cuda") * 0.05], 1)
    return clean + po.ve_marginal_std(t)[:, None] * torch.randn(N, 9, generator=g, device="cuda")


def _times(pattern, N, rpo, g):
    """one t per call (a float), one per object ("object": runs end inside tiles) or one per row ("row")"""
    if isinstance(pattern, float):
        return torch.full((N,), pattern, device="cuda")
    n = -(-N // rpo) if pattern == "object" else N
    t = torch.rand(n, generator=g, device="cuda") * (1 - 1e-5) + 1e-5
    return t.repeat_interleave(rpo)[:N].contiguous() if pattern == "object" else t


_CASES = {}


def _case(sd, feats, N, rpo, pattern, kind):
    """(inputs, (want, S, R)) of a score / energy case"""
    key = (N, rpo, pattern, kind)
    if key not in _CASES:
        if len(_CASES) > 24:
            _CASES.clear()
        g = torch.Generator(device="cuda").manual_seed(zlib.crc32(repr(key).encode()))
        B = -(-N // rpo)
        t = _times(pattern, N, rpo, g)
        x = _poses(t, g)
        if kind == "score":
            ref = po.trunk_f64(sd, feats[:B], rpo, x, t, device="cuda", rss=True)
            inp = dict(x=x, t=t)
        else:
            centre = torch.randn(B, 3, generator=g, device="cuda") * 0.1 + torch.tensor([0.0, 0.0, 0.8], device="cuda")
            centre = centre.repeat_interleave(rpo, 0)[:N].contiguous()
            poses = x.double()
            poses[:, 6:] += centre.double()
            ref = po.trunk_f64(sd, feats[:B], rpo, poses, t, energy=centre, device="cuda", rss=True)
            inp = dict(poses=poses, centre=centre, t=t)
        _CASES[key] = (inp, ref)
    return _CASES[key]


def _mode_arg(shape, mode):
    return MLP_MODES[MLP[mode]] | (EVAL_SHAPES[shape] if mode != "ffma" else 0)


def _run(kind, blob, proj, inp, N, rpo, shape, mode):
    """gp_scorenet_eval / gp_energy through the C ABI (which takes a partial last object) into a NaN-padded buffer"""
    buf, out = _nan_rows(N, 9 if kind == "score" else 2)
    if kind == "score":
        _lib.call("gp_scorenet_eval", _lib.ptr(blob), _lib.ptr(proj), _lib.ptr(inp["x"]), _lib.ptr(inp["t"]), N, rpo,
                  _lib.ptr(out), _mode_arg(shape, mode))
    else:
        _lib.call("gp_energy", _lib.ptr(blob), _lib.ptr(proj), _lib.ptr(inp["poses"]), _lib.ptr(inp["centre"]),
                  _lib.ptr(inp["t"]), N, rpo, _lib.ptr(out), _mode_arg(shape, mode))
    _check_spare(buf, N)
    return out


def _tile_rows(mode, N, sms):
    """tile height: 128 rows on the tensor cores; launch_eval's FFMA rule: 16 rows up to 16 rows per SM, 32 above"""
    return RT if mode != "ffma" else (16 if N <= 16 * sms else 32)


def _evaluator(shape, mode, N, sms):
    rt = _tile_rows(mode, N, sms)
    if mode == "ffma":
        return f"SimtEval<{rt // 4}>"
    solo = shape in ("solo", "solo_smem_a") or (shape == "auto" and -(-N // RT) > 32)
    return f"TcEval<{NPASS[mode]}>" if not solo else f"TcSolo{'' if shape == 'solo_smem_a' else 'T'}<{NPASS[mode]}>"


def _tiles(N, rpo, rt):
    """begin_tile's arithmetic restated: first row, first and last object of every tile"""
    r0 = torch.arange(0, N, rt)
    return r0, r0 // rpo, (torch.clamp(r0 + rt, max=N) - 1) // rpo


def _label(kind, shape, mode, N, rpo, pattern, sms):
    rt = _tile_rows(mode, N, sms)
    _, first, last = _tiles(N, rpo, rt)
    span = last - first + 1
    return (f"{kind} {_evaluator(shape, mode, N, sms)} [{mode}] N={N} rpo={rpo} t={pattern}: {first.numel()} tiles of "
            f"{rt} rows, {int(span.min())}-{int(span.max())} objects per tile")


# ------------------------------------------------------------------------------------------------------------------
# 1. the projection
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("B", [1, 7, 8, 9, 64, 1024, 8192])
def test_project_matches_float64(sd, blobs, feats, B):
    """gp_trunk_project: 8-object blocks, a partial last block (7, 9), C2 and C5 object counts"""
    buf, out = _nan_rows(B, 768)
    _lib.call("gp_trunk_project", _lib.ptr(blobs["split"]), _lib.ptr(feats[:B]), B, _lib.ptr(out))
    _check_spare(buf, B)
    heads = [(sd[f"pose_score_net.fusion_tail_{h}.0.weight"].double().cuda(),
              sd[f"pose_score_net.fusion_tail_{h}.0.bias"].double().cuda()) for h in ("rot_x", "rot_y", "trans")]
    w = torch.cat([w0[:, :1024] for w0, _ in heads])
    b = torch.cat([b0 for _, b0 in heads])
    f = feats[:B].double()
    ref = (f @ w.t() + b, f.abs() @ w.abs().t() + b.abs(), ((f * f) @ (w * w).t() + b * b).sqrt())
    _check(out, ref, "ffma", f"gp_trunk_project B={B}: {-(-B // 8)} blocks of 8 objects", kappa=KAPPA_PROJECT,
           kappa_r=KAPPA_R_PROJECT)


# ------------------------------------------------------------------------------------------------------------------
# 2. every evaluator at production sizes
# ------------------------------------------------------------------------------------------------------------------

# C2; 32 and 33 tiles (the second with a one-row last tile); a 1024-object shard; C5
ROWS = [3200, 4096, 4097, 51200, 409600]


@pytest.mark.parametrize("shape,mode", EVALUATORS, ids=[f"{s}-{m}" for s, m in EVALUATORS])
@pytest.mark.parametrize("N", ROWS)
def test_eval_and_energy_match_float64(sd, blobs, feats, proj, sms, N, shape, mode):
    """gp_scorenet_eval and gp_energy, 50 rows per object, one t per call (1e-5, 0.55, 1), one per object and (up to
    4097 rows) one per row"""
    patterns = [1e-5, 0.55, 1.0, "object"] + (["row"] if N <= 4097 else [])
    if N == 409600 and mode != "ffma":
        assert -(-N // RT) == 3200
    for kind in ("score", "energy"):
        for pattern in patterns:
            inp, ref = _case(sd, feats, N, RPO, pattern, kind)
            got = _run(kind, blobs[mode], proj, inp, N, RPO, shape, mode)
            _check(got, ref, mode, _label(kind, shape, mode, N, RPO, pattern, sms))


# ------------------------------------------------------------------------------------------------------------------
# 3. the projection table's boundaries
# ------------------------------------------------------------------------------------------------------------------

SLOT_RPO = [1, 25, 26, 32, 33, 43, 127, 128, 129, 300]
TC_EVALUATORS = [e for e in EVALUATORS if e[1] != "ffma"]


@pytest.mark.parametrize("shape,mode", TC_EVALUATORS, ids=[f"{s}-{m}" for s, m in TC_EVALUATORS])
def test_projection_table_boundaries(sd, blobs, feats, proj, sms, shape, mode):
    """A tile copies the projection rows of its objects into shared memory when it spans at most MAX_SLOTS = 5
    (cluster, trunk_tc.cuh) or SLOTS = 4 (one CTA per tile, trunk_solo*.cuh) objects, and reads global memory
    otherwise; the cluster shape then also switches from local to global head columns.  At 5 objects the two shapes
    take different paths.  4097 rows (a one-row last tile), one t per object, every object count per tile from 1 to
    128, objects spanning tiles (rpo > 128) and a partial last object (4097 % rpo != 0 for every rpo > 1)."""
    N = 4097
    limit = 5 if shape == "cluster" else 4
    spans, head_cut, tail_cut = set(), False, False
    for rpo in SLOT_RPO:
        r0, first, last = _tiles(N, rpo, RT)
        span = last - first + 1
        end = torch.clamp(r0 + RT, max=N)
        spans |= set(span.tolist())
        head_cut |= bool((r0 % rpo != 0).any())                       # the tile's first object began in an earlier tile
        tail_cut |= bool(((end % rpo != 0) & (end < N)).any())        # its last object goes on in the next tile
        table = int((span <= limit).sum())
        for kind in ("score", "energy"):
            inp, ref = _case(sd, feats, N, rpo, "object", kind)
            got = _run(kind, blobs[mode], proj, inp, N, rpo, shape, mode)
            _check(got, ref, mode, _label(kind, shape, mode, N, rpo, "object", sms) +
                   f", {table} of {span.numel()} tiles from the table")
    assert {4, 5} <= spans and max(spans) >= 6, sorted(spans)
    assert head_cut and tail_cut
    assert all(N % rpo != 0 for rpo in SLOT_RPO if rpo > 1)


# ------------------------------------------------------------------------------------------------------------------
# 4. thresholds
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", ["bf16", "split", "tf32"])
def test_auto_shape_switches_at_33_tiles(sd, blobs, feats, proj, mode):
    """The default runs a 4-CTA cluster per tile up to 32 tiles and one CTA per tile above: at 4096 rows auto is
    forced cluster bit for bit, at 4097 forced solo (and the two shapes differ, so the comparison tells them apart)"""
    for N, same, other in ((4096, "cluster", "solo"), (4097, "solo", "cluster")):
        inp, _ = _case(sd, feats, N, RPO, "object", "score")
        auto = _run("score", blobs[mode], proj, inp, N, RPO, "auto", mode)
        assert torch.equal(auto, _run("score", blobs[mode], proj, inp, N, RPO, same, mode)), (N, same)
        assert not torch.equal(auto, _run("score", blobs[mode], proj, inp, N, RPO, other, mode)), (N, other)
        print(f"[{mode}] N={N} ({-(-N // RT)} tiles): auto == {same}, != {other}")


def test_ffma_tile_height_switch(sd, blobs, feats, proj, sms):
    """launch_eval's FFMA tile: 16 rows up to 16 rows per SM, 32 rows above"""
    for N in (16 * sms, 16 * sms + 1):
        for kind in ("score", "energy"):
            for pattern in ("object", "row"):
                inp, ref = _case(sd, feats, N, RPO, pattern, kind)
                got = _run(kind, blobs["ffma"], proj, inp, N, RPO, "auto", "ffma")
                _check(got, ref, "ffma", _label(kind, "auto", "ffma", N, RPO, pattern, sms))


# ------------------------------------------------------------------------------------------------------------------
# 5. the bound can fail
# ------------------------------------------------------------------------------------------------------------------

def test_negative_controls_against_the_bound(sd, blobs, feats, proj):
    """The check rejects, in every mode: (1) the reference with one row given the next object's projection row, (2) the
    reference with one object's t-run evaluated at the previous run's t; and (3) the bf16 output held to the
    split-bf16 bound.  Rejected means above kappa_R against the control's own R; the worst-case bound (units of S) is
    printed beside it: S being 1e3 - 1e4 times the outputs, it misses (1) and (3) in every mode and (2) in bf16 / tf32."""
    N = 4097
    inp, ref = _case(sd, feats, N, RPO, "object", "score")
    want, S, R = ref
    x, t = inp["x"], inp["t"]
    modes = ("split", "ffma", "bf16", "tf32")
    got = {m: _run("score", blobs[m], proj, inp, N, RPO, "auto", m) for m in modes}
    for m in modes:
        _check(got[m], ref, m, f"control baseline [{m}]")

    def rejected(name, rows, bad):
        bw, bS, bR = (a.clone() for a in ref)
        bw[rows], bS[rows], bR[rows] = bad
        for m in modes:
            rs, rr = _ratio(got[m], bw, bS, m), _ratio(got[m], bw, bR, m)
            print(f"{name} [{m}]: max |got - want| / (u R) = {rr:.3g} (kappa_R {KAPPA_R[m]:g}); / (u S) = {rs:.3g} "
                  f"(kappa {KAPPA[m]:g})")
            assert rr > KAPPA_R[m], (name, m, rr)

    # 1. row r of object o evaluated with object o + 1's projection row
    o = 40
    r = o * RPO + 7
    rejected(f"wrong proj row (row {r}: object {o + 1}'s)", slice(r, r + 1),
             po.trunk_f64(sd, feats[o + 1:o + 2], 1, x[r:r + 1], t[r:r + 1], device="cuda", rss=True))
    # 2. object o's run at the previous run's t: the smallest step between neighbouring objects' t of at least 0.05
    tobj = t[::RPO]
    dt = (tobj[1:] - tobj[:-1]).abs()
    o = int(torch.where(dt >= 0.05, dt, torch.full_like(dt, 2.0)).argmin()) + 1
    rows = slice(o * RPO, (o + 1) * RPO)
    rejected(f"wrong t (object {o}: t {float(tobj[o]):.4f} -> {float(tobj[o - 1]):.4f})", rows,
             po.trunk_f64(sd, feats[o:o + 1], RPO, x[rows], torch.full((RPO,), float(tobj[o - 1]), device="cuda"),
                          device="cuda", rss=True))
    # 3. a missing split pass: the bf16 output against the split-bf16 bound
    rr, rs = _ratio(got["bf16"], want, R, "split"), _ratio(got["bf16"], want, S, "split")
    print(f"bf16 output against the split bound: max |got - want| / (u_split R) = {rr:.3g} "
          f"(kappa_R {KAPPA_R['split']:g}); "
          f"/ (u_split S) = {rs:.3g} (kappa {KAPPA['split']:g})")
    assert rr > KAPPA_R["split"], rr


# ------------------------------------------------------------------------------------------------------------------
# 6. tile replication of the multi-tile sampler kernels
# ------------------------------------------------------------------------------------------------------------------

PERIOD_OBJ = 64
PERIOD_ROWS = PERIOD_OBJ * RPO            # 3200 rows = 25 tiles
T0, PC_STEPS, DENSE_STEPS = 0.55, 3, 5


@pytest.fixture(scope="module")
def period():
    """one period: 64 objects' features, centres (per row), ODE start noise, PC start and PC noise"""
    g = torch.Generator().manual_seed(31)
    feat = torch.relu(torch.randn(PERIOD_OBJ, 1024, generator=g))
    centre = torch.randn(PERIOD_OBJ, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 0.8])
    return dict(feat=feat.cuda(), centre=centre.repeat_interleave(RPO, 0).cuda(),
                noise=(torch.randn(PERIOD_ROWS, 9, generator=g) * po.ve_marginal_std(T0)).cuda(),
                pc_init=(torch.randn(PERIOD_ROWS, 9, generator=g) * po.ve_marginal_std(1.0)).cuda(),
                pc_noise=torch.randn(PC_STEPS, 2, PERIOD_ROWS, 9, generator=g).cuda())


def _sample(net, sampler, period, k):
    """the sampler on k copies of the period -> (outputs, nfev or None)"""
    rep = lambda a: a.repeat(k, *([1] * (a.dim() - 1))).contiguous()
    N = k * PERIOD_ROWS
    data = {"pts": torch.empty(N, 0), "pts_center": rep(period["centre"]), "_gp_pts_feat_obj": rep(period["feat"]),
            "_gp_rows_per_object": RPO}
    if sampler == "pc":
        xs, mean_x = samplers.cond_pc_sampler(net, data, None, None, num_steps=PC_STEPS, device="cuda", eps=1e-5,
                                              pose_mode="rot_matrix", init_x=rep(period["pc_init"]),
                                              noise=period["pc_noise"].repeat(1, 1, k, 1))
        return [xs, mean_x], None
    noise = rep(period["noise"])
    xs, x = samplers.cond_ode_sampler(net, data, lambda shape, T: noise, None, device="cuda", T=T0, eps=1e-5,
                                      pose_mode="rot_matrix", return_trajectory=False,
                                      num_steps=DENSE_STEPS if sampler == "ode_dense" else None)
    st = samplers.ode_stats()
    assert st["status"] == 0, st
    return ([xs, x] if sampler == "ode_dense" else [x]), st["nfev"]


_BASE = {}


@pytest.mark.parametrize("mode", ["split", "bf16"])
@pytest.mark.parametrize("shape,objects", [("auto", 1024), ("auto", 8192), ("cluster", 1024)])
@pytest.mark.parametrize("sampler", ["ode", "ode_dense", "pc"])
def test_tile_replication_is_bitwise(sd, period, sms, sampler, shape, objects, mode):
    """gp_scorenet_ode / _ode_dense / _pc on 16 or 128 copies of a 25-tile period: every tile equal to its copy in the
    first period bit for bit; the first period against a separate 64-object run in the same shape (north-star gates:
    the batch error norm / gradient norm sums its partials in another order)"""
    k = objects // PERIOD_OBJ
    tiles = k * 25
    forced = "solo" if (shape == "auto" and tiles > 32) else shape
    outs, nfev = _sample(_module(sd, mode, shape), sampler, period, k)
    per_cta = tiles / (sms if forced == "solo" else 33)      # the cooperative grid: one CTA per SM, or 33 clusters
    label = (f"{sampler} {objects} objects [{mode}] shape {shape} ({forced}): {tiles} tiles, ~{per_cta:.1f} per "
             f"{'CTA' if forced == 'solo' else 'cluster'}")
    for a in outs:
        assert bool(torch.isfinite(a).all()), label
        v = a.reshape(k, 25, RT, -1)
        same = (v == v[:1]).flatten(2).all(2)                  # [copy, tile]
        bad = torch.nonzero(~same).tolist()
        assert not bad, f"{label}: tiles (copy, tile) differing from the first period: {bad[:10]} ({len(bad)} in all)"
    # the 1024-object forced-cluster ode_dense case is the regression case of the cluster evaluator's t-branch barrier
    # (TcEval::stage_tq): without it, rank 0's dense-output writes let the peers' partials overwrite its t-branch
    # scratch; at ~12 tiles per cluster copies differed by up to 0.15 and reruns disagreed (not seen at 3 per cluster)
    key = (sampler, forced, mode)
    if key not in _BASE:
        _BASE[key] = _sample(_module(sd, mode, forced), sampler, period, 1)
    base, base_nfev = _BASE[key]
    rot, trans = pose_errors(outs[-1][:PERIOD_ROWS].cpu().numpy(), base[-1].cpu().numpy())
    print(f"{label}: all {k} copies bitwise equal; first period vs 64 objects ({forced}): rot {rot:.2e} rad, trans "
          f"{trans:.2e}" + ("" if nfev is None else f", nfev {nfev} vs {base_nfev}"))
    assert rot <= 1e-3 and trans <= 1e-4, (label, rot, trans)

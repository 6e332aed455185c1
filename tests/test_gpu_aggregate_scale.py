"""GPU: the three kernels of csrc/aggregate.cu (gp_scalenet, gp_aggregate, gp_pose_to_quat) against float64 at
production batch sizes, at every launch shape and at the edges of their limits; batch invariance of the aggregation at
C5; non-finite energies; a failed object carried through the whole pipeline.

Every output lands in the middle of a NaN-filled (labels: -7-filled) buffer: the outputs are all written and finite
where they should be, the spare rows untouched.  Each case prints its measured ratios against their bounds.

ScaleNet (gp_scalenet).  B <= SMs runs one object per block (OB 1), B < 8 SMs two (OB 2), larger batches eight (OB 8);
each OB gets another number of weight rows in flight per warp (dense_rows' NB).  C2 (64 objects) runs OB 1, a
1024-object shard OB 2, C5 on one GPU (8192) OB 8.  Against po.scalenet_f64 per element, u = 2^-24:

* worst case |got - want| <= kappa u S, S the float64 chain on absolute values.  A dense_rows output is a chain of
  4 ceil(K / 128) FMAs per lane, a 5-level shuffle tree and the bias add, every rounding at most u times a partial sum
  bounded by the layer's S; errors of the inputs travel through |W| into S unchanged.  K = 180: 8 + 5 + 1 = 14,
  K = 256: 14, K = 1280: 40 + 6 = 46, K = 256: 14; sincosf is within 2 ulp of sin / cos of the same float32 argument
  (2^k a is exact in float32).  Total 90: kappa = 100.
* random-signed |got - want| <= kappa_R u R, R the root-sum-square scale of po.scalenet_f64(rss=True) (defined as in
  po.trunk_f64, see tests/test_gpu_trunk_scale.py): a chain of n roundings adds a variance <= (n / 3) u^2 R^2, so the
  90 above give std <= 5.5 u R; with the tail factor 10 of the trunk test, kappa_R = 60.  Here S is thousands of
  times R (on a B200 the worst case used 0.002 of kappa, the R bound up to 7.4 of 60), so only the R bound can see a
  transposed axes read, a zeroed feature channel or an object reading its neighbour's features (the bug that staging
  OB objects per block can make): test_scalenet_negative_controls shows that it rejects each of them in each OB path.

Aggregation (gp_aggregate, one warp per object) against po.aggregate_pose(stable=True, float64=True):

* labels and the ranked poses (sorted_out) exactly: both are integer / gather results.  DBSCAN on distances within
  1e-12 of eps is a coin toss between two correct float64 summations: such objects are left out of the label check
  and counted (0 with these seeds).
* translation: the float64 mean of the same float64 rows, rounded to float32 once: within one float32 ulp.
* rotation, per element: the kernel's float64 eigenvector (cyclic Jacobi) and eigh's are exact eigenvectors of A + E
  with ||E|| <= c1 2^-52 ||A|| (forming A from the oriented quaternions, which the two compute in different orders,
  and each solver's backward error), so by Davis-Kahan they differ by <= 2 c1 2^-52 ||A|| / gap, and a rotation
  element (quadratic in q, |dM / dq| <= 4) by <= 8 c1 2^-52 ||A|| / gap; the float32 store adds <= 2^-25.  Bound
  2^-24 + KAPPA_ROT 2^-52 ||A|| / gap with KAPPA_ROT = 2048 (c1 = 256).
* Rayleigh-quotient deficit lambda_max - q^T A q, q read back from the float32 matrix (po.matrix_to_quaternion,
  normalised): it holds whatever the gap is.  An exact eigenvector of A + E has a deficit <= 2 ||E||; reading q back
  from a matrix rounded to float32 moves it by <= 4 * 2^-24 (each component is a sum of two elements over 2 |q_max|,
  |q_max| >= 1/2), which costs <= 16 * 2^-48 ||A||.  Bound ||A|| (KAPPA_DEF_32 2^-48 + KAPPA_DEF_64 2^-52) with 32 and
  1024.

gp_pose_to_quat: the same float64 operations as po.matrix_to_quaternion(po.get_rot_matrix(.)) up to order (the 6D
normalisation, the cross product); every branch divides by 2 max(|q_max|, 0.1) with |q_max| >= 1, and near a tie of
the argmax both branches give the quaternion (or its negative) to rounding.  min(|q - q'|, |q + q'|) <= KAPPA_Q 2^-52
per component, KAPPA_Q = 64.
"""
import ctypes

import numpy as np
import pytest
import torch

from genpose2_b200 import _lib, samplers, synthetic
from genpose2_b200.scalenet import ScaleNet
from oracle import pose_oracle as po

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
KAPPA_SCALE, KAPPA_R_SCALE = 100.0, 60.0
KAPPA_ROT, KAPPA_DEF_32, KAPPA_DEF_64, KAPPA_Q = 2048.0, 32.0, 1024.0, 64.0
SPARE = 5
NAN = float("nan")
EPS, MARGIN = 0.05, 1e-12


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _ob(B, sms):
    """gp_scalenet's launch rule"""
    return 1 if B <= sms else (2 if B < 8 * sms else 8)


# ------------------------------------------------------------------------------------------------------------------
# 1. ScaleNet
# ------------------------------------------------------------------------------------------------------------------

SCALE_B = {"1": lambda s: 1, "64": lambda s: 64, "SMs": lambda s: s, "SMs+1": lambda s: s + 1,
           "1024": lambda s: 1024, "8SMs-1": lambda s: 8 * s - 1, "8SMs": lambda s: 8 * s, "8192": lambda s: 8192,
           "8193": lambda s: 8193}


def _resolve(name, sms):
    return SCALE_B[name](sms)


@pytest.fixture(scope="module")
def scale():
    sd = synthetic.random_scalenet_state_dict(300)
    net = ScaleNet(1024, 0, 180).cuda()
    net.load_state_dict(sd)
    p, keep = net._params()
    g = torch.Generator().manual_seed(17)
    B = 8193
    feat = torch.relu(torch.randn(B, 1024, generator=g)).cuda()
    rot = torch.from_numpy(synthetic._random_rotations(np.random.default_rng(17), B)).float().cuda()
    return dict(sd=sd, p=p, keep=keep, feat=feat, rot=rot, refs={})


def _scale_ref(scale, B, axes=None, feat=None):
    if axes is None and feat is None:
        if B not in scale["refs"]:
            scale["refs"][B] = po.scalenet_f64(scale["sd"], scale["rot"][:B], scale["feat"][:B], rss=True, device="cuda")
        return scale["refs"][B]
    return po.scalenet_f64(scale["sd"], scale["rot"][:B] if axes is None else axes,
                           scale["feat"][:B] if feat is None else feat, rss=True, device="cuda")


def _scalenet(scale, B, layout):
    """gp_scalenet through the C ABI: contiguous [B,3,3] axes, or the [B,4,4] view the pipeline passes (its unused
    elements NaN: a misread would show)"""
    rot = scale["rot"][:B]
    if layout == "contiguous":
        axes, bs, rs = rot.contiguous(), 9, 3
    else:
        pose = torch.full((B, 4, 4), NAN, device="cuda")
        pose[:, :3, :3] = rot
        axes, bs, rs = pose[:, :3, :3], 16, 4
    buf = torch.full((B + 2 * SPARE, 3), NAN, device="cuda")
    out = buf[SPARE:SPARE + B]
    _lib.call("gp_scalenet", ctypes.byref(scale["p"]), _lib.ptr(axes), bs, rs, _lib.ptr(scale["feat"][:B]), B,
              _lib.ptr(out))
    assert bool(buf[:SPARE].isnan().all()) and bool(buf[SPARE + B:].isnan().all()), "spare rows written"
    return out


def _scale_ratios(got, ref):
    want, S, R = ref
    d = (got.double() - want).abs()
    return float((d / (U * S)).max()), float((d / (U * R)).max())


@pytest.mark.parametrize("layout", ["contiguous", "pose4x4"])
@pytest.mark.parametrize("name", list(SCALE_B))
def test_scalenet_matches_float64(scale, sms, name, layout):
    B = _resolve(name, sms)
    ob = _ob(B, sms)
    got = _scalenet(scale, B, layout)
    assert bool(torch.isfinite(got).all()), "non-finite lengths (an object was skipped)"
    rs, rr = _scale_ratios(got, _scale_ref(scale, B))
    blocks = -(-B // ob)
    print(f"gp_scalenet OB={ob} B={B} ({name}, {layout}): {blocks} blocks, last holds {B - (blocks - 1) * ob}: "
          f"max |got - want| / (u S) = {rs:.3g} (kappa {KAPPA_SCALE:g}), / (u R) = {rr:.3g} (kappa_R {KAPPA_R_SCALE:g})")
    assert rs <= KAPPA_SCALE and rr <= KAPPA_R_SCALE, (rs, rr)


def test_scalenet_negative_controls(scale, sms):
    """the R bound rejects, in each OB path: the axes transposed, one feature channel zeroed, object o given object
    o + 1's features (o in the middle of a block)"""
    paths = {1: sms, 2: 1024, 8: 8192}
    for ob, B in paths.items():
        assert _ob(B, sms) == ob, (ob, B)
        got = _scalenet(scale, B, "pose4x4")
        rot, feat = scale["rot"][:B], scale["feat"][:B]
        c = int((feat > 0).sum(0).argmax())
        zeroed = feat.clone()
        zeroed[:, c] = 0
        o = 5 * ob + ob // 2
        shifted = feat.clone()
        shifted[o] = feat[o + 1]
        controls = {"axes transposed": _scale_ref(scale, B, axes=rot.transpose(1, 2)),
                    f"feature channel {c} zeroed": _scale_ref(scale, B, feat=zeroed),
                    f"object {o} reads object {o + 1}'s features": _scale_ref(scale, B, feat=shifted)}
        for what, ref in controls.items():
            rs, rr = _scale_ratios(got, ref)
            print(f"control OB={ob} B={B}, {what}: max |got - want| / (u R) = {rr:.3g} (kappa_R {KAPPA_R_SCALE:g}); "
                  f"/ (u S) = {rs:.3g} (kappa {KAPPA_SCALE:g})")
            assert rr > KAPPA_R_SCALE, (ob, what, rr)


def test_scalenet_nan_axes_give_nan_length(scale, sms):
    """a NaN in the axes (the aggregated pose of a failed object) turns that object's length into NaN, like
    torch.relu, in each OB path; no other object changes"""
    for B in (sms, 1024, 8192):
        good = _scalenet(scale, B, "contiguous")
        o = 3 * _ob(B, sms) + 1
        saved = scale["rot"][o].clone()
        scale["rot"][o, 2, 1] = NAN
        try:
            bad = _scalenet(scale, B, "contiguous")
        finally:
            scale["rot"][o] = saved
        keep = torch.arange(B, device="cuda") != o
        assert bool(bad[o].isnan().all()), (B, bad[o])
        assert torch.equal(bad[keep], good[keep]), B


# ------------------------------------------------------------------------------------------------------------------
# 2. aggregation against float64
# ------------------------------------------------------------------------------------------------------------------

def _aggregate(poses, energy, retain, clustering, eps, min_samples):
    """gp_aggregate through the C ABI into -7 / NaN-filled buffers -> (pose [B,4,4], labels [B,retain], sorted)"""
    B, R = poses.shape[:2]
    poses = poses.to("cuda", torch.float64).contiguous()
    energy = energy.to("cuda", torch.float32).contiguous()
    pb = torch.full((B + 2 * SPARE, 4, 4), NAN, device="cuda")
    lb = torch.full((B + 2 * SPARE, retain), -7, dtype=torch.int32, device="cuda")
    sb = torch.full((B + 2 * SPARE, R, 9), NAN, dtype=torch.float64, device="cuda")
    out, labels, srt = pb[SPARE:SPARE + B], lb[SPARE:SPARE + B], sb[SPARE:SPARE + B]
    _lib.call("gp_aggregate", _lib.ptr(poses), _lib.ptr(energy), B, R, int(retain), int(bool(clustering)), float(eps),
              int(min_samples), _lib.ptr(out), _lib.ptr(labels), _lib.ptr(srt))
    for b in (pb, sb):
        assert bool(b[:SPARE].isnan().all()) and bool(b[SPARE + B:].isnan().all()), "spare rows written"
    assert bool((lb[:SPARE] == -7).all()) and bool((lb[SPARE + B:] == -7).all()), "spare labels written"
    assert bool((labels != -7).all()), "labels not written"
    return out, labels, srt


def _same_bits(a, b):
    """equal bit patterns where finite, NaN at the same places"""
    nan = a.isnan()
    if not torch.equal(nan, b.isnan()):
        return False
    return torch.equal(torch.where(nan, 0, a).view(torch.int64), torch.where(nan, 0, b).view(torch.int64))


def _check_aggregate(poses, energy, retain, clustering, eps, min_samples, label, got=None):
    """every check of the module docstring; returns (pose, labels, sorted) of the kernel"""
    poses, energy = poses.to(torch.float64).cpu(), energy.to(torch.float32).cpu()
    B = poses.shape[0]
    if got is None:
        got = _aggregate(poses, energy, retain, clustering, eps, min_samples)
    out, labels, srt = (t.cpu() for t in got)
    want, wl, info = po.aggregate_pose(poses, energy, retain_num=retain, clustering=bool(clustering),
                                       clustering_eps=eps, min_samples=min_samples, stable=True, float64=True)
    assert _same_bits(srt, po._sorted_stable(poses, energy)), f"{label}: sorted_out is not the stable-sorted gather"
    sure = ~(info["margin"] <= MARGIN)       # NaN distances (a NaN pose) are never neighbours: no coin toss
    assert np.array_equal(labels.numpy()[sure], wl[sure]), f"{label}: labels"
    np.testing.assert_array_equal(out[:, 3].numpy(), np.tile(np.float32([0, 0, 0, 1]), (B, 1)))
    g, w = out[:, :3].double(), want[:, :3]
    assert torch.equal(g.isnan(), w.isnan()), f"{label}: NaN pattern differs"
    fin = bool(torch.isfinite(w).all())
    ok = torch.isfinite(w).flatten(1).all(1)
    g, w, A, ev = g[ok], w[ok], info["A"][ok], info["evals"][ok]
    t_want = w[:, :, 3].numpy()
    t_ratio = float((np.abs(g[:, :, 3].numpy() - t_want) / np.spacing(np.abs(t_want.astype(np.float32)))).max()) \
        if len(w) else 0.0
    norm, gap = ev[:, 3], ev[:, 3] - ev[:, 2]
    rot_bound = 2.0 ** -24 + KAPPA_ROT * 2.0 ** -52 * norm / gap
    rot_ratio = float(((g[:, :, :3] - w[:, :, :3]).abs().flatten(1).amax(1) / rot_bound).max()) if len(w) else 0.0
    q = po.matrix_to_quaternion(g[:, :, :3].contiguous())
    q = q / q.norm(dim=1, keepdim=True)
    deficit = norm - torch.einsum("bi,bij,bj->b", q, A, q)
    def_ratio = float((deficit / (norm * (KAPPA_DEF_32 * 2.0 ** -48 + KAPPA_DEF_64 * 2.0 ** -52))).max()) \
        if len(w) else 0.0
    print(f"{label}: translation {t_ratio:.3g} ulp (1); rotation {rot_ratio:.3g} of 2^-24 + {KAPPA_ROT:g} 2^-52 "
          f"|A| / gap (1), min gap / |A| {float((gap / norm).min()) if len(w) else 0:.2g}; Rayleigh deficit "
          f"{def_ratio:.3g} of |A| ({KAPPA_DEF_32:g} 2^-48 + {KAPPA_DEF_64:g} 2^-52) (1); {int((~sure).sum())} of {B} "
          f"objects within {MARGIN:g} of eps left out of the label check" + ("" if fin else f"; {int((~ok).sum())} "
                                                                                                 "NaN objects"))
    assert t_ratio <= 1 and rot_ratio <= 1 and def_ratio <= 1, (label, t_ratio, rot_ratio, def_ratio)
    return got


_POSES = {}


def _cluster_poses(B, R):
    """thirds at 1, 4 and 12 degrees of jitter (one tight cluster / a second mode / no cluster to speak of), drawn at
    64 hypotheses and cut to R"""
    if B not in _POSES:
        n = [B // 3, B // 3, B - 2 * (B // 3)]
        _POSES[B] = torch.cat([synthetic.make_cluster_quaternion_poses(k, 64, seed=B + i, jitter_deg=j)
                               for i, (k, j) in enumerate(zip(n, (1.0, 4.0, 12.0)))])
    return _POSES[B][:, :R].contiguous()


def _energy(B, R, seed):
    return torch.randn(B, R, 2, generator=torch.Generator().manual_seed(seed))


AGG_CONFIGS = [(50, 20, True), (64, 32, True), (64, 64, False), (33, 13, True), (2, 1, False)]


@pytest.mark.parametrize("R,retain,clustering", AGG_CONFIGS, ids=[f"R{r}-k{k}-{'on' if c else 'off'}"
                                                                  for r, k, c in AGG_CONFIGS])
@pytest.mark.parametrize("B", [64, 1024])
def test_aggregate_matches_float64(B, R, retain, clustering):
    """C2 and a 1024-object shard; R = 64 (the limit), retain 32 with clustering (full 32-bit neighbourhood masks),
    retain 64 without (the upper half of the member mask), R < 32 (idle lanes), a ragged last block for 33 x 13"""
    min_samples = int(0.1667 * retain)
    if clustering:
        assert min_samples >= 1
    _check_aggregate(_cluster_poses(B, R), _energy(B, R, B + R), retain, clustering, EPS, max(min_samples, 1),
                     f"gp_aggregate B={B} R={R} retain={retain} clustering={int(clustering)} "
                     f"min_samples={max(min_samples, 1)}")


def test_aggregate_retain_one_and_min_samples_one():
    """aggregation._run (the Python entry point): one retained hypothesis with clustering, min_samples = 1 at
    retain 20, 63 objects (a ragged last block)"""
    from genpose2_b200.aggregation import _run
    B = 63
    poses, energy = _cluster_poses(64, 50)[:B], _energy(B, 50, 3)
    for retain in (1, 20):
        out, labels, srt = _run(poses.cuda(), energy.cuda(), retain, True, EPS, 1, want_sorted=True, want_labels=True)
        _check_aggregate(poses, energy, retain, True, EPS, 1, f"_run retain={retain} min_samples=1",
                         got=(out, labels, srt))
        if retain == 1:
            assert bool((labels == 0).all())


def _quat_to_6d(q):
    M = po.quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True))
    return torch.cat([M[..., :, 0], M[..., :, 1]], -1)


def _jitter(q, deg, g):
    """q (wxyz, [..., 4]) times a random rotation of about `deg` degrees"""
    ax = torch.randn(q.shape[:-1] + (3,), generator=g, dtype=torch.float64)
    ax = ax / ax.norm(dim=-1, keepdim=True)
    h = np.deg2rad(deg) * torch.randn(q.shape[:-1] + (1,), generator=g, dtype=torch.float64) / 2
    d = torch.cat([torch.cos(h), torch.sin(h) * ax], -1)
    w1, x1, y1, z1 = d.unbind(-1)
    w2, x2, y2, z2 = q.unbind(-1)
    return torch.stack([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                        w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2], -1)


def _with_trans(rot6, g):
    return torch.cat([rot6, torch.randn(rot6.shape[:-1] + (3,), generator=g, dtype=torch.float64) * 0.01 + 0.8], -1)


def test_aggregate_hand_built_cases():
    g = torch.Generator().manual_seed(21)
    B, R, retain = 12, 50, 20
    energy = -torch.arange(R, dtype=torch.float32).repeat(B, 1).unsqueeze(-1).repeat(1, 1, 2)   # rank = index
    # two clusters of 10 among the 20 retained, interleaved: the label tie goes to the first label (A)
    qa, qb = torch.randn(B, 1, 4, generator=g, dtype=torch.float64), torch.randn(B, 1, 4, generator=g, dtype=torch.float64)
    which = (torch.arange(R) % 2 == 1).reshape(1, R, 1)
    q = torch.where(which, qb, qa).expand(B, R, 4)
    q = torch.where(torch.arange(R).reshape(1, R, 1) < retain, _jitter(q, 0.5, g), torch.randn(B, R, 4, generator=g,
                                                                                               dtype=torch.float64))
    poses = _with_trans(_quat_to_6d(q), g)
    out, labels, _ = _check_aggregate(poses, energy, retain, True, EPS, 3, "two equal clusters")
    lab = labels.cpu()
    assert bool((lab[:, 0::2] == 0).all()) and bool((lab[:, 1::2] == 1).all()), lab
    ra = po.quaternion_to_matrix(qa[:, 0] / qa[:, 0].norm(dim=1, keepdim=True))
    assert float((out[:, :3, :3].cpu().double() - ra).abs().max()) < 0.05   # cluster A's average, not B's
    # all points noise: min_samples above any neighbourhood
    _, labels, _ = _check_aggregate(poses, energy, retain, True, EPS, retain + 1, "all noise (min_samples = 21)")
    assert bool((labels == -1).all())
    # identical hypotheses
    same = poses[:, :1].expand(B, R, 9).contiguous()
    out, labels, _ = _check_aggregate(same, _energy(B, R, 4), retain, True, EPS, 3, "identical hypotheses")
    assert bool((labels.cpu() == 0).all())
    # rotations near 180 degrees (w ~ 0: rot6d_to_quat takes branches 1-3), about random and coordinate axes
    axes = torch.cat([torch.eye(3, dtype=torch.float64), torch.randn(B - 3, 3, generator=g, dtype=torch.float64)])
    axes = axes / axes.norm(dim=1, keepdim=True)
    off = torch.tensor([0, 1e-12, 1e-6, 1e-3] * 3, dtype=torch.float64)[:, None]   # distance of the angle from pi
    base = torch.cat([torch.sin(off / 2), torch.cos(off / 2) * axes], -1)
    for deg, (ms, clus) in ((0.2, (3, True)), (2.0, (3, True)), (2.0, (1, False))):
        q = _jitter(base[:, None].expand(B, R, 4), deg, g)
        poses = _with_trans(_quat_to_6d(q), g)
        _check_aggregate(poses, _energy(B, R, int(deg * 10)), retain, clus, EPS, ms,
                         f"near 180 degrees, jitter {deg} deg, clustering={int(clus)}")
        qk = torch.empty(B * R, 7, dtype=torch.float64, device="cuda")
        _lib.call("gp_pose_to_quat", _lib.ptr(poses.reshape(-1, 9).cuda().contiguous()), B * R, _lib.ptr(qk))
        assert int((qk[:, 0].abs() < qk[:, 1:4].abs().amax(1)).sum()) > 0      # the w ~ 0 branches were taken


# ------------------------------------------------------------------------------------------------------------------
# 3. batch invariance at C5
# ------------------------------------------------------------------------------------------------------------------

def test_aggregate_batch_invariance_c5():
    """8192 objects (C5 on one GPU, 2048 blocks): each object equal bit for bit to its result alone, in C2-sized
    batches of 64, after a permutation, and in batches of 8191 / 8190 / 8189 objects (B % 4 != 0)"""
    B, R, retain = 8192, 50, 20
    base = _cluster_poses(1024, R)
    g = torch.Generator().manual_seed(8)
    poses = base.repeat(8, 1, 1)
    poses[:, :, 6:] += torch.randn(B, 1, 3, generator=g, dtype=torch.float64) * 0.05
    energy = torch.randn(B, R, 2, generator=g)          # another ranking for every copy
    args = (retain, True, EPS, 3)
    full = _aggregate(poses, energy, *args)

    def same(part, idx, what):
        for a, b, name in zip(part, full, ("pose", "labels", "sorted")):
            assert _same_bits(a.double(), b[idx].double()), f"{what}: {name}"

    for lo in range(0, B, 64):
        same(_aggregate(poses[lo:lo + 64], energy[lo:lo + 64], *args), slice(lo, lo + 64), f"batch of 64 at {lo}")
    perm = torch.from_numpy(np.random.default_rng(2).permutation(B))
    same(_aggregate(poses[perm], energy[perm], *args), perm.cuda(), "permuted")
    for n in (8191, 8190, 8189):
        same(_aggregate(poses[:n], energy[:n], *args), slice(0, n), f"first {n}")
    alone = [0, 1, 3, 4, 4095, 8188, 8189, 8190, 8191] + np.random.default_rng(3).choice(B, 23, replace=False).tolist()
    for b in alone:
        same(_aggregate(poses[b:b + 1], energy[b:b + 1], *args), slice(b, b + 1), f"object {b} alone")
    print(f"C5 batch invariance: 8192 objects, {full[1].eq(-1).sum().item()} noise labels, {len(alone)} objects alone, "
          f"128 batches of 64, a permutation, 3 ragged prefixes: bit-identical")


# ------------------------------------------------------------------------------------------------------------------
# 4. non-finite energies and NaN poses
# ------------------------------------------------------------------------------------------------------------------

def _nonfinite_energies(B, R, g):
    """one pattern per object, in turn: ties, +-0 only, +-inf among finite, NaN in some rows, NaN in every row, NaN in
    channel 0 only, NaN in channel 1 only, NaN / inf / ties mixed"""
    e = torch.randn(B, R, 2, generator=g)
    pick = lambda k: torch.randperm(R, generator=g)[:k]
    for b in range(B):
        kind = b % 8
        if kind == 0:
            e[b] = torch.round(e[b] * 2) / 2
        elif kind == 1:
            e[b] = torch.where(torch.rand(R, 2, generator=g) < 0.5, -0.0, 0.0)
        elif kind == 2:
            e[b, pick(5)] = float("inf")
            e[b, pick(5)] = -float("inf")
        elif kind == 3:
            e[b, pick(7)] = NAN
        elif kind == 4:
            e[b] = NAN
        elif kind == 5:
            e[b, pick(9), 0] = NAN
        elif kind == 6:
            e[b, pick(9), 1] = NAN
        else:
            e[b] = torch.round(e[b])
            e[b, pick(4)] = NAN
            e[b, pick(4)] = float("inf")
            e[b, pick(4), 1] = -float("inf")
    return e


@pytest.mark.parametrize("R,retain,clustering", [(50, 20, True), (64, 32, True), (64, 64, False)])
def test_aggregate_nonfinite_energies(R, retain, clustering):
    """the ranks follow torch.sort(descending=True, stable=True): NaN first (in index order), then +inf, ..., -inf,
    +-0 and every other tie in index order.  The poses are finite, so a NaN energy only moves its row to the front:
    it is retained and the result stays finite"""
    B = 64
    g = torch.Generator().manual_seed(R + retain)
    energy = _nonfinite_energies(B, R, g)
    poses = _cluster_poses(64, R)
    out, _, srt = _check_aggregate(poses, energy, retain, clustering, EPS, max(int(0.1667 * retain), 1),
                                   f"non-finite energies R={R} retain={retain} clustering={int(clustering)}")
    assert bool(torch.isfinite(out).all())
    nan_first = energy[:, :, 0].isnan()
    for b in range(B):
        k = int(nan_first[b].sum())
        if k:
            rows = torch.nonzero(nan_first[b])[:, 0]
            assert torch.equal(srt[b, :k, :6].cpu(), poses[b, rows, :6]), b   # NaN rows first, in index order


def test_aggregate_nan_poses_poison_only_their_object():
    """What a failed integration hands to the aggregation: NaN in all nine columns of some rows, so NaN energies.
    Object 5 has every row NaN (the failed object of object-mode step control), object 9 three rows; both come out NaN
    in rows 0-2 with [0, 0, 0, 1] in row 3 and labels -1.  Object 12 has a NaN pose whose finite energy is the lowest:
    it is not retained and the result is finite.  Every other object equals the healthy batch bit for bit."""
    B, R, retain = 16, 50, 20
    poses = _cluster_poses(64, R)[:B].clone()
    energy = _energy(B, R, 12)
    for clustering, ms in ((True, 3), (False, 1)):
        healthy = _aggregate(poses, energy, retain, clustering, EPS, ms)
        bp, be = poses.clone(), energy.clone()
        bp[5], be[5] = NAN, NAN
        bp[9, [2, 17, 40]], be[9, [2, 17, 40]] = NAN, NAN
        low = int(energy[12, :, 0].argmin())
        bp[12, low, :6] = NAN
        be[12, low, 0] = -1e30
        got = _check_aggregate(bp, be, retain, clustering, EPS, ms, f"NaN poses, clustering={int(clustering)}")
        out, labels, _ = (t.cpu() for t in got)
        for b in (5, 9):
            assert bool(out[b, :3].isnan().all()) and out[b, 3].tolist() == [0, 0, 0, 1] and bool((labels[b] == -1).all())
        assert bool(torch.isfinite(out[12]).all())
        keep = [b for b in range(B) if b not in (5, 9, 12)]
        for a, h in zip(got, healthy):
            assert _same_bits(a[keep].double(), h[keep].double())
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------------
# 5. gp_pose_to_quat
# ------------------------------------------------------------------------------------------------------------------

def _branch_rows(g):
    """quaternions whose argmax branch is each of w, x, y, z; two-, three- and four-way ties of |components| with
    offsets from 0 to 1e-6; unnormalised, non-orthogonal 6D"""
    rows = []
    for i in range(4):
        q = torch.randn(20000, 4, generator=g, dtype=torch.float64) * 0.3
        q[:, i] = torch.sign(torch.randn(20000, generator=g, dtype=torch.float64)) * (1 + torch.rand(20000, generator=g))
        rows.append(q)
    n = 8000
    for k in (2, 3, 4):
        for off in (0.0, 1e-15, 1e-12, 1e-9, 1e-6):
            q = torch.randn(n, 4, generator=g, dtype=torch.float64) * 0.2
            idx = torch.rand(n, 4, generator=g).argsort(1)[:, :k]
            q.scatter_(1, idx, torch.sign(torch.randn(n, k, generator=g, dtype=torch.float64)))
            q[torch.arange(n), idx[:, 0]] *= 1 + off
            rows.append(q)
    return _quat_to_6d(torch.cat(rows))


def test_pose_to_quat_matches_float64():
    """409 600 rows (C5 x 50): random rotations plus rows for every argmax branch and near ties between branches; a
    quarter of the 6D rows unnormalised and non-orthogonal (the kernel Gram-Schmidts them like get_rot_matrix)"""
    N = 409600
    g = torch.Generator().manual_seed(40)
    special = _branch_rows(g)
    rest = _quat_to_6d(torch.randn(N - special.shape[0], 4, generator=g, dtype=torch.float64))
    rot6 = torch.cat([special, rest])[torch.randperm(N, generator=g)]
    skew = torch.rand(N, generator=g) < 0.25
    scale = 0.5 + torch.rand(N, 2, generator=g, dtype=torch.float64)
    rot6[skew, :3] *= scale[skew, :1]
    rot6[skew, 3:] = rot6[skew, 3:] * scale[skew, 1:] + 0.3 * rot6[skew, :3]
    poses = _with_trans(rot6, g).cuda().contiguous()
    buf = torch.full((N + 2 * SPARE, 7), NAN, dtype=torch.float64, device="cuda")
    out = buf[SPARE:SPARE + N]
    _lib.call("gp_pose_to_quat", _lib.ptr(poses), N, _lib.ptr(out))
    assert bool(buf[:SPARE].isnan().all()) and bool(buf[SPARE + N:].isnan().all()), "spare rows written"
    assert bool(torch.isfinite(out).all())
    assert torch.equal(out[:, 4:], poses[:, 6:]), "translations are not copied bit for bit"
    want = po.matrix_to_quaternion(po.get_rot_matrix(poses[:, :6]))
    d = torch.minimum((out[:, :4] - want).abs().amax(1), (out[:, :4] + want).abs().amax(1))
    ratio = float(d.max() / (KAPPA_Q * 2.0 ** -52))
    flips = int(((out[:, :4] - want).abs().amax(1) > (out[:, :4] + want).abs().amax(1)).sum())
    branch = want.abs().argmax(1).bincount(minlength=4).tolist()
    print(f"gp_pose_to_quat N={N}: max min(|q - q'|, |q + q'|) = {ratio:.3g} of {KAPPA_Q:g} 2^-52 (1); rows per "
          f"largest component {branch}; {flips} rows of the opposite sign (another branch at a tie)")
    assert ratio <= 1, ratio
    assert min(branch) > 20000


# ------------------------------------------------------------------------------------------------------------------
# 6. a failed object through the whole pipeline
# ------------------------------------------------------------------------------------------------------------------

def test_pipeline_failed_object_poisons_only_its_results():
    """PosePipeline(step_control="object") with a NaN in object 2's prior noise: its integration fails (status -1),
    its poses are NaN, and energy, aggregation and ScaleNet carry that to NaN pose rows 0-2 and a NaN length for that
    object alone; every other object is bit-identical to the healthy step, and a healthy step afterwards is too"""
    from genpose2_b200.pipeline import PosePipeline
    pipe = PosePipeline(device="cuda", step_control="object").load_synthetic_weights()
    B, R, T0, bad_obj = 8, 50, 0.55, 2
    pts, center = synthetic.make_point_clouds(B, 1024, seed=61)
    noise = po.ve_prior((B * R, 9), T=T0).float()
    bad = noise.clone()
    bad[bad_obj * R + 5, 4] = NAN
    cur = {}
    pipe.score_agent.net.prior_fn = lambda shape, T=1.0: cur["noise"].clone()

    def step(n):
        cur["noise"] = n
        return pipe({"pts": pts.cuda(), "pts_center": center.cuda()}, repeat_num=R, T0=T0)

    ok_pose, ok_len = step(noise)
    assert samplers.ode_stats()["status"] == 0
    pose, length = step(bad)
    with pytest.raises(RuntimeError, match="status -1"):
        samplers.ode_stats()
    st = samplers.ode_stats()
    assert [int(s) for s in st["obj_status"]] == [0] * bad_obj + [-1] + [0] * (B - bad_obj - 1), st["obj_status"]
    torch.cuda.synchronize()
    assert bool(pose[bad_obj, :3].isnan().all()) and pose[bad_obj, 3].tolist() == [0, 0, 0, 1]
    assert bool(length[bad_obj].isnan().all()), length[bad_obj]
    keep = [b for b in range(B) if b != bad_obj]
    assert torch.equal(pose[keep], ok_pose[keep]) and torch.equal(length[keep], ok_len[keep])
    again_pose, again_len = step(noise)
    assert samplers.ode_stats()["status"] == 0
    assert torch.equal(again_pose, ok_pose) and torch.equal(again_len, ok_len)
    print(f"failed object {bad_obj}: NaN pose rows 0-2 and length; {B - 1} other objects bit-identical; "
          f"obj_status {st['obj_status'].tolist()}")

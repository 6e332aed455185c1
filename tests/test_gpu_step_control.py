"""GPU: per-object RK45 step control (cond_ode_sampler(..., step_control="object"), gp_scorenet_ode_objects).

An object's result must be a function of its own features, noise and the weights only: "object" mode on a batch is
bit-identical to one-object "batch" calls (same evaluator shape), under permutation, sharding and embedding in a larger
batch; it agrees with the per-object CPU oracle at the north-star gates with equal step counts; a failed object poisons
only its own rows.  The default ("batch") is untouched."""
import functools

import numpy as np
import pytest
import torch

from genpose2_b200 import samplers, synthetic
from oracle import pose_oracle as po
from tests.test_gpu_sampler import BF16_ROT_TOL, BF16_TRANS_TOL, ROT_TOL, TRANS_TOL, make_net
from tests.util import geodesic_6d, pose_errors, rep

pytestmark = pytest.mark.gpu

MODES = ["fp32", "bf16", "fp32_ffma"]


def inputs(B, R, T0, seed, with_init=False):
    g = torch.Generator().manual_seed(seed)
    feat = torch.relu(torch.randn(B, 1024, generator=g))
    center = torch.randn(B, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 0.8])
    noise = torch.randn(B * R, 9, generator=g) * po.ve_marginal_std(T0)
    init = None
    if with_init:
        init = torch.randn(B, 9, generator=g)
        init[:, 6:] *= 0.05
    return feat, center, noise, init


def run(net, feat, center, noise, R, T0, step_control="batch", init=None, num_steps=None, **kw):
    B = feat.shape[0]
    data = {"pts": torch.zeros(B * R, 1, 3), "pts_center": rep(center, R).cuda(), "_gp_pts_feat_obj": feat.cuda(),
            "_gp_rows_per_object": R}
    extra = {} if step_control is None else {"step_control": step_control}
    xs, x = samplers.cond_ode_sampler(net, data, lambda shape, T: noise.clone(), net.sde_fn, device="cuda", T=T0,
                                      pose_mode="rot_matrix", num_steps=num_steps, return_trajectory=False,
                                      init_x=None if init is None else rep(init, R).cuda(), **extra, **kw)
    return xs.cpu().numpy(), x.cpu().numpy(), samplers.ode_stats()


def rows(b, R):
    return slice(b * R, (b + 1) * R)


def shaped_net(mlp_mode, shape):
    net = make_net(100, mlp_mode=mlp_mode)
    net.pose_score_net.eval_shape = shape
    return net


@pytest.mark.parametrize("mlp_mode,shape", [("fp32", "cluster"), ("fp32", "solo"), ("bf16", "cluster"),
                                            ("bf16", "solo"), ("fp32_ffma", "auto")])
def test_object_mode_is_batch_invariant(mlp_mode, shape):
    net = shaped_net(mlp_mode, shape)
    B, R, T0 = 13, 50, 0.55
    feat, center, noise, _ = inputs(B, R, T0, seed=1)
    _, x, st = run(net, feat, center, noise, R, T0, "object")
    assert st["status"] == 0 and len(st["obj_nfev"]) == B
    assert st["nfev"] == st["obj_nfev"].max() and st["accepted"] == st["obj_accepted"].sum()
    assert st["rejected"] == st["obj_rejected"].sum() and (st["obj_status"] == 0).all()
    # 13 one-object batch calls with the same noise rows
    for b in range(B):
        _, xb, sb = run(net, feat[b:b + 1], center[b:b + 1], noise[rows(b, R)], R, T0, "batch")
        assert np.array_equal(x[rows(b, R)], xb), b
        assert (st["obj_nfev"][b], st["obj_accepted"][b], st["obj_rejected"][b]) == \
            (sb["nfev"], sb["accepted"], sb["rejected"]), b
    print(f"object [{mlp_mode}/{shape}]: nfev per object {st['obj_nfev'].min()}..{st['obj_nfev'].max()}")
    # permuted
    perm = np.random.default_rng(0).permutation(B)
    nz = noise.view(B, R, 9)
    _, xp, _ = run(net, feat[perm], center[perm], nz[perm].reshape(B * R, 9), R, T0, "object")
    assert np.array_equal(xp.reshape(B, R, 9), x.reshape(B, R, 9)[perm])
    # two shards
    _, x1, _ = run(net, feat[:6], center[:6], noise[:6 * R], R, T0, "object")
    _, x2, _ = run(net, feat[6:], center[6:], noise[6 * R:], R, T0, "object")
    assert np.array_equal(np.concatenate([x1, x2]), x)
    # embedded in a 200-object batch
    fe, ce, ne, _ = inputs(200, R, T0, seed=2)
    at = np.sort(np.random.default_rng(1).choice(200, B, replace=False))
    fe[at], ce[at] = feat, center
    ne = ne.view(200, R, 9)
    ne[at] = nz
    _, xe, se = run(net, fe, ce, ne.reshape(200 * R, 9), R, T0, "object")
    assert np.array_equal(xe.reshape(200, R, 9)[at], x.reshape(B, R, 9))
    assert np.array_equal(se["obj_nfev"][at], st["obj_nfev"])


@pytest.mark.parametrize("mlp_mode", ["fp32", "bf16"])
def test_object_mode_across_automatic_shape_change(mlp_mode):
    """13 objects run as clusters by default, 200 objects one CTA per object: the two shapes sum the head columns in
    different orders, so the same objects agree at the solo-vs-cluster gate of test_gpu_solo, not bit for bit.  Each
    object has its own controller, so an error norm that sits at an accept / reject threshold in one shape can cost one
    more attempt (6 evaluations) in the other: 1 of these 13 objects does (152 vs 158 nfev on a B200)."""
    net = shaped_net(mlp_mode, "auto")
    B, R, T0 = 13, 50, 0.55
    feat, center, noise, _ = inputs(B, R, T0, seed=1)
    _, x, st = run(net, feat, center, noise, R, T0, "object")
    fe, ce, ne, _ = inputs(200, R, T0, seed=2)
    fe[:B], ce[:B] = feat, center
    ne[:B * R] = noise
    _, xe, se = run(net, fe, ce, ne, R, T0, "object")
    a, b = x, xe[:B * R]
    rot = geodesic_6d(a[:, :6], b[:, :6])
    trans = np.linalg.norm(a[:, 6:] - b[:, 6:], axis=1)
    print(f"cluster vs solo [{mlp_mode}]: rot max {rot.max():.3e} trans max {trans.max():.3e}")
    if mlp_mode == "fp32":
        dn = np.abs(st["obj_nfev"] - se["obj_nfev"][:B])
        print(f"   nfev differs on {int((dn > 0).sum())} of {B} objects")
        assert dn.max() <= 6 and (dn == 0).sum() >= B - 2
        assert np.abs(st["obj_accepted"] - se["obj_accepted"][:B]).max() <= 1
        assert rot.max() <= ROT_TOL and trans.max() <= TRANS_TOL
    else:
        assert rot.max() <= BF16_ROT_TOL and trans.max() <= BF16_TRANS_TOL


@functools.lru_cache(maxsize=None)
def oracle(B, R, T0, with_init, num_steps=None, seed=5):
    """per-object CPU oracle: po.cond_ode_sampler on each object alone -> (xs, x, nfev, accepted, rejected)"""
    feat, center, noise, init = inputs(B, R, T0, seed, with_init)
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(100))
    out = []
    for b in range(B):
        xs, x, s = po.cond_ode_sampler(trunk, rep(feat[b:b + 1], R), rep(center[b:b + 1], R), noise[rows(b, R)],
                                       init_x=None if init is None else rep(init[b:b + 1], R), T=T0,
                                       num_steps=num_steps)
        out.append((xs.numpy(), x.numpy(), s["nfev"], s["n_accepted"], s["n_rejected"]))
    return out


@pytest.mark.parametrize("mlp_mode", MODES)
@pytest.mark.parametrize("B,R,T0,with_init", [(5, 7, 0.55, False), (3, 50, 0.55, False), (2, 128, 0.55, False),
                                              (3, 50, 0.25, True), (2, 128, 0.25, True)])
def test_object_mode_matches_per_object_oracle(mlp_mode, B, R, T0, with_init):
    want = oracle(B, R, T0, with_init)
    feat, center, noise, init = inputs(B, R, T0, 5, with_init)
    net = make_net(100, mlp_mode=mlp_mode)
    _, x, st = run(net, feat, center, noise, R, T0, "object", init=init)
    assert st["status"] == 0
    for b in range(B):
        rot, trans = pose_errors(x[rows(b, R)], want[b][1])
        print(f"[{mlp_mode}] B={B} R={R} T0={T0} object {b}: rot {rot:.2e} trans {trans:.2e} nfev "
              f"{st['obj_nfev'][b]} (oracle {want[b][2]})")
        if mlp_mode == "bf16":
            assert rot <= BF16_ROT_TOL and trans <= BF16_TRANS_TOL
        else:
            assert rot <= ROT_TOL and trans <= TRANS_TOL, (b, rot, trans)
            assert (st["obj_nfev"][b], st["obj_accepted"][b], st["obj_rejected"][b]) == want[b][2:], b


@pytest.mark.parametrize("mlp_mode", ["fp32", "fp32_ffma"])
def test_object_mode_dense_output_matches_per_object_oracle(mlp_mode):
    B, R, T0, S = 3, 50, 0.55, 20
    want = oracle(B, R, T0, False, S)
    feat, center, noise, _ = inputs(B, R, T0, 5)
    net = make_net(100, mlp_mode=mlp_mode)
    xs, x, st = run(net, feat, center, noise, R, T0, "object", num_steps=S)
    assert st["status"] == 0 and xs.shape == (B * R, S, 9)
    for b in range(B):
        assert st["obj_nfev"][b] == want[b][2]
        rot, trans = pose_errors(x[rows(b, R)], want[b][1])
        assert rot <= ROT_TOL and trans <= TRANS_TOL, (b, rot, trans)
        for s in range(S):
            rot, trans = pose_errors(xs[rows(b, R), s], want[b][0][:, s])
            assert rot <= ROT_TOL and trans <= TRANS_TOL, (b, s, rot, trans)


@pytest.mark.parametrize("mlp_mode", MODES)
def test_failed_object_poisons_only_its_rows(mlp_mode):
    """A NaN in object 2's initial state makes its error norm NaN, so every attempt is rejected until the step size
    underflows (status -1).  (NaN features would not do: the ReLUs of the trunk map NaN to 0.)"""
    net = make_net(100, mlp_mode=mlp_mode)
    B, R, T0 = 4, 50, 0.55
    feat, center, noise, _ = inputs(B, R, T0, seed=7)
    _, x_ok, _ = run(net, feat, center, noise, R, T0, "object")
    bad = noise.clone()
    bad[2 * R + 5, 4] = float("nan")
    data = {"pts": torch.zeros(B * R, 1, 3), "pts_center": rep(center, R).cuda(), "_gp_pts_feat_obj": feat.cuda(),
            "_gp_rows_per_object": R}
    _, x = samplers.cond_ode_sampler(net, data, lambda shape, T: bad.clone(), net.sde_fn, device="cuda", T=T0,
                                     pose_mode="rot_matrix", return_trajectory=False, step_control="object")
    x = x.cpu().numpy()
    with pytest.raises(RuntimeError, match="status -1"):
        samplers.ode_stats()
    st = samplers.ode_stats()
    assert list(st["obj_status"]) == [0, 0, -1, 0]
    assert np.isnan(x[rows(2, R)]).all()
    keep = np.r_[0:2 * R, 3 * R:4 * R]
    assert np.array_equal(x[keep], x_ok[keep])


@pytest.mark.parametrize("mlp_mode", MODES)
def test_default_step_control_is_batch(mlp_mode):
    net = make_net(100, mlp_mode=mlp_mode)
    B, R, T0 = 3, 50, 0.55
    feat, center, noise, _ = inputs(B, R, T0, seed=8)
    _, a, sa = run(net, feat, center, noise, R, T0, None)
    _, b, sb = run(net, feat, center, noise, R, T0, "batch")
    assert np.array_equal(a, b) and sa == sb and "obj_nfev" not in sb


def test_pipeline_object_mode_graph_and_shards():
    """PosePipeline(step_control="object"): the graphed step equals the eager step bit for bit, and the two halves of a
    batch run as separate steps reproduce the full batch bit for bit (every stage after the sampler works per object)."""
    from genpose2_b200.pipeline import PosePipeline
    eager = PosePipeline(device="cuda", step_control="object").load_synthetic_weights()
    graph = PosePipeline(device="cuda", use_graph=True, step_control="object").load_synthetic_weights()
    B, R, T0 = 8, 50, 0.55
    pts, center = synthetic.make_point_clouds(B, 1024, seed=60)
    noise = po.ve_prior((B * R, 9), T=T0).float()
    cur = {}
    for pipe in (eager, graph):
        pipe.score_agent.net.prior_fn = lambda shape, T=1.0: cur["noise"].clone()

    def step(pipe, lo, hi):
        cur["noise"] = noise[lo * R:hi * R]
        return pipe({"pts": pts[lo:hi].cuda(), "pts_center": center[lo:hi].cuda()}, repeat_num=R, T0=T0)

    a_pose, a_len = step(eager, 0, B)
    st = samplers.ode_stats()
    assert st["status"] == 0 and len(st["obj_nfev"]) == B
    g_pose, g_len = step(graph, 0, B)
    assert torch.equal(a_pose, g_pose) and torch.equal(a_len, g_len)
    assert len(st_g := samplers.ode_stats()["obj_nfev"]) == B and np.array_equal(st_g, st["obj_nfev"])
    p1, l1 = step(eager, 0, B // 2)
    p2, l2 = step(eager, B // 2, B)
    assert torch.equal(torch.cat([p1, p2]), a_pose) and torch.equal(torch.cat([l1, l2]), a_len)

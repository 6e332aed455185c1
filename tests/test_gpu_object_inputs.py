"""GPU: per-object start times and keyed per-object noise of the ODE sampler (step_control="object").

An object's result must depend only on its own inputs: with mixed start times every object equals a one-object call
from its scalar T0 with the same noise rows, bit for bit (dense output included, and within the north-star gates of the
per-object oracle); a constant T0 vector is the scalar T0; gp_object_noise matches the CPU restatement and a key gives
the same block wherever it sits; and PosePipeline with keys and mixed T0 gives each object the same aggregated pose and
length under permutation and embedding, graphed, with one graph serving every mixed frame of a batch size."""
import functools

import numpy as np
import pytest
import torch

from genpose2_b200 import samplers, synthetic
from oracle import object_noise as on
from oracle import pose_oracle as po
from tests.test_gpu_sampler import BF16_ROT_TOL, BF16_TRANS_TOL, ROT_TOL, TRANS_TOL
from tests.test_gpu_step_control import rows, shaped_net
from tests.util import pose_errors, rep

pytestmark = pytest.mark.gpu

SHAPES = [("fp32", "cluster"), ("fp32", "solo"), ("bf16", "auto"), ("fp32_ffma", "auto")]
T_CYCLE = (0.55, 0.4, 0.25, 0.15)


def inputs(B, R, seed):
    """features, centres, per-object T0 (cycling T_CYCLE) and warm starts (zero rows for the T0 = 0.55 objects)"""
    g = torch.Generator().manual_seed(seed)
    feat = torch.relu(torch.randn(B, 1024, generator=g))
    center = torch.randn(B, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 0.8])
    T = np.array([T_CYCLE[b % len(T_CYCLE)] for b in range(B)])
    init = torch.randn(B, 9, generator=g)
    init[:, 6:] *= 0.05
    init[T == 0.55] = 0.0
    return feat, center, T, init


def call(net, feat, center, R, T, prior, init=None, num_steps=None, **kw):
    """cond_ode_sampler -> (xs, x, device obj_stats [B, 7]) as numpy"""
    B = feat.shape[0]
    data = {"pts": torch.zeros(B * R, 1, 3), "pts_center": rep(center, R).cuda(), "_gp_pts_feat_obj": feat.cuda(),
            "_gp_rows_per_object": R}
    xs, x = samplers.cond_ode_sampler(net, data, prior, net.sde_fn, device="cuda", T=T, pose_mode="rot_matrix",
                                      num_steps=num_steps, return_trajectory=False, step_control="object",
                                      init_x=None if init is None else rep(init, R).cuda(), **kw)
    obj = samplers.last_ode_stats["device_obj_stats"][:, :7].cpu().numpy()
    st = samplers.ode_stats()
    assert st["status"] == 0, st
    return xs.cpu().numpy(), x.cpu().numpy(), obj


def scaled_noise(seed, T, R):
    """the rows the unkeyed per-object draw gives after torch.manual_seed(seed)"""
    torch.manual_seed(seed)
    return samplers.object_prior_noise(samplers.object_sigmas(T, None, len(T)), R)


def solo(net, feat, center, init, T, noise, R, b, num_steps=None):
    warm = None if not init[b].any() else init[b:b + 1]
    return call(net, feat[b:b + 1], center[b:b + 1], R, float(T[b]), lambda shape, T: noise[rows(b, R)].clone(),
                init=warm, num_steps=num_steps)


@pytest.mark.parametrize("mlp_mode,shape", SHAPES)
def test_mixed_T0_equals_solo_calls(mlp_mode, shape):
    net = shaped_net(mlp_mode, shape)
    B, R, seed = 12, 50, 21
    feat, center, T, init = inputs(B, R, seed=1)
    torch.manual_seed(seed)
    _, x, obj = call(net, feat, center, R, T, None, init=init)
    noise = scaled_noise(seed, T, R)
    for b in range(B):
        _, xb, ob = solo(net, feat, center, init, T, noise, R, b)
        assert np.array_equal(x[rows(b, R)], xb), b
        assert np.array_equal(obj[b], ob[0]), (b, obj[b], ob[0])
    print(f"mixed T0 [{mlp_mode}/{shape}]: nfev per object {obj[:, 0].astype(int).tolist()}")


@pytest.mark.parametrize("mlp_mode,shape", SHAPES)
def test_constant_T0_vector_equals_scalar(mlp_mode, shape):
    net = shaped_net(mlp_mode, shape)
    B, R = 6, 50
    feat, center, _, _ = inputs(B, R, seed=2)
    torch.manual_seed(5)
    _, a, oa = call(net, feat, center, R, 0.55, net.prior_fn)
    torch.manual_seed(5)
    _, b, ob = call(net, feat, center, R, torch.full((B,), 0.55, dtype=torch.float64), net.prior_fn)
    assert np.array_equal(a, b) and np.array_equal(oa, ob)


@functools.lru_cache(maxsize=None)
def dense_oracle(B, R, S, seed):
    feat, center, T, init = inputs(B, R, seed=3)
    noise = scaled_noise(seed, T, R)
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(100))
    out = []
    for b in range(B):
        xs, x, s = po.cond_ode_sampler(trunk, rep(feat[b:b + 1], R), rep(center[b:b + 1], R), noise[rows(b, R)],
                                       init_x=rep(init[b:b + 1], R) if init[b].any() else None, T=float(T[b]),
                                       num_steps=S)
        out.append((xs.numpy(), x.numpy(), s["nfev"]))
    return out


@pytest.mark.parametrize("mlp_mode,shape", SHAPES)
def test_mixed_T0_dense_output(mlp_mode, shape):
    net = shaped_net(mlp_mode, shape)
    B, R, S, seed = 4, 50, 20, 33
    feat, center, T, init = inputs(B, R, seed=3)
    torch.manual_seed(seed)
    xs, x, obj = call(net, feat, center, R, T, None, init=init, num_steps=S)
    assert xs.shape == (B * R, S, 9)
    noise = scaled_noise(seed, T, R)
    want = dense_oracle(B, R, S, seed)
    for b in range(B):
        xsb, xb, ob = solo(net, feat, center, init, T, noise, R, b, num_steps=S)
        assert np.array_equal(xs[rows(b, R)], xsb) and np.array_equal(x[rows(b, R)], xb), b
        assert np.array_equal(obj[b], ob[0]), b
        rot_tol, trans_tol = (BF16_ROT_TOL, BF16_TRANS_TOL) if mlp_mode == "bf16" else (ROT_TOL, TRANS_TOL)
        rot, trans = pose_errors(x[rows(b, R)], want[b][1])
        assert rot <= rot_tol and trans <= trans_tol, (b, rot, trans)
        for s in range(S):
            rot, trans = pose_errors(xs[rows(b, R), s], want[b][0][:, s])
            assert rot <= rot_tol and trans <= trans_tol, (b, s, rot, trans)
        if mlp_mode != "bf16":
            assert int(obj[b, 0]) == want[b][2], (b, obj[b, 0], want[b][2])


KEYS = [0, 1, -1, 7, 1 << 40, -(1 << 62), 123456789012345, 42]


@pytest.mark.parametrize("R", [1, 7, 50, 128])
def test_keyed_noise_matches_oracle(R):
    keys = torch.tensor(KEYS, dtype=torch.int64)
    sig = torch.tensor([1.0, 0.5, 2.0, 1.0, 3.25, 1.0, 0.01, 1.0], dtype=torch.float32)
    got = samplers.keyed_noise(keys.cuda(), sig.cuda(), R).cpu().numpy()
    want = on.object_noise(KEYS, sig.numpy(), R)
    unit = samplers.keyed_noise(keys.cuda(), torch.ones(len(KEYS), device="cuda"), R).cpu().numpy()
    normals = np.concatenate([on.object_normals(k, R) for k in KEYS])
    # the normals: within 1 float32 ulp of the restatement (float64 log / cos / sin of device and numpy may differ in
    # their last bit); then scaled by sigma in float32 exactly as the restatement scales them
    ulps = np.abs(unit.view(np.int32).astype(np.int64) - normals.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, ulps.max()
    print(f"R={R}: {int((ulps > 0).sum())} of {ulps.size} normals differ by 1 ulp")
    assert np.array_equal(got, unit * np.repeat(sig.numpy(), R)[:, None])
    close = ulps.reshape(len(KEYS), R * 9).max(axis=1) == 0
    assert np.array_equal(got.reshape(len(KEYS), -1)[close], want.reshape(len(KEYS), -1)[close])


def test_keyed_noise_block_depends_on_its_key_only():
    R = 50
    sig = torch.ones(16, device="cuda")
    full = samplers.keyed_noise(torch.arange(100, 116, device="cuda"), sig, R).cpu()
    for B, at in ((1, [5]), (3, [0, 2, 1]), (16, list(range(15, -1, -1)))):
        keys = torch.tensor([100 + a for a in at], device="cuda")
        got = samplers.keyed_noise(keys, sig[:B], R).cpu()
        for i, a in enumerate(at):
            assert torch.equal(got[rows(i, R)], full[rows(a, R)]), (B, i, a)


def test_keyed_call_leaves_the_global_generator_alone():
    net = shaped_net("fp32", "auto")
    B, R = 4, 50
    feat, center, T, init = inputs(B, R, seed=4)
    torch.manual_seed(9)
    before = torch.get_rng_state()
    keys = torch.arange(B, dtype=torch.int64)
    _, a, _ = call(net, feat, center, R, T, None, init=init, noise_keys=keys)
    _, b, _ = call(net, feat, center, R, 0.55, None, noise_keys=keys.cuda())
    assert torch.equal(torch.get_rng_state(), before)
    # the keyed noise is gp_object_noise with sigma(T_b): the same as injecting it
    sig = samplers.object_sigmas(T, None, B)
    noise = samplers.keyed_noise(keys.cuda(), sig.cuda(), R).cpu()
    for i in range(B):
        _, xb, _ = solo(net, feat, center, init, T, noise, R, i)
        assert np.array_equal(a[rows(i, R)], xb), i


def frame(B, seed):
    pts, center = synthetic.make_point_clouds(B, 1024, seed=seed)
    g = torch.Generator().manual_seed(seed)
    T = np.array([T_CYCLE[b % len(T_CYCLE)] for b in range(B)])
    init = torch.randn(B, 9, generator=g)
    init[:, 6:] *= 0.05
    init[T == 0.55] = 0.0
    keys = torch.randint(-(1 << 62), 1 << 62, (B,), generator=g, dtype=torch.int64)
    return pts, center, T, init, keys


def test_pipeline_keyed_mixed_frame_is_invariant():
    """8 objects; the same 8 permuted; the same 8 embedded in 16 objects (both sizes run the score net as clusters
    and the energy net on the same shape): each object's aggregated pose and length are bit-identical."""
    from genpose2_b200.pipeline import PosePipeline
    pipe = PosePipeline(device="cuda", use_graph=True, step_control="object").load_synthetic_weights()
    R = 50
    pts, center, T, init, keys = frame(8, seed=70)

    def step(idx, P=pts, C=center, TT=T, I=init, K=keys):
        return pipe({"pts": P[idx].cuda(), "pts_center": C[idx].cuda()}, repeat_num=R, T0=TT[idx],
                    init_x=I[idx].cuda(), noise_keys=K[idx])

    pose, length = step(np.arange(8))
    assert torch.isfinite(pose).all() and torch.isfinite(length).all()
    perm = np.random.default_rng(0).permutation(8)
    pp, lp = step(perm)
    assert torch.equal(pp, pose[perm]) and torch.equal(lp, length[perm])
    p16, c16, T16, i16, k16 = frame(16, seed=71)
    at = np.sort(np.random.default_rng(1).choice(16, 8, replace=False))
    p16[at], c16[at], T16[at], i16[at], k16[at] = pts, center, T, init, keys
    pe, le = step(np.arange(16), p16, c16, T16, i16, k16)
    assert torch.equal(pe[at], pose) and torch.equal(le[at], length)


def test_one_graph_serves_every_mixed_frame():
    """One captured graph replays frames with different T0 vectors and keys (len(_graphs) stays 1), each equal to the
    eager step bit for bit; per-object T0 without keys is a second graph, equal to the eager step with the same seed."""
    from genpose2_b200.pipeline import PosePipeline
    eager = PosePipeline(device="cuda", step_control="object").load_synthetic_weights()
    graph = PosePipeline(device="cuda", use_graph=True, step_control="object").load_synthetic_weights()
    R, B = 50, 8
    for k, seed in enumerate((80, 81, 82)):
        pts, center, T, init, keys = frame(B, seed)
        T = np.roll(T, k) if k else T
        data = {"pts": pts.cuda(), "pts_center": center.cuda()}
        a = eager(dict(data), repeat_num=R, T0=T, init_x=init.cuda(), noise_keys=keys)
        g = graph(dict(data), repeat_num=R, T0=T, init_x=init.cuda(), noise_keys=keys.cuda() if k == 1 else keys)
        assert torch.equal(a[0], g[0]) and torch.equal(a[1], g[1]), k
        assert len(graph._graphs) == 1
    for seed in (83, 84):
        pts, center, T, init, _ = frame(B, seed)
        data = {"pts": pts.cuda(), "pts_center": center.cuda()}
        torch.manual_seed(seed)
        a = eager(dict(data), repeat_num=R, T0=T, init_x=init.cuda())
        torch.manual_seed(seed)
        g = graph(dict(data), repeat_num=R, T0=T, init_x=init.cuda())
        assert torch.equal(a[0], g[0]) and torch.equal(a[1], g[1]), seed
    assert len(graph._graphs) == 2

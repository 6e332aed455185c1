"""CPU: pins the oracle restatements (oracle/pose_oracle.py) against the golden fixtures that
tests/golden/make_golden.py produced by running the reference itself, and the restated
third-party algorithms (scipy RK45, sklearn DBSCAN) against the libraries on the reference's
call sites."""
import os

import numpy as np
import pytest
import torch

from genpose2_b200 import synthetic
from oracle import pose_oracle as po


@pytest.fixture(autouse=True)
def golden_thread_count():
    """tests/golden/make_golden.py ran the reference with torch.set_num_threads(8), and torch-CPU's summation order
    depends on the thread count: the restatement runs with the same count so that it agrees with the goldens to
    rounding on a host with any number of cores."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name + ".npz")))


def geodesic(x, y):
    """angle between rotations given as 6D (first two columns) tensors [N,6]."""
    Rx = po.get_rot_matrix(torch.as_tensor(x, dtype=torch.float64))
    Ry = po.get_rot_matrix(torch.as_tensor(y, dtype=torch.float64))
    tr = torch.einsum("bij,bij->b", Rx, Ry)
    return torch.acos(torch.clamp((tr - 1) / 2, -1, 1))


def rep(a, R):
    return a.unsqueeze(1).repeat(1, R, 1).view(a.shape[0] * R, -1)


@pytest.mark.parametrize("name", ["ode_c1_T1", "ode_b4_T055", "ode_track_T025"])
@pytest.mark.parametrize("integrator", ["restated", "scipy"])
def test_ode_sampler_matches_reference(golden_dir, name, integrator):
    g = load(golden_dir, name)
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(int(g["score_seed"])))
    R = int(g["R"])
    feat, center = torch.from_numpy(g["feat"]), torch.from_numpy(g["center"])
    init = rep(torch.from_numpy(g["init_x"]), R) if "init_x" in g else None
    xs, x, stats = po.cond_ode_sampler(trunk, rep(feat, R), rep(center, R), torch.from_numpy(g["noise"]),
                                       init_x=init, T=float(g["T0"]), integrator=integrator)
    assert stats["nfev"] + 1 == int(g["nfev"])  # +1: the denoise evaluation outside the solver
    assert xs.shape[1] == int(g["S"])
    # same torch-CPU kernels in the same order -> agreement to rounding
    np.testing.assert_allclose(x.numpy(), g["x"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(xs[:, -1].numpy(), g["xs_last"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(xs[:, xs.shape[1] // 2].numpy(), g["xs_mid"], rtol=0, atol=1e-9)
    assert x.dtype == torch.float64


def test_ode_sampler_dense_output(golden_dir):
    g = load(golden_dir, "ode_b2_T055_steps20")
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(int(g["score_seed"])))
    R = int(g["R"])
    feat, center = torch.from_numpy(g["feat"]), torch.from_numpy(g["center"])
    xs, x, stats = po.cond_ode_sampler(trunk, rep(feat, R), rep(center, R), torch.from_numpy(g["noise"]),
                                       T=float(g["T0"]), num_steps=20, integrator="restated")
    assert xs.shape[1] == 20
    np.testing.assert_allclose(x.numpy(), g["x"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(xs[:, 10].numpy(), g["xs_mid"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(xs[:, 0].numpy(), g["xs_first"], rtol=0, atol=1e-9)


def test_pc_sampler_matches_reference(golden_dir):
    g = load(golden_dir, "pc_b2")
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(int(g["score_seed"])))
    R = int(g["R"])
    feat, center = torch.from_numpy(g["feat"]), torch.from_numpy(g["center"])
    xs, mean_x = po.cond_pc_sampler(trunk, rep(feat, R), rep(center, R), torch.from_numpy(g["init"]),
                                    torch.from_numpy(g["noises"]), num_steps=int(g["steps"]))
    np.testing.assert_allclose(mean_x.numpy(), g["mean_x"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(xs.numpy(), g["xs"], rtol=0, atol=1e-6)


def test_energy_matches_reference(golden_dir):
    g = load(golden_dir, "energy_b3")
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(int(g["energy_seed"])))
    poses = torch.from_numpy(g["poses"])
    B, R = poses.shape[:2]
    feat, center = torch.from_numpy(g["feat"]), torch.from_numpy(g["center"])
    sp = poses.clone().view(B * R, -1).float()
    sp[:, -3:] -= rep(center, R)
    e = trunk.energy(rep(feat, R), sp, torch.ones(B * R, 1) * 1e-5).reshape(B, R, 2)
    np.testing.assert_allclose(e.numpy(), g["energy"], rtol=1e-6, atol=1e-6)


def test_aggregation_with_clusters_matches_reference(golden_dir):
    g = load(golden_dir, "aggregate_clusters")
    poses, energy = torch.from_numpy(g["poses"]), torch.from_numpy(g["energy"])
    sp, se = po.sort_poses_by_energy(poses, energy)
    np.testing.assert_array_equal(sp.numpy(), g["sorted_pose"])
    np.testing.assert_array_equal(se.numpy(), g["sorted_energy"])
    for mode in ("restated", "sklearn"):
        agg, labels = po.aggregate_pose(poses, energy, dbscan=mode)
        np.testing.assert_array_equal(labels, g["labels"])
        np.testing.assert_allclose(agg.numpy(), g["aggregated_pose"], rtol=0, atol=1e-6)
    assert (g["labels"] >= 0).any() and (g["labels"] == -1).any()


def test_scalenet_matches_reference(golden_dir):
    g = load(golden_dir, "scalenet_b5")
    sd = synthetic.random_scalenet_state_dict(int(g["scale_seed"]))
    out = po.scalenet_forward(sd, torch.from_numpy(g["axes"]), torch.from_numpy(g["feat"]))
    np.testing.assert_allclose(out.numpy(), g["length"], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("name", ["full_b3_T055", "full_track_b2_T025"])
def test_full_path_matches_reference(golden_dir, name):
    g = load(golden_dir, name)
    ssd = synthetic.random_gfobjectpose_state_dict(int(g["score_seed"]))
    esd = synthetic.random_gfobjectpose_state_dict(int(g["energy_seed"]))
    csd = synthetic.random_scalenet_state_dict(int(g["scale_seed"]))
    init = torch.from_numpy(g["init_x"]) if "init_x" in g else None
    out = po.full_pipeline(ssd, esd, csd, torch.from_numpy(g["pts"]), torch.from_numpy(g["center"]),
                           torch.from_numpy(g["noise"]), repeat_num=int(g["R"]), T0=float(g["T0"]),
                           init_x=init, integrator="restated",
                           score_feat=torch.from_numpy(g["score_feat"]),
                           energy_feat=torch.from_numpy(g["energy_feat"]))
    np.testing.assert_allclose(out["pred_pose"].numpy(), g["pred_pose"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(out["energy"].numpy(), g["energy"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(out["aggregated_pose"].numpy(), g["aggregated_pose"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(out["length"].numpy(), g["length"], rtol=1e-5, atol=1e-6)
    np.testing.assert_array_equal(out["labels"], g["labels"])


def test_rk45_restated_matches_scipy_on_stiffish_problem():
    from scipy import integrate

    rng = np.random.default_rng(0)
    A = rng.normal(size=(12, 12)) * 0.7

    def fun(t, y):
        return np.tanh(A @ y) * (1 + 5 * t) - 0.3 * y

    y0 = rng.normal(size=12)
    ref = integrate.solve_ivp(fun, (1.0, 1e-5), y0, method="RK45", rtol=1e-5, atol=1e-5)
    mine = po.rk45_restated(fun, 1.0, 1e-5, y0, 1e-5, 1e-5)
    assert mine["nfev"] == ref.nfev
    np.testing.assert_array_equal(mine["t"], ref.t)
    np.testing.assert_allclose(mine["y"], ref.y, rtol=0, atol=1e-14)
    assert mine["n_rejected"] >= 0 and mine["n_accepted"] == len(ref.t) - 1
    te = np.linspace(1.0, 1e-5, 17)
    ref = integrate.solve_ivp(fun, (1.0, 1e-5), y0, method="RK45", rtol=1e-5, atol=1e-5, t_eval=te)
    mine = po.rk45_restated(fun, 1.0, 1e-5, y0, 1e-5, 1e-5, t_eval=te)
    np.testing.assert_allclose(mine["y"], ref.y, rtol=0, atol=1e-13)


def test_dbscan_restated_matches_sklearn_random():
    from sklearn.cluster import DBSCAN

    rng = np.random.default_rng(1)
    for trial in range(40):
        n = 20
        centers = rng.normal(size=(3, 4))
        pts = centers[rng.integers(0, 3, n)] + rng.normal(size=(n, 4)) * rng.choice([0.05, 0.15, 0.4])
        D = np.sqrt(((pts[:, None] - pts[None]) ** 2).sum(-1))
        eps = rng.choice([0.2, 0.5, 1.0])
        a = DBSCAN(eps=eps, min_samples=3).fit(D).labels_
        b = po.dbscan_restated(D, eps, 3)
        np.testing.assert_array_equal(a, b)


def test_fps_of_an_fps_ordered_cloud_is_its_prefix():
    """The identity gp_fps_chain relies on (DESIGN.md 4.1), on the reference restatement alone: sampling the
    centres of the previous level again returns 0, 1, ..., m-1 as long as no step tied; with exact ties between
    different locations (a lattice) it does not have to, which is why the kernel keeps the tie bookkeeping."""
    from oracle import pointnet2_oracle as p2
    pts, _ = synthetic.make_point_clouds(6, 1024, seed=3, dup_fraction=0.0)
    xyz = pts.numpy()
    idx = p2.furthest_point_sample(xyz, 512)
    level1 = np.take_along_axis(xyz, idx[..., None].astype(np.int64), 1)
    for m in (256, 128, 64):
        again = p2.furthest_point_sample(level1, m)
        np.testing.assert_array_equal(again, np.broadcast_to(np.arange(m, dtype=again.dtype), again.shape))
        level1 = level1[:, :m]
    g = np.stack(np.meshgrid(*[np.arange(8.0)] * 3, indexing="ij"), -1).reshape(1, -1, 3).astype(np.float32)
    lat = g[:, np.random.default_rng(0).permutation(g.shape[1])]
    i1 = p2.furthest_point_sample(lat, 256)
    l1 = np.take_along_axis(lat, i1[..., None].astype(np.int64), 1)
    assert not np.array_equal(p2.furthest_point_sample(l1, 128)[0], np.arange(128))

"""CPU: the per-object step control of the ODE sampler (step_control="object") -- argument validation before any
device work, the C ABI's validation and workspace sizing, the graph key of PosePipeline, and the per-object oracle
(oracle.pose_oracle.cond_ode_sampler run on one object at a time) against scipy's solve_ivp on the restated trunk."""
import ctypes
import types

import numpy as np
import pytest
import torch

from genpose2_b200 import _lib, samplers, synthetic
from oracle import pose_oracle as po
from tests.util import rep


def _no_prior(shape, T=1.0):
    raise AssertionError("the prior was drawn: validation must come before any sampler work")


def _data(B, R):
    return {"pts": torch.zeros(B * R, 1, 3), "pts_center": torch.zeros(B * R, 3),
            "_gp_pts_feat_obj": torch.zeros(B, 1024), "_gp_rows_per_object": R}


# stands in for a GFObjectPose: the samplers only look for `packed` before validating
FAKE_NET = types.SimpleNamespace(packed=lambda: None)


def test_bad_step_control_values_raise_before_device_work():
    with pytest.raises(ValueError, match="step_control"):
        samplers.cond_ode_sampler(FAKE_NET, _data(2, 50), _no_prior, None, pose_mode="rot_matrix",
                                  return_trajectory=False, step_control="tile")
    with pytest.raises(NotImplementedError, match="128"):
        samplers.cond_ode_sampler(FAKE_NET, _data(2, 129), _no_prior, None, pose_mode="rot_matrix",
                                  return_trajectory=False, step_control="object")
    with pytest.raises(NotImplementedError, match="trajectory"):
        samplers.cond_ode_sampler(FAKE_NET, _data(2, 50), _no_prior, None, pose_mode="rot_matrix",
                                  step_control="object")
    with pytest.raises(NotImplementedError, match="ODE sampler only"):
        samplers.cond_pc_sampler(FAKE_NET, _data(2, 50), _no_prior, None, num_steps=4, pose_mode="rot_matrix",
                                 step_control="object")
    with pytest.raises(ValueError, match="step_control"):
        samplers.cond_pc_sampler(FAKE_NET, _data(2, 50), _no_prior, None, num_steps=4, pose_mode="rot_matrix",
                                 step_control="tile")
    from genpose2_b200.pipeline import PosePipeline
    with pytest.raises(ValueError, match="step_control"):
        PosePipeline(device="cpu", step_control="objects")


def test_step_control_is_keyword_only():
    with pytest.raises(TypeError):
        samplers.cond_ode_sampler(FAKE_NET, _data(1, 1), _no_prior, None, 1e-5, 1e-5, "cuda", 1e-5, 1.0, None,
                                  "rot_matrix", True, None, False, "object")


def test_graph_key_includes_step_control():
    from genpose2_b200.pipeline import PosePipeline
    pts = torch.zeros(2, 16, 3)
    keys = {sc: PosePipeline(device="cpu", step_control=sc)._graph_key(pts, 50, 0.55, None)
            for sc in samplers.STEP_CONTROLS}
    assert keys["batch"] != keys["object"]
    assert keys["batch"][:-1] == keys["object"][:-1]
    cfg = PosePipeline(device="cpu", step_control="object").score_agent.net.cfg
    assert cfg.step_control == "object"


def test_objects_workspace_sizing():
    lib = _lib.load()
    per_obj = 128 * 9 * 8   # one padded 128-row tile of float64 state
    for B in (1, 13, 64, 1024):
        for R in (1, 7, 50, 128):
            ws = lib.gp_scorenet_ode_objects_workspace_bytes(B, R)
            # y, y_new, K0..K6 for each of the 4 CTAs of a cluster, 256-byte aligned, plus alignment slack
            assert ws == ((B * per_obj + 255) // 256 * 256) * 9 * 4 + 256, (B, R, ws)
    assert lib.gp_scorenet_ode_objects_workspace_bytes(4, 129) == 0
    assert lib.gp_scorenet_ode_objects_workspace_bytes(0, 50) == 0
    assert lib.gp_scorenet_ode_objects_workspace_bytes(4, 0) == 0


def test_objects_c_abi_validation():
    """The entries reject unsupported sizes before touching the device (dummy non-null pointers are never read)."""
    lib = _lib.load()
    p = ctypes.c_void_p(256)

    def call(N, R, ws_bytes=1 << 40):
        return lib.gp_scorenet_ode_objects(p, p, p, p, N, R, 0.55, 1e-5, 1e-5, 1e-5, 1, p, p, p, p, ws_bytes, 2, None)

    assert call(2 * 129, 129) == -2 and "128" in _lib.last_error()        # GP_ERR_UNSUPPORTED
    assert call(101, 50) == -1 and "B * rows_per_object" in _lib.last_error()
    assert call(100, 50, ws_bytes=1024) == -3 and "workspace" in _lib.last_error()
    rc = lib.gp_scorenet_ode_dense_objects(p, p, p, p, 100, 50, 0.55, 1e-5, 1e-5, 1e-5, 1, p, None, 0, None, p, p, p,
                                           1 << 40, 2, None)
    assert rc == -1
    rc = lib.gp_scorenet_ode_objects(None, p, p, p, 100, 50, 0.55, 1e-5, 1e-5, 1e-5, 1, p, p, p, p, 1 << 40, 2, None)
    assert rc == -1 and "null" in _lib.last_error()


@pytest.mark.parametrize("T0,with_init", [(0.55, False), (0.25, True)])
def test_per_object_oracle_matches_scipy_per_object(T0, with_init):
    """The oracle the GPU tests hold "object" mode to: the restated RK45 run on each object alone equals scipy's
    solve_ivp run on each object alone (same trunk), step counts included; and objects integrated alone differ from
    the same objects integrated as one batch (the property the mode exists for)."""
    trunk = po.Trunk(synthetic.random_gfobjectpose_state_dict(100))
    g = torch.Generator().manual_seed(3)
    B, R = 3, 7
    feat = torch.relu(torch.randn(B, 1024, generator=g))
    center = torch.randn(B, 3, generator=g) * 0.1
    noise = torch.randn(B * R, 9, generator=g) * po.ve_marginal_std(T0)
    init = rep(torch.randn(B, 9, generator=g), R) if with_init else None
    xs_alone = []
    for b in range(B):
        rows = slice(b * R, (b + 1) * R)
        args = (trunk, rep(feat[b:b + 1], R), rep(center[b:b + 1], R), noise[rows])
        kw = dict(init_x=None if init is None else init[rows], T=T0)
        xs_r, x_r, st_r = po.cond_ode_sampler(*args, **kw, integrator="restated")
        xs_s, x_s, st_s = po.cond_ode_sampler(*args, **kw, integrator="scipy")
        assert st_r["nfev"] == st_s["nfev"] and xs_r.shape == xs_s.shape
        np.testing.assert_allclose(x_r.numpy(), x_s.numpy(), rtol=0, atol=1e-12)
        xs_alone.append(x_r)
    _, x_batch, _ = po.cond_ode_sampler(trunk, rep(feat, R), rep(center, R), noise, init_x=init, T=T0)
    assert not np.array_equal(torch.cat(xs_alone).numpy(), x_batch.numpy())

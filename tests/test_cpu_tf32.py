"""CPU: mlp_mode "tf32" (trunk mode 3) -- the `mode` argument it produces, refusal of the shared-memory-A shape before
any device work, the C ABI's checks of mode 3 and of gp_trunk_pack_tf32, the configuration plumbing, and the oracle's
restatement of cvt.rna.tf32.f32 against hand-computed values."""
import ctypes

import numpy as np
import pytest
import torch

from genpose2_b200 import _lib, samplers
from genpose2_b200.scorenet import EVAL_SHAPES, MLP_MODES, PoseScoreNet
from oracle.tf32 import tf32_round
from tests.test_cpu_step_control import _data, _no_prior

GP_MODE_SOLO, GP_MODE_CLUSTER, GP_MODE_SMEM_A = 16, 32, 64


def _net(shape="auto"):
    net = PoseScoreNet(None, 0, "rot_matrix", "Rx_Ry_and_T")
    net.mlp_mode, net.eval_shape = "tf32", shape
    return net


def test_mode_arg_is_3_with_shape_flags():
    assert MLP_MODES["tf32"] == 3
    assert _net("auto").mode_arg() == 3
    assert _net("solo").mode_arg() == 3 | GP_MODE_SOLO
    assert _net("cluster").mode_arg() == 3 | GP_MODE_CLUSTER
    assert EVAL_SHAPES["solo_smem_a"] == GP_MODE_SOLO | GP_MODE_SMEM_A


def test_solo_smem_a_raises_before_device_work():
    net = _net("solo_smem_a")
    with pytest.raises(ValueError, match="solo_smem_a"):
        net.mode_arg()
    # the parameters are on the CPU: reaching the packing would raise RuntimeError instead
    with pytest.raises(ValueError, match="solo_smem_a"):
        net.packed()
    with pytest.raises(ValueError, match="solo_smem_a"):
        samplers.cond_ode_sampler(net, _data(2, 50), _no_prior, None, pose_mode="rot_matrix", return_trajectory=False)
    with pytest.raises(ValueError, match="solo_smem_a"):
        samplers.cond_pc_sampler(net, _data(2, 50), _no_prior, None, num_steps=4, pose_mode="rot_matrix")


def test_c_abi_refuses_bad_tf32_modes():
    """Dummy non-null pointers: the entries must refuse before touching the device."""
    lib = _lib.load()
    p = ctypes.c_void_p(256)
    for mode, rc, msg in ((3 | GP_MODE_SMEM_A, -2, "GP_MODE_SMEM_A"), (3 | GP_MODE_SOLO | GP_MODE_SMEM_A, -2, "GP_MODE_SMEM_A"),
                          (3 | GP_MODE_SOLO | GP_MODE_CLUSTER, -1, "mode must be"), (3 | 128, -1, "mode must be")):
        assert lib.gp_scorenet_eval(p, p, p, p, 100, 50, p, mode, None) == rc and msg in _lib.last_error()
        assert lib.gp_energy(p, p, p, p, p, 100, 50, p, mode, None) == rc and msg in _lib.last_error()
        assert lib.gp_scorenet_ode(p, p, p, p, 100, 50, 0.55, 1e-5, 1e-5, 1e-5, 1, p, None, 0, p, p, 1 << 40, mode,
                                   None) == rc and msg in _lib.last_error()
        assert lib.gp_scorenet_ode_objects(p, p, p, p, 100, 50, 0.55, 1e-5, 1e-5, 1e-5, 1, p, p, p, p, 1 << 40, mode,
                                           None) == rc and msg in _lib.last_error()
        assert lib.gp_scorenet_ode_objects_t0(p, p, p, p, 100, 50, p, 1e-5, 1e-5, 1e-5, 1, p, None, 0, None, p, p, p,
                                              1 << 40, mode, None) == rc and msg in _lib.last_error()
        assert lib.gp_scorenet_pc(p, p, p, p, p, p, 100, 50, 25, 0.16, p, p, p, 1 << 40, mode,
                                  None) == rc and msg in _lib.last_error()


def test_pack_tf32_refuses_null_pointers():
    lib = _lib.load()
    assert lib.gp_trunk_pack_tf32(None, ctypes.c_void_p(256), None) == -1 and "null" in _lib.last_error()
    assert "gp_trunk_pack_tf32" in _lib.last_error()
    params = _lib.TrunkParams()   # every parameter pointer null
    assert lib.gp_trunk_pack_tf32(ctypes.byref(params), ctypes.c_void_p(256), None) == -1
    assert "null" in _lib.last_error()
    assert lib.gp_trunk_pack_tf32(ctypes.byref(params), None, None) == -1 and "null" in _lib.last_error()


def test_config_plumbing():
    from genpose2_b200.config import get_config
    from genpose2_b200.pipeline import PosePipeline
    assert get_config(["--mlp_mode", "tf32"]).mlp_mode == "tf32"
    pipe = PosePipeline(device="cpu", mlp_mode="tf32")
    for agent in (pipe.score_agent, pipe.energy_agent):
        assert agent.net.pose_score_net.mlp_mode == "tf32"
        # the point-cloud encoder stays fp32-class (split bf16): only the trunk runs in tf32
        assert {sa.gemm_mode for sa in agent.net.pts_encoder.SA_modules} == {"bf16x3"}


def _bits(v):
    return int(np.array([v], dtype=np.float32).view(np.uint32)[0])


def _from_bits(b):
    return float(np.array([b], dtype=np.uint32).view(np.float32)[0])


def test_oracle_tf32_rounding_hand_values():
    one = _bits(1.0)                                   # 0x3f800000; the tf32 ulp at 1 is 2^-10 (bit 13)
    cases = [
        (1.0, 1.0),
        (_from_bits(one + 0x0FFF), 1.0),                # below half an ulp: down
        (_from_bits(one + 0x1000), 1.0 + 2.0 ** -10),   # exactly half: tie, away from zero (to even would give 1)
        (_from_bits(one + 0x1001), 1.0 + 2.0 ** -10),
        (_from_bits(one + 0x2000 + 0x1000), 1.0 + 2.0 ** -9),   # tie above 1 + 2^-10: away from zero again
        (1.0 + 2.0 ** -11, 1.0 + 2.0 ** -10),           # 1 + half an ulp
        (1.0 + 2.0 ** -12, 1.0),
        (0.0, 0.0),
        (3.0, 3.0),
        (1.0 / 3.0, _from_bits(0x3eaaa000)),            # 0x3eaaaaab: dropped bits 0x0aab < 0x1000, down
        (float(np.float32(np.pi)), _from_bits(0x40490000)),   # 0x40490fdb: dropped bits 0x0fdb < 0x1000, down
        (float(np.float32(np.e)), _from_bits(0x402e0000)),    # 0x402df854: dropped bits 0x1854 > 0x1000, up
        (float(np.finfo(np.float32).max), np.inf),      # past the largest float32
    ]
    for x, want in cases:
        got = float(tf32_round(np.float32(x)))
        assert got == want, (x, got, want)
        # the sign is carried: ties go away from zero on both sides
        assert float(tf32_round(np.float32(-x))) == -want, x
    assert np.signbit(tf32_round(np.float32(-0.0)))
    assert np.isinf(tf32_round(np.float32(np.inf))) and np.isnan(tf32_round(np.float32(np.nan)))


def test_oracle_tf32_rounding_properties():
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(100_000) * np.exp(rng.uniform(-20, 20, 100_000))).astype(np.float32)
    r = tf32_round(x)
    assert r.dtype == np.float32 and r.shape == x.shape
    assert (r.view(np.uint32) & 0x1FFF == 0).all()           # 10 explicit significand bits left
    assert np.array_equal(tf32_round(r), r)                    # idempotent
    assert np.array_equal(tf32_round(-x), -r)                  # odd
    # nearest: within half a tf32 ulp of the input
    err = np.abs(r.astype(np.float64) - x.astype(np.float64))
    ulp = np.exp2(np.floor(np.log2(np.abs(x.astype(np.float64)))) - 10)
    assert (err <= ulp / 2).all()
    # float64 inputs are taken as float32 first; shapes are kept
    assert tf32_round(np.ones((3, 4))).shape == (3, 4)
    assert torch.equal(torch.from_numpy(tf32_round(np.ones(2))), torch.ones(2))

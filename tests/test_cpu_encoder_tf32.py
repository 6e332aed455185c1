"""CPU: encoder_mode (the operand precision of the encoder's tensor-core SharedMLP GEMMs) -- the configuration
plumbing, "tf32" (npass = 2) sizes and the C ABI's refusal of npass values outside {1, 2, 3} before any device work."""
import ctypes

import pytest

from genpose2_b200 import _lib
from genpose2_b200 import pointnet2_utils as pu
from genpose2_b200.pointnet2 import ClsMSG_CFG_Light, GEMM_NPASS


def _encoder_modes(pipe):
    """gemm_mode of every SA module and SharedMLP of both encoders"""
    modes = set()
    for agent in (pipe.score_agent, pipe.energy_agent):
        for sa in agent.net.pts_encoder.SA_modules:
            modes.add(sa.gemm_mode)
            modes.update(m.gemm_mode for m in sa.mlps)
    return modes


def _pipeline(**kw):
    from genpose2_b200.pipeline import PosePipeline
    return PosePipeline(device="cpu", **kw)


@pytest.mark.parametrize("mlp_mode,want", [("fp32", "bf16x3"), ("fp32_ffma", "bf16x3"), ("tf32", "bf16x3"),
                                           ("bf16", "bf16")])
def test_auto_keeps_the_mlp_mode_mapping(mlp_mode, want):
    assert _encoder_modes(_pipeline(mlp_mode=mlp_mode)) == {want}
    assert _encoder_modes(_pipeline(mlp_mode=mlp_mode, encoder_mode="auto")) == {want}


@pytest.mark.parametrize("mlp_mode", ["fp32", "tf32", "bf16"])
def test_encoder_mode_tf32_sets_every_level(mlp_mode):
    from genpose2_b200.config import get_config
    assert get_config().encoder_mode == "auto"
    assert get_config(["--encoder_mode", "tf32"]).encoder_mode == "tf32"
    pipe = _pipeline(mlp_mode=mlp_mode, encoder_mode="tf32")
    assert _encoder_modes(pipe) == {"tf32"}
    for agent in (pipe.score_agent, pipe.energy_agent):   # the trunk keeps its own mode
        assert agent.net.pose_score_net.mlp_mode == mlp_mode
    assert _encoder_modes(_pipeline(encoder_mode="bf16")) == {"bf16"}


def test_bad_encoder_mode_raises_before_device_work():
    # "cuda:7" does not exist on any test host: reaching device work would raise something else
    from genpose2_b200.config import get_config
    from genpose2_b200.posenet import GFObjectPose
    with pytest.raises(ValueError, match="encoder_mode"):
        _pipeline(encoder_mode="fp32")
    cfg = get_config(["--encoder_mode", "tf16", "--device", "cuda:7"])
    with pytest.raises(ValueError, match="encoder_mode"):
        GFObjectPose(cfg, None, None, None, 1e-5, 1.0)


def test_set_gemm_mode_accepts_the_table():
    from genpose2_b200.pointnet2 import Pointnet2ClsMSG
    assert GEMM_NPASS == {"bf16x3": 3, "tf32": 2, "bf16": 1}
    enc = Pointnet2ClsMSG(0).set_gemm_mode("tf32")
    assert all(sa.gemm_mode == "tf32" for sa in enc.SA_modules)
    with pytest.raises(ValueError):
        enc.set_gemm_mode("tf16")


def _encoder_layers():
    """(N, K) of every tensor-core GEMM layer of the encoder: the SharedMLP layers of levels 2-5 (plus the padding of
    their first layers' input to 4 columns), the merged first layers, and the level-1 fused scale's layers 2-3"""
    shapes = {(32, 32), (64, 32)}
    cin = sum(m[-1] for m in ClsMSG_CFG_Light["MLPS"][0])
    for mlps in ClsMSG_CFG_Light["MLPS"][1:]:
        k0 = cin + 3
        shapes.add((sum(m[0] for m in mlps), (k0 + 3) // 4 * 4))
        for m in mlps:
            spec = [k0] + list(m)
            shapes.add((spec[1], (k0 + 3) // 4 * 4))
            shapes.update((spec[j + 1], spec[j]) for j in range(1, len(spec) - 1))
        cin = sum(m[-1] for m in mlps)
    return sorted(shapes)


def test_tf32_packed_bytes_equal_split_mode():
    lib = _lib.load()
    shapes = _encoder_layers()
    assert (196, 128) in shapes and (512, 515 + 1) in shapes
    for N, K in shapes:
        assert lib.gp_gemm_packed_bytes(N, K, 2) == lib.gp_gemm_packed_bytes(N, K, 3) > 0, (N, K)
        assert lib.gp_gemm_packed_bytes(N, K, 2) == 2 * lib.gp_gemm_packed_bytes(N, K, 1)
    for npass in (0, 4, -1):
        assert lib.gp_gemm_packed_bytes(128, 64, npass) == 0


FUSED_SPECS = [(32, 32, 64), (64, 64, 128), (64, 96, 128), (128, 196, 256), (256, 256, 512), (256, 384, 512),
               (64, 64, 256), (64, 384, 512)]


def test_tf32_fused_fits_equals_split_mode():
    for spec in FUSED_SPECS + [(256, 384, 512), (252, 384, 512)]:
        for ns in (8, 16, 32):
            assert pu.sa_mlp2_fused_fits(*spec, 2, ns) == pu.sa_mlp2_fused_fits(*spec, 3, ns), (spec, ns)
    assert pu.sa_mlp2_fused_fits(256, 384, 512, 2, 32)


@pytest.mark.parametrize("npass", [0, 4])
def test_c_abi_refuses_bad_npass(npass):
    """Dummy non-null pointers: the entries must refuse before touching the device."""
    lib = _lib.load()
    p = ctypes.c_void_p(256)
    w = (ctypes.c_float * 192)()
    checks = [
        ("gp_gemm_pack", lambda: lib.gp_gemm_pack(p, 128, 64, npass, p, None)),
        ("gp_gemm_bias_relu", lambda: lib.gp_gemm_bias_relu(p, 1024, 64, p, p, 128, 64, npass, p, 128, 0, None, 0, None)),
        ("gp_gemm_linear", lambda: lib.gp_gemm_linear(p, 1024, 64, p, 128, 64, npass, p, 128, None)),
        ("gp_gemm_gather_bias_relu", lambda: lib.gp_gemm_gather_bias_relu(p, 256, 64, p, 1024, 512, p, 64, 32, p, p, 128,
                                                                          64, npass, p, 128, 0, None, 0, None)),
        ("gp_sa_mlp2_fused", lambda: lib.gp_sa_mlp2_fused(p, 256, 64, p, 1024, 512, p, 64, 32, p, p, 64, 64, p, p, 128,
                                                          npass, 32, p, 128, None)),
        ("gp_sa_mlp2_fused_xyz", lambda: lib.gp_sa_mlp2_fused_xyz(p, p, 1024, p, 1024, 512, 32, w, w, p, p, 32, 32, p, p,
                                                                  64, npass, 32, p, 64, None)),
    ]
    for name, fn in checks:
        assert fn() == -1, name
        assert name in _lib.last_error() and "npass must be 1, 2 or 3" in _lib.last_error(), (name, _lib.last_error())

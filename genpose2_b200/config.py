"""The reference's configuration keys (configs/config.py:5-135) with the same names and defaults,
WITHOUT parsing argv at import time (the reference does, from pointnet2.py:28).  `--dino` defaults
to "none" here: the fork's "pointwise" default needs a dinov3 checkout that is not in the tree
(SURVEY.md naming corrections)."""
import argparse


def build_parser():
    p = argparse.ArgumentParser()
    p.add_argument("--data_path", type=str)
    p.add_argument("--batch_size", type=int, default=192)
    p.add_argument("--pose_mode", type=str, default="rot_matrix")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--device", type=str, default="cuda")
    p.add_argument("--num_points", type=int, default=1024)
    p.add_argument("--sampler_mode", nargs="+", default=["ode"])
    p.add_argument("--sampling_steps", type=int)
    p.add_argument("--sde_mode", type=str, default="ve")
    p.add_argument("--regression_head", type=str, default="Rx_Ry_and_T")
    p.add_argument("--pointnet2_params", type=str, default="light")
    p.add_argument("--pts_encoder", type=str, default="pointnet2")
    p.add_argument("--energy_mode", type=str, default="IP")
    p.add_argument("--s_theta_mode", type=str, default="score")
    p.add_argument("--norm_energy", type=str, default="identical")
    p.add_argument("--dino", type=str, default="none")
    p.add_argument("--scale_embedding", type=int, default=180)
    p.add_argument("--agent_type", type=str, default="score")
    p.add_argument("--pretrained_score_model_path", type=str)
    p.add_argument("--pretrained_energy_model_path", type=str)
    p.add_argument("--pretrained_scale_model_path", type=str)
    p.add_argument("--parallel", default=False, action="store_true")
    p.add_argument("--num_gpu", type=int, default=4)
    p.add_argument("--is_train", default=False, action="store_true")
    p.add_argument("--eval", default=False, action="store_true")
    p.add_argument("--pred", default=False, action="store_true")
    p.add_argument("--eval_repeat_num", type=int, default=50)
    p.add_argument("--save_video", default=False, action="store_true")
    p.add_argument("--T0", type=float, default=1.0)
    p.add_argument("--clustering", type=int, default=1)
    p.add_argument("--clustering_eps", type=float, default=0.05)
    p.add_argument("--clustering_minpts", type=float, default=0.1667)
    p.add_argument("--retain_ratio", type=float, default=0.4)
    # not in the reference: numerical mode of the fused MLP kernels (fp32 | fp32_ffma | tf32 | bf16), see scorenet.MLP_MODES
    p.add_argument("--mlp_mode", type=str, default="fp32")
    # not in the reference: operand precision of the encoder's tensor-core SharedMLP GEMMs (auto | bf16x3 | bf16 | tf32);
    # auto follows mlp_mode, see posenet.ENCODER_MODES
    p.add_argument("--encoder_mode", type=str, default="auto")
    # not in the reference: RK45 step-size control shared by the batch (batch) or per object (object), see
    # samplers.STEP_CONTROLS
    p.add_argument("--step_control", type=str, default="batch")
    return p


def get_config(argv=None):
    """argv=None -> defaults only (never reads sys.argv implicitly)."""
    cfg = build_parser().parse_args([] if argv is None else list(argv))
    assert cfg.dino in ["none", "global", "pointwise"]
    return cfg

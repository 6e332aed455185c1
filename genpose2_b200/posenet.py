"""Drop-in for `GFObjectPose` (networks/posenet.py:27-345): same constructor arguments, the same
state-dict keys (`pts_encoder.*`, `pose_score_net.*`) and the same `forward(data, mode, init_x, T0)`
mode dispatcher and `sample(...)` signature.  Accelerated configuration: dino=none,
pts_encoder=pointnet2, sde_mode=ve, pose_mode=rot_matrix, regression_head=Rx_Ry_and_T; anything else
raises NotImplementedError (no fallback / multi-backend dispatch)."""
import torch
import torch.nn as nn

from .pointnet2 import GEMM_NPASS, Pointnet2ClsMSG
from .samplers import cond_ode_sampler, cond_pc_sampler
from .scorenet import PoseEnergyNet, PoseScoreNet

# cfg.encoder_mode: "auto" or a SharedMLP operand precision (pointnet2.GEMM_NPASS).  "auto" follows mlp_mode: fp32,
# fp32_ffma and tf32 -> split-bf16 x3 (fp32-class, 2e-5 of the reference's fp32 features; mlp_mode tf32 runs only the
# trunk in tf32), bf16 -> bf16
ENCODER_MODES = ("auto",) + tuple(GEMM_NPASS)
_AUTO_ENCODER_MODE = {"fp32": "bf16x3", "fp32_ffma": "bf16x3", "tf32": "bf16x3", "bf16": "bf16"}


def encoder_gemm_mode(cfg):
    """The encoder's SharedMLP operand precision for cfg (ValueError for an unknown encoder_mode)."""
    mode = getattr(cfg, "encoder_mode", "auto")
    if mode not in ENCODER_MODES:
        raise ValueError(f"encoder_mode={mode!r}: expected one of {ENCODER_MODES}")
    return _AUTO_ENCODER_MODE[getattr(cfg, "mlp_mode", "fp32")] if mode == "auto" else mode


class GFObjectPose(nn.Module):
    def __init__(self, cfg, prior_fn, marginal_prob_fn, sde_fn, sampling_eps, T):
        super().__init__()
        self.cfg = cfg
        encoder_mode = encoder_gemm_mode(cfg)
        self.device = cfg.device
        self.is_testing = False
        self.prior_fn, self.marginal_prob_fn, self.sde_fn = prior_fn, marginal_prob_fn, sde_fn
        self.sampling_eps, self.T = sampling_eps, T
        if cfg.dino != "none":
            raise NotImplementedError(
                "dino=%r needs the networks/dinov3 checkout that is absent from the reference tree; the "
                "accelerated path covers --dino none (SURVEY.md section 8, row f3)" % cfg.dino)
        if cfg.pts_encoder != "pointnet2":
            raise NotImplementedError("pts_encoder=%r: only pointnet2 is on the accelerated path" % cfg.pts_encoder)
        if getattr(cfg, "pointnet2_params", "light") != "light":
            raise NotImplementedError("pointnet2_params=%r: only 'light' (ClsMSG_CFG_Light)" % cfg.pointnet2_params)
        self.pts_encoder = Pointnet2ClsMSG(0)
        self.pts_encoder.set_gemm_mode(encoder_mode)
        if cfg.agent_type == "score":
            self.pose_score_net = PoseScoreNet(self.marginal_prob_fn, 0, cfg.pose_mode, cfg.regression_head, False)
        elif cfg.agent_type == "energy":
            self.pose_score_net = PoseEnergyNet(
                marginal_prob_func=self.marginal_prob_fn, dino_dim=0, pose_mode=cfg.pose_mode,
                regression_head=cfg.regression_head, energy_mode=cfg.energy_mode,
                s_theta_mode=cfg.s_theta_mode, norm_energy=cfg.norm_energy)
        else:
            raise NotImplementedError(f"agent_type={cfg.agent_type!r}")
        self.pose_score_net.mlp_mode = getattr(cfg, "mlp_mode", "fp32")

    def extract_pts_feature(self, data, geometry=None, return_geometry=False):
        """posenet.py:127-228 with dino=none: pts_encoder(pts) -> [bs,1024]."""
        return self.pts_encoder(data["pts"], geometry=geometry, return_geometry=return_geometry)

    def sample(self, data, sampler, atol=1e-5, rtol=1e-5, snr=0.16, denoise=True, init_x=None, T0=None,
               return_trajectory=True, *, noise_keys=None):
        """posenet.py:230-276.  T0 may be one start time per object and `noise_keys` (not in the reference) int64 [B]
        keys of per-object noise, see samplers.cond_ode_sampler."""
        if sampler == "pc":
            return cond_pc_sampler(
                score_model=self, data=data, prior=self.prior_fn, sde_coeff=self.sde_fn,
                num_steps=self.cfg.sampling_steps, snr=snr, device=self.device, eps=self.sampling_eps,
                pose_mode=self.cfg.pose_mode, init_x=init_x, step_control=getattr(self.cfg, "step_control", "batch"),
                noise_keys=noise_keys)
        if sampler == "ode":
            T0 = self.T if T0 is None else T0
            return cond_ode_sampler(
                score_model=self, data=data, prior=self.prior_fn, sde_coeff=self.sde_fn, atol=atol, rtol=rtol,
                device=self.device, eps=self.sampling_eps, T=T0, num_steps=self.cfg.sampling_steps,
                pose_mode=self.cfg.pose_mode, denoise=denoise, init_x=init_x,
                return_trajectory=return_trajectory, step_control=getattr(self.cfg, "step_control", "batch"),
                noise_keys=noise_keys)
        raise NotImplementedError

    def forward(self, data, mode="score", init_x=None, T0=None, **kw):
        """posenet.py:294-345."""
        if mode == "score":
            return self.pose_score_net(data)
        if mode == "energy":
            return self.pose_score_net(data, return_item="energy")
        if mode == "likelihood":
            raise NotImplementedError("likelihood needs autograd through the net (training/eval only)")
        if mode == "pts_feature":
            return self.extract_pts_feature(data, **kw)
        if mode == "rgb_feature":
            return None  # cfg.dino != "global" (posenet.py:313-315)
        if mode == "pc_sample":
            return self.sample(data, "pc", init_x=init_x, noise_keys=kw.get("noise_keys"))
        if mode == "ode_sample":
            return self.sample(data, "ode", init_x=init_x, T0=T0, **kw)
        raise NotImplementedError

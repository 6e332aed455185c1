"""Drop-in for the `PoseNet` agent (networks/posenet_agent.py:52-823), inference surface:
`pred_func` (:490-584), `get_energy` (:608-705), `pred_scale_func` (:586-606), `load_ckpt`
(:171-203).  Training / evaluation-metric / tensorboard methods are out of scope (SURVEY.md 2).

Same signatures, shapes and dtypes.  Differences that do not change results:
  * nothing is repeated x repeat_num on the host (the reference repeats every dict entry,
    posenet_agent.py:512-520): the kernels index the per-object features by row // repeat_num;
  * `pred_func` may be handed / return the FPS + ball-query geometry so that the energy agent's
    encoder (second pass over the same cloud, posenet_agent.py:636-640) reuses it.
"""
import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .posenet import GFObjectPose
from .rotation import get_rot_matrix, matrix_to_quaternion
from .scalenet import ScaleNet
from .sde import init_sde


class PoseNet(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg
        self.is_testing = False
        self.pts_feature = False
        if getattr(cfg, "is_train", False):
            raise NotImplementedError("training is not on the accelerated path")
        if getattr(cfg, "parallel", False):
            raise NotImplementedError("nn.DataParallel is replaced by one process per GPU (see genpose2_b200.pipeline)")
        self.prior_fn, self.marginal_prob_fn, self.sde_fn, self.sampling_eps, self.T = init_sde(cfg.sde_mode)
        self.net = self.build_net()

    def get_network(self, name):
        if name == "GFObjectPose":
            return GFObjectPose(self.cfg, self.prior_fn, self.marginal_prob_fn, self.sde_fn, self.sampling_eps, self.T)
        if name == "ScaleNet":
            return ScaleNet(self.cfg.num_points, dino_dim=0, embedding_dim=self.cfg.scale_embedding)
        raise NotImplementedError(f"Got name '{name}'")

    def build_net(self):
        net = self.get_network("GFObjectPose" if self.cfg.agent_type != "scale" else "ScaleNet")
        return net.to(self.cfg.device)

    def load_ckpt(self, model_dir, model_path=False, load_model_only=False):
        """posenet_agent.py:171-203 (inference use: model_path=True, load_model_only=True)."""
        if not model_path:
            raise NotImplementedError("load by epoch name is a training-time convenience")
        checkpoint = torch.load(model_dir, map_location=self.cfg.device)
        self.net.load_state_dict(checkpoint["model_state_dict"])
        if not load_model_only:
            raise NotImplementedError("optimizer / scheduler state is training-only")

    # ------------------------------------------------------------------------------------------
    def pred_func(self, data, repeat_num, save_path="./visualization_results", return_average_res=False,
                  init_x: torch.Tensor = None, T0=None, return_process=False, geometry=None,
                  return_geometry=False, pts_feat=None, want_quat=True, *, noise_keys=None):
        """T0: a scalar, or one start time per object (step_control="object"); noise_keys (not in the reference):
        int64 [bs] keys of per-object noise.  See samplers.cond_ode_sampler."""
        self.is_testing = True
        if self.net.training:   # eval() walks every sub-module: only when the flag actually has to change
            self.net.eval()
        if getattr(self.cfg, "save_video", False):
            raise NotImplementedError("save_video (visualisation) is out of scope")
        with torch.no_grad():
            if pts_feat is not None:   # features already extracted by the caller (PosePipeline overlaps the encoders)
                feat = pts_feat
            else:
                feat = self.net(data, mode="pts_feature", geometry=geometry, return_geometry=return_geometry)
                if return_geometry:
                    feat, geometry = feat
            data["pts_feat"] = feat
            data["rgb_feat"] = self.net(data, mode="rgb_feature")  # None
            bs = data["pts"].shape[0]
            self.pts_feature = True
            N = bs * repeat_num
            center = data["pts_center"].to(torch.float32)
            sampler_data = {
                "pts": _RowCount(N),  # the samplers read only data["pts"].shape[0] (samplers.py:196)
                "pts_center": center.unsqueeze(1).expand(bs, repeat_num, 3).reshape(N, 3).contiguous(),
                "_gp_pts_feat_obj": feat,
                "_gp_rows_per_object": repeat_num,
            }
            repeated_init_x = (None if init_x is None
                               else init_x.unsqueeze(1).repeat(1, repeat_num, 1).view(N, -1))
            mode = f"{self.cfg.sampler_mode[0]}_sample"
            kw = {"return_trajectory": bool(return_process)} if mode == "ode_sample" else {}
            if noise_keys is not None:
                kw["noise_keys"] = noise_keys
            in_process_sample, res = self.net(sampler_data, mode=mode, init_x=repeated_init_x, T0=T0, **kw)
            pred_pose = res.reshape(bs, repeat_num, -1)
            in_process_sample = in_process_sample.reshape(bs, repeat_num, in_process_sample.shape[1], -1)
            self.pts_feature = False

            pred_pose_q_wxyz = None
            if want_quat or return_average_res:   # (the runners drop it: `pred_pose, _ = pred_results`)
                resc = _lib.check_cuda(res.contiguous(), "res", torch.float64)
                qt = torch.empty((N, 7), dtype=torch.float64, device=res.device)
                _lib.call("gp_pose_to_quat", _lib.ptr(resc), N, _lib.ptr(qt), device=res.device)
                pred_pose_q_wxyz = qt.reshape(bs, repeat_num, -1)
            extra = (geometry,) if return_geometry else ()
            if return_average_res:
                from .aggregation import _run
                # average_quaternion_batch over all hypotheses + mean translation (posenet_agent.py:561-570)
                ones = torch.zeros((bs, repeat_num, 2), dtype=torch.float32, device=res.device)
                if repeat_num > 64:
                    raise NotImplementedError("return_average_res with more than 64 hypotheses")
                avg, _, _ = _run(pred_pose, ones, repeat_num, False, 0.0, 1)
                avg_q = torch.zeros((bs, 7), device=res.device)
                avg_q[:, :4] = matrix_to_quaternion(avg[:, :3, :3])
                avg_q[:, 4:] = avg[:, :3, 3]
                if return_process:
                    return (pred_pose, pred_pose_q_wxyz, avg_q, in_process_sample) + extra
                return (pred_pose, pred_pose_q_wxyz, avg_q) + extra
            if return_process:
                return [pred_pose, in_process_sample] + list(extra)
            return (pred_pose, pred_pose_q_wxyz) + extra

    def pred_scale_func(self, data):
        """posenet_agent.py:586-606 -> (axes, length [bs,3])."""
        self.is_testing = True
        if self.net.training:   # eval() walks every sub-module: only when the flag actually has to change
            self.net.eval()
        with torch.no_grad():
            pred_len = self.net(data)
        return data["axes"], pred_len

    def energy_prepare(self, pts_feat, pts_center, repeat_num, T):
        """The pose-independent inputs of get_energy(T=T, extract_feature=False) for `data["_gp_energy_pre"]`:
        (per-row centres [N,3], per-row times [N], per-object head projection [B,768])."""
        bs, dev = pts_feat.shape[0], pts_feat.device
        N = bs * repeat_num
        with torch.no_grad():
            t_rows = torch.ones(N, dtype=torch.float32, device=dev) * T
            center = pts_center.to(dev, torch.float32)
            center_rows = center.unsqueeze(1).expand(bs, repeat_num, 3).reshape(N, 3).contiguous()
            proj = self.net.pose_score_net.project(pts_feat)
        return center_rows, t_rows, proj

    def get_energy(self, data, pose_samples, T=None, mode="test", extract_feature=True, geometry=None):
        """posenet_agent.py:608-705 -> energy [bs, repeat_num, 2] f32."""
        if mode != "test":
            raise NotImplementedError("get_energy(mode='train') is training-only")
        self.is_testing = True
        if self.net.training:   # eval() walks every sub-module: only when the flag actually has to change
            self.net.eval()
        bs, repeat_num = pose_samples.shape[0], pose_samples.shape[1]
        with torch.no_grad():
            pts_feat = data["pts_feat"] if not extract_feature else self.net(data, mode="pts_feature", geometry=geometry)
            self.pts_feature = True
            dev = pts_feat.device
            N = bs * repeat_num
            pre = data.get("_gp_energy_pre") if T is not None else None
            if pre is not None:
                pass
            elif T is not None:
                t_rows = torch.ones(N, dtype=torch.float32, device=dev) * T
            else:  # posenet_agent.py:677-687: one random T in [1e-5, 1e-4) per object
                T_samples = torch.randint(int(1e-5 * 1e5), int(1e-4 * 1e5), (bs, 1)).to(dev).type_as(pts_feat) / 1e5
                t_rows = T_samples.repeat([1, repeat_num]).view(N).contiguous()
            net = self.net.pose_score_net
            # what does not depend on the poses may come precomputed (PosePipeline prepares it beside the sampler, on the
            # stream of the energy encoder): the per-row centres and times, the per-object head projection
            if pre is not None:
                center_rows, t_rows, proj = pre
            else:
                center = data["pts_center"].to(dev, torch.float32)
                center_rows = center.unsqueeze(1).expand(bs, repeat_num, 3).reshape(N, 3).contiguous()
                proj = net.project(pts_feat)
            poses = _lib.check_cuda(pose_samples.to(dev, torch.float64).reshape(N, -1).contiguous(), "pose_samples")
            energy = net.energy_from_poses(proj, poses, center_rows, t_rows, repeat_num)
        return energy.reshape(bs, repeat_num, -1)


class _RowCount:
    """Stands in for the x repeat_num copy of `pts` that the reference materialises only to read
    its leading dimension (samplers.py:196)."""

    def __init__(self, n):
        self.shape = (n,)

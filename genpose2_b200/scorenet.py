"""Drop-ins for `PoseScoreNet` (networks/gf_algorithms/scorenet.py:103-275) and `PoseEnergyNet`
(networks/gf_algorithms/energynet.py:32-235) for the configuration on the hot path
(regression_head=Rx_Ry_and_T, pose_mode=rot_matrix, dino=none, energy_mode=IP,
s_theta_mode=score, norm_energy=identical).  Anything else raises NotImplementedError.

The modules own parameters under the reference's state-dict keys; the arithmetic runs in
libgenpose_b200.so on a packed copy of the weights (re-packed automatically when they change).
"""
import ctypes

import numpy as np
import torch
import torch.nn as nn

from . import _lib


# numerical mode of the fused MLP kernels:
#   "fp32"      split-bf16 x3 on the tcgen05 tensor cores (every operand = hi + lo bf16, products accumulated
#               as hi*hi + lo*hi + hi*lo in fp32): fp32-class results (same distance to the reference as a
#               different fp32 summation order)
#   "fp32_ffma" plain FP32 FFMA on the CUDA cores
#   "tf32"      tf32 operands (round to nearest, 11 significand bits) on the tensor cores, fp32 accumulation: 2 MMAs
#               per 16 k instead of 3 (DESIGN 4.6g); weights packed by gp_trunk_pack_tf32
#   "bf16"      bf16 operands on the tensor cores, fp32 accumulation (stated looser bound)
MLP_MODES = {"fp32_ffma": 0, "bf16": 1, "fp32": 2, "tf32": 3}
# shape of the tensor-core evaluator (include/genpose_b200.h, gp_mode_flag): "auto" = one CTA per 128-row tile for
# batches of more than 32 tiles, a 4-CTA cluster per tile below; "solo" / "cluster" force one
EVAL_SHAPES = {"auto": 0, "solo": 16, "cluster": 32, "solo_smem_a": 16 | 64}


def zero_module(module):
    """scorenet.py:15-21"""
    for p in module.parameters():
        p.detach().zero_()
    return module


class GaussianFourierProjection(nn.Module):
    """scorenet.py:77-88 (parameter holder; evaluated inside the kernels)."""

    def __init__(self, embed_dim, scale=30.0):
        super().__init__()
        self.W = nn.Parameter(torch.randn(embed_dim // 2) * scale, requires_grad=False)

    def forward(self, x):
        x_proj = x[:, None] * self.W[None, :] * 2 * np.pi
        return torch.cat([torch.sin(x_proj), torch.cos(x_proj)], dim=-1)


class _Trunk(nn.Module):
    """Shared parameter layout + packing of PoseScoreNet / PoseEnergyNet."""

    def __init__(self, marginal_prob_func, dino_dim, pose_mode, regression_head):
        super().__init__()
        if regression_head != "Rx_Ry_and_T" or pose_mode != "rot_matrix" or dino_dim:
            raise NotImplementedError(
                "accelerated trunk supports regression_head=Rx_Ry_and_T, pose_mode=rot_matrix, dino=none only")
        self.regression_head = regression_head
        self.dino_dim = dino_dim
        self.act = nn.ReLU(True)
        self.pose_encoder = nn.Sequential(nn.Linear(9, 256), self.act, nn.Linear(256, 256), self.act)
        self.t_encoder = nn.Sequential(GaussianFourierProjection(embed_dim=128), nn.Linear(128, 128), self.act)
        for name in ("rot_x", "rot_y", "trans"):
            setattr(self, f"fusion_tail_{name}",
                    nn.Sequential(nn.Linear(128 + 256 + 1024, 256), self.act, zero_module(nn.Linear(256, 3))))
        self.marginal_prob_func = marginal_prob_func
        self.mlp_mode = "fp32"  # see MLP_MODES (set by GFObjectPose from cfg.mlp_mode)
        self.eval_shape = "auto"  # see EVAL_SHAPES
        self._packed = None
        self._packed_key = None

    # ---- packed weights -------------------------------------------------------------------
    def _raw_tensors(self):
        heads = [getattr(self, f"fusion_tail_{n}") for n in ("rot_x", "rot_y", "trans")]
        return ([self.pose_encoder[0].weight, self.pose_encoder[0].bias, self.pose_encoder[2].weight,
                 self.pose_encoder[2].bias, self.t_encoder[0].W, self.t_encoder[1].weight, self.t_encoder[1].bias],
                heads)

    def packed(self):
        """Device blob in the layout of csrc/trunk.cuh (gp_trunk_pack_tf32's for mlp_mode "tf32"); rebuilt when any
        parameter or the kind of blob was modified."""
        self.mode_arg()   # an unsupported mode / shape pair raises before any device work
        base, heads = self._raw_tensors()
        tensors = base + [t for h in heads for t in (h[0].weight, h[0].bias, h[2].weight, h[2].bias)]
        pack = "gp_trunk_pack_tf32" if self.mlp_mode == "tf32" else "gp_trunk_pack"
        key = (pack,) + tuple((t.data_ptr(), t._version) for t in tensors)
        if self._packed is None or key != self._packed_key:
            dev = tensors[0].device
            if dev.type != "cuda":
                raise RuntimeError("the accelerated trunk needs its parameters on a CUDA device (no CPU path)")
            keep = [t.detach().to(torch.float32).contiguous() for t in tensors]
            p = _lib.TrunkParams()
            (p.pose_w0, p.pose_b0, p.pose_w1, p.pose_b1, p.fourier_w, p.t_w, p.t_b) = [t.data_ptr() for t in keep[:7]]
            for h in range(3):
                w0, b0, w1, b1 = keep[7 + 4 * h: 11 + 4 * h]
                p.head_w0[h], p.head_b0[h], p.head_w1[h], p.head_b1[h] = (
                    w0.data_ptr(), b0.data_ptr(), w1.data_ptr(), b1.data_ptr())
            nbytes = _lib.load().gp_trunk_packed_bytes()
            blob = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
            _lib.call(pack, ctypes.byref(p), _lib.ptr(blob), device=dev)
            self._packed, self._packed_key = blob, key
        return self._packed

    def mode_arg(self):
        """the `mode` argument of the C entries: arithmetic | evaluator-shape flag"""
        m = MLP_MODES[self.mlp_mode]
        if self.mlp_mode == "tf32" and self.eval_shape == "solo_smem_a":
            raise ValueError("mlp_mode='tf32' runs with the A operand in tensor memory only: eval_shape='solo_smem_a' "
                             "is not supported")
        return m | (EVAL_SHAPES[self.eval_shape] if m else 0)

    def project(self, pts_feat):
        """Per-object hoisted head projection [B,768] (gp_trunk_project)."""
        pts_feat = _lib.check_cuda(pts_feat.contiguous(), "pts_feat", torch.float32)
        B = pts_feat.shape[0]
        proj = torch.empty((B, 768), dtype=torch.float32, device=pts_feat.device)
        _lib.call("gp_trunk_project", _lib.ptr(self.packed()), _lib.ptr(pts_feat), B, _lib.ptr(proj),
                  device=pts_feat.device)
        return proj


def _object_features(data, n_rows):
    """(pts_feat per object [B,1024], rows_per_object).  The reference repeats every dict entry
    x repeat_num (posenet_agent.py:512-520); callers that know the repeat pass the un-repeated
    features as data["_gp_pts_feat_obj"] + data["_gp_rows_per_object"], anything else is handled
    as one object per row."""
    if "_gp_pts_feat_obj" in data and data["_gp_pts_feat_obj"] is not None:
        rpo = int(data["_gp_rows_per_object"])
        feat = data["_gp_pts_feat_obj"]
        if feat.shape[0] * rpo != n_rows:
            raise ValueError("_gp_pts_feat_obj / _gp_rows_per_object inconsistent with the batch")
        return feat, rpo
    return data["pts_feat"], 1


class PoseScoreNet(_Trunk):
    def __init__(self, marginal_prob_func, dino_dim, pose_mode="quat_wxyz", regression_head="RT",
                 per_point_feature=False):
        if per_point_feature:
            raise NotImplementedError("per_point_feature is a dead branch in the reference (scorenet.py:240)")
        super().__init__(marginal_prob_func, dino_dim, pose_mode, regression_head)
        self.per_point_feature = per_point_feature

    def forward(self, data):
        """scorenet.py:215-275: data{pts_feat [N,1024], sampled_pose [N,9], t [N,1]} -> score [N,9]."""
        x = data["sampled_pose"]
        N = x.shape[0]
        feat, rpo = _object_features(data, N)
        proj = self.project(feat)
        x = _lib.check_cuda(x.to(torch.float32).contiguous(), "sampled_pose", torch.float32)
        t = data["t"].reshape(-1).to(torch.float32).contiguous()
        out = torch.empty((N, 9), dtype=torch.float32, device=x.device)
        _lib.call("gp_scorenet_eval", _lib.ptr(self.packed()), _lib.ptr(proj), _lib.ptr(x), _lib.ptr(t), N, rpo,
                  _lib.ptr(out), self.mode_arg(), device=x.device)
        return out


class PoseEnergyNet(_Trunk):
    def __init__(self, marginal_prob_func, dino_dim, pose_mode="quat_wxyz", regression_head="Rx_Ry_and_T",
                 energy_mode="IP", s_theta_mode="score", norm_energy="identical"):
        if (energy_mode, s_theta_mode, norm_energy) != ("IP", "score", "identical"):
            raise NotImplementedError("accelerated energy net supports energy_mode=IP, s_theta_mode=score, "
                                      "norm_energy=identical only")
        super().__init__(marginal_prob_func, dino_dim, pose_mode, regression_head)
        self.energy_mode, self.s_theta_mode, self.norm_energy = energy_mode, s_theta_mode, norm_energy

    def energy_from_poses(self, proj, poses_f64, pts_center, t_rows, rows_per_object):
        """gp_energy: poses [N,9] f64 in the camera frame, centre subtracted inside the kernel."""
        N = poses_f64.shape[0]
        out = torch.empty((N, 2), dtype=torch.float32, device=poses_f64.device)
        _lib.call("gp_energy", _lib.ptr(self.packed()), _lib.ptr(proj), _lib.ptr(poses_f64), _lib.ptr(pts_center),
                  _lib.ptr(t_rows), N, int(rows_per_object), _lib.ptr(out), self.mode_arg(),
                  device=poses_f64.device)
        return out

    def forward(self, data, return_item="score"):
        """energynet.py:211-235; only return_item="energy" is on the inference path (the score /
        likelihood branches need autograd through the net and are training-time)."""
        if return_item != "energy":
            raise NotImplementedError("PoseEnergyNet: only return_item='energy' is accelerated")
        x = data["sampled_pose"]
        N = x.shape[0]
        feat, rpo = _object_features(data, N)
        proj = self.project(feat)
        zeros = torch.zeros((N, 3), dtype=torch.float32, device=x.device)
        t = data["t"].reshape(-1).to(torch.float32).contiguous()
        return self.energy_from_poses(proj, x.to(torch.float64).contiguous(), zeros, t, rpo)

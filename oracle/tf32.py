"""The trunk of oracle/pose_oracle.py with the operands of its tensor-core products rounded to tf32: the arithmetic the
library's mlp_mode "tf32" (trunk mode 3) implements, restated in numpy / float64.

Rounded (what the tensor cores multiply): x . W1^T, h1 . W2^T and h2 . W_head[:, pose_feat columns]^T, activations
and weights alike.  Left in fp32: the per-object projection (pts_feat columns), the t-branch and the 256 -> 3 output
layers, which the kernels evaluate on the CUDA cores.  Products are accumulated in float64.  Using TF32Trunk instead of
pose_oracle.Trunk is the opt-in; pose_oracle.Trunk stays the fp32 reference."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import pose_oracle as po


def tf32_round(a):
    """cvt.rna.tf32.f32 restated: float32 -> the nearest value with 10 explicit significand bits, rounding to nearest
    on the 13 dropped bits with ties away from zero (add half of the dropped range to the magnitude bits, then
    truncate; the sign bit is untouched).  Finite values that round past the largest float32 become +-inf.  Returns
    float32 of the same shape."""
    a = np.asarray(a, dtype=np.float32)
    b = np.ascontiguousarray(a).view(np.uint32)
    b = np.where(np.isfinite(a), b + np.uint32(0x1000), b) & np.uint32(0xFFFFE000)
    return b.astype(np.uint32).view(np.float32).reshape(a.shape)


def _r64(t):
    """torch float32 tensor -> its tf32 rounding as float64 numpy"""
    return tf32_round(t.detach().cpu().numpy()).astype(np.float64)


class TF32Trunk(po.Trunk):
    """pose_oracle.Trunk evaluated as mlp_mode "tf32" does (module docstring); score() / energy() follow."""

    def f_theta(self, pts_feat, sampled_pose, t):
        tt = t.squeeze(1)
        x_proj = tt[:, None] * self.four_w[None, :] * 2 * np.pi  # scorenet.py:87
        four = torch.cat([torch.sin(x_proj), torch.cos(x_proj)], dim=-1)
        t_feat = torch.relu(F.linear(four, self.t_w, self.t_b)).double().numpy()
        f64 = lambda v: v.detach().double().numpy()
        h1 = np.maximum(_r64(sampled_pose.float()) @ _r64(self.pose_w0).T + f64(self.pose_b0), 0.0)
        h1 = torch.from_numpy(h1.astype(np.float32))   # the epilogue rounds relu(acc + b) from fp32
        h2 = np.maximum(_r64(h1) @ _r64(self.pose_w1).T + f64(self.pose_b1), 0.0)
        h2 = torch.from_numpy(h2.astype(np.float32))
        feat = f64(pts_feat)
        outs = []
        for w0, b0, w1, b1 in self.heads:
            pre = (feat @ f64(w0[:, :1024]).T + f64(b0) + t_feat @ f64(w0[:, 1024:1152]).T
                   + _r64(h2) @ _r64(w0[:, 1152:]).T)
            outs.append(np.maximum(pre, 0.0) @ f64(w1).T + f64(b1))
        return torch.from_numpy(np.concatenate(outs, axis=1).astype(np.float32)), po.ve_marginal_std(t)

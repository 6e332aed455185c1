"""Drop-in for networks/pts_encoder/pointnet2_utils/pointnet2/pointnet2_utils.py (inference side).

Same names, argument order, dtypes and shapes as the reference (`furthest_point_sample`,
`gather_operation`, `ball_query`, `grouping_operation`, `QueryAndGroup`, `GroupAll`), backed by
libgenpose_b200.so.  Indices are bit-exact with the reference extension.  Backward passes are out
of scope (training is not on the hot path) and raise.
"""
from typing import Tuple

import torch
import torch.nn as nn

from . import _lib


def furthest_point_sample(xyz: torch.Tensor, npoint: int) -> torch.Tensor:
    """pointnet2_utils.py:16-37.  xyz (B, N, 3) f32 -> (B, npoint) int32."""
    assert xyz.is_contiguous()
    _lib.check_cuda(xyz, "xyz", torch.float32)
    B, N, _ = xyz.size()
    output = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
    _lib.call("gp_fps", _lib.ptr(xyz), B, N, int(npoint), _lib.ptr(output), None, device=xyz.device)
    return output


def furthest_point_sample_gather(xyz: torch.Tensor, npoint: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """FPS fused with the gather of pointnet2_modules.py:43-47: returns (idx, new_xyz (B,npoint,3))."""
    assert xyz.is_contiguous()
    _lib.check_cuda(xyz, "xyz", torch.float32)
    B, N, _ = xyz.size()
    idx = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
    new_xyz = torch.empty((B, npoint, 3), dtype=torch.float32, device=xyz.device)
    _lib.call("gp_fps", _lib.ptr(xyz), B, N, int(npoint), _lib.ptr(idx), _lib.ptr(new_xyz), device=xyz.device)
    return idx, new_xyz


def furthest_point_sample_chain(xyz: torch.Tensor, npoint: int, tie_free: torch.Tensor = None):
    """FPS + gather for a cascade of levels (gp_fps_chain): returns (idx, new_xyz, tie_free_out).

    `tie_free` must be the third result of the call that PRODUCED `xyz` (i.e. xyz is the previous level's new_xyz, in
    FPS order); objects whose earlier sampling was tie-free for at least `npoint` steps get the prefix
    0..npoint-1, which is what sampling them again would return -- bit-exact, tested against the reference ext.
    Pass None for the first level."""
    assert xyz.is_contiguous()
    _lib.check_cuda(xyz, "xyz", torch.float32)
    B, N, _ = xyz.size()
    idx = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
    new_xyz = torch.empty((B, npoint, 3), dtype=torch.float32, device=xyz.device)
    out = torch.empty((B,), dtype=torch.int32, device=xyz.device)
    if tie_free is not None:
        _lib.check_cuda(tie_free, "tie_free", torch.int32)
        assert tie_free.numel() == B
    _lib.call("gp_fps_chain", _lib.ptr(xyz), B, N, int(npoint), _lib.ptr(idx), _lib.ptr(new_xyz),
              _lib.ptr(tie_free), _lib.ptr(out), device=xyz.device)
    return idx, new_xyz, out


def gather_operation(features: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """pointnet2_utils.py:50-72.  features (B, C, N), idx (B, npoint) -> (B, C, npoint)."""
    assert features.is_contiguous()
    assert idx.is_contiguous()
    _lib.check_cuda(features, "features", torch.float32)
    _lib.check_cuda(idx, "idx", torch.int32)
    B, npoint = idx.size()
    _, C, N = features.size()
    output = torch.empty((B, C, npoint), dtype=torch.float32, device=features.device)
    _lib.call("gp_gather", _lib.ptr(features), _lib.ptr(idx), B, C, N, npoint, _lib.ptr(output),
              device=features.device)
    return output


def ball_query(radius: float, nsample: int, xyz: torch.Tensor, new_xyz: torch.Tensor) -> torch.Tensor:
    """pointnet2_utils.py:229-253.  -> idx (B, npoint, nsample) int32."""
    assert new_xyz.is_contiguous()
    assert xyz.is_contiguous()
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    B, N, _ = xyz.size()
    npoint = new_xyz.size(1)
    idx = torch.empty((B, npoint, nsample), dtype=torch.int32, device=xyz.device)
    _lib.call("gp_ball_query", _lib.ptr(new_xyz), _lib.ptr(xyz), B, N, npoint, float(radius), int(nsample),
              _lib.ptr(idx), device=xyz.device)
    return idx


def ball_query2(radii, nsamples, xyz: torch.Tensor, new_xyz: torch.Tensor):
    """Both radii of an MSG level in one scan of the cloud -> (idx0, idx1)."""
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    B, N, _ = xyz.size()
    npoint = new_xyz.size(1)
    idx0 = torch.empty((B, npoint, nsamples[0]), dtype=torch.int32, device=xyz.device)
    idx1 = torch.empty((B, npoint, nsamples[1]), dtype=torch.int32, device=xyz.device)
    _lib.call("gp_ball_query2", _lib.ptr(new_xyz), _lib.ptr(xyz), B, N, npoint, float(radii[0]),
              int(nsamples[0]), _lib.ptr(idx0), float(radii[1]), int(nsamples[1]), _lib.ptr(idx1),
              device=xyz.device)
    return idx0, idx1


def ball_query2_tails(radii, nsamples, xyz: torch.Tensor, new_xyz: torch.Tensor, shift: torch.Tensor, tail_absolute: bool):
    """ball_query2 plus the encoder's per-centre by-products from the same launch (gp_ball_query2_tails):
    returns ((idx0, idx1), rel [B,M,3] = new_xyz - shift, tail [B,M,4] = [rel | 0] or [new_xyz | 0])."""
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    _lib.check_cuda(shift, "shift", torch.float32)
    B, N, _ = xyz.size()
    npoint = new_xyz.size(1)
    assert shift.numel() == 3 * B
    idx0 = torch.empty((B, npoint, nsamples[0]), dtype=torch.int32, device=xyz.device)
    idx1 = torch.empty((B, npoint, nsamples[1]), dtype=torch.int32, device=xyz.device)
    rel = torch.empty((B, npoint, 3), dtype=torch.float32, device=xyz.device)
    tail = torch.empty((B, npoint, 4), dtype=torch.float32, device=xyz.device)
    _lib.call("gp_ball_query2_tails", _lib.ptr(new_xyz), _lib.ptr(xyz), B, N, npoint, float(radii[0]),
              int(nsamples[0]), _lib.ptr(idx0), float(radii[1]), int(nsamples[1]), _lib.ptr(idx1),
              _lib.ptr(shift), _lib.ptr(rel), _lib.ptr(tail), int(bool(tail_absolute)), device=xyz.device)
    return (idx0, idx1), rel, tail


def grouping_operation(features: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """pointnet2_utils.py:179-203.  features (B, C, N), idx (B, npoint, nsample) -> (B, C, npoint, nsample)."""
    assert features.is_contiguous()
    assert idx.is_contiguous()
    _lib.check_cuda(features, "features", torch.float32)
    _lib.check_cuda(idx, "idx", torch.int32)
    B, nfeatures, nsample = idx.size()
    _, C, N = features.size()
    output = torch.empty((B, C, nfeatures, nsample), dtype=torch.float32, device=features.device)
    _lib.call("gp_group", _lib.ptr(features), _lib.ptr(idx), B, C, N, nfeatures, nsample, _lib.ptr(output),
              device=features.device)
    return output


def query_group(xyz, new_xyz, features, idx) -> torch.Tensor:
    """Fused tail of QueryAndGroup.forward (pointnet2_utils.py:279-296): (B, 3 + C, npoint, nsample)."""
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    _lib.check_cuda(idx, "idx", torch.int32)
    B, N, _ = xyz.size()
    _, M, ns = idx.size()
    C = 0
    if features is not None:
        _lib.check_cuda(features, "features", torch.float32)
        C = features.size(1)
    out = torch.empty((B, 3 + C, M, ns), dtype=torch.float32, device=xyz.device)
    _lib.call("gp_query_group", _lib.ptr(xyz), _lib.ptr(new_xyz), _lib.ptr(features), _lib.ptr(idx), B, C, N, M,
              ns, _lib.ptr(out), device=xyz.device)
    return out


def group_rows(xyz, new_xyz, feat_cl, idx, pad_to=1) -> torch.Tensor:
    """Channels-last QueryAndGroup tail: one row per (centre, sample): [B*M*ns, ld] with
    row = [xyz[idx] - new_xyz | feat_cl[idx] | zeros]; feat_cl is [B, N, C] (channels last) or None;
    ld = 3 + C rounded up to a multiple of `pad_to`."""
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    _lib.check_cuda(idx, "idx", torch.int32)
    B, N, _ = xyz.size()
    _, M, ns = idx.size()
    C = 0
    if feat_cl is not None:
        _lib.check_cuda(feat_cl, "feat_cl", torch.float32)
        C = feat_cl.size(2)
    ld = (3 + C + pad_to - 1) // pad_to * pad_to
    out = torch.empty((B * M * ns, ld), dtype=torch.float32, device=xyz.device)
    _lib.call("gp_group_rows", _lib.ptr(xyz), _lib.ptr(new_xyz), _lib.ptr(feat_cl), _lib.ptr(idx), B, C, N, M, ns,
              ld, _lib.ptr(out), device=xyz.device)
    return out


def maxpool_rows(h, groups, nsample, out=None):
    """max over the `nsample` consecutive rows of each group: h [groups*nsample, C] -> out [groups, C]
    (`out` may be a column slice of a wider row-major tensor: both MSG scales land in one tensor)."""
    _lib.check_cuda(h, "h", torch.float32)
    C = h.size(1)
    if out is None:
        out = torch.empty((groups, C), dtype=torch.float32, device=h.device)
    if out.stride(-1) != 1 or out.dtype != torch.float32:
        raise ValueError("out must be float32 with unit inner stride")
    _lib.call("gp_maxpool_rows", _lib.ptr(h), int(groups), int(nsample), C, int(out.stride(-2)), _lib.ptr(out),
              device=h.device)
    return out


def sa_small_mlp(xyz, new_xyz, idx, layers, out):
    """Fused first-level scale (no point features): grouping -> 3-layer SharedMLP -> max-pool, written into
    `out` [B*M, >= C3] (may be a column slice).  `layers` = [(W [Cout,Cin], b [Cout])] x 3, BatchNorm folded."""
    import ctypes
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    _lib.check_cuda(idx, "idx", torch.int32)
    B, N, _ = xyz.size()
    _, M, ns = idx.size()
    ws = (ctypes.c_void_p * 3)(*[w.data_ptr() for w, _ in layers])
    bs = (ctypes.c_void_p * 3)(*[b.data_ptr() for _, b in layers])
    C1, C2, C3 = (w.shape[0] for w, _ in layers)
    _lib.call("gp_sa_small_mlp", _lib.ptr(xyz), _lib.ptr(new_xyz), _lib.ptr(idx), B, N, M, ns, ws, bs, C1, C2, C3,
              _lib.ptr(out), int(out.stride(-2)), device=xyz.device)
    return out


def sa_small_mlp_hostw(xyz, new_xyz, idx, host_layers, out, tail=None, tail_col=0):
    """sa_small_mlp with HOST copies of the folded weights (gp_sa_small_mlp_hostw): they travel in the launch's
    parameter space and the kernel reads them as constant operands.  `host_layers` = [(W, b)] x 3, CPU fp32.
    tail [B,M,4] (optional): also copied to out[..., tail_col : tail_col + 4] (gp_sa_small_mlp_hostw_tail)."""
    import ctypes
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    _lib.check_cuda(idx, "idx", torch.int32)
    for w, b in host_layers:
        if w.is_cuda or b.is_cuda or w.dtype != torch.float32 or not w.is_contiguous() or not b.is_contiguous():
            raise TypeError("host_layers must be contiguous fp32 CPU tensors")
    B, N, _ = xyz.size()
    _, M, ns = idx.size()
    ws = (ctypes.c_void_p * 3)(*[w.data_ptr() for w, _ in host_layers])
    bs = (ctypes.c_void_p * 3)(*[b.data_ptr() for _, b in host_layers])
    C1, C2, C3 = (w.shape[0] for w, _ in host_layers)
    if tail is not None:
        _lib.check_cuda(tail, "tail", torch.float32)
        _lib.call("gp_sa_small_mlp_hostw_tail", _lib.ptr(xyz), _lib.ptr(new_xyz), _lib.ptr(idx), B, N, M, ns, ws, bs, C1, C2,
                  C3, _lib.ptr(out), int(out.stride(-2)), _lib.ptr(tail), int(tail_col), device=xyz.device)
        return out
    _lib.call("gp_sa_small_mlp_hostw", _lib.ptr(xyz), _lib.ptr(new_xyz), _lib.ptr(idx), B, N, M, ns, ws, bs, C1, C2, C3,
              _lib.ptr(out), int(out.stride(-2)), device=xyz.device)
    return out


def ctypes_ptr(host_tensor):
    """Pointer to a CPU tensor's storage (host-side operands that travel in a launch's parameter space)."""
    import ctypes
    return ctypes.c_void_p(host_tensor.data_ptr())


def zeros(shape, device):
    """A zero-filled fp32 tensor through a stream-ordered memset (gp_zero), not a fill kernel."""
    t = torch.empty(shape, dtype=torch.float32, device=device)
    _lib.call("gp_zero", _lib.ptr(t), t.numel() * 4, device=t.device)
    return t


def gemm_pack(weight: torch.Tensor, npass: int) -> torch.Tensor:
    """Pack W [N, K] fp32 into the pre-swizzled bf16 (npass=1) / bf16 hi+lo (npass=3) / tf32 k 0..31 + k 32..63
    (npass=2, rounded to nearest tf32) chunk images the tcgen05 GEMM streams with TMA (gp_gemm_pack).  Do once per
    checkpoint."""
    w = _lib.check_cuda(weight.detach().to(torch.float32).contiguous(), "weight", torch.float32)
    N, K = w.shape
    nbytes = _lib.load().gp_gemm_packed_bytes(N, K, npass)
    packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
    _lib.call("gp_gemm_pack", _lib.ptr(w), N, K, npass, _lib.ptr(packed), device=w.device)
    return packed


def gemm_bias_relu(x, packed, bias, N, K, npass, pool_ns=0, pooled_out=None):
    """relu(x @ W^T + bias) on the tensor cores (gp_gemm_bias_relu).  x [R, ldx] fp32 with ldx % 4 == 0.
    pool_ns == 0 -> returns y [R, round_up(N, 32)] (columns >= N are zero);
    pool_ns  > 0 -> max over each pool_ns consecutive rows into `pooled_out` (zero-initialised,
    [R / pool_ns, >= N] row-major, may be a column slice) and returns it."""
    _lib.check_cuda(x, "x", torch.float32, rows=True)    # may be a column slice of a wider row-major matrix
    R, ldx = x.shape[0], int(x.stride(0))
    if pool_ns:
        if pooled_out is None:
            pooled_out = torch.zeros((R // pool_ns, N), dtype=torch.float32, device=x.device)
        _lib.call("gp_gemm_bias_relu", _lib.ptr(x), R, ldx, _lib.ptr(packed), _lib.ptr(bias), N, K, npass, None, 0,
                  int(pool_ns), _lib.ptr(pooled_out), int(pooled_out.stride(-2)), device=x.device)
        return pooled_out
    ldy = (N + 31) // 32 * 32
    y = torch.empty((R, ldy), dtype=torch.float32, device=x.device)
    _lib.call("gp_gemm_bias_relu", _lib.ptr(x), R, ldx, _lib.ptr(packed), _lib.ptr(bias), N, K, npass, _lib.ptr(y), ldy,
              0, None, 0, device=x.device)
    return y


def gemm_linear(x, packed, N, K, npass):
    """x @ W^T on the tensor cores, no bias / activation (gp_gemm_linear): [R, round_up(N, 32)]."""
    _lib.check_cuda(x, "x", torch.float32)
    R, ldx = x.shape
    ldy = (N + 31) // 32 * 32
    y = torch.empty((R, ldy), dtype=torch.float32, device=x.device)
    _lib.call("gp_gemm_linear", _lib.ptr(x), R, ldx, _lib.ptr(packed), N, K, npass, _lib.ptr(y), ldy, device=x.device)
    return y


def gemm_gather_bias_relu(P, n_src, gidx, rows_per_batch, Q, q_ns, packed, bias, N, K, npass, pool_ns=0,
                          pooled_out=None):
    """relu(relu(P[batch * n_src + gidx] - Q[row // q_ns]) @ W^T + bias)  (gp_gemm_gather_bias_relu)."""
    _lib.check_cuda(P, "P", torch.float32, rows=True)
    _lib.check_cuda(Q, "Q", torch.float32, rows=True)
    _lib.check_cuda(gidx, "gidx", torch.int32)
    R = gidx.numel()
    if pool_ns:
        _lib.call("gp_gemm_gather_bias_relu", _lib.ptr(P), int(n_src), int(P.stride(0)), _lib.ptr(gidx), R,
                  int(rows_per_batch), _lib.ptr(Q), int(Q.stride(0)), int(q_ns), _lib.ptr(packed), _lib.ptr(bias), N, K,
                  npass, None, 0, int(pool_ns), _lib.ptr(pooled_out), int(pooled_out.stride(-2)), device=P.device)
        return pooled_out
    ldy = (N + 31) // 32 * 32
    y = torch.empty((R, ldy), dtype=torch.float32, device=P.device)
    _lib.call("gp_gemm_gather_bias_relu", _lib.ptr(P), int(n_src), int(P.stride(0)), _lib.ptr(gidx), R,
              int(rows_per_batch), _lib.ptr(Q), int(Q.stride(0)), int(q_ns), _lib.ptr(packed), _lib.ptr(bias), N, K,
              npass, _lib.ptr(y), ldy, 0, None, 0, device=P.device)
    return y


def centre_term(new_xyz_rows, w0_xyz_t, b0, ldq, tail=None, tail_dst=None):
    """Q [rows, ldq]: per-centre term  new_xyz @ W0_xyz^T - b0  of a hoisted first layer, zero-padded (gp_centre_term).
    With tail [rows,4] and tail_dst (a 4-column slice of the level buffer) the same launch copies the tail rows
    (gp_centre_term_tail)."""
    _lib.check_cuda(new_xyz_rows, "new_xyz", torch.float32)
    rows, c1 = new_xyz_rows.shape[0], w0_xyz_t.shape[1]
    Q = torch.empty((rows, ldq), dtype=torch.float32, device=new_xyz_rows.device)
    if tail is not None:
        _lib.check_cuda(tail, "tail", torch.float32)
        assert tail_dst.shape[-1] == 4 and tail_dst.stride(-1) == 1 and tail.numel() == rows * 4
        _lib.call("gp_centre_term_tail", _lib.ptr(new_xyz_rows), rows, _lib.ptr(w0_xyz_t), _lib.ptr(b0), int(c1), _lib.ptr(Q),
                  int(ldq), _lib.ptr(tail), _lib.ptr(tail_dst), int(tail_dst.stride(-2)), device=new_xyz_rows.device)
        return Q
    _lib.call("gp_centre_term", _lib.ptr(new_xyz_rows), rows, _lib.ptr(w0_xyz_t), _lib.ptr(b0), int(c1), _lib.ptr(Q),
              int(ldq), device=new_xyz_rows.device)
    return Q


def sa_mlp2_fused(P, n_src, gidx, rows_per_batch, Q, q_ns, packed1, bias1, c1, c2, packed2, bias2, c3, npass, pool_ns,
                  pooled_out):
    """pooled_out[g] = max_rows relu(relu(relu(P[gather] - Q) @ W1^T + b1) @ W2^T + b2)  (gp_sa_mlp2_fused):
    the last two SharedMLP layers of a scale and its max-pool without materialising any (centre, sample) matrix."""
    _lib.check_cuda(P, "P", torch.float32, rows=True)
    _lib.check_cuda(Q, "Q", torch.float32, rows=True)
    _lib.check_cuda(gidx, "gidx", torch.int32)
    _lib.call("gp_sa_mlp2_fused", _lib.ptr(P), int(n_src), int(P.stride(0)), _lib.ptr(gidx), gidx.numel(),
              int(rows_per_batch), _lib.ptr(Q), int(Q.stride(0)), int(q_ns), _lib.ptr(packed1), _lib.ptr(bias1), int(c1),
              int(c2), _lib.ptr(packed2), _lib.ptr(bias2), int(c3), int(npass), int(pool_ns), _lib.ptr(pooled_out),
              int(pooled_out.stride(-2)), device=P.device)
    return pooled_out


def sa_mlp2_fused_xyz(xyz, new_xyz, bq_idx, w0, b0, packed1, bias1, c1, c2, packed2, bias2, c3, npass, pooled_out):
    """A feature-less scale (first level) on the fused tensor-core kernel (gp_sa_mlp2_fused_xyz): the K = 3 first layer
    relu(W0 . (xyz[idx] - new_xyz) + b0) is evaluated in the operand loader, layers 2, 3 and the max-pool as sa_mlp2_fused.
    xyz [B,N,3], new_xyz [B,M,3], bq_idx [B,M,ns]; w0 [c1,3], b0 [c1]: HOST copies of the folded first layer."""
    _lib.check_cuda(xyz, "xyz", torch.float32)
    _lib.check_cuda(new_xyz, "new_xyz", torch.float32)
    _lib.check_cuda(bq_idx, "bq_idx", torch.int32)
    for t in (w0, b0):
        if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise TypeError("w0 / b0 must be contiguous fp32 CPU tensors (they travel in the launch's parameter space)")
    B, N, _ = xyz.shape
    _, M, ns = bq_idx.shape
    _lib.call("gp_sa_mlp2_fused_xyz", _lib.ptr(xyz), _lib.ptr(new_xyz), int(N), _lib.ptr(bq_idx), bq_idx.numel(), int(M * ns),
              int(ns), ctypes_ptr(w0), ctypes_ptr(b0), _lib.ptr(packed1), _lib.ptr(bias1), int(c1), int(c2), _lib.ptr(packed2),
              _lib.ptr(bias2), int(c3), int(npass), int(ns), _lib.ptr(pooled_out), int(pooled_out.stride(-2)),
              device=xyz.device)
    return pooled_out


def sa_mlp2_fused_fits(c1, c2, c3, npass, pool_ns):
    """Shapes the fused kernel takes (the plan of csrc/sa_fused.cu): H = relu(layer 2) lives in tensor memory as packed
    bf16 (32 columns per 64-wide k-atom, hi + lo in split mode; tf32: 64 columns per k-atom) next to at least 128
    accumulator columns, and the gathered A operand plus a ring of at least two weight chunks (hi + lo, or the two tf32
    images) must fit in shared memory."""
    if c1 % 4 or c1 > 256 or c2 > 384 or c3 > 512 or pool_ns not in (8, 16, 32):
        return False
    images = 1 if npass == 1 else 2
    if 512 - ((c2 + 63) // 64) * 32 * images < 128:
        return False
    return images * ((c1 + 63) // 64) * 16384 + 2 * images * 16384 + 2048 + 1536 <= 227 * 1024


class QueryAndGroup(nn.Module):
    """pointnet2_utils.py:259-298."""

    def __init__(self, radius: float, nsample: int, use_xyz: bool = True):
        super().__init__()
        self.radius, self.nsample, self.use_xyz = radius, nsample, use_xyz

    def forward(self, xyz: torch.Tensor, new_xyz: torch.Tensor, features: torch.Tensor = None):
        idx = ball_query(self.radius, self.nsample, xyz, new_xyz)
        if features is not None and not self.use_xyz:
            return grouping_operation(features, idx)
        assert self.use_xyz, "Cannot have not features and not use xyz as a feature!"
        return query_group(xyz, new_xyz, features, idx)


class GroupAll(nn.Module):
    """pointnet2_utils.py:301-328 (pure views/concat, no kernel needed)."""

    def __init__(self, use_xyz: bool = True):
        super().__init__()
        self.use_xyz = use_xyz

    def forward(self, xyz: torch.Tensor, new_xyz: torch.Tensor, features: torch.Tensor = None):
        grouped_xyz = xyz.transpose(1, 2).unsqueeze(2)
        if features is not None:
            grouped_features = features.unsqueeze(2)
            if self.use_xyz:
                return torch.cat([grouped_xyz, grouped_features], dim=1)
            return grouped_features
        return grouped_xyz

"""Drop-in for `Pointnet2ClsMSG` (networks/pts_encoder/pointnet2.py:211-252) with the
`ClsMSG_CFG_Light` configuration (pointnet2.py:77-89) and its set-abstraction module
(pointnet2_utils/pointnet2/pointnet2_modules.py:19-74, 77-121).

The module tree reproduces the reference's state-dict keys exactly
(`SA_modules.{k}.mlps.{i}.layer{j}.conv.weight`, `...bn.bn.{weight,bias,running_mean,running_var}`)
so reference checkpoints load with `load_state_dict`.

FPS, gather, ball query and grouping run on the hand-written kernels (libgenpose_b200.so): one
fused FPS+gather launch, one two-radius ball query and one fused query-and-group per scale per
level, instead of the reference's FPS, 3 gathers / transposes, 2 ball queries and 4 groupings.
The geometry (FPS / ball-query indices) depends on xyz only, so `forward` can return it and accept
it back: the score and the energy encoder see the same cloud and share one geometry pass.

The per-scale SharedMLP (conv1x1 + BatchNorm(eval) + ReLU, pytorch_utils.py:5-33) is row f1 of SURVEY.md
section 8: BatchNorm is folded into the weights once per checkpoint, activations are channels-last (one GEMM
row per sample) and every layer runs on the tcgen05 kernels of libgenpose_b200.so (csrc/gemm_tc.cu,
csrc/sa_fused.cu; level 1 on the FP32 kernel of csrc/pointnet2.cu).  There is no library-GEMM backend:
`gemm_mode` only selects the operand precision, see GEMM_NPASS.
"""
from typing import List, Optional

import torch
import torch.nn as nn

from . import pointnet2_utils as pu

# operand precision of the tensor-core SharedMLP GEMMs -> the kernels' npass: "bf16x3" = split-bf16 x3 (fp32-class),
# "tf32" = tcgen05 kind::tf32 with operands rounded to nearest tf32, "bf16" = bf16 operands
GEMM_NPASS = {"bf16x3": 3, "tf32": 2, "bf16": 1}

ClsMSG_CFG_Light = {
    "NPOINTS": [512, 256, 128, 64, None],
    "RADIUS": [[0.01, 0.02], [0.02, 0.04], [0.04, 0.08], [0.08, 0.16], [None, None]],
    "NSAMPLE": [[16, 32], [16, 32], [16, 32], [16, 32], [None, None]],
    "MLPS": [
        [[16, 16, 32], [32, 32, 64]],
        [[64, 64, 128], [64, 96, 128]],
        [[128, 196, 256], [128, 196, 256]],
        [[256, 256, 512], [256, 384, 512]],
        [[512, 512], [512, 512]],
    ],
    "DP_RATIO": 0.5,
}


class _BatchNorm2d(nn.Module):
    """pytorch_utils.py BatchNorm2d wrapper: child named `bn`."""

    def __init__(self, c):
        super().__init__()
        self.bn = nn.BatchNorm2d(c)


class _Conv2d(nn.Module):
    """pytorch_utils.py Conv2d(_ConvBase): children `conv` (1x1, no bias) and `bn`."""

    def __init__(self, cin, cout):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, kernel_size=(1, 1), bias=False)
        self.bn = _BatchNorm2d(cout)

    def folded(self):
        bn = self.bn.bn
        scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
        w = self.conv.weight[:, :, 0, 0] * scale[:, None]
        b = bn.bias - bn.running_mean * scale
        return w, b


class SharedMLP(nn.Module):
    """pytorch_utils.py:5-33: children `layer{i}`."""

    def __init__(self, spec: List[int]):
        super().__init__()
        self.n_layers = len(spec) - 1
        for i in range(self.n_layers):
            self.add_module(f"layer{i}", _Conv2d(spec[i], spec[i + 1]))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """Reference layout: x (B, C, M, ns) -> (B, Cout, M): conv+BN+ReLU stack then max over ns."""
        B, C, M, ns = x.shape
        rows = x.permute(0, 2, 3, 1).reshape(B * M * ns, C)
        if C % 4:   # the GEMM loader reads 16-byte groups; padding columns meet zero weights
            rows = torch.nn.functional.pad(rows, (0, 4 - C % 4))
        cout = getattr(self, f"layer{self.n_layers - 1}").conv.out_channels
        out = torch.empty((B * M, cout), dtype=torch.float32, device=x.device)
        self.forward_rows_pooled(rows.contiguous(), B * M, ns, out, self.gemm_mode)
        return out.view(B, M, -1).permute(0, 2, 1).contiguous()

    gemm_mode = "bf16x3"   # operand precision of the tensor-core GEMMs: a key of GEMM_NPASS

    _trusted = False  # set by Pointnet2ClsMSG.forward for the duration of one pass, after it has checked the cache

    def _folded_layers(self):
        """BatchNorm(eval) folded into the 1x1 convs, cached until a parameter / buffer changes."""
        if self._trusted:
            return self._fold
        ts = []
        for i in range(self.n_layers):
            l = getattr(self, f"layer{i}")
            ts += [l.conv.weight, l.bn.bn.weight, l.bn.bn.bias, l.bn.bn.running_mean, l.bn.bn.running_var]
        key = tuple((t.data_ptr(), t._version) for t in ts)
        if getattr(self, "_fold_key", None) != key:
            with torch.no_grad():
                self._fold = [tuple(t.contiguous() for t in getattr(self, f"layer{i}").folded())
                              for i in range(self.n_layers)]
            self._fold_key = key
        return self._fold

    def _folded_layers_host(self):
        """CPU copies of the folded layers (one device-to-host copy per checkpoint), for kernels that take their
        weights through the launch's parameter space."""
        fold = self._folded_layers()
        if getattr(self, "_fh_key", None) != self._fold_key:
            self._fh = [(w.detach().float().cpu().contiguous(), b.detach().float().cpu().contiguous()) for w, b in fold]
            self._fh_key = self._fold_key
        return self._fh

    def _tc_layers(self, npass):
        """(packed weights, bias, N, K) per layer for the tcgen05 GEMM, cached like the folded weights."""
        fold = self._folded_layers()
        key = (self._fold_key, npass)
        if getattr(self, "_tc_key", None) != key:
            self._tc = [(pu.gemm_pack(w, npass), b, w.shape[0], w.shape[1]) for w, b in fold]
            self._tc_key = key
        return self._tc

    def _tc_layers_featfirst(self, npass):
        """_tc_layers with the first layer's columns permuted to the [feat | xyz] row layout of the encoder's
        level buffers (the reference concatenates [xyz | feat], pointnet2_utils.py:321-326)."""
        fold = self._folded_layers()
        key = (self._fold_key, npass, "featfirst")
        if getattr(self, "_tf_key", None) != key:
            (w0, b0), rest = fold[0], fold[1:]
            w0p = torch.cat([w0[:, 3:], w0[:, :3]], dim=1).contiguous()
            self._tf = [(pu.gemm_pack(w0p, npass), b0, w0p.shape[0], w0p.shape[1])] + \
                       [(pu.gemm_pack(w, npass), b, w.shape[0], w.shape[1]) for w, b in rest]
            self._tf_key = key
        return self._tf

    def _tc_hoisted(self, npass):
        """Operands for the hoisted form of a 3-layer scale (see forward_hoisted), cached."""
        fold = self._folded_layers()
        key = (self._fold_key, npass, "hoisted")
        if getattr(self, "_th_key", None) != key:
            (w0, b0), (w1, b1), (w2, b2) = fold
            w0p = torch.cat([w0[:, 3:], w0[:, :3]], dim=1).contiguous()  # feature columns first, xyz last
            self._th = dict(p0=pu.gemm_pack(w0p, npass), k0=w0p.shape[1], c1=w0.shape[0], w0p=w0p,
                            w0_xyz_t=w0[:, :3].t().contiguous(), b0=b0,
                            p1=pu.gemm_pack(w1, npass), b1=b1, c2=w1.shape[0],
                            p2=pu.gemm_pack(w2, npass), b2=b2, c3=w2.shape[0])
            self._th_key = key
        return self._th

    def forward_hoisted(self, pts_rows, n_src, new_xyz, bq_idx, out, gemm_mode):
        """A whole scale with point features on the tensor cores, first layer hoisted to the points.
        The first 1x1 conv is linear before its ReLU, so
            W0 . [xyz[idx] - new_xyz ; feat[idx]] + b0  =  (W0 . [xyz ; feat])[idx]  -  (W0_xyz . new_xyz - b0)
        : it is evaluated once per POINT (nsample x fewer multiply-adds, exact algebra), and the gathered
        (centre, sample) activation matrix of the reference (pointnet2_utils.py:279-296) never exists in HBM --
        the second layer's operand loader gathers the per-point rows by ball-query index, subtracts the per-centre
        term and applies the ReLU on the fly.  pts_rows = [feat | xyz | 0-pad] per point, [B*n_src, ld]."""
        npass = GEMM_NPASS[gemm_mode]
        t = self._tc_hoisted(npass)
        B, M, ns = bq_idx.shape
        P = pu.gemm_linear(pts_rows, t["p0"], t["c1"], t["k0"], npass)                 # [B*n_src, ldp]
        Q = pu.centre_term(new_xyz.reshape(B * M, 3).contiguous(), t["w0_xyz_t"], t["b0"], P.shape[1])
        return self.hoisted_tail(P, Q, n_src, bq_idx, out, gemm_mode)

    def hoisted_tail(self, P, Q, n_src, bq_idx, out, gemm_mode):
        """Layers 2, 3 and the max-pool of forward_hoisted, given the per-point table P and the per-centre term Q
        (both may be column slices of tables shared by the scales of a level)."""
        npass = GEMM_NPASS[gemm_mode]
        t = self._tc_hoisted(npass)
        B, M, ns = bq_idx.shape
        if pu.sa_mlp2_fused_fits(t["c1"], t["c2"], t["c3"], npass, ns):
            # layers 2, 3 and the max-pool in one kernel: no (centre, sample) matrix in HBM at all
            return pu.sa_mlp2_fused(P, n_src, bq_idx.reshape(-1), M * ns, Q, ns, t["p1"], t["b1"], t["c1"], t["c2"],
                                    t["p2"], t["b2"], t["c3"], npass, ns, out)
        h2 = pu.gemm_gather_bias_relu(P, n_src, bq_idx.reshape(-1), M * ns, Q, ns, t["p1"], t["b1"], t["c2"], t["c1"],
                                      npass)
        out.zero_()
        pu.gemm_bias_relu(h2, t["p2"], t["b2"], t["c3"], t["c2"], npass, pool_ns=ns, pooled_out=out)
        return out

    def forward_rows_pooled(self, rows, groups, nsample, out, gemm_mode, feat_first=False, zeroed=False):
        """rows (R, ld) -> SharedMLP -> max over `nsample` rows per group, written into `out` (groups, Cout).
        gemm_mode: a key of GEMM_NPASS (tcgen05 operand precision).
        feat_first: the rows are [feat | xyz | 0] (the encoder's level buffers) instead of [xyz | feat]."""
        npass = GEMM_NPASS[gemm_mode]
        layers = self._tc_layers_featfirst(npass) if feat_first else self._tc_layers(npass)
        h = rows
        for i, (packed, b, N, K) in enumerate(layers):
            if i + 1 < len(layers):
                h = pu.gemm_bias_relu(h, packed, b, N, K, npass)
            else:
                if not zeroed:
                    out.zero_()
                pu.gemm_bias_relu(h, packed, b, N, K, npass, pool_ns=nsample, pooled_out=out)
        return out


class PointnetSAModuleMSG(nn.Module):
    """pointnet2_modules.py:77-121 + forward :19-74 (max_pool, use_xyz=True, bn=True)."""

    def __init__(self, *, npoint, radii, nsamples, mlps):
        super().__init__()
        self.npoint, self.radii, self.nsamples = npoint, radii, nsamples
        self.gemm_mode = "bf16x3"  # a key of GEMM_NPASS (see SharedMLP.forward_rows_pooled)
        # feature-less scales (first level) that take the fused tensor-core kernel instead of the FP32 kernel
        self.level1_tc_specs = ((32, 32, 64),)
        self.groupers = nn.ModuleList(
            [pu.QueryAndGroup(r, n) if npoint is not None else pu.GroupAll() for r, n in zip(radii, nsamples)])
        self.mlps = nn.ModuleList([SharedMLP([spec[0] + 3] + spec[1:]) for spec in mlps])

    def forward(self, xyz, features=None, geometry=None):
        """Reference layout (pointnet2_modules.py:19-74): xyz (B,N,3), features (B,C,N) ->
        new_xyz (B,npoint,3), new_features (B,sum Cout,npoint), geometry."""
        feat_cl = None if features is None else features.transpose(1, 2).contiguous()
        new_xyz, out_cl, geometry = self.forward_cl(xyz, feat_cl, geometry)
        return new_xyz, out_cl.transpose(1, 2).contiguous(), geometry

    def _merged_first_layer(self, npass):
        """The hoisted first layers of all scales of this level as ONE per-point GEMM and ONE per-centre term: the
        scales read the same rows, so their weights are stacked along the output channels and each scale takes its
        column slice of P / Q.  None when a slice would not start on a 64-column (one operand atom) boundary."""
        ths = [m._tc_hoisted(npass) for m in self.mlps]
        if len(ths) < 2 or any(t["c1"] % 64 for t in ths) or len({t["k0"] for t in ths}) != 1:
            return None
        key = tuple(m._th_key for m in self.mlps)
        if getattr(self, "_mf_key", None) != key:
            self._mf = dict(p0=pu.gemm_pack(torch.cat([t["w0p"] for t in ths], dim=0).contiguous(), npass),
                            k0=ths[0]["k0"], n=sum(t["c1"] for t in ths),
                            w0_xyz_t=torch.cat([t["w0_xyz_t"] for t in ths], dim=1).contiguous(),
                            b0=torch.cat([t["b0"] for t in ths]).contiguous())
            self._mf_key = key
        return self._mf

    def _merged_groupall_first(self, npass, feat_first):
        """GroupAll level with two-layer scales: the first layers of all scales as ONE GEMM (they read the same rows).
        None when the scales are not two-layer MLPs of equal input width with hidden widths that keep every slice on a
        64-column boundary."""
        if len(self.mlps) < 2 or any(m.n_layers != 2 for m in self.mlps):
            return None
        lays = [(m._tc_layers_featfirst(npass) if feat_first else m._tc_layers(npass)) for m in self.mlps]
        if len({l[0][3] for l in lays}) != 1 or any(l[0][2] % 64 or l[1][3] != l[0][2] for l in lays):
            return None
        key = (tuple(m._fold_key for m in self.mlps), npass, feat_first)
        if getattr(self, "_mg_key", None) != key:
            ws, bs = [], []
            for m in self.mlps:
                w0, b0 = m._folded_layers()[0]
                ws.append(torch.cat([w0[:, 3:], w0[:, :3]], dim=1) if feat_first else w0)
                bs.append(b0)
            w = torch.cat(ws, dim=0).contiguous()
            self._mg = dict(p0=pu.gemm_pack(w, npass), b0=torch.cat(bs).contiguous(), n=w.shape[0], k=w.shape[1])
            self._mg_key = key
        return self._mg

    def forward_cl(self, xyz, feat_cl=None, geometry=None, pts_rows=None, return_rows=False):
        """Channels-last fast path: feat_cl (B,N,C) -> new_xyz (B,npoint,3), out (B,npoint,sum Cout).
        FPS+gather, one two-radius ball query, then per scale: fused gather into GEMM rows, the SharedMLP
        as a row-major GEMM chain, max-pool over the samples written straight into the concatenated output.

        Level buffers: the tensor-core scales read one row [feat | xyz | 0] per point.  With return_rows the output
        is allocated four columns wider, the centres are copied into the tail, and the buffer comes back as a fourth
        result to be handed to the next level as `pts_rows` -- no concatenation between levels."""
        B = xyz.shape[0]
        couts = [getattr(m, f"layer{m.n_layers - 1}").conv.out_channels for m in self.mlps]
        C = sum(couts)
        tc = True   # every SharedMLP layer runs on the library's own kernels
        if self.npoint is not None:
            if geometry is None:
                idx, new_xyz = pu.furthest_point_sample_gather(xyz, self.npoint)
                bq = pu.ball_query2(self.radii, self.nsamples, xyz, new_xyz)
                geometry = (idx, new_xyz, bq)
            idx, new_xyz, bq = geometry[:3]
            M = self.npoint
            pad_rows = return_rows and tc and C % 4 == 0
            out_full = torch.empty((B, M, C + 4 if pad_rows else C), dtype=torch.float32, device=xyz.device)
            out, out2d = out_full[..., :C], out_full.view(B * M, -1)
            off = 0
            hoist = feat_cl is not None and tc and feat_cl.shape[2] % 4 == 0
            P_all = Q_all = None
            # [x y z 0] of the centres for the tail of the level buffer: written by a kernel of this level as a by-product
            tail = None
            if pad_rows:
                tail = geometry[3] if len(geometry) > 3 else torch.nn.functional.pad(new_xyz, (0, 1))
            tail_written = False
            if hoist:
                shifted = len(geometry) > 5      # compute_geometry's per-object shift (see there)
                q_xyz = geometry[4] if shifted else new_xyz
                if pts_rows is None:  # [feat | xyz | 0] per point, shared by both scales
                    N = xyz.shape[1]
                    pts_rows = torch.cat([feat_cl, xyz - geometry[5] if shifted else xyz,
                                          torch.zeros((B, N, 1), dtype=torch.float32, device=xyz.device)],
                                         dim=-1).reshape(B * N, -1)
                if all(m.n_layers == 3 for m in self.mlps):
                    npass = GEMM_NPASS[self.gemm_mode]
                    mf = self._merged_first_layer(npass)
                    if mf is not None:
                        P_all = pu.gemm_linear(pts_rows, mf["p0"], mf["n"], mf["k0"], npass)
                        Q_all = pu.centre_term(q_xyz.reshape(B * M, 3), mf["w0_xyz_t"], mf["b0"], P_all.shape[1],
                                               tail=tail, tail_dst=None if tail is None else out2d[:, C:C + 4])
                        tail_written = tail is not None
            col = 0
            for i, mlp in enumerate(self.mlps):
                if hoist and mlp.n_layers == 3:
                    dst = out2d[:, off:off + couts[i]]
                    if P_all is not None:
                        c1 = mlp.layer0.conv.out_channels
                        mlp.hoisted_tail(P_all[:, col:col + c1], Q_all[:, col:col + c1], xyz.shape[1], bq[i], dst,
                                         self.gemm_mode)
                        col += c1
                    else:
                        mlp.forward_hoisted(pts_rows, xyz.shape[1], q_xyz, bq[i], dst, self.gemm_mode)
                    off += couts[i]
                    continue
                spec = tuple(getattr(mlp, f"layer{j}").conv.out_channels for j in range(mlp.n_layers))
                if (feat_cl is None and tc and self.nsamples[i] in (16, 32) and spec in self.level1_tc_specs
                        and pu.sa_mlp2_fused_fits(*spec, GEMM_NPASS[self.gemm_mode], self.nsamples[i])):
                    # first level, wide scale: layers 2, 3 and the max-pool on the tensor cores, the K = 3 first layer
                    # evaluated in the fused kernel's operand loader
                    npass = GEMM_NPASS[self.gemm_mode]
                    t = mlp._tc_hoisted(npass)
                    w0, b0 = mlp._folded_layers_host()[0]
                    pu.sa_mlp2_fused_xyz(xyz, new_xyz, bq[i], w0, b0, t["p1"], t["b1"], t["c1"], t["c2"], t["p2"], t["b2"],
                                         t["c3"], npass, out2d[:, off:off + couts[i]])
                    off += couts[i]
                    continue
                if (feat_cl is None and tc and self.nsamples[i] in (16, 32)
                        and spec in ((16, 16, 32), (32, 32, 64))):
                    # first level: the whole scale in one FP32 kernel (channels too narrow for tensor cores)
                    first = tail is not None and not tail_written
                    pu.sa_small_mlp_hostw(xyz, new_xyz, bq[i], mlp._folded_layers_host(), out2d[:, off:off + couts[i]],
                                          tail=tail if first else None, tail_col=C - off)
                    tail_written = tail_written or first
                    off += couts[i]
                    continue
                rows = pu.group_rows(xyz, new_xyz, feat_cl, bq[i], pad_to=4 if tc else 1)
                mlp.forward_rows_pooled(rows, B * M, self.nsamples[i], out2d[:, off:off + couts[i]], self.gemm_mode)
                off += couts[i]
            if pad_rows and not tail_written:
                out_full[..., C:].copy_(tail)  # [x y z 0] of the centres
            res = (new_xyz, out, geometry)
            return res + (out2d if pad_rows else None,) if return_rows else res
        # GroupAll (pointnet2_utils.py:306-328): every point of the level is one sample of a single group
        N = xyz.shape[1]
        if not (N % 32 == 0 or 32 % N == 0):
            raise NotImplementedError(
                f"GroupAll over {N} points: the pooled tensor-core GEMM needs N to divide or be a multiple of 32 "
                "(GP_ERR_UNSUPPORTED; there is no library fallback)")
        feat_first = pts_rows is not None
        if feat_first:
            rows, gm = pts_rows, self.gemm_mode
        else:
            parts = [xyz] if feat_cl is None else [xyz, feat_cl]
            width = sum(p.shape[-1] for p in parts)
            if tc and width % 4:
                parts.append(torch.zeros((B, N, 4 - width % 4), dtype=torch.float32, device=xyz.device))
            rows = torch.cat(parts, dim=-1).reshape(B * N, -1)
            gm = self.gemm_mode
        out = pu.zeros((B, 1, C), xyz.device)   # the pooled GEMMs take the max into a zero-initialised output
        off = 0
        npass = GEMM_NPASS[gm]
        mg = self._merged_groupall_first(npass, feat_first)
        if mg is not None:
            # the scales read the same rows: their first layers are ONE GEMM (weights stacked along the output channels,
            # twice the CTAs of a launch per scale -- at 64 objects a scale alone covers 64 of the 148 SMs); each scale's
            # pooled second layer then reads its column slice
            h = pu.gemm_bias_relu(rows, mg["p0"], mg["b0"], mg["n"], mg["k"], npass)
            col = 0
            for i, mlp in enumerate(self.mlps):
                packed, b, N2, K2 = (mlp._tc_layers_featfirst(npass) if feat_first else mlp._tc_layers(npass))[1]
                pu.gemm_bias_relu(h[:, col:col + K2], packed, b, N2, K2, npass, pool_ns=N,
                                  pooled_out=out.view(B, -1)[:, off:off + couts[i]])
                col += K2
                off += couts[i]
            res = (None, out, geometry)
            return res + (None,) if return_rows else res
        for i, mlp in enumerate(self.mlps):
            mlp.forward_rows_pooled(rows, B, N, out.view(B, -1)[:, off:off + couts[i]], gm, feat_first=feat_first, zeroed=True)
            off += couts[i]
        res = (None, out, geometry)
        return res + (None,) if return_rows else res


class Pointnet2ClsMSG(nn.Module):
    def __init__(self, input_channels=0):
        super().__init__()
        cfg = ClsMSG_CFG_Light
        self.SA_modules = nn.ModuleList()
        channel_in = input_channels
        for k in range(len(cfg["NPOINTS"])):
            mlps = [[channel_in] + list(m) for m in cfg["MLPS"][k]]
            self.SA_modules.append(PointnetSAModuleMSG(
                npoint=cfg["NPOINTS"][k], radii=cfg["RADIUS"][k], nsamples=cfg["NSAMPLE"][k], mlps=mlps))
            channel_in = sum(m[-1] for m in mlps)

    def set_gemm_mode(self, mode):
        """Operand precision of the tensor-core SharedMLP GEMMs for every level: "bf16x3" (split-bf16 x3,
        fp32-class accuracy), "tf32" (tf32 operands, rounded to nearest) or "bf16"."""
        if mode not in GEMM_NPASS:
            raise ValueError(mode)
        for sa in self.SA_modules:
            sa.gemm_mode = mode
            for m in sa.mlps:
                m.gemm_mode = mode
        return self

    @staticmethod
    def _break_up_pc(pc):
        xyz = pc[..., 0:3].contiguous()
        features = pc[..., 3:].transpose(1, 2).contiguous() if pc.size(-1) > 3 else None
        return xyz, features

    def compute_geometry(self, pointcloud: torch.Tensor):
        """FPS + both ball queries of every level (they depend on the coordinates only: level k samples the centres
        of level k-1), as the list `forward(..., geometry=...)` takes.  Lets two encoders that see the same cloud
        share one pass and start side by side."""
        xyz = pointcloud[..., 0:3].contiguous()
        # Per-object shift for the hoisted first layers.  W0 . [xyz[idx] - new_xyz ; feat[idx]] only sees coordinate
        # DIFFERENCES, so the per-point table P = W0_xyz . (xyz - c) and the per-centre term Q = W0_xyz . (new_xyz - c) - b0
        # give the same result for any c.  The clouds are in the camera frame (|xyz| ~ 1 m, posenet.py:135) while the
        # differences are <= the ball radius (0.02 .. 0.16 m): with c = the object's first point (FPS starts there, so it
        # is also every level's first centre) the GEMM operands are object-sized and their bf16 / split-bf16 rounding
        # scales with the object, not with its distance from the camera.
        shift = xyz[:, 0:1, :].contiguous()
        n_levels = sum(1 for sa in self.SA_modules if sa.npoint is not None)
        geometry, tie_free = [], None
        for k, sa in enumerate(self.SA_modules):
            if sa.npoint is None:
                geometry.append(None)
                continue
            # each level samples the previous level's centres: an FPS-ordered cloud, whose FPS is its own prefix
            # unless the earlier sampling hit an exact tie (pointnet2_utils.furthest_point_sample_chain)
            idx, new_xyz, tie_free = pu.furthest_point_sample_chain(xyz, sa.npoint, tie_free)
            # rel = new_xyz - shift and the tail of this level's buffer = the [x y z 0] columns the NEXT level reads
            # (shifted for a hoisted level, absolute for the GroupAll level: its SharedMLP sees the coordinates
            # themselves, pointnet2_utils.py:321-326) come out of the ball-query launch
            bq, rel, tail = pu.ball_query2_tails(sa.radii, sa.nsamples, xyz, new_xyz, shift, k + 1 >= n_levels)
            geometry.append((idx, new_xyz, bq, tail, rel, shift))
            xyz = new_xyz
        return geometry

    def forward(self, pointcloud: torch.Tensor, geometry: Optional[list] = None, return_geometry=False,
                levels: Optional[list] = None):
        """pointcloud (B, N, 3 + C) -> (B, 1024).  `geometry`: per-level FPS / ball-query results of an
        earlier call on the same cloud (they depend on xyz only).  `levels`: a list that receives every level's
        (new_xyz, pooled features channels-last) -- the reference's l_xyz / l_features (pointnet2.py:247-251)."""
        xyz = pointcloud[..., 0:3].contiguous()
        feat_cl = pointcloud[..., 3:].contiguous() if pointcloud.size(-1) > 3 else None
        geo_out = []
        if geometry is None:
            geometry = self.compute_geometry(pointcloud)
        # the folded / packed weight caches are validated once per pass (parameter versions), not once per use
        mlps = [m for sa in self.SA_modules for m in sa.mlps]
        for m in mlps:
            m._trusted = False
            m._folded_layers()
            m._trusted = True
        try:
            rows = None
            for k, sa in enumerate(self.SA_modules):
                g = geometry[k]
                xyz, feat_cl, g, rows = sa.forward_cl(xyz, feat_cl, g, pts_rows=rows, return_rows=True)
                geo_out.append(g)
                if levels is not None:
                    levels.append((xyz, feat_cl))
        finally:
            for m in mlps:
                m._trusted = False
        out = feat_cl.squeeze(1)
        return (out, geo_out) if return_geometry else out

"""Drop-in for the reference's util/lpdnet_model.py: LPDNet, LPDNetOrign, TranformNet, knn,
get_graph_feature, get_graph_feature_Origin — same constructor signatures, attribute names and
state_dict keys, same tensor layouts at the public boundary ([B,1,N,3] in, [B,emb,N,1] out, knn()
takes channel-major [B,C,N] and returns int64 [B,N,k]).

Inside, feature maps are point-major [B*N, C] and every arithmetic step is a call into
liblpd_b200.so (see include/lpd_b200.h).  The EdgeConv layers use the exact decomposition
W.[f_j ; f_i] = Wn.f_j + Wc.f_i (per-point GEMM + neighbour gather), so the [B,2C,N,k] edge tensor of
get_graph_feature (reference :331-363) is only materialised if a caller asks for it through the public
get_graph_feature() function.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from .._host import Prepared, fold_bn, require_cuda, training_unsupported, w2d

__all__ = ["LPDNet", "LPDNetOrign", "TranformNet", "knn", "get_graph_feature", "get_graph_feature_Origin"]

cat_or_stack = True  # reference :17 (module-level switch, always True there)


# ------------------------------------------------------------------------------------------------
# public free functions (reference :317-363, :116-145)
# ------------------------------------------------------------------------------------------------
def knn(x: torch.Tensor, k: int) -> torch.Tensor:
    """x [B, C, N] (channel-major, as in the reference :317) -> int64 [B, N, k], nearest first, self first.
    Ties are broken towards the lower index (canonical order, include/lpd_b200.h lpd_knn)."""
    require_cuda(x, "knn")
    return ops.knn(ops.transpose(x.detach()), k, int64=True)


def _gather_edges(x: torch.Tensor, k: int, idx):
    """shared by the two public get_graph_feature variants: returns (point-major x [B,N,C], neighbours [B,N,k,C])"""
    require_cuda(x, "get_graph_feature")
    B, N = x.size(0), x.size(2)
    x = x.detach().reshape(B, -1, N)
    x_pm = ops.transpose(x)                                    # [B, N, C]
    if idx is None:
        idx = ops.knn(x_pm, k, int64=True)
    C = x_pm.size(2)
    # gather with an identity EdgeConv: out[i] = p[j(i,m)] for each m separately (k launches of the gather kernel)
    idx32 = idx.to(torch.int32).contiguous()
    feat = torch.empty(B, N, k, C, device=x.device, dtype=torch.float32)
    Cp = (C + 3) // 4 * 4
    src = x_pm if Cp == C else torch.nn.functional.pad(x_pm, (0, Cp - C))
    tmp = torch.empty(B * N, Cp, device=x.device, dtype=torch.float32)
    for m in range(k):
        ops.edge_gather_ext(src, Cp, None, 0, idx32[:, :, m].contiguous(), B, N, 1, Cp, None, None, ops.ACT_NONE, 0.0, tmp, Cp)
        feat[:, :, m, :] = tmp.view(B, N, Cp)[:, :, :C]
    return x_pm, feat


def get_graph_feature(x: torch.Tensor, k: int = 20, idx=None) -> torch.Tensor:
    """Reference :331-363: [B, C, N] -> [B, 2C, N, k] = cat(neighbour, centre).  Compatibility entry point only —
    LPDNet.forward never builds this tensor."""
    x_pm, feat = _gather_edges(x, k, idx)
    centre = x_pm.unsqueeze(2).expand_as(feat)
    return torch.cat((feat, centre), dim=3).permute(0, 3, 1, 2)


def get_graph_feature_Origin(x: torch.Tensor, k: int = 20, idx=None, cat: bool = True) -> torch.Tensor:
    """Reference :116-145: cat(centre, neighbour - centre) -> [B, 2C, N, k], or gather only -> [B, C, N, k]."""
    x_pm, feat = _gather_edges(x, k, idx)
    if cat:
        centre = x_pm.unsqueeze(2).expand_as(feat)
        feat = torch.cat((centre, feat - centre), dim=3)
    return feat.permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------------
# shared building blocks
# ------------------------------------------------------------------------------------------------
def _act_code(module) -> tuple:
    return (ops.ACT_RELU, 0.0) if isinstance(module.act_f, nn.ReLU) else (ops.ACT_LEAKY, module.negative_slope)


def _split_input(x: torch.Tensor, use_mFea: bool, who: str, spatial_order: bool = False):
    """[B,1,N,D] -> (point-major rows [B*N, D] contiguous, xyz [B,N,3] contiguous, B, N, D).
    spatial_order: the points of every cloud are re-ordered into grid-cell order first (ops.cell_order); valid whenever the
    caller consumes the per-point result through a permutation-invariant reduction (NetVLAD)."""
    require_cuda(x, who)
    if x.dim() != 4 or x.size(1) != 1:
        raise ValueError(f"{who}: expected input [B, 1, N, dims], got {tuple(x.shape)}")
    B, _, N, D = x.shape
    rows = x.detach().reshape(B * N, D).contiguous()
    if spatial_order and D == 3 and N >= 64:
        _, _, xs = ops.cell_order(rows.view(B, N, 3))
        rows = xs.view(B * N, 3)
    if D > 3 or use_mFea:
        if D != 8:
            raise ValueError(f"{who}: use_mFea expects 8 input dims (xyz + 5 features), got {D}")
        xyz = rows.view(B, N, D)[:, :, :3].contiguous()
    else:
        xyz = rows.view(B, N, 3)
    return rows, xyz, B, N, D


def _apply_transform(rows: torch.Tensor, trans: torch.Tensor, B: int, N: int, C: int, ld: int) -> torch.Tensor:
    """rows[b] <- rows[b][:, :C] . trans[b]   (torch.bmm at reference :86,:93,:229,:241), other columns kept"""
    out = rows.clone() if ld != C else torch.empty_like(rows)
    ops.gemm(rows, trans, a_layout=ops.A_MK, b_layout=ops.B_KN, M=N, N=C, K=C, lda=ld, ldb=C, out=out, ldc=ld,
             batch=B, strideA=N * ld, strideB=C * C, strideC=N * ld)
    return out


class TranformNet(nn.Module):
    """Reference :273-313 (spelling kept).  T-Net: k -> 64 -> 128 -> 1024, max over N, 512 -> 256 -> k*k + I."""

    def __init__(self, k=3, negative_slope=1e-2, use_relu=True):
        super().__init__()
        self.conv1 = nn.Conv1d(k, 64, 1)
        self.conv2 = nn.Conv1d(64, 128, 1)
        self.conv3 = nn.Conv1d(128, 1024, 1)
        self.fc1 = nn.Linear(1024, 512)
        self.fc2 = nn.Linear(512, 256)
        self.fc3 = nn.Linear(256, k * k)
        self.relu = nn.ReLU if use_relu else nn.LeakyReLU(negative_slope=negative_slope, inplace=True)  # unused, as in the reference
        self.bn1 = nn.BatchNorm1d(64)
        self.bn2 = nn.BatchNorm1d(128)
        self.bn3 = nn.BatchNorm1d(1024)
        self.bn4 = nn.BatchNorm1d(512)
        self.bn5 = nn.BatchNorm1d(256)
        self.k = k
        self._prep = Prepared()

    def _build(self):
        p = {}
        for i, (lin, bn) in enumerate(((self.conv1, self.bn1), (self.conv2, self.bn2), (self.conv3, self.bn3),
                                       (self.fc1, self.bn4), (self.fc2, self.bn5)), 1):
            p[f"w{i}"] = w2d(lin.weight)
            p[f"s{i}"], p[f"t{i}"] = fold_bn(bn, lin.bias)
        p["w6"] = w2d(self.fc3.weight)
        p["t6"] = self.fc3.bias.detach() + torch.eye(self.k, device=self.fc3.bias.device).reshape(-1)
        return p

    def forward_pm(self, rows: torch.Tensor, B: int, N: int, ld: int) -> torch.Tensor:
        """rows [B*N, ld] point-major (first k columns used) -> [B, k, k]"""
        training_unsupported(self, "TranformNet")
        p = self._prep.get(self, self._build)
        M, R = B * N, ops.ACT_RELU
        h = ops.linear(rows, p["w1"], M=M, N=64, K=self.k, lda=ld, scale=p["s1"], shift=p["t1"], act=R)
        h = ops.linear(h, p["w2"], M=M, N=128, K=64, scale=p["s2"], shift=p["t2"], act=R)
        h = ops.linear(h, p["w3"], M=M, N=1024, K=128, scale=p["s3"], shift=p["t3"], act=R)
        g = ops.colmax(h, B, N, 1024)
        g = ops.linear(g, p["w4"], M=B, N=512, K=1024, scale=p["s4"], shift=p["t4"], act=R)
        g = ops.linear(g, p["w5"], M=B, N=256, K=512, scale=p["s5"], shift=p["t5"], act=R)
        g = ops.linear(g, p["w6"], M=B, N=self.k * self.k, K=256, shift=p["t6"])
        return g.view(B, self.k, self.k)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [B, k, N] (channel-major, reference :295) -> [B, k, k]"""
        require_cuda(x, "TranformNet")
        B, _, N = x.shape
        return self.forward_pm(ops.transpose(x.detach()).view(B * N, self.k), B, N, self.k)


class _LPDBase(nn.Module):
    """Common forward plumbing of LPDNet / LPDNetOrign."""

    def _front(self, x, p, who, spatial_order=False):
        """input split, optional T-Nets, conv1/conv2 -> (h2 [M,64], xyz_init [B,N,3], B, N).
        Everything here feeds the feature-space kNN, so it always runs in strict fp32 arithmetic (a TF32-rounded
        feature would move points across the k-th-neighbour boundary far beyond the few-ulp near-ties)."""
        prev = ops.set_precision("fp32")
        try:
            rows, xyz_init, B, N, D = _split_input(x, self.use_mFea, who, spatial_order)
            M = B * N
            act, slope = _act_code(self)
            if self.t3d:
                trans = self.t_net3d.forward_pm(rows, B, N, D)           # T-Net sees the raw xyz columns
                rows = _apply_transform(rows, trans, B, N, 3, D)         # kNN below still uses xyz_init (reference :226,:255)
            if D <= 8 and p["w1"].shape[0] == 64 and tuple(p["w2"].shape) == (64, 64):
                h = ops.pointwise_mlp2(rows, D, M, p["w1"], p["s1"], p["t1"], p["w2"], p["s2"], p["t2"], act, slope)
            else:
                h = ops.linear(rows, p["w1"], M=M, N=64, K=D, scale=p["s1"], shift=p["t1"], act=act, slope=slope)
                h = ops.linear(h, p["w2"], M=M, N=64, K=64, scale=p["s2"], shift=p["t2"], act=act, slope=slope)
            if self.tfea:
                tf = self.t_net_fea.forward_pm(h, B, N, 64)
                h = _apply_transform(h, tf, B, N, 64, 64)
        finally:
            ops.set_precision(prev)
        return h, xyz_init, B, N

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """[B, 1, N, dims] -> [B, emb_dims, N, 1] (reference layout)."""
        f, B, N = self.forward_pm(x, keep_order=True)
        return ops.transpose(f.view(B, N, self.emb_dims)).unsqueeze(-1)


class LPDNet(_LPDBase):
    """Reference :147-268.  conv1/2 (3->64->64) -> feature-space kNN EdgeConv DG1 (x1) / DG2 (x2) ->
    Cartesian kNN EdgeConv SN1 on x2 (x3) -> cat 512 -> conv3 512->emb."""

    def __init__(self, emb_dims=512, use_mFea=False, t3d=True, tfea=False, use_relu=False):
        super().__init__()
        self.negative_slope = 1e-2
        self.act_f = nn.ReLU(inplace=True) if use_relu else nn.LeakyReLU(negative_slope=self.negative_slope, inplace=True)
        self.use_mFea = use_mFea
        self.k = 20
        self.t3d = t3d
        self.tfea = tfea
        self.emb_dims = emb_dims
        if self.t3d:
            self.t_net3d = TranformNet(3)
        if self.tfea:
            self.t_net_fea = TranformNet(64)
        self.useBN = True
        mult = 2 if cat_or_stack else 1
        self.convDG1 = nn.Sequential(nn.Conv2d(64 * mult, 128, kernel_size=1, bias=False), nn.BatchNorm2d(128), self.act_f)
        self.convDG2 = nn.Sequential(nn.Conv2d(128, 128, kernel_size=1, bias=False), nn.BatchNorm2d(128), self.act_f)
        self.convSN1 = nn.Sequential(nn.Conv2d(128 * mult, 256, kernel_size=1, bias=False), nn.BatchNorm2d(256), self.act_f)
        self.conv1_lpd = nn.Conv1d(8 if use_mFea else 3, 64, kernel_size=1, bias=False)
        self.conv2_lpd = nn.Conv1d(64, 64, kernel_size=1, bias=False)
        self.conv3_lpd = nn.Conv1d(512, self.emb_dims, kernel_size=1, bias=False)
        self.bn1_lpd = nn.BatchNorm1d(64)
        self.bn2_lpd = nn.BatchNorm1d(64)
        self.bn3_lpd = nn.BatchNorm1d(self.emb_dims)
        self._prep = Prepared()

    def _build(self):
        p = {"w1": w2d(self.conv1_lpd.weight), "w2": w2d(self.conv2_lpd.weight), "w3": w2d(self.conv3_lpd.weight)}
        p["s1"], p["t1"] = fold_bn(self.bn1_lpd)
        p["s2"], p["t2"] = fold_bn(self.bn2_lpd)
        p["s3"], p["t3"] = fold_bn(self.bn3_lpd)
        wdg1 = w2d(self.convDG1[0].weight)                     # [128, 128] = [Wn | Wc] (neighbour first, reference :357)
        wsn1 = w2d(self.convSN1[0].weight)                     # [256, 256]
        p["wpq1"] = torch.cat((wdg1[:, :64], wdg1[:, 64:]), 0).contiguous()      # [256, 64]: rows 0..127 -> P, 128..255 -> Q
        p["wpq3"] = torch.cat((wsn1[:, :128], wsn1[:, 128:]), 0).contiguous()    # [512, 128]
        p["wdg2"] = w2d(self.convDG2[0].weight)
        p["sdg1"], p["tdg1"] = fold_bn(self.convDG1[1])
        p["sdg2"], p["tdg2"] = fold_bn(self.convDG2[1])
        p["ssn1"], p["tsn1"] = fold_bn(self.convSN1[1])
        # epilogue vectors of the projection GEMMs for the pre-scaled edge kernels: [s | s] and [0 | t]
        p["spq1"] = torch.cat((p["sdg1"], p["sdg1"])).contiguous()
        p["tpq1"] = torch.cat((torch.zeros_like(p["tdg1"]), p["tdg1"])).contiguous()
        p["spq3"] = torch.cat((p["ssn1"], p["ssn1"])).contiguous()
        p["tpq3"] = torch.cat((torch.zeros_like(p["tsn1"]), p["tsn1"])).contiguous()
        if p["w3"].is_cuda:      # fp16 copies of the weights the "f16" precision mode multiplies with (rounded to nearest, once)
            p["wdg2_h"], p["wpq3_h"], p["w3_h"] = ops.to_f16(p["wdg2"]), ops.to_f16(p["wpq3"]), ops.to_f16(p["w3"])
        return p

    def forward_pm(self, x: torch.Tensor, keep_order: bool = False, f16: bool = False):
        """-> (F [B*N, emb] point-major, B, N).  Unless keep_order, the rows of every cloud are in spatial (grid-cell)
        order (ops.SPATIAL_ORDER): PointNetVlad feeds them to NetVLAD, which sums over the points.
        f16 (PointNetVlad.forward in "f16" precision mode, k == 20 or 32): F and every activation downstream of the feature-space kNN
        are fp16 tensors; conv1 / conv2 and both kNN graphs stay exact fp32."""
        require_cuda(x, "LPDNet")
        training_unsupported(self, "LPDNet")
        p = self._prep.get(self, self._build)
        h, xyz_init, B, N = self._front(x, p, "LPDNet", ops.SPATIAL_ORDER and not keep_order)
        M, k = B * N, self.k
        act, slope = _act_code(self)
        dev = h.device
        idx_f = ops.knn(h.view(B, N, 64), k)
        if f16 and k in (20, 32) and M >= 128 and self.emb_dims % 4 == 0:
            pq1 = ops.gemm_tf32_out16(h, p["wpq1"], M=M, N=256, K=64, scale=p["spq1"], shift=p["tpq1"])
            pyr = torch.empty(M, 512, device=dev, dtype=torch.float16)
            ops.edgeconv_dg20_f16(pq1, 256, pq1[:, 128:], 256, idx_f, B, N, p["wdg2_h"], p["sdg2"], p["tdg2"], act, slope,
                                  pyr, 512, pyr[:, 128:], 512)
            del pq1
            idx_x = ops.knn(xyz_init, k)
            pq3 = ops.gemm_f16(pyr[:, 128:], p["wpq3_h"], M=M, N=512, K=128, lda=512, out_half=True, scale=p["spq3"], shift=p["tpq3"])
            ops.edge_gather_max_f16(pq3, 512, pq3[:, 256:], 512, idx_x, B, N, k, 256, act, slope, pyr[:, 256:], 512)
            del pq3
            f = ops.gemm_f16(pyr, p["w3_h"], M=M, N=self.emb_dims, K=512, out_half=True, scale=p["s3"], shift=p["t3"], act=act, slope=slope)
            return f, B, N
        # feature-space graph: DG1 + DG2 fused, x1 | x2 land in columns 0..255 of the 512-wide pyramid buffer
        pyr = torch.empty(M, 512, device=dev, dtype=torch.float32)
        if ops.get_precision() != "fp32" and k == 20 and M >= 128:
            # the reference's own shape: DG1's folded BatchNorm goes into the projection GEMM's epilogue
            # (P' = s1 * Wn h, Q' = s1 * Wc h + t1), the edge kernel only adds, activates and feeds the tensor cores
            pq1 = ops.linear(h, p["wpq1"], M=M, N=256, K=64, scale=p["spq1"], shift=p["tpq1"])
            ops.edgeconv_dg(pq1, 256, pq1[:, 128:], 256, idx_f, B, N, k, 128, 128, None, None, p["wdg2"],
                            p["sdg2"], p["tdg2"], act, slope, pyr, 512, pyr[:, 128:], 512)
        else:
            pq1 = ops.linear(h, p["wpq1"], M=M, N=256, K=64)
            ops.edgeconv_dg(pq1, 256, pq1[:, 128:], 256, idx_f, B, N, k, 128, 128, p["sdg1"], p["tdg1"], p["wdg2"],
                            p["sdg2"], p["tdg2"], act, slope, pyr, 512, pyr[:, 128:], 512)
        del pq1
        # Cartesian graph on the untransformed input coordinates: SN1 over x2
        idx_x = ops.knn(xyz_init, k)
        # SN1's folded BatchNorm rides in the projection GEMM's epilogue (P' = s Wn x2, Q' = s Wc x2 + t): the gather kernel
        # then only needs max_m P'_j + Q'_i (no min branch for negative scales, no per-channel constants)
        pq3 = ops.linear(pyr[:, 128:], p["wpq3"], M=M, N=512, K=128, lda=512, scale=p["spq3"], shift=p["tpq3"])
        ops.edge_gather_ext(pq3, 512, pq3[:, 256:], 512, idx_x, B, N, k, 256, None, None, act, slope, pyr[:, 256:], 512)
        del pq3
        f = ops.linear(pyr, p["w3"], M=M, N=self.emb_dims, K=512, scale=p["s3"], shift=p["t3"], act=act, slope=slope)
        return f, B, N


class LPDNetOrign(_LPDBase):
    """Reference :18-114 (spelling kept; the CLI default featnet).  DGCNN-style edges [f_i ; f_j - f_i] for
    DG1 (128->64) + DG2 (64->64) + max, gather-only edges for SN1/SN2 (64->64) + max, conv3/4/5 64->64->128->emb."""

    def __init__(self, emb_dims=512, use_mFea=False, t3d=True, tfea=False, use_relu=False):
        super().__init__()
        self.negative_slope = 1e-2
        self.act_f = nn.ReLU(inplace=True) if use_relu else nn.LeakyReLU(negative_slope=self.negative_slope, inplace=True)
        self.use_mFea = use_mFea
        self.k = 20
        self.t3d = t3d
        self.tfea = tfea
        self.emb_dims = emb_dims
        if self.t3d:
            self.t_net3d = TranformNet(3)
        if self.tfea:
            self.t_net_fea = TranformNet(64)
        self.useBN = True
        a = self.act_f

        def c2(i, o):
            return nn.Sequential(nn.Conv2d(i, o, kernel_size=1, bias=False), nn.BatchNorm2d(o), a)

        def c1(i, o):
            return nn.Sequential(nn.Conv1d(i, o, kernel_size=1, bias=False), nn.BatchNorm1d(o), a)

        self.convDG1, self.convDG2 = c2(128, 64), c2(64, 64)
        self.convSN1, self.convSN2 = c2(64, 64), c2(64, 64)
        self.conv1_lpd, self.conv2_lpd = c1(8 if use_mFea else 3, 64), c1(64, 64)
        self.conv3_lpd, self.conv4_lpd, self.conv5_lpd = c1(64, 64), c1(64, 128), c1(128, self.emb_dims)
        self._prep = Prepared()

    def _build(self):
        p = {}
        for i, seq in enumerate((self.conv1_lpd, self.conv2_lpd, self.conv3_lpd, self.conv4_lpd, self.conv5_lpd), 1):
            p[f"w{i}"] = w2d(seq[0].weight)
            p[f"s{i}"], p[f"t{i}"] = fold_bn(seq[1])
        wdg1 = w2d(self.convDG1[0].weight)                     # [64, 128] = [Wa | Wb] on [f_i ; f_j - f_i] (reference :142)
        wa, wb = wdg1[:, :64], wdg1[:, 64:]
        p["wpq1"] = torch.cat((wb, wa - wb), 0).contiguous()   # P = Wb.f_j ; Q = (Wa - Wb).f_i
        p["wdg2"] = w2d(self.convDG2[0].weight)
        p["sdg1"], p["tdg1"] = fold_bn(self.convDG1[1])
        p["sdg2"], p["tdg2"] = fold_bn(self.convDG2[1])
        p["wsn1"], p["wsn2"] = w2d(self.convSN1[0].weight), w2d(self.convSN2[0].weight)
        p["ssn1"], p["tsn1"] = fold_bn(self.convSN1[1])
        p["ssn2"], p["tsn2"] = fold_bn(self.convSN2[1])
        # epilogue vectors of the DG1 projection for the pre-scaled f16 edge kernel: P' = s1 P, Q' = s1 Q + t1
        p["spq1"] = torch.cat((p["sdg1"], p["sdg1"])).contiguous()
        p["tpq1"] = torch.cat((torch.zeros_like(p["tdg1"]), p["tdg1"])).contiguous()
        if p["w3"].is_cuda:      # fp16 copies of the weights the "f16" precision mode multiplies with (rounded to nearest, once)
            for name in ("wdg2", "wsn1", "wsn2", "w3", "w4", "w5"):
                p[name + "_h"] = ops.to_f16(p[name])
        return p

    def forward_pm(self, x: torch.Tensor, keep_order: bool = False, f16: bool = False):
        """-> (F [B*N, emb] point-major, B, N), rows in spatial order unless keep_order (see LPDNet.forward_pm).
        f16 (PointNetVlad.forward in "f16" precision mode, k == 20 or 32): F and every activation downstream of the feature-space kNN
        are fp16 tensors; conv1 / conv2 and both kNN graphs stay exact fp32."""
        require_cuda(x, "LPDNetOrign")
        training_unsupported(self, "LPDNetOrign")
        p = self._prep.get(self, self._build)
        h, xyz_init, B, N = self._front(x, p, "LPDNetOrign", ops.SPATIAL_ORDER and not keep_order)
        M, k = B * N, self.k
        act, slope = _act_code(self)
        dev = h.device
        idx_f = ops.knn(h.view(B, N, 64), k)
        if f16 and k in (20, 32) and M >= 128 and self.emb_dims % 8 == 0:
            pq1 = ops.gemm_tf32_out16(h, p["wpq1"], M=M, N=128, K=64, scale=p["spq1"], shift=p["tpq1"])
            xdg = torch.empty(M, 64, device=dev, dtype=torch.float16)
            ops.edgeconv_dg64_f16(pq1, 128, pq1[:, 64:], 128, idx_f, B, N, p["wdg2_h"], p["sdg2"], p["tdg2"], act, slope, xdg, 64)
            del pq1
            idx_x = ops.knn(xyz_init, k)
            g = ops.gemm_f16(xdg, p["wsn1_h"], M=M, N=64, K=64, out_half=True, scale=p["ssn1"], shift=p["tsn1"], act=act, slope=slope)
            g = ops.gemm_f16(g, p["wsn2_h"], M=M, N=64, K=64, out_half=True, scale=p["ssn2"], shift=p["tsn2"], act=act, slope=slope)
            xsn = torch.empty(M, 64, device=dev, dtype=torch.float16)
            ops.edge_gather_max_f16(g, 64, None, 0, idx_x, B, N, k, 64, ops.ACT_NONE, 0.0, xsn, 64)
            f = ops.gemm_f16(xsn, p["w3_h"], M=M, N=64, K=64, out_half=True, scale=p["s3"], shift=p["t3"], act=act, slope=slope)
            f = ops.gemm_f16(f, p["w4_h"], M=M, N=128, K=64, out_half=True, scale=p["s4"], shift=p["t4"], act=act, slope=slope)
            f = ops.gemm_f16(f, p["w5_h"], M=M, N=self.emb_dims, K=128, out_half=True, scale=p["s5"], shift=p["t5"], act=act, slope=slope)
            return f, B, N
        pq1 = ops.linear(h, p["wpq1"], M=M, N=128, K=64)
        xdg = torch.empty(M, 64, device=dev, dtype=torch.float32)
        ops.edgeconv_dg(pq1, 128, pq1[:, 64:], 128, idx_f, B, N, k, 64, 64, p["sdg1"], p["tdg1"], p["wdg2"],
                        p["sdg2"], p["tdg2"], act, slope, None, 0, xdg, 64)
        # gather-only edges: SN1 and SN2 act on each neighbour independently -> evaluate them per POINT, then max-gather
        idx_x = ops.knn(xyz_init, k)
        g = ops.linear(xdg, p["wsn1"], M=M, N=64, K=64, scale=p["ssn1"], shift=p["tsn1"], act=act, slope=slope)
        g = ops.linear(g, p["wsn2"], M=M, N=64, K=64, scale=p["ssn2"], shift=p["tsn2"], act=act, slope=slope)
        xsn = torch.empty(M, 64, device=dev, dtype=torch.float32)
        ops.edge_gather_ext(g, 64, None, 0, idx_x, B, N, k, 64, None, None, ops.ACT_NONE, 0.0, xsn, 64)
        f = ops.linear(xsn, p["w3"], M=M, N=64, K=64, scale=p["s3"], shift=p["t3"], act=act, slope=slope)
        f = ops.linear(f, p["w4"], M=M, N=128, K=64, scale=p["s4"], shift=p["t4"], act=act, slope=slope)
        f = ops.linear(f, p["w5"], M=M, N=self.emb_dims, K=128, scale=p["s5"], shift=p["t5"], act=act, slope=slope)
        return f, B, N

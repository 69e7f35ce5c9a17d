"""Drop-in for the reference's util/PointNetVlad.py: PointNetVlad, NetVLADLoupe, GatingContext, STN3d,
PointNetfeat, Flatten — same constructor signatures, attribute names, state_dict keys and public tensor
layouts.  All arithmetic is in liblpd_b200.so.

PointNetVlad.forward hands the point-major [B*N, D] feature map of the feature net straight to NetVLAD,
which removes the [B,D,N,1] -> [B,N,D] transpose copy of the reference (:46-47); the individual modules
still honour the reference layouts when called on their own.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import ops
from .._host import Prepared, fold_bn, require_cuda, training_unsupported, w2d
from .lpdnet_model import LPDNet, LPDNetOrign

__all__ = ["PointNetVlad", "NetVLADLoupe", "GatingContext", "STN3d", "PointNetfeat", "Flatten"]


class GatingContext(nn.Module):
    """Reference :86-115: x * sigmoid(BN(x . W_g)) (or + gating_biases)."""

    def __init__(self, dim, add_batch_norm=True):
        super().__init__()
        self.dim = dim
        self.add_batch_norm = add_batch_norm
        self.gating_weights = nn.Parameter(torch.randn(dim, dim) * 1 / math.sqrt(dim))
        self.sigmoid = nn.Sigmoid()
        if add_batch_norm:
            self.gating_biases = None
            self.bn1 = nn.BatchNorm1d(dim)
        else:
            self.gating_biases = nn.Parameter(torch.randn(dim) * 1 / math.sqrt(dim))
            self.bn1 = None
        self._prep = Prepared()

    def _build(self):
        if self.add_batch_norm:
            s, t = fold_bn(self.bn1)
        else:
            s, t = None, self.gating_biases.detach()
        return {"w": self.gating_weights.detach().contiguous(), "s": s, "t": t}

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        require_cuda(x, "GatingContext")
        training_unsupported(self, "GatingContext")
        p = self._prep.get(self, self._build)
        x = x.detach().contiguous()
        B = x.size(0)
        return ops.gemm(x, p["w"], b_layout=ops.B_KN, M=B, N=self.dim, K=self.dim, scale=p["s"], shift=p["t"],
                        act=ops.ACT_GATE, aux=x)


class NetVLADLoupe(nn.Module):
    """Reference :12-83."""

    HIDDEN_SPLITS = 128  # split-K factor of the (K*D) x output_dim hidden projection

    def __init__(self, feature_size, max_samples, cluster_size, output_dim,
                 gating=True, add_batch_norm=True, is_training=True):
        super().__init__()
        self.feature_size = feature_size
        self.max_samples = max_samples
        self.output_dim = output_dim
        self.is_training = is_training
        self.gating = gating
        self.add_batch_norm = add_batch_norm
        self.cluster_size = cluster_size
        self.softmax = nn.Softmax(dim=-1)
        self.cluster_weights = nn.Parameter(torch.randn(feature_size, cluster_size) * 1 / math.sqrt(feature_size))
        self.cluster_weights2 = nn.Parameter(torch.randn(1, feature_size, cluster_size) * 1 / math.sqrt(feature_size))
        self.hidden1_weights = nn.Parameter(torch.randn(cluster_size * feature_size, output_dim) * 1 / math.sqrt(feature_size))
        if add_batch_norm:
            self.cluster_biases = None
            self.bn1 = nn.BatchNorm1d(cluster_size)
        else:
            self.cluster_biases = nn.Parameter(torch.randn(cluster_size) * 1 / math.sqrt(feature_size))
            self.bn1 = None
        self.bn2 = nn.BatchNorm1d(output_dim)
        if gating:
            self.context_gating = GatingContext(output_dim, add_batch_norm=add_batch_norm)
        self._prep = Prepared()

    def _build(self):
        p = {"wc": self.cluster_weights.detach().contiguous(), "wc2": self.cluster_weights2.detach()[0].contiguous(),
             "wh": self.hidden1_weights.detach().contiguous()}
        p["wct"] = ops.transpose(p["wc"].unsqueeze(0))[0]      # [K, D]: K-contiguous operand for the tensor-core path
        if p["wct"].is_cuda:
            p["wct_h"] = ops.to_f16(p["wct"])                  # "f16" precision mode
            p["wh3"] = ops.split3_tf32(p["wh"], 1)             # TF32 hi / lo split of the hidden weights, stacked [hi; lo; hi]
        if self.add_batch_norm:
            p["s1"], p["t1"] = fold_bn(self.bn1)
        else:
            p["s1"], p["t1"] = None, self.cluster_biases.detach()
        p["s2"], p["t2"] = fold_bn(self.bn2)
        return p

    def forward_pm(self, f: torch.Tensor, B: int) -> torch.Tensor:
        """f [B*max_samples, feature_size] point-major -> [B, output_dim]"""
        training_unsupported(self, "NetVLADLoupe")
        if self.cluster_size != 64:
            raise NotImplementedError("the NetVLAD kernels are specialised for cluster_size == 64 (the reference's value)")
        p = self._prep.get(self, self._build)
        N, D, K, O = self.max_samples, self.feature_size, self.cluster_size, self.output_dim
        M = B * N
        # softmax (and the 32-row partial sums of a_sum) as the epilogue of the assignment GEMM; the cluster finish kernel takes the partials
        fused = N % 32 == 0 and D % 128 == 0 and D <= 1024 and M >= 128
        apart = None
        if f.dtype == torch.float16:                                                          # "f16" mode: F arrives as fp16
            if fused:
                a, a_h, apart = ops.gemm_softmax64(f, p["wct_h"], M=M, K=D, scale=p["s1"], shift=p["t1"], want32=False, want16=True,
                                                   want_parts=True)                           # :48-59
            else:
                a, a_h = ops.softmax64_f16(ops.gemm_f16(f, p["wct_h"], M=M, N=K, K=D, scale=p["s1"], shift=p["t1"]), M)
            vraw = ops.gemm_f16_tn(f, a_h, M=D, N=K, K=N, lda=D, ldb=K, batch=B)              # :64-66 -> [B, D, K]
        elif ops.get_precision() != "fp32" and M >= 128 and D % 4 == 0:                       # :48-59
            if fused:
                a, _, apart = ops.gemm_softmax64(f, p["wct"], M=M, K=D, scale=p["s1"], shift=p["t1"], want_parts=True)
            else:
                a = ops.softmax64(ops.gemm_tf32(f, p["wct"], M=M, N=K, K=D, scale=p["s1"], shift=p["t1"]), M)
        else:
            a = ops.netvlad_assign(f, M, D, p["wc"], p["s1"], p["t1"], K)
        if f.dtype == torch.float16:
            pass
        elif ops._tn_ok(f, a, D, K, N, D, K, B):
            vraw = ops.gemm_tf32_tn(f, a, M=D, N=K, K=N, lda=D, ldb=K, batch=B)               # :64-66 -> [B, D, K]
        else:
            vraw = ops.gemm(f, a, a_layout=ops.A_KM, b_layout=ops.B_KN, M=D, N=K, K=N, lda=D, ldb=K, batch=B,
                            strideA=N * D, strideB=N * K)
        if B == 1:
            vraw = vraw.view(1, D, K)
        if apart is not None:
            v = ops.netvlad_finish_parts(vraw, apart, N // 32, p["wc2"], B, D, K)             # :61-62,:68-74 -> [B, D*K]
        else:
            v = ops.netvlad_finish(vraw, a, p["wc2"], B, N, D, K)
        KD = D * K
        splits = self.HIDDEN_SPLITS
        while KD % splits:
            splits //= 2
        kc = KD // splits
        if ops.get_precision() != "fp32" and (3 * kc) % 32 == 0 and O % 4 == 0 and O <= 256 and "wh3" in p:
            # the (K*D) x output_dim projection on the tensor cores at fp32 accuracy ("3xTF32"): out[b][o] = sum_r vT[r][b] W_h[r][o] is
            # a contraction over the ROWS of two row-major matrices (vT = the transposed descriptors, W_h as stored), both split
            # into TF32 hi + lo parts stacked along the rows ([hi; hi; lo] x [hi; lo; hi]: hi.hi + hi.lo + lo.hi), cut into
            # `splits` slices = one tcgen05 tile per CTA; the partial sums are reduced in fixed order with the BatchNorm affine.
            # (A single-pass TF32 / fp16 projection is 2 x faster still but doubles the descriptor error: this layer feeds a
            # BatchNorm whose scale amplifies it.)
            Bp = (B + 3) // 4 * 4
            part = ops.gemm_tf32_tn(ops.transpose_split3(v, Bp), p["wh3"], M=B, N=O, K=3 * kc, lda=Bp, ldb=O, batch=splits)   # :76
        else:
            part = torch.empty(splits, B, O, device=f.device, dtype=torch.float32)
            ops.gemm(v, p["wh"], a_layout=ops.A_MK, b_layout=ops.B_KN, M=B, N=O, K=kc, lda=KD, ldb=O, out=part, ldc=O,
                     batch=splits, strideA=kc, strideB=kc * O, strideC=B * O)                 # :76
        if self.gating and O <= 1024:                                                         # :78-81 in one launch
            g = self.context_gating._prep.get(self.context_gating, self.context_gating._build)
            return ops.hidden_gate(part, splits, B, O, p["s2"], p["t2"], g["w"], g["s"], g["t"])
        h = ops.splitk_reduce(part, splits, B, O, p["s2"], p["t2"])                           # :78
        if self.gating:
            h = self.context_gating(h)                                                        # :80-81
        return h

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [B, feature_size, max_samples, 1] (reference layout, :45-47) -> [B, output_dim]"""
        require_cuda(x, "NetVLADLoupe")
        B = x.size(0)
        f = ops.transpose(x.detach().reshape(B, self.feature_size, -1))                       # [B, N, D]
        if f.size(1) != self.max_samples:
            raise ValueError(f"NetVLADLoupe: got {f.size(1)} samples, constructed for max_samples={self.max_samples}")
        return self.forward_pm(f.view(B * self.max_samples, self.feature_size), B)


class Flatten(nn.Module):
    def forward(self, input):
        return input.view(input.size(0), -1)


class STN3d(nn.Module):
    """Reference :126-179.  Spatial transformer: (1,k')-conv 64 -> 128 -> 1024, max over num_points, 512 -> 256 -> k*k + I."""

    def __init__(self, num_points=2500, k=3, use_bn=True):
        super().__init__()
        self.k = k
        self.kernel_size = 3 if k == 3 else 1
        self.channels = 1 if k == 3 else k
        self.num_points = num_points
        self.use_bn = use_bn
        self.conv1 = nn.Conv2d(self.channels, 64, (1, self.kernel_size))
        self.conv2 = nn.Conv2d(64, 128, (1, 1))
        self.conv3 = nn.Conv2d(128, 1024, (1, 1))
        self.mp1 = nn.MaxPool2d((num_points, 1), 1)
        self.fc1 = nn.Linear(1024, 512)
        self.fc2 = nn.Linear(512, 256)
        self.fc3 = nn.Linear(256, k * k)
        self.fc3.weight.data.zero_()
        self.fc3.bias.data.zero_()
        self.relu = nn.ReLU()
        if use_bn:
            self.bn1 = nn.BatchNorm2d(64)
            self.bn2 = nn.BatchNorm2d(128)
            self.bn3 = nn.BatchNorm2d(1024)
            self.bn4 = nn.BatchNorm1d(512)
            self.bn5 = nn.BatchNorm1d(256)
        self._prep = Prepared()

    def _build(self):
        p = {}
        layers = (self.conv1, self.conv2, self.conv3, self.fc1, self.fc2)
        for i, lin in enumerate(layers, 1):
            p[f"w{i}"] = w2d(lin.weight)
            if self.use_bn:
                p[f"s{i}"], p[f"t{i}"] = fold_bn(getattr(self, f"bn{i}"), lin.bias)
            else:
                p[f"s{i}"], p[f"t{i}"] = None, lin.bias.detach()
        p["w6"] = w2d(self.fc3.weight)
        p["t6"] = self.fc3.bias.detach() + torch.eye(self.k, device=self.fc3.bias.device).reshape(-1)
        if p["w3"].is_cuda:      # fp16 copies of the weights the "f16" precision mode multiplies with (rounded to nearest, once)
            p["w3_h"] = ops.to_f16(p["w3"])
            if self.k == 64:
                p["w2_h"] = ops.to_f16(p["w2"])
        return p

    def forward_pm(self, rows: torch.Tensor, B: int, N: int, f16: bool = False) -> torch.Tensor:
        """rows [B*N, k] point-major -> [B, k, k].
        f16 (PointNetfeat.forward_pm in "f16" precision mode; needs N % 32 == 0): the per-point activations that feed conv3 (and conv2 for
        k == 64) are fp16 tensors, and conv3 + ReLU + max over the points run in one call without writing the [B*N, 1024] map;
        fc1-fc3 stay fp32."""
        if self.use_bn:
            training_unsupported(self, "STN3d")
        if N != self.num_points:
            raise ValueError(f"STN3d: got {N} points, constructed for num_points={self.num_points} "
                             f"(the reference's MaxPool2d((num_points,1)) silently mis-pools here)")
        p = self._prep.get(self, self._build)
        M, R = B * N, ops.ACT_RELU
        if f16:
            if self.k == 3:     # K = 3: fp32 CUDA-core layer, fp32 operands of conv2 consumed as TF32
                h = ops.linear(rows, p["w1"], M=M, N=64, K=3, scale=p["s1"], shift=p["t1"], act=R)
                h = ops.gemm_tf32_out16(h, p["w2"], M=M, N=128, K=64, scale=p["s2"], shift=p["t2"], act=R)
            else:
                h = ops.gemm_tf32_out16(rows, p["w1"], M=M, N=64, K=self.k, scale=p["s1"], shift=p["t1"], act=R)
                h = ops.gemm_f16(h, p["w2_h"], M=M, N=128, K=64, out_half=True, scale=p["s2"], shift=p["t2"], act=R)
            g = ops.gemm_f16_colmax(h, p["w3_h"], M=M, N=1024, K=128, R=N, scale=p["s3"], shift=p["t3"], act=R, slope=0.0)
        else:
            h = ops.linear(rows, p["w1"], M=M, N=64, K=self.k, scale=p["s1"], shift=p["t1"], act=R)
            h = ops.linear(h, p["w2"], M=M, N=128, K=64, scale=p["s2"], shift=p["t2"], act=R)
            h = ops.linear(h, p["w3"], M=M, N=1024, K=128, scale=p["s3"], shift=p["t3"], act=R)
            g = ops.colmax(h, B, N, 1024)
        g = ops.linear(g, p["w4"], M=B, N=512, K=1024, scale=p["s4"], shift=p["t4"], act=R)
        g = ops.linear(g, p["w5"], M=B, N=256, K=512, scale=p["s5"], shift=p["t5"], act=R)
        g = ops.linear(g, p["w6"], M=B, N=self.k * self.k, K=256, shift=p["t6"])
        return g.view(B, self.k, self.k)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [B, 1, N, 3] (k == 3) or [B, k, N, 1] -> [B, k, k]"""
        require_cuda(x, "STN3d")
        B = x.size(0)
        if self.k == 3:
            N = x.size(2)
            rows = x.detach().reshape(B * N, 3).contiguous()
        else:
            N = x.size(2)
            rows = ops.transpose(x.detach().reshape(B, self.k, N)).view(B * N, self.k)
        return self.forward_pm(rows, B, N)


class PointNetfeat(nn.Module):
    """Reference :181-241."""

    def __init__(self, num_points=2500, global_feat=True, feature_transform=False, max_pool=True, emb_dims=1024):
        super().__init__()
        self.stn = STN3d(num_points=num_points, k=3, use_bn=False)
        self.feature_trans = STN3d(num_points=num_points, k=64, use_bn=False)
        self.apply_feature_trans = feature_transform
        self.conv1 = nn.Conv2d(1, 64, (1, 3))
        self.conv2 = nn.Conv2d(64, 64, (1, 1))
        self.conv3 = nn.Conv2d(64, 64, (1, 1))
        self.conv4 = nn.Conv2d(64, 128, (1, 1))
        self.conv5 = nn.Conv2d(128, emb_dims, (1, 1))
        self.bn1 = nn.BatchNorm2d(64)
        self.bn2 = nn.BatchNorm2d(64)
        self.bn3 = nn.BatchNorm2d(64)
        self.bn4 = nn.BatchNorm2d(128)
        self.bn5 = nn.BatchNorm2d(emb_dims)
        self.mp1 = nn.MaxPool2d((num_points, 1), 1)
        self.num_points = num_points
        self.global_feat = global_feat
        self.max_pool = max_pool
        self.emb_dims = emb_dims
        self._prep = Prepared()

    def _build(self):
        p = {}
        for i in range(1, 6):
            conv, bn = getattr(self, f"conv{i}"), getattr(self, f"bn{i}")
            p[f"w{i}"] = w2d(conv.weight)
            p[f"s{i}"], p[f"t{i}"] = fold_bn(bn, conv.bias)
        if p["w4"].is_cuda:      # fp16 copies of the weights the "f16" precision mode multiplies with (rounded to nearest, once)
            p["w4_h"], p["w5_h"] = ops.to_f16(p["w4"]), ops.to_f16(p["w5"])
        return p

    def forward_pm(self, x: torch.Tensor, f16: bool = False):
        """x [B,1,N,3] -> (F [B*N, emb] point-major (before any pooling), trans [B,3,3], h2 [B*N,64], B, N).
        f16 (PointNetVlad.forward in "f16" precision mode; needs N % 32 == 0): both STNs take their f16 form, conv3-conv5 keep fp16
        activations and F is an fp16 tensor; the input transform, conv1 / conv2 (h2) and the feature transform stay fp32."""
        require_cuda(x, "PointNetfeat")
        training_unsupported(self, "PointNetfeat")
        p = self._prep.get(self, self._build)
        B, _, N, _ = x.shape
        M, R = B * N, ops.ACT_RELU
        rows = x.detach().reshape(M, 3).contiguous()
        trans = self.stn.forward_pm(rows, B, N, f16=f16)                                      # :205
        xt = ops.gemm(rows, trans, b_layout=ops.B_KN, M=N, N=3, K=3, lda=3, ldb=3, batch=B,
                      strideA=N * 3, strideB=9, strideC=N * 3,
                      out=torch.empty(M, 3, device=x.device, dtype=torch.float32), ldc=3)     # :209
        if f16:                                                                               # :213-215 in one strict-fp32 pass
            h2 = ops.pointwise_mlp2(xt, 3, M, p["w1"], p["s1"], p["t1"], p["w2"], p["s2"], p["t2"], act=R)
        else:
            h = ops.linear(xt, p["w1"], M=M, N=64, K=3, scale=p["s1"], shift=p["t1"], act=R)     # :213
            h2 = ops.linear(h, p["w2"], M=M, N=64, K=64, scale=p["s2"], shift=p["t2"], act=R)    # :215
        h = h2
        if self.apply_feature_trans:                                                          # :218-225
            ft = self.feature_trans.forward_pm(h2, B, N, f16=f16)
            h = ops.gemm(h2, ft, b_layout=ops.B_KN, M=N, N=64, K=64, lda=64, ldb=64, batch=B,
                         strideA=N * 64, strideB=64 * 64, strideC=N * 64,
                         out=torch.empty(M, 64, device=x.device, dtype=torch.float32), ldc=64)
        if f16:
            h = ops.gemm_tf32_out16(h, p["w3"], M=M, N=64, K=64, scale=p["s3"], shift=p["t3"], act=R)                 # :226
            h = ops.gemm_f16(h, p["w4_h"], M=M, N=128, K=64, out_half=True, scale=p["s4"], shift=p["t4"], act=R)       # :228
            f = ops.gemm_f16(h, p["w5_h"], M=M, N=self.emb_dims, K=128, out_half=True, scale=p["s5"], shift=p["t5"])   # :230
            return f, trans, h2, B, N
        h = ops.linear(h, p["w3"], M=M, N=64, K=64, scale=p["s3"], shift=p["t3"], act=R)         # :226
        h = ops.linear(h, p["w4"], M=M, N=128, K=64, scale=p["s4"], shift=p["t4"], act=R)        # :228
        f = ops.linear(h, p["w5"], M=M, N=self.emb_dims, K=128, scale=p["s5"], shift=p["t5"])    # :230 (no ReLU)
        return f, trans, h2, B, N

    def forward(self, x: torch.Tensor):
        f, trans, h2, B, N = self.forward_pm(x)
        if not self.max_pool:
            return ops.transpose(f.view(B, N, self.emb_dims)).unsqueeze(-1)                   # [B, emb, N, 1]
        if N != self.num_points:
            raise ValueError(f"PointNetfeat: got {N} points, constructed for num_points={self.num_points}")
        g = ops.colmax(f, B, N, self.emb_dims)                                                # :235-236
        if self.global_feat:
            return g, trans
        pointfeat = ops.transpose(h2.view(B, N, 64)).unsqueeze(-1)                            # [B, 64, N, 1]
        g = g.view(B, self.emb_dims, 1).repeat(1, 1, self.num_points)
        return torch.cat([g, pointfeat], 1), trans                                            # as written at :240-241


class PointNetVlad(nn.Module):
    """Reference :244-270: featnet switch (lpdnet / pointnet / lpdnetorigin) + NetVLADLoupe(K=64) -> [B, output_dim]."""

    def __init__(self, num_points=4096, global_feat=True, feature_transform=False, max_pool=False, output_dim=256,
                 emb_dims=1024, featnet="lpdnet", xyz_trans=False):
        super().__init__()
        if featnet == "lpdnet":
            self.emb_nn = LPDNet(emb_dims=emb_dims, tfea=feature_transform, t3d=xyz_trans)
        elif featnet == "pointnet":
            self.emb_nn = None
            self.point_net = PointNetfeat(num_points=num_points, global_feat=global_feat,
                                          feature_transform=feature_transform, max_pool=max_pool, emb_dims=emb_dims)
        elif featnet == "lpdnetorigin":
            self.emb_nn = LPDNetOrign(emb_dims=emb_dims, tfea=feature_transform, t3d=xyz_trans)
        else:
            print("featnet error")  # the reference only prints (:256) and fails later; fail here instead
            raise ValueError(f"featnet error: {featnet!r}")
        self.net_vlad = NetVLADLoupe(feature_size=emb_dims, max_samples=num_points, cluster_size=64,
                                     output_dim=output_dim, gating=True, add_batch_norm=True, is_training=True)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.training:
            # batch-statistics BatchNorm + hand-written backward behind one autograd node (lpdnet_b200/train.py)
            from ..train import forward_train
            return forward_train(self, x)
        # "f16" precision mode: fp16 activations (downstream of the kNN for the LPD nets), for the configurations the kernels are
        # specialised for.  N % 64 == 0: the fp16 NetVLAD aggregate contracts each cloud's N rows in 64-row k-blocks.
        f16 = (ops.get_precision() == "f16" and x.size(2) % 64 == 0 and x.size(0) * x.size(2) >= 128
               and self.net_vlad.cluster_size == 64 and self.net_vlad.feature_size % 8 == 0)
        if self.emb_nn is not None:
            f16 = f16 and isinstance(self.emb_nn, (LPDNet, LPDNetOrign)) and self.emb_nn.k in (20, 32)
            f, B, N = self.emb_nn.forward_pm(x, f16=True) if f16 else self.emb_nn.forward_pm(x)
        else:
            if self.point_net.max_pool:
                raise ValueError("PointNetVlad needs the per-point feature map: construct with max_pool=False")
            f, _, _, B, N = self.point_net.forward_pm(x, f16=f16)
        if N != self.net_vlad.max_samples:
            raise ValueError(f"PointNetVlad: got {N} points per cloud, constructed for num_points={self.net_vlad.max_samples}")
        return self.net_vlad.forward_pm(f, B)

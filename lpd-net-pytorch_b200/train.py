"""Train-mode execution of the hot path: forward with batch-statistics BatchNorm, hand-written backward, all through
the C ABI (include/lpd_b200.h, "TRAIN MODE").  Replaces what torch autograd does for the reference in
train_pointnetvlad.py:121-130,150-159 (model.train(); output = model(feed); loss.backward(); optimizer.step()).

The public entry is `forward_train(model, x)`: it returns the [B, output_dim] descriptors as a tensor that is attached
to the autograd graph through ONE torch.autograd.Function whose backward runs the kernels below and hands the
parameter gradients back to torch (so `loss.backward()` fills `.grad` exactly as in the reference and any
torch.optim optimizer, or lpdnet_b200.optim.Adam, can step).  torch itself does no arithmetic here: it owns the device
memory, the current stream and the parameter / gradient storage.

Layout: feature maps are point-major [rows, C]; every layer object below keeps what its backward needs.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from ._host import require_cuda, w2d
from ._lib import LpdError

A_MK, A_KM, B_NK, B_KN = ops.A_MK, ops.A_KM, ops.B_NK, ops.B_KN


def dgrad(dz, lddz, w, rows, N, K, out=None, ldc=None, accumulate=False, tf32_ok=True):
    """da[r][k] (+)= sum_n dz[r][n] * w[n][k]   (input gradient of z = a . w^T, w [N, K]).
    In "tf32" precision mode the product runs on the tensor cores against a transposed copy of the (small) weight."""
    if (tf32_ok and ops.get_precision() != "fp32" and N >= 32 and N % 4 == 0 and lddz % 4 == 0 and K >= 64
            and K % 4 == 0 and rows >= 128 and (ldc is None or ldc % 4 == 0) and dz.data_ptr() % 16 == 0
            and (out is None or out.data_ptr() % 16 == 0)):
        wt = ops.transpose(w.unsqueeze(0))[0]                                   # [K, N]
        return ops.gemm_tf32(dz, wt, M=rows, N=K, K=N, lda=lddz, out=out, ldc=ldc, accumulate=accumulate)
    return ops.gemm(dz, w, a_layout=A_MK, b_layout=B_KN, M=rows, N=K, K=N, lda=lddz, ldb=K, out=out, ldc=ldc,
                    act=ops.ACT_ADD if accumulate else ops.ACT_NONE, aux=out if accumulate else None)


# ----------------------------------------------------------------------------------------------------------------------
# layer records
# ----------------------------------------------------------------------------------------------------------------------
class _Grads:
    """parameter -> gradient tensor (in the parameter's own shape); accumulates when a parameter is hit twice.
    A gradient declared `final` (no later contribution in this backward) is offered to the parameter's gradient sink, if it
    has one: lpdnet_b200.optim.Adam registers itself on its large parameters so that their data-parallel all-reduce starts
    while the rest of the backward is still running."""

    def __init__(self):
        self.by_param = {}

    def add(self, param: torch.Tensor, g: torch.Tensor, final: bool = False):
        g = g.reshape(param.shape)
        if final and param not in self.by_param:
            sink = getattr(param, "_lpd_grad_sink", None)
            sink = sink() if sink is not None else None
            if sink is not None and sink.grad_ready(param, g.contiguous()):
                return                                       # the optimizer owns it now: autograd gets None for this parameter
        cur = self.by_param.get(param)
        if cur is None:
            self.by_param[param] = g.contiguous()
        else:
            n = cur.numel()
            ops.axpy(cur.view(1, n), n, g.contiguous().view(1, n), n, 1, n, 1.0)


class Linear:
    """z = a . W^T (+ bias)     a [rows, K] (lda), W [N, K] (a conv1x1 / nn.Linear weight)"""

    def fwd(self, a, lda, rows, weight: nn.Parameter, bias=None, tf32_ok=True):
        self.a, self.lda, self.rows = a, lda, rows
        self.weight, self.bias = weight, bias
        self.w = w2d(weight)
        self.N, self.K = self.w.shape
        self.tf32_ok = tf32_ok
        lin = ops.linear if tf32_ok else ops.gemm
        return lin(a, self.w, M=rows, N=self.N, K=self.K, lda=lda, shift=None if bias is None else bias.detach())

    def bwd(self, dz, lddz, grads: _Grads, need_da=True, da_out=None, ldda=None, accumulate=False):
        grads.add(self.weight, ops.wgrad(dz, lddz, self.a, self.lda, self.rows, self.N, self.K))
        if self.bias is not None:
            if self.N % 4 == 0 and lddz % 4 == 0:
                part, nparts = ops.bn_stats(dz, self.rows, self.N, lddz)
                grads.add(self.bias, ops.colsum_finalize(part, nparts, 2 * self.N)[: self.N])
            else:   # few columns (fc3 of the 3x3 T-Net): ones . dz
                ones = torch.ones(1, self.rows, device=dz.device, dtype=torch.float32)
                grads.add(self.bias, ops.gemm(ones, dz, a_layout=A_MK, b_layout=B_KN, M=1, N=self.N, K=self.rows, ldb=lddz))
        if not need_da:
            return None
        return dgrad(dz, lddz, self.w, self.rows, self.N, self.K, out=da_out, ldc=ldda, accumulate=accumulate, tf32_ok=self.tf32_ok)


def _bn_params(bn: nn.modules.batchnorm._BatchNorm):
    g = bn.weight.detach() if bn.affine else None
    b = bn.bias.detach() if bn.affine else None
    mom = 0.1 if bn.momentum is None else bn.momentum
    return g, b, mom


def _bn_finalize(bn: nn.modules.batchnorm._BatchNorm, part, nparts, count, C):
    g, b, mom = _bn_params(bn)
    track = bn.track_running_stats and bn.running_mean is not None
    blk = ops.bn_finalize(part, nparts, count, C, g, b, bn.eps, mom, bn.running_mean if track else None,
                          bn.running_var if track else None)
    if track and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)       # bookkeeping counter (int64 buffer), as torch does
    return blk


class BNAct:
    """y = act(BatchNorm_batch(z))   z [rows, C] (ldz); statistics over the rows"""

    def fwd(self, z, ldz, rows, C, bn: nn.modules.batchnorm._BatchNorm, act=ops.ACT_NONE, slope=0.0, aux=None, ldaux=0,
            out=None, ldo=None):
        self.z, self.ldz, self.rows, self.C, self.bn_mod = z, ldz, rows, C, bn
        self.act, self.slope, self.aux, self.ldaux = act, slope, aux, ldaux
        part, nparts = ops.bn_stats(z, rows, C, ldz)
        self.bn = _bn_finalize(bn, part, nparts, rows, C)
        return ops.affine_act(z, rows, C, ldz, self.bn[0], self.bn[1], act, slope, aux, ldaux, out, ldo)

    def bwd(self, dy, lddy, grads: _Grads, inplace=True):
        dz, S = ops.bn_bwd(dy, lddy, self.z, self.ldz, self.rows, self.C, self.bn, self.act, self.slope, aux=self.aux,
                           ldaux=self.ldaux, dz=dy if inplace else None, lddz=lddy if inplace else None)
        if self.bn_mod.affine:
            grads.add(self.bn_mod.bias, S[0])
            grads.add(self.bn_mod.weight, S[1])
        return dz


class ActOnly:
    """y = act(z) after a BatchNorm-free layer (STN3d(use_bn=False), reference PointNetVlad.py:160-167)"""

    def fwd(self, z, ldz, rows, C, act, slope=0.0):
        self.z, self.ldz, self.rows, self.C, self.act, self.slope = z, ldz, rows, C, act, slope
        return ops.affine_act(z, rows, C, ldz, None, None, act, slope)

    def bwd(self, dy, lddy, grads=None):
        return ops.act_bwd(dy, lddy, self.z, self.ldz, self.rows, self.C, self.act, self.slope, dz=dy, lddz=lddy)


def _norm_act(bn_mod):
    """BNAct when the layer has a BatchNorm module, else ActOnly (same fwd/bwd call shape)"""
    return BNAct() if bn_mod is not None else ActOnly()


def _fwd_norm_act(layer, z, ldz, rows, C, bn_mod, act, slope=0.0):
    if bn_mod is not None:
        return layer.fwd(z, ldz, rows, C, bn_mod, act, slope)
    return layer.fwd(z, ldz, rows, C, act, slope)


class ColMax:
    """g[b][c] = max_n h[b][n][c]  (torch.max(x, 2) lpdnet_model.py:300 / MaxPool2d((num_points,1)) PointNetVlad.py:169)"""

    def fwd(self, h, B, N, C):
        self.B, self.N, self.C = B, N, C
        g, self.arg = ops.colmax_arg(h, B, N, C)
        return g

    def bwd(self, dg):
        dh = torch.zeros(self.B * self.N, self.C, device=dg.device, dtype=torch.float32)
        return ops.colmax_bwd(dg.contiguous(), self.arg, self.B, self.N, self.C, dh, self.C)


class Transform:
    """out[b][:, :C] = rows[b][:, :C] . T[b]   (torch.bmm / matmul with a T-Net output: lpdnet_model.py:86,93,229,241;
    PointNetVlad.py:209,223).  keep_tail: rows wider than C (the 8-d use_mFea input, lpdnet_model.py:215-222) keep their
    remaining columns, i.e. the output is [B*N, ld] again."""

    def fwd(self, rows, ld, trans, B, N, C, keep_tail=False):
        self.rows, self.ld, self.trans, self.B, self.N, self.C = rows, ld, trans.contiguous(), B, N, C
        self.ldo = ld if (keep_tail and ld != C) else C
        out = rows.clone() if self.ldo != C else torch.empty(B * N, C, device=rows.device, dtype=torch.float32)
        ops.gemm(rows, self.trans, a_layout=A_MK, b_layout=B_KN, M=N, N=C, K=C, lda=ld, ldb=C, out=out, ldc=self.ldo,
                 batch=B, strideA=N * ld, strideB=C * C, strideC=N * self.ldo)
        return out

    def bwd(self, dout, need_drows, lddout=None):
        B, N, C = self.B, self.N, self.C
        ldd = C if lddout is None else lddout
        # dT[b] = rows[b]^T . dout[b]
        dtrans = ops.gemm(self.rows, dout, a_layout=A_KM, b_layout=B_KN, M=C, N=C, K=N, lda=self.ld, ldb=ldd, batch=B,
                          strideA=N * self.ld, strideB=N * ldd, strideC=C * C,
                          out=torch.empty(B, C, C, device=dout.device, dtype=torch.float32), ldc=C)
        drows = None
        if need_drows:   # drows[b][n][c] = sum_c' dout[b][n][c'] T[b][c][c']
            drows = ops.gemm(dout, self.trans, a_layout=A_MK, b_layout=B_NK, M=N, N=C, K=C, lda=ldd, ldb=C, batch=B,
                             strideA=N * ldd, strideB=C * C, strideC=N * C,
                             out=torch.empty(B * N, C, device=dout.device, dtype=torch.float32), ldc=C)
        return drows, dtrans


class TNetTrain:
    """TranformNet (lpdnet_model.py:273-313, BatchNorm everywhere) and STN3d (PointNetVlad.py:126-179, BatchNorm optional):
    k -> 64 -> 128 -> 1024 (+norm +ReLU), max over the points, 1024 -> 512 -> 256 (+norm +ReLU) -> k*k, + identity."""

    def __init__(self, net):
        self.net = net
        self.has_bn = getattr(net, "use_bn", True)

    def _bn(self, i):
        return getattr(self.net, f"bn{i}") if self.has_bn else None

    def fwd(self, rows, ld, B, N):
        net, k, R = self.net, self.net.k, ops.ACT_RELU
        M = B * N
        self.B, self.N, self.M = B, N, M
        self.lin = [Linear() for _ in range(6)]
        self.na = [_norm_act(self._bn(i)) for i in range(1, 6)]
        h, ldh = rows, ld
        for i, (conv, C) in enumerate(((net.conv1, 64), (net.conv2, 128), (net.conv3, 1024))):
            z = self.lin[i].fwd(h, ldh, M, conv.weight, conv.bias, tf32_ok=False)
            h = _fwd_norm_act(self.na[i], z, C, M, C, self._bn(i + 1), R)
            ldh = C
        self.pool = ColMax()
        g = self.pool.fwd(h, B, N, 1024)
        for i, (fc, C) in enumerate(((net.fc1, 512), (net.fc2, 256)), 3):
            z = self.lin[i].fwd(g, g.shape[1], B, fc.weight, fc.bias, tf32_ok=False)
            g = _fwd_norm_act(self.na[i], z, C, B, C, self._bn(i + 1), R)
        t = self.lin[5].fwd(g, 256, B, net.fc3.weight, net.fc3.bias, tf32_ok=False)               # [B, k*k]
        eye = torch.eye(k, device=t.device, dtype=torch.float32).reshape(1, k * k)
        ops.axpy(t, k * k, eye.expand(B, -1).contiguous(), k * k, B, k * k, 1.0)                    # + identity
        return t.view(B, k, k)

    def bwd(self, dtrans, grads, need_drows):
        B, M, k = self.B, self.M, self.net.k
        d = dtrans.reshape(B, k * k).contiguous()
        d = self.lin[5].bwd(d, k * k, grads)
        for i in (4, 3):
            C = (512, 256)[i - 3]
            d = self.na[i].bwd(d, C, grads)
            d = self.lin[i].bwd(d, C, grads)
        d = self.pool.bwd(d)                                                                        # [M, 1024]
        for i in (2, 1, 0):
            C = (64, 128, 1024)[i]
            d = self.na[i].bwd(d, C, grads)
            d = self.lin[i].bwd(d, C, grads, need_da=(i > 0 or need_drows))
        return d


def _act_of(module):
    return (ops.ACT_RELU, 0.0) if isinstance(module.act_f, nn.ReLU) else (ops.ACT_LEAKY, module.negative_slope)


# ----------------------------------------------------------------------------------------------------------------------
# LPDNet (reference lpdnet_model.py:147-268), train mode
# ----------------------------------------------------------------------------------------------------------------------
class LPDNetTrain:
    def __init__(self, net):
        self.net = net

    # conv1 / conv2 (+BN+act) with the optional T-Nets around them (reference :226-241); strict fp32: they feed the kNN
    def _front_fwd(self, rows, D, B, N, conv1, bn1, conv2, bn2, act, slope):
        net, M = self.net, B * N
        self.t3, self.tf = None, None
        if net.t3d:
            self.t3, self.x3 = TNetTrain(net.t_net3d), Transform()
            rows = self.x3.fwd(rows, D, self.t3.fwd(rows, D, B, N), B, N, 3, keep_tail=True)
        self.l1, self.b1, self.l2, self.b2 = Linear(), BNAct(), Linear(), BNAct()
        z1 = self.l1.fwd(rows, D, M, conv1.weight, tf32_ok=False)
        h1 = self.b1.fwd(z1, 64, M, 64, bn1, act, slope)
        z2 = self.l2.fwd(h1, 64, M, conv2.weight, tf32_ok=False)
        h2 = self.b2.fwd(z2, 64, M, 64, bn2, act, slope)
        if net.tfea:
            self.tf, self.xf = TNetTrain(net.t_net_fea), Transform()
            h2 = self.xf.fwd(h2, 64, self.tf.fwd(h2, 64, B, N), B, N, 64)
        return h2

    def _front_bwd(self, dh2, grads):
        if self.tf is not None:
            da, dtf = self.xf.bwd(dh2, need_drows=True)
            db = self.tf.bwd(dtf, grads, need_drows=True)
            ops.axpy(da, 64, db, 64, self.M, 64, 1.0)
            dh2 = da
        dz2 = self.b2.bwd(dh2, 64, grads)
        dh1 = self.l2.bwd(dz2, 64, grads)
        dz1 = self.b1.bwd(dh1, 64, grads)
        if self.t3 is None:
            self.l1.bwd(dz1, 64, grads, need_da=False)
            return
        drows = self.l1.bwd(dz1, 64, grads)                                        # [M, D]: gradient of the transformed xyz (+ the mFea columns)
        _, dt3 = self.x3.bwd(drows, need_drows=False, lddout=drows.shape[1])
        self.t3.bwd(dt3, grads, need_drows=False)

    def fwd(self, x):
        net = self.net
        self.f16 = ops.get_train_precision() == "f16"
        if self.f16 and ops.get_precision() == "fp32":
            raise LpdError('set_train_precision("f16") needs precision "tf32" or "f16": "fp32" stays strict fp32')
        require_cuda(x, "LPDNet")
        B, _, N, D = x.shape
        M, k = B * N, net.k
        self.B, self.N, self.M, self.k = B, N, M, k
        act, slope = _act_of(net)
        self.act, self.slope = act, slope
        dev = x.device
        rows = x.detach().reshape(M, D).contiguous()
        if D != 3 and not (D == 8 and net.use_mFea):
            raise ValueError(f"LPDNet: expected 3 input dims (or 8 with use_mFea: xyz + 5 features), got {D}")
        if ops.SPATIAL_ORDER and N >= 64 and D == 3:
            # grid-cell order per cloud: every stage below is per-point equivariant, NetVLAD and the BatchNorm statistics
            # sum over the points, and no input gradient is needed, so the parameter gradients are unchanged
            rows = ops.cell_order(rows.view(B, N, 3))[2].view(M, 3)
        xyz = rows.view(B, N, D)[:, :, :3].contiguous() if D != 3 else rows.view(B, N, 3)   # kNN uses the untransformed xyz (:216,:255)
        h2 = self._front_fwd(rows, D, B, N, net.conv1_lpd, net.bn1_lpd, net.conv2_lpd, net.bn2_lpd, act, slope)
        self.h2 = h2
        # ---- feature-space graph: DG1 (decomposed) -> x1, DG2 (dense edge GEMM) -> x2 --------------------------------
        self.idx_f = ops.knn(h2.view(B, N, 64), k)
        wdg1 = w2d(net.convDG1[0].weight)                                         # [128, 128] = [Wn | Wc]
        self.wpq1 = torch.cat((wdg1[:, :64], wdg1[:, 64:]), 0).contiguous()       # [256, 64]
        self.pq1 = ops.linear(h2, self.wpq1, M=M, N=256, K=64)
        p1, q1 = self.pq1, self.pq1[:, 128:]
        bn_dg1, bn_dg2, bn_sn1 = net.convDG1[1], net.convDG2[1], net.convSN1[1]
        self.zsel1, self.arg1, part, nparts = ops.edge_sel_stats(p1, 256, q1, 256, self.idx_f, B, N, k, 128, bn_dg1.weight.detach())
        self.bn1e = _bn_finalize(bn_dg1, part, nparts, M * k, 128)
        self.pyr = torch.empty(M, 512, device=dev, dtype=torch.float32)
        pyr = self.pyr
        ops.affine_act(self.zsel1, M, 128, 128, self.bn1e[0], self.bn1e[1], act, slope, out=pyr, ldo=512)
        self.wdg2 = w2d(net.convDG2[0].weight)
        if self.f16:
            # DG2 edge tensors in fp16 (ops.set_train_precision): y1 rounded to nearest, z2e = y1 . W2^T with fp32 accumulation
            self.y1 = ops.edge_materialize_f16(p1, 256, q1, 256, self.idx_f, B, N, k, 128, self.bn1e[0], self.bn1e[1], act, slope)
            self.wdg2_h = ops.to_f16(self.wdg2)
            self.z2e = ops.gemm_f16(self.y1, self.wdg2_h, M=M * k, N=128, K=128, out_half=True)
            part, nparts, self.z2e_minmax = ops.bn_stats_f16(self.z2e, M * k, 128, 128)
            self.bn2e = _bn_finalize(bn_dg2, part, nparts, M * k, 128)
            self.zsel2, self.arg2 = ops.edge_sel_dense_f16(self.z2e, M, k, 128, bn_dg2.weight.detach())
        else:
            self.y1 = ops.edge_materialize(p1, 256, q1, 256, self.idx_f, B, N, k, 128, self.bn1e[0], self.bn1e[1], act, slope)
            self.z2e = ops.linear(self.y1, self.wdg2, M=M * k, N=128, K=128)
            part, nparts = ops.bn_stats(self.z2e, M * k, 128, 128)
            self.bn2e = _bn_finalize(bn_dg2, part, nparts, M * k, 128)
            self.zsel2, self.arg2 = ops.edge_sel_dense(self.z2e, M, k, 128, bn_dg2.weight.detach())
        ops.affine_act(self.zsel2, M, 128, 128, self.bn2e[0], self.bn2e[1], act, slope, out=pyr[:, 128:], ldo=512)
        # ---- Cartesian graph on the input coordinates: SN1 (decomposed) over x2 -> x3 ---------------------------------
        self.idx_x = ops.knn(xyz, k)
        wsn1 = w2d(net.convSN1[0].weight)                                         # [256, 256]
        self.wpq3 = torch.cat((wsn1[:, :128], wsn1[:, 128:]), 0).contiguous()     # [512, 128]
        self.pq3 = ops.linear(pyr[:, 128:], self.wpq3, M=M, N=512, K=128, lda=512)
        p3, q3 = self.pq3, self.pq3[:, 256:]
        self.zsel3, self.arg3, part, nparts = ops.edge_sel_stats(p3, 512, q3, 512, self.idx_x, B, N, k, 256, bn_sn1.weight.detach())
        self.bn3e = _bn_finalize(bn_sn1, part, nparts, M * k, 256)
        ops.affine_act(self.zsel3, M, 256, 256, self.bn3e[0], self.bn3e[1], act, slope, out=pyr[:, 256:], ldo=512)
        # ---- conv3 512 -> emb ---------------------------------------------------------------------------------------------
        self.l3, self.b3 = Linear(), BNAct()
        z3 = self.l3.fwd(pyr, 512, M, net.conv3_lpd.weight)
        f = self.b3.fwd(z3, net.emb_dims, M, net.emb_dims, net.bn3_lpd, act, slope)
        return f, B, N

    def bwd(self, df, grads: _Grads):
        """df [M, emb] (consumed in place)"""
        net, B, N, M, k = self.net, self.B, self.N, self.M, self.k
        act, slope = self.act, self.slope
        dev = df.device
        dz3 = self.b3.bwd(df, net.emb_dims, grads)
        dpyr = self.l3.bwd(dz3, net.emb_dims, grads)                               # [M, 512]
        del dz3, df
        # ---- SN1: arg-routed gradient only -------------------------------------------------------------------------------
        bn_dg1, bn_dg2, bn_sn1 = net.convDG1[1], net.convDG2[1], net.convSN1[1]
        dx3 = dpyr[:, 256:]
        S3 = ops.bn_bwd_sums(dx3, 512, self.zsel3, 256, M, 256, self.bn3e, act, slope)
        dpq3 = torch.empty(M, 512, device=dev, dtype=torch.float32)
        ops.edge_bwd(self.pq3, 512, self.pq3[:, 256:], 512, self.idx_x, B, N, k, 256, self.bn3e, act, slope, dx3, 512, self.arg3,
                     None, dpq3, 512, dpq3[:, 256:], 512, S=S3)
        grads.add(bn_sn1.bias, S3[0])
        grads.add(bn_sn1.weight, S3[1])
        dwpq3 = ops.wgrad(dpq3, 512, self.pyr[:, 128:], 512, M, 512, 128)          # [512, 128]
        grads.add(net.convSN1[0].weight, torch.cat((dwpq3[:256], dwpq3[256:]), 1))
        dx2 = dpyr[:, 128:]
        dgrad(dpq3, 512, self.wpq3, M, 512, 128, out=dx2, ldc=512, accumulate=True)
        del dpq3
        # ---- DG2: dense edge layer whose only consumer is the max ----------------------------------------------------
        S2 = ops.bn_bwd_sums(dx2, 512, self.zsel2, 128, M, 128, self.bn2e, act, slope)
        grads.add(bn_dg2.bias, S2[0])
        grads.add(bn_dg2.weight, S2[1])
        dpq1 = torch.empty(M, 256, device=dev, dtype=torch.float32)
        if self.f16:
            # fp16 gradients stored as 2^E * value: scale = [2^E; 2^-E], E from the bound of include/lpd_b200.h
            gs = ops.edge_grad_scale_f16(dx2, 512, M, 128, self.bn2e, S2, M * k, act, slope, self.z2e_minmax, self.wdg2_h)
            dz2e = ops.edge_dense_bwd_apply_f16(self.z2e, M, k, 128, self.bn2e, S2, M * k, act, slope, dx2, 512, self.zsel2, self.arg2, gs[0])
            grads.add(net.convDG2[0].weight, ops.wgrad_f16(dz2e, 128, self.y1, 128, M * k, 128, 128, gs[1]))
            w2t_h = ops.to_f16(ops.transpose(self.wdg2.unsqueeze(0))[0])
            dy1 = ops.gemm_f16(dz2e, w2t_h, M=M * k, N=128, K=128, out=self.y1, ldc=128)      # 2^E * dy1, over the dead y1
            # ---- DG1: dense gradient from DG2 + arg-routed gradient of x1 -------------------------------------------
            S1 = ops.edge_bwd_f16(self.pq1, 256, self.pq1[:, 128:], 256, self.idx_f, B, N, k, 128, self.bn1e, act, slope, dpyr, 512,
                                  self.arg1, dy1, gs[1], dpq1, 256, dpq1[:, 128:], 256)
        else:
            dz2e = ops.edge_dense_bwd_apply(self.z2e, M, k, 128, self.bn2e, S2, M * k, act, slope, dx2, 512, self.zsel2, self.arg2)
            grads.add(net.convDG2[0].weight, ops.wgrad(dz2e, 128, self.y1, 128, M * k, 128, 128))
            dy1 = dgrad(dz2e, 128, self.wdg2, M * k, 128, 128, out=self.y1, ldc=128)   # y1 is dead after the wgrad: reuse it
            # ---- DG1: dense gradient from DG2 + arg-routed gradient of x1 -------------------------------------------
            S1 = ops.edge_bwd(self.pq1, 256, self.pq1[:, 128:], 256, self.idx_f, B, N, k, 128, self.bn1e, act, slope, dpyr, 512,
                              self.arg1, dy1, dpq1, 256, dpq1[:, 128:], 256)
        grads.add(bn_dg1.bias, S1[0])
        grads.add(bn_dg1.weight, S1[1])
        dwpq1 = ops.wgrad(dpq1, 256, self.h2, 64, M, 256, 64)                      # [256, 64]
        grads.add(net.convDG1[0].weight, torch.cat((dwpq1[:128], dwpq1[128:]), 1))
        dh2 = dgrad(dpq1, 256, self.wpq1, M, 256, 64)
        del dpq1, dy1, dpyr
        self._front_bwd(dh2, grads)


# ----------------------------------------------------------------------------------------------------------------------
# LPDNetOrign (reference lpdnet_model.py:18-114, the CLI default featnet), train mode
# ----------------------------------------------------------------------------------------------------------------------
class LPDNetOrignTrain(LPDNetTrain):
    def fwd(self, x):
        net = self.net
        require_cuda(x, "LPDNetOrign")
        B, _, N, D = x.shape
        M, k = B * N, net.k
        self.B, self.N, self.M, self.k = B, N, M, k
        act, slope = _act_of(net)
        self.act, self.slope = act, slope
        rows = x.detach().reshape(M, D).contiguous()
        if D != 3 and not (D == 8 and net.use_mFea):
            raise ValueError(f"LPDNetOrign: expected 3 input dims (or 8 with use_mFea), got {D}")
        if ops.SPATIAL_ORDER and N >= 64 and D == 3:
            rows = ops.cell_order(rows.view(B, N, 3))[2].view(M, 3)
        xyz = rows.view(B, N, D)[:, :, :3].contiguous() if D != 3 else rows.view(B, N, 3)
        h2 = self._front_fwd(rows, D, B, N, net.conv1_lpd[0], net.conv1_lpd[1], net.conv2_lpd[0], net.conv2_lpd[1], act, slope)
        self.h2 = h2
        # ---- feature-space graph: edges [f_i ; f_j - f_i] -> DG1 (decomposed: P = Wb f_j, Q = (Wa - Wb) f_i), DG2 (dense), max ----
        self.idx_f = ops.knn(h2.view(B, N, 64), k)
        wdg1 = w2d(net.convDG1[0].weight)                                          # [64, 128] = [Wa | Wb]
        wa, wb = wdg1[:, :64], wdg1[:, 64:]
        self.wpq1 = torch.cat((wb, wa - wb), 0).contiguous()                       # [128, 64]
        self.pq1 = ops.linear(h2, self.wpq1, M=M, N=128, K=64)
        p1, q1 = self.pq1, self.pq1[:, 64:]
        bn_dg1, bn_dg2 = net.convDG1[1], net.convDG2[1]
        _, _, part, nparts = ops.edge_sel_stats(p1, 128, q1, 128, self.idx_f, B, N, k, 64, bn_dg1.weight.detach())
        self.bn1e = _bn_finalize(bn_dg1, part, nparts, M * k, 64)
        self.y1 = ops.edge_materialize(p1, 128, q1, 128, self.idx_f, B, N, k, 64, self.bn1e[0], self.bn1e[1], act, slope)
        self.wdg2 = w2d(net.convDG2[0].weight)
        self.z2e = ops.linear(self.y1, self.wdg2, M=M * k, N=64, K=64)
        part, nparts = ops.bn_stats(self.z2e, M * k, 64, 64)
        self.bn2e = _bn_finalize(bn_dg2, part, nparts, M * k, 64)
        self.zsel2, self.arg2 = ops.edge_sel_dense(self.z2e, M, k, 64, bn_dg2.weight.detach())
        self.xdg = ops.affine_act(self.zsel2, M, 64, 64, self.bn2e[0], self.bn2e[1], act, slope)
        # ---- Cartesian graph, gather-only edges e = f_j: SN1, SN2 over the materialised edges (BatchNorm2d statistics are
        #      over all B*N*k edges, i.e. weighted by the in-degree of every point), max ----
        self.idx_x = ops.knn(xyz, k)
        one, zero = torch.ones(64, device=x.device), torch.zeros(64, device=x.device)
        self.e3 = ops.edge_materialize(self.xdg, 64, None, 0, self.idx_x, B, N, k, 64, one, zero, ops.ACT_NONE, 0.0)
        self.ls1, self.bs1, self.ls2 = Linear(), BNAct(), Linear()
        zs1 = self.ls1.fwd(self.e3, 64, M * k, net.convSN1[0].weight)
        ys1 = self.bs1.fwd(zs1, 64, M * k, 64, net.convSN1[1], act, slope)
        self.zs2 = self.ls2.fwd(ys1, 64, M * k, net.convSN2[0].weight)
        part, nparts = ops.bn_stats(self.zs2, M * k, 64, 64)
        self.bns2 = _bn_finalize(net.convSN2[1], part, nparts, M * k, 64)
        self.zsel4, self.arg4 = ops.edge_sel_dense(self.zs2, M, k, 64, net.convSN2[1].weight.detach())
        xsn = ops.affine_act(self.zsel4, M, 64, 64, self.bns2[0], self.bns2[1], act, slope)
        # ---- conv3/4/5: 64 -> 64 -> 128 -> emb ----
        self.tail = []
        f, ldf = xsn, 64
        for seq, C in ((net.conv3_lpd, 64), (net.conv4_lpd, 128), (net.conv5_lpd, net.emb_dims)):
            lin, bna = Linear(), BNAct()
            z = lin.fwd(f, ldf, M, seq[0].weight)
            f = bna.fwd(z, C, M, C, seq[1], act, slope)
            ldf = C
            self.tail.append((lin, bna, C))
        return f, B, N

    def bwd(self, df, grads: _Grads):
        net, B, N, M, k = self.net, self.B, self.N, self.M, self.k
        act, slope = self.act, self.slope
        d = df
        for lin, bna, C in reversed(self.tail):
            d = bna.bwd(d, C, grads)
            d = lin.bwd(d, C, grads)
        dxsn = d                                                                   # [M, 64]
        # SN2: dense edge layer whose only consumer is the max
        bn_sn2 = net.convSN2[1]
        S = ops.bn_bwd_sums(dxsn, 64, self.zsel4, 64, M, 64, self.bns2, act, slope)
        dzs2 = ops.edge_dense_bwd_apply(self.zs2, M, k, 64, self.bns2, S, M * k, act, slope, dxsn, 64, self.zsel4, self.arg4)
        grads.add(bn_sn2.bias, S[0])
        grads.add(bn_sn2.weight, S[1])
        dys1 = self.ls2.bwd(dzs2, 64, grads)
        dzs1 = self.bs1.bwd(dys1, 64, grads)
        de3 = self.ls1.bwd(dzs1, 64, grads)                                        # [M*k, 64]
        dxdg = ops.edge_scatter_add(de3, self.idx_x, B, N, k, 64)                  # [M, 64]
        del de3, dzs1, dys1, dzs2
        # DG2
        bn_dg1, bn_dg2 = net.convDG1[1], net.convDG2[1]
        S2 = ops.bn_bwd_sums(dxdg, 64, self.zsel2, 64, M, 64, self.bn2e, act, slope)
        dz2e = ops.edge_dense_bwd_apply(self.z2e, M, k, 64, self.bn2e, S2, M * k, act, slope, dxdg, 64, self.zsel2, self.arg2)
        grads.add(bn_dg2.bias, S2[0])
        grads.add(bn_dg2.weight, S2[1])
        grads.add(net.convDG2[0].weight, ops.wgrad(dz2e, 64, self.y1, 64, M * k, 64, 64))
        dy1 = dgrad(dz2e, 64, self.wdg2, M * k, 64, 64, out=self.y1, ldc=64)
        # DG1 (decomposed, dense incoming gradient only)
        dpq1 = torch.empty(M, 128, device=df.device, dtype=torch.float32)
        S1 = ops.edge_bwd(self.pq1, 128, self.pq1[:, 64:], 128, self.idx_f, B, N, k, 64, self.bn1e, act, slope, None, 0, None,
                          dy1, dpq1, 128, dpq1[:, 64:], 128)
        grads.add(bn_dg1.bias, S1[0])
        grads.add(bn_dg1.weight, S1[1])
        dwpq1 = ops.wgrad(dpq1, 128, self.h2, 64, M, 128, 64)                      # [128, 64] = [dW_P ; dW_Q]
        dwp, dwq = dwpq1[:64], dwpq1[64:]
        dwb = dwp.clone()
        ops.axpy(dwb, 64, dwq.contiguous(), 64, 64, 64, -1.0)                      # Wb enters P (+) and Q = Wa - Wb (-)
        grads.add(net.convDG1[0].weight, torch.cat((dwq, dwb), 1))
        dh2 = dgrad(dpq1, 128, self.wpq1, M, 128, 64)
        self._front_bwd(dh2, grads)


# ----------------------------------------------------------------------------------------------------------------------
# PointNetfeat (reference PointNetVlad.py:181-241), train mode
# ----------------------------------------------------------------------------------------------------------------------
class PointNetTrain:
    def __init__(self, net):
        self.net = net

    def fwd(self, x):
        net = self.net
        require_cuda(x, "PointNetfeat")
        B, _, N, _ = x.shape
        M, R = B * N, ops.ACT_RELU
        self.B, self.N, self.M = B, N, M
        if N != net.num_points:
            raise ValueError(f"PointNetfeat: got {N} points, constructed for num_points={net.num_points}")
        rows = x.detach().reshape(M, 3).contiguous()
        self.stn, self.x3 = TNetTrain(net.stn), Transform()
        xt = self.x3.fwd(rows, 3, self.stn.fwd(rows, 3, B, N), B, N, 3)                              # :205-209
        self.lins = [Linear() for _ in range(5)]
        self.bnas = [BNAct() for _ in range(5)]
        h, ldh = xt, 3
        self.ft = None
        for i, C in enumerate((64, 64, 64, 128, net.emb_dims)):
            conv, bn = getattr(net, f"conv{i + 1}"), getattr(net, f"bn{i + 1}")
            if i == 2 and net.apply_feature_trans:                                                   # :218-225
                self.ft, self.xf = TNetTrain(net.feature_trans), Transform()
                h = self.xf.fwd(h, 64, self.ft.fwd(h, 64, B, N), B, N, 64)
            z = self.lins[i].fwd(h, ldh, M, conv.weight, conv.bias, tf32_ok=(i >= 2))
            h = self.bnas[i].fwd(z, C, M, C, bn, R if i < 4 else ops.ACT_NONE)                       # :213-230 (no ReLU after bn5)
            ldh = C
        return h, B, N

    def bwd(self, df, grads: _Grads):
        d = df
        chans = (64, 64, 64, 128, self.net.emb_dims)
        for i in (4, 3, 2, 1, 0):
            d = self.bnas[i].bwd(d, chans[i], grads)
            d = self.lins[i].bwd(d, chans[i], grads)
            if i == 2 and self.ft is not None:
                da, dft = self.xf.bwd(d, need_drows=True)
                db = self.ft.bwd(dft, grads, need_drows=True)
                ops.axpy(da, 64, db, 64, self.M, 64, 1.0)
                d = da
        _, dt3 = self.x3.bwd(d, need_drows=False)                                                    # d: gradient of x . T  [M, 3]
        self.stn.bwd(dt3, grads, need_drows=False)


# ----------------------------------------------------------------------------------------------------------------------
# NetVLADLoupe + GatingContext (reference PointNetVlad.py:12-115), train mode
# ----------------------------------------------------------------------------------------------------------------------
class NetVLADTrain:
    def __init__(self, nv):
        if nv.cluster_size != 64:
            raise NotImplementedError("the NetVLAD kernels are specialised for cluster_size == 64 (the reference's value)")
        if not nv.add_batch_norm:
            raise LpdError("train mode without add_batch_norm is not built yet")
        self.nv = nv

    def fwd(self, f, B):
        nv = self.nv
        N, D, K, O = nv.max_samples, nv.feature_size, nv.cluster_size, nv.output_dim
        M = B * N
        self.f, self.B, self.M = f, B, M
        wc = nv.cluster_weights.detach()
        # soft assignment: a = softmax(BN(f . Wc))                                            :48-59
        if ops.get_precision() != "fp32" and M >= 128 and D % 4 == 0:
            self.apre = ops.gemm_tf32(f, ops.transpose(wc.unsqueeze(0))[0], M=M, N=K, K=D)
        else:
            self.apre = ops.gemm(f, wc, a_layout=A_MK, b_layout=B_KN, M=M, N=K, K=D, lda=D, ldb=K)
        self.bn_a = BNAct()
        a = self.bn_a.fwd(self.apre, K, M, K, nv.bn1)
        self.a = ops.softmax64(a, M)
        if ops._tn_ok(f, self.a, D, K, N, D, K, B):
            vraw = ops.gemm_tf32_tn(f, self.a, M=D, N=K, K=N, lda=D, ldb=K, batch=B)          # :64-66 -> [B, D, K]
        else:
            vraw = ops.gemm(f, self.a, a_layout=A_KM, b_layout=B_KN, M=D, N=K, K=N, lda=D, ldb=K, batch=B,
                            strideA=N * D, strideB=N * K)
        vraw = vraw.view(B, D, K)
        self.v, self.asum, self.n1, self.n2 = ops.netvlad_finish_train(vraw, self.a, nv.cluster_weights2.detach()[0].contiguous(),
                                                                       B, N, D, K)            # :61-74
        KD = D * K
        splits = nv.HIDDEN_SPLITS
        while KD % splits:
            splits //= 2
        kc = KD // splits
        wh = nv.hidden1_weights.detach()
        part = torch.empty(splits, B, O, device=f.device, dtype=torch.float32)
        ops.gemm(self.v, wh, a_layout=A_MK, b_layout=B_KN, M=B, N=O, K=kc, lda=KD, ldb=O, out=part, ldc=O,
                 batch=splits, strideA=kc, strideB=kc * O, strideC=B * O)                     # :76
        hpre = ops.splitk_reduce(part, splits, B, O)
        self.bn_h = BNAct()
        h = self.bn_h.fwd(hpre, O, B, O, nv.bn2)                                              # :78
        self.h = h
        if not nv.gating:
            return h
        cg = nv.context_gating
        self.g = ops.gemm(h, cg.gating_weights.detach(), a_layout=A_MK, b_layout=B_KN, M=B, N=O, K=O)   # :104
        self.bn_g = BNAct()
        return self.bn_g.fwd(self.g, O, B, O, cg.bn1, ops.ACT_GATE, 0.0, aux=h, ldaux=O)        # :106-113

    def bwd(self, dout, grads: _Grads):
        """dout [B, O] -> df [M, D]"""
        nv = self.nv
        N, D, K, O = nv.max_samples, nv.feature_size, nv.cluster_size, nv.output_dim
        B, M = self.B, self.M
        dout = dout.contiguous()
        if nv.gating:
            cg = nv.context_gating
            wg = cg.gating_weights.detach()
            # out = h * sigmoid(BN(g)):  dh (direct) = dout * sigmoid(.) ; dg through the BN
            dh = ops.affine_act(self.g, B, O, O, self.bn_g.bn[0], self.bn_g.bn[1], ops.ACT_GATE, 0.0, aux=dout, ldaux=O)
            dg = self.bn_g.bwd(dout, O, grads, inplace=False)
            grads.add(cg.gating_weights, ops.gemm(self.h, dg, a_layout=A_KM, b_layout=B_KN, M=O, N=O, K=B, lda=O, ldb=O))
            ops.gemm(dg, wg, a_layout=A_MK, b_layout=B_NK, M=B, N=O, K=O, lda=O, ldb=O, out=dh, ldc=O, act=ops.ACT_ADD, aux=dh)
        else:
            dh = dout.clone()
        dhpre = self.bn_h.bwd(dh, O, grads)
        wh = nv.hidden1_weights.detach()
        KD = D * K
        # the 64 MiB hidden-projection gradient is 95 % of all gradient bytes and the FIRST one to be complete: final -> its
        # NCCL all-reduce overlaps the whole rest of the backward (optim.Adam.grad_ready)
        grads.add(nv.hidden1_weights, ops.gemm(self.v, dhpre, a_layout=A_KM, b_layout=B_KN, M=KD, N=O, K=B, lda=KD, ldb=O), final=True)
        dv = ops.gemm(dhpre, wh, a_layout=A_MK, b_layout=B_NK, M=B, N=KD, K=O, lda=O, ldb=O)   # [B, D*K]
        wc2 = nv.cluster_weights2.detach()[0].contiguous()
        dvraw, dasum, dwc2 = ops.netvlad_finish_bwd(dv, self.v, wc2, self.asum, self.n1, self.n2, B, D, K)
        grads.add(nv.cluster_weights2, dwc2)
        f, a = self.f, self.a
        # vraw[b] = f[b]^T a[b]:  da[b] = f[b] . dvraw[b] ;  df[b] = a[b] . dvraw[b]^T (accumulated below)
        tc_ok = ops.get_precision() != "fp32" and N >= 128 and D % 4 == 0
        if tc_ok:
            dvraw_t = ops.transpose(dvraw.view(B, D, K))                            # [B, K, D]: K-contiguous weight slices
            da = ops.gemm_tf32(f, dvraw_t, M=N, N=K, K=D, lda=D, batch=B,
                               out=torch.empty(M, K, device=f.device, dtype=torch.float32), ldc=K)
        else:
            da = ops.gemm(f, dvraw, a_layout=A_MK, b_layout=B_KN, M=N, N=K, K=D, lda=D, ldb=K, batch=B,
                          strideA=N * D, strideB=D * K, strideC=N * K,
                          out=torch.empty(M, K, device=f.device, dtype=torch.float32), ldc=K)
        ds = ops.softmax64_bwd(da, a, dasum, M, N)
        dapre = self.bn_a.bwd(ds, K, grads)
        wc = nv.cluster_weights.detach()
        grads.add(nv.cluster_weights, ops.wgrad(f, D, dapre, K, M, D, K))           # dWc[d][k] = sum_m f[m][d] dapre[m][k]
        # df = dapre . Wc^T  (z = f . Wc  <=>  weight [N=K][K=D] = Wc^T, i.e. "w" of dgrad is Wc^T [K, D])
        df = torch.empty(M, D, device=f.device, dtype=torch.float32)
        if ops.get_precision() != "fp32" and M >= 128:
            ops.gemm_tf32(dapre, wc, M=M, N=D, K=K, lda=K, out=df, ldc=D)           # Wc [D][K] is already K-contiguous
        else:
            ops.gemm(dapre, wc, a_layout=A_MK, b_layout=B_NK, M=M, N=D, K=K, lda=K, ldb=K, out=df, ldc=D)
        if tc_ok:
            ops.gemm_tf32(a, dvraw, M=N, N=D, K=K, lda=K, batch=B, out=df, ldc=D, accumulate=True)
        else:
            ops.gemm(a, dvraw, a_layout=A_MK, b_layout=B_NK, M=N, N=D, K=K, lda=K, ldb=K, batch=B,
                     strideA=N * K, strideB=D * K, strideC=N * D, out=df, ldc=D, act=ops.ACT_ADD, aux=df)
        return df


# ----------------------------------------------------------------------------------------------------------------------
# whole model
# ----------------------------------------------------------------------------------------------------------------------
class _PointNetVladTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, model, *params):
        from .util.lpdnet_model import LPDNet, LPDNetOrign
        feat = model.emb_nn
        with torch.no_grad():
            if isinstance(feat, LPDNet):
                fe = LPDNetTrain(feat)
            elif isinstance(feat, LPDNetOrign):
                fe = LPDNetOrignTrain(feat)
            else:
                if model.point_net.max_pool:
                    raise ValueError("PointNetVlad needs the per-point feature map: construct with max_pool=False")
                fe = PointNetTrain(model.point_net)
            f, B, N = fe.fwd(x)
            if N != model.net_vlad.max_samples:
                raise ValueError(f"PointNetVlad: got {N} points per cloud, constructed for num_points={model.net_vlad.max_samples}")
            nv = NetVLADTrain(model.net_vlad)
            out = nv.fwd(f, B)
        ctx.fe, ctx.nv, ctx.params = fe, nv, params
        return out

    @staticmethod
    def backward(ctx, dout):
        grads = _Grads()
        with torch.no_grad():
            df = ctx.nv.bwd(dout, grads)
            ctx.fe.bwd(df, grads)
        out = [grads.by_param.get(p) for p in ctx.params]
        ctx.fe = ctx.nv = None
        return (None, None, *out)


def forward_train(model, x: torch.Tensor) -> torch.Tensor:
    """train-mode PointNetVlad.forward (reference PointNetVlad.py:261-270 under model.train())"""
    require_cuda(x, "PointNetVlad")
    params = [p for p in model.parameters() if p.requires_grad]
    if not torch.is_grad_enabled() or not params:
        with torch.no_grad():
            return _PointNetVladTrainFn.forward(_NullCtx(), x, model, *params)
    return _PointNetVladTrainFn.apply(x, model, *params)


class _NullCtx:
    pass

"""Drop-in modules for the reference's 1-D graph convolutions (torch_src/models/mmargcn/graph_convolution.py; SURVEY 8 f2).

``AGCNGraphConvolution`` (:56-113) is the adaptive graph convolution of the AGCN unit WITHOUT the time axis -- Conv1d 1x1
projections, per-sample ``softmax(theta^T phi / Ci)`` attention, ``X (A + B + P)`` aggregation, BatchNorm1d, ``down`` residual,
ReLU -- on graphs of up to T * signals = 652 nodes (``ImuGCN``, torch_src/models/mmargcn/imu_feature_models.py:63-102;
``GCN``, gcn.py:18-83).  It runs on the same kernels as ``SpatialGraphConv`` with t = 1: the V x V stages switch to batched FFMA
GEMMs over the node axis for V > 32 (csrc/joint_big.cu).  ``STGCNGraphConvolution`` (:12-53) is ``relu(dropout(conv(x) adj^T) +
residual(x))`` with one fixed adjacency for the whole batch (``agcn_node_mix``).

Same constructors, forward signatures ((N, C, V) in, (N, C_out, V) out), parameter / buffer names and initial distributions
as the reference classes; ``nn.Conv1d`` / ``nn.BatchNorm1d`` objects are parameter containers only.
"""
import numpy as np
import torch
import torch.nn as nn

from . import functional as FN
from . import ops as K_default  # noqa: F401  (functional.K is the switchable backend; imported here for the type checker)
from . import modules as M
from .modules import _bn_buffers, bn_init, conv_branch_init, conv_init


def _to_cl(x):       # (N, C, V) -> (N, 1, V, C)
    return M._prep(x.permute(0, 2, 1)).unsqueeze(1)


def _from_cl(y):     # (N, 1, V, C) -> contiguous (N, C, V)
    return y.squeeze(1).permute(0, 2, 1).contiguous()


class AGCNGraphConvolution(nn.Module):
    """relu(BN(sum_k conv_d[k](x . (adj_a[k] + adj_b[k] + softmax(theta_k^T phi_k / Ci)))) + down(x))  (graph_convolution.py:56-113)."""

    def __init__(self, in_features, out_features, adj, **kwargs):
        super().__init__()
        coff_embedding = kwargs.get("coff_embedding", 4)
        num_subset = kwargs.get("num_subset", 3)
        adj = np.asarray(adj)
        if num_subset != 3 or adj.shape[0] != 3:
            raise ValueError("fusion_gcn_b200 implements the 3-subset spatial partition (K = 3) only")
        inter_channels = out_features // coff_embedding
        self.inter_c = inter_channels
        self.in_features, self.out_features = in_features, out_features
        self.adj_b = nn.Parameter(torch.from_numpy(adj.astype(np.float32)))
        nn.init.constant_(self.adj_b, 1e-6)
        self.register_buffer("adj_a", torch.from_numpy(adj.astype(np.float32)))
        self.num_subset = num_subset
        self.adj_c = [None] * num_subset
        self.conv_a, self.conv_b, self.conv_d = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        for _ in range(num_subset):
            self.conv_a.append(nn.Conv1d(in_features, inter_channels, 1))
            self.conv_b.append(nn.Conv1d(in_features, inter_channels, 1))
            self.conv_d.append(nn.Conv1d(in_features, out_features, 1))
        if in_features != out_features:
            self.down = nn.Sequential(nn.Conv1d(in_features, out_features, 1), nn.BatchNorm1d(out_features))
        else:
            self.down = lambda x: x
        self.bn = nn.BatchNorm1d(out_features)
        for m in self.modules():
            if isinstance(m, nn.Conv1d):
                conv_init(m)
            elif isinstance(m, nn.BatchNorm1d):
                bn_init(m, 1)
        bn_init(self.bn, 1e-6)
        for i in range(num_subset):
            conv_branch_init(self.conv_d[i], num_subset)
        self._agcn_precision = M._default_precision

    @property
    def has_down(self):
        return isinstance(self.down, nn.Sequential)

    def _params(self):
        p = [self.adj_a, self.adj_b]
        for k in range(3):
            p += [self.conv_a[k].weight, self.conv_a[k].bias, self.conv_b[k].weight, self.conv_b[k].bias,
                  self.conv_d[k].weight, self.conv_d[k].bias]
        p += [self.bn.weight, self.bn.bias]
        p += [self.down[0].weight, self.down[0].bias, self.down[1].weight, self.down[1].bias] if self.has_down else [None] * 4
        return p

    def forward(self, x):
        spec = FN.UnitSpec(cin=self.in_features, cout=self.out_features, training=self.training, precision=self._agcn_precision,
                           has_down=self.has_down, bn_gcn=_bn_buffers(self.bn),
                           bn_down=_bn_buffers(self.down[1]) if self.has_down else None, attention_out=self.adj_c)
        return _from_cl(FN.GcnFn.apply(_to_cl(x), spec, *self._params()))


class _NodeMixFn(torch.autograd.Function):
    """y[b, v, :] = sum_u adj[v, u] x[b, u, :]  (support . adj^T in the reference's (N, C, V) layout, graph_convolution.py:45)."""

    @staticmethod
    def forward(ctx, x, adj):
        ctx.save_for_backward(adj)
        return FN.K.node_mix(x, adj)

    @staticmethod
    def backward(ctx, dy):
        adj, = ctx.saved_tensors
        return FN.K.node_mix(dy.contiguous(), adj, transpose=True), None


class _RowBnFn(torch.autograd.Function):
    """BatchNorm1d over the channels of a [rows, C] tensor (statistics over rows), training or eval."""

    @staticmethod
    def forward(ctx, x, gamma, beta, buf: FN.BnBuffers, training: bool):
        sc, sh, mean, invstd = FN.K.bn_stats(x, gamma, beta, buf.running_mean, buf.running_var, buf.num_batches_tracked,
                                             FN.BN_MOMENTUM, FN.BN_EPS, training)
        ctx.save_for_backward(x, gamma, mean, invstd)
        ctx.training = training
        return FN.K.bn_apply(x, sc, sh)[0]

    @staticmethod
    def backward(ctx, dy):
        x, gamma, mean, invstd = ctx.saved_tensors
        dx, dgamma, dbeta, _ = FN.K.bn_bwd(dy.contiguous(), None, x, mean, invstd, gamma, frozen=not ctx.training)
        return dx, dgamma, dbeta, None, None


class _AddReluFn(torch.autograd.Function):
    """relu(y + r) (graph_convolution.py:50-52) through the BN-apply kernel with unit scale; r may be None."""

    @staticmethod
    def forward(ctx, y, r):
        c = y.shape[-1]
        one, zero = torch.ones(c, device=y.device, dtype=y.dtype), torch.zeros(c, device=y.device, dtype=y.dtype)
        out = FN.K.bn_apply(y, one, zero, res_mode=FN.K.RES_NONE if r is None else FN.K.RES_TENSOR, res=r, relu=True)[0]
        ctx.save_for_backward(out)
        ctx.has_r = r is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        out, = ctx.saved_tensors
        c = out.shape[-1]
        zero, one = torch.zeros(c, device=out.device, dtype=out.dtype), torch.ones(c, device=out.device, dtype=out.dtype)
        g = torch.empty_like(out)
        FN.K.bn_bwd(dout.contiguous(), out, out, zero, one, None, want_dy=False, dres=g)      # g = dout * [out > 0]
        return g, (g if ctx.has_r else None)


class STGCNGraphConvolution(nn.Module):
    """relu(dropout(conv(x) adj^T) + residual(x))  (graph_convolution.py:12-53).  ``sparse=True`` adjacencies are densified: the
    graphs have at most a few hundred nodes and the reference's per-sample ``torch.sparse.mm`` loop is its own "very slow" path."""

    def __init__(self, in_features: int, out_features: int, adj: torch.Tensor, bias: bool = True, residual: bool = True, **kwargs):
        super().__init__()
        dropout = kwargs.get("dropout", 0.)
        self.sparse = kwargs.get("sparse", False)
        self.conv = nn.Conv1d(in_features, out_features, 1, bias=bias)
        adj = adj.to_dense() if adj.is_sparse else adj
        self.register_buffer("adj", adj.to(torch.float32).contiguous())
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(dropout) if dropout > 0 else None
        if not residual:
            self.residual = lambda x: 0
            self._residual_kind = "none"
        elif in_features == out_features:
            self.residual = lambda x: x
            self._residual_kind = "identity"
        else:
            self.residual = nn.Sequential(nn.Conv1d(in_features, out_features, 1), nn.BatchNorm1d(out_features))
            self._residual_kind = "conv"
        self._agcn_precision = M._default_precision

    def forward(self, x):
        n, c, v = x.shape
        xc = M._prep(x.permute(0, 2, 1))                                               # (N, V, C)
        rows = xc.view(n * v, c)
        cout = self.conv.out_channels
        support = FN.LinearFn.apply(rows, self.conv.weight.view(cout, c), self.conv.bias, self._agcn_precision)
        y = _NodeMixFn.apply(support.view(n, v, cout), self.adj)
        if self.dropout is not None:
            y = self.dropout(y)
        if self._residual_kind == "identity":
            r = xc
        elif self._residual_kind == "conv":
            conv, bn = self.residual[0], self.residual[1]
            r = FN.LinearFn.apply(rows, conv.weight.view(cout, c), conv.bias, self._agcn_precision)
            r = _RowBnFn.apply(r, bn.weight, bn.bias, _bn_buffers(bn), self.training).view(n, v, cout)
        else:
            r = None
        out = _AddReluFn.apply(y.contiguous(), r)
        return out.permute(0, 2, 1).contiguous()

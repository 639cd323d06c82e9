"""Drop-in modules for the MMARGCN variant of the AGCN unit (reference: torch_src/models/mmargcn/agcn.py).

Same constructors, forward signatures, attribute names, parameter / buffer names (state-dict keys),
initial distributions and ``adj_c`` side output as the reference classes ``TemporalConv`` (:37),
``SpatialGraphConv`` (:54), ``SpatialTemporalConv`` (:118) and ``Model`` (:139) -- but the arithmetic
runs in the sm_100a kernels of libagcn_b200.so.  ``nn.Conv2d`` / ``nn.BatchNorm2d`` objects are used
only as parameter containers (so checkpoints, optimizers and ``named_parameters`` filters of the
reference's session code keep working); their ``forward`` is never called.

Layout: the standalone modules take and return the reference's (N', C, T, V) tensors; inside ``Model``
the units exchange channels-last (N', T, V, C) tensors through ``forward_cl`` so that no transposes remain
(the model input (N, M, T, V, C) already is channels-last).
"""
import math
from typing import Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as FN
from .capi import PREC_BF16X3, PREC_FP32, PREC_FP32_FFMA, PREC_TF32
from .graph import adjacency_from_graph

_PRECISIONS = {"fp32": PREC_FP32, "tf32": PREC_TF32, "fp32_ffma": PREC_FP32_FFMA, "bf16x3": PREC_BF16X3,
               PREC_FP32: PREC_FP32, PREC_TF32: PREC_TF32, PREC_FP32_FFMA: PREC_FP32_FFMA, PREC_BF16X3: PREC_BF16X3}


_default_precision = PREC_FP32


def set_default_precision(precision) -> None:
    """Precision mode given to modules constructed from now on (used by the drop-in launcher, where the reference's own
    session code builds the model)."""
    global _default_precision
    _default_precision = _PRECISIONS[precision]


def set_precision(module: nn.Module, precision) -> nn.Module:
    """'fp32' (parity mode: 3xTF32 tensor cores + FFMA), 'tf32' (single-pass tensor cores) or 'fp32_ffma' (FFMA only)
    for every unit under ``module``."""
    code = _PRECISIONS[precision]
    for m in module.modules():
        if hasattr(m, "_agcn_precision"):
            m._agcn_precision = code
    return module


_default_recompute = False


def set_default_recompute(flag: bool) -> None:
    """Activation-recompute policy given to units constructed from now on (see ``set_recompute``)."""
    global _default_recompute
    _default_recompute = bool(flag)


def set_recompute(module: nn.Module, flag: bool = True) -> nn.Module:
    """Recompute policy of every unit under ``module``: with ``flag`` the theta / phi embeddings and the aggregated tensor
    (1.5 + 3 of the ~8.5 activation planes a unit saves) are not kept for the backward but produced again there by the same two
    kernels -- same bits, ~45 % less activation memory, two more launches per unit in the backward."""
    for m in module.modules():
        if hasattr(m, "_agcn_recompute"):
            m._agcn_recompute = bool(flag)
    return module


def set_sync_batchnorm(module: nn.Module, sync=True) -> nn.Module:
    """Synchronised BatchNorm for every unit (and the model's data_bn) under ``module``: training-mode statistics and their backward
    sums are taken over all ranks of a process group, so a batch sharded over R GPUs normalises exactly like the unsharded batch
    (the reference is single-process: its nn.BatchNorm sees the whole batch, agcn.py:44,78,83,150).  ``sync``: True (default group),
    a ``distributed.SyncBatchNorm``, or None / False to go back to per-replica statistics.  The ranks' local batch sizes may differ
    (``distributed.split_batch``; multiply a mean-reduced loss by its ``loss_weight`` before ``backward()``)."""
    if sync is True:
        from .distributed import SyncBatchNorm
        sync = SyncBatchNorm()
    elif sync is False:
        sync = None
    for m in module.modules():
        if hasattr(m, "_agcn_sync"):
            m._agcn_sync = sync
    return module


def conv_branch_init(conv, branches):            # agcn.py:18-24
    weight = conv.weight
    n, k1, k2 = weight.size(0), weight.size(1), weight.size(2)
    nn.init.normal_(weight, 0, math.sqrt(2. / (n * k1 * k2 * branches)))
    nn.init.constant_(conv.bias, 0)


def conv_init(conv):                             # agcn.py:27-29
    nn.init.kaiming_normal_(conv.weight, mode="fan_out")
    nn.init.constant_(conv.bias, 0)


def bn_init(bn, scale):                          # agcn.py:32-34
    nn.init.constant_(bn.weight, scale)
    nn.init.constant_(bn.bias, 0)


def _bn_buffers(bn: nn.BatchNorm2d) -> FN.BnBuffers:
    return FN.BnBuffers(bn.running_mean, bn.running_var, bn.num_batches_tracked)


def _prep(x: torch.Tensor) -> torch.Tensor:
    # device / dtype are enforced by fusion_gcn_b200.ops (CUDA fp32 only, no CPU path)
    return x.float().contiguous()


def _to_cl(x):       # (N', C, T, V) -> (N', T, V, C)
    return _prep(x.permute(0, 2, 3, 1))


def _from_cl(y):     # (N', T, V, C) -> contiguous (N', C, T, V), as the reference returns
    return y.permute(0, 3, 1, 2).contiguous()


class TemporalConv(nn.Module):
    """BN(Conv2d(C_in, C_out, (k,1), pad ((k-1)/2, 0), stride (s,1))) -- no activation (agcn.py:37-51)."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int = 9, stride: int = 1):
        super().__init__()
        pad = int((kernel_size - 1) / 2)
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=(kernel_size, 1), padding=(pad, 0), stride=(stride, 1))
        self.bn = nn.BatchNorm2d(out_channels)
        conv_init(self.conv)
        bn_init(self.bn, 1)
        self._agcn_precision = _default_precision
        self._agcn_sync = None

    def _params(self):
        return (self.conv.weight, self.conv.bias, self.bn.weight, self.bn.bias)

    def forward_cl(self, x):
        spec = FN.UnitSpec(cin=self.conv.in_channels, cout=self.conv.out_channels, stride=self.conv.stride[0], residual="none",
                           kernel_size=self.conv.kernel_size[0], relu_out=False, training=self.training,
                           precision=self._agcn_precision, bn_tcn=_bn_buffers(self.bn), sync=self._agcn_sync)
        return FN.TcnFn.apply(x, None, spec, *self._params(), None, None, None, None)

    def forward(self, x):
        return _from_cl(self.forward_cl(_to_cl(x)))


class SpatialGraphConv(nn.Module):
    """relu(BN(sum_k conv_d[k](x . (adj_a[k] + adj_b[k] + softmax(theta_k^T phi_k)))) + down(x)) (agcn.py:54-115)."""

    def __init__(self, in_channels: int, out_channels: int, adj: np.ndarray, coff_embedding: int = 4, num_subsets: int = 3):
        super().__init__()
        if num_subsets != 3 or adj.shape[0] != 3:
            raise ValueError("fusion_gcn_b200 implements the 3-subset spatial partition (K = 3) only")
        inter_channels = out_channels // coff_embedding
        self.inter_channels = inter_channels
        self.num_subsets = num_subsets
        self.in_channels, self.out_channels = in_channels, out_channels

        self.adj_b = nn.Parameter(torch.from_numpy(adj.astype(np.float32)))
        nn.init.constant_(self.adj_b, 1e-6)
        self.register_buffer("adj_a", torch.from_numpy(adj.astype(np.float32)))
        self.adj_c = [None] * self.num_subsets

        self.conv_a = nn.ModuleList()
        self.conv_b = nn.ModuleList()
        self.conv_d = nn.ModuleList()
        for _ in range(self.num_subsets):
            self.conv_a.append(nn.Conv2d(in_channels, inter_channels, 1))
            self.conv_b.append(nn.Conv2d(in_channels, inter_channels, 1))
            self.conv_d.append(nn.Conv2d(in_channels, out_channels, 1))

        if in_channels != out_channels:
            self.down = nn.Sequential(nn.Conv2d(in_channels, out_channels, 1), nn.BatchNorm2d(out_channels))
        else:
            self.down = lambda x: x

        self.bn = nn.BatchNorm2d(out_channels)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                conv_init(m)
            elif isinstance(m, nn.BatchNorm2d):
                bn_init(m, 1)
        bn_init(self.bn, 1e-6)
        for i in range(self.num_subsets):
            conv_branch_init(self.conv_d[i], self.num_subsets)
        self._agcn_precision = _default_precision
        self._agcn_recompute = _default_recompute
        self._agcn_sync = None

    # hooks for the original-variant subclass (parameter called PA, adjacency not a buffer)
    def _adj_fixed(self, x):
        return self.adj_a

    def _adj_learned(self):
        return self.adj_b

    @property
    def has_down(self):
        return isinstance(self.down, nn.Sequential)

    def _params(self, x):
        p = [self._adj_fixed(x), self._adj_learned()]
        for k in range(3):
            p += [self.conv_a[k].weight, self.conv_a[k].bias, self.conv_b[k].weight, self.conv_b[k].bias,
                  self.conv_d[k].weight, self.conv_d[k].bias]
        p += [self.bn.weight, self.bn.bias]
        if self.has_down:
            p += [self.down[0].weight, self.down[0].bias, self.down[1].weight, self.down[1].bias]
        else:
            p += [None, None, None, None]
        return p

    def _fill_spec(self, spec: FN.UnitSpec):
        spec.has_down = self.has_down
        spec.bn_gcn = _bn_buffers(self.bn)
        spec.bn_down = _bn_buffers(self.down[1]) if self.has_down else None
        spec.attention_out = self.adj_c          # list of 3 (N', V, V) tensors refreshed every forward, detached (SURVEY D10)
        return spec

    def forward_cl(self, x):
        spec = self._fill_spec(FN.UnitSpec(cin=self.in_channels, cout=self.out_channels, training=self.training,
                                           precision=self._agcn_precision, recompute=self._agcn_recompute, sync=self._agcn_sync))
        params = self._params(x)
        spec.cin = _pad_input_weights(params, self.in_channels, x.shape[-1])
        return FN.GcnFn.apply(x, spec, *params)

    def forward(self, x):
        return _from_cl(self.forward_cl(_to_cl(x)))


def _pad_input_weights(params, in_channels: int, actual: int) -> int:
    """Channel-padded input (Model pads wide odd channel counts such as the 515-channel skeleton + RGB fusion to a multiple of 32 so
    that the first unit runs on the TMA / tcgen05 kernels): the gcn weights that read x (conv_a / conv_b / conv_d / down) get matching
    zero columns, in place in ``params``.  F.pad is differentiable, so their gradients come back in the parameters' own shapes."""
    cpad = actual - in_channels
    if cpad < 0:
        raise RuntimeError(f"input has {actual} channels, the unit expects {in_channels}")
    if cpad > 0:
        for i, prm in enumerate(params[:FN.GCN_NPARAMS]):
            if prm is not None and prm.dim() == 4 and prm.shape[1] == in_channels:
                params[i] = F.pad(prm, (0, 0, 0, 0, 0, cpad))
    return actual



def _padded_channels(c: int) -> int:
    """Channel count the first unit actually runs on: wide counts that are not a multiple of 32 (C = 515: skeleton + 512-d RGB patch
    embeddings, early_fusion_models.py:53-60) are zero-padded up so that every contraction of the unit takes the tensor-core path."""
    return (c + 31) // 32 * 32 if (c > 64 and c % 32) else c


class SpatialTemporalConv(nn.Module):
    """relu(tcn1(gcn1(x)) + residual(x)) (agcn.py:118-136)."""

    _gcn_cls = SpatialGraphConv
    _tcn_cls = TemporalConv

    def __init__(self, in_channels, out_channels, adj, stride=1, residual=True):
        super().__init__()
        self.gcn1 = self._gcn_cls(in_channels, out_channels, adj)
        self.tcn1 = self._tcn_cls(out_channels, out_channels, stride=stride)
        self.out_channels = out_channels
        self.stride = stride
        if not residual:
            self.residual = lambda x: 0
            self._residual_kind = "none"
        elif (in_channels == out_channels) and (stride == 1):
            self.residual = lambda x: x
            self._residual_kind = "identity"
        else:
            self.residual = self._tcn_cls(in_channels, out_channels, kernel_size=1, stride=stride)
            self._residual_kind = "conv"
        self._agcn_precision = _default_precision
        self._agcn_recompute = _default_recompute
        self._agcn_sync = None

    def forward_cl(self, x, pool_groups: int = 0):
        """``pool_groups`` > 0: return the mean over the (T, V) positions and bodies of every sample, [pool_groups, C_out], instead
        of the feature map (the model's tail, agcn.py:194-196, fused into this unit's last pass)."""
        g, t = self.gcn1, self.tcn1
        spec = FN.UnitSpec(cin=g.in_channels, cout=self.out_channels, stride=self.stride, residual=self._residual_kind,
                           kernel_size=t.conv.kernel_size[0], relu_out=True, training=self.training,
                           precision=self._agcn_precision, bn_tcn=_bn_buffers(t.bn), pool_groups=pool_groups,
                           recompute=self._agcn_recompute, sync=self._agcn_sync)
        g._fill_spec(spec)
        params = g._params(x) + list(t._params())
        spec.cin = _pad_input_weights(params, g.in_channels, x.shape[-1])
        if self._residual_kind == "conv":
            spec.bn_res = _bn_buffers(self.residual.bn)
            params += list(self.residual._params())
        else:
            params += [None, None, None, None]
        return FN.UnitFn.apply(x, spec, *params)

    def forward(self, x):
        return _from_cl(self.forward_cl(_to_cl(x)))


class Model(nn.Module):
    """AGCN backbone: data_bn -> up to 10 units -> mean over (T, V) and bodies -> fc (agcn.py:139-200).

    ``forward(x)`` takes the reference's live layout x: (N, M, T, V, C) (SURVEY D1).
    """

    _unit_cls = SpatialTemporalConv

    def __init__(self, data_shape: tuple, num_classes: int, graph, num_layers: int = 10, start_feature_size: int = 64,
                 without_fc=False, dropout: float = 0., adjacency_matrix: Optional[np.ndarray] = None):
        super().__init__()
        num_persons, _, num_joints, num_channels = data_shape
        adj = adjacency_matrix if adjacency_matrix is not None else adjacency_from_graph(graph)
        if adj.shape[-1] != num_joints:
            raise ValueError(f"graph has {adj.shape[-1]} vertices but data_shape has {num_joints} joints")
        self.data_bn = nn.BatchNorm1d(num_persons * num_channels * num_joints)
        s = start_feature_size
        U = self._unit_cls
        self.layers = [
            U(num_channels, s, adj, residual=False), U(s, s, adj), U(s, s, adj), U(s, s, adj),
            U(s, s * 2, adj, stride=2), U(s * 2, s * 2, adj), U(s * 2, s * 2, adj),
            U(s * 2, s * 4, adj, stride=2), U(s * 4, s * 4, adj), U(s * 4, s * 4, adj)]
        self.layers = self.layers[:min(len(self.layers), num_layers)]
        if dropout > 0:      # dropout modules take their own l<idx> names, exactly like the reference (agcn.py:166-172)
            for i in range(1, len(self.layers) * 2 - 1, 2):
                self.layers.insert(i, nn.Dropout(dropout, inplace=True))
        self._register_layers()
        last = [m for m in self.layers if not isinstance(m, nn.Dropout)][-1].out_channels
        if without_fc:
            self.fc = None
            self.out_channels = last
        else:
            self.fc = nn.Linear(last, num_classes)
            nn.init.normal_(self.fc.weight, 0, math.sqrt(2. / num_classes))
            self.out_channels = num_classes
        bn_init(self.data_bn, 1)
        self._agcn_precision = _default_precision
        self._agcn_sync = None

    def _register_layers(self):
        for layer_idx, layer in enumerate(self.layers):
            setattr(self, f"l{layer_idx}", layer)

    def features_cl(self, x):
        """(N, M, T, V, C) -> channels-last feature map (N*M, T', V, C_out) of the last unit."""
        x = _prep(x)
        buf = FN.BnBuffers(self.data_bn.running_mean, self.data_bn.running_var, self.data_bn.num_batches_tracked)
        h = FN.DataBnFn.apply(x, self.data_bn.weight, self.data_bn.bias, buf, self.training, self._agcn_sync)
        cp = _padded_channels(h.shape[-1])
        if cp != h.shape[-1] and self.layers and self.layers[0]._residual_kind == "none":
            h = F.pad(h, (0, cp - h.shape[-1]))
        for layer in self.layers:
            h = layer(h) if isinstance(layer, nn.Dropout) else layer.forward_cl(h)
        return h

    def pooled_features(self, x):
        """(N, M, T, V, C) -> (N, C_out): features_cl followed by the mean over (T, V) and bodies, with the pool fused into the last
        unit's normalise / residual / ReLU pass (the last feature map is never written)."""
        n = x.shape[0]
        x = _prep(x)
        buf = FN.BnBuffers(self.data_bn.running_mean, self.data_bn.running_var, self.data_bn.num_batches_tracked)
        h = FN.DataBnFn.apply(x, self.data_bn.weight, self.data_bn.bias, buf, self.training, self._agcn_sync)
        cp = _padded_channels(h.shape[-1])
        if cp != h.shape[-1] and self.layers and self.layers[0]._residual_kind == "none":
            h = F.pad(h, (0, cp - h.shape[-1]))
        for i, layer in enumerate(self.layers):
            if isinstance(layer, nn.Dropout):
                h = layer(h)
            elif i == len(self.layers) - 1:
                h = layer.forward_cl(h, pool_groups=n)
            else:
                h = layer.forward_cl(h)
        return h if h.dim() == 2 else FN.PoolFn.apply(h, n)       # (layouts the fused tail does not cover pool separately)

    def loss(self, x, labels):
        """(loss, logits) of nn.CrossEntropyLoss()(self(x), labels) with the classifier and the loss fused into one kernel
        (the reference computes them separately, procedures/step.py:41-42).  Mean reduction, no class weights / smoothing."""
        if self.fc is None:
            raise RuntimeError("Model(without_fc=True) has no classifier to fuse the loss with")
        feat = self.pooled_features(x)
        return FN.LinearCrossEntropyFn.apply(feat, self.fc.weight, self.fc.bias, labels)

    def forward(self, x):
        x = self.pooled_features(x)
        if self.fc is not None:
            x = FN.LinearFn.apply(x, self.fc.weight, self.fc.bias, self._agcn_precision)
        return x

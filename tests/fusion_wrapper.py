"""A two-modality fusion model built from package modules only, for the CUDA-graph step tests and tools/bench_graph_step.py.

It takes the dict batches the reference's ``MultiModalDataset`` yields when a config loads two modalities (torch_src/dataset.py:42-49):
``{"skeleton": (N, M, T, V, C), "inertial": (N, C_i, V_i)}``.  The skeleton branch is the AGCN backbone without its classifier on
the UTD-MHAD graph; the inertial branch is an adaptive graph convolution on a 40-node IMU graph (more than 32 nodes: the large-graph
kernels, ``agcn_joint_mix_big`` / ``agcn_node_mix``, run inside the capture) followed by an ST-GCN graph convolution with a conv
residual; an ``nn.Linear`` head reads both feature vectors, as the reference's late-fusion wrappers do.  The model has no ``loss``
method, so the graphed step takes ``loss_fn(model(x), y)``."""
import numpy as np
import torch
import torch.nn as nn

from fusion_gcn_b200 import graph as G, graphconv as GC, modules as M

IMU_STEPS, IMU_SIGNALS = 10, 4          # V_i = 40 nodes


def imu_adjacency(steps=IMU_STEPS, signals=IMU_SIGNALS):
    """The IMU graph of imu_feature_models.py:11-61 restated: nodes = (time step, signal), all signals of a step connected both
    ways, every node pointing to the same signal one step later.  Returns (3-subset partition for the adaptive convolution,
    row-normalised undirected adjacency with self loops for the ST-GCN convolution)."""
    v = steps * signals
    edges = []
    for i in range(0, v, signals):
        edges += [(i + j, i + k) for j in range(signals) for k in range(signals) if j != k]
        if i >= signals:
            edges += [(i - signals + k, i + k) for k in range(signals)]
    a = np.zeros((v, v))
    e = np.asarray(edges)
    a[e[:, 0], e[:, 1]] = 1.0
    a = np.maximum(a, a.T) + np.eye(v)
    return G.partition_adjacency(edges, v), torch.from_numpy(a / a.sum(axis=1, keepdims=True)).float()


class SkeletonInertialNet(nn.Module):
    def __init__(self, skeleton_shape=(1, 40, 20, 3), inertial_channels=6, num_classes=27, start_feature_size=16, num_layers=10):
        super().__init__()
        self.skeleton = M.Model(skeleton_shape, num_classes, G.SkeletonGraph(G.UTD_EDGES, center_joint=G.UTD_CENTER),
                                num_layers=num_layers, start_feature_size=start_feature_size, without_fc=True)
        adj3, adj1 = imu_adjacency()
        self.inertial_agcn = GC.AGCNGraphConvolution(inertial_channels, 32, adj3)
        self.inertial_stgcn = GC.STGCNGraphConvolution(32, 64, adj1)          # 32 -> 64: conv + BatchNorm residual
        self.head = nn.Linear(self.skeleton.out_channels + 64, num_classes)

    def forward(self, x):
        a = self.skeleton(x["skeleton"])
        b = self.inertial_stgcn(self.inertial_agcn(x["inertial"])).mean(dim=2)
        return self.head(torch.cat([a, b], dim=1))


def batch(n, skeleton_shape=(1, 40, 20, 3), inertial_channels=6, num_classes=27, seed=0, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    x = {"skeleton": torch.randn(n, *skeleton_shape, generator=g),
         "inertial": torch.randn(n, inertial_channels, IMU_STEPS * IMU_SIGNALS, generator=g)}
    y = torch.randint(num_classes, (n,), generator=g)
    return {k: v.to(device) for k, v in x.items()}, y.to(device)

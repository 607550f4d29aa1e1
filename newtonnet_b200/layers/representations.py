"""Edge embedding modules; mirror the module tree of newtonnet/layers/representations.py so state dicts
and pickled checkpoints map one to one (`embedding_layers.edge_embedding.embedding.frequencies`).

The arithmetic lives in the CUDA library: RadiusGraph -> csrc/nbr.cu (cell list, bit-identical edge set),
ScaledNorm / PolynomialCutoff / RadialBesselLayer -> csrc/pair_ops.cu (k_edge_geom_fwd / _bwd).
`EdgeEmbedding.forward` exposes that path for tests and users of the layer API.
"""
import ctypes as C

import torch
from torch import nn

__all__ = ['EdgeEmbedding', 'RadiusGraph', 'ScaledNorm', 'PolynomialCutoff', 'RadialBesselLayer']


class RadiusGraph(nn.Module):
    def __init__(self, r):
        super().__init__()
        self.r = r

    def forward(self, pos, cell=None, batch=None):
        """-> (edge_index [2,E] int64, disp [E,3]); same edges, order and fp32 values as
        representations.py:57-100."""
        from newtonnet_b200.engine import get_engine
        if batch is None:
            batch = torch.zeros(pos.shape[0], dtype=torch.long, device=pos.device)
        if cell is None:
            cell = torch.zeros(int(batch.max().item()) + 1 if batch.numel() else 1, 3, 3, device=pos.device)
        nl = get_engine(pos.device).checked_neighbor_list(pos, cell, batch, float(self.r))
        ei = nl.edge_index()
        ep = nl.edge_pair[:nl.n_edges].long()
        sign = torch.where(ep < 0, -1.0, 1.0).to(torch.float32).unsqueeze(1)
        disp = nl.pair_disp[(ep & 0x7fffffff)] * sign
        return ei, disp.to(pos.dtype)

    def __repr__(self):
        return f'{self.__class__.__name__}(r={self.r})'


class ScaledNorm(nn.Module):
    def __init__(self, r):
        super().__init__()
        self.r = r

    def __repr__(self):
        return f'{self.__class__.__name__}(r={self.r})'


class PolynomialCutoff(nn.Module):
    def __init__(self, p):
        super().__init__()
        self.p = p

    def __repr__(self):
        return f'{self.__class__.__name__}(p={self.p})'


class RadialBesselLayer(nn.Module):
    def __init__(self, n_basis):
        super().__init__()
        self.n_basis = n_basis
        # fp32(n * pi), non-trainable but part of the state dict (representations.py:220)
        self.frequencies = nn.Parameter(torch.arange(1, n_basis + 1) * torch.pi, requires_grad=False)
        self.epsilon = 1.0e-8

    def __repr__(self):
        return f'{self.__class__.__name__}(basis={self.n_basis})'


class EdgeEmbedding(nn.Module):
    def __init__(self, cutoff, n_basis=20):
        super().__init__()
        self.radius_graph = RadiusGraph(r=cutoff)
        self.norm = ScaledNorm(r=cutoff)
        self.envelope = PolynomialCutoff(p=9)
        self.embedding = RadialBesselLayer(n_basis=n_basis)

    def forward(self, pos, cell=None, batch=None):
        """-> (dist_edge [E,n_basis], dir_edge [E,3], edge_index [2,E]) as representations.py:20-43."""
        from newtonnet_b200 import _lib as L
        from newtonnet_b200.engine import stream
        edge_index, disp = self.radius_graph(pos, cell, batch)
        E = disp.shape[0]
        dev = pos.device
        d32 = disp.to(torch.float32).contiguous()
        rbf = torch.empty(E, L.NN_NB, dtype=torch.float32, device=dev)
        unit = torch.empty(E, 3, dtype=torch.float32, device=dev)
        dist = torch.empty(E, dtype=torch.float32, device=dev)
        freq = self.embedding.frequencies.detach().to(device=dev, dtype=torch.float32).contiguous()
        if E:
            L.check(L.load().nn_edge_geom_fwd(d32.data_ptr(), freq.data_ptr(), float(self.norm.r), None, E,
                                             rbf.data_ptr(), None, unit.data_ptr(), dist.data_ptr(), stream()),
                    'nn_edge_geom_fwd')
        return rbf.to(pos.dtype), unit.to(pos.dtype), edge_index

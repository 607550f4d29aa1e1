"""CPU oracle for the NewtonNet energy/force/stress path.  TEST INFRASTRUCTURE ONLY.

This file is a CPU restatement (PyTorch-on-CPU tensor ops, no CUDA, no custom kernels) of the
algorithm in the reference THGLab/NewtonNet v2.1.0.  Only `tests/`, `__graft_entry__.smoke()` and the
`cpu_baseline` / `--impl reference` legs of `bench.py` may import it; the product package
`newtonnet_b200` never does, and fails loudly when its CUDA library is missing.

Parity status: PINNED.  `tests/test_oracle.py` checks every function below against
  * the reference's own golden trajectory `scripts/md17_md/md.traj` + shipped checkpoint
    (tests/golden/md17_kat.npz, weights_md17.npz), and
  * outputs of the unmodified reference imported in the build container
    (tests/golden/case_*.npz, written by tests/golden/make_golden.py).

All file:line citations are relative to the reference repository root.

The state dict `sd` uses the reference's parameter names (SURVEY.md §8b):
  embedding_layers.node_embedding.weight [119,F]
  embedding_layers.edge_embedding.embedding.frequencies [nb]
  interaction_layers.{l}.message_nodepart.{0,2}.{weight,bias}
  interaction_layers.{l}.message_edgepart.weight [F,nb]
  interaction_layers.{l}.equiv_message{1,2}.{0,2}.weight
  interaction_layers.{l}.equiv_update.weight
  output_layers.0.layers.{0,2,4}.{weight,bias}
  scalers.0.{scale,shift}.weight [119,1]
"""
import math

import numpy as np
import torch

CUTOFF = 5.0
POLY_P = 9


def as_torch_sd(sd, dtype):
    """Cast a {name: ndarray|tensor} state dict to `dtype`.

    The Bessel frequencies are created as fp32(n*pi) (layers/representations.py:220) and keep that
    rounding when the model is cast to fp64 - casting the stored fp32 values up reproduces this.
    """
    return {k: torch.as_tensor(np.asarray(v)).to(dtype) for k, v in sd.items()}


def n_layers(sd):
    return 1 + max(int(k.split('.')[1]) for k in sd if k.startswith('interaction_layers.'))


# ----------------------------------------------------------------------------- R2 neighbour search
def radius_graph_dense(pos, cell, batch, cutoff=CUTOFF):
    """Dense minimum-image neighbour search; layers/representations.py:57-100.

    Ordered pairs (i, j) of the same system, i-major / j ascending (:74-77), i != j (:82);
    disp = pos[i]-pos[j] (:85); when any cell entry is non-zero (:86) the fractional shift
    n = round(solve(cell^T, disp)) (:92) is removed as cell @ n (:93) - NOT cell^T @ n, a reference
    quirk that is part of the behaviour to match; keep ||disp|| < cutoff, strict (:96-98).
    Returns edge_index [2,E] int64 (row 0 = destination i, row 1 = source j) and disp [E,3].
    """
    rows, cols = [], []
    for b in torch.unique(batch):
        members = torch.nonzero(batch == b).flatten()
        n = members.numel()
        rows.append(members.repeat_interleave(n))
        cols.append(members.repeat(n))
    i = torch.cat(rows) if rows else torch.zeros(0, dtype=torch.long)
    j = torch.cat(cols) if cols else torch.zeros(0, dtype=torch.long)
    keep = i != j
    i, j = i[keep], j[keep]
    disp = pos[i] - pos[j]
    if cell is not None and bool((cell != 0).any()):
        h = cell[batch][i]                                   # [E,3,3]
        frac = torch.linalg.solve(h.transpose(1, 2), disp)   # :92
        disp = disp - torch.bmm(h, torch.round(frac).unsqueeze(-1)).squeeze(-1)   # :93
    inside = disp.norm(dim=1) < cutoff
    return torch.stack([i[inside], j[inside]]), disp[inside]


def radius_graph_cell_list(pos, cell, batch, cutoff=CUTOFF):
    """O(N) restatement of `radius_graph_dense` for large boxes (numpy, fp32 arithmetic).

    Candidate pairs come from a cell list; each candidate is then tested with exactly the
    reference arithmetic (SURVEY.md §8a R2): per component d = fl(p_i - p_j), n = rint(d / L),
    d' = fl(d - fl(L*n)), keep sqrt(fma(dz,dz,fma(dy,dy,dx*dx))) < cutoff.  Diagonal cells or zero
    cells only (anything else goes through the dense path).  Validated against the dense path in
    tests/test_oracle.py; used where the dense path cannot run (C4, 100k atoms).
    Returns (edge_index [2,E] int64 sorted i-major / j-ascending, disp [E,3] float32).
    """
    pos = np.asarray(pos, dtype=np.float32)
    cell = np.asarray(cell, dtype=np.float32)
    batch = np.asarray(batch)
    periodic = bool((cell != 0).any())
    out_i, out_j, out_d = [], [], []
    for b in np.unique(batch):
        idx = np.nonzero(batch == b)[0]
        p = pos[idx]
        if periodic:
            h = cell[b]
            assert np.count_nonzero(h - np.diag(np.diag(h))) == 0, 'diagonal cells only'
            L = np.diag(h).astype(np.float32)
            frac = p.astype(np.float64) / L.astype(np.float64)
            frac -= np.floor(frac)
            nc = np.maximum(1, np.floor(L.astype(np.float64) / (cutoff * 1.0001)).astype(np.int64))
        else:
            L = None
            lo = p.min(0).astype(np.float64)
            ext = np.maximum(p.max(0).astype(np.float64) - lo, 1e-6)
            nc = np.maximum(1, np.floor(ext / (cutoff * 1.0001)).astype(np.int64))
            frac = (p.astype(np.float64) - lo) / ext
        ci = np.minimum((frac * nc).astype(np.int64), nc - 1)
        cid = (ci[:, 0] * nc[1] + ci[:, 1]) * nc[2] + ci[:, 2]
        order = np.argsort(cid, kind='stable')
        start = np.searchsorted(cid[order], np.arange(nc.prod() + 1))
        # neighbour cell offsets, de-duplicated per axis when fewer than 3 cells
        def axis_offsets(n):
            return [0] if n == 1 else ([0, 1] if n == 2 else [-1, 0, 1])
        offs = [(a, bb, c) for a in axis_offsets(nc[0]) for bb in axis_offsets(nc[1]) for c in axis_offsets(nc[2])]
        for (a, bb, c) in offs:
            nb = ci + np.array([a, bb, c])
            if periodic:
                nb %= nc
                ok = np.ones(len(p), dtype=bool)
            else:
                ok = ((nb >= 0) & (nb < nc)).all(1)
                nb = np.clip(nb, 0, nc - 1)
            ncid = (nb[:, 0] * nc[1] + nb[:, 1]) * nc[2] + nb[:, 2]
            cnt = np.where(ok, start[ncid + 1] - start[ncid], 0)
            ii = np.repeat(np.arange(len(p)), cnt)
            within = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
            jj = order[np.repeat(start[ncid], cnt) + within]
            m = ii != jj
            ii, jj = ii[m], jj[m]
            d = p[ii] - p[jj]
            if periodic:
                n = np.rint(d / L).astype(np.float32)
                d = d - (L * n).astype(np.float32)
            dd = d.astype(np.float64)   # fma chain == exact fp64 accumulate then one rounding per step
            r2 = np.float32(dd[:, 0] * dd[:, 0])
            r2 = (dd[:, 1] * dd[:, 1] + r2.astype(np.float64)).astype(np.float32)
            r2 = (dd[:, 2] * dd[:, 2] + r2.astype(np.float64)).astype(np.float32)
            keep = np.sqrt(r2) < np.float32(cutoff)
            out_i.append(idx[ii[keep]]); out_j.append(idx[jj[keep]]); out_d.append(d[keep])
    i = np.concatenate(out_i); j = np.concatenate(out_j); d = np.concatenate(out_d)
    key = i.astype(np.int64) * (len(pos) + 1) + j
    o = np.argsort(key, kind='stable')
    return np.stack([i[o], j[o]]).astype(np.int64), d[o]


# ----------------------------------------------------------------------------- R3-R6 edge features
def scaled_norm(disp, cutoff=CUTOFF):
    """layers/representations.py:129-131: d=|disp| (keepdim), dir=disp/d, x=d/cutoff."""
    d = torch.linalg.vector_norm(disp, dim=-1, keepdim=True)
    return d / cutoff, disp / d


def polynomial_cutoff(x, p=POLY_P):
    """layers/representations.py:166-169 (p=9 at :17): 1 - 55 x^9 + 99 x^10 - 45 x^11."""
    return (1.0 - 0.5 * (p + 1) * (p + 2) * x.pow(p) + p * (p + 2) * x.pow(p + 1)
            - 0.5 * p * (p + 1) * x.pow(p + 2))


def radial_bessel(x, frequencies):
    """layers/representations.py:233: sin(f_n x)/x, no normalisation."""
    return torch.sin(frequencies * x) / x


def edge_embedding(sd, pos, cell, batch, cutoff=CUTOFF):
    """layers/representations.py:20-43 -> (rbf [E,nb], dir [E,3], edge_index [2,E])."""
    edge_index, disp = radius_graph_dense(pos, cell, batch, cutoff)
    x, direction = scaled_norm(disp, cutoff)
    freq = sd['embedding_layers.edge_embedding.embedding.frequencies']
    return polynomial_cutoff(x) * radial_bessel(x, freq), direction, edge_index


# ----------------------------------------------------------------------------- R7 interaction layer
def silu(x):
    return x * torch.sigmoid(x)


def _segment_sum(src, index, n):
    """torch_geometric.utils.scatter(reduce='sum') == new_zeros(size).scatter_add_(0, index, src)."""
    out = src.new_zeros((n,) + tuple(src.shape[1:]))
    view = index.view((-1,) + (1,) * (src.dim() - 1)).expand_as(src)
    return out.scatter_add_(0, view, src)


def interaction(sd, l, a, f, direction, rbf, edge_index):
    """models/newtonnet.py:207-237 (layer_norm=False)."""
    k = f'interaction_layers.{l}.'
    i, j = edge_index[0], edge_index[1]
    n = a.shape[0]
    hidden = silu(a @ sd[k + 'message_nodepart.0.weight'].T + sd[k + 'message_nodepart.0.bias'])
    mn = hidden @ sd[k + 'message_nodepart.2.weight'].T + sd[k + 'message_nodepart.2.bias']   # :209
    me = rbf @ sd[k + 'message_edgepart.weight'].T                                            # :210
    m = me * mn[i] * mn[j]                                                                    # :211
    a = a + _segment_sum(m, i, n)                                                             # :213-215
    e1 = silu(m @ sd[k + 'equiv_message1.0.weight'].T) @ sd[k + 'equiv_message1.2.weight'].T  # :218
    e2 = silu(m @ sd[k + 'equiv_message2.0.weight'].T) @ sd[k + 'equiv_message2.2.weight'].T  # :222
    vec = e1.unsqueeze(1) * direction.unsqueeze(2) + e2.unsqueeze(1) * f[j]                   # :219-224
    f = f + _segment_sum(vec, i, n)                                                           # :226-227
    a = a + (f * (f @ sd[k + 'equiv_update.weight'].T)).sum(dim=1)                            # :230-231
    if (k + 'layer_norm.weight') in sd:                                                       # :234-235, nn.LayerNorm(F)
        a = torch.nn.functional.layer_norm(a, (a.shape[1],), sd[k + 'layer_norm.weight'], sd[k + 'layer_norm.bias'], 1e-5)
    return a, f


# ----------------------------------------------------------------------------- R8/R9 energy head
def atomic_energy(sd, a, z, head=0):
    """models/output.py:98-100 then layers/scalers.py:55-58."""
    k = f'output_layers.{head}.layers.'
    h = silu(a @ sd[k + '0.weight'].T + sd[k + '0.bias'])
    h = silu(h @ sd[k + '2.weight'].T + sd[k + '2.bias'])
    o = h @ sd[k + '4.weight'].T + sd[k + '4.bias']
    return o * sd[f'scalers.{head}.scale.weight'][z] + sd[f'scalers.{head}.shift.weight'][z]


def direct_force(sd, a, f, z, head):
    """DirectForceOutput (models/output.py:115-132) + ScaleShift(scale only) (layers/scalers.py:11,55-56):
    F_i[c] = scale[z_i] * sum_f MLP(a_i)[f] * f_i[c][f]."""
    k = f'output_layers.{head}.layers.'
    h = silu(a @ sd[k + '0.weight'].T + sd[k + '0.bias'])
    h = silu(h @ sd[k + '2.weight'].T + sd[k + '2.bias'])
    h = h @ sd[k + '4.weight'].T + sd[k + '4.bias']
    return (h.unsqueeze(1) * f).sum(-1) * sd[f'scalers.{head}.scale.weight'][z]


# ----------------------------------------------------------------------------- R0/R1/R10 full path
def forward(sd, z, pos, cell, batch, dtype=torch.float64, stress=False, return_layers=False,
            cutoff=CUTOFF, direct_force_head=None):
    """NewtonNet.forward, models/newtonnet.py:74-104, heads energy + gradient_force (+ stress/virial).

    Follows the reference's strain trick (models/newtonnet.py:146-155): D = I, S = (D + D^T)/2,
    pos' = pos @ S[batch], cell' = cell @ S; forces/virial come from one autograd.grad of the summed
    energies w.r.t. (pos, D) (models/output.py:66-73); force = -dE/dpos (:112), virial = -dE/dD
    (:164), stress = dE/dD / det(cell) (:176-179).
    Returns a dict of numpy arrays.
    """
    sd = as_torch_sd(sd, dtype)
    z = torch.as_tensor(np.asarray(z)).long()
    batch = torch.as_tensor(np.asarray(batch)).long()
    pos = torch.as_tensor(np.asarray(pos)).to(dtype).clone().requires_grad_(True)
    cell = torch.as_tensor(np.asarray(cell)).to(dtype)
    n_sys = cell.shape[0]
    D = torch.eye(3, dtype=dtype).repeat(n_sys, 1, 1).requires_grad_(True)
    S = 0.5 * (D + D.transpose(-1, -2))
    pos_s = torch.bmm(pos.unsqueeze(1), S[batch]).squeeze(1)
    cell_s = torch.bmm(cell, S)
    rbf, direction, edge_index = edge_embedding(sd, pos_s, cell_s, batch, cutoff)
    a = sd['embedding_layers.node_embedding.weight'][z]            # :142 (row 0 = padding)
    f = torch.zeros(z.shape[0], 3, a.shape[1], dtype=dtype)        # :143
    layers = []
    for l in range(n_layers(sd)):
        a, f = interaction(sd, l, a, f, direction, rbf, edge_index)
        if return_layers:
            layers.append((a.detach().numpy().copy(), f.detach().numpy().copy()))
    e_atom = atomic_energy(sd, a, z)
    energy = _segment_sum(e_atom, batch, n_sys).reshape(-1)        # models/output.py:246
    g_pos, g_D = torch.autograd.grad(energy, (pos, D), torch.ones_like(energy))
    out = {'energy': energy.detach().numpy(), 'forces': (-g_pos).numpy(),
           'edge_index': edge_index.numpy(), 'atom_node': a.detach().numpy(),
           'force_node': f.detach().numpy()}
    if stress:
        out['virial'] = (-g_D).numpy()
        out['stress'] = (g_D / torch.linalg.det(cell).view(-1, 1, 1)).numpy()
    if return_layers:
        out['layers'] = layers
    if direct_force_head is not None:
        out['direct_force'] = direct_force(sd, a, f, z, direct_force_head).detach().numpy()
    return out


# ----------------------------------------------------------------------------- row B: analytic backward
def silu_grad(x):
    s = torch.sigmoid(x)
    return s * (1.0 + x * (1.0 - s))


def forward_analytic(sd, z, pos, cell, batch, dtype=torch.float64, cutoff=CUTOFF, edge_index=None,
                     disp=None):
    """Hand-derived reverse sweep (SURVEY.md §8a row B) in the pair-symmetric staged form the CUDA
    path uses; no autograd.  It is checked against `forward` (autograd) in tests/test_oracle.py and is
    the blueprint for the kernels in newtonnet_b200/csrc.

    Undirected pairs p = (i<j) with disp_p = pos_i - pos_j (minimum image).  m, e1, e2 are symmetric
    in (i,j) so they are evaluated once per pair; the directed sums run over a destination-sorted
    adjacency with an orientation sign.
    """
    sd = as_torch_sd(sd, dtype)
    z = torch.as_tensor(np.asarray(z)).long()
    batch = torch.as_tensor(np.asarray(batch)).long()
    pos = torch.as_tensor(np.asarray(pos)).to(dtype)
    cell = torch.as_tensor(np.asarray(cell)).to(dtype)
    N = z.shape[0]
    n_sys = cell.shape[0]
    if edge_index is None:
        edge_index, disp = radius_graph_dense(pos, cell, batch, cutoff)
    else:
        edge_index = torch.as_tensor(np.asarray(edge_index)).long()
        disp = torch.as_tensor(np.asarray(disp)).to(dtype)
    fwd = edge_index[0] < edge_index[1]
    pi, pj, dp = edge_index[0][fwd], edge_index[1][fwd], disp[fwd]
    freq = sd['embedding_layers.edge_embedding.embedding.frequencies']
    d = dp.norm(dim=1, keepdim=True)
    u = dp / d
    x = d / cutoff
    env = polynomial_cutoff(x)
    sb = torch.sin(freq * x) / x
    rbf = env * sb
    L = n_layers(sd)
    F = sd['embedding_layers.node_embedding.weight'].shape[1]
    a = sd['embedding_layers.node_embedding.weight'][z]
    f = torch.zeros(N, 3, F, dtype=dtype)

    def both(t_i, t_j):   # sum of a per-pair quantity into both endpoints
        return _segment_sum(t_i, pi, N) + _segment_sum(t_j, pj, N)

    saved = []
    for l in range(L):
        k = f'interaction_layers.{l}.'
        W1, b1 = sd[k + 'message_nodepart.0.weight'], sd[k + 'message_nodepart.0.bias']
        W2, b2 = sd[k + 'message_nodepart.2.weight'], sd[k + 'message_nodepart.2.bias']
        We = sd[k + 'message_edgepart.weight']
        U1, U2 = sd[k + 'equiv_message1.0.weight'], sd[k + 'equiv_message1.2.weight']
        V1, V2 = sd[k + 'equiv_message2.0.weight'], sd[k + 'equiv_message2.2.weight']
        Wu = sd[k + 'equiv_update.weight']
        pre = a @ W1.T + b1
        mn = silu(pre) @ W2.T + b2
        me = rbf @ We.T
        m = me * (mn[pi] * mn[pj])
        a = a + both(m, m)
        q1 = m @ U1.T
        q2 = m @ V1.T
        e1 = silu(q1) @ U2.T
        e2 = silu(q2) @ V2.T
        f_in = f
        # destination i gets +u, destination j gets -u
        df = both(e1.unsqueeze(1) * u.unsqueeze(2) + e2.unsqueeze(1) * f_in[pj],
                  -e1.unsqueeze(1) * u.unsqueeze(2) + e2.unsqueeze(1) * f_in[pi])
        f = f_in + df
        g = f @ Wu.T
        a = a + (f * g).sum(1)
        saved.append(dict(pre=pre, mn=mn, me=me, m=m, q1=q1, q2=q2, e1=e1, e2=e2, f_in=f_in, f_out=f, g=g))
    # energy head forward + backward
    kh = 'output_layers.0.layers.'
    h1p = a @ sd[kh + '0.weight'].T + sd[kh + '0.bias']
    h2p = silu(h1p) @ sd[kh + '2.weight'].T + sd[kh + '2.bias']
    o = silu(h2p) @ sd[kh + '4.weight'].T + sd[kh + '4.bias']
    scale = sd['scalers.0.scale.weight'][z]
    e_atom = o * scale + sd['scalers.0.shift.weight'][z]
    energy = _segment_sum(e_atom, batch, n_sys).reshape(-1)
    gh2 = (scale @ sd[kh + '4.weight']) * silu_grad(h2p)
    gh1 = (gh2 @ sd[kh + '2.weight']) * silu_grad(h1p)
    abar = gh1 @ sd[kh + '0.weight']
    fbar = torch.zeros_like(f)
    rbf_bar = torch.zeros_like(rbf)
    ubar = torch.zeros_like(u)
    for l in reversed(range(L)):
        k = f'interaction_layers.{l}.'
        W1 = sd[k + 'message_nodepart.0.weight']; W2 = sd[k + 'message_nodepart.2.weight']
        We = sd[k + 'message_edgepart.weight']
        U1, U2 = sd[k + 'equiv_message1.0.weight'], sd[k + 'equiv_message1.2.weight']
        V1, V2 = sd[k + 'equiv_message2.0.weight'], sd[k + 'equiv_message2.2.weight']
        Wu = sd[k + 'equiv_update.weight']
        s = saved[l]
        dfb = fbar + abar.unsqueeze(1) * s['g'] + (abar.unsqueeze(1) * s['f_out']) @ Wu     # [N,3,F]
        w = dfb[pi] - dfb[pj]                                                                # [P,3,F]
        e1b = (w * u.unsqueeze(2)).sum(1)
        ubar = ubar + (w * s['e1'].unsqueeze(1)).sum(2)
        e2b = (dfb[pi] * s['f_in'][pj] + dfb[pj] * s['f_in'][pi]).sum(1)
        fbar = dfb + both(dfb[pj] * s['e2'].unsqueeze(1), dfb[pi] * s['e2'].unsqueeze(1))
        mb = ((e1b @ U2) * silu_grad(s['q1'])) @ U1 + ((e2b @ V2) * silu_grad(s['q2'])) @ V1 \
            + abar[pi] + abar[pj]
        mnprod = s['mn'][pi] * s['mn'][pj]
        rbf_bar = rbf_bar + (mb * mnprod) @ We
        t = mb * s['me']
        mnb = both(t * s['mn'][pj], t * s['mn'][pi])
        abar = abar + ((mnb @ W2) * silu_grad(s['pre'])) @ W1
    # edge geometry backward
    fx = freq * x
    envp = -0.5 * POLY_P * (POLY_P + 1) * (POLY_P + 2) * x.pow(POLY_P - 1) * (1 - x) ** 2
    sbp = (fx * torch.cos(fx) - torch.sin(fx)) / (x * x)
    xbar = (rbf_bar * (envp * sb + env * sbp)).sum(1, keepdim=True)
    G = (xbar / cutoff) * u + (ubar - (ubar * u).sum(1, keepdim=True) * u) / d
    g_pos = _segment_sum(G, pi, N) - _segment_sum(G, pj, N)
    # dE/dD through the strain trick (models/newtonnet.py:153-155): pos' = pos @ S feeds the raw
    # difference dpos = pos_i - pos_j, cell' = cell @ S feeds the image shift cell' @ n, so
    # M[a,b] = sum_p dpos_a G_b - (cell^T G)_a n_b ; dE/dD = (M + M^T)/2.  For cubic cells this equals
    # sum_p disp (x) G; for other cells it is the reference's (quirky) value that parity is held to.
    dpos = pos[pi] - pos[pj]
    M = dpos.unsqueeze(2) * G.unsqueeze(1)
    if bool((cell != 0).any()):
        h = cell[batch[pi]]
        nimg = torch.round(torch.linalg.solve(h.transpose(1, 2), dpos))
        M = M - torch.bmm(h.transpose(1, 2), G.unsqueeze(2)) * nimg.unsqueeze(1)
    M_pair = M
    M = _segment_sum(M, batch[pi], n_sys)
    g_D = 0.5 * (M + M.transpose(1, 2))
    # per-pair terms too (pairs [2,P] = (i<j), G = dE/d disp, M before the per-system sum): what one atom or one pair
    # contributes to the virial, for tests that must notice an atom dropped from or counted twice in a sum
    out = {'energy': energy.numpy(), 'forces': (-g_pos).numpy(), 'virial': (-g_D).numpy(),
           'atom_node': a.numpy(), 'force_node': f.numpy(), 'pairs': torch.stack([pi, pj]).numpy(),
           'G': G.numpy(), 'M': M_pair.numpy()}
    if bool((cell != 0).any()):
        out['stress'] = (g_D / torch.linalg.det(cell).view(-1, 1, 1)).numpy()
    return out


def hessian(sd, z, pos, cell, batch, dtype=torch.float64, cutoff=CUTOFF):
    """HessianOutput, models/output.py:134-152: d(pos_grad)/d pos, [N,3,N,3]."""
    sd = as_torch_sd(sd, dtype)
    z = torch.as_tensor(np.asarray(z)).long()
    batch = torch.as_tensor(np.asarray(batch)).long()
    pos = torch.as_tensor(np.asarray(pos)).to(dtype).clone().requires_grad_(True)
    cell = torch.as_tensor(np.asarray(cell)).to(dtype)
    rbf, direction, edge_index = edge_embedding(sd, pos, cell, batch, cutoff)
    a = sd['embedding_layers.node_embedding.weight'][z]
    f = torch.zeros(z.shape[0], 3, a.shape[1], dtype=dtype)
    for l in range(n_layers(sd)):
        a, f = interaction(sd, l, a, f, direction, rbf, edge_index)
    energy = _segment_sum(atomic_energy(sd, a, z), batch, cell.shape[0]).reshape(-1)
    g, = torch.autograd.grad(energy, pos, torch.ones_like(energy), create_graph=True)
    flat = g.reshape(-1)
    rows = [torch.autograd.grad(flat[r], pos, retain_graph=True)[0] for r in range(flat.numel())]
    n = z.shape[0]
    return torch.stack(rows).reshape(n, 3, n, 3).numpy()


# ----------------------------------------------------------------------------- row T: training step
def training_gradients(sd, z, pos, cell, batch, e_target, f_target, force_weight=50.0, dtype=torch.float64,
                       cutoff=CUTOFF):
    """Loss and parameter gradients of one training step: forward with create_graph=True
    (models/newtonnet.py:106-113, models/output.py:66-73), loss = MSE(E) + w MSE(F) (train/loss.py:48,
    104-138), loss.backward() (train/trainer.py:310) - the double backward through the force graph.
    Returns (loss, {parameter name: gradient ndarray})."""
    params = {k: torch.as_tensor(np.asarray(v)).to(dtype).requires_grad_(k.split('.')[-1] != 'frequencies')
              for k, v in sd.items()}
    z = torch.as_tensor(np.asarray(z)).long()
    batch = torch.as_tensor(np.asarray(batch)).long()
    pos = torch.as_tensor(np.asarray(pos)).to(dtype).clone().requires_grad_(True)
    cell = torch.as_tensor(np.asarray(cell)).to(dtype)
    n_sys = cell.shape[0]
    rbf, direction, edge_index = edge_embedding(params, pos, cell, batch, cutoff)
    a = torch.nn.functional.embedding(z, params['embedding_layers.node_embedding.weight'], padding_idx=0)
    f = torch.zeros(z.shape[0], 3, a.shape[1], dtype=dtype)
    for l in range(n_layers(sd)):
        a, f = interaction(params, l, a, f, direction, rbf, edge_index)
    energy = _segment_sum(atomic_energy(params, a, z), batch, n_sys).reshape(-1)
    g_pos, = torch.autograd.grad(energy, pos, torch.ones_like(energy), create_graph=True)
    e_t = torch.as_tensor(np.asarray(e_target)).to(dtype)
    f_t = torch.as_tensor(np.asarray(f_target)).to(dtype)
    loss = torch.mean((energy - e_t) ** 2) + force_weight * torch.mean((-g_pos - f_t) ** 2)
    names = [k for k, v in params.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [params[k] for k in names], allow_unused=True)
    out = {k: (np.zeros(params[k].shape) if g is None else g.detach().numpy()) for k, g in zip(names, grads)}
    return float(loss), out


# ----------------------------------------------------------------------------- synthetic workloads
def water_box(nside, seed=0):
    """Synthetic periodic water lattice of SURVEY.md §8d C3/C4 (numpy restatement of the generator in
    tests/golden/make_golden.py; same distribution, numpy RNG).  Returns z,pos,cell,batch."""
    rng = np.random.default_rng(seed)
    a = 3.104
    idx = np.stack(np.meshgrid(*[np.arange(nside)] * 3, indexing='ij'), -1).reshape(-1, 3).astype(np.float64)
    n = idx.shape[0]
    O = (idx + 0.5) * a + (rng.random((n, 3)) - 0.5) * 0.4
    Q, _ = np.linalg.qr(rng.standard_normal((n, 3, 3)))
    ang = math.radians(104.52)
    H1 = O + Q @ np.array([0.9572, 0.0, 0.0])
    H2 = O + Q @ np.array([0.9572 * math.cos(ang), 0.9572 * math.sin(ang), 0.0])
    L = nside * a
    pos = (np.stack([O, H1, H2], 1).reshape(-1, 3) % L).astype(np.float32)
    pos = np.where(pos >= np.float32(L), np.float32(0), pos)
    z = np.tile(np.array([8, 1, 1], dtype=np.int64), n)
    cell = (np.eye(3) * L).astype(np.float32)[None]
    return z, pos, cell, np.zeros(3 * n, dtype=np.int64)


def molecule_batch(n_mol, seed=1, lo=4, hi=65, sizes=None):
    """Synthetic ANI-1x-shaped ragged batch of SURVEY.md §8d C2 (numpy RNG).  Returns z,pos,cell,batch."""
    rng = np.random.default_rng(seed)
    if sizes is None:
        sizes = rng.integers(lo, hi, n_mol)
    zs, ps, bs = [], [], []
    for b, n in enumerate(sizes):
        n = int(n)
        m = int(math.ceil(n ** (1 / 3))) + 1
        sites = rng.permutation(m ** 3)[:n]
        ijk = np.stack([sites // (m * m), (sites // m) % m, sites % m], 1).astype(np.float64)
        ps.append(ijk * 1.4 + (rng.random((n, 3)) - 0.5) * 0.5)
        zs.append(np.array([1, 6, 7, 8])[rng.integers(0, 4, n)])
        bs.append(np.full(n, b, dtype=np.int64))
    return (np.concatenate(zs).astype(np.int64), np.concatenate(ps).astype(np.float32),
            np.zeros((len(sizes), 3, 3), dtype=np.float32), np.concatenate(bs))

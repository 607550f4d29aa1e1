"""Hessians in batched blocks of rows (reference models/output.py:141-152 batches the rows of d pos_grad / d pos with vmap).

One reverse pass gives k rows, exactly: a pass puts k copies of frames into one molecule batch, copy c being its own
system, and differentiates <seed, pos_grad> with respect to the replicated positions, where the seed holds a one-hot for
row r_c in copy c's block.  Copy c's block of that gradient is row r_c of its frame's Hessian; nothing crosses between
copies.  One forward, one create_graph first backward and one second backward over k n atoms therefore give k rows,
where the per-row loop (train.hessian_rows) needs one second backward over the whole batch for every row.

Every primitive on the path treats rows independently or sums over per-system segments of the destination-sorted CSR in
a fixed order, and each copy's neighbour list is that of its frame, so each row is bit-identical to the row the per-row
loop computes (tests/test_gpu_hessian.py).

    job    one (frame, row) pair; a padding job (row -1) copies a frame and gets a zero seed
    pass   k jobs whose frames have the same atom count n: k n replicated atoms, at most the atom budget (one oversized
           frame still runs at k = 1); the last pass of a group is padded, so all passes of a group share one shape
    group  the passes of the frames of one atom count

The pass (csrc/hessian.cu nn_hessian_expand -> neighbour rebuild -> differentiable_forward on the replicated batch ->
two reverse sweeps -> nn_hessian_scatter) reads its jobs from a plan in device memory and advances a device-side pass
counter, so it is captured once as a CUDA graph and replayed once per pass; graphs are cached by (frame sizes, selection,
budget, parameter addresses) and reused when the same molecule comes back at new positions.  Edge capacity is tight, as in
GraphedTrainingStep; a pass whose list outgrows it leaves a flag that is read after the group's replays, and the group is
then recaptured with more room and run again.  NN_HESSIAN_GRAPH=0 runs the same passes eagerly.
"""
import os

import numpy as np
import torch

from . import _lib as L
from .engine import NeighborList, all_pairs_bound, capture, count_edges, edge_capacity, get_engine, stream, warm_up

# Device memory one replicated atom costs on the differentiable path (forward + create_graph backward + second backward):
# peak allocated bytes of a call over the atoms of its largest pass, MEASURED with tools/bench_hessian.py on a B200
# (1000 W): 1.59 MB for the 81-atom periodic water box (~54 directed edges per atom, the densest case measured), 0.46 MB
# for aspirin.
BYTES_PER_ATOM = 1_600_000
MEMORY_FRACTION = 0.25          # of the device memory free at the first call: the rest stays with the caller
# Default budget ceiling.  Measured on the same B200, graphed water box: 12 / 49 / 81 / 122 rows per pass -> 87.8 / 61.8 /
# 58.8 / 57.6 ms, so passes beyond ~4k replicated atoms gain little while their memory keeps growing.
MAX_ATOMS = 8192

stats = {'captures': 0, 'passes': 0}      # CUDA-graph captures and passes run since import (tests, tools/bench_hessian.py)


# ----------------------------------------------------------------------------- planner (host only)
class Group:
    """Passes over frames of n atoms: plan [n_pass, k, 3] int32 rows {frame, local row or -1, output row}."""

    def __init__(self, n, k, plan):
        self.n, self.k, self.plan = int(n), int(k), plan

    @property
    def n_pass(self):
        return self.plan.shape[0]


def plan_passes(frame_sizes, atoms=None, budget=MAX_ATOMS):
    """Jobs for every row of every frame (atoms=None: output row 3 i + d of global atom i) or for the rows of the selected
    global atoms (output row 3 m + d of the m-th selected atom), packed into passes of at most `budget` replicated atoms.
    Returns (groups, n_output_rows).  Jobs keep their order within a group; the pass count of a group is the least the
    budget allows, and its jobs are spread evenly over those passes (the last one is padded)."""
    sizes = np.asarray(frame_sizes, dtype=np.int64).reshape(-1)
    if sizes.size == 0 or (sizes < 0).any():
        raise ValueError('frame sizes must be a non-empty list of non-negative atom counts')
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    N = int(ptr[-1])
    budget = max(int(budget), 1)
    if atoms is None:
        sel = np.arange(N, dtype=np.int64)
    else:
        sel = np.asarray(atoms, dtype=np.int64).reshape(-1)
        if sel.size == 0:
            raise ValueError('atoms= selects no atom')
        if (sel < 0).any() or (sel >= N).any():
            raise IndexError(f'atoms= holds an index outside [0, {N})')
    frame = np.searchsorted(ptr, sel, side='right') - 1
    local = sel - ptr[frame]
    jobs = {}                                          # n -> list of (frame, local row, output row)
    for m, (f, a) in enumerate(zip(frame.tolist(), local.tolist())):
        for d in range(3):
            jobs.setdefault(int(sizes[f]), []).append((f, 3 * a + d, 3 * m + d))
    groups = []
    for n, js in jobs.items():
        k = max(min(budget // max(n, 1), len(js)), 1)
        n_pass = -(-len(js) // k)
        k = -(-len(js) // n_pass)                      # same pass count, least padding
        plan = np.empty((n_pass * k, 3), dtype=np.int32)
        plan[:len(js)] = js
        plan[len(js):] = (js[0][0], -1, -1)            # padding jobs copy the group's first frame
        groups.append(Group(n, k, plan.reshape(n_pass, k, 3)))
    return groups, 3 * sel.size


_budgets = {}


def default_budget(device):
    """Replicated atoms per pass: NN_HESSIAN_ATOMS, else MEMORY_FRACTION of the device memory free at the first call over
    BYTES_PER_ATOM (kept for the device's later calls, so the cached graphs stay valid), at most MAX_ATOMS."""
    env = os.environ.get('NN_HESSIAN_ATOMS')
    if env:
        return max(int(env), 1)
    key = str(device)
    if key not in _budgets:
        free, _ = torch.cuda.mem_get_info(device)
        free += torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
        _budgets[key] = int(min(max(MEMORY_FRACTION * free // BYTES_PER_ATOM, 1), MAX_ATOMS))
    return _budgets[key]


# ----------------------------------------------------------------------------- device side
class _GroupRunner:
    """The passes of one group on static buffers; one CUDA graph replayed once per pass (or the same pass run eagerly).
    It holds no reference to its _Blocks (which is passed in): an evicted _Blocks then frees its graphs at once, by
    reference count, instead of whenever the cyclic collector runs - possibly in the middle of a later capture."""

    HEADROOM = (1.05, 256)         # tight edge capacity, as in GraphedTrainingStep: factor and slack over the counted edges

    def __init__(self, b, group, max_edges):
        dev = b.device
        self.group = group
        k, n = group.k, group.n
        self.plan = torch.as_tensor(group.plan, device=dev).contiguous()
        self.z_rep = torch.empty(k * n, dtype=torch.int64, device=dev)
        self.pos_rep = torch.empty(k * n, 3, dtype=torch.float32, device=dev)
        self.cell_rep = torch.empty(k, 3, 3, dtype=torch.float32, device=dev)
        self.batch_rep = torch.empty(k * n, dtype=torch.int64, device=dev)
        self.seed = torch.empty(k * n, 3, dtype=torch.float32, device=dev)
        self.bound = all_pairs_bound(b.cell, torch.arange(k).repeat_interleave(n))     # k copies of an n-atom frame
        self.graph = None
        self.recaptures = 0
        self._build(b, self._capacity(k * max_edges))

    def _capacity(self, n_edges):
        return edge_capacity(n_edges, *self.HEADROOM, self.bound)

    def _build(self, b, cap_edges):
        self.graph = None                              # the previous capture's graph goes first
        self.nl = NeighborList(b.engine, self.pos_rep, self.cell_rep, self.batch_rep, cap_edges=cap_edges)
        if not b.graphed:
            return

        def first_pass():
            b.ctr.zero_()
            self._pass(b)
        warm_up(first_pass, b.device, 1)
        self.graph, _, _ = capture(lambda: self._pass(b), b.device, pool=b.pool)
        stats['captures'] += 1

    def _pass(self, b):
        from newtonnet_b200.train import _skip_weight_grads, differentiable_forward
        g, lib, s = self.group, b.lib, stream()
        L.check(lib.nn_hessian_expand(self.plan.data_ptr(), b.ctr.data_ptr(), g.k, g.n, b.z.data_ptr(), b.pos.data_ptr(),
                                      b.cell.data_ptr(), b.frame_ptr.data_ptr(), self.z_rep.data_ptr(), self.pos_rep.data_ptr(),
                                      self.cell_rep.data_ptr(), self.batch_rep.data_ptr(), self.seed.data_ptr(), s),
                'nn_hessian_expand')
        self.nl.rebuild(b.model.cutoff)
        pos = self.pos_rep.detach().requires_grad_(True)
        out = differentiable_forward(b.model, self.z_rep, pos, self.cell_rep, self.batch_rep, static_nl=self.nl,
                                     properties=('energy',))
        with _skip_weight_grads():                     # only d/d pos is asked for in both sweeps
            pos_grad, = torch.autograd.grad(out.energy, pos, torch.ones_like(out.energy), create_graph=True)
            rows, = torch.autograd.grad(pos_grad, pos, self.seed)
        L.check(lib.nn_hessian_scatter(self.plan.data_ptr(), b.ctr.data_ptr(), g.k, g.n, b.frame_ptr.data_ptr(),
                                       rows.contiguous().data_ptr(), b.H.data_ptr(), b.H.shape[1], b.ticket.data_ptr(), s),
                'nn_hessian_scatter')
        torch.maximum(b.sticky, self.nl.status[L.ST_EDGE_OVERFLOW:L.ST_EDGE_OVERFLOW + 1], out=b.sticky)

    def run(self, b):
        for attempt in range(4):
            b.ctr.zero_()
            b.sticky.zero_()
            for _ in range(self.group.n_pass):
                if self.graph is not None:
                    self.graph.replay()
                else:
                    self._pass(b)
            stats['passes'] += self.group.n_pass
            need = int(b.sticky.item())                 # edges the fullest pass needed, 0 = every pass fit
            if need == 0:
                return
            if attempt == 3:
                break
            self._build(b, max(self._capacity(need), self.nl.cap_edges + 2))
            self.recaptures += 1
        raise RuntimeError(f'Hessian pass: edge capacity {self.nl.cap_edges} still overflowed after regrowing')


class _Blocks:
    """Static inputs / output of one Hessian shape and the runners of its groups."""

    def __init__(self, model, z, pos, cell, batch, frame_sizes, atoms, budget, graphed):
        dev = pos.device
        self.model, self.device, self.graphed = model, dev, graphed
        self.engine = get_engine(dev)
        self.lib = L.load()
        N, B = pos.shape[0], cell.shape[0]
        self.groups, n_rows = plan_passes(frame_sizes, atoms, budget)
        i32 = dict(dtype=torch.int32, device=dev)
        self.z = torch.empty(N, dtype=torch.int64, device=dev)
        self.pos = torch.empty(N, 3, dtype=torch.float32, device=dev)
        self.cell = torch.empty(B, 3, 3, dtype=torch.float32, device=dev)
        self.frame_ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(frame_sizes)]), **i32)
        self.H = torch.empty(n_rows, 3 * N, dtype=torch.float32, device=dev)
        self.ctr = torch.zeros(1, **i32)
        self.ticket = torch.zeros(1, **i32)
        self.sticky = torch.zeros(1, **i32)
        self.pool = torch.cuda.graph_pool_handle() if graphed else None     # one pool for the groups' graphs
        self.copy_in(z, pos, cell)
        # edges per frame from a counting pass over the input batch size the first capture
        probe = count_edges(self.engine, self.pos, self.cell, batch.to(torch.int64).contiguous(), model.cutoff)
        per_frame = (probe.row_ptr[probe.sys_ptr[1:].long()] - probe.row_ptr[probe.sys_ptr[:-1].long()]).cpu().numpy()
        self.runners = []
        for g in self.groups:
            frames = np.unique(g.plan[:, :, 0])
            self.runners.append(_GroupRunner(self, g, int(per_frame[frames].max())))

    def copy_in(self, z, pos, cell):
        self.z.copy_(z)
        self.pos.copy_(pos.detach())
        self.cell.copy_(cell.detach().reshape(-1, 3, 3))

    def __call__(self):
        for r in self.runners:
            r.run(self)
        return self.H.clone()


_cache = {}
_CACHE_SIZE = 4


def hessian_blocks(model, z, pos, cell, batch, atoms=None):
    """d^2 E / d pos d pos in batched blocks of rows: [N,3,N,3], or [M,3,N,3] for the M selected atoms (global indices)."""
    if not pos.is_cuda:
        raise RuntimeError('newtonnet_b200: inputs must be CUDA tensors - there is no CPU fallback')
    if pos.dtype != torch.float32 or next(model.parameters()).dtype != torch.float32:
        raise NotImplementedError('the Hessian path computes in fp32: cast the model and inputs to float32')
    cell = cell.reshape(-1, 3, 3)
    N, B = pos.shape[0], cell.shape[0]
    b_host = batch.detach().to('cpu', torch.int64).numpy()
    if b_host.size and ((np.diff(b_host) < 0).any() or b_host[0] < 0 or b_host[-1] >= B):
        raise ValueError('batch must be non-decreasing with values in [0, n_systems)')
    if b_host.size != N:
        raise ValueError('batch must hold one system index per atom')
    sizes = np.bincount(b_host, minlength=B)
    sel = None if atoms is None else torch.as_tensor(atoms).detach().to('cpu', torch.int64).reshape(-1).numpy()
    graphed = os.environ.get('NN_HESSIAN_GRAPH', '1') != '0'
    budget = default_budget(pos.device)
    # a captured pass reads the parameters where they were at capture time: a model whose tensors moved gets new graphs
    params = tuple(p.data_ptr() for p in model.parameters())
    key = (str(pos.device), id(model), params, tuple(sizes.tolist()), None if sel is None else tuple(sel.tolist()), budget, graphed)
    blocks = _cache.pop(key, None)
    if blocks is None:
        blocks = _Blocks(model, z, pos, cell, batch, sizes, sel, budget, graphed)
        while len(_cache) >= _CACHE_SIZE:
            _cache.pop(next(iter(_cache)))
    else:
        blocks.copy_in(z, pos, cell)
    _cache[key] = blocks                               # most recently used last
    H = blocks()
    M = H.shape[0] // 3
    return H.reshape(M, 3, N, 3)


def hessian(model, z, pos, cell, batch, atoms=None):
    """Hessian of the model's energy with respect to the positions.

    z [N] int64, pos [N,3] fp32, cell [B,3,3] (zeros = not periodic), batch [N] non-decreasing system index, all on one
    CUDA device; atoms: optional global atom indices.  Returns hessian[i,a,j,b] = d^2 E / d pos_ia d pos_jb as [N,3,N,3],
    or [M,3,N,3] for the M selected atoms (rows of an adsorbate or active site, as partial vibrational analyses use).
    Blocks between atoms of different systems are exactly zero."""
    return hessian_blocks(model, z, pos, cell, batch, atoms)

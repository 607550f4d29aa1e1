"""Host driver of the CUDA path: neighbour list, weight pack, one-call evaluation.

PyTorch is used for device memory and streams only; all arithmetic happens in
libnewtonnet_b200.so (include/newtonnet_b200.h).
"""
import ctypes as C
import gc
import os

import numpy as np
import torch

from . import _lib as L


def stream():
    """Raw handle of the current CUDA stream, as the library's entry points take it."""
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(f'newtonnet_b200: `{name}` must be a CUDA tensor - this package has no CPU fallback '
                           f'(use the reference implementation or oracle/ for CPU).')


class WeightPack:
    """fp32 device copies of the reference parameters in both orientations (nn_weights)."""

    def __init__(self, state, cutoff, device):
        """`state`: mapping with the reference's parameter names (SURVEY.md section 8b) -> tensors."""
        self.keep = []
        dev = device

        def f32(t):
            t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
            self.keep.append(t)
            return t

        lib = L.load()
        stream = torch.cuda.current_stream(dev).cuda_stream

        def image(b):
            img = torch.empty(L.NN_B_IMAGE_FLOATS, dtype=torch.float32, device=dev)
            self.keep.append(img)
            L.check(lib.nn_gemm128_prepare_b(b.data_ptr(), img.data_ptr(), stream), 'nn_gemm128_prepare_b')
            return img.data_ptr()

        def mat(dst, t):
            """Both orientations of a [128,128] weight plus their tensor-core operand images."""
            w = f32(t)
            wt = f32(t.detach().t())
            dst.w, dst.wt = w.data_ptr(), wt.data_ptr()
            dst.w_img, dst.wt_img = image(w), image(wt)

        def both(t):
            w = f32(t)
            wt = f32(t.detach().t())
            return w.data_ptr(), wt.data_ptr()

        w = L.Weights()
        n_layers = 1 + max(int(k.split('.')[1]) for k in state if k.startswith('interaction_layers.'))
        if n_layers > L.NN_MAX_LAYERS:
            raise ValueError(f'n_interactions={n_layers} > {L.NN_MAX_LAYERS}')
        emb = state['embedding_layers.node_embedding.weight']
        if emb.shape[1] != L.NN_F:
            raise NotImplementedError(f'kernels are specialised for n_features={L.NN_F}, got {emb.shape[1]}')
        freq = state['embedding_layers.edge_embedding.embedding.frequencies']
        if freq.numel() != L.NN_NB:
            raise NotImplementedError(f'kernels are specialised for n_basis={L.NN_NB}, got {freq.numel()}')
        w.n_layers = n_layers
        w.cutoff = float(cutoff)
        w.embedding = f32(emb).data_ptr()
        w.frequencies = f32(freq).data_ptr()
        for l in range(n_layers):
            k = f'interaction_layers.{l}.'
            lw = w.layer[l]
            if (k + 'layer_norm.weight') in state:
                lw.ln_gamma = f32(state[k + 'layer_norm.weight']).data_ptr()
                lw.ln_beta = f32(state[k + 'layer_norm.bias']).data_ptr()
            mat(lw.W1, state[k + 'message_nodepart.0.weight'])
            lw.b1 = f32(state[k + 'message_nodepart.0.bias']).data_ptr()
            mat(lw.W2, state[k + 'message_nodepart.2.weight'])
            lw.b2 = f32(state[k + 'message_nodepart.2.bias']).data_ptr()
            lw.We, lw.Wet = both(state[k + 'message_edgepart.weight'])
            we_img = torch.empty(L.NN_WE_IMAGE_FLOATS, dtype=torch.float32, device=dev)
            self.keep.append(we_img)
            L.check(lib.nn_message_prepare_b(lw.We, we_img.data_ptr(), stream), 'nn_message_prepare_b')
            lw.We_img = we_img.data_ptr()
            mat(lw.U1, state[k + 'equiv_message1.0.weight'])
            mat(lw.U2, state[k + 'equiv_message1.2.weight'])
            mat(lw.V1, state[k + 'equiv_message2.0.weight'])
            mat(lw.V2, state[k + 'equiv_message2.2.weight'])
            mat(lw.Wu, state[k + 'equiv_update.weight'])
        h = 'output_layers.0.layers.'
        hk = [k for k in state if k.endswith('layers.0.weight') and k.startswith('output_layers.')]
        if hk:
            h = hk[0][:-len('0.weight')]
        idx = h.split('.')[1]
        mat(w.H1, state[h + '0.weight'])
        w.hb1 = f32(state[h + '0.bias']).data_ptr()
        mat(w.H2, state[h + '2.weight'])
        w.hb2 = f32(state[h + '2.bias']).data_ptr()
        w.w3 = f32(state[h + '4.weight'].reshape(-1)).data_ptr()
        w.hb3 = f32(state[h + '4.bias'].reshape(-1)).data_ptr()
        w.scale = f32(state[f'scalers.{idx}.scale.weight'].reshape(-1)).data_ptr()
        w.shift = f32(state[f'scalers.{idx}.shift.weight'].reshape(-1)).data_ptr()
        self.has_direct_force = 'direct_head.layers.0.weight' in state
        if self.has_direct_force:
            mat(w.D1, state['direct_head.layers.0.weight']); w.db1 = f32(state['direct_head.layers.0.bias']).data_ptr()
            mat(w.D2, state['direct_head.layers.2.weight']); w.db2 = f32(state['direct_head.layers.2.bias']).data_ptr()
            mat(w.D3, state['direct_head.layers.4.weight']); w.db3 = f32(state['direct_head.layers.4.bias']).data_ptr()
            w.dscale = f32(state['direct_head.scale'].reshape(-1)).data_ptr()
        self.struct = w
        self.n_layers = n_layers
        self.cutoff = float(cutoff)


class NeighborList:
    """Destination-sorted CSR + undirected pair list on the device (nn_nbr)."""

    def __init__(self, engine, pos, cell, batch, cap_edges, cap_pairs=None, n_owned=0):
        """cap_pairs: capacity of the pair table; default cap_edges / 2 (complete lists have P = E / 2 - lists with empty
        ghost rows, domain decomposition, have up to P = E pairs and pass it explicitly).
        n_owned > 0: atoms [n_owned, N) are ghosts, and pairs between two ghosts are left out."""
        N, B = pos.shape[0], cell.shape[0]
        dev = pos.device
        i32 = dict(dtype=torch.int32, device=dev)
        self.pos, self.cell, self.batch = pos, cell, batch
        self.n_atoms, self.n_systems = N, B
        self.cap_edges = int(cap_edges)
        self.cap_pairs = (self.cap_edges + 1) // 2 if cap_pairs is None else int(cap_pairs)
        self.sys_ptr = torch.empty(B + 1, **i32)
        self.row_ptr = torch.empty(N + 1, **i32)
        self.pair_ptr = torch.empty(N + 1, **i32)
        self.col = torch.empty(max(self.cap_edges, 1), **i32)
        self.edge_pair = torch.empty(max(self.cap_edges, 1), **i32)
        self.pair_i = torch.empty(max(self.cap_pairs, 1), **i32)
        self.pair_j = torch.empty(max(self.cap_pairs, 1), **i32)
        self.pair_disp = torch.empty(max(self.cap_pairs, 1), 3, dtype=torch.float32, device=dev)
        self.status = torch.zeros(L.NN_STATUS_WORDS, **i32)
        ws_bytes = engine.lib.nn_nbr_workspace_bytes(N, B)
        self.workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        s = L.Nbr()
        s.n_atoms, s.n_systems = N, B
        s.cap_edges, s.cap_pairs, s.cap_cells = self.cap_edges, self.cap_pairs, 2 * N + B
        s.n_owned = n_owned
        s.pos, s.cell, s.batch = pos.data_ptr(), cell.data_ptr(), batch.data_ptr()
        s.sys_ptr, s.row_ptr, s.col = self.sys_ptr.data_ptr(), self.row_ptr.data_ptr(), self.col.data_ptr()
        s.edge_pair, s.pair_ptr = self.edge_pair.data_ptr(), self.pair_ptr.data_ptr()
        s.pair_i, s.pair_j, s.pair_disp = self.pair_i.data_ptr(), self.pair_j.data_ptr(), self.pair_disp.data_ptr()
        s.status = self.status.data_ptr()
        s.workspace, s.workspace_bytes = self.workspace.data_ptr(), ws_bytes
        self.struct = s
        self.n_edges = None   # known on the host after `check()`
        self.generation = 0   # bumped every time the list is rebuilt in place

    def rebind(self, pos, cell, batch):
        """Point the list at new input tensors of the same shapes (next MD step)."""
        self.pos, self.cell, self.batch = pos, cell, batch
        self.struct.pos, self.struct.cell, self.struct.batch = pos.data_ptr(), cell.data_ptr(), batch.data_ptr()

    def rebuild(self, cutoff):
        """Count + fill on the current stream.  A list that outgrows its capacity is not filled: the status words say so."""
        lib, s = L.load(), stream()
        self.n_edges = None
        L.check(lib.nn_nbr_count(C.byref(self.struct), cutoff, s), 'nn_nbr_count')
        L.check(lib.nn_nbr_fill(C.byref(self.struct), cutoff, s), 'nn_nbr_fill')

    def check(self):
        """Read the status words (one small D2H copy, synchronises the stream)."""
        st = self.status.cpu().tolist()
        if st[L.ST_BATCH_UNSORTED] == 1:
            raise ValueError('batch must be non-decreasing with values in [0, n_systems)')
        if st[L.ST_BATCH_UNSORTED] == 3:
            raise ValueError('atomic numbers must be in [0, 118]')
        if st[L.ST_BATCH_UNSORTED] == 2:
            raise RuntimeError('internal error: asymmetric edge set')
        if st[L.ST_SINGULAR_CELL]:
            # the reference raises torch._C._LinAlgError from linalg.solve (representations.py:92)
            raise RuntimeError('singular cell in a periodic batch (mixed periodic / non-periodic systems or '
                               'partially periodic cells are not supported, as in the reference)')
        if st[L.ST_ROW_OVERFLOW]:
            raise RuntimeError(f'an atom has {st[L.ST_ROW_OVERFLOW]} neighbours (> {512})')
        self.n_edges = st[L.ST_N_EDGES]
        return st

    def edge_index(self, generation=None):
        """[2,E] int64, reference order (i-major, j ascending)."""
        if generation is not None and generation != self.generation:
            raise RuntimeError('edge_index of an earlier forward() was requested after the neighbour list had been '
                               'rebuilt in place by a later call; read it before the next forward()')
        if self.n_edges is None:
            self.check()
        out = torch.empty(2, self.n_edges, dtype=torch.int64, device=self.pos.device)
        if self.n_edges:
            lib = L.load()
            L.check(lib.nn_nbr_edge_index(C.byref(self.struct), out.data_ptr(), self.n_edges, stream()), 'nn_nbr_edge_index')
        return out


def count_edges(engine, pos, cell, batch, cutoff, n_owned=0):
    """Count-only pass over a list of capacity 0.  Returns that list, checked: `n_edges` holds the directed edges the
    inputs need, and `row_ptr` / `sys_ptr` the count per atom / per system."""
    probe = NeighborList(engine, pos, cell, batch, cap_edges=0, n_owned=n_owned)
    L.check(engine.lib.nn_nbr_count(C.byref(probe.struct), cutoff, stream()), 'nn_nbr_count')
    probe.check()
    return probe


def edge_capacity(n_edges, factor, slack, bound=None):
    """Edge capacity for `n_edges` edges: int(n_edges * factor) + slack, at most `bound`, made even and at least 2."""
    c = int(n_edges * factor) + slack
    if bound is not None:
        c = min(c, bound)
    return max(c + c % 2, 2)


def edges_needed(status):
    """Edges a list must hold after its status words reported an overflow."""
    return max(status[L.ST_EDGE_OVERFLOW], status[L.ST_N_EDGES])


def all_pairs_bound(cell, batch):
    """Most directed edges a batch without a periodic cell can have: every ordered pair within each system.  None when a
    cell is periodic (periodic images make pairs repeat)."""
    if bool((cell != 0).any()):
        return None
    n = torch.bincount(batch, minlength=cell.shape[0])
    return int((n * (n - 1)).sum())


def eval_outputs(N, B, device, want_forces, want_virial, want_nodes, want_direct):
    """The output tensors nn_eval writes for these requests (the virial needs the forces' reverse sweep)."""
    f32 = dict(dtype=torch.float32, device=device)
    out = {'energy': torch.empty(B, **f32)}
    if want_forces or want_virial:
        out['forces'] = torch.empty(N, 3, **f32)
    if want_virial:
        out['virial'] = torch.empty(B, 3, 3, **f32)
        out['stress'] = torch.empty(B, 3, 3, **f32)
    if want_nodes:
        out['atom_node'] = torch.empty(N, L.NN_F, **f32)
        out['force_node'] = torch.empty(N, 3, L.NN_F, **f32)
    if want_direct:
        out['direct_force'] = torch.empty(N, 3, **f32)
    return out


def eval_args(nl, weights, z, out, ws, want_forces, want_virial, n_owned=0):
    """nn_eval's arguments: outputs are the tensors of `out` (a missing key passes NULL), `ws` is the workspace."""
    a = L.EvalArgs()
    a.nbr, a.w, a.z = C.pointer(nl.struct), C.pointer(weights.struct), z.data_ptr()
    a.want_forces, a.want_virial, a.n_owned = int(want_forces or want_virial), int(want_virial), n_owned
    a.energy = out['energy'].data_ptr()
    for k in ('forces', 'virial', 'stress', 'atom_node', 'force_node', 'direct_force'):
        setattr(a, k, L.ptr(out.get(k)))
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    return a


class _gc_paused:
    """Python's cyclic collector off while a graph is captured.  Collected cycles may own CUDA graphs or events; destroying
    one while a capture is running is not a stream operation and invalidates the capture.  torch.cuda.graph no longer
    collects before it captures."""

    def __enter__(self):
        self.was = gc.isenabled()
        gc.disable()

    def __exit__(self, *exc):
        if self.was:
            gc.enable()
        return False


def capture(fn, device, pool=None):
    """Synchronise the device, then capture fn() as a CUDA graph with the cyclic collector paused.  Returns (graph, what
    fn returned, launches of this library the graph holds)."""
    lib = L.load()
    torch.cuda.synchronize(device)
    graph = torch.cuda.CUDAGraph()
    before = lib.nn_launch_count(0)
    with _gc_paused(), torch.cuda.graph(graph, pool=pool):
        result = fn()
    return graph, result, int(lib.nn_launch_count(0) - before)


def warm_up(fn, device, times):
    """Run fn() `times` times on a side stream that then joins the current one: the warm-up torch asks for before a
    capture, so that lazy initialisation does not happen inside it."""
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        for _ in range(times):
            fn()
    torch.cuda.current_stream(device).wait_stream(side)


def driver_inputs(model, z, pos, cell, batch, who):
    """Inputs of a device-resident driver (DeviceMD, DeviceFIRE), on the model's CUDA device.  Returns (device, engine,
    weight pack, as_t, z [N] int64, x [N,3] fp64 (a copy), batch [N] int64, cell [B,3,3] fp32); as_t(array, dtype)
    moves one more input there.  cell None = not periodic, batch None = one system."""
    dev = next(model.parameters()).device
    if dev.type != 'cuda':
        raise RuntimeError(f'{who} needs the model on a CUDA device (no CPU fallback)')
    as_t = lambda a, dt: torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a).to(device=dev, dtype=dt).contiguous()
    z = as_t(z, torch.int64)
    N = z.shape[0]
    x = as_t(pos, torch.float64).reshape(N, 3).clone()
    batch = torch.zeros(N, dtype=torch.int64, device=dev) if batch is None else as_t(batch, torch.int64)
    B = int(batch.max().item()) + 1 if N else 1
    cell = torch.zeros(B, 3, 3, dtype=torch.float32, device=dev) if cell is None else as_t(cell, torch.float32).reshape(-1, 3, 3)
    if cell.shape[0] != B:
        raise ValueError(f'cell has {cell.shape[0]} systems, batch has {B}')
    return dev, get_engine(dev), model._weight_pack(dev), as_t, z, x, batch, cell


class ForceStep:
    """Energy + forces of a device-resident driver's fixed buffers: a neighbour list over (pos, cell, batch) with room for
    the edges counted plus `headroom`, nn_eval's workspace and arguments.  Calling it rebuilds the list and evaluates, on
    the current stream and capturable.  Use `force_step` to get one that holds every edge."""

    def __init__(self, engine, weights, z, pos, cell, batch, energy, force, n_edges, headroom):
        self.engine, self.weights = engine, weights
        self.nl = NeighborList(engine, pos, cell, batch, cap_edges=edge_capacity(n_edges, *headroom))
        nbytes = engine.lib.nn_eval_workspace_bytes(self.nl.n_atoms, self.nl.n_systems, self.nl.cap_pairs, weights.n_layers, 1)
        self.ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=pos.device)
        self.args = eval_args(self.nl, weights, z, {'energy': energy, 'forces': force}, self.ws, True, False)

    def __call__(self):
        self.nl.rebuild(self.weights.cutoff)
        L.check(self.engine.lib.nn_eval(C.byref(self.args), stream()), 'nn_eval')


def force_step(engine, weights, z, pos, cell, batch, energy, force, n_edges, headroom):
    """A ForceStep for `n_edges` edges that has evaluated energy and forces at the current positions, regrown until its
    neighbour list holds every edge."""
    while True:
        fs = ForceStep(engine, weights, z, pos, cell, batch, energy, force, n_edges, headroom)
        fs()
        st = fs.nl.check()
        if not st[L.ST_EDGE_OVERFLOW]:
            return fs
        n_edges = edges_needed(st)


def replay_chunk(graph, n, sticky, state):
    """Replay a device-resident driver's step graph n times, then read its sticky status words {edges needed, max degree,
    singular cell} once (synchronises).  Raises on a singular cell or an over-full row.  Returns 0, or after a capacity
    overflow somewhere in the chunk the edges a list must hold: every tensor of `state` is then back at its value before
    the chunk and `sticky` is cleared, so the caller regrows and redoes the chunk."""
    snap = [t.clone() for t in state]
    for _ in range(n):
        graph.replay()
    st = sticky.cpu().tolist()
    if st[2]:
        raise RuntimeError('singular cell in a periodic system')
    if st[1]:
        raise RuntimeError(f'an atom has {st[1]} neighbours (> 512)')
    if st[0]:
        for t, s in zip(state, snap):
            t.copy_(s)
        sticky.zero_()
    return st[0]


class Engine:
    """Per-device driver.  Keeps capacities and workspaces between calls so a steady-state evaluation
    allocates nothing and synchronises once (the status read that accompanies the results)."""

    HEADROOM = (1.08, 64)          # edge capacity: factor and slack over the counted edges

    def __init__(self, device):
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('newtonnet_b200 runs on CUDA devices only (no CPU fallback)')
        self.lib = L.load()
        self._nl = None
        self._ws = None
        self.use_cuda_graphs = os.environ.get('NN_CUDA_GRAPHS', '1') != '0'
        self._graphs = {}
        self._last_key = None

    # ------------------------------------------------------------------ neighbour list
    def neighbor_list(self, pos, cell, batch, cutoff):
        for t, n in ((pos, 'pos'), (cell, 'cell'), (batch, 'batch')):
            _require_cuda(t, n)
        pos = pos.detach().to(torch.float32).contiguous()
        cell = cell.detach().to(torch.float32).contiguous().reshape(-1, 3, 3)
        batch = batch.to(torch.int64).contiguous()
        N, B = pos.shape[0], cell.shape[0]
        nl = self._nl
        reuse = nl is not None and nl.n_atoms == N and nl.n_systems == B and nl.pos.device == pos.device
        if reuse:
            nl.rebind(pos, cell, batch)
            nl.generation += 1
            nl.rebuild(cutoff)
            return nl   # overflow (if any) is detected by the caller's status check
        return self._build_with_capacity(pos, cell, batch, cutoff, count_edges(self, pos, cell, batch, cutoff).n_edges)

    def _build_with_capacity(self, pos, cell, batch, cutoff, n_edges):
        nl = NeighborList(self, pos, cell, batch, cap_edges=edge_capacity(n_edges, *self.HEADROOM))
        nl.rebuild(cutoff)
        self._nl = nl
        return nl

    def checked_neighbor_list(self, pos, cell, batch, cutoff):
        """neighbor_list + status read; a cached list whose capacity the new positions outgrow is rebuilt larger
        (the sync-free `neighbor_list` leaves that to the caller).  Returns a list that is complete."""
        nl = self.neighbor_list(pos, cell, batch, cutoff)
        st = nl.check()
        if st[L.ST_EDGE_OVERFLOW]:
            nl = self._build_with_capacity(nl.pos, nl.cell, nl.batch, cutoff, edges_needed(st))
            st = nl.check()
            if st[L.ST_EDGE_OVERFLOW]:
                raise RuntimeError('neighbour list capacity overflow after regrow')
        return nl

    # ------------------------------------------------------------------ evaluation
    def _workspace(self, nbytes):
        if self._ws is None or self._ws.numel() < nbytes or self._ws.device != self.device:
            self._ws = torch.empty(int(nbytes * 1.05) + 256, dtype=torch.uint8, device=self.device)
        return self._ws

    def evaluate(self, nl, weights, z, want_forces=True, want_virial=False, want_nodes=False, want_direct=False):
        _require_cuda(z, 'z')
        z = z.to(torch.int64).contiguous()
        out = eval_outputs(nl.n_atoms, nl.n_systems, nl.pos.device, want_forces, want_virial, want_nodes, want_direct)
        ws = self._workspace(self.lib.nn_eval_workspace_bytes(nl.n_atoms, nl.n_systems, nl.cap_pairs, weights.n_layers,
                                                              int(want_forces or want_virial)))
        a = eval_args(nl, weights, z, out, ws, want_forces, want_virial)
        L.check(self.lib.nn_eval(C.byref(a), stream()), 'nn_eval')
        out['_z'] = z   # keep alive until the stream has consumed it
        return out

    def energy_forces(self, weights, z, pos, cell, batch, want_forces=True, want_virial=False, want_nodes=False,
                      want_direct=False):
        """Neighbour list + evaluation + status check, regrowing capacities when needed.  From the second
        call with the same shapes on, the whole step (neighbour rebuild + ~80 kernels) is replayed as one
        CUDA graph."""
        if self.use_cuda_graphs:
            key = (pos.shape[0], cell.reshape(-1, 9).shape[0], bool(want_forces), bool(want_virial), bool(want_nodes),
                   bool(want_direct), id(weights), str(pos.device))
            g = self._graphs.get(key)
            if g is not None:
                out = g.replay(z, pos, cell, batch)
                if out is not None:
                    return out
                del self._graphs[key]                         # capacity overflow: fall through, recapture later
            elif self._last_key == key and self._nl is not None and self._nl.n_atoms == pos.shape[0]:
                if len(self._graphs) >= 4:
                    self._graphs.pop(next(iter(self._graphs)))
                self._graphs[key] = GraphedStep(self, weights, z, pos, cell, batch, want_forces, want_virial, want_nodes,
                                                self._nl.cap_edges, want_direct)
                out = self._graphs[key].replay(z, pos, cell, batch)
                if out is not None:
                    return out
                del self._graphs[key]
            self._last_key = key
        nl = self.neighbor_list(pos, cell, batch, weights.cutoff)
        out = self.evaluate(nl, weights, z, want_forces, want_virial, want_nodes, want_direct)
        st = nl.check()
        if st[L.ST_EDGE_OVERFLOW]:
            nl = self._build_with_capacity(nl.pos, nl.cell, nl.batch, weights.cutoff, edges_needed(st))
            out = self.evaluate(nl, weights, z, want_forces, want_virial, want_nodes, want_direct)
            st = nl.check()
            if st[L.ST_EDGE_OVERFLOW]:
                raise RuntimeError('neighbour list capacity overflow after regrow')
        out['_nl'] = nl
        return out


class GraphedStep:
    """One evaluation (neighbour rebuild + nn_eval) captured as a CUDA graph over static buffers."""

    def __init__(self, engine, weights, z, pos, cell, batch, want_forces, want_virial, want_nodes, cap_edges,
                 want_direct=False):
        dev = pos.device
        self.engine, self.weights = engine, weights
        self.z = torch.empty(z.shape, dtype=torch.int64, device=dev)
        self.pos = torch.empty(pos.shape, dtype=torch.float32, device=dev)
        self.cell = torch.empty(cell.reshape(-1, 3, 3).shape, dtype=torch.float32, device=dev)
        self.batch = torch.empty(batch.shape, dtype=torch.int64, device=dev)
        self._copy_in(z, pos, cell, batch)
        self.nl = NeighborList(engine, self.pos, self.cell, self.batch, cap_edges=cap_edges)
        N, B = self.nl.n_atoms, self.nl.n_systems
        self.out = eval_outputs(N, B, dev, want_forces, want_virial, want_nodes, want_direct)
        nbytes = engine.lib.nn_eval_workspace_bytes(N, B, self.nl.cap_pairs, weights.n_layers, int(want_forces or want_virial))
        self.ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
        self.args = eval_args(self.nl, weights, self.z, self.out, self.ws, want_forces, want_virial)
        self.graph, _, _ = capture(self._launch, dev)

    def _launch(self):
        self.nl.rebuild(self.weights.cutoff)
        L.check(self.engine.lib.nn_eval(C.byref(self.args), stream()), 'nn_eval')

    def _copy_in(self, z, pos, cell, batch):
        self.z.copy_(z, non_blocking=True)
        self.pos.copy_(pos.detach(), non_blocking=True)
        self.cell.copy_(cell.detach().reshape(-1, 3, 3), non_blocking=True)
        self.batch.copy_(batch, non_blocking=True)

    def replay(self, z, pos, cell, batch):
        """Returns the result dict, or None when the captured capacities overflowed (caller regrows)."""
        for t, n in ((pos, 'pos'), (cell, 'cell'), (batch, 'batch'), (z, 'z')):
            _require_cuda(t, n)
        self._copy_in(z, pos, cell, batch)
        self.nl.n_edges = None
        self.nl.generation += 1
        self.graph.replay()
        out = {k: v.clone() for k, v in self.out.items()}
        st = self.nl.check()
        if st[L.ST_EDGE_OVERFLOW]:
            return None
        out['_nl'] = self.nl
        return out


_engines = {}


def get_engine(device):
    device = torch.device(device)
    if device.type == 'cuda' and device.index is None:
        device = torch.device('cuda', torch.cuda.current_device())
    key = str(device)
    if key not in _engines:
        _engines[key] = Engine(device)
    return _engines[key]

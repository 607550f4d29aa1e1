"""Multi-GPU evaluation: one process per GPU, torch.distributed (NCCL over NVLink) for the plumbing.

Two partitionings, as SURVEY.md section 8e lays out (the reference itself is single-process):

* independent molecule batches - `shard_batch` splits the systems of a batch into contiguous,
  atom-balanced ranges; every rank evaluates its range with the ordinary single-GPU path, there is no
  data-path collective (edges never cross systems, reference layers/representations.py:74-77);

* one large periodic box - `DomainDecomposition` splits space into a px x py x pz grid of bricks.  A
  rank owns the atoms inside its brick and keeps ghost copies of every atom within the cutoff of it.
  Pairs with at least one owned endpoint are evaluated locally (owned-ghost pairs on both sides, ~10 %
  redundant edge-MLP work for 50 A bricks), so every per-atom sum of an owned atom is complete locally
  and the only communication is owner -> ghost copies of per-atom feature rows, three times per
  direction: forward mn(l) [+ f(l-1)], reverse dfb(l) + abar(l).  Ghost rows are ordered by owner rank,
  so a peer's rows land contiguously: the receive side needs no unpack kernel.
  Energy, virial and forces are completed with one all-reduce each.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from .engine import NeighborList, capture, count_edges, edge_capacity, edges_needed, eval_args, get_engine, stream

GRIDS = {1: (1, 1, 1), 2: (2, 1, 1), 3: (3, 1, 1), 4: (2, 2, 1), 6: (3, 2, 1), 8: (2, 2, 2)}


# ----------------------------------------------------------------------------- molecule batches
def shard_batch(z, pos, cell, batch, rank, world):
    """Contiguous range of systems for `rank`, balanced by atom count (numpy or torch inputs).
    Returns (z, pos, cell, batch_local, system_slice) with batch re-based to start at 0."""
    b = np.asarray(batch.cpu() if torch.is_tensor(batch) else batch)
    n_sys = cell.shape[0]
    counts = np.bincount(b, minlength=n_sys)
    csum = np.concatenate([[0], np.cumsum(counts)])
    total = csum[-1]
    bounds = [int(np.searchsorted(csum, total * r / world, side='left')) for r in range(world)] + [n_sys]
    bounds[0] = 0
    for r in range(1, world + 1):
        bounds[r] = max(bounds[r], bounds[r - 1])
    s0, s1 = bounds[rank], bounds[rank + 1]
    a0, a1 = int(csum[s0]), int(csum[s1])
    return z[a0:a1], pos[a0:a1], cell[s0:s1], batch[a0:a1] - s0, slice(s0, s1)


# ----------------------------------------------------------------------------- spatial decomposition
class HaloPlan:
    """Host-side description of one rank's brick: who is owned, who is a ghost, what to send to whom."""

    def __init__(self, pos, cell, rank, world, cutoff, grid=None, skin=0.0):
        pos = np.asarray(pos, dtype=np.float64)
        cell = np.asarray(cell, dtype=np.float64).reshape(3, 3)
        if np.count_nonzero(cell - np.diag(np.diag(cell))) or np.any(np.diag(cell) <= 0):
            raise ValueError('domain decomposition needs an orthorhombic periodic cell')
        grid = tuple(grid) if grid is not None else GRIDS.get(world)
        if grid is None or int(np.prod(grid)) != world:
            raise ValueError(f'no brick grid for world size {world}')
        Ld = np.diag(cell)
        width = Ld / np.array(grid)
        halo = cutoff * 1.0001 + skin + 16 * np.finfo(np.float32).eps * np.abs(pos).max(initial=0.0)
        for d in range(3):
            if grid[d] > 1 and width[d] < halo:
                raise ValueError('bricks must be at least one cutoff wide')
        self.grid, self.rank, self.world = grid, rank, world
        frac = pos / Ld
        frac -= np.floor(frac)
        wrapped = frac * Ld
        ix = np.minimum((frac * np.array(grid)).astype(np.int64), np.array(grid) - 1)
        owner = (ix[:, 0] * grid[1] + ix[:, 1]) * grid[2] + ix[:, 2]
        self.owner = owner
        all_idx = np.arange(len(pos))

        def ghosts_of(r):
            """Atoms not owned by r within `halo` of r's brick (per-axis periodic distance)."""
            rc = np.array([r // (grid[1] * grid[2]), (r // grid[2]) % grid[1], r % grid[2]])
            lo, hi = rc * width, (rc + 1) * width
            near = np.ones(len(pos), dtype=bool)
            for d in range(3):
                if grid[d] == 1:
                    continue
                x = wrapped[:, d]
                below = np.minimum(np.abs(lo[d] - x), Ld[d] - np.abs(lo[d] - x))
                above = np.minimum(np.abs(x - hi[d]), Ld[d] - np.abs(x - hi[d]))
                inside = (x >= lo[d]) & (x < hi[d])
                near &= inside | (np.minimum(below, above) <= halo)
            g = all_idx[near & (owner != r)]
            return g[np.lexsort((g, owner[g]))]            # grouped by owner rank, ascending global index

        self.owned = all_idx[owner == rank]
        self.ghost = ghosts_of(rank)
        self.n_owned, self.n_ghost = len(self.owned), len(self.ghost)
        self.local_to_global = np.concatenate([self.owned, self.ghost])
        g_owner = owner[self.ghost]
        self.recv_counts = [int((g_owner == r).sum()) for r in range(world)]
        # rows this rank sends: its owned atoms that are ghosts of peer s, in s's ghost order
        local_of = -np.ones(len(pos), dtype=np.int64)
        local_of[self.owned] = np.arange(self.n_owned)
        send = []
        self.send_counts = []
        self.send_row_offset = []        # first row of this rank's block in peer s's ghost order
        for s in range(world):
            if s == rank:
                self.send_counts.append(0)
                self.send_row_offset.append(0)
                continue
            gs = ghosts_of(s)
            mine = gs[owner[gs] == rank]
            send.append(local_of[mine])
            self.send_counts.append(len(mine))
            self.send_row_offset.append(int((owner[gs] < rank).sum()))
        self.send_index = np.concatenate(send).astype(np.int32) if send else np.zeros(0, np.int32)


class HaloExchange:
    """Owner -> ghost copy of per-atom rows: pack kernel + all_to_all_single into the ghost tail."""

    def __init__(self, plan, device, group=None):
        self.plan, self.group = plan, group
        self.device = torch.device(device)
        self.send_index = torch.from_numpy(plan.send_index).to(self.device)
        self.n_send = int(plan.send_index.shape[0])
        self._buf = {}

    def _pack(self, rows, width):
        key = width
        buf = self._buf.get(key)
        if buf is None or buf.shape[0] < self.n_send:
            buf = torch.empty(max(self.n_send, 1), width, dtype=torch.float32, device=self.device)
            self._buf[key] = buf
        out = buf[:self.n_send]
        if self.n_send == 0:
            return out
        if rows.is_cuda:
            L.check(L.load().nn_halo_pack(rows.data_ptr(), self.send_index.data_ptr(), self.n_send, width,
                                          out.data_ptr(), stream()), 'nn_halo_pack')
        else:   # host tensors: used only by the gloo tests of the plan / exchange logic
            torch.index_select(rows, 0, self.send_index.long(), out=out)
        return out

    def exchange(self, rows):
        """rows: [n_local, width] float32 (contiguous); ghost rows [n_owned:] are overwritten."""
        p = self.plan
        if p.world == 1:
            return
        width = rows.shape[1]
        send = self._pack(rows, width)
        recv = rows[p.n_owned:]
        if dist.get_backend(self.group) == 'nccl':
            dist.all_to_all_single(recv, send, output_split_sizes=p.recv_counts, input_split_sizes=p.send_counts,
                                   group=self.group)
        else:
            ops, so, ro = [], 0, 0
            for r in range(p.world):
                if p.send_counts[r]:
                    ops.append(dist.P2POp(dist.isend, send[so:so + p.send_counts[r]], r, group=self.group))
                if p.recv_counts[r]:
                    ops.append(dist.P2POp(dist.irecv, recv[ro:ro + p.recv_counts[r]], r, group=self.group))
                so += p.send_counts[r]; ro += p.recv_counts[r]
            for req in (dist.batch_isend_irecv(ops) if ops else []):
                req.wait()


class PeerArena:
    """One cudaMalloc arena per rank that every peer maps through CUDA IPC (csrc/p2p.cu): landing buffers of the
    two exchange channels, flag words, the complete force array, the table of per-rank partial sums.  Collective:
    every rank of the group constructs it at the same time."""

    def __init__(self, plan, n_atoms_total, device, group, strides):
        self.plan, self.group, self.device = plan, group, torch.device(device)
        self.lib = L.load()
        self.rank, self.world = plan.rank, plan.world
        self.n_atoms_total = int(n_atoms_total)
        if not 2 <= self.world <= L.DD_MAX_RANKS:
            raise ValueError(f'peer-memory transport supports 2..{L.DD_MAX_RANKS} ranks')
        al = lambda n: (int(n) + 255) // 256 * 256
        # room for the ghost count to grow: a later plan of the same box (atoms drift, the ghost shell is re-cut) reuses
        # the arena and its IPC mappings (`rebind`) instead of paying cudaMalloc + handle exchange + mapping again
        self.ghost_cap = int(plan.n_ghost * 1.25) + 1024
        landing = al(self.ghost_cap * L.DD_MAX_WIDTH * 4)
        off, cur = {}, 0
        for ch in range(L.DD_CHANNELS):
            for par in range(2):
                off['landing', ch, par] = cur; cur += landing
        off['forces'] = cur; cur += al(n_atoms_total * 12)
        off['partials'] = cur; cur += al(self.world * L.DD_PARTIAL * 4)
        for ch in range(L.DD_CHANNELS):
            off['flags', ch] = cur; cur += al(self.world * 4)
        self.nbytes = cur
        p = C.c_void_p()
        L.check(self.lib.nn_p2p_alloc(cur, C.byref(p)), 'nn_p2p_alloc')
        self.base = p.value
        h = C.create_string_buffer(64)
        L.check(self.lib.nn_p2p_get_handle(self.base, h), 'nn_p2p_get_handle')
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (h.raw, off), group=group)
        self.opened = {}
        for s in range(self.world):
            if s == self.rank:
                continue
            q = C.c_void_p()
            L.check(self.lib.nn_p2p_open_handle(C.create_string_buffer(gathered[s][0], 64), C.byref(q)), 'nn_p2p_open_handle')
            self.opened[s] = q.value
        i32 = dict(dtype=torch.int32, device=self.device)
        self.send_index = torch.from_numpy(plan.send_index).to(self.device)
        self.step = torch.zeros(1, **i32)
        self.done = torch.zeros(L.DD_CHANNELS, **i32)
        self.status = torch.zeros(L.DD_STATUS_WORDS, **i32)
        c = L.DDComm()
        c.world, c.rank, c.n_atoms_total = self.world, self.rank, int(n_atoms_total)
        c.n_owned, c.n_ghost = plan.n_owned, plan.n_ghost
        for ch in range(L.DD_CHANNELS):
            c.stride[ch] = int(strides[ch])
            c.flags[ch] = self.base + off['flags', ch]
            for par in range(2):
                c.landing[ch][par] = self.base + off['landing', ch, par]
        c.forces_full = self.base + off['forces']
        c.partials = self.base + off['partials']
        for s in range(self.world):
            if s == self.rank:
                continue
            o = gathered[s][1]
            for ch in range(L.DD_CHANNELS):
                c.peer_flags[ch][s] = self.opened[s] + o['flags', ch]
                for par in range(2):
                    c.peer_landing[ch][par][s] = self.opened[s] + o['landing', ch, par]
            c.peer_forces_full[s] = self.opened[s] + o['forces']
            c.peer_partials[s] = self.opened[s] + o['partials']
        c.step, c.done, c.status = self.step.data_ptr(), self.done.data_ptr(), self.status.data_ptr()
        self.comm = c
        self._bind_plan(plan)
        dist.barrier(group=group)

    def _bind_plan(self, plan):
        c = self.comm
        self.plan = plan
        self.send_index = torch.from_numpy(plan.send_index).to(self.device)
        c.n_owned, c.n_ghost = plan.n_owned, plan.n_ghost
        begin = 0
        for s in range(self.world):
            c.send_begin[s] = begin
            begin += plan.send_counts[s]
            c.send_end[s] = begin
            c.row_offset[s] = plan.send_row_offset[s]
        c.send_idx = self.send_index.data_ptr()

    def fits(self, plan, n_atoms_total):
        return plan.n_ghost <= self.ghost_cap and int(n_atoms_total) == self.n_atoms_total and plan.world == self.world

    def rebind(self, plan):
        """Adopt a new brick / ghost plan of the same box (same ranks, same arena, same peer mappings).  Every rank does this
        after the same step (the stale flag is OR-ed over ranks), and a rank can only have finished that step after all
        its peers consumed what it sent, so nobody still reads landing data of the old plan.  The sticky status words are
        cleared; the step counter and the flag epochs keep running."""
        torch.cuda.synchronize(self.device)
        self.status.zero_()
        self._bind_plan(plan)

    def close(self):
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        for q in self.opened.values():
            self.lib.nn_p2p_close_handle(q)
        if self.base:
            self.lib.nn_p2p_free(self.base)
        self.opened, self.base = {}, None


class _PeerStep:
    """One decomposed evaluation over static buffers: launched eagerly the first time, then captured and replayed
    as ONE CUDA graph (two streams: halo exchanges off the critical path run on the side stream)."""

    HEADROOM = (1.08, 64)          # both capacities: factor and slack over the trial fill's edge and pair counts

    def __init__(self, dd, z, pos, cell3, want_virial, reuse=None):
        """reuse: the step object of the previous plan of the same box - its arena (peer mappings) and its neighbour-list
        capacities are taken over when they fit, and the first call is captured right away (every kernel has run before)."""
        self.dd = dd
        dev = pos.device
        self.device = dev
        model = dd.model
        self.engine = get_engine(dev)
        self.lib = self.engine.lib
        self.pack = model._weight_pack(dev)
        self.want_virial = bool(want_virial)
        N = pos.shape[0]
        self.N = N
        cutoff = self.pack.cutoff
        plan = HaloPlan(pos.detach().cpu().numpy(), cell3[0].detach().cpu().numpy(), dd.rank, dd.world, cutoff, dd.grid,
                        skin=dd.skin)
        self.plan = plan
        nL = self.pack.n_layers
        self.strides = (2 * nL + 1, max(2 * nL - 1, 1))
        fits = reuse is not None and reuse.arena is not None and reuse.arena.fits(plan, N) and reuse.strides == self.strides
        if dd.world > 1:      # the same decision on every rank (a collective constructor must not be entered by some ranks only)
            flag = torch.tensor([0.0 if fits else 1.0], device=dev)
            dist.all_reduce(flag, group=dd.group)
            fits = bool(flag.item() == 0)
        if fits:
            self.arena = reuse.arena
            reuse.arena = None                   # ownership moves here
            self.arena.rebind(plan)
        else:
            if reuse is not None:
                reuse.close()
            self.arena = PeerArena(plan, N, dev, dd.group, self.strides)
        f32 = dict(dtype=torch.float32, device=dev)
        self.n_local, self.n_owned = len(plan.local_to_global), plan.n_owned
        self.l2g = torch.from_numpy(plan.local_to_global.astype(np.int32)).to(dev)
        # static inputs (graph replays read these) and the plan's reference state
        self.z_in = z.to(torch.int64).contiguous().clone()
        self.pos_in = pos.detach().to(torch.float32).contiguous().clone()
        self.cell_in = cell3.detach().to(torch.float32).contiguous().clone()
        self.pos_ref = self.pos_in.clone()
        self.cell_ref = self.cell_in.clone()
        self.z_l = self.z_in[self.l2g.long()].contiguous()
        self.pos_l = self.pos_in[self.l2g.long()].contiguous()
        self.batch_l = torch.zeros(self.n_local, dtype=torch.int64, device=dev)
        # outputs
        self.energy = torch.zeros(1, **f32); self.forces_l = torch.zeros(max(self.n_owned, 1), 3, **f32)
        self.virial = torch.zeros(1, 3, 3, **f32); self.stress = torch.zeros(1, 3, 3, **f32)
        self.forces_out = torch.zeros(N, 3, **f32)
        self.small = torch.zeros(19, **f32)
        self.out_status = torch.zeros(L.DD_STATUS_WORDS, dtype=torch.int32, device=dev)
        self.side = torch.cuda.Stream(device=dev)
        self.graph = None
        self.calls = 0
        self.stale = False
        self.nl = None
        if fits and reuse.nl is not None:
            # capacities of the previous plan, scaled by the change of the owned count, plus headroom (an overflow is caught by
            # the status words like any other)
            g = max(1.0, self.n_owned / max(reuse.n_owned, 1)) * 1.02
            self._bind_list(edge_capacity(reuse.nl.cap_edges, g, 64), int(reuse.nl.cap_pairs * g) + 64)
            self.calls = 1               # no eager first step: capture immediately
        else:
            self._size_neighbor_list()

    # ---- capacities
    def _new_list(self, cap_edges, cap_pairs):
        return NeighborList(self.engine, self.pos_l, self.cell_in, self.batch_l, cap_edges, cap_pairs, self.n_owned)

    def _size_neighbor_list(self, needed=0):
        """Probe: count (-> directed edges of the owned rows), then a trial fill with room for one pair per edge (ghost rows
        are empty, so an owned-ghost pair has a single directed edge and P lies between E / 2 and E) -> final capacities."""
        probe = count_edges(self.engine, self.pos_l, self.cell_in, self.batch_l, self.pack.cutoff, self.n_owned)
        n_edges = max(probe.n_edges, needed)
        probe = self._new_list(n_edges + 2, n_edges + 2)
        probe.rebuild(self.pack.cutoff)
        st = probe.check()
        del probe
        factor, slack = self.HEADROOM
        self._bind_list(edge_capacity(st[L.ST_N_EDGES], factor, slack), int(st[L.ST_N_PAIRS] * factor) + slack)

    def _bind_list(self, cap_edges, cap_pairs):
        self.nl = self._new_list(cap_edges, cap_pairs)
        nbytes = self.lib.nn_eval_workspace_bytes(self.n_local, 1, self.nl.cap_pairs, self.pack.n_layers, 1)
        self.ws = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=self.device)
        out = {'energy': self.energy, 'forces': self.forces_l}
        if self.want_virial:
            out.update(virial=self.virial, stress=self.stress)
        self.args = eval_args(self.nl, self.pack, self.z_l, out, self.ws, True, self.want_virial, self.n_owned)
        self.graph = None
        self.calls = 0

    # ---- one step on the current stream (+ side stream)
    def _launch(self):
        lib, a, comm = self.lib, self.args, C.byref(self.arena.comm)
        main = torch.cuda.current_stream()
        side = self.side if self.dd.overlap else main
        s = main.cuda_stream
        nL, F = self.pack.n_layers, L.NN_F
        n_owned = self.n_owned
        ghost = lambda which, l, width: lib.nn_eval_buffer(C.byref(a), which, l) + n_owned * width * 4
        rows = lambda which, l: lib.nn_eval_buffer(C.byref(a), which, l)

        def phase(ph, l=0):
            L.check(lib.nn_eval_phase(C.byref(a), ph, l, s), f'nn_eval_phase({ph},{l})')

        seq = [0, 0]

        def exchange(stream, ch, which, l, width):
            st = stream.cuda_stream
            L.check(lib.nn_dd_halo_push(comm, ch, seq[ch], rows(which, l), width, st), 'nn_dd_halo_push')
            L.check(lib.nn_dd_halo_wait(comm, ch, seq[ch], ghost(which, l, width), width, st), 'nn_dd_halo_wait')
            seq[ch] += 1

        def fork():          # side stream continues from here
            if side is not main:
                side.wait_stream(main)

        def join():
            if side is not main:
                main.wait_stream(side)

        L.check(lib.nn_dd_begin(comm, self.pos_in.data_ptr(), self.pos_ref.data_ptr(), self.cell_in.data_ptr(),
                                self.cell_ref.data_ptr(), self.z_in.data_ptr(), self.l2g.data_ptr(), self.n_local,
                                self.dd.skin, self.pos_l.data_ptr(), self.z_l.data_ptr(), s), 'nn_dd_begin')
        self.nl.rebuild(self.pack.cutoff)
        phase(L.PH_BEGIN)
        pending = False
        for l in range(nL):
            phase(L.PH_FWD_NODE, l)
            exchange(main, 0, L.BUF_MN, l, F)
            if pending:
                join(); pending = False
            phase(L.PH_FWD_PAIR_A, l)
            if l + 1 < nL:           # f_out(l) is needed by the NEXT layer's pair phase only: exchange it behind FWD_PAIR_B / FWD_NODE
                fork()
                exchange(side, 1, L.BUF_F_OUT, l, 3 * F)
                pending = True
            phase(L.PH_FWD_PAIR_B, l)
        phase(L.PH_HEAD)
        phase(L.PH_BWD_SEED)
        for l in reversed(range(nL)):
            phase(L.PH_BWD_NORM, l)
            fork()                   # abar(l) is final here and needed by BWD_PAIR_B only
            exchange(side, 1, L.BUF_ABAR, 0, F)
            phase(L.PH_BWD_NODE_B, l)
            exchange(main, 0, L.BUF_DFB, 0, 3 * F)
            phase(L.PH_BWD_PAIR_A, l)
            join()
            phase(L.PH_BWD_PAIR_B, l)
        phase(L.PH_FINISH)
        assert seq[0] == self.strides[0] - 1 and seq[1] == self.strides[1], (seq, self.strides)
        L.check(lib.nn_dd_finish(comm, seq[0], self.forces_l.data_ptr(), self.l2g.data_ptr(), self.energy.data_ptr(),
                                 self.virial.data_ptr() if self.want_virial else None,
                                 self.stress.data_ptr() if self.want_virial else None, self.nl.status.data_ptr(),
                                 self.forces_out.data_ptr(), self.small.data_ptr(), self.out_status.data_ptr(), s), 'nn_dd_finish')

    def run(self, z, pos, cell3):
        self.z_in.copy_(z, non_blocking=True)
        self.pos_in.copy_(pos.detach(), non_blocking=True)
        self.cell_in.copy_(cell3.detach(), non_blocking=True)
        self.calls += 1
        if self.calls == 1 or not self.dd.use_cuda_graph:
            self._launch()
            return
        if self.graph is None:
            self.graph, _, _ = capture(self._launch, self.device)
        self.graph.replay()

    def status(self):
        """Status words of the last step (one small D2H copy, synchronises); raises when a peer timed out or a rank's
        inputs broke its neighbour list."""
        st = self.out_status.cpu().tolist()
        if st[L.DD_ST_TIMEOUT]:
            raise RuntimeError('halo exchange timed out waiting for a peer rank')
        if st[L.DD_ST_BAD_INPUT]:
            self.nl.check()
            raise RuntimeError('neighbour list failure on a peer rank (degree overflow / singular cell)')
        return st

    def halo_bytes_per_step(self):
        """Bytes this rank stores into peer memory per step (feature rows + forces), and the number of exchanges."""
        F, nL = L.NN_F, self.pack.n_layers
        n_send = int(self.plan.send_index.shape[0])
        rows = n_send * 4 * F * (nL + 3 * (nL - 1) + nL + 3 * nL)
        return rows + (self.plan.world - 1) * self.n_owned * 12, self.strides[0] + self.strides[1]

    def close(self):
        self.graph = None
        if self.arena is not None:
            self.arena.close()
            self.arena = None


class DomainDecomposition:
    """Energy / forces / stress of ONE periodic box across the ranks of a process group.

    dd = DomainDecomposition(model); out = dd(z, pos, cell)   (same full inputs on every rank)
    -> CustomOutputSet with energy [1], gradient_force [N,3] (complete on every rank), stress, virial.
    """

    HEADROOM = (1.08, 64)          # eager path's edge capacity: factor and slack over the counted edges

    def __init__(self, model, group=None, grid=None, skin=1.0, transport='p2p', overlap=True, use_cuda_graph=True):
        """skin (A): the brick/ghost plan is kept while no atom has moved more than skin/2 since it was
        made (the ghost shell is cutoff + skin thick); the neighbour list itself is rebuilt every call.
        transport: 'p2p' = the whole step is one CUDA graph, halo rows and results travel as stores into peer
        memory over NVLink (csrc/p2p.cu); 'nccl' = eager phases, pack kernel + all_to_all_single + all-reduce.
        overlap: exchange f_out / abar rows on a second stream behind the node-level work."""
        self.model, self.group, self.grid, self.skin = model, group, grid, float(skin)
        self.transport = transport
        self.overlap, self.use_cuda_graph = bool(overlap), bool(use_cuda_graph)
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.plan = None
        self._ws = None
        self._nl = None
        self._state = None
        self._peer = None
        self.n_plans = 0

    # ------------------------------------------------------------------ peer-memory path (CUDA graph)
    def _use_peer(self):
        return self.transport == 'p2p' and self.world > 1 and dist.get_backend(self.group) == 'nccl'

    def check(self):
        """Read the status of the last step (one small D2H copy, synchronises).  Returns the status words;
        raises on conditions that invalidate the result.  `__call__(..., sync=True)` does this itself."""
        st = self._peer.status()
        if st[L.DD_ST_STALE]:
            raise RuntimeError('an atom moved more than skin/2 since the brick/ghost plan was made and the step ran with '
                               'sync=False: call with sync=True (replans automatically) or increase skin')
        if st[L.DD_ST_OVERFLOW]:
            raise RuntimeError('neighbour-list capacity overflow in a step run with sync=False')
        return st

    def _call_peer(self, z, pos, cell, want_virial, sync):
        from newtonnet_b200.models.output import CustomOutputSet
        cell3 = cell.reshape(-1, 3, 3)
        N = pos.shape[0]
        for attempt in range(4):
            p = self._peer
            if p is None or p.N != N or p.want_virial != bool(want_virial) or p.stale:
                same_box = p is not None and p.N == N and p.want_virial == bool(want_virial)
                if p is not None and not same_box:
                    p.close()
                p = self._peer = _PeerStep(self, z, pos, cell3, want_virial, reuse=p if same_box else None)
                self.plan = p.plan
                self.n_plans += 1
            p.run(z, pos, cell3)
            if not sync:
                break
            st = p.status()                             # the one host synchronisation of the step
            if st[L.DD_ST_STALE]:                        # same decision on every rank: the flags were OR-ed by nn_dd_finish
                p.stale = True                           # re-cut the bricks for the new positions, keep arena and capacities
                continue
            if st[L.DD_ST_OVERFLOW]:
                p._size_neighbor_list(edges_needed(p.nl.status.cpu().tolist()))
                continue
            break
        else:
            raise RuntimeError('domain decomposition did not converge (plan / capacity kept changing)')
        dt = pos.dtype
        out = CustomOutputSet(z=z, pos=pos, cell=cell, batch=torch.zeros(N, dtype=torch.int64, device=pos.device))
        small = p.small.clone()
        out.energy = small[:1].to(dt)
        out.gradient_force = p.forces_out.clone().to(dt)
        out.virial = small[1:10].reshape(1, 3, 3).to(dt)
        out.stress = small[10:19].reshape(1, 3, 3).to(dt)
        out.n_owned, out.n_ghost = p.n_owned, p.plan.n_ghost
        return out

    def close(self):
        if self._peer is not None:
            self._peer.close()
            self._peer = None

    # ------------------------------------------------------------------ eager path (NCCL / gloo collectives)
    def _workspace(self, nbytes, device):
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(int(nbytes * 1.05) + 256, dtype=torch.uint8, device=device)
        return self._ws

    def _view(self, ws, ptr, rows, width):
        off = ptr - ws.data_ptr()
        return ws[off:off + rows * width * 4].view(torch.float32).view(rows, width)

    def _replan(self, z, pos, cell3, cutoff, dev):
        plan = HaloPlan(pos.detach().cpu().numpy(), cell3[0].detach().cpu().numpy(), self.rank, self.world,
                        cutoff, self.grid, skin=self.skin)
        self.plan = plan
        self.n_plans += 1
        l2g = torch.from_numpy(plan.local_to_global).to(dev)
        halo = HaloExchange(plan, dev, self.group)
        self._state = dict(l2g=l2g, halo=halo, pos_ref=pos.detach().clone(),
                           z_l=z.to(torch.int64)[l2g].contiguous(), n=pos.shape[0],
                           batch_l=torch.zeros(len(plan.local_to_global), dtype=torch.int64, device=dev))
        self._nl = None

    def __call__(self, z, pos, cell, want_virial=True, sync=True):
        """sync=False (peer-memory transport only): no host synchronisation at all - the caller checks a batch of
        steps afterwards with `check()`; a stale plan or a capacity overflow then raises instead of being repaired."""
        if self._use_peer():
            if cell.reshape(-1, 3, 3).shape[0] != 1:
                raise ValueError('DomainDecomposition evaluates one periodic system')
            return self._call_peer(z, pos, cell, want_virial, sync)
        return self._call_eager(z, pos, cell, want_virial)

    def _call_eager(self, z, pos, cell, want_virial=True):
        from newtonnet_b200.models.output import CustomOutputSet
        model = self.model
        dev = pos.device
        engine = get_engine(dev)
        lib = engine.lib
        pack = model._weight_pack(dev)
        N = pos.shape[0]
        cell3 = cell.reshape(-1, 3, 3)
        if cell3.shape[0] != 1:
            raise ValueError('DomainDecomposition evaluates one periodic system')
        st = self._state
        stale = st is None or st['n'] != N
        if not stale:   # one scalar read-back decides whether the cached plan still covers the cutoff
            moved = float((pos.detach() - st['pos_ref']).square().sum(1).max().sqrt())
            flag = torch.tensor([1.0 if moved > 0.5 * self.skin else 0.0], device=dev)
            if self.world > 1:
                dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=self.group)
            stale = bool(flag.item() > 0)
        if stale:
            self._replan(z, pos, cell3, pack.cutoff, dev)
            st = self._state
        plan, halo, l2g, z_l, batch_l = self.plan, st['halo'], st['l2g'], st['z_l'], st['batch_l']
        pos_l = pos.detach().to(torch.float32)[l2g].contiguous()
        cell_l = cell3.detach().to(torch.float32).contiguous()
        n_local, n_owned = int(l2g.shape[0]), plan.n_owned
        s = stream()

        # ---- neighbour list over owned + ghost atoms (ghost-ghost pairs dropped); capacities are kept
        if self._nl is None:
            cap = edge_capacity(count_edges(engine, pos_l, cell_l, batch_l, pack.cutoff, n_owned).n_edges, *self.HEADROOM)
            # ghost rows of the list stay empty, so an owned-ghost pair has ONE directed edge: up to one pair per edge
            self._nl = NeighborList(engine, pos_l, cell_l, batch_l, cap, cap, n_owned)
        nl = self._nl
        nl.rebind(pos_l, cell_l, batch_l)
        nl.rebuild(pack.cutoff)
        n_layers = pack.n_layers

        # ---- phased evaluation with halo exchanges
        f32 = dict(dtype=torch.float32, device=dev)
        energy = torch.zeros(1, **f32); forces_l = torch.zeros(max(n_owned, 1), 3, **f32)
        virial = torch.zeros(1, 3, 3, **f32); stress = torch.zeros(1, 3, 3, **f32)
        ws = self._workspace(lib.nn_eval_workspace_bytes(n_local, 1, nl.cap_pairs, n_layers, 1), dev)
        outputs = {'energy': energy, 'forces': forces_l}
        if want_virial:
            outputs.update(virial=virial, stress=stress)
        a = eval_args(nl, pack, z_l, outputs, ws, True, want_virial, n_owned)

        def phase(ph, l=0):
            L.check(lib.nn_eval_phase(C.byref(a), ph, l, s), f'nn_eval_phase({ph},{l})')

        def buf(which, l, width):
            return self._view(ws, lib.nn_eval_buffer(C.byref(a), which, l), n_local, width)

        phase(L.PH_BEGIN)
        for l in range(n_layers):
            phase(L.PH_FWD_NODE, l)
            halo.exchange(buf(L.BUF_MN, l, L.NN_F))
            if l > 0:
                halo.exchange(buf(L.BUF_F_OUT, l - 1, 3 * L.NN_F))
            phase(L.PH_FWD_PAIR, l)
        phase(L.PH_HEAD)
        phase(L.PH_BWD_SEED)
        for l in reversed(range(n_layers)):
            phase(L.PH_BWD_NODE, l)
            halo.exchange(buf(L.BUF_DFB, 0, 3 * L.NN_F))
            halo.exchange(buf(L.BUF_ABAR, 0, L.NN_F))
            phase(L.PH_BWD_PAIR, l)
        phase(L.PH_FINISH)

        # ---- complete the sums across ranks: ONE all-reduce of [forces | energy, virial, stress (hi, lo) | flags]
        status_dev = nl.status.to(torch.float32)
        small = torch.cat([energy.double(), virial.double().reshape(-1), stress.double().reshape(-1)])
        hi = small.float()
        lo = (small - hi.double()).float()                       # fp64 partial sums travel as two fp32 parts
        over_flag = (status_dev[L.ST_EDGE_OVERFLOW:L.ST_EDGE_OVERFLOW + 1] != 0).float()
        buf = torch.zeros(3 * N + 2 * 19 + 1, **f32)
        buf[:3 * N].view(N, 3)[l2g[:n_owned]] = forces_l[:n_owned]
        buf[3 * N:3 * N + 19] = hi
        buf[3 * N + 19:3 * N + 38] = lo
        buf[3 * N + 38:] = over_flag
        if self.world > 1:
            dist.all_reduce(buf, group=self.group)
        forces = buf[:3 * N].view(N, 3)
        tail = buf[3 * N:].cpu()                                  # the one host synchronisation of the step
        red = tail[:19].double() + tail[19:38].double()
        status = nl.check()
        if float(tail[38]) > 0:      # some rank's list outgrew its capacity: resize everywhere and repeat
            self._nl = None
            return self._call_eager(z, pos, cell, want_virial)
        dt = pos.dtype
        out = CustomOutputSet(z=z, pos=pos, cell=cell, batch=torch.zeros(N, dtype=torch.int64, device=dev))
        red = red.to(dev)
        out.energy = red[:1].to(dt)
        out.gradient_force = forces.to(dt)
        out.virial = red[1:10].reshape(1, 3, 3).to(dt)
        out.stress = red[10:19].reshape(1, 3, 3).to(dt)
        out.n_owned, out.n_ghost, out.n_local_edges = n_owned, plan.n_ghost, status[L.ST_N_EDGES]
        out._keep = (nl, z_l, pos_l, cell_l, batch_l, halo)
        return out

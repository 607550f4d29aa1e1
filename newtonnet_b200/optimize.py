"""Device-resident geometry optimisation: ASE's FIRE for every system of a batch at once.

Relaxing structures through ASE runs on the host, one Atoms at a time: every step calls
MLAseCalculator.calculate (utils/ase_interface.py:52-81: numpy -> H2D -> forward -> D2H -> numpy) and then the
optimiser's numpy step.  `DeviceFIRE` keeps positions, FIRE velocities, forces and each system's FIRE state in HBM and
replays one CUDA graph per step (nn_fire_step -> neighbour rebuild -> nn_eval -> nn_fire_check); the host enqueues
graph launches and reads the status and the converged flags once per `check_interval` steps.

The step is `ase.optimize.FIRE.step` (ASE 3.22 / 3.23, downhill_check=False) run independently per system, with ASE's
parameter names and defaults; convergence is `Optimizer.converged` (max_i |f_i|^2 < fmax^2) checked before every step,
and a converged system is frozen.  oracle/opt_oracle.py restates both in numpy.  Relaxations have long tails: once the
unconverged systems hold at most half of the graph's atoms they are gathered into a smaller graph (`compaction_plan`).
"""
import types

import numpy as np
import torch

from newtonnet_b200 import _lib as L
from newtonnet_b200.engine import capture, count_edges, driver_inputs, force_step, replay_chunk, stream
from newtonnet_b200.md import atoms_cell

__all__ = ['DeviceFIRE', 'compaction_plan']

# per-system state columns (csrc/md_ops.cu): sf [B,3] fp64, si [B,4] int32
DT, A, F2 = 0, 1, 2
NSTEPS, STARTED, CONVERGED, STEPS = 0, 1, 2, 3


def segment_rows(ptr, sel):
    """Row indices of segments `sel` (ascending) of an array cut at offsets `ptr`: rows [ptr[s], ptr[s+1]) of every s in
    sel, in order.  The rows a step graph gathers for the systems it keeps."""
    ptr, sel = np.asarray(ptr, dtype=np.int64), np.asarray(sel, dtype=np.int64)
    n = ptr[sel + 1] - ptr[sel]
    return np.repeat(ptr[sel], n) + np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n)


def gather_state(w, master, index, keys):
    """w.<key> = master[key][index] as a fresh contiguous tensor, for every key."""
    for k in keys:
        setattr(w, k, master[k][index].contiguous())


def scatter_state(master, w, index, keys):
    """master[key][index] = w.<key>, for every key: the inverse of gather_state."""
    for k in keys:
        master[k].index_copy_(0, index, getattr(w, k))


def fixed_mask(atoms, who):
    """[len(atoms)] bool: the atoms FixAtoms-like constraints (any object with get_indices()) hold in place.  Any other
    constraint raises NotImplementedError."""
    f = np.zeros(len(atoms), dtype=bool)
    for c in getattr(atoms, 'constraints', None) or ():
        if not hasattr(c, 'get_indices'):
            raise NotImplementedError(f'{who} supports FixAtoms-like constraints only, not {type(c).__name__}')
        f[np.asarray(c.get_indices(), dtype=np.int64)] = True
    return f


def compaction_plan(active, n_atoms):
    """Which systems a relaxation keeps in its step graph at a chunk boundary.  active: bool [S], the systems of the
    graph's batch that have not converged; n_atoms: [S] atoms per system.  Returns None while the active systems hold
    more than half of the graph's atoms (or there are none), else (keep: [K] indices of the active systems in batch
    order, batch: [n_atoms[keep].sum()] their atoms' system ids 0..K-1 in the smaller graph)."""
    active = np.asarray(active, dtype=bool)
    n = np.asarray(n_atoms, dtype=np.int64)
    if not active.any() or 2 * int(n[active].sum()) > int(n.sum()):
        return None
    keep = np.flatnonzero(active)
    return keep, np.repeat(np.arange(len(keep)), n[keep])


class DeviceFIRE:
    """FIRE relaxation at fixed cell of one system or a batch of independent systems, state resident on the GPU.

    model: newtonnet_b200 NewtonNet (CUDA, energy head); z [N]; pos [N,3] (Angstrom); cell [B,3,3] or None (not
    periodic); batch [N] or None (one system); fixed [N] bool or None: atoms held in place, as ASE's FixAtoms (their
    forces are zero in the step, the convergence test and `forces`).  dt ... a: ASE's FIRE parameters, per system.
    check_interval: steps replayed between two reads of the status and the converged flags."""

    HEADROOM = (1.15, 64)          # edge capacity: factor and slack over the counted edges

    def __init__(self, model, z, pos, cell=None, batch=None, fixed=None, dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1,
                 fdec=0.5, astart=0.1, fa=0.99, a=0.1, check_interval=16):
        self.lib = L.load()
        self.model = model
        dev, self.engine, self.weights, as_t, z, x, batch, cell = driver_inputs(model, z, pos, cell, batch, 'DeviceFIRE')
        self.device = dev
        N, B = z.shape[0], cell.shape[0]
        self.n_atoms, self.n_systems = N, B
        self.params = (float(maxstep), float(dtmax), float(finc), float(fdec), float(astart), float(fa), int(Nmin))
        self.check_interval = max(1, int(check_interval))
        self.sys_atoms = torch.bincount(batch, minlength=B).cpu().numpy()
        self.sys_ptr = np.concatenate([[0], np.cumsum(self.sys_atoms)])
        f64, f32 = dict(dtype=torch.float64, device=dev), dict(dtype=torch.float32, device=dev)
        sf = torch.zeros(B, 3, **f64)
        sf[:, DT], sf[:, A] = float(dt), float(a)
        # state of every system; the step graph works on a gathered copy of some of them (`_use`)
        self.master = dict(z=z, x=x, v=torch.zeros(N, 3, **f64), force=torch.zeros(N, 3, **f32), energy=torch.zeros(B, **f32),
                           cell=cell, sf=sf, si=torch.zeros(B, 4, dtype=torch.int32, device=dev),
                           fixed=torch.zeros(N, dtype=torch.bool, device=dev) if fixed is None else as_t(fixed, torch.bool).reshape(N))
        self.fmax2 = torch.zeros(1, **f64)
        self.graph_launches = 0        # step graph replays, rolled-back chunks included
        self.compactions = 0
        self.work = None
        self._use(np.arange(B), batch.cpu().numpy())     # evaluates the input positions
        self._scatter()

    # ------------------------------------------------------------------ construction helpers
    @staticmethod
    def _atoms_list(atoms):
        return [atoms] if hasattr(atoms, 'get_atomic_numbers') else list(atoms)

    @classmethod
    def from_atoms(cls, atoms, calc, **kwargs):
        """From one ASE-like Atoms or a list (one system each) and an MLAseCalculator.  FixAtoms-like constraints (any
        object with get_indices()) become `fixed`; any other constraint raises NotImplementedError."""
        atoms_list = cls._atoms_list(atoms)
        fixed = [fixed_mask(at, 'DeviceFIRE') for at in atoms_list]
        kw = dict(kwargs)
        if any(f.any() for f in fixed):
            kw.setdefault('fixed', np.concatenate(fixed))
        return cls(calc.model, np.concatenate([at.get_atomic_numbers() for at in atoms_list]),
                   np.concatenate([at.get_positions() for at in atoms_list]), np.stack([atoms_cell(at) for at in atoms_list]),
                   np.repeat(np.arange(len(atoms_list)), [len(at) for at in atoms_list]), **kw)

    def update_atoms(self, atoms):
        """Write the current positions into the Atoms (or list of Atoms) the optimiser was built from."""
        x = self.positions
        for b, at in enumerate(self._atoms_list(atoms)):
            at.set_positions(x[self.sys_ptr[b]:self.sys_ptr[b + 1]])
        return atoms

    # ------------------------------------------------------------------ the step graph
    def _use(self, sel, batch):
        """Point the step graph at master systems `sel` (ascending) with atom system ids `batch`: gather their state into
        fresh buffers, evaluate and capture."""
        m, dev = self.master, self.device
        atoms = segment_rows(self.sys_ptr, sel)
        ai, si = torch.as_tensor(atoms, device=dev), torch.as_tensor(sel, device=dev)
        w = types.SimpleNamespace(sel=np.asarray(sel), sys_atoms=self.sys_atoms[sel], atoms=ai, sys=si, n_atoms=len(atoms),
                                  n_systems=len(sel))
        gather_state(w, m, ai, ('z', 'x', 'v', 'force', 'fixed'))
        gather_state(w, m, si, ('energy', 'cell', 'sf', 'si'))
        w.batch = torch.as_tensor(batch, dtype=torch.int64, device=dev)
        w.pos_model = torch.empty(len(atoms), 3, dtype=torch.float32, device=dev)
        w.step_ctr = torch.zeros(1, dtype=torch.int64, device=dev)
        w.sticky = torch.zeros(4, dtype=torch.int32, device=dev)
        w.ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        self.work = w
        self._wrap()
        self._build(count_edges(self.engine, w.pos_model, w.cell, w.batch, self.weights.cutoff).n_edges)

    def _scatter(self):
        """Copy the graph's systems back into the master state."""
        w, m = self.work, self.master
        scatter_state(m, w, w.atoms, ('x', 'v', 'force'))
        scatter_state(m, w, w.sys, ('energy', 'sf', 'si'))

    def _wrap(self):
        w = self.work
        L.check(self.lib.nn_wrap_positions(w.n_atoms, w.x.data_ptr(), w.cell.data_ptr(), w.batch.data_ptr(),
                                           w.pos_model.data_ptr(), stream()), 'nn_wrap_positions')

    def _fire_step(self):
        w = self.work
        L.check(self.lib.nn_fire_step(w.n_systems, w.nl.sys_ptr.data_ptr(), w.x.data_ptr(), w.v.data_ptr(), w.force.data_ptr(),
                                      w.cell.data_ptr(), w.pos_model.data_ptr(), w.sf.data_ptr(), w.si.data_ptr(),
                                      *self.params, stream()), 'nn_fire_step')

    def _check(self, advance):
        w = self.work
        L.check(self.lib.nn_fire_check(w.n_systems, w.nl.sys_ptr.data_ptr(), w.force.data_ptr(), w.fixed.data_ptr(),
                                       self.fmax2.data_ptr(), w.sf.data_ptr(), w.si.data_ptr(), advance, w.step_ctr.data_ptr(),
                                       w.nl.status.data_ptr(), w.sticky.data_ptr(), w.ticket.data_ptr(), stream()),
                'nn_fire_check')

    def _step(self):
        self._fire_step()
        self.work.forces_step()
        self._check(1)

    def _build(self, n_edges):
        """(Re)allocate the neighbour list for `n_edges`, evaluate forces and the convergence test at the current
        positions and capture the step."""
        w = self.work
        w.forces_step = force_step(self.engine, self.weights, w.z, w.pos_model, w.cell, w.batch, w.energy, w.force, n_edges,
                                   self.HEADROOM)
        w.nl = w.forces_step.nl
        self._check(0)
        w.graph, _, self.kernels_per_step = capture(self._step, self.device)     # kernels one graph replay launches

    # ------------------------------------------------------------------ run
    def run(self, fmax=0.05, steps=100_000_000):
        """Relax until every system has max_i |f_i| < fmax (eV/A) or `steps` steps of this call have been taken; returns
        True when every system has converged (ASE's Optimizer.run).  A second call continues from the stored state
        (velocities, dt, a, Nsteps); every system whose current max |f| is at least the new fmax steps again."""
        f2 = float(fmax) ** 2
        self.fmax2.fill_(f2)
        m = self.master
        active = ~(m['sf'][:, F2].cpu().numpy() < f2)
        m['si'][:, CONVERGED] = torch.as_tensor(~active, dtype=torch.int32, device=self.device)
        if not active.any():
            return True
        plan = compaction_plan(active, self.sys_atoms)
        sel, batch = (np.arange(self.n_systems), np.repeat(np.arange(self.n_systems), self.sys_atoms)) if plan is None else plan
        if not np.array_equal(sel, self.work.sel):
            self._use(sel, batch)
        else:
            self._check(0)                                   # the new fmax's converged flags
        done = 0
        while done < steps:
            w = self.work
            n = min(self.check_interval, steps - done)
            need = replay_chunk(w.graph, n, w.sticky, (w.x, w.v, w.force, w.energy, w.sf, w.si, w.step_ctr))
            self.graph_launches += n
            if need:                                         # capacity overflow somewhere in the chunk: rolled back; regrow, redo
                self._wrap()
                self._build(need)
                continue
            done += n
            active = w.si[:, CONVERGED].cpu().numpy() == 0
            if not active.any():
                break
            plan = compaction_plan(active, w.sys_atoms)
            if plan is not None and done < steps:
                self._scatter()
                self._use(w.sel[plan[0]], plan[1])
                self.compactions += 1
        self._scatter()
        return bool(m['si'][:, CONVERGED].all())

    # ------------------------------------------------------------------ state (numpy; per atom [N,...] or per system [B])
    @property
    def positions(self):
        return self.master['x'].cpu().numpy()

    @property
    def forces(self):
        return self.master['force'].cpu().numpy().astype(np.float64)

    @property
    def energy(self):
        return self.master['energy'].cpu().numpy().astype(np.float64)

    @property
    def fmax(self):
        """max_i |f_i| per system at the current positions."""
        return np.sqrt(self.master['sf'][:, F2].cpu().numpy())

    @property
    def converged(self):
        return self.master['si'][:, CONVERGED].cpu().numpy() != 0

    @property
    def nsteps(self):
        """Steps each system has taken, over all run() calls."""
        return self.master['si'][:, STEPS].cpu().numpy().astype(np.int64)

    @property
    def state(self):
        """FIRE state per system: velocities [N,3], dt [B], a [B], Nsteps [B]."""
        m = self.master
        sf, si = m['sf'].cpu().numpy(), m['si'].cpu().numpy()
        return {'v': m['v'].cpu().numpy(), 'dt': sf[:, DT], 'a': sf[:, A], 'Nsteps': si[:, NSTEPS]}

"""Device-resident molecular dynamics (SURVEY.md section 8f rank 1).

The reference runs MD from ASE on the host: scripts/simulate.py:21-31 builds `Langevin(atoms, 0.5 fs, 300 K,
friction 1/(500 fs))` and every step calls MLAseCalculator.calculate (utils/ase_interface.py:52-81): numpy -> torch
-> H2D -> forward -> D2H -> numpy.  `DeviceMD` keeps positions, velocities and forces in HBM and replays one CUDA
graph per step (integrator half step, neighbour rebuild, network forward + reverse sweep, second half kick, log
row) - the host only enqueues graph launches and reads the status / energy log once per `check_interval` steps.

Integrator: BAOAB splitting (velocity Verlet when no thermostat is requested).  ASE's own Langevin scheme is a
third-party algorithm that is not part of /root/reference; trajectories of a stochastic thermostat are not
comparable step by step anyway, so parity is (a) NVE trajectories against a host fp64 velocity Verlet driven through
the calculator and (b) the thermostat's temperature.  Units are ASE's: Angstrom, eV, amu, time in
Angstrom*sqrt(amu/eV) (`FS` converts femtoseconds), `KB` in eV/K.
"""
import math

import numpy as np
import torch

from newtonnet_b200 import _lib as L
from newtonnet_b200.engine import capture, count_edges, driver_inputs, force_step, replay_chunk, stream

__all__ = ['DeviceMD', 'FS', 'KB', 'ATOMIC_MASSES']

FS = 1e-15 * 1e10 * math.sqrt(1.6021766208e-19 / 1.660539040e-27)     # one femtosecond in ASE time units (0.0982269...)
KB = 8.6173303e-5                                                      # eV / K
ATOMIC_MASSES = np.array([0.0, 1.008, 4.002602, 6.94, 9.0121831, 10.81, 12.011, 14.007, 15.999, 18.998403163, 20.1797,
                          22.98976928, 24.305, 26.9815385, 28.085, 30.973761998, 32.06, 35.45, 39.948, 39.0983, 40.078,
                          44.955908, 47.867, 50.9415, 51.9961, 54.938044, 55.845, 58.933194, 58.6934, 63.546, 65.38,
                          69.723, 72.630, 74.921595, 78.971, 79.904, 83.798])


def atoms_cell(atoms):
    """[3,3] fp64 cell of an ASE-like Atoms with the rows of non-periodic directions zeroed (ase_interface.py:134-138)."""
    cell = np.array(getattr(atoms.get_cell(), 'array', atoms.get_cell()), dtype=np.float64).reshape(3, 3)
    cell[~np.asarray(atoms.get_pbc(), dtype=bool).reshape(3)] = 0.0
    return cell


class DeviceMD:
    """NVE / Langevin MD of one system or a batch of independent systems, state resident on the GPU.

    model: newtonnet_b200 NewtonNet (CUDA, energy head); z [N]; pos [N,3]; cell [B,3,3] or None (not periodic);
    batch [N] or None (one system); masses [N] amu (default: standard weights, H-Kr); timestep in ASE time units;
    temperature_K + friction (1 / ASE time) switch the Ornstein-Uhlenbeck step on; velocities [N,3] or None
    (Maxwell-Boltzmann at temperature_K when given, else zero)."""

    HEADROOM = (1.15, 64)          # edge capacity: factor and slack over the counted edges

    def __init__(self, model, z, pos, cell=None, batch=None, masses=None, timestep=0.5 * FS, temperature_K=None,
                 friction=None, velocities=None, seed=0, log_capacity=1024, check_interval=64):
        self.lib = L.load()
        self.model = model
        dev, self.engine, self.weights, as_t, self.z, self.x, self.batch, self.cell = driver_inputs(model, z, pos, cell, batch, 'DeviceMD')
        self.device = dev
        N, B = self.z.shape[0], self.cell.shape[0]
        if masses is None:
            zc = self.z.cpu().numpy()
            if zc.max() >= len(ATOMIC_MASSES):
                raise ValueError('pass `masses` for elements beyond Kr')
            masses = ATOMIC_MASSES[zc]
        m = as_t(masses, torch.float64)
        self.masses = m
        self.inv_mass = torch.where(m > 0, 1.0 / m, torch.zeros_like(m))
        self.dt = float(timestep)
        self.kT = 0.0 if temperature_K is None else KB * float(temperature_K)
        self.ou_c = 1.0 if (friction is None or temperature_K is None) else math.exp(-float(friction) * self.dt)
        self.seed = int(seed)
        if velocities is None:
            self.v = torch.zeros(N, 3, dtype=torch.float64, device=dev)
            if temperature_K is not None:
                g = torch.Generator(device='cpu').manual_seed(self.seed)
                self.v = (torch.randn(N, 3, dtype=torch.float64, generator=g).to(dev) * torch.sqrt(self.kT * self.inv_mass)[:, None])
        else:
            self.v = as_t(velocities, torch.float64).reshape(N, 3).clone()
        self.n_atoms, self.n_systems = N, B
        self.pos_model = torch.empty(N, 3, dtype=torch.float32, device=dev)
        self.energy = torch.empty(B, dtype=torch.float32, device=dev)
        self.force = torch.zeros(N, 3, dtype=torch.float32, device=dev)
        self.step_ctr = torch.zeros(1, dtype=torch.int64, device=dev)
        self.sticky = torch.zeros(4, dtype=torch.int32, device=dev)
        self.ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        self.log_capacity = int(log_capacity)
        self.check_interval = max(1, min(int(check_interval), self.log_capacity))
        self.log = torch.zeros(self.log_capacity, B, 2, dtype=torch.float64, device=dev)
        self.graph_launches = 0
        self._wrap()
        self._build(count_edges(self.engine, self.pos_model, self.cell, self.batch, self.weights.cutoff).n_edges)

    # ------------------------------------------------------------------ construction helpers
    @classmethod
    def from_atoms(cls, atoms, calc, **kwargs):
        """From an ASE-like Atoms object and an MLAseCalculator (scripts/simulate.py:10-31)."""
        kw = dict(kwargs)
        if hasattr(atoms, 'get_masses'):
            kw.setdefault('masses', atoms.get_masses())
        if hasattr(atoms, 'get_velocities') and atoms.get_velocities() is not None and np.any(atoms.get_velocities()):
            kw.setdefault('velocities', atoms.get_velocities())
        return cls(calc.model, atoms.get_atomic_numbers(), atoms.get_positions(), atoms_cell(atoms)[None], **kw)

    def update_atoms(self, atoms):
        atoms.set_positions(self.positions)
        if hasattr(atoms, 'set_velocities'):
            atoms.set_velocities(self.velocities)
        return atoms

    def _advance(self, dt, ou_c):
        L.check(self.lib.nn_md_advance(self.n_atoms, self.x.data_ptr(), self.v.data_ptr(), self.force.data_ptr(),
                                       self.inv_mass.data_ptr(), self.cell.data_ptr(), self.batch.data_ptr(),
                                       self.pos_model.data_ptr(), dt, ou_c, self.kT, self.seed, self.step_ctr.data_ptr(),
                                       stream()), 'nn_md_advance')

    def _wrap(self):
        L.check(self.lib.nn_wrap_positions(self.n_atoms, self.x.data_ptr(), self.cell.data_ptr(), self.batch.data_ptr(),
                                           self.pos_model.data_ptr(), stream()), 'nn_wrap_positions')

    def _finish(self):
        L.check(self.lib.nn_md_finish(self.n_systems, self.nl.sys_ptr.data_ptr(), self.v.data_ptr(), self.force.data_ptr(),
                                      self.inv_mass.data_ptr(), self.dt, self.energy.data_ptr(), self.log.data_ptr(),
                                      self.log_capacity, self.step_ctr.data_ptr(), self.nl.status.data_ptr(),
                                      self.sticky.data_ptr(), self.ticket.data_ptr(), stream()), 'nn_md_finish')

    def _step(self):
        self._advance(self.dt, self.ou_c)
        self.forces_step()
        self._finish()

    def _build(self, n_edges):
        """(Re)allocate the neighbour list for `n_edges`, evaluate forces at the current positions and capture the step."""
        self.forces_step = force_step(self.engine, self.weights, self.z, self.pos_model, self.cell, self.batch, self.energy,
                                      self.force, n_edges, self.HEADROOM)
        self.nl = self.forces_step.nl
        self.graph, _, self.kernels_per_step = capture(self._step, self.device)     # kernels one graph replay launches

    # ------------------------------------------------------------------ run
    def run(self, steps, trajectory_interval=None):
        """Advance `steps` time steps.  Returns {'energy': [steps, B], 'kinetic': [steps, B]} (numpy fp64, eV) and, with
        trajectory_interval = k, 'positions': [steps // k, N, 3] (unwrapped, fp64) sampled after every k-th step - the
        device-side counterpart of the `trajectory=..., loginterval=k` arguments of the reference's ASE driver
        (scripts/simulate.py:21-30); the copy happens at chunk boundaries, so chunks are cut at multiples of k."""
        pe, ke, traj = [], [], []
        done = 0
        while done < steps:
            n = min(self.check_interval, steps - done)
            if trajectory_interval:
                n = min(n, trajectory_interval - (done % trajectory_interval))
            s0 = self.step
            need = replay_chunk(self.graph, n, self.sticky, (self.x, self.v, self.force, self.step_ctr))
            self.graph_launches += n
            if need:                                           # capacity overflow somewhere in the chunk: rolled back; regrow, redo
                self._wrap()
                self._build(need)
                continue
            rows = (torch.arange(s0, s0 + n, device=self.device) % self.log_capacity)
            chunk = self.log[rows].cpu().numpy()
            pe.append(chunk[:, :, 0]); ke.append(chunk[:, :, 1])
            done += n
            if trajectory_interval and done % trajectory_interval == 0:
                traj.append(self.x.cpu().numpy())
        empty = np.zeros((0, self.n_systems))
        out = {'energy': np.concatenate(pe) if pe else empty, 'kinetic': np.concatenate(ke) if ke else empty}
        if trajectory_interval:
            out['positions'] = np.stack(traj) if traj else np.zeros((0, self.n_atoms, 3))
        return out

    # ------------------------------------------------------------------ state
    @property
    def step(self):
        return int(self.step_ctr.item())

    @property
    def positions(self):
        return self.x.cpu().numpy()

    @property
    def velocities(self):
        return self.v.cpu().numpy()

    @property
    def forces(self):
        return self.force.cpu().numpy().astype(np.float64)

    def temperature(self):
        """Instantaneous temperature per system [B] (K), 3N degrees of freedom as ASE's get_temperature."""
        ke = torch.zeros(self.n_systems, dtype=torch.float64, device=self.device).index_add_(
            0, self.batch, 0.5 * self.masses * (self.v * self.v).sum(-1))
        n = torch.bincount(self.batch, minlength=self.n_systems).clamp(min=1)
        return (2.0 * ke / (3.0 * n * KB)).cpu().numpy()

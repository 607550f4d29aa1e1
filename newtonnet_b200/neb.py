"""Device-resident climbing-image NEB: reaction paths and saddle points for a batch of bands at once.

Finding the minimum-energy path between two minima through ASE runs on the host: every step of FIRE(NEB(images)) calls
MLAseCalculator.calculate on the interior images (utils/ase_interface.py:52-81: numpy -> H2D -> forward -> D2H ->
numpy), then the NEB projection and the FIRE update in numpy.  `DeviceNEB` keeps every band's positions, FIRE velocities,
model forces, NEB forces and FIRE state in HBM and replays one CUDA graph per step: nn_fire_step (one system per band)
-> neighbour rebuild -> nn_eval (one system per interior image) -> nn_neb_forces -> nn_fire_check (one system per band).

The method is ASE 3.22's NEB with method='improvedtangent', a scalar spring constant and an optional climbing image,
optimised by ASE's FIRE with one optimiser state per band - the whole band is one optimisable, as FIRE sees an NEB object
- and converged when max |F_neb| over the band's interior atoms is below fmax.  oracle/neb_oracle.py restates it in
numpy.  The NEB force is stored in fp32 because the FIRE kernels read fp32 forces; it is computed in fp64.
"""
import types
import warnings

import numpy as np
import torch

from newtonnet_b200 import _lib as L
from newtonnet_b200.engine import capture, count_edges, driver_inputs, force_step, replay_chunk, stream
from newtonnet_b200.md import atoms_cell
from newtonnet_b200.optimize import (A, CONVERGED, DT, F2, NSTEPS, STEPS, compaction_plan, fixed_mask, gather_state,
                                     scatter_state, segment_rows)

__all__ = ['DeviceNEB', 'align_band', 'band_layout', 'bands_from_inputs']

ATOM_KEYS = ('z', 'x', 'v', 'force', 'true_force', 'fixed')
IMAGE_KEYS = ('energy', 'img_cell')
BAND_KEYS = ('cell', 'sf', 'si', 'climb', 'imax', 'failed', 'ends_energy', 'band_ends')
INDEX_KEYS = ('band_ptr', 'img_ptr', 'img_band', 'band_img')


def _host(a, dtype):
    return (a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)).astype(dtype)


def align_band(R, cell):
    """Positions of a band [n+2, n_atoms, 3] with every image shifted by lattice vectors so that its displacement from
    the image before it is the minimum image by fractional rounding; image 0 stays as it is.  cell [3,3] (rows are the
    lattice vectors; all zero = not periodic, returned unchanged).  An aligned displacement longer than half the smallest
    cell height is ambiguous and raises ValueError."""
    R = np.array(R, dtype=np.float64)
    cell = np.asarray(cell, dtype=np.float64).reshape(3, 3)
    if not (cell != 0).any():
        return R
    if np.linalg.det(cell) == 0:
        raise ValueError('partially periodic cells are not supported')
    inv = np.linalg.inv(cell)
    half = 0.5 / np.linalg.norm(inv, axis=0).max()          # half the smallest distance between opposite faces
    for i in range(1, len(R)):
        R[i] -= np.rint((R[i] - R[i - 1]) @ inv) @ cell
        d = np.linalg.norm(R[i] - R[i - 1], axis=1)
        if (d > half).any():
            raise ValueError(f'image {i}: atom {int(d.argmax())} moves {d.max():.3f} A from image {i - 1}, more than half '
                             f'the smallest cell height ({half:.3f} A): its periodic image is ambiguous')
    return R


def bands_from_inputs(z, images, cell=None, fixed=None):
    """DeviceNEB's inputs as a list of bands (z [n_atoms] int64, R [n+2, n_atoms, 3] fp64 aligned, cell [3,3] fp64,
    fixed [n_atoms] bool).  One band: images is an array or tensor [n+2, n_atoms, 3], z [n_atoms], cell [3,3] or None,
    fixed [n_atoms] or None.  Several bands: lists of those (cell and fixed may also be None for all)."""
    one = torch.is_tensor(images) or isinstance(images, np.ndarray)
    if one:
        z, images, cell, fixed = [z], [images], [cell], [fixed]
    B = len(images)
    cell = [None] * B if cell is None else list(cell)
    fixed = [None] * B if fixed is None else list(fixed)
    if not (len(z) == len(cell) == len(fixed) == B) or B == 0:
        raise ValueError(f'{B} bands of images, but {len(z)} z, {len(cell)} cells and {len(fixed)} fixed masks')
    out = []
    for b in range(B):
        zb = _host(z[b], np.int64).reshape(-1)
        R = _host(images[b], np.float64)
        na = len(zb)
        if R.ndim != 3 or R.shape[1:] != (na, 3):
            raise ValueError(f'band {b}: images must be [n+2, {na}, 3] for {na} atoms, got {list(R.shape)}')
        if R.shape[0] < 3:
            raise ValueError(f'band {b}: a band needs at least one interior image between its end points')
        c = np.zeros((3, 3)) if cell[b] is None else _host(cell[b], np.float64).reshape(3, 3)
        f = np.zeros(na, dtype=bool) if fixed[b] is None else _host(fixed[b], bool).reshape(na)
        R = align_band(R, c)
        if f.any() and np.abs(R[:, f] - R[0, f]).max() > 1e-6:
            raise ValueError(f'band {b}: fixed atoms must sit at the same place in every image (ASE keeps them still, and '
                             f'their force counts as zero)')
        d = np.linalg.norm((R[1:] - R[:-1]).reshape(len(R) - 1, -1), axis=1)
        if (d == 0).any():
            i = int(np.flatnonzero(d == 0)[0])
            raise ValueError(f'band {b}: images {i} and {i + 1} coincide (the tangent between them is undefined)')
        out.append((zb, R, c, f))
    return out


def band_layout(n_atoms, n_interior):
    """Offsets of bands stored band-major with their interior images image-major, so that each band's interior atoms are
    one contiguous range.  n_atoms [B] atoms per image, n_interior [B] interior images per band.  Returns int64 arrays:
    band_ptr [B+1] first interior atom of each band, band_img [B+1] first interior image of each band, img_ptr [I+1] first
    atom of each interior image, img_band [I] band of each interior image, ends_ptr [B] first end-point row of each band
    (its image 0, then its image n+1)."""
    na, ni = np.asarray(n_atoms, dtype=np.int64), np.asarray(n_interior, dtype=np.int64)
    img_band = np.repeat(np.arange(len(na)), ni)
    return dict(band_ptr=np.concatenate([[0], np.cumsum(na * ni)]), band_img=np.concatenate([[0], np.cumsum(ni)]),
                img_ptr=np.concatenate([[0], np.cumsum(na[img_band])]), img_band=img_band,
                ends_ptr=np.concatenate([[0], np.cumsum(2 * na)])[:-1])


class DeviceNEB:
    """Climbing-image NEB of one band or a batch of bands, state resident on the GPU.

    model: newtonnet_b200 NewtonNet (CUDA, energy head); images: [n+2, n_atoms, 3] positions of one band, end points
    included (Angstrom), with z [n_atoms], cell [3,3] or None (not periodic) and fixed [n_atoms] bool or None (atoms held
    in place, as ASE's FixAtoms); or lists of those, one per band (bands may differ in molecule and image count).
    k: spring constant (eV/A^2); climb: climbing image on.  dt ... a: ASE's FIRE parameters, per band.  check_interval:
    steps replayed between two reads of the status and the converged flags.  Only ASE's method='improvedtangent' with a
    scalar k, no remove_rotation_and_translation and no preconditioner is built; the others raise NotImplementedError.
    Periodic bands are aligned once (`align_band`); end-point energies are evaluated once, here."""

    HEADROOM = (1.15, 64)          # edge capacity: factor and slack over the counted edges

    def __init__(self, model, z, images, cell=None, fixed=None, k=0.1, climb=False, method='improvedtangent',
                 remove_rotation_and_translation=False, precon=None, dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1,
                 fdec=0.5, astart=0.1, fa=0.99, a=0.1, check_interval=16):
        if method != 'improvedtangent':
            raise NotImplementedError(f"DeviceNEB implements method='improvedtangent' only, not {method!r}")
        if remove_rotation_and_translation or precon is not None:
            raise NotImplementedError('DeviceNEB supports neither remove_rotation_and_translation nor a preconditioner')
        if np.ndim(k) != 0:
            raise NotImplementedError('DeviceNEB takes one scalar spring constant k, not one per spring')
        if not float(k) > 0:
            raise ValueError(f'the spring constant k must be > 0, got {k}')
        self.lib = L.load()
        self.model = model
        bands = bands_from_inputs(z, images, cell, fixed)
        self.n_bands = B = len(bands)
        self.band_atoms = np.array([len(zb) for zb, _, _, _ in bands], dtype=np.int64)
        self.band_images = np.array([len(R) - 2 for _, R, _, _ in bands], dtype=np.int64)
        self.layout = lay = band_layout(self.band_atoms, self.band_images)
        self.k, self.climb = float(k), bool(climb)
        self.params = (float(maxstep), float(dtmax), float(finc), float(fdec), float(astart), float(fa), int(Nmin))
        self.check_interval = max(1, int(check_interval))
        self._ends = [R[[0, -1]] for _, R, _, _ in bands]
        n_img = self.band_images
        z_all = np.concatenate([np.tile(zb, n) for (zb, _, _, _), n in zip(bands, n_img)])
        x_all = np.concatenate([R[1:-1].reshape(-1, 3) for _, R, _, _ in bands])
        img_cell = np.repeat(np.stack([c for _, _, c, _ in bands]), n_img, axis=0)
        img_batch = np.repeat(np.arange(len(lay['img_band'])), self.band_atoms[lay['img_band']])
        dev, self.engine, self.weights, as_t, z_t, x, _, img_cell_t = driver_inputs(model, z_all, x_all, img_cell, img_batch,
                                                                                   'DeviceNEB')
        self.device = dev
        N, I = len(z_all), len(lay['img_band'])
        f64, f32, i32 = (dict(dtype=t, device=dev) for t in (torch.float64, torch.float32, torch.int32))
        sf = torch.zeros(B, 3, **f64)
        sf[:, DT], sf[:, A] = float(dt), float(a)
        # end points: fp64 positions the springs of the first and last interior images read, energies evaluated once
        ends = torch.as_tensor(np.concatenate([e.reshape(-1, 3) for e in self._ends]), **f64)
        self.master = dict(z=z_t, x=x, v=torch.zeros(N, 3, **f64), force=torch.zeros(N, 3, **f32),
                           true_force=torch.zeros(N, 3, **f32),
                           fixed=as_t(np.concatenate([np.tile(f, n) for (_, _, _, f), n in zip(bands, n_img)]), torch.bool),
                           energy=torch.zeros(I, **f32), img_cell=img_cell_t, cell=img_cell_t[torch.as_tensor(lay['band_img'][:-1], device=dev)].contiguous(),
                           sf=sf, si=torch.zeros(B, 4, **i32), climb=torch.full((B,), int(self.climb), **i32),
                           imax=torch.zeros(B, **i32), failed=torch.zeros(B, **i32), ends_energy=self._end_energies(bands, ends),
                           band_ends=torch.as_tensor(lay['ends_ptr'], **i32))
        self.ends = ends
        bad = ~torch.isfinite(self.master['ends_energy']).all(1).cpu().numpy()
        if bad.any():
            raise ValueError(f'the model gives non-finite energies for the end points of bands {np.flatnonzero(bad).tolist()}')
        self.master_index = types.SimpleNamespace(**{k: torch.as_tensor(lay[k], **i32) for k in INDEX_KEYS})
        self.fmax2 = torch.zeros(1, **f64)
        self.graph_launches = 0        # step graph replays, rolled-back chunks included
        self.compactions = 0
        self.work = None
        self._use(np.arange(B))        # evaluates the input images
        self._scatter()

    def _end_energies(self, bands, ends):
        """[B,2] fp64 energies of every band's end points, through the engine's evaluation path at the fp32 wrapped
        positions the step graph would use."""
        dev = self.device
        B = len(bands)
        na = self.band_atoms
        z = torch.as_tensor(np.concatenate([np.tile(zb, 2) for zb, _, _, _ in bands]), dtype=torch.int64, device=dev)
        cell = torch.as_tensor(np.repeat(np.stack([c for _, _, c, _ in bands]), 2, axis=0), dtype=torch.float32, device=dev)
        batch = torch.as_tensor(np.repeat(np.arange(2 * B), np.repeat(na, 2)), dtype=torch.int64, device=dev)
        pos = torch.empty(len(z), 3, dtype=torch.float32, device=dev)
        L.check(self.lib.nn_wrap_positions(len(z), ends.data_ptr(), cell.data_ptr(), batch.data_ptr(), pos.data_ptr(),
                                           stream()), 'nn_wrap_positions')
        out = self.engine.energy_forces(self.weights, z, pos, cell, batch)
        return out['energy'].double().reshape(B, 2).contiguous()

    # ------------------------------------------------------------------ construction from Atoms
    @staticmethod
    def _band_list(images):
        return [list(images)] if hasattr(images[0], 'get_atomic_numbers') else [list(b) for b in images]

    @classmethod
    def from_images(cls, images, calc, **kwargs):
        """From one band or a list of bands, each a list of ASE-like Atoms with its end points (as ase.neb.NEB(images)),
        and an MLAseCalculator.  FixAtoms-like constraints become `fixed`; any other constraint raises
        NotImplementedError.  The images of a band must agree in atom count, atomic numbers, cell and fixed atoms."""
        zs, Rs, cells, fixed = [], [], [], []
        for b, band in enumerate(cls._band_list(images)):
            z0, c0, f0 = np.asarray(band[0].get_atomic_numbers()), atoms_cell(band[0]), fixed_mask(band[0], 'DeviceNEB')
            for i, at in enumerate(band[1:], 1):
                if len(at) != len(z0) or not np.array_equal(at.get_atomic_numbers(), z0):
                    raise ValueError(f'band {b}: image {i} has other atoms than image 0')
                if not np.array_equal(atoms_cell(at), c0):
                    raise ValueError(f'band {b}: image {i} has another cell than image 0')
                if not np.array_equal(fixed_mask(at, 'DeviceNEB'), f0):
                    raise ValueError(f'band {b}: image {i} fixes other atoms than image 0')
            zs.append(z0)
            Rs.append(np.stack([at.get_positions() for at in band]))
            cells.append(c0)
            fixed.append(f0)
        return cls(calc.model, zs, Rs, cells, fixed, **kwargs)

    def update_images(self, images):
        """Write the current interior positions into the Atoms of the band (or list of bands) it was built from."""
        for band, R in zip(self._band_list(images), self.positions):
            for i in range(1, len(band) - 1):
                band[i].set_positions(R[i])
        return images

    # ------------------------------------------------------------------ the step graph
    def _use(self, sel):
        """Point the step graph at master bands `sel` (ascending): gather their state into fresh buffers, evaluate and
        capture."""
        m, dev, lay = self.master, self.device, self.layout
        sel = np.asarray(sel)
        ai = torch.as_tensor(segment_rows(lay['band_ptr'], sel), device=dev)
        ii = torch.as_tensor(segment_rows(lay['band_img'], sel), device=dev)
        bi = torch.as_tensor(sel, device=dev)
        sub = band_layout(self.band_atoms[sel], self.band_images[sel])
        w = types.SimpleNamespace(sel=sel, band_atoms=self.band_atoms[sel] * self.band_images[sel], atoms=ai, images=ii,
                                  bands=bi, n_atoms=len(ai), n_images=len(ii), n_bands=len(sel))
        gather_state(w, m, ai, ATOM_KEYS)
        gather_state(w, m, ii, IMAGE_KEYS)
        gather_state(w, m, bi, BAND_KEYS)
        for k in INDEX_KEYS:
            setattr(w, k, torch.as_tensor(sub[k], dtype=torch.int32, device=dev))
        w.img_batch = torch.as_tensor(np.repeat(np.arange(w.n_images), self.band_atoms[sel][sub['img_band']]), device=dev)
        w.pos_model = torch.empty(w.n_atoms, 3, dtype=torch.float32, device=dev)
        w.step_ctr = torch.zeros(1, dtype=torch.int64, device=dev)
        w.sticky = torch.zeros(4, dtype=torch.int32, device=dev)
        w.ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        self.work = w
        self._wrap()
        self._build(count_edges(self.engine, w.pos_model, w.img_cell, w.img_batch, self.weights.cutoff).n_edges)

    def _scatter(self):
        """Copy the graph's bands back into the master state."""
        w, m = self.work, self.master
        scatter_state(m, w, w.atoms, ('x', 'v', 'force', 'true_force'))
        scatter_state(m, w, w.images, ('energy',))
        scatter_state(m, w, w.bands, ('sf', 'si', 'imax', 'failed'))

    def _wrap(self):
        w = self.work
        L.check(self.lib.nn_wrap_positions(w.n_atoms, w.x.data_ptr(), w.img_cell.data_ptr(), w.img_batch.data_ptr(),
                                           w.pos_model.data_ptr(), stream()), 'nn_wrap_positions')

    def _fire_step(self):
        w = self.work
        L.check(self.lib.nn_fire_step(w.n_bands, w.band_ptr.data_ptr(), w.x.data_ptr(), w.v.data_ptr(), w.force.data_ptr(),
                                      w.cell.data_ptr(), w.pos_model.data_ptr(), w.sf.data_ptr(), w.si.data_ptr(),
                                      *self.params, stream()), 'nn_fire_step')

    def _neb(self, s):
        """NEB forces of the bands of `s` (the step graph's buffers, or the master state with its index arrays)."""
        L.check(self.lib.nn_neb_forces(len(s.img_band), s.img_ptr.data_ptr(), s.img_band.data_ptr(), s.band_img.data_ptr(),
                                       s.x.data_ptr(), self.ends.data_ptr(), s.band_ends.data_ptr(), s.energy.data_ptr(),
                                       s.ends_energy.data_ptr(), s.true_force.data_ptr(), s.fixed.data_ptr(),
                                       s.climb.data_ptr(), s.si.data_ptr(), self.k, s.force.data_ptr(), s.imax.data_ptr(),
                                       s.failed.data_ptr(),                                        stream()), 'nn_neb_forces')

    def _check(self, s, advance):
        """nn_fire_check on the bands of `s`; advance = 1 is the captured step's, 0 only measures."""
        st = (s.step_ctr, s.nl.status, s.sticky, s.ticket) if advance else (None,) * 4
        L.check(self.lib.nn_fire_check(len(s.sf), s.band_ptr.data_ptr(), s.force.data_ptr(), s.fixed.data_ptr(),
                                       self.fmax2.data_ptr(), s.sf.data_ptr(), s.si.data_ptr(), advance,
                                       *(L.ptr(t) for t in st), stream()), 'nn_fire_check')

    def _step(self):
        w = self.work
        self._fire_step()
        w.forces_step()
        self._neb(w)
        self._check(w, 1)

    def _build(self, n_edges):
        """(Re)allocate the neighbour list for `n_edges`, evaluate the model, the NEB forces and the convergence test at
        the current positions and capture the step."""
        w = self.work
        w.forces_step = force_step(self.engine, self.weights, w.z, w.pos_model, w.img_cell, w.img_batch, w.energy,
                                   w.true_force, n_edges, self.HEADROOM)
        w.nl = w.forces_step.nl
        self._neb(w)
        self._check(w, 0)
        w.graph, _, self.kernels_per_step = capture(self._step, self.device)     # kernels one graph replay launches

    # ------------------------------------------------------------------ run
    def run(self, fmax=0.05, steps=100_000_000, climb=None):
        """Optimise until every band has max |F_neb| < fmax (eV/A) over its interior atoms or `steps` steps of this call
        have been taken; returns True when every band has converged.  climb: switch the climbing image on or off (None
        keeps the current setting).  A second call continues from the stored state (velocities, dt, a, Nsteps); every
        band whose current max |F_neb| is at least the new fmax steps again.  A band for which the model returns a non-finite
        energy or force stops where it is, is reported in `failed` and never steps again (a warning names it)."""
        f2 = float(fmax) ** 2
        self.fmax2.fill_(f2)
        m = self.master
        if climb is not None and bool(climb) != self.climb:
            # the stored NEB forces and convergence flags belong to the other projection: recompute both for every band at
            # the current positions (model energies and forces there are stored), then regather the step graph
            self._scatter()
            self.climb = bool(climb)
            m['climb'].fill_(int(self.climb))
            m['si'][:, CONVERGED] = 0
            s = types.SimpleNamespace(**m, **vars(self.master_index))
            self._neb(s)
            self._check(s, 0)
            self.work.sel = None
        failed0 = self.failed
        active = ~(m['sf'][:, F2].cpu().numpy() < f2) & ~failed0
        m['si'][:, CONVERGED] = torch.as_tensor(~active, dtype=torch.int32, device=self.device)
        if not active.any():
            return not failed0.any()
        n_band_atoms = self.band_atoms * self.band_images
        plan = compaction_plan(active, n_band_atoms)
        sel = np.arange(self.n_bands) if plan is None else plan[0]
        if self.work.sel is None or not np.array_equal(sel, self.work.sel):
            self._use(sel)
        else:
            self._check(self.work, 0)                            # the new fmax's converged flags
        done = 0
        while done < steps:
            w = self.work
            n = min(self.check_interval, steps - done)
            need = replay_chunk(w.graph, n, w.sticky, (w.x, w.v, w.force, w.true_force, w.energy, w.sf, w.si, w.imax,
                                                       w.failed, w.step_ctr))
            self.graph_launches += n
            if need:                                         # capacity overflow somewhere in the chunk: rolled back; regrow, redo
                self._wrap()
                self._build(need)
                continue
            done += n
            active = ((w.si[:, CONVERGED] == 0) & (w.failed == 0)).cpu().numpy()
            if not active.any():
                break
            plan = compaction_plan(active, w.band_atoms)
            if plan is not None and done < steps:
                self._scatter()
                self._use(w.sel[plan[0]])
                self.compactions += 1
        self._scatter()
        new = np.flatnonzero(self.failed & ~failed0)
        if len(new):
            warnings.warn(f'DeviceNEB: the model returned non-finite energies or forces for bands {new.tolist()}; they were '
                          f'stopped where that happened (see `failed`)', RuntimeWarning, stacklevel=2)
        return bool(self.converged.all())

    # ------------------------------------------------------------------ results (numpy, one entry per band)
    def _per_band(self, t, shape_fn):
        a = t.cpu().numpy()
        p = self.layout['band_ptr']
        return [a[p[b]:p[b + 1]].reshape(shape_fn(b)) for b in range(self.n_bands)]

    def _interior(self, t):
        return [f.astype(np.float64) for f in
                self._per_band(t, lambda b: (self.band_images[b], self.band_atoms[b], 3))]

    @property
    def positions(self):
        """Per band [n+2, n_atoms, 3]: the end points (aligned) and the current interior images."""
        return [np.concatenate([e[:1], x, e[1:]]) for e, x in zip(self._ends, self._interior(self.master['x']))]

    @property
    def energies(self):
        """Per band [n+2] fp64: end-point energies and the interior images' energies at their current positions."""
        e, ends, p = self.master['energy'].cpu().numpy().astype(np.float64), self.master['ends_energy'].cpu().numpy(), self.layout['band_img']
        return [np.concatenate([ends[b, :1], e[p[b]:p[b + 1]], ends[b, 1:]]) for b in range(self.n_bands)]

    @property
    def forces(self):
        """Per band [n, n_atoms, 3]: the NEB forces the optimiser steps with (zero for fixed atoms)."""
        return self._interior(self.master['force'])

    @property
    def true_forces(self):
        """Per band [n, n_atoms, 3]: the model forces of the interior images (zero for fixed atoms)."""
        f = self.master['true_force'].masked_fill(self.master['fixed'][:, None], 0.0)
        return self._interior(f)

    @property
    def imax(self):
        """Per band: index in 1..n of the highest interior image (the climbing image when climb is on)."""
        return self.master['imax'].cpu().numpy().astype(np.int64)

    @property
    def fmax(self):
        """max |F_neb| over each band's interior atoms at the current positions (NaN for a failed band)."""
        return np.where(self.failed, np.nan, np.sqrt(self.master['sf'][:, F2].cpu().numpy()))

    @property
    def converged(self):
        return (self.master['si'][:, CONVERGED].cpu().numpy() != 0) & ~self.failed

    @property
    def failed(self):
        """Bands stopped because the model returned a non-finite energy or force for one of their interior images."""
        return self.master['failed'].cpu().numpy() != 0

    @property
    def nsteps(self):
        """Steps each band has taken, over all run() calls."""
        return self.master['si'][:, STEPS].cpu().numpy().astype(np.int64)

    @property
    def state(self):
        """FIRE state per band: velocities [n, n_atoms, 3], dt, a, Nsteps."""
        sf, si = self.master['sf'].cpu().numpy(), self.master['si'].cpu().numpy()
        return {'v': self._interior(self.master['v']), 'dt': sf[:, DT], 'a': sf[:, A], 'Nsteps': si[:, NSTEPS]}

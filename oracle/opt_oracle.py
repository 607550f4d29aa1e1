"""TEST INFRASTRUCTURE - CPU restatement of the device-resident FIRE optimiser (newtonnet_b200/csrc/md_ops.cu,
nn_fire_step / nn_fire_check).

Only tests/ and tools/bench_relax.py (its host-loop leg) may import this.

What it pins: ASE's FIRE (ase/optimize/fire.py, `FIRE.step`, ASE 3.22 / 3.23, `downhill_check=False`) and the
convergence test of `Optimizer.converged` (ase/optimize/optimize.py: `(forces ** 2).sum(axis=1).max() < fmax ** 2`),
transcribed line for line in numpy fp64 for one system.  ASE is not a dependency of this project and FIRE is a
third-party algorithm (Bitzek et al., PRL 97, 170201 (2006)); this file restates ASE's version of it, with ASE's
parameter names and defaults, so that the device kernels can be compared with it.  `step_batch` runs one step for
every system of a batch, each with its own state, as the device does.
"""
import numpy as np

DEFAULTS = dict(dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1, fdec=0.5, astart=0.1, fa=0.99, a=0.1)


class FIRE:
    """State of one system's FIRE optimiser: v (None before the first step, as in ASE), dt, a, Nsteps."""

    def __init__(self, dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1, fdec=0.5, astart=0.1, fa=0.99, a=0.1):
        self.dt, self.maxstep, self.dtmax, self.Nmin = dt, maxstep, dtmax, Nmin
        self.finc, self.fdec, self.astart, self.fa, self.a = finc, fdec, astart, fa, a
        self.v = None
        self.Nsteps = 0

    def step(self, r, f):
        """FIRE.step: returns the new positions r + dr.  r [n,3] fp64, f [n,3] forces at r (cast to fp64)."""
        f = np.asarray(f, dtype=np.float64)
        if self.v is None:
            self.v = np.zeros((len(r), 3))
        else:
            vf = np.vdot(f, self.v)
            if vf > 0.0:
                self.v = (1.0 - self.a) * self.v + self.a * f / np.sqrt(np.vdot(f, f)) * np.sqrt(np.vdot(self.v, self.v))
                if self.Nsteps > self.Nmin:
                    self.dt = min(self.dt * self.finc, self.dtmax)
                    self.a *= self.fa
                self.Nsteps += 1
            else:
                self.v[:] *= 0.0
                self.a = self.astart
                self.dt *= self.fdec
                self.Nsteps = 0
        self.v += self.dt * f
        dr = self.dt * self.v
        normdr = np.sqrt(np.vdot(dr, dr))
        if normdr > self.maxstep:
            dr = self.maxstep * dr / normdr
        return r + dr


def max_force2(f):
    """max_i sum_c f_ic^2 in fp64 (0 for a system without atoms)."""
    f = np.asarray(f, dtype=np.float64)
    return float((f ** 2).sum(axis=1).max()) if len(f) else 0.0


def converged(f, fmax):
    """Optimizer.converged: strictly below fmax."""
    return max_force2(f) < fmax ** 2


def step_batch(opts, r, f, batch, fixed=None):
    """One FIRE step of every system b of the batch (opts[b] its optimiser).  Fixed atoms' forces are zero (ASE's
    FixAtoms.adjust_forces).  A system whose forces are converged already is left as it is; `fmax` is not known here,
    so the caller passes only the optimisers to step: opts[b] = None skips system b.  Returns the new positions."""
    f = np.array(f, dtype=np.float64)
    if fixed is not None:
        f[np.asarray(fixed, dtype=bool)] = 0.0
    out = np.array(r, dtype=np.float64)
    for b, opt in enumerate(opts):
        if opt is None:
            continue
        m = batch == b
        out[m] = opt.step(out[m], f[m])
    return out


def relax(opts, r, batch, forces, fmax, steps, fixed=None):
    """Host loop of an ASE optimiser run per system: `forces(r)` gives fp forces [N,3] of the whole batch; every system
    steps until it is converged (checked before each step) or `steps` steps have been taken.  Returns (r, nsteps [B],
    history: per step a list of (dt, a, Nsteps) per system, None for a system that did not step)."""
    r = np.array(r, dtype=np.float64)
    B = len(opts)
    fixed = np.zeros(len(r), bool) if fixed is None else np.asarray(fixed, dtype=bool)
    nsteps = np.zeros(B, dtype=np.int64)
    history = []
    f = np.array(forces(r), dtype=np.float64)
    f[fixed] = 0.0
    for _ in range(steps):
        active = [opts[b] if not converged(f[batch == b], fmax) else None for b in range(B)]
        if all(o is None for o in active):
            break
        r = step_batch(active, r, f, batch)
        nsteps += np.array([o is not None for o in active])
        history.append([None if o is None else (o.dt, o.a, o.Nsteps) for o in active])
        f = np.array(forces(r), dtype=np.float64)
        f[fixed] = 0.0
    return r, nsteps, history

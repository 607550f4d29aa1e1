"""TEST INFRASTRUCTURE - CPU restatement of the device-resident climbing-image NEB (newtonnet_b200/neb.py,
nn_neb_forces in csrc/neb.cu).

Only tests/ and tools/bench_neb.py (its host-loop leg) may import this.

What it pins: ASE's NEB.get_forces (ase/neb.py, ASE 3.22) with method='improvedtangent' - the improved tangent of
Henkelman & Jonsson, J. Chem. Phys. 113, 9978 (2000) - a scalar spring constant k, and the climbing image of Henkelman,
Uberuaga & Jonsson, J. Chem. Phys. 113, 9901 (2000), transcribed in numpy fp64; and ASE's FIRE(NEB(images)) around it:
one FIRE optimiser (opt_oracle.FIRE) per band, over all interior atoms of the band, with Optimizer.converged on the NEB
forces.  ASE is not a dependency of this project; this file restates ASE's version of the method so that the device
kernels can be compared with it.  The climbing image is the highest interior image, ties going to the highest index.
One deliberate difference: where an image and both neighbours have the same energy, ASE's tangent is zero and its NEB
force NaN; here it is t+ + t-, the limit of the weighted tangent when the two energy differences become equal.
"""
import numpy as np

from oracle import opt_oracle as O


def imax(E):
    """Index of the climbing image in 1..n: the highest interior energy, ties to the highest index."""
    e = np.asarray(E, dtype=np.float64)[1:-1]
    return 1 + int(np.flatnonzero(e == e.max())[-1])


def tangent(R, E, i):
    """Improved tangent of interior image i (unit vector, [n_atoms,3]) and the spring lengths |t+|, |t-|."""
    tp, tm = R[i + 1] - R[i], R[i] - R[i - 1]
    if E[i + 1] > E[i] > E[i - 1]:
        tau = tp.copy()
    elif E[i + 1] < E[i] < E[i - 1]:
        tau = tm.copy()
    else:
        vmax = max(abs(E[i + 1] - E[i]), abs(E[i - 1] - E[i]))
        vmin = min(abs(E[i + 1] - E[i]), abs(E[i - 1] - E[i]))
        if vmax == 0.0:                  # three equal energies: the limit dV_max = dV_min (ASE divides 0 by 0 here)
            vmax = vmin = 1.0
        tau = tp * vmax + tm * vmin if E[i + 1] > E[i - 1] else tp * vmin + tm * vmax
    tau /= np.linalg.norm(tau)
    return tau, np.linalg.norm(tp), np.linalg.norm(tm)


def neb_forces(R, E, F, k, climb, fixed=None):
    """NEB forces of the interior images of one band.  R [n+2, n_atoms, 3] positions (end points included), E [n+2]
    energies, F [n, n_atoms, 3] model forces of the interior images, k > 0, climb: bool; fixed [n_atoms] bool or None
    (their forces count as zero, as under FixAtoms, and their NEB force is zero).  Returns (F_neb [n, n_atoms, 3] fp64,
    imax).  A band whose model output is not finite (an interior energy, or a force of a free atom) has failed: its NEB
    force is zero everywhere, so the optimiser stops it where it is, and imax is None."""
    R = np.asarray(R, dtype=np.float64)
    E = np.asarray(E, dtype=np.float64)
    F = np.array(F, dtype=np.float64)
    if fixed is not None:
        F[:, np.asarray(fixed, dtype=bool)] = 0.0
    if not (np.isfinite(E[1:-1]).all() and np.isfinite(F).all()):
        return np.zeros_like(F), None
    top = imax(E)
    out = np.empty_like(F)
    for i in range(1, len(R) - 1):
        tau, ntp, ntm = tangent(R, E, i)
        f = F[i - 1].copy()
        fpar = np.vdot(f, tau)
        if climb and i == top:
            f -= 2 * fpar * tau
        else:
            f -= fpar * tau
            f += (ntp * k - ntm * k) * tau
        out[i - 1] = f
    if fixed is not None:
        out[:, np.asarray(fixed, dtype=bool)] = 0.0
    return out, top


def relax_bands(bands, ends_energy, forces, fmax, steps, k=0.1, climb=False, fixed=None, opts=None, store=np.float64):
    """Host loop of ASE's FIRE(NEB(band)) for every band at once, one optimiser per band.
    bands: list of [n+2, n_atoms, 3]; ends_energy: list of (E_0, E_{n+1}); forces(list of [n, n_atoms, 3]) -> list of
    (E [n], F [n, n_atoms, 3]) per band; fixed: list of [n_atoms] bool or None; opts: list of opt_oracle.FIRE (new ones
    by default; passing the ones a previous call returned continues that run); store: dtype the NEB forces are rounded to
    before FIRE and the convergence test read them (np.float32 mirrors the device's force buffer).  Every band steps until
    its NEB forces are converged (checked before each step) or `steps` steps have been taken.  Returns (bands, nsteps [B],
    history: per step a list of (dt, a, Nsteps) per band, None for a band that did not step, opts, F_neb per band,
    imax per band)."""
    R = [np.array(b, dtype=np.float64) for b in bands]
    B = len(R)
    fixed = [None] * B if fixed is None else fixed
    opts = [O.FIRE() for _ in range(B)] if opts is None else opts
    nsteps = np.zeros(B, dtype=np.int64)
    history = []

    def project():
        ef = forces([r[1:-1] for r in R])
        out = []
        for b in range(B):
            E = np.concatenate([[ends_energy[b][0]], np.asarray(ef[b][0], dtype=np.float64), [ends_energy[b][1]]])
            f, top = neb_forces(R[b], E, ef[b][1], k, climb, fixed[b])
            out.append((f.astype(store).astype(np.float64), top))
        return out

    fn = project()
    for _ in range(steps):
        active = [not O.converged(fn[b][0].reshape(-1, 3), fmax) for b in range(B)]
        if not any(active):
            break
        for b in range(B):
            if active[b]:
                n = len(R[b]) - 2
                R[b][1:-1] = opts[b].step(R[b][1:-1].reshape(-1, 3), fn[b][0].reshape(-1, 3)).reshape(n, -1, 3)
        nsteps += np.array(active)
        history.append([(o.dt, o.a, o.Nsteps) if a else None for o, a in zip(opts, active)])
        fn = project()
    return R, nsteps, history, opts, [f for f, _ in fn], [t for _, t in fn]

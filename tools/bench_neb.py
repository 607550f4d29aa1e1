"""Time climbing-image NEB on the device (newtonnet_b200.neb.DeviceNEB) against the host loop users run today: the NEB
projection and ASE's FIRE in numpy (oracle/neb_oracle.py restates both) around MLAseCalculator.calculate on the list of
all interior images per step.

    python tools/bench_neb.py [--fmax 0.05] [--max-steps 3000] [--cases aspirin1,aspirin64,aspirin512,water81] > out.jsonl

Cases, 7 interior images per band, climb on, k = 0.1: aspirin bands between a relaxed MD17 frame and the same frame with
its methyl group turned by 120 degrees and relaxed (interior images: the methyl group turned by equal angles - a straight
line would pull its hydrogens through the rotation axis - plus seeded 0.05 A noise per band, MD17 weights)
as 1, 64 and 512 bands; one periodic water band (the 81-molecule box of `case_water81_smallL`, relaxed, and the same box
with one molecule moved 0.6 A, relaxed with that molecule's oxygen held; linear interpolation plus the same noise; its
weights).  One JSON line per case: wall time to converge (device: run() after construction, ending in its final host
read; the median of three identical runs after a first, untimed one, all four listed; host: the whole loop after three
warm-up calls of the calculator), steps per band (max and median), ms per graph replay (CUDA events over 50 replays on a
fresh optimiser whose bands are all active) and nn_neb_forces' share of it (20 launches captured in one graph, CUDA
events over 10 replays of it), compactions, bands stopped because the model returned non-finite values on either path,
whether both paths took the same per-band step counts, and the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_relax import _Atoms, _events, _gpu, _model  # noqa: E402
from newtonnet_b200.engine import capture  # noqa: E402

G = os.path.join(ROOT, 'tests', 'golden')
DEV = 'cuda:0'
N_INTERIOR = 7


def _rotate_methyl(x, deg):
    """Aspirin (MD17 atom order) with the methyl hydrogens 18-20 turned by `deg` about the C11 -> C4 axis."""
    x = x.copy()
    axis = (x[4] - x[11]) / np.linalg.norm(x[4] - x[11])
    t = np.deg2rad(deg)
    for h in (18, 19, 20):
        r = x[h] - x[4]
        x[h] = x[4] + r * np.cos(t) + np.cross(axis, r) * np.sin(t) + axis * (axis @ r) * (1 - np.cos(t))
    return x


def _band(a, b, noise, seed, turn=False):
    """[n+2, N, 3] from a to b with seeded noise on the interior images: a straight line, or for the methyl rotation the
    first end point turned by equal angles (a straight line would pull the hydrogens through the rotation axis)."""
    t = np.linspace(0.0, 1.0, N_INTERIOR + 2)
    if turn:
        R = np.stack([a] + [_rotate_methyl(a, 120.0 * s) for s in t[1:-1]] + [b])
    else:
        R = (1 - t[:, None, None]) * a[None] + t[:, None, None] * b[None]
    R[1:-1] += np.random.default_rng(seed).normal(size=R[1:-1].shape) * noise
    return R


def _cases(names):
    from newtonnet_b200.optimize import DeviceFIRE
    kat = np.load(os.path.join(G, 'md17_kat.npz'))
    md17 = dict(np.load(os.path.join(G, 'weights_md17.npz')))
    z = kat['numbers'].astype(np.int64)
    ends = None
    out = []
    for name in names:
        if name.startswith('aspirin'):
            if ends is None:
                x0 = kat['positions'][0].astype(np.float64)
                r = DeviceFIRE(_model(md17), np.tile(z, 2), np.concatenate([x0, _rotate_methyl(x0, 120.0)]),
                               batch=np.repeat([0, 1], 21))
                r.run(fmax=0.005, steps=5000)
                ends = r.positions.reshape(2, 21, 3)
            n = int(name[len('aspirin'):])
            out.append((name, md17, [z] * n, [_band(ends[0], ends[1], 0.05, q, turn=True) for q in range(n)], None))
        elif name == 'water81':
            d = dict(np.load(os.path.join(G, 'case_water81_smallL.npz')))
            w = dict(np.load(os.path.join(G, f'weights_{d["weights"]}.npz')))
            cell = d['cell'][0].astype(np.float64)
            a = d['pos'].astype(np.float64)
            b = a.copy()
            b[3:6] += [0.6, -0.3, 0.4]
            held = np.arange(len(a)) == 3         # the moved molecule's oxygen: otherwise it relaxes back
            r = DeviceFIRE(_model(w), np.tile(d['z'], 2), np.concatenate([a, b]), cell=np.stack([cell, cell]),
                           batch=np.repeat([0, 1], len(a)), fixed=np.concatenate([np.zeros(len(a), bool), held]))
            r.run(fmax=0.005, steps=5000)
            a, b = r.positions.reshape(2, -1, 3)
            out.append((name, w, [d['z'].astype(np.int64)], [_band(a, b, 0.05, 0)], [cell]))
        else:
            raise ValueError(name)
    return out


def device(model, zs, bands, cells, fmax, max_steps):
    from newtonnet_b200.neb import DeviceNEB
    kw = dict(cell=cells, climb=True)
    # replay and kernel timing on a throwaway optimiser whose bands are all active
    probe = DeviceNEB(model, zs, bands, **kw)
    probe.fmax2.fill_(0.0)
    probe._check(probe.work, 0)
    w = probe.work
    _events(w.graph.replay, 5)
    replay_ms = _events(w.graph.replay, 50)
    neb_graph, _, _ = capture(lambda: [probe._neb(w) for _ in range(20)], probe.device)
    neb_graph.replay()
    neb_ms = _events(neb_graph.replay, 10) / 20
    del probe, neb_graph
    walls, regather = [], []
    for _ in range(4):                   # the first run also pays first-use costs of every compacted shape
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt = DeviceNEB(model, zs, bands, **kw)
        spent = [0.0]

        def timed_use(*a, _use=opt._use):          # time spent gathering and recapturing at compactions
            torch.cuda.synchronize()
            s = time.perf_counter()
            _use(*a)
            torch.cuda.synchronize()
            spent[0] += time.perf_counter() - s
        opt._use = timed_use
        t1 = time.perf_counter()
        done = opt.run(fmax=fmax, steps=max_steps)
        t2 = time.perf_counter()
        walls.append(t2 - t1)
        regather.append(spent[0])
    k = 1 + int(np.argsort(walls[1:])[1])           # the median of the three timed runs
    return opt, dict(build_s=round(t1 - t0, 4), wall_s=round(walls[k], 4), wall_s_all=[round(t, 4) for t in walls],
                     compaction_s=round(regather[k], 4), compaction_s_all=[round(t, 4) for t in regather],
                     failed_bands=np.flatnonzero(opt.failed).tolist(),
                     all_converged=bool(done), ms_per_replay=round(replay_ms, 4), neb_kernel_ms=round(neb_ms, 4),
                     neb_share=round(neb_ms / replay_ms, 4), graph_replays=opt.graph_launches,
                     compactions=opt.compactions, kernels_per_step=opt.kernels_per_step)


def host(model, zs, bands, cells, fmax, max_steps, ends_energy):
    from newtonnet_b200.neb import bands_from_inputs
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    from oracle import neb_oracle as N
    from oracle import opt_oracle as O
    calc = MLAseCalculator(model, properties=['energy', 'forces'], device=DEV)
    aligned = bands_from_inputs(zs, bands, cells)
    B = len(aligned)
    R = [r for _, r, _, _ in aligned]
    atoms = [_Atoms(zb, r[i], c, np.any(c != 0, axis=1)) for zb, r, c, _ in aligned for i in range(1, len(r) - 1)]
    opts = [O.FIRE() for _ in range(B)]
    nsteps = np.zeros(B, np.int64)
    failed = np.zeros(B, bool)
    for _ in range(3):                   # the calculator captures its graphed step on the second call of a shape
        calc.calculate(atoms)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(max_steps + 1):
        calc.calculate(atoms)
        e, f = np.asarray(calc.results['energy'], dtype=np.float64).reshape(-1), calc.results['forces'].reshape(-1, 3)
        fneb, i, a = [], 0, 0
        for b in range(B):
            n, na = len(R[b]) - 2, len(aligned[b][0])
            E = np.concatenate([[ends_energy[b][0]], e[i:i + n], [ends_energy[b][1]]])
            fb, top = N.neb_forces(R[b], E, f[a:a + n * na].reshape(n, na, 3), 0.1, True)
            fneb.append(fb.astype(np.float32))
            failed[b] |= top is None
            i, a = i + n, a + n * na
        active = [not O.converged(fneb[b].reshape(-1, 3), fmax) for b in range(B)]
        if not any(active) or nsteps.max() == max_steps:
            break
        k = 0
        for b in range(B):
            n = len(R[b]) - 2
            if active[b]:
                R[b][1:-1] = opts[b].step(R[b][1:-1].reshape(-1, 3), fneb[b].reshape(-1, 3)).reshape(n, -1, 3)
                nsteps[b] += 1
                for q in range(n):
                    atoms[k + q].positions = R[b][1 + q]
            k += n
    return nsteps, time.perf_counter() - t0, failed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--fmax', type=float, default=0.05)
    ap.add_argument('--max-steps', type=int, default=3000)
    ap.add_argument('--cases', default='aspirin1,aspirin64,aspirin512,water81')
    ap.add_argument('--no-host', action='store_true', help='skip the host loop')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_neb.py needs a CUDA device')
    gpu = _gpu()
    for name, weights, zs, bands, cells in _cases(args.cases.split(',')):
        model = _model(weights)
        opt, rec = device(model, zs, bands, cells, args.fmax, args.max_steps)
        rec.update(case=name, bands=len(bands), images_per_band=N_INTERIOR, atoms=int(sum(len(z) * N_INTERIOR for z in zs)),
                   fmax=args.fmax, steps_max=int(opt.nsteps.max()), steps_median=float(np.median(opt.nsteps)))
        if not args.no_host:
            ends = [(e[0], e[-1]) for e in opt.energies]
            n_host, wall, failed = host(model, zs, bands, cells, args.fmax, args.max_steps, ends)
            differ = np.flatnonzero(n_host != opt.nsteps)
            rec.update(host_wall_s=round(wall, 4), speedup=round(wall / rec['wall_s'], 2),
                       host_failed_bands=np.flatnonzero(failed).tolist(),
                       same_step_counts=bool(len(differ) == 0), bands_with_other_step_counts=differ.tolist()[:32],
                       host_steps_of_those=n_host[differ].tolist()[:32], device_steps_of_those=opt.nsteps[differ].tolist()[:32])
        rec.update(gpu)
        print(json.dumps(rec), flush=True)


if __name__ == '__main__':
    main()

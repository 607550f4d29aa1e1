"""Time FIRE relaxations on the device (newtonnet_b200.optimize.DeviceFIRE) against the host loop users run today: ASE's
FIRE in numpy (oracle/opt_oracle.py restates it) around MLAseCalculator.calculate on the whole list of Atoms per step.

    python tools/bench_relax.py [--fmax 0.05] [--max-steps 3000] [--cases aspirin1,aspirin64,aspirin1024,water3000] > out.jsonl

Cases: perturbed aspirin conformers (MD17 frames plus seeded Gaussian noise of 0.05 A, MD17 weights) as 1, 64 and 1,024
molecules; the c3 water box (3,000 atoms, fixed cell, `case_water375` weights).  One JSON line per case: wall time to
converge (device: run() after construction, ending in its final host read, second of two identical relaxations, the
first one's time beside it; host: the whole loop after three warm-up calls of the calculator), steps taken (max and
median over systems), ms per graph replay and the FIRE kernels' share of it (CUDA events over 50 launches each, on a
fresh optimiser whose systems are all active), compactions, whether both paths took the same per-system step counts,
and the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
G = os.path.join(ROOT, 'tests', 'golden')
DEV = 'cuda:0'


def _gpu():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unavailable'
    return {'gpu': name, 'power_limit_and_max_sm_clock': q}


class _Atoms:
    """The part of ase.Atoms MLAseCalculator reads (ASE is not a dependency)."""

    def __init__(self, numbers, positions, cell, pbc):
        self.numbers, self.positions, self.cell, self.pbc = numbers, np.array(positions, dtype=np.float64), cell, pbc

    def __len__(self):
        return len(self.numbers)

    def get_atomic_numbers(self):
        return self.numbers

    def get_positions(self, wrap=False):
        if wrap and self.pbc.any():
            frac = np.linalg.solve(self.cell.T, self.positions.T).T
            return (frac % 1.0) @ self.cell
        return self.positions

    def get_cell(self):
        return self.cell

    def get_pbc(self):
        return self.pbc


def _model(weights):
    from newtonnet_b200.compat import model_from_state_dict
    m = model_from_state_dict({k: torch.tensor(v) for k, v in weights.items()}, output_properties=['energy', 'gradient_force'])
    return m.to(DEV).eval()


def _cases(names):
    from newtonnet_b200 import workloads
    kat = np.load(os.path.join(G, 'md17_kat.npz'))
    md17 = dict(np.load(os.path.join(G, 'weights_md17.npz')))
    out = []
    for name in names:
        if name.startswith('aspirin'):
            n = int(name[len('aspirin'):])
            frames = kat['positions'][(np.arange(n) * 7) % len(kat['positions'])].astype(np.float64)
            frames += np.random.default_rng(n).normal(size=frames.shape) * 0.05
            out.append((name, md17, np.tile(kat['numbers'], n).astype(np.int64), frames.reshape(-1, 3),
                        np.zeros((n, 3, 3)), np.repeat(np.arange(n), 21)))
        elif name == 'water3000':
            w375 = dict(np.load(os.path.join(G, 'case_water375.npz')))
            ws = dict(np.load(os.path.join(G, f'weights_{w375["weights"]}.npz')))
            z, pos, cell, batch = workloads.water_box(10, seed=0)
            out.append((name, ws, z, pos.astype(np.float64), cell.astype(np.float64), batch))
        else:
            raise ValueError(name)
    return out


def _events(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def device(model, z, pos, cell, batch, fmax, max_steps):
    from newtonnet_b200.optimize import DeviceFIRE
    # replay and kernel timing on a throwaway optimiser whose systems are all active
    probe = DeviceFIRE(model, z, pos, cell=cell, batch=batch)
    probe.fmax2.fill_(0.0)
    probe._check(0)
    w = probe.work
    _events(w.graph.replay, 5)
    replay_ms = _events(w.graph.replay, 50)
    fire_ms = _events(lambda: (probe._fire_step(), probe._check(1)), 50)
    del probe
    walls, regather = [], []
    for _ in range(2):                   # the first relaxation also pays first-use costs of every compacted shape
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt = DeviceFIRE(model, z, pos, cell=cell, batch=batch)
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
    return opt, dict(build_s=round(t1 - t0, 4), wall_s=round(walls[1], 4), wall_s_first=round(walls[0], 4),
                     compaction_s=round(regather[1], 4), compaction_s_first=round(regather[0], 4),
                     all_converged=bool(done),
                     ms_per_replay=round(replay_ms, 4), fire_kernels_ms=round(fire_ms, 4),
                     fire_share=round(fire_ms / replay_ms, 4), graph_replays=opt.graph_launches, compactions=opt.compactions,
                     kernels_per_step=opt.kernels_per_step)


def host(model, z, pos, cell, batch, fmax, max_steps):
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    from oracle import opt_oracle as O
    B = cell.shape[0]
    calc = MLAseCalculator(model, properties=['energy', 'forces'], device=DEV)
    pbc = [np.any(cell[b] != 0, axis=1) for b in range(B)]
    atoms = [_Atoms(z[batch == b], pos[batch == b], cell[b], pbc[b]) for b in range(B)]
    opts = [O.FIRE() for _ in range(B)]
    nsteps = np.zeros(B, np.int64)
    for _ in range(3):                   # the calculator captures its graphed step on the second call of a shape
        calc.calculate(atoms if B > 1 else atoms[0])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(max_steps + 1):
        calc.calculate(atoms if B > 1 else atoms[0])
        f = calc.results['forces'].reshape(B, -1, 3)
        active = [not O.converged(f[b], fmax) for b in range(B)]
        if not any(active) or nsteps.max() == max_steps:
            break
        for b in range(B):
            if active[b]:
                atoms[b].positions = opts[b].step(atoms[b].positions, f[b])
                nsteps[b] += 1
    return nsteps, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--fmax', type=float, default=0.05)
    ap.add_argument('--max-steps', type=int, default=3000)
    ap.add_argument('--cases', default='aspirin1,aspirin64,aspirin1024,water3000')
    ap.add_argument('--no-host', action='store_true', help='skip the host loop')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_relax.py needs a CUDA device')
    gpu = _gpu()
    for name, weights, z, pos, cell, batch in _cases(args.cases.split(',')):
        model = _model(weights)
        opt, rec = device(model, z, pos, cell, batch, args.fmax, args.max_steps)
        rec.update(case=name, systems=int(cell.shape[0]), atoms=int(len(z)), fmax=args.fmax,
                   steps_max=int(opt.nsteps.max()), steps_median=float(np.median(opt.nsteps)))
        if not args.no_host:
            n_host, wall = host(model, z, pos, cell, batch, args.fmax, args.max_steps)
            differ = np.flatnonzero(n_host != opt.nsteps)
            rec.update(host_wall_s=round(wall, 4), speedup=round(wall / rec['wall_s'], 2),
                       same_step_counts=bool(len(differ) == 0), systems_with_other_step_counts=differ.tolist()[:32],
                       host_steps_of_those=n_host[differ].tolist()[:32], device_steps_of_those=opt.nsteps[differ].tolist()[:32])
        rec.update(gpu)
        print(json.dumps(rec), flush=True)


if __name__ == '__main__':
    main()

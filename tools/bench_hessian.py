"""Time one Hessian three ways: the per-row loop (train.hessian_rows: one second backward over the whole batch per row),
the block path run eagerly (NN_HESSIAN_GRAPH=0) and the block path replayed as CUDA graphs (default).

    python tools/bench_hessian.py [--runs 7] [--budgets 1024,4096,8192] > out.jsonl

Cases: aspirin (21 atoms, MD17 weights), a batch of 4 aspirin frames, the 81-atom periodic water box (case_water81_smallL).
Every time is the median of --runs calls after a warm-up call, between CUDA events, each call ending in the copy of the
result to a fresh tensor (the block path) or the stacked rows (the per-row loop).  One JSON line per case and mode, with
the rows per pass (k), the passes, the peak device memory of the call over its replicated atoms, and the GPU's name and
power limit.  --budgets also times the graphed path of each case at those NN_HESSIAN_ATOMS values."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
G = os.path.join(ROOT, 'tests', 'golden')


def _gpu():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unavailable'
    return {'gpu': name, 'power_limit_and_max_sm_clock': q}


def _cases():
    kat = np.load(os.path.join(G, 'md17_kat.npz'))
    md17 = dict(np.load(os.path.join(G, 'weights_md17.npz')))
    z = kat['numbers'].astype(np.int64)
    one = dict(z=z, pos=kat['positions'][0].astype(np.float32), cell=np.zeros((1, 3, 3), np.float32), batch=np.zeros(21, np.int64))
    four = dict(z=np.tile(z, 4), pos=kat['positions'][:4].reshape(-1, 3).astype(np.float32), cell=np.zeros((4, 3, 3), np.float32),
                batch=np.repeat(np.arange(4), 21))
    w81 = dict(np.load(os.path.join(G, 'case_water81_smallL.npz')))
    ws = dict(np.load(os.path.join(G, f'weights_{w81["weights"]}.npz')))
    return [('aspirin', md17, one), ('aspirin_x4', md17, four), ('water81_smallL', ws, w81)]


def _time(fn, runs):
    fn()                                                    # warm-up: captures, lazy initialisation
    torch.cuda.synchronize()
    ms = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), [round(x, 3) for x in ms]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--runs', type=int, default=7)
    ap.add_argument('--budgets', default='')
    ap.add_argument('--skip-per-row', action='store_true')
    args = ap.parse_args()
    from newtonnet_b200.compat import model_from_state_dict
    from newtonnet_b200 import hessian
    from newtonnet_b200.hessian import default_budget, plan_passes, stats
    from newtonnet_b200.train import _skip_weight_grads, differentiable_forward, hessian_rows
    dev = torch.device('cuda:0')
    info = _gpu()
    for name, w, d in _cases():
        model = model_from_state_dict({k: torch.tensor(v) for k, v in w.items()}).to(dev).eval()
        t = lambda a, dt: torch.as_tensor(np.asarray(a), device=dev, dtype=dt)
        z, pos, cell, batch = t(d['z'], torch.int64), t(d['pos'], torch.float32), t(d['cell'], torch.float32), t(d['batch'], torch.int64)
        sizes = np.bincount(d['batch'])

        def per_row():
            p = pos.clone().requires_grad_(True)
            out = differentiable_forward(model, z, p, cell, batch, properties=('energy',))
            with _skip_weight_grads():
                g, = torch.autograd.grad(out.energy, p, torch.ones_like(out.energy), create_graph=True)
            return hessian_rows(g, p)

        def block():
            return hessian(model, z, pos, cell, batch)

        modes = [] if args.skip_per_row else [('per_row', None, None)]
        modes += [('block_eager', '0', None), ('block_graph', '1', None)]
        modes += [('block_graph', '1', b) for b in args.budgets.split(',') if b]
        ref = None
        for mode, graph, budget in modes:
            os.environ['NN_HESSIAN_GRAPH'] = graph or '1'
            if budget:
                os.environ['NN_HESSIAN_ATOMS'] = budget
            else:
                os.environ.pop('NN_HESSIAN_ATOMS', None)
            fn = per_row if mode == 'per_row' else block
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats(dev)
            base = torch.cuda.memory_allocated(dev)
            caps0, passes0 = stats['captures'], stats['passes']
            med, all_ms = _time(fn, args.runs)
            peak = torch.cuda.max_memory_allocated(dev) - base
            H = fn()
            torch.cuda.synchronize()
            ref = H if ref is None else ref
            row = dict(case=name, mode=mode, atoms=int(len(d['z'])), rows=int(3 * len(d['z'])), ms=round(med, 3), runs_ms=all_ms,
                       equal_to_first_mode=bool(torch.equal(H, ref)))
            if mode != 'per_row':
                bud = default_budget(dev)
                groups, _ = plan_passes(sizes, budget=bud)
                rep = max(g.k * g.n for g in groups)
                row.update(budget=bud, rows_per_pass=[g.k for g in groups], passes=sum(g.n_pass for g in groups),
                           captures=stats['captures'] - caps0, passes_run=stats['passes'] - passes0,
                           peak_bytes=int(peak), peak_bytes_per_replicated_atom=int(peak / rep))
            else:
                row.update(passes=int(3 * len(d['z'])), peak_bytes=int(peak))
            row.update(info)
            print(json.dumps(row), flush=True)
        os.environ.pop('NN_HESSIAN_ATOMS', None)
        os.environ.pop('NN_HESSIAN_GRAPH', None)


if __name__ == '__main__':
    main()

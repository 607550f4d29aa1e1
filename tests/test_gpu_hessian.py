"""Hessians in batched blocks of rows (newtonnet_b200/hessian.py, csrc/hessian.cu) against the per-row loop
(train.hessian_rows), the golden of the unmodified reference and the fp64 oracle.

Each row of the block path is expected to be bit-identical to the row of the per-row loop: a pass evaluates k independent
copies of frames, and every primitive of the differentiable path treats rows independently or sums over per-system
segments in a fixed order.  So block vs per-row, block sizes against each other, graph vs eager and a frame in a batch vs
the frame alone are compared with torch.equal.

Against the fp64 oracle the rule of test_gpu_fwd_ops.py is used, |got - ref| <= c * 2^-24 * mag, with mag = the largest
|entry| of the frame's fp64 Hessian: every entry is a sum of second-derivative terms of that order, through three
interaction layers of fp32 arithmetic (3xTF32 contractions, fp32 segment sums of up to ~60 neighbours, SiLU'' and the
radial basis' second derivative).  Measured on a B200: at most 130 (aspirin 73, water81_smallL 123, mols_edge frames
69-130); C_HESS = 512 leaves a factor 4 for other GEMM back-ends and GPUs.  Each test prints its worst ratio.
"""
import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_case, load_weights

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
U = 2.0 ** -24
C_HESS = 512


def _model(weights, props=('energy', 'gradient_force')):
    from newtonnet_b200.compat import model_from_state_dict
    m = model_from_state_dict({k: torch.tensor(v) for k, v in weights.items()}, output_properties=list(props)).to(DEV)
    m.eval()
    return m


def _t(a, dt=None):
    return torch.as_tensor(np.asarray(a), device=DEV) if dt is None else torch.as_tensor(np.asarray(a), device=DEV, dtype=dt)


def _inputs(d):
    return _t(d['z'], torch.int64), _t(d['pos'], torch.float32), _t(d['cell'], torch.float32), _t(d['batch'], torch.int64)


def _aspirin():
    d = np.load(f'{GOLDEN}/hessian_aspirin1.npz')
    return dict(z=d['z'], pos=d['pos'], cell=np.zeros((1, 3, 3), np.float32), batch=np.zeros(21, np.int64)), d['hessian']


def _block(model, d, atoms=None):
    from newtonnet_b200 import hessian
    out = hessian(model, *_inputs(d), atoms=atoms)
    torch.cuda.synchronize()
    return out


def _per_row(model, d):
    """The per-row loop as the hessian head ran it: pos_grad with create_graph, then one reverse pass per row."""
    from newtonnet_b200.train import _skip_weight_grads, differentiable_forward, hessian_rows
    z, pos, cell, batch = _inputs(d)
    pos = pos.clone().requires_grad_(True)
    out = differentiable_forward(model, z, pos, cell, batch, properties=('energy',))
    with _skip_weight_grads():
        g, = torch.autograd.grad(out.energy, pos, torch.ones_like(out.energy), create_graph=True, retain_graph=True)
    return hessian_rows(g, pos)


def _oracle(w, d):
    from oracle import newtonnet_oracle as O
    return O.hessian(w, d['z'], d['pos'], d['cell'], d['batch'])


def _within_oracle(got, ref, what):
    got = got.detach().cpu().double().numpy()
    mag = np.abs(ref).max()
    err = np.abs(got - ref).max()
    ratio = err / (U * mag)
    print(f'{what}: max |H - oracle| = {err:.3e}, max |H| = {mag:.3e}, {ratio:.0f} * 2^-24 * mag')
    assert ratio <= C_HESS, f'{what}: {ratio:.0f} * 2^-24 * mag > {C_HESS}'


def _frame(d, b):
    sel = d['batch'] == b
    return dict(z=d['z'][sel], pos=d['pos'][sel], cell=d['cell'][b:b + 1], batch=np.zeros(int(sel.sum()), np.int64))


def test_aspirin_matches_per_row_golden_and_oracle():
    w = load_weights('md17')
    d, golden = _aspirin()
    model = _model(w)
    H = _block(model, d)
    assert H.shape == (21, 3, 21, 3) and H.dtype == torch.float32
    assert torch.equal(H, _per_row(model, d))
    assert np.abs(H.cpu().numpy() - golden).max() < 2e-3 and np.abs(golden).max() > 50
    _within_oracle(H, _oracle(w, d), 'aspirin')


@pytest.mark.parametrize('budget,k,padded', [(21, 1, False), (147, 7, False), (1323, 63, False), (168, 8, True)])
def test_block_size_invariance(monkeypatch, budget, k, padded):
    from newtonnet_b200.hessian import plan_passes
    w = load_weights('md17')
    d, _ = _aspirin()
    model = _model(w)
    g, = plan_passes([21], budget=budget)[0]
    assert g.k == k and bool((g.plan[:, :, 1] < 0).any()) == padded
    ref = _block(model, d)                                  # default budget: one pass of 63 rows
    monkeypatch.setenv('NN_HESSIAN_ATOMS', str(budget))
    assert torch.equal(_block(model, d), ref)


def test_ragged_batch():
    d, w = load_case('mols_edge')
    model = _model(w)
    H = _block(model, d)
    N = d['z'].shape[0]
    assert H.shape == (N, 3, N, 3)
    assert torch.equal(H, _per_row(model, d))
    Hc = H.cpu()
    ptr = np.concatenate([[0], np.cumsum(np.bincount(d['batch']))])
    for b in range(len(ptr) - 1):
        lo, hi = int(ptr[b]), int(ptr[b + 1])
        rows = Hc[lo:hi]
        assert torch.count_nonzero(rows[:, :, :lo]) == 0 and torch.count_nonzero(rows[:, :, hi:]) == 0   # cross-frame blocks
        f = _frame(d, b)
        assert torch.equal(rows[:, :, lo:hi], _block(model, f).cpu()), f'frame {b} in the batch != frame {b} alone'
        if hi - lo > 1:
            _within_oracle(rows[:, :, lo:hi], _oracle(w, f), f'mols_edge frame {b} ({hi - lo} atoms)')


def test_periodic_small_box_against_oracle():
    d, w = load_case('water81_smallL')                     # L = 9.3 A < 2 r_c: an atom sees several images of a neighbour
    model = _model(w)
    H = _block(model, d)
    assert torch.equal(H, _per_row(model, d))
    _within_oracle(H, _oracle(w, d), 'water81_smallL')


def test_selected_atoms_are_rows_of_the_full_hessian():
    d, w = load_case('mols_edge')
    model = _model(w)
    full = _block(model, d)
    atoms = [0, 1, 2, 70, 156, 3]                          # across frames, out of order
    part = _block(model, d, atoms=atoms)
    assert part.shape == (len(atoms), 3) + full.shape[2:]
    assert torch.equal(part, full[atoms])
    da, _ = _aspirin()
    ma = _model(load_weights('md17'))
    assert torch.equal(_block(ma, da, atoms=[20, 5]), _block(ma, da)[[20, 5]])


def test_graph_eager_reuse_and_overflow(monkeypatch):
    from newtonnet_b200.hessian import stats
    w = load_weights('md17')
    d, _ = _aspirin()
    model = _model(w)

    def eager(dd):
        monkeypatch.setenv('NN_HESSIAN_GRAPH', '0')
        try:
            return _block(model, dd)
        finally:
            monkeypatch.delenv('NN_HESSIAN_GRAPH')

    g0 = _block(model, d)
    assert torch.equal(g0, eager(d))
    # the same molecule at new positions replays the cached graph
    moved = dict(d, pos=d['pos'] + np.random.default_rng(0).normal(0, 0.02, d['pos'].shape).astype(np.float32))
    caps = stats['captures']
    g1 = _block(model, moved)
    assert stats['captures'] == caps
    assert torch.equal(g1, eager(moved)) and not torch.equal(g1, g0)
    # compressed to 55 %: every pair within the cutoff, more edges than the captured capacity -> recapture with more room
    dense = dict(d, pos=(d['pos'] - d['pos'].mean(0)) * np.float32(0.55))
    g2 = _block(model, dense)
    assert stats['captures'] > caps
    assert torch.equal(g2, eager(dense))
    assert torch.isfinite(g2).all() and torch.count_nonzero(g2) > 0


def test_training_mode_keeps_the_per_row_loop():
    from newtonnet_b200.hessian import stats
    from newtonnet_b200.train import hessian_rows
    w = load_weights('md17')
    d, _ = _aspirin()
    model = _model(w, ('energy', 'gradient_force', 'hessian'))
    model.train()                                           # create_graph on every derivative head
    assert model.output_layers[2].create_graph
    passes = stats['passes']
    z, pos, cell, batch = _inputs(d)
    pos = pos.clone().requires_grad_(True)
    out = model(z, pos, cell, batch)
    assert stats['passes'] == passes                        # no block pass ran
    assert out.gradient_force.grad_fn is not None
    assert torch.equal(out.hessian, hessian_rows(out.pos_grad, pos))
    # eval mode with create_graph heads (what MLAseCalculator sets up): the block path, same values
    model.eval()
    for layer in model.output_layers[1:]:
        layer.create_graph = True
    out2 = model(z, pos.detach().clone(), cell, batch)
    assert stats['passes'] > passes
    assert out2.hessian.shape == (21, 3, 21, 3) and out2.hessian.grad_fn is None
    assert torch.equal(out2.hessian, out.hessian)


def test_evicted_graphs_are_freed_without_the_cyclic_collector():
    """A cached Hessian shape that the cache evicts must free its CUDA graphs at once, by reference count: left to the
    cyclic collector, the graphs would be destroyed whenever it runs, possibly in the middle of a later capture."""
    import gc
    import weakref
    from newtonnet_b200.hessian import _CACHE_SIZE, _cache
    d, _ = _aspirin()
    model = _model(load_weights('md17'))
    was = gc.isenabled()
    gc.disable()
    try:
        refs = []
        for i in range(_CACHE_SIZE + 1):                   # distinct selections: distinct cache entries
            _block(model, d, atoms=[i])
            refs.append(weakref.ref(list(_cache.values())[-1]))
        assert refs[0]() is None, 'an evicted entry is kept alive by a reference cycle'
        assert all(r() is not None for r in refs[1:])
    finally:
        if was:
            gc.enable()

"""Host plumbing the drivers share (newtonnet_b200/engine.py): capacity policy, all-pairs bound, graph capture."""
import contextlib
import gc
from types import SimpleNamespace

import pytest
import torch

from newtonnet_b200 import _lib as L
from newtonnet_b200.distributed import DomainDecomposition, _PeerStep
from newtonnet_b200.engine import Engine, _gc_paused, all_pairs_bound, capture, edge_capacity
from newtonnet_b200.hessian import _GroupRunner
from newtonnet_b200.md import DeviceMD
from newtonnet_b200.train import GraphedTrainingStep

EDGES = [0, 1, 7, 8, 30_209, 12_345_678]          # zero, one, odd, even, a c5 batch, large
BOUNDS = [0, 2, 5, 100, 31_000, 10 ** 9, None]    # None: a periodic batch


# the capacity formulas as each driver wrote them before they shared edge_capacity
def _engine(n):
    cap = int(n * 1.08) + 64
    cap += cap % 2
    return cap


def _md(n):
    cap = int(n * 1.15) + 64
    cap += cap % 2
    return cap


def _training_headroom(n, bound):
    cap = int(n * 1.05) + 256
    if bound is not None:
        cap = min(cap, bound)
    return cap


def _training(cap_edges):                          # what _capture made of the capacity it was given
    return max(int(cap_edges) + int(cap_edges) % 2, 2)


def _hessian(n, bound):
    cap = int(n * 1.05) + 256
    if bound is not None:
        cap = min(cap, bound)
    return max(cap + cap % 2, 2)


def _peer_fresh(n):
    cap = int(n * 1.08) + 64
    return cap + cap % 2


def _peer_reused(cap, g):
    c = int(cap * g) + 64
    return c + c % 2


def _eager_dd(n):
    cap = int(n * 1.08) + 64
    return cap + cap % 2


def _runner(bound):
    return SimpleNamespace(HEADROOM=_GroupRunner.HEADROOM, bound=bound)


def _training_step(periodic):                      # 100 molecules of 21 atoms
    cell = torch.eye(3).repeat(100, 1, 1) * 20.0 if periodic else torch.zeros(100, 3, 3)
    return SimpleNamespace(HEADROOM=GraphedTrainingStep.HEADROOM, cell=cell, batch=torch.arange(100).repeat_interleave(21))


@pytest.mark.parametrize('n', EDGES)
def test_edge_capacity_matches_every_driver(n):
    assert edge_capacity(n, *Engine.HEADROOM) == _engine(n)
    assert edge_capacity(n, *DeviceMD.HEADROOM) == _md(n)
    assert edge_capacity(n, *_PeerStep.HEADROOM) == _peer_fresh(n)
    assert edge_capacity(n, *DomainDecomposition.HEADROOM) == _eager_dd(n)
    for g in (1.02, 1.02 * 1.37):
        assert edge_capacity(n, g, 64) == _peer_reused(n, g)
    for bound in BOUNDS:
        assert edge_capacity(n, *GraphedTrainingStep.HEADROOM, bound) == _training(_training_headroom(n, bound))
        assert _GroupRunner._capacity(_runner(bound), n) == _hessian(n, bound)
    for periodic, bound in ((True, None), (False, 100 * 21 * 20)):
        assert GraphedTrainingStep._capacity(_training_step(periodic), n) == _training(_training_headroom(n, bound))
    assert edge_capacity(n, 1, 0) == _training(n)  # a capacity given to GraphedTrainingStep


@pytest.mark.parametrize('need', EDGES)
@pytest.mark.parametrize('cap', [2, 8, 31_000, 40_000])
def test_regrow_rule_matches_every_driver(need, cap):
    """After an overflow, training and the Hessian take max(capacity for the need, old capacity + 2)."""
    for bound in BOUNDS:
        assert max(_GroupRunner._capacity(_runner(bound), need), cap + 2) == max(_hessian(need, bound), cap + 2)
        assert (max(edge_capacity(need, *GraphedTrainingStep.HEADROOM, bound), cap + 2)
                == _training(max(_training_headroom(need, bound), cap + 2)))


def test_all_pairs_bound():
    batch = torch.tensor([0, 0, 0, 1, 1, 3, 3, 3, 3])
    cell = torch.zeros(4, 3, 3)
    n = torch.bincount(batch, minlength=4)
    assert all_pairs_bound(cell, batch) == int((n * (n - 1)).sum()) == 3 * 2 + 2 * 1 + 0 + 4 * 3
    cell[2, 1, 1] = 5.0                            # one periodic system: no bound
    assert all_pairs_bound(cell, batch) is None
    k, n = 6, 21                                   # the Hessian's replicated batch: k copies of an n-atom frame
    assert all_pairs_bound(torch.zeros(1, 3, 3), torch.arange(k).repeat_interleave(n)) == k * n * (n - 1)


def test_gc_paused_restores_the_collector_state():
    was = gc.isenabled()
    try:
        for before in (True, False):
            (gc.enable if before else gc.disable)()
            with _gc_paused():
                assert not gc.isenabled()
            assert gc.isenabled() == before
    finally:
        (gc.enable if was else gc.disable)()


def test_capture_with_fakes(monkeypatch):
    """capture(): synchronise, then capture fn() with the collector off; the launch count is a delta, never reset."""
    events = []

    class FakeLib:
        launches = 1000

        def nn_launch_count(self, reset):
            events.append(('count', reset))
            return self.launches

    class FakeGraph:
        pass

    @contextlib.contextmanager
    def fake_graph(graph, pool=None):
        events.append(('begin', graph, pool))
        yield
        events.append(('end', graph))

    lib = FakeLib()
    monkeypatch.setattr(L, 'load', lambda: lib)
    monkeypatch.setattr(torch.cuda, 'CUDAGraph', FakeGraph)
    monkeypatch.setattr(torch.cuda, 'graph', fake_graph)
    monkeypatch.setattr(torch.cuda, 'synchronize', lambda device=None: events.append(('sync', device)))

    def fn():
        events.append(('fn', gc.isenabled()))
        lib.launches += 37
        return 'loss'

    def failing():
        events.append(('fn', gc.isenabled()))
        raise ValueError('inside the capture')

    was = gc.isenabled()
    try:
        for before in (True, False):
            (gc.enable if before else gc.disable)()
            events.clear()
            graph, result, kernels = capture(fn, 'cuda:3', pool='pool')
            assert isinstance(graph, FakeGraph) and result == 'loss' and kernels == 37
            assert events == [('sync', 'cuda:3'), ('count', 0), ('begin', graph, 'pool'), ('fn', False), ('end', graph),
                              ('count', 0)]
            assert gc.isenabled() == before
            events.clear()
            with pytest.raises(ValueError, match='inside the capture'):
                capture(failing, 'cuda:0')
            assert events[0] == ('sync', 'cuda:0') and ('fn', False) in events
            assert gc.isenabled() == before
    finally:
        (gc.enable if was else gc.disable)()

"""Planner of the block Hessian (newtonnet_b200/hessian.py: plan_passes), on the host: which rows go into which pass."""
import numpy as np
import pytest

from newtonnet_b200.hessian import plan_passes

SIZES = [
    [21],
    [21, 21, 21, 21],
    [1, 2, 64, 3, 1, 17, 64, 5],          # case_mols_edge: ragged, with 1- and 2-atom molecules
    [81],
    [0, 4, 0, 7],                         # empty systems plan no rows
]


def _jobs(groups):
    """All real jobs as (frame, local row, output row), and every job with its group."""
    real, every = [], []
    for g in groups:
        for job in g.plan.reshape(-1, 3).tolist():
            every.append((g, job))
            if job[1] >= 0:
                real.append(tuple(job))
    return real, every


def _expected(sizes, atoms):
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    sel = range(int(ptr[-1])) if atoms is None else atoms
    out = []
    for m, i in enumerate(sel):
        f = int(np.searchsorted(ptr, i, side='right') - 1)
        out += [(f, 3 * (i - int(ptr[f])) + d, 3 * m + d) for d in range(3)]
    return out


@pytest.mark.parametrize('sizes', SIZES)
@pytest.mark.parametrize('budget', [1, 5, 21, 100, 147, 1000, 10 ** 6])
def test_every_row_exactly_once(sizes, budget):
    groups, n_rows = plan_passes(sizes, budget=budget)
    real, _ = _jobs(groups)
    assert n_rows == 3 * sum(sizes)
    assert sorted(real) == sorted(_expected(sizes, None))
    assert sorted(j[2] for j in real) == list(range(n_rows))        # each output row once


@pytest.mark.parametrize('sizes', SIZES[:3])
def test_selected_atoms(sizes):
    N = sum(sizes)
    rng = np.random.default_rng(sum(sizes))
    atoms = rng.choice(N, size=min(N, 5), replace=False).tolist()
    groups, n_rows = plan_passes(sizes, atoms=atoms, budget=50)
    real, _ = _jobs(groups)
    assert n_rows == 3 * len(atoms)
    assert sorted(real) == sorted(_expected(sizes, atoms))


@pytest.mark.parametrize('sizes', SIZES)
@pytest.mark.parametrize('budget', [1, 5, 21, 100, 147, 1000])
def test_budget_and_group_shape(sizes, budget):
    groups, _ = plan_passes(sizes, budget=budget)
    for g in groups:
        assert g.plan.dtype == np.int32 and g.plan.shape == (g.n_pass, g.k, 3)
        assert all(sizes[f] == g.n for f in g.plan[:, :, 0].reshape(-1))     # one atom count per group
        if g.n <= budget:
            assert g.k * g.n <= budget
        else:
            assert g.k == 1                                                 # an oversized frame still runs, alone
        assert len({g.n for g in groups}) == len(groups)
        # the least pass count the budget allows
        jobs = int((g.plan[:, :, 1] >= 0).sum())
        k_max = max(min(budget // max(g.n, 1), jobs), 1)
        assert g.n_pass == -(-jobs // k_max)


def test_oversized_frame_runs_alone():
    groups, _ = plan_passes([81, 2], budget=50)
    big = [g for g in groups if g.n == 81][0]
    assert big.k == 1 and big.n_pass == 243
    small = [g for g in groups if g.n == 2][0]
    assert small.k == 6 and small.n_pass == 1


def test_padding_jobs_are_marked_and_last():
    groups, _ = plan_passes([21], budget=168)          # at most 8 rows per pass: 63 rows -> 8 passes of 8, one padding job
    g, = groups
    assert (g.k, g.n_pass) == (8, 8)
    pad = g.plan[:, :, 1] < 0
    assert int(pad.sum()) == 1 and bool(pad[-1, -1])
    assert (g.plan[pad][:, 2] == -1).all()             # padding writes no output row
    assert (g.plan[pad][:, 0] == 0).all()              # ... and copies a frame of the group
    for budget in (21, 147, 1323):                     # 1, 7, 63 rows per pass: no padding
        g, = plan_passes([21], budget=budget)[0]
        assert g.k == budget // 21 and not (g.plan[:, :, 1] < 0).any()


def test_jobs_mix_frames_of_one_size():
    groups, _ = plan_passes([21, 21, 21, 21], budget=21 * 100)
    g, = groups
    assert g.n_pass == 3 and g.k == 84
    assert len(set(g.plan[0, :, 0].tolist())) == 2     # the first pass holds rows of frames 0 and 1


def test_bad_selection():
    with pytest.raises(IndexError):
        plan_passes([3, 4], atoms=[7])
    with pytest.raises(IndexError):
        plan_passes([3, 4], atoms=[-1])
    with pytest.raises(ValueError):
        plan_passes([3, 4], atoms=[])


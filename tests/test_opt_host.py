"""CPU checks of the FIRE oracle (oracle/opt_oracle.py) on hand-made states, and of DeviceFIRE's compaction plan."""
import numpy as np

from oracle import opt_oracle as O


def _downhill(opt, n=1):
    """Take n steps with the force along v: every step after the first is downhill."""
    r, f = np.zeros((2, 3)), np.array([[1e-3, 0, 0], [0, 2e-3, 0]])
    for _ in range(n):
        r = opt.step(r, f)
    return r


def test_first_step_keeps_dt_and_a():
    opt = O.FIRE()
    r = _downhill(opt)
    assert opt.dt == 0.1 and opt.a == 0.1 and opt.Nsteps == 0
    f = np.array([[1e-3, 0, 0], [0, 2e-3, 0]])
    np.testing.assert_array_equal(opt.v, 0.1 * f)
    np.testing.assert_array_equal(r, 0.1 * (0.1 * f))


def test_dt_and_a_change_only_after_nmin_downhill_steps():
    opt = O.FIRE()
    _downhill(opt, 1 + 6)                     # first step + Nsteps 0..5: none has Nsteps > Nmin
    assert opt.Nsteps == 6 and opt.dt == 0.1 and opt.a == 0.1
    _downhill(opt, 1)
    assert opt.Nsteps == 7 and opt.dt == 0.1 * 1.1 and opt.a == 0.1 * 0.99


def test_dt_capped_at_dtmax():
    opt = O.FIRE()
    _downhill(opt, 60)
    assert opt.dt == 1.0
    opt = O.FIRE(dtmax=0.5)
    _downhill(opt, 60)
    assert opt.dt == 0.5


def test_uphill_step_resets():
    opt = O.FIRE()
    _downhill(opt, 10)
    dt = opt.dt
    f = np.array([[-1e-3, 0, 0], [0, -2e-3, 0]])
    opt.step(np.zeros((2, 3)), f)
    assert opt.a == 0.1 and opt.dt == 0.5 * dt and opt.Nsteps == 0
    np.testing.assert_array_equal(opt.v, opt.dt * f)            # v reset to 0, then v += dt f


def test_maxstep_clips_the_step():
    opt = O.FIRE()
    r0 = np.zeros((3, 3))
    r = opt.step(r0, np.full((3, 3), 50.0))
    assert abs(np.linalg.norm(r - r0) - 0.2) < 1e-15
    opt = O.FIRE(maxstep=0.05)
    r = opt.step(r0, np.full((3, 3), 50.0))
    assert abs(np.linalg.norm(r - r0) - 0.05) < 1e-15
    r = O.FIRE().step(r0, np.full((3, 3), 1e-3))                  # small: not clipped
    np.testing.assert_array_equal(r, 0.1 * (0.1 * np.full((3, 3), 1e-3)))


def test_fmax_is_strict():
    f = np.array([[0.375, 0.5, 0.0], [0.25, 0.0, 0.0]])         # |f_0| = 0.625, every square exact in fp64
    assert O.max_force2(f) == 0.625 ** 2
    assert not O.converged(f, 0.625)
    assert O.converged(f, np.nextafter(0.625, 1.0))
    assert O.converged(np.zeros((2, 3)), 1e-12)


def test_converges_on_a_quadratic_well():
    k = np.array([1.0, 4.0, 9.0])
    center = np.array([[0.3, -0.2, 0.1], [1.0, 2.0, -1.0]])
    r0 = center + np.array([[0.8, -0.5, 0.3], [-0.4, 0.2, 0.6]])
    forces = lambda r: -(r - center) * k
    batch = np.array([0, 1])
    r, nsteps, hist = O.relax([O.FIRE(), O.FIRE()], r0, batch, forces, fmax=1e-4, steps=2000)
    assert (nsteps > 0).all() and (nsteps < 2000).all()
    assert np.abs(forces(r)).max() < 1e-4 and np.abs(r - center).max() < 1e-4
    assert len(hist) == nsteps.max() and sum(h[0] is not None for h in hist) == nsteps[0]
    # the same system alone takes the same steps: systems of a batch are independent
    ra, na, _ = O.relax([O.FIRE()], r0[:1], np.array([0]), lambda r: forces(np.vstack([r, center[1:]]))[:1], 1e-4, 2000)
    assert na[0] == nsteps[0] and np.array_equal(ra, r[:1])


def test_fixed_atoms_do_not_move():
    center = np.zeros((3, 3))
    r0 = np.array([[1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0]])
    fixed = np.array([False, True, False])
    r, _, _ = O.relax([O.FIRE()], r0, np.zeros(3, np.int64), lambda r: -(r - center), 1e-3, 500, fixed=fixed)
    np.testing.assert_array_equal(r[1], r0[1])
    assert np.abs(r[[0, 2]]).max() < 1e-2


def test_compaction_plan():
    from newtonnet_b200.optimize import compaction_plan
    n = np.array([21, 3, 21, 5])                                 # 50 atoms
    assert compaction_plan([True, True, True, True], n) is None
    assert compaction_plan([False] * 4, n) is None
    assert compaction_plan([True, False, True, False], n) is None           # 42 of 50 atoms
    keep, batch = compaction_plan([False, True, True, False], n)           # 24 of 50 atoms
    np.testing.assert_array_equal(keep, [1, 2])
    np.testing.assert_array_equal(batch, [0] * 3 + [1] * 21)
    # exactly half the atoms: compacted; one atom more: not
    keep, batch = compaction_plan([True, False, False, True], [5, 6, 4, 5])     # 10 of 20
    np.testing.assert_array_equal(keep, [0, 3])
    np.testing.assert_array_equal(batch, [0] * 5 + [1] * 5)
    assert compaction_plan([True, False, False, True], [5, 5, 4, 5]) is None    # 10 of 19

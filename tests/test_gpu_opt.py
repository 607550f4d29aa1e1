"""GPU tests of the device-resident FIRE optimiser (newtonnet_b200/optimize.py, nn_fire_step / nn_fire_check in
csrc/md_ops.cu) against the CPU oracle (oracle/opt_oracle.py) and against a host FIRE loop driven through the public
model API."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_case, load_weights

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _model(weights='md17'):
    from newtonnet_b200.compat import model_from_state_dict
    m = model_from_state_dict({k: torch.tensor(v) for k, v in load_weights(weights).items()},
                              output_properties=['energy', 'gradient_force']).to(DEV)
    m.eval()
    return m


def _aspirins(n_sys, noise=0.0, seed=0):
    kat = np.load(f'{GOLDEN}/md17_kat.npz')
    z = np.tile(kat['numbers'], n_sys)
    pos = np.concatenate([kat['positions'][(7 * k) % len(kat['positions'])] for k in range(n_sys)]).astype(np.float64)
    pos += np.random.default_rng(seed).normal(size=pos.shape) * noise
    return z, pos, np.repeat(np.arange(n_sys), 21)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def test_fire_kernels_match_oracle():
    from newtonnet_b200 import _lib as L
    from oracle import md_oracle as M
    from oracle import opt_oracle as O
    lib = L.load()
    rng = np.random.default_rng(0)
    sizes = [1, 21, 21, 21, 21, 21, 3000, 700, 21, 30]
    # (started, Nsteps, dt, force scale, v relative to f): every branch of FIRE.step
    cases = [(0, 0, 0.1, 1e-2, None),       # first step, 1 atom
             (1, 2, 0.1, 1e-2, 0.5),        # downhill, Nsteps <= Nmin, not clipped
             (1, 9, 0.3, 1e-2, 0.5),        # downhill, Nsteps > Nmin
             (1, 9, 0.95, 1e-2, 0.5),       # dt reaches dtmax
             (1, 4, 0.2, 1e-2, -0.7),       # uphill: reset
             (1, 3, 0.1, 5.0, 0.5),         # clipped step
             (1, 7, 0.5, 3.0, 0.3),         # 3000 atoms, downhill, clipped
             (1, 1, 0.2, 1e-3, -0.2),       # 700 atoms, uphill, not clipped
             (1, 3, 0.1, 1e-2, 0.5),        # converged: frozen
             (0, 0, 0.1, 1e-2, None)]       # first step, triclinic cell, 30 atoms, some fixed
    B, N = len(sizes), sum(sizes)
    ptr = np.concatenate([[0], np.cumsum(sizes)])
    batch = np.repeat(np.arange(B), sizes)
    cell = np.zeros((B, 3, 3))
    cell[9] = [[7.0, 0, 0], [1.5, 8.0, 0], [0.5, -1.0, 9.0]]
    x = rng.uniform(-10, 20, (N, 3))
    f = np.zeros((N, 3), np.float32)
    v = np.zeros((N, 3))
    sf, si = np.zeros((B, 3)), np.zeros((B, 4), np.int32)
    fixed = np.zeros(N, bool)
    fixed[ptr[9]:ptr[10]:4] = True
    for b, (started, n, dt, fs, vr) in enumerate(cases):
        s = slice(ptr[b], ptr[b + 1])
        f[s] = (rng.normal(size=(sizes[b], 3)) * fs).astype(np.float32)
        f[s][fixed[s]] = 0.0
        if vr is not None:
            v[s] = vr * f[s] + rng.normal(size=(sizes[b], 3)) * 0.1 * fs
        sf[b] = (dt, 0.1 * 0.99 ** n, 0.0)
        si[b] = (n, started, 1 if b == 8 else 0, 17)
    t = lambda a, d: torch.tensor(a, dtype=d, device=DEV)
    X, V, F, CELL = t(x, torch.float64), t(v, torch.float64), t(f, torch.float32), t(cell, torch.float32)
    SF, SI, PTR = t(sf, torch.float64), t(si, torch.int32), t(ptr, torch.int32)
    P = torch.full((N, 3), -7.0, device=DEV)
    params = (0.2, 1.0, 1.1, 0.5, 0.1, 0.99, 5)
    L.check(lib.nn_fire_step(B, PTR.data_ptr(), X.data_ptr(), V.data_ptr(), F.data_ptr(), CELL.data_ptr(), P.data_ptr(),
                             SF.data_ptr(), SI.data_ptr(), *params, _stream()), 'nn_fire_step')
    xd, vd, sfd, sid, pd = X.cpu().numpy(), V.cpu().numpy(), SF.cpu().numpy(), SI.cpu().numpy(), P.cpu().numpy()
    for b, (started, n, dt, fs, vr) in enumerate(cases):
        s = slice(ptr[b], ptr[b + 1])
        if b == 8:
            np.testing.assert_array_equal(xd[s], x[s]); np.testing.assert_array_equal(vd[s], v[s])
            np.testing.assert_array_equal(sfd[b], sf[b]); np.testing.assert_array_equal(sid[b], si[b])
            assert (pd[s] == -7.0).all()
            continue
        opt = O.FIRE(dt=dt, a=sf[b, 1])
        opt.Nsteps, opt.v = n, (v[s].copy() if started else None)
        xo = opt.step(x[s], f[s])
        np.testing.assert_allclose(vd[s], opt.v, rtol=1e-12, atol=1e-300, err_msg=f'system {b}')
        np.testing.assert_allclose(xd[s], xo, rtol=1e-12, atol=1e-300, err_msg=f'system {b}')
        assert abs(sfd[b, 0] - opt.dt) <= 1e-12 * opt.dt and abs(sfd[b, 1] - opt.a) <= 1e-12 * opt.a, b
        assert sid[b, 0] == opt.Nsteps and sid[b, 1] == 1 and sid[b, 2] == 0 and sid[b, 3] == 17, b
        w = M.wrap(xo, cell[b].astype(np.float32).astype(np.float64))
        if b == 9:
            d = (pd[s].astype(np.float64) - w) @ np.linalg.inv(cell[b])
            d -= np.rint(d)
            assert np.abs(d @ cell[b]).max() < 5e-6
        else:
            np.testing.assert_array_equal(pd[s], xd[s].astype(np.float32))
    # every branch was taken
    assert sfd[3, 0] == 1.0 and sid[4, 0] == 0 and sfd[4, 1] == 0.1 and sid[2, 0] == 10 and sid[1, 0] == 3
    assert abs(np.linalg.norm(xd[ptr[5]:ptr[6]] - x[ptr[5]:ptr[6]]) - 0.2) < 1e-12
    assert abs(np.linalg.norm(xd[ptr[6]:ptr[7]] - x[ptr[6]:ptr[7]]) - 0.2) < 1e-12
    np.testing.assert_array_equal(xd[fixed], x[fixed])

    # convergence test on new forces: fixed atoms zeroed, max |f|^2 exact, one step counted for every active system
    f2 = (rng.normal(size=(N, 3)) * np.repeat(rng.choice([1e-3, 1.0], B), sizes)[:, None]).astype(np.float32)
    F.copy_(t(f2, torch.float32))
    FIX = t(fixed, torch.bool)
    fmax2 = 0.05 ** 2
    FM = t([fmax2], torch.float64)
    CTR, STICKY, TICKET = t([41], torch.int64), t([0] * 4, torch.int32), t([0], torch.int32)
    status = np.zeros(L.NN_STATUS_WORDS, np.int32)
    status[L.ST_EDGE_OVERFLOW] = 1234
    ST = t(status, torch.int32)
    sid0 = SI.cpu().numpy()
    L.check(lib.nn_fire_check(B, PTR.data_ptr(), F.data_ptr(), FIX.data_ptr(), FM.data_ptr(), SF.data_ptr(), SI.data_ptr(), 1,
                              CTR.data_ptr(), ST.data_ptr(), STICKY.data_ptr(), TICKET.data_ptr(), _stream()), 'nn_fire_check')
    fz = f2.copy()
    fz[fixed] = 0.0
    np.testing.assert_array_equal(F.cpu().numpy(), fz)
    sfd, sid = SF.cpu().numpy(), SI.cpu().numpy()
    for b in range(B):
        s = slice(ptr[b], ptr[b + 1])
        assert sfd[b, 2] == O.max_force2(fz[s]), b
        assert sid[b, 2] == int(O.converged(fz[s], 0.05)), b
        assert sid[b, 3] == sid0[b, 3] + (0 if sid0[b, 2] else 1), b
    assert 0 < sid[:, 2].sum() < B
    assert CTR.item() == 42 and TICKET.item() == 0 and STICKY.cpu().tolist() == [1234, 0, 0, 0]
    L.check(lib.nn_fire_check(B, PTR.data_ptr(), F.data_ptr(), None, FM.data_ptr(), SF.data_ptr(), SI.data_ptr(), 0,
                              None, None, None, None, _stream()), 'nn_fire_check')
    np.testing.assert_array_equal(SI.cpu().numpy(), sid)          # measuring only: no step counted
    assert CTR.item() == 42


def test_matches_host_fire_loop():
    from newtonnet_b200.optimize import DeviceFIRE
    from oracle import opt_oracle as O
    model = _model()
    z, pos, batch = _aspirins(3)
    fmax, steps = 0.05, 40
    opt = DeviceFIRE(model, z, pos, batch=batch, check_interval=1)
    hist_dev = []
    for _ in range(steps):
        if opt.converged.all():
            break
        opt.run(fmax=fmax, steps=1)
        st = opt.state
        hist_dev.append(list(zip(st['dt'], st['a'], st['Nsteps'])))
    zt, bt = torch.tensor(z, device=DEV), torch.tensor(batch, device=DEV)
    cell = torch.zeros(3, 3, 3, device=DEV)
    forces = lambda p: model(zt, torch.tensor(p, dtype=torch.float32, device=DEV), cell, bt).gradient_force.double().cpu().numpy()
    x, nsteps, hist = O.relax([O.FIRE() for _ in range(3)], pos, batch, forces, fmax, steps)
    assert np.abs(opt.positions - x).max() < 2e-6
    np.testing.assert_array_equal(opt.nsteps, nsteps)
    assert len(hist) == len(hist_dev) > 0
    for k, row in enumerate(hist):            # branch history: dt, a, Nsteps after every step
        for b, h in enumerate(row):
            if h is not None:
                assert h[2] == hist_dev[k][b][2], (k, b)
                assert abs(h[0] - hist_dev[k][b][0]) <= 1e-12 * h[0] and abs(h[1] - hist_dev[k][b][1]) <= 1e-12 * h[1], (k, b)
    assert opt.kernels_per_step > 2


def test_batch_independence_compaction_and_check_interval():
    from newtonnet_b200.optimize import DeviceFIRE
    model = _model()
    kw = dict(fmax=0.05, steps=400)
    # 15 molecules near their minimum (relaxed, then nudged) and one far from it
    z, pos, batch = _aspirins(15)
    pre = DeviceFIRE(model, z, pos, batch=batch)
    pre.run(**kw)
    near = pre.positions + np.random.default_rng(3).normal(size=pos.shape) * 0.01
    zf, far, _ = _aspirins(1, noise=0.08, seed=5)
    Z = np.concatenate([z[:21 * 7], zf, z[21 * 7:]]).astype(np.int64)
    P = np.concatenate([near[:21 * 7], far, near[21 * 7:]])
    Bt = np.repeat(np.arange(16), 21)
    alone = DeviceFIRE(model, zf, far)
    alone.run(**kw)
    runs = {}
    for ci in (1, 16):
        o = DeviceFIRE(model, Z, P, batch=Bt, check_interval=ci)
        o.run(**kw)
        runs[ci] = o
    big = runs[16]
    assert big.compactions >= 1
    s = slice(7 * 21, 8 * 21)
    np.testing.assert_array_equal(big.positions[s], alone.positions)
    np.testing.assert_array_equal(big.state['v'][s], alone.state['v'])
    for k in ('dt', 'a', 'Nsteps'):
        np.testing.assert_array_equal(big.state[k][7], alone.state[k][0])
    assert big.nsteps[7] == alone.nsteps[0]
    np.testing.assert_array_equal(big.energy[7], alone.energy[0])
    np.testing.assert_array_equal(big.forces[s], alone.forces)
    a, b = runs[1], runs[16]
    np.testing.assert_array_equal(a.positions, b.positions)
    np.testing.assert_array_equal(a.nsteps, b.nsteps)
    np.testing.assert_array_equal(a.energy, b.energy)
    np.testing.assert_array_equal(a.state['v'], b.state['v'])


def test_converges_and_agrees_with_calculator():
    from newtonnet_b200.optimize import DeviceFIRE
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    from test_gpu_parity import FakeAtoms
    model = _model()
    z, pos, batch = _aspirins(8)
    opt = DeviceFIRE(model, z, pos, batch=batch)
    e0 = opt.energy
    done = opt.run(fmax=0.05, steps=2000)
    assert done and opt.converged.all() and (opt.fmax < 0.05).all()
    calc = MLAseCalculator(_model(), properties=['energy', 'forces'], device=DEV)
    calc.calculate([FakeAtoms(z[:21], opt.positions[batch == b]) for b in range(8)])
    fc = calc.results['forces'].reshape(-1, 3)
    assert np.abs(fc - opt.forces).max() < 1e-5
    fmax_calc = np.sqrt((fc.reshape(8, 21, 3) ** 2).sum(-1).max(-1))
    assert (fmax_calc[opt.converged] < 0.05).all()
    assert (calc.results['energy'] < e0).all()
    np.testing.assert_allclose(calc.results['energy'], opt.energy, rtol=1e-6)


def test_repeated_run_continues():
    from newtonnet_b200.optimize import DeviceFIRE
    model = _model()
    z, pos, batch = _aspirins(4)
    a = DeviceFIRE(model, z, pos, batch=batch)
    a.run(fmax=0.01, steps=30)
    b = DeviceFIRE(model, z, pos, batch=batch)
    b.run(fmax=0.01, steps=10)
    b.run(fmax=0.01, steps=20)
    np.testing.assert_array_equal(a.positions, b.positions)
    np.testing.assert_array_equal(a.state['v'], b.state['v'])
    np.testing.assert_array_equal(a.nsteps, b.nsteps)
    # converged at 0.05; a second run at 0.01 reactivates every system still above it
    c = DeviceFIRE(model, z, pos, batch=batch)
    assert c.run(fmax=0.05, steps=2000)
    n1, x1, v1 = c.nsteps, c.positions, c.state['v']
    assert c.run(fmax=0.05)                                  # nothing to do: zero steps, positions bit-unchanged
    np.testing.assert_array_equal(c.nsteps, n1)
    np.testing.assert_array_equal(c.positions, x1)
    above = c.fmax >= 0.01
    assert above.any()
    c.run(fmax=0.01, steps=25)
    assert (c.nsteps[above] > n1[above]).all() and (c.nsteps[~above] == n1[~above]).all()
    # inputs already below fmax take zero steps
    d = DeviceFIRE(model, z, x1, batch=batch)
    assert d.run(fmax=0.05)
    assert (d.nsteps == 0).all()
    np.testing.assert_array_equal(d.positions, x1)
    assert np.abs(v1).max() > 0


def test_periodic_fixed_atoms_and_overflow_rollback():
    from newtonnet_b200.compat import model_from_state_dict
    from newtonnet_b200.optimize import DeviceFIRE
    d, w = load_case('water375')
    model = model_from_state_dict({k: torch.tensor(v) for k, v in w.items()}, output_properties=['energy', 'gradient_force']).to(DEV)
    model.eval()
    fixed = d['z'] == 8
    kw = dict(cell=d['cell'], fixed=fixed, check_interval=8)
    a = DeviceFIRE(model, d['z'], d['pos'], **kw)
    a.run(fmax=1e-9, steps=24)
    x0 = d['pos'].astype(np.float64)
    np.testing.assert_array_equal(a.positions[fixed], x0[fixed])
    assert np.abs(a.positions[~fixed] - x0[~fixed]).max() > 0
    assert (a.forces[fixed] == 0).all() and a.nsteps[0] == 24
    frac = a.work.pos_model.double().cpu().numpy() @ np.linalg.inv(d['cell'][0].astype(np.float64))
    assert frac.min() > -1e-6 and frac.max() < 1 + 1e-6
    b = DeviceFIRE(model, d['z'], d['pos'], **kw)
    cap0 = b.work.nl.cap_edges
    b.work.sticky[0] = int(cap0 * 1.3)                  # pretend the first chunk overflowed: roll back, regrow, redo
    b.run(fmax=1e-9, steps=24)
    assert b.work.nl.cap_edges > cap0 and b.graph_launches == 32
    np.testing.assert_array_equal(a.positions, b.positions)
    np.testing.assert_array_equal(a.energy, b.energy)
    np.testing.assert_array_equal(a.nsteps, b.nsteps)


def test_from_atoms_and_update():
    from newtonnet_b200.optimize import DeviceFIRE
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    from test_gpu_parity import FakeAtoms

    class Fix:
        def __init__(self, idx):
            self.idx = idx

        def get_indices(self):
            return np.asarray(self.idx)

    class FixBondLength:
        pass

    kat = np.load(f'{GOLDEN}/md17_kat.npz')
    atoms = [FakeAtoms(kat['numbers'], kat['positions'][k]) for k in (0, 50, 100)]
    atoms[1].constraints = [Fix([0, 3, 20])]
    calc = MLAseCalculator(_model(), properties=['energy', 'forces'], device=DEV)
    opt = DeviceFIRE.from_atoms(atoms, calc)
    opt.run(fmax=0.05, steps=20)
    assert opt.nsteps.tolist() == [20, 20, 20]
    x = opt.positions
    np.testing.assert_array_equal(x[21 + np.array([0, 3, 20])], kat['positions'][50][[0, 3, 20]])
    assert (opt.forces[21 + np.array([0, 3, 20])] == 0).all()
    moved = []
    for at in atoms:
        at.set_positions = lambda p, at=at: moved.append(p)
    opt.update_atoms(atoms)
    assert len(moved) == 3
    for k in range(3):
        np.testing.assert_array_equal(moved[k], x[21 * k:21 * (k + 1)])
    single = DeviceFIRE.from_atoms(FakeAtoms(kat['numbers'], kat['positions'][0]), calc)
    assert single.n_systems == 1
    atoms[2].constraints = [FixBondLength()]
    with pytest.raises(NotImplementedError):
        DeviceFIRE.from_atoms(atoms, calc)

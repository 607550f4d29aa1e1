"""GPU tests of the device-resident climbing-image NEB (newtonnet_b200/neb.py, nn_neb_forces in csrc/neb.cu) against the
CPU oracle (oracle/neb_oracle.py) and against a host NEB + FIRE loop driven through the public model API."""
import functools

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_case, load_weights

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
U = 2.0 ** -24
# |got - ref| <= C_NEB * 2^-24 * mag element-wise, ref the fp64 oracle and mag = |F| + |F_par tau^| + |spring tau^| (the
# climbing image: |F| + |2 F_par tau^|).  The kernel computes in fp64 and rounds once to fp32 (<= 2^-24 |F_neb| <=
# 2^-24 mag); the fp64 reductions add ~1e-16 mag.  C_NEB = 2 leaves a factor 2 over that.
C_NEB = 2.0
METHYL_C, CARBONYL_C, METHYL_H = 4, 11, [18, 19, 20]      # MD17 aspirin atom order


def _model(weights='md17'):
    from newtonnet_b200.compat import model_from_state_dict
    m = model_from_state_dict({k: torch.tensor(v) for k, v in load_weights(weights).items()},
                              output_properties=['energy', 'gradient_force']).to(DEV)
    m.eval()
    return m


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _kat():
    return np.load(f'{GOLDEN}/md17_kat.npz')


def _band(a, b, n, noise=0.0, seed=0):
    """[n+2, N, 3]: linear interpolation from a to b with seeded Gaussian noise on the interior images."""
    t = np.linspace(0.0, 1.0, n + 2)[:, None, None]
    R = (1 - t) * a[None] + t * b[None]
    R[1:-1] += np.random.default_rng(seed).normal(size=R[1:-1].shape) * noise
    return R


def _rotate_methyl(x, deg):
    """Aspirin positions with the methyl hydrogens rotated by `deg` about the carbonyl C -> methyl C axis."""
    x = x.copy()
    axis = x[METHYL_C] - x[CARBONYL_C]
    axis /= np.linalg.norm(axis)
    t = np.deg2rad(deg)
    for h in METHYL_H:
        r = x[h] - x[METHYL_C]
        x[h] = x[METHYL_C] + r * np.cos(t) + np.cross(axis, r) * np.sin(t) + axis * (axis @ r) * (1 - np.cos(t))
    return x


@functools.lru_cache(maxsize=None)
def _methyl_ends():
    """[2, 21, 3]: MD17 aspirin frame 0 relaxed, and the same frame with its methyl group turned by 120 degrees, relaxed -
    two symmetry-equivalent minima (the hydrogens trade places) joined by a methyl-rotation saddle."""
    from newtonnet_b200.optimize import DeviceFIRE
    x0 = _kat()['positions'][0].astype(np.float64)
    r = DeviceFIRE(_model(), np.tile(_kat()['numbers'], 2), np.concatenate([x0, _rotate_methyl(x0, 120.0)]),
                   batch=np.repeat([0, 1], 21))
    assert r.run(fmax=0.005, steps=5000)
    return r.positions.reshape(2, 21, 3)


def _methyl_band(n, noise=0.0, seed=0):
    """[n+2, 21, 3]: the two minima of `_methyl_ends` with n interior images that turn the methyl group of the first by
    equal angles (a straight line between the end points would pull the hydrogens through the axis), plus seeded noise."""
    a, b = _methyl_ends()
    R = np.stack([a] + [_rotate_methyl(a, 120.0 * i / (n + 1)) for i in range(1, n + 1)] + [b])
    R[1:-1] += np.random.default_rng(seed).normal(size=R[1:-1].shape) * noise
    return R


def _forward_forces(model, z_list):
    """forces() of neb_oracle.relax_bands through the public forward: every interior image of every band in one batch."""
    def forces(Rs):
        z = np.concatenate([np.tile(z_list[b], len(R)) for b, R in enumerate(Rs)])
        pos = np.concatenate([R.reshape(-1, 3) for R in Rs])
        sizes = [len(z_list[b]) for b, R in enumerate(Rs) for _ in range(len(R))]
        batch = np.repeat(np.arange(len(sizes)), sizes)
        out = model(torch.tensor(z, device=DEV), torch.tensor(pos, dtype=torch.float32, device=DEV),
                    torch.zeros(len(sizes), 3, 3, device=DEV), torch.tensor(batch, device=DEV))
        e, f = out.energy.double().cpu().numpy(), out.gradient_force.double().cpu().numpy()
        res, i, a = [], 0, 0
        for b, R in enumerate(Rs):
            n, na = len(R), len(z_list[b])
            res.append((e[i:i + n], f[a:a + n * na].reshape(n, na, 3)))
            i, a = i + n, a + n * na
        return res
    return forces


def test_neb_kernel_matches_oracle():
    from newtonnet_b200 import _lib as L
    from newtonnet_b200.neb import band_layout
    from oracle import neb_oracle as N
    lib = L.load()
    rng = np.random.default_rng(0)
    # (atoms, energies of images 0..n+1, climb, frozen, fixed every k-th atom or 0); branches per interior image noted
    bands = [(21, [0, 1, 2, 3, 4], 0, 0, 0),        # monotone up
             (21, [4, 3, 2, 1, 0], 1, 0, 0),        # monotone down; the first interior image climbs
             (21, [0, 2, 5, 3, 1], 1, 0, 0),        # up; maximum with E+ > E- (climbs, middle); down
             (21, [0, 3, 2, 6, 1], 1, 0, 0),        # maximum E+ > E-; minimum; maximum E+ < E- (climbs, last)
             (21, [1, 1, 2, 2, 3], 1, 0, 0),        # exact ties E = E-, E = E+ ... and a tie for the climbing image
             (5, [0, 1, 0.5], 1, 0, 2),             # n = 1, climbing, fixed atoms
             (21, [0, 1, 2, 3], 0, 1, 0),           # frozen band: nothing written
             (3000, [0, 2, 1], 0, 0, 0),            # n = 1, a 3,000-atom image
             (30, [0, 1.5, 1, 0.25], 0, 0, 3),      # fixed atoms: maximum E+ > E-, then monotone down
             (21, [2, 2, 2], 1, 0, 0),              # three equal energies: tau = t+ + t-
             (21, [0, 1, np.nan, 2, 0], 1, 0, 0),   # a non-finite energy: the band fails
             (21, [0, 1, 2, 1, 0], 1, 0, 0),        # a non-finite force (set below): the band fails
             (21, [0, 1, 0], 0, 0, 2)]              # a NaN force on a fixed atom (set below) counts as zero
    na = np.array([b[0] for b in bands])
    ni = np.array([len(b[1]) - 2 for b in bands])
    lay = band_layout(na, ni)
    B, N_ = len(bands), int(lay['band_ptr'][-1])
    Rs = [rng.uniform(-3, 3, (na[b], 3))[None] + np.cumsum(rng.normal(size=(ni[b] + 2, na[b], 3)) * 0.1, axis=0)
          for b in range(B)]
    Fs = [(rng.normal(size=(ni[b], na[b], 3)) * 0.5).astype(np.float32) for b in range(B)]
    fixed = [np.arange(na[b]) % bands[b][4] == 0 if bands[b][4] else np.zeros(na[b], bool) for b in range(B)]
    Fs[11][2, 5, 1] = np.inf
    Fs[12][0, 0, 0] = np.nan
    k = 0.37
    t = lambda a, d: torch.tensor(np.asarray(a), dtype=d, device=DEV)
    i32 = torch.int32
    X = t(np.concatenate([R[1:-1].reshape(-1, 3) for R in Rs]), torch.float64)
    ENDS = t(np.concatenate([R[[0, -1]].reshape(-1, 3) for R in Rs]), torch.float64)
    E = t(np.concatenate([np.asarray(bd[1][1:-1]) for bd in bands]), torch.float32)
    EE = t([[bd[1][0], bd[1][-1]] for bd in bands], torch.float64)
    F = t(np.concatenate([f.reshape(-1, 3) for f in Fs]), torch.float32)
    FIX = t(np.concatenate([np.tile(f, n) for f, n in zip(fixed, ni)]), torch.bool)
    CLIMB = t([bd[2] for bd in bands], i32)
    SI = t([[0, 1, bd[3], 0] for bd in bands], i32)
    OUT = torch.full((N_, 3), -7.0, device=DEV)
    IMAX = torch.full((B,), -1, dtype=i32, device=DEV)
    FAILED = torch.zeros(B, dtype=i32, device=DEV)
    idx = {key: t(lay[key], i32) for key in ('img_ptr', 'img_band', 'band_img', 'ends_ptr')}
    L.check(lib.nn_neb_forces(len(lay['img_band']), idx['img_ptr'].data_ptr(), idx['img_band'].data_ptr(),
                              idx['band_img'].data_ptr(), X.data_ptr(), ENDS.data_ptr(), idx['ends_ptr'].data_ptr(),
                              E.data_ptr(), EE.data_ptr(), F.data_ptr(), FIX.data_ptr(), CLIMB.data_ptr(), SI.data_ptr(), k,
                              OUT.data_ptr(), IMAX.data_ptr(), FAILED.data_ptr(), _stream()), 'nn_neb_forces')
    out, imax, failed = OUT.cpu().numpy(), IMAX.cpu().numpy(), FAILED.cpu().numpy()
    for b, (n_at, en, climb, frozen, _) in enumerate(bands):
        got = out[lay['band_ptr'][b]:lay['band_ptr'][b + 1]].reshape(ni[b], n_at, 3)
        if frozen:
            assert (got == -7.0).all() and imax[b] == -1
            continue
        ref, top = N.neb_forces(Rs[b], np.asarray(en, dtype=np.float32), Fs[b], k, bool(climb), fixed[b])
        if top is None:                                     # failed: zero NEB force on every image, imax not written
            assert failed[b] == 1 and imax[b] == -1 and (got == 0).all(), b
            continue
        assert imax[b] == top and failed[b] == 0, b
        f64 = Fs[b].astype(np.float64)
        f64[:, fixed[b]] = 0.0
        mag = np.empty_like(ref)
        for i in range(1, ni[b] + 1):
            tau, ntp, ntm = N.tangent(Rs[b], np.asarray(en, dtype=np.float64), i)
            fpar = abs(np.vdot(f64[i - 1], tau))
            extra = 2 * fpar if climb and i == top else fpar + abs(ntp * k - ntm * k)
            mag[i - 1] = np.abs(f64[i - 1]) + extra * np.abs(tau)
        err = np.abs(got - ref)
        assert (err <= C_NEB * U * mag).all(), (b, float((err / (U * mag + 1e-300)).max()))
        assert (got[:, fixed[b]] == 0).all()
    assert imax.tolist() == [3, 1, 2, 3, 3, 1, -1, 1, 1, 1, -1, -1, 1]
    assert failed.tolist() == [0] * 10 + [1, 1, 0]


def test_matches_host_neb_loop():
    from newtonnet_b200.neb import DeviceNEB
    from oracle import neb_oracle as N
    model = _model()
    kat = _kat()
    z = kat['numbers'].astype(np.int64)
    bands = [_methyl_band(5, 0.02, 1), _methyl_band(3, 0.02, 2)]
    fmax, steps = 0.05, 40
    opt = DeviceNEB(model, [z, z], bands, climb=True, check_interval=1)
    hist_dev = []
    for _ in range(steps):
        if opt.converged.all():
            break
        opt.run(fmax=fmax, steps=1)
        st = opt.state
        hist_dev.append(list(zip(st['dt'], st['a'], st['Nsteps'])))
    forces = _forward_forces(model, [z, z])
    ends = [(e[0], e[-1]) for e in opt.energies]
    for b, R in enumerate(bands):
        e_fwd = forces([R[[0, -1]]])[0][0]
        assert e_fwd[0] == ends[b][0] and e_fwd[1] == ends[b][1]
    R, nsteps, hist, _, F, top = N.relax_bands(bands, ends, forces, fmax, steps, climb=True, store=np.float32)
    for b in range(2):
        assert np.abs(opt.positions[b] - R[b]).max() < 2e-6, b
        np.testing.assert_array_equal(opt.positions[b][[0, -1]], bands[b][[0, -1]])
    np.testing.assert_array_equal(opt.nsteps, nsteps)
    np.testing.assert_array_equal(opt.imax, top)
    assert len(hist) == len(hist_dev) > 0
    for kk, row in enumerate(hist):            # branch history: dt, a, Nsteps after every step
        for b, h in enumerate(row):
            if h is not None:
                assert h[2] == hist_dev[kk][b][2], (kk, b)
                assert abs(h[0] - hist_dev[kk][b][0]) <= 1e-12 * h[0] and abs(h[1] - hist_dev[kk][b][1]) <= 1e-12 * h[1], (kk, b)
    assert opt.kernels_per_step > 3


def test_batch_independence_compaction_and_check_interval():
    from newtonnet_b200.neb import DeviceNEB
    model = _model()
    kat = _kat()
    z = kat['numbers'].astype(np.int64)
    kw = dict(fmax=0.1, steps=600)
    # six bands near their converged path (relaxed, then nudged) and one far from it
    pre = DeviceNEB(model, [z] * 6, [_methyl_band(3, 0.01, q) for q in range(6)])
    assert pre.run(fmax=0.1, steps=3000)
    near = []
    for q, R in enumerate(pre.positions):
        R = R.copy()
        R[1:-1] += np.random.default_rng(10 + q).normal(size=R[1:-1].shape) * 0.003
        near.append(R)
    far = _methyl_band(4, 0.05, 5)
    bands = near[:3] + [far] + near[3:]
    alone = DeviceNEB(model, z, far, climb=True)
    alone.run(**kw)
    runs = {ci: DeviceNEB(model, [z] * 7, bands, climb=True, check_interval=ci) for ci in (1, 16)}
    for o in runs.values():
        o.run(**kw)
    big = runs[16]
    assert big.compactions >= 1 and alone.nsteps[0] > big.nsteps[[0, 1, 2, 4, 5, 6]].max()
    np.testing.assert_array_equal(big.positions[3], alone.positions[0])
    np.testing.assert_array_equal(big.state['v'][3], alone.state['v'][0])
    for key in ('dt', 'a', 'Nsteps'):
        np.testing.assert_array_equal(big.state[key][3], alone.state[key][0])
    assert big.nsteps[3] == alone.nsteps[0] and big.imax[3] == alone.imax[0]
    np.testing.assert_array_equal(big.energies[3], alone.energies[0])
    np.testing.assert_array_equal(big.forces[3], alone.forces[0])
    np.testing.assert_array_equal(big.true_forces[3], alone.true_forces[0])
    a, b = runs[1], runs[16]
    for q in range(7):
        np.testing.assert_array_equal(a.positions[q], b.positions[q])
        np.testing.assert_array_equal(a.energies[q], b.energies[q])
        np.testing.assert_array_equal(a.state['v'][q], b.state['v'][q])
    np.testing.assert_array_equal(a.nsteps, b.nsteps)


def test_climb_switched_on_between_runs_matches_oracle():
    from newtonnet_b200.neb import DeviceNEB
    from oracle import neb_oracle as N
    model = _model()
    kat = _kat()
    z = kat['numbers'].astype(np.int64)
    band = _methyl_band(5, 0.03, 7)
    opt = DeviceNEB(model, z, band, check_interval=4)
    forces = _forward_forces(model, [z])
    ends = [(opt.energies[0][0], opt.energies[0][-1])]
    opt.run(fmax=0.5, steps=300)
    R, n1, _, opts, _, _ = N.relax_bands([band], ends, forces, 0.5, 300, store=np.float32)
    assert opt.converged[0] and n1[0] == opt.nsteps[0] > 0
    assert np.abs(opt.positions[0] - R[0]).max() < 2e-6
    f_off = opt.forces[0]
    assert opt.run(fmax=0.5, climb=False)                    # same setting: nothing to do
    opt.run(fmax=0.05, steps=30, climb=True)
    R, n2, _, _, F, top = N.relax_bands(R, ends, forces, 0.05, 30, climb=True, opts=opts, store=np.float32)
    assert opt.nsteps[0] == n1[0] + n2[0] and n2[0] > 0
    assert np.abs(opt.positions[0] - R[0]).max() < 2e-6
    assert opt.imax[0] == top[0] and opt.climb
    assert np.abs(opt.forces[0] - F[0]).max() < 1e-5
    assert not np.array_equal(opt.forces[0], f_off)
    # switching back re-projects at the current positions before deciding what is converged
    fm = opt.fmax[0]
    opt.run(fmax=10.0, climb=False)
    assert opt.nsteps[0] == n1[0] + n2[0] and opt.fmax[0] != fm


def test_band_stopped_where_the_model_fails():
    """Seed 487 of tools/bench_neb.py's aspirin bands: after ~2,700 steps its last interior image has walked into a region
    of the MD17 model with no repulsive wall (two atoms 0.1-0.3 A apart, energies down to -1e35 eV) and the model returns
    NaN.  Device and host loop stop the band at the same step; the positions stay finite."""
    from newtonnet_b200.neb import DeviceNEB
    from oracle import neb_oracle as N
    model = _model()
    z = _kat()['numbers'].astype(np.int64)
    band = _methyl_band(7, 0.05, 487)
    good = _methyl_band(7, 0.05, 0)
    opt = DeviceNEB(model, [z, z], [band, good], climb=True)
    with pytest.warns(RuntimeWarning, match=r'bands \[0\]'):
        assert not opt.run(fmax=0.05, steps=4000)
    assert opt.failed.tolist() == [True, False] and opt.converged.tolist() == [False, True]
    assert np.isnan(opt.fmax[0]) and opt.fmax[1] < 0.05
    assert np.isfinite(opt.positions[0]).all() and not np.isfinite(opt.energies[0]).all()
    n0 = opt.nsteps.copy()
    assert 0 < n0[0] < 4000
    assert not opt.run(fmax=0.05, steps=100) and (opt.nsteps == n0).all()     # a failed band never steps again
    ends = [(opt.energies[0][0], opt.energies[0][-1])]
    _, nh, _, _, _, top = N.relax_bands([band], ends, _forward_forces(model, [z]), 0.05, 4000, climb=True, store=np.float32)
    assert top[0] is None and nh[0] == n0[0]


def test_periodic_fixed_atoms_and_overflow_rollback():
    from newtonnet_b200.compat import model_from_state_dict
    from newtonnet_b200.neb import DeviceNEB, align_band
    d, w = load_case('water81_smallL')
    model = model_from_state_dict({k: torch.tensor(v) for k, v in w.items()}, output_properties=['energy', 'gradient_force']).to(DEV)
    model.eval()
    cell = d['cell'][0].astype(np.float64)
    a = d['pos'].astype(np.float64)
    b = a.copy()
    b[3:6] += [0.6, -0.3, 0.4]                              # one molecule displaced
    R = _band(a, b, 3)
    rng = np.random.default_rng(4)
    wrapped = R + rng.integers(-1, 2, R.shape[:2] + (3,)) @ cell    # every atom of every image in another cell
    fixed = (d['z'] == 8) & (np.arange(81) != 3)
    kw = dict(cell=cell, fixed=fixed, climb=True, check_interval=8)
    x = DeviceNEB(model, d['z'], wrapped, **kw)
    aligned = align_band(wrapped, cell)
    np.testing.assert_allclose(aligned - aligned[0], R - R[0], atol=1e-9)
    x.run(fmax=1e-9, steps=24)
    got = x.positions[0]
    np.testing.assert_array_equal(got[:, fixed], aligned[:, fixed])
    assert np.abs(got[1:-1, ~fixed] - aligned[1:-1, ~fixed]).max() > 0
    assert (x.forces[0][:, fixed] == 0).all() and (x.true_forces[0][:, fixed] == 0).all() and x.nsteps[0] == 24
    frac = x.work.pos_model.double().cpu().numpy() @ np.linalg.inv(cell)
    assert frac.min() > -1e-6 and frac.max() < 1 + 1e-6
    y = DeviceNEB(model, d['z'], wrapped, **kw)
    cap0 = y.work.nl.cap_edges
    y.work.sticky[0] = int(cap0 * 1.3)                      # pretend the first chunk overflowed: roll back, regrow, redo
    y.run(fmax=1e-9, steps=24)
    assert y.work.nl.cap_edges > cap0 and y.graph_launches == 32
    np.testing.assert_array_equal(x.positions[0], y.positions[0])
    np.testing.assert_array_equal(x.energies[0], y.energies[0])
    np.testing.assert_array_equal(x.forces[0], y.forces[0])
    np.testing.assert_array_equal(x.nsteps, y.nsteps)


def test_from_images_and_update():
    from newtonnet_b200.neb import DeviceNEB
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    from test_gpu_parity import FakeAtoms

    class Fix:
        def __init__(self, idx):
            self.idx = idx

        def get_indices(self):
            return np.asarray(self.idx)

    kat = _kat()
    z = kat['numbers']
    R1, R2 = _methyl_band(3, 0.01, 1), _methyl_band(2, 0.01, 2)
    held = [0, 3, 7]                                        # fixed atoms sit still in every image
    R2[:, held] = R2[0, held]
    band1 = [FakeAtoms(z, r) for r in R1]
    band2 = [FakeAtoms(z, r) for r in R2]
    for at in band2:
        at.constraints = [Fix(held)]
    calc = MLAseCalculator(_model(), properties=['energy', 'forces'], device=DEV)
    opt = DeviceNEB.from_images([band1, band2], calc, climb=True)
    ref = DeviceNEB(_model(), [z, z], [R1, R2], fixed=[None, np.isin(np.arange(21), held)], climb=True)
    opt.run(fmax=0.05, steps=12)
    ref.run(fmax=0.05, steps=12)
    assert opt.nsteps.tolist() == [12, 12]
    for b in range(2):
        np.testing.assert_array_equal(opt.positions[b], ref.positions[b])
    np.testing.assert_array_equal(opt.positions[1][:, held], R2[:, held])
    moved = {}
    for b, band in enumerate((band1, band2)):
        for i, at in enumerate(band):
            at.set_positions = lambda p, key=(b, i): moved.__setitem__(key, p)
    opt.update_images([band1, band2])
    assert sorted(moved) == [(0, 1), (0, 2), (0, 3), (1, 1), (1, 2)]
    for (b, i), p in moved.items():
        np.testing.assert_array_equal(p, opt.positions[b][i])
    single = DeviceNEB.from_images(band1, calc)
    assert single.n_bands == 1 and single.energies[0].shape == (5,)


def _negative_modes(model, z, x, tol):
    """Eigenvalues of the Hessian below -tol after projecting out rigid translations and rotations."""
    from newtonnet_b200 import hessian
    n = len(z)
    H = hessian(model, torch.tensor(z, device=DEV), torch.tensor(x, dtype=torch.float32, device=DEV),
                torch.zeros(1, 3, 3, device=DEV), torch.zeros(n, dtype=torch.int64, device=DEV))
    H = H.reshape(3 * n, 3 * n).double().cpu().numpy()
    H = 0.5 * (H + H.T)
    c = x - x.mean(0)
    rigid = [np.tile(e, n) for e in np.eye(3)] + [np.cross(e, c).reshape(-1) for e in np.eye(3)]
    Q, _ = np.linalg.qr(np.stack(rigid, 1))
    Pm = np.eye(3 * n) - Q @ Q.T
    ev = np.linalg.eigvalsh(Pm @ H @ Pm)
    return ev[ev < -tol], ev


def test_aspirin_methyl_rotation_saddle():
    from newtonnet_b200.neb import DeviceNEB
    model = _model()
    z = _kat()['numbers'].astype(np.int64)
    ends = _methyl_ends()
    n = 7
    band = _methyl_band(n)
    opt = DeviceNEB(model, z, band, climb=True)
    assert opt.run(fmax=0.01, steps=5000)
    i = opt.imax[0]
    E = opt.energies[0]
    assert 0 < i < n + 1 and E[i] == E.max() and E[i] > max(E[0], E[-1])
    tol = 1e-3
    neg, ev = _negative_modes(model, z, opt.positions[0][i], tol)
    print(f'methyl rotation: barrier {E[i] - E[0]:.4f} eV at image {i} after {opt.nsteps[0]} steps, '
          f'lowest projected Hessian eigenvalues {np.round(ev[:8], 5).tolist()} eV/A^2')
    assert len(neg) == 1, ev[:8]
    for x in ends:
        neg, ev = _negative_modes(model, z, x, tol)
        assert len(neg) == 0, ev[:8]

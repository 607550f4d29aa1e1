"""CPU tests of the NEB oracle (oracle/neb_oracle.py) and of DeviceNEB's host-side input handling and band layout
(newtonnet_b200/neb.py)."""
import numpy as np
import pytest

from oracle import neb_oracle as N

# Mueller-Brown potential, scaled to energies of order 1: three minima and two saddle points in the plane
MB_A = np.array([-200.0, -100.0, -170.0, 15.0]) * 0.01
MB_a, MB_b, MB_c = np.array([-1.0, -1.0, -6.5, 0.7]), np.array([0.0, 0.0, 11.0, 0.6]), np.array([-10.0, -10.0, -6.5, 0.7])
MB_x0, MB_y0 = np.array([1.0, 0.0, -0.5, -1.0]), np.array([0.0, 0.5, 1.5, 1.0])


def _mb(p):
    """Energy [...] and gradient [..., 3] of one 'atom' at p [..., 3] (the potential does not depend on z)."""
    dx, dy = p[..., 0:1] - MB_x0, p[..., 1:2] - MB_y0
    e = MB_A * np.exp(MB_a * dx * dx + MB_b * dx * dy + MB_c * dy * dy)
    g = np.stack([(e * (2 * MB_a * dx + MB_b * dy)).sum(-1), (e * (MB_b * dx + 2 * MB_c * dy)).sum(-1), 0 * dx[..., 0]], -1)
    return e.sum(-1), g


def _mb_min(p):
    p = np.array([p[0], p[1], 0.0])
    for _ in range(200):                      # Newton on the analytic gradient with a finite-difference Hessian
        H = np.array([(_mb(p + e)[1] - _mb(p - e)[1])[:2] / 2e-6 for e in np.eye(3)[:2] * 1e-6])
        p[:2] -= np.linalg.solve(0.5 * (H + H.T), _mb(p)[1][:2])
    return p


def test_oracle_climbing_image_finds_mueller_brown_saddle():
    a, c = _mb_min([-0.55, 1.44]), _mb_min([-0.05, 0.47])
    assert np.abs(_mb(a)[1]).max() < 1e-10 and np.abs(_mb(c)[1]).max() < 1e-10
    n = 7
    t = np.linspace(0.0, 1.0, n + 2)[:, None]
    R = ((1 - t) * a + t * c)[:, None, :]
    ends = [(_mb(R[0, 0])[0], _mb(R[-1, 0])[0])]
    forces = lambda Rs: [(_mb(r[:, 0])[0], -_mb(r)[1]) for r in Rs]
    Rs, n1, _, opts, _, _ = N.relax_bands([R], ends, forces, fmax=0.5, steps=2000, k=1.0)
    fmax = 0.005
    Rs, n2, _, _, F, top = N.relax_bands(Rs, ends, forces, fmax=fmax, steps=5000, k=1.0, climb=True, opts=opts)
    assert 0 < n2[0] < 5000 and np.abs(F[0]).max() < fmax
    i = top[0]
    p = Rs[0][i, 0]
    assert np.linalg.norm(_mb(p)[1]) < fmax                 # the climbing image feels the full force: |grad V| < fmax
    E = _mb(Rs[0][:, 0])[0]
    assert E[i] == E.max() and 0 < i < n + 1
    H = np.array([(_mb(p + e)[1] - _mb(p - e)[1])[:2] / 2e-5 for e in np.eye(3)[:2] * 1e-5])
    ev = np.linalg.eigvalsh(0.5 * (H + H.T))
    assert ev[0] < -1.0 and ev[1] > 1.0                     # exactly one negative eigenvalue: a first-order saddle
    assert np.abs(p[:2] - [-0.822, 0.624]).max() < 2e-3     # the known saddle between these two minima


# 1-D-like bands in the plane: R0 = (0,0), R1 = (1,0), R2 = (1,2), so t- = (1,0), |t-| = 1 and t+ = (0,2), |t+| = 2
R3 = np.array([[[0.0, 0.0, 0.0]], [[1.0, 0.0, 0.0]], [[1.0, 2.0, 0.0]]])
F1 = np.array([[[0.3, -0.5, 0.25]]])


@pytest.mark.parametrize('E, tau', [
    ([0.0, 1.0, 2.0], [0.0, 1.0, 0.0]),                      # monotone up: tau = t+
    ([2.0, 1.0, 0.0], [1.0, 0.0, 0.0]),                      # monotone down: tau = t-
    ([0.0, 3.0, 1.0], [2.0, 6.0, 0.0]),                      # maximum, E+ > E-: t+ dVmax + t- dVmin = (0,2) 3 + (1,0) 2
    ([1.0, 3.0, 0.0], [3.0, 4.0, 0.0]),                      # maximum, E+ < E-: t+ dVmin + t- dVmax = (0,2) 2 + (1,0) 3
    ([2.0, 0.0, 1.0], [2.0, 2.0, 0.0]),                      # minimum, E+ < E-: (0,2) 1 + (1,0) 2
    ([1.0, 1.0, 2.0], [0.0, 1.0, 0.0]),                      # tie E = E-: not monotone, dVmin = 0, so tau = t+
    ([1.0, 1.0, 1.0], [1.0, 2.0, 0.0]),                      # three equal energies: t+ + t-, the limit dVmax = dVmin
])
def test_tangent_branches(E, tau):
    tau = np.array(tau) / np.linalg.norm(tau)
    k = 0.7
    for climb in (False, True):
        got, top = N.neb_forces(R3, E, F1, k, climb)
        fpar = F1[0, 0] @ tau
        want = F1[0, 0] - 2 * fpar * tau if climb else F1[0, 0] - fpar * tau + k * (2.0 - 1.0) * tau
        assert top == 1
        np.testing.assert_allclose(got[0, 0], want, rtol=0, atol=1e-15)


def test_climbing_image_ties_and_fixed_atoms():
    R = np.array([[[0.0, 0, 0], [5.0, 0, 0]], [[1.0, 0, 0], [5.0, 0, 0]], [[2.0, 0.5, 0], [5.0, 0, 0]],
                  [[3.0, 0, 0], [5.0, 0, 0]]])
    assert N.imax([0.0, 2.0, 2.0, 0.0]) == 2 and N.imax([0.0, 3.0, 2.0, 0.0]) == 1 and N.imax([5.0, 1.0, 2.0, 9.0]) == 2
    F = np.array([[[0.1, 0.2, 0.3], [1.0, 1.0, 1.0]], [[-0.1, 0.4, 0.0], [2.0, 2.0, 2.0]]])
    fixed = np.array([False, True])
    got, top = N.neb_forces(R, [0.0, 2.0, 2.0, 0.0], F, 0.1, True, fixed)
    assert top == 2
    assert (got[:, 1] == 0).all()                           # fixed atoms: their force counts as 0 and their NEB force is 0
    tau, _, _ = N.tangent(R, [0.0, 2.0, 2.0, 0.0], 2)
    np.testing.assert_allclose(got[1, 0], F[1, 0] - 2 * (F[1, 0] @ tau[0]) * tau[0], atol=1e-15)
    assert np.abs(tau[1]).max() == 0.0                      # the fixed atom does not move along the band


def test_non_finite_model_output_fails_the_band():
    R = np.array([[[0.0, 0, 0], [5.0, 0, 0]], [[1.0, 0, 0], [5.0, 0, 0]], [[2.0, 0.5, 0], [5.0, 0, 0]],
                  [[3.0, 0, 0], [5.0, 0, 0]]])
    F = np.ones((2, 2, 3))
    for E, Fb in (([0.0, np.nan, 1.0, 0.0], F), ([0.0, 1.0, np.inf, 0.0], F), ([0.0, 1.0, 2.0, 0.0], F * [[[1]], [[np.inf]]])):
        got, top = N.neb_forces(R, E, Fb, 0.1, True)
        assert top is None and (got == 0).all()
    Fb = F.copy()
    Fb[1, 1] = np.nan                                       # a fixed atom's force counts as zero, even when it is NaN
    got, top = N.neb_forces(R, [0.0, 1.0, 2.0, 0.0], Fb, 0.1, True, fixed=[False, True])
    assert top == 2 and np.isfinite(got).all() and (got[:, 0] != 0).any()


def test_band_layout_and_segment_rows():
    from newtonnet_b200.neb import band_layout
    from newtonnet_b200.optimize import segment_rows
    lay = band_layout([2, 3, 1], [1, 2, 3])
    np.testing.assert_array_equal(lay['band_ptr'], [0, 2, 8, 11])
    np.testing.assert_array_equal(lay['band_img'], [0, 1, 3, 6])
    np.testing.assert_array_equal(lay['img_ptr'], [0, 2, 5, 8, 9, 10, 11])
    np.testing.assert_array_equal(lay['img_band'], [0, 1, 1, 2, 2, 2])
    np.testing.assert_array_equal(lay['ends_ptr'], [0, 4, 10])
    np.testing.assert_array_equal(segment_rows(lay['band_ptr'], [0, 2]), [0, 1, 8, 9, 10])
    np.testing.assert_array_equal(segment_rows(lay['band_img'], [1, 2]), [1, 2, 3, 4, 5])
    np.testing.assert_array_equal(segment_rows(lay['band_ptr'], []), np.zeros(0))


def test_periodic_alignment():
    from newtonnet_b200.neb import align_band
    cell = np.array([[10.0, 0, 0], [2.0, 9.0, 0], [0, 0, 8.0]])
    rng = np.random.default_rng(0)
    R = rng.uniform(0, 1, (5, 4, 3)) @ cell
    for i in range(1, 5):
        R[i] = R[i - 1] + rng.normal(size=(4, 3)) * 0.3
    wrapped = R + rng.integers(-2, 3, (5, 4, 3)) @ cell
    got = align_band(wrapped, cell)
    np.testing.assert_allclose(got - got[0], R - R[0], atol=1e-12)   # image 0 keeps its own lattice shift
    np.testing.assert_array_equal(got[0], wrapped[0])
    np.testing.assert_array_equal(align_band(R, np.zeros((3, 3))), R)
    far = R.copy()
    far[3, 1] = far[2, 1] + [3.5, 3.0, 2.0]                 # |d| = 5.0 after rounding; half the smallest height is 4
    with pytest.raises(ValueError, match='ambiguous'):
        align_band(far, cell)
    with pytest.raises(ValueError, match='partially periodic'):
        align_band(R, np.diag([10.0, 10.0, 0.0]))


def test_input_checks():
    from newtonnet_b200.neb import DeviceNEB, bands_from_inputs
    z = np.array([1, 8, 1])
    R = np.random.default_rng(1).normal(size=(4, 3, 3))
    (zb, Rb, c, f), = bands_from_inputs(z, R)
    assert Rb.shape == (4, 3, 3) and (c == 0).all() and not f.any()
    Rc = R[:3, :2].copy()
    Rc[:, 0] = Rc[0, 0]
    assert len(bands_from_inputs([z, z[:2]], [R, Rc], fixed=[None, [True, False]])) == 2
    with pytest.raises(ValueError, match='interior image'):
        bands_from_inputs(z, R[[0, 3]])
    R2 = R.copy()
    R2[2] = R2[1]
    with pytest.raises(ValueError, match='coincide'):
        bands_from_inputs(z, R2)
    with pytest.raises(ValueError, match=r'\[n\+2, 3, 3\]'):
        bands_from_inputs(z, R[:, :2])
    with pytest.raises(ValueError, match='bands'):
        bands_from_inputs([z], [R, R])
    with pytest.raises(ValueError, match='fixed atoms must sit'):
        bands_from_inputs(z, R, fixed=[True, False, False])
    Rf = R.copy()
    Rf[:, 0] = Rf[0, 0]
    assert len(bands_from_inputs(z, Rf, fixed=[True, False, False])) == 1
    for kw, err in ((dict(k=0.0), ValueError), (dict(k=-1.0), ValueError), (dict(k=[0.1, 0.2, 0.1]), NotImplementedError),
                    (dict(method='aseneb'), NotImplementedError), (dict(remove_rotation_and_translation=True), NotImplementedError),
                    (dict(precon='Exp'), NotImplementedError)):
        with pytest.raises(err):
            DeviceNEB(None, z, R, **kw)


class _Atoms:
    def __init__(self, numbers, positions, cell=None, constraints=()):
        self.numbers, self.positions = np.asarray(numbers), np.asarray(positions, dtype=np.float64)
        self.cell = np.zeros((3, 3)) if cell is None else np.asarray(cell, dtype=np.float64)
        self.constraints = list(constraints)

    def __len__(self):
        return len(self.numbers)

    def get_atomic_numbers(self):
        return self.numbers

    def get_positions(self):
        return self.positions

    def get_cell(self):
        return self.cell

    def get_pbc(self):
        return np.array([(self.cell != 0).any()] * 3)


class _Fix:
    def __init__(self, idx):
        self.idx = idx

    def get_indices(self):
        return np.asarray(self.idx)


def test_from_images_rejects_inconsistent_bands():
    from newtonnet_b200.neb import DeviceNEB
    calc = type('Calc', (), {'model': None})()
    z = np.array([6, 1, 1])
    p = np.random.default_rng(2).normal(size=(3, 3, 3))
    cases = [([_Atoms(z, p[0]), _Atoms(z[:2], p[1, :2]), _Atoms(z, p[2])], 'other atoms'),
             ([_Atoms(z, p[0]), _Atoms([6, 1, 8], p[1]), _Atoms(z, p[2])], 'other atoms'),
             ([_Atoms(z, p[0]), _Atoms(z, p[1], cell=np.eye(3) * 9), _Atoms(z, p[2])], 'another cell'),
             ([_Atoms(z, p[0], constraints=[_Fix([0])]), _Atoms(z, p[1]), _Atoms(z, p[2])], 'other atoms than image 0')]
    for band, msg in cases:
        with pytest.raises(ValueError, match=msg):
            DeviceNEB.from_images(band, calc)
        with pytest.raises(ValueError, match=msg):
            DeviceNEB.from_images([[_Atoms(z, q) for q in p], band], calc)
    with pytest.raises(NotImplementedError):
        DeviceNEB.from_images([_Atoms(z, p[0], constraints=[object()]), _Atoms(z, p[1]), _Atoms(z, p[2])], calc)

"""The forward-sweep operators of the C ABI, one by one, against fp64 restatements of their formulas, and the two-level
(sliced) per-system energy and virial sums of nn_eval end to end against the fp64 oracle.  The reverse-sweep operators
are checked the same way in test_gpu_bwd_ops.py.

Tolerance rule (every comparison here):  |got - ref| <= c * 2^-24 * mag,  where `ref` is the operation evaluated in fp64
from the same fp32 operands and `mag` is the same expression evaluated in fp64 on the absolute values of the operands
(e.g. sum_k |We_fk| |rbf_pk| |mn_if| |mn_jf| for the message).  A rounding error of every fp32 operation is at most 2^-24
of the magnitude it works on, so the bound holds under cancellation where a fixed atol would not, and stays tight where
the result is large.  `c` is stated once per kernel family below, with its reason.

Lists come from the engine (Engine.neighbor_list), which leaves spare capacity (HEADROOM), so cap_pairs > P; every pair
row at index P or above of an output is filled with a sentinel before the call and must be unchanged after it, and every
pair row at index P or above of an input is NaN, so a kernel that reads past the count poisons its result.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from conftest import load_case, load_weights

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
U = 2.0 ** -24
CUTOFF = 5.0

# c per kernel family
C_EW = 8        # element-wise kernels (a few fp32 roundings per output: unit, dist, equivariant update)
C_GEOM = 32     # rbf / drbf: Horner envelope (9 fmaf), 1/x, sincosf (<= 2 ulp), 3-4 products; cos/sin cancellation is in mag
C_SUM = 32      # SIMT sums and dot products: fp32 fma chains of 20 (We rbf) to 400 (longest aggregation row) terms, whose
                # error grows like sqrt(n) 2^-24 of the sum of |terms| in practice; warp-tree dot products of 128 terms
C_TC = 64       # 3xTF32 (hi*hi + hi*lo + lo*hi): the dropped lo*lo term and the tf32 rounding of the lo parts are about
                # 2^-22 of each product, 96 products are accumulated in fp32 in the tensor core, then two fp32 products


def _lib():
    from newtonnet_b200 import _lib as L
    return L, L.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _within(got, ref, mag, c, what):
    """Assert the tolerance rule element-wise; returns the largest |got - ref| / (2^-24 mag) for reporting."""
    got, ref, mag = got.double(), ref.double(), mag.double()
    err = (got - ref).abs()
    bound = c * U * mag
    bad = ~(err <= bound)
    if bool(bad.any()):
        k = int(bad.reshape(-1).nonzero()[0])
        raise AssertionError(f'{what}: {int(bad.sum())} of {bad.numel()} elements exceed {c} * 2^-24 * mag; first at flat '
                             f'index {k}: got {float(got.reshape(-1)[k])!r}, ref {float(ref.reshape(-1)[k])!r}, '
                             f'mag {float(mag.reshape(-1)[k])!r}')
    return float((err / (U * mag).clamp_min(1e-300)).max())


def _engine_list(pos, cell, batch):
    """A complete neighbour list of the engine (fresh engine: a cached list of the same shape would be rebuilt in place)."""
    from newtonnet_b200 import _lib as L
    from newtonnet_b200.engine import Engine
    t = lambda a: torch.as_tensor(np.asarray(a), device=DEV)
    nl = Engine(torch.device(DEV)).neighbor_list(t(pos), t(cell).float(), t(batch), CUTOFF)
    st = nl.check()
    assert st[L.ST_EDGE_OVERFLOW] == 0
    P = st[L.ST_N_PAIRS]
    assert nl.cap_pairs > P
    return nl, P


def _chains(P, seed=0):
    """Non-periodic straight chains with 4 A spacing (nearest neighbours only: k atoms give k - 1 pairs) whose pair counts
    sum to exactly P: 128-pair chains plus one shorter chain for the remainder."""
    rng = np.random.default_rng(seed)
    lens = [128] * (P // 128) + ([P % 128] if P % 128 else [])
    pos, batch = [], []
    for b, k in enumerate(lens):
        x = np.arange(k + 1) * 4.0
        pos.append(np.stack([x, rng.uniform(-0.2, 0.2, k + 1), rng.uniform(-0.2, 0.2, k + 1)], 1))
        batch.append(np.full(k + 1, b, np.int64))
    return np.concatenate(pos).astype(np.float32), np.zeros((len(lens), 3, 3), np.float32), np.concatenate(batch)


def _ball(rng, n, r_lo, r_hi):
    v = rng.standard_normal((n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return v * rng.uniform(r_lo, r_hi, (n, 1))


def _mixed_list():
    """One non-periodic batch with the row shapes the reductions must handle: a dense cluster whose centre atom has 400
    neighbours (> 256; NN_MAX_DEGREE is 512), stars whose centre rows hold exactly 32 and 33 edges, a one-atom system, a
    chain (end rows of 1 edge) with an isolated atom in the same system, and an empty system."""
    rng = np.random.default_rng(11)
    parts = [np.vstack([np.zeros((1, 3)), _ball(rng, 400, 0.05, 4.95)]),       # system 0: centre row of 400 edges
             np.vstack([np.zeros((1, 3)), _ball(rng, 32, 1.5, 4.9)]),         # system 1: centre row of 32 edges
             np.vstack([np.zeros((1, 3)), _ball(rng, 33, 1.5, 4.9)]),         # system 2: centre row of 33 edges
             np.zeros((1, 3)),                                                 # system 3: one atom
             None,                                                             # system 4: no atoms
             np.vstack([np.stack([np.arange(20) * 4.0, np.zeros(20), np.zeros(20)], 1), [[-50.0, 0.0, 0.0]]])]   # 5
    pos = np.concatenate([p for p in parts if p is not None]).astype(np.float32)
    batch = np.concatenate([np.full(len(p), b, np.int64) for b, p in enumerate(parts) if p is not None])
    cell = np.zeros((len(parts), 3, 3), np.float32)
    return _engine_list(pos, cell, batch)


@pytest.fixture
def backend_state():
    """Restores the library's default backend after a test that switches it."""
    _, lib = _lib()
    yield lib
    lib.nn_set_gemm_backend(2)


def _rand(g, *shape):
    return torch.randn(*shape, generator=g).to(DEV)


def _pair_rows(g, cap, P, width, fill=float('nan')):
    """[cap, width] random rows; rows P.. hold `fill`."""
    t = _rand(g, cap, width)
    t[P:] = fill
    return t


def _np_count(nl):
    from newtonnet_b200 import _lib as L
    return nl.status[L.ST_N_PAIRS:].data_ptr()       # device pointer to the pair count


# ----------------------------------------------------------------------------- nn_edge_geom_fwd
def _geom_ref(disp, dist_got, freq, cutoff):
    """fp64 reference of rbf / drbf at the kernel's own fp32 argument: x = fp32(dist / rc) and f_n x rounded to fp32 as
    the kernel computes them (the rounding of an argument up to 20 pi ~ 63 alone moves sin by ~63 * 2^-24; that error is
    in the input, not in the kernel).  dist itself is checked against the fp64 norm."""
    x32 = (dist_got.cpu().float() / np.float32(cutoff)).double()          # IEEE division, as __fdiv_rn
    fx32 = (freq.cpu().float()[None, :] * x32.float()[:, None]).double()  # fp32 product, as the kernel's fr * x
    x = x32[:, None]
    t = 1.0 - x
    env = 1 - 55 * x ** 9 + 99 * x ** 10 - 45 * x ** 11
    env_fact = t ** 3 * sum(math.comb(k + 2, 2) * x ** k for k in range(9))     # same polynomial, no cancellation
    envp = -495 * x ** 8 * t ** 2
    sn, cs = torch.sin(fx32), torch.cos(fx32)
    rbf = env_fact * sn / x
    drbf = envp * sn / x + env_fact * (fx32 * cs - sn) / (x * x)
    mag_rbf = env_fact.abs() * sn.abs() / x
    mag_drbf = envp.abs() * sn.abs() / x + env_fact.abs() * ((fx32 * cs).abs() + sn.abs()) / (x * x)
    assert torch.allclose(env, env_fact, rtol=0, atol=1e-12)
    return rbf, drbf, mag_rbf, mag_drbf, fx32, env_fact / x


@pytest.mark.parametrize('count', ['device_count_below_cap', 'null_count'])
def test_edge_geom_fwd(count):
    L, lib = _lib()
    nl, P = _mixed_list()
    cap = nl.cap_pairs
    freq = torch.tensor(load_weights('seed0')['embedding_layers.edge_embedding.embedding.frequencies'], device=DEV)
    assert freq.numel() == 20 and float(freq.max()) > 62.0          # all 20 frequencies, arguments up to 20 pi
    disp = nl.pair_disp
    if count == 'null_count':                                       # no device count: every row of `cap` is a pair
        disp, cap = nl.pair_disp[:P].clone(), P
    n_dev = _np_count(nl) if count != 'null_count' else None
    sent = 7.0
    outs = {k: torch.full((cap, w), sent, device=DEV) for k, w in (('rbf', 20), ('drbf', 20), ('unit', 3), ('dist', 1))}
    L.check(lib.nn_edge_geom_fwd(disp.data_ptr(), freq.data_ptr(), CUTOFF, n_dev, cap, outs['rbf'].data_ptr(),
                                 outs['drbf'].data_ptr(), outs['unit'].data_ptr(), outs['dist'].data_ptr(), _stream()),
            'nn_edge_geom_fwd')
    # drbf = NULL: the same rbf / unit / dist, nothing else written
    o2 = {k: torch.full_like(v, sent) for k, v in outs.items()}
    L.check(lib.nn_edge_geom_fwd(disp.data_ptr(), freq.data_ptr(), CUTOFF, n_dev, cap, o2['rbf'].data_ptr(), None,
                                 o2['unit'].data_ptr(), o2['dist'].data_ptr(), _stream()), 'nn_edge_geom_fwd')
    torch.cuda.synchronize()
    for k in ('rbf', 'unit', 'dist'):
        assert torch.equal(o2[k], outs[k]), k
    assert bool((o2['drbf'] == sent).all())
    for k, v in outs.items():
        assert bool((v[P:] == sent).all()), f'{k}: rows past the pair count were written'
    d64 = disp[:P].double()
    dist_ref = d64.norm(dim=1)
    x = dist_ref / CUTOFF
    assert float(dist_ref.min()) < 0.5 and float(x.max()) > 0.999        # distances from below 0.5 A to just under rc
    _within(outs['dist'][:P, 0], dist_ref, dist_ref, C_EW, 'dist')
    _within(outs['unit'][:P], d64 / dist_ref[:, None], (d64 / dist_ref[:, None]).abs(), C_EW, 'unit')
    rbf, drbf, mag_r, mag_d, fx32, env_over_x = _geom_ref(disp[:P], outs['dist'][:P, 0], freq, CUTOFF)
    got_r, got_d = outs['rbf'][:P].cpu(), outs['drbf'][:P].cpu()
    _within(got_r, rbf, mag_r, C_GEOM, 'rbf')
    _within(got_d, drbf, mag_d, C_GEOM, 'drbf')
    # the rbf bound has teeth: a sine whose argument is reduced in fp32 (__sinf class: absolute error ~ |f x| 2^-24 on
    # top of its 2^-21.41 core error) would exceed it at every argument above 32
    big = fx32 > 32
    assert int(big.sum()) > 1000
    sinf_err = (fx32 * U + 2.0 ** -21.41) * env_over_x
    assert bool((sinf_err[big] > C_GEOM * U * mag_r[big]).all())


# ----------------------------------------------------------------------------- nn_edge_geom_bwd
@pytest.mark.parametrize('n_slots', [1, 2, 6])
def test_edge_geom_bwd(n_slots):
    L, lib = _lib()
    nl, P = _mixed_list()
    cap = nl.cap_pairs
    g = torch.Generator().manual_seed(20 + n_slots)
    unit = torch.full((cap, 3), float('nan'), device=DEV)
    dist = torch.full((cap,), float('nan'), device=DEV)
    freq = torch.tensor(load_weights('seed0')['embedding_layers.edge_embedding.embedding.frequencies'], device=DEV)
    rbf = torch.empty(cap, 20, device=DEV)
    L.check(lib.nn_edge_geom_fwd(nl.pair_disp.data_ptr(), freq.data_ptr(), CUTOFF, _np_count(nl), cap, rbf.data_ptr(), None,
                                 unit.data_ptr(), dist.data_ptr(), _stream()), 'nn_edge_geom_fwd')
    x_bar = torch.randn(n_slots, cap, generator=g).to(DEV)
    x_bar[:, P:] = float('nan')
    ubar = _pair_rows(g, cap, P, 3)
    out = torch.full((cap, 3), 7.0, device=DEV)
    L.check(lib.nn_edge_geom_bwd(x_bar.data_ptr(), n_slots, ubar.data_ptr(), unit.data_ptr(), dist.data_ptr(), CUTOFF,
                                 _np_count(nl), cap, out.data_ptr(), _stream()), 'nn_edge_geom_bwd')
    torch.cuda.synchronize()
    assert bool((out[P:] == 7.0).all())
    u, d, ub, xb = unit[:P].double(), dist[:P].double()[:, None], ubar[:P].double(), x_bar[:, :P].double()
    ref = (xb.sum(0)[:, None] / CUTOFF) * u + (ub - (ub * u).sum(1, keepdim=True) * u) / d
    mag = (xb.abs().sum(0)[:, None] / CUTOFF) * u.abs() + (ub.abs() + (ub.abs() * u.abs()).sum(1, keepdim=True) * u.abs()) / d
    _within(out[:P], ref, mag, C_EW + n_slots, 'disp_bar')


# ----------------------------------------------------------------------------- nn_edge_message_fwd
def _tf32(x):
    """Round fp32 to tf32 (10-bit mantissa, nearest, ties away) as cvt.rna.tf32.f32 does."""
    b = x.float().contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1fff).view(torch.float32)


@pytest.mark.parametrize('P', [100, 640, 641, 18945, 37888, 37889])
@pytest.mark.parametrize('backend', [0, 2], ids=['simt', 'tcgen05'])
def test_edge_message_fwd(backend, P, backend_state):
    """P: below one 128-pair tile; 5 tiles exactly and one pair more; 149 tiles (a CTA of the persistent tensor-core kernel
    takes a second tile: the other TMEM accumulator); 2 * 148 tiles exactly and one pair more (a third tile: the first
    accumulator is reused with its phase flipped, and the epilogue's gather window crosses two tile boundaries)."""
    L, lib = _lib()
    lib.nn_set_gemm_backend(backend)
    pos, cell, batch = _chains(P)
    nl, P_got = _engine_list(pos, cell, batch)
    assert P_got == P
    cap, N = nl.cap_pairs, nl.n_atoms
    g = torch.Generator().manual_seed(P)
    rbf, mn, We = _pair_rows(g, cap, P, 20), _rand(g, N, 128), _rand(g, 128, 20) / 4
    Wet = We.t().contiguous()
    img = torch.empty(L.NN_WE_IMAGE_FLOATS, device=DEV)
    L.check(lib.nn_message_prepare_b(We.data_ptr(), img.data_ptr(), _stream()), 'nn_message_prepare_b')
    msg = torch.full((cap, 128), 7.0, device=DEV)
    L.check(lib.nn_edge_message_fwd(C.byref(nl.struct), rbf.data_ptr(), mn.data_ptr(), Wet.data_ptr(),
                                    img.data_ptr() if backend else None, msg.data_ptr(), _stream()), 'nn_edge_message_fwd')
    torch.cuda.synchronize()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles, grid = -(-P // 128), min(-(-cap // 128), sms)
    per_cta = -(-tiles // grid)
    print(f'P={P} cap_pairs={cap} tiles={tiles} CTAs={grid} max tiles per CTA={per_cta}')
    assert per_cta == {18945: 2, 37888: 2, 37889: 3}.get(P, 1)
    assert bool((msg[P:] == 7.0).all()), 'rows past the pair count were written'
    i, j = nl.pair_i[:P].long(), nl.pair_j[:P].long()
    R, W, MN = rbf[:P].double(), We.double(), mn.double()
    ref = (R @ W.t()) * MN[i] * MN[j]
    mag = (R.abs() @ W.abs().t()) * MN[i].abs() * MN[j].abs()
    worst = _within(msg[:P], ref, mag, C_TC if backend else C_SUM, 'msg')
    print(f'largest error {worst:.2f} * 2^-24 * mag')
    if backend:
        # the bound has teeth: single-pass TF32 (no hi/lo correction) must violate it
        one_pass = (_tf32(rbf[:P]).double() @ _tf32(We).double().t()) * MN[i] * MN[j]
        assert bool(((one_pass - ref).abs() > C_TC * U * mag).any())


# ----------------------------------------------------------------------------- nn_node_aggregate_fwd
@pytest.mark.parametrize('first_layer', [0, 1])
def test_node_aggregate_fwd(first_layer):
    L, lib = _lib()
    nl, P = _mixed_list()
    cap, N = nl.cap_pairs, nl.n_atoms
    deg = (nl.row_ptr[1:] - nl.row_ptr[:-1]).cpu()
    for k in (0, 1, 32, 33):
        assert bool((deg == k).any()), f'no row of {k} edges'
    assert int(deg.max()) > 256
    g = torch.Generator().manual_seed(30 + first_layer)
    msg, e1, e2 = _pair_rows(g, cap, P, 128), _pair_rows(g, cap, P, 128), _pair_rows(g, cap, P, 128)
    unit = _pair_rows(g, cap, P, 3)
    a_in, f_in = _rand(g, N, 128), _rand(g, N, 3, 128)
    a_out, f_out = torch.full((N, 128), 7.0, device=DEV), torch.full((N, 3, 128), 7.0, device=DEV)
    L.check(lib.nn_node_aggregate_fwd(C.byref(nl.struct), msg.data_ptr(), e1.data_ptr(), e2.data_ptr(), unit.data_ptr(),
                                      a_in.data_ptr(), None if first_layer else f_in.data_ptr(), a_out.data_ptr(),
                                      f_out.data_ptr(), first_layer, _stream()), 'nn_node_aggregate_fwd')
    torch.cuda.synchronize()
    ei = nl.edge_index()
    E = ei.shape[1]
    assert E == 2 * P
    ep = nl.edge_pair[:E].long()
    pair, sgn = ep & 0x7fffffff, torch.where(ep < 0, -1.0, 1.0).double()
    assert bool((sgn < 0).any()) and bool((sgn > 0).any())              # both orientations (bit 31) occur
    k, j = ei[0], ei[1]
    M, E1, E2, Un, A, Fi = msg.double(), e1.double(), e2.double(), unit.double(), a_in.double(), f_in.double()
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=DEV)
    ref_a = A.clone().index_add_(0, k, M[pair])
    mag_a = A.abs().index_add_(0, k, M[pair].abs())
    su = sgn[:, None] * Un[pair]                                        # [E,3]: the edge's own orientation
    vec = su[:, :, None] * E1[pair][:, None, :]
    avec = su.abs()[:, :, None] * E1[pair].abs()[:, None, :]
    if not first_layer:
        vec = vec + E2[pair][:, None, :] * Fi[j]
        avec = avec + E2[pair].abs()[:, None, :] * Fi[j].abs()
    ref_f = (z(N, 3, 128) if first_layer else Fi.clone()).index_add_(0, k, vec)
    mag_f = (z(N, 3, 128) if first_layer else Fi.abs()).index_add_(0, k, avec)
    _within(a_out, ref_a, mag_a, C_SUM, 'a_out')
    _within(f_out, ref_f, mag_f, C_SUM, 'f_out')
    iso = (deg == 0).nonzero()[:, 0].to(DEV)
    assert torch.equal(a_out[iso], a_in[iso])
    assert torch.equal(f_out[iso], torch.zeros_like(f_out[iso]) if first_layer else f_in[iso])


# ----------------------------------------------------------------------------- nn_equiv_update_fwd
@pytest.mark.parametrize('N', [1, 77, 3001])
def test_equiv_update_fwd(N):
    L, lib = _lib()
    g = torch.Generator().manual_seed(N)
    a, f, gg = _rand(g, N, 128), _rand(g, N, 3, 128), _rand(g, N, 3, 128)
    out = torch.full((N + 1, 128), 7.0, device=DEV)
    L.check(lib.nn_equiv_update_fwd(a.data_ptr(), f.data_ptr(), gg.data_ptr(), out.data_ptr(), N, _stream()),
            'nn_equiv_update_fwd')
    torch.cuda.synchronize()
    assert bool((out[N] == 7.0).all())
    ref = a.double() + (f.double() * gg.double()).sum(1)
    mag = a.double().abs() + (f.double().abs() * gg.double().abs()).sum(1)
    _within(out[:N], ref, mag, C_EW, 'a_out')


# ----------------------------------------------------------------------------- nn_energy_head_fwd
def test_energy_head_fwd():
    """Shifts of 10^3 - 10^4 eV, z over the whole table 1..118, an empty and a one-atom system in the batch."""
    L, lib = _lib()
    g = torch.Generator().manual_seed(40)
    sizes = [300, 0, 1, 2000, 77]
    N, B = sum(sizes), len(sizes)
    sys_ptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32, device=DEV)
    z = (torch.arange(N) % 118 + 1).to(DEV)
    h2, w3, b3 = _rand(g, N, 128) * 2, _rand(g, 128) / 8, _rand(g, 1)
    scale = (torch.rand(119, generator=g) + 0.5).to(DEV)
    shift = (-(10.0 ** (3 + torch.rand(119, generator=g)))).to(DEV)
    e_atom, energy = torch.full((N + 8,), 7.0, device=DEV), torch.full((B + 1,), 7.0, device=DEV)
    L.check(lib.nn_energy_head_fwd(h2.data_ptr(), w3.data_ptr(), b3.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                   z.data_ptr(), sys_ptr.data_ptr(), N, B, e_atom.data_ptr(), energy.data_ptr(), _stream()),
            'nn_energy_head_fwd')
    torch.cuda.synchronize()
    assert bool((e_atom[N:] == 7.0).all()) and float(energy[B]) == 7.0
    hd = h2.double()
    s = hd * torch.sigmoid(hd)
    o = s @ w3.double() + b3.double()
    ref = o * scale.double()[z] + shift.double()[z]
    mag = ((s.abs() @ w3.double().abs()) + b3.double().abs()) * scale.double()[z] + shift.double()[z].abs()
    _within(e_atom[:N], ref, mag, C_SUM, 'e_atom')
    # per-system energy = the fp64 sum of the kernel's own e_atom, rounded to fp32 once (within one fp32 ulp)
    ea = e_atom[:N].double().cpu().numpy()
    ptr = sys_ptr.cpu().numpy()
    want = np.array([ea[ptr[b]:ptr[b + 1]].sum() for b in range(B)])
    got = energy[:B].cpu().numpy()
    w32 = want.astype(np.float32)
    assert np.all(np.abs(got.astype(np.float64) - w32) <= np.spacing(np.abs(w32))), (got, want)
    assert got[1] == 0.0                                                     # empty system
    assert got[2] == np.float32(ea[ptr[2]])                                  # one atom: its own energy, exactly
    e_ref = np.array([ref.cpu().numpy()[ptr[b]:ptr[b + 1]].sum() for b in range(B)])
    e_mag = np.array([mag.cpu().numpy()[ptr[b]:ptr[b + 1]].sum() for b in range(B)])
    assert np.all(np.abs(got - e_ref) <= C_SUM * U * e_mag + np.spacing(np.abs(w32)))


# ----------------------------------------------------------------------------- nn_force_virial_reduce
def _virial_ref(nl, P, G, pos, cell, batch):
    """forces = -dE/dpos and the virial / stress of the reference's strain convention (oracle.forward_analytic): per pair
    M = dpos (x) G - (cell^T G) (x) n with the image n solved in fp64, summed per system, symmetrised."""
    N, B = pos.shape[0], cell.shape[0]
    i, j = nl.pair_i[:P].long(), nl.pair_j[:P].long()
    Gd = G[:P].double()
    F = torch.zeros(N, 3, dtype=torch.float64, device=DEV)
    F = F.index_add(0, i, -Gd).index_add(0, j, Gd)
    Fm = torch.zeros(N, 3, dtype=torch.float64, device=DEV).index_add(0, i, Gd.abs()).index_add(0, j, Gd.abs())
    dpos = pos[i] - pos[j]
    M = dpos[:, :, None] * Gd[:, None, :]
    Mm = dpos.abs()[:, :, None] * Gd.abs()[:, None, :]
    if bool((cell != 0).any()):
        h = cell[batch[i]]
        n = torch.round(torch.linalg.solve(h.transpose(1, 2), dpos))
        M = M - torch.bmm(h.transpose(1, 2), Gd[:, :, None]) * n[:, None, :]
        Mm = Mm + torch.bmm(h.abs().transpose(1, 2), Gd.abs()[:, :, None]) * n.abs()[:, None, :]
    sb = batch[i]
    M = torch.zeros(B, 3, 3, dtype=torch.float64, device=DEV).index_add(0, sb, M)
    Mm = torch.zeros(B, 3, 3, dtype=torch.float64, device=DEV).index_add(0, sb, Mm)
    gD = 0.5 * (M + M.transpose(1, 2))
    gDm = 0.5 * (Mm + Mm.transpose(1, 2))
    return F, Fm, -gD, gDm


def _run_force_virial(nl, G, want_stress):
    L, lib = _lib()
    N, B = nl.n_atoms, nl.n_systems
    forces, virial = torch.full((N + 1, 3), 7.0, device=DEV), torch.full((B + 1, 9), 7.0, device=DEV)
    stress = torch.full((B + 1, 9), 7.0, device=DEV) if want_stress else None
    ws = torch.empty(N * 9, device=DEV)
    L.check(lib.nn_force_virial_reduce(C.byref(nl.struct), G.data_ptr(), forces.data_ptr(), virial.data_ptr(),
                                       L.ptr(stress), ws.data_ptr(), _stream()), 'nn_force_virial_reduce')
    torch.cuda.synchronize()
    assert bool((forces[N] == 7.0).all()) and bool((virial[B] == 7.0).all())
    if want_stress:
        assert bool((stress[B] == 7.0).all())
    return forces[:N], virial[:B].reshape(B, 3, 3), None if stress is None else stress[:B].reshape(B, 3, 3)


@pytest.mark.parametrize('name', ['water375', 'water192_ortho_unwrapped', 'water192_triclinic', 'mols24'])
def test_force_virial_reduce(name):
    """A cubic box (no strain-quirk term), a non-cubic orthorhombic box (quirk mode 1), a triclinic box (mode 2) and a
    molecule batch with zero cells (stress = NULL)."""
    d, _ = load_case(name)
    periodic = bool(np.any(d['cell'] != 0))
    nl, P = _engine_list(d['pos'], d['cell'], d['batch'])
    g = torch.Generator().manual_seed(50)
    G = _pair_rows(g, nl.cap_pairs, P, 3)
    forces, virial, stress = _run_force_virial(nl, G, periodic)
    pos, cell = nl.pos.double(), nl.cell.double()
    F, Fm, V, Vm = _virial_ref(nl, P, G, pos, cell, nl.batch)
    _within(forces, F, Fm, C_SUM, 'forces')
    _within(virial, V, Vm, C_SUM, 'virial')
    if periodic:
        det = torch.linalg.det(cell)[:, None, None]
        _within(stress, -V / det, Vm / det.abs(), C_SUM, 'stress')
        # the strain-quirk term matters on the non-cubic cells: the plain sum of disp (x) G would miss it
        i, j = nl.pair_i[:P].long(), nl.pair_j[:P].long()
        plain = (nl.pair_disp[:P].double()[:, :, None] * G[:P].double()[:, None, :]).sum(0)
        plain = -0.5 * (plain + plain.t())
        off = float((plain - V[0]).abs().max()) / float(Vm[0].max())
        assert (off > 100 * C_SUM * U) == (name != 'water375'), off


def test_force_virial_reduce_oracle_G():
    """The oracle's own fp64 dE/d disp, cast to fp32, reduced by the kernel: forces, virial and stress of the oracle."""
    from oracle import newtonnet_oracle as O
    d, w = load_case('water192_triclinic')
    nl, P = _engine_list(d['pos'], d['cell'], d['batch'])
    ei = nl.edge_index()
    ep = nl.edge_pair[:ei.shape[1]].long()
    sgn = torch.where(ep < 0, -1.0, 1.0)[:, None]
    disp = (sgn * nl.pair_disp[ep & 0x7fffffff]).double()                  # per directed edge: pos_i - pos_j, min image
    ref = O.forward_analytic(w, d['z'], d['pos'], d['cell'], d['batch'], edge_index=ei.cpu().numpy(),
                             disp=disp.cpu().numpy())
    pairs = ref['pairs']
    assert pairs.shape[1] == P
    key_nl = (nl.pair_i[:P].long() * nl.n_atoms + nl.pair_j[:P].long()).cpu().numpy()
    key_or = pairs[0] * nl.n_atoms + pairs[1]
    order = np.argsort(key_or)
    at = order[np.searchsorted(key_or[order], key_nl)]
    assert np.array_equal(key_or[at], key_nl)
    G = torch.full((nl.cap_pairs, 3), float('nan'), device=DEV)
    G[:P] = torch.tensor(ref['G'][at], dtype=torch.float32, device=DEV)
    forces, virial, stress = _run_force_virial(nl, G, True)
    Gd = torch.tensor(ref['G'][at], device=DEV).abs()
    i, j = nl.pair_i[:P].long(), nl.pair_j[:P].long()
    Fm = torch.zeros(nl.n_atoms, 3, dtype=torch.float64, device=DEV).index_add(0, i, Gd).index_add(0, j, Gd)
    _, _, _, Vm = _virial_ref(nl, P, G, nl.pos.double(), nl.cell.double(), nl.batch)
    # one more rounding per G element (the cast) than the kernel's own error
    _within(forces, torch.tensor(ref['forces'], device=DEV), Fm, C_SUM + 1, 'forces')
    _within(virial, torch.tensor(ref['virial'], device=DEV), Vm, C_SUM + 1, 'virial')
    det = abs(float(np.linalg.det(d['cell'][0].astype(np.float64))))
    _within(stress, torch.tensor(ref['stress'], device=DEV), Vm / det, C_SUM + 1, 'stress')


# ----------------------------------------------------------------------------- sliced per-system sums (nn_eval)
def _slice_bounds(n_atoms, sizes):
    """Atom indices on both sides of every slice boundary of nn_eval's two-level per-system sums (pair_ops.cu
    nn_sum_slices / k_sys_sum_partial: S = clamp(mean atoms per system / 2048, 1, 64) equal slices per system)."""
    S = min(max(n_atoms // len(sizes) // 2048, 1), 64)
    out, first = [], 0
    for n in sizes:
        for sl in range(1, S if n else 1):
            b = first + n * sl // S
            out += [b - 1, b]
        first += n
    return S, np.array(out, dtype=np.int64)


def _water_boxes(parts):
    from oracle import newtonnet_oracle as O
    zs, ps, cs, bs, sizes, boxes = [], [], [], [], [], []
    for b, (nside, seed) in enumerate(parts):
        if nside is None:                                                   # an empty system
            cs.append(np.eye(3, dtype=np.float32)[None] * 20.0); sizes.append(0); boxes.append(None)
            continue
        z, p, c, _ = O.water_box(nside, seed=seed)
        zs.append(z); ps.append(p); cs.append(c); bs.append(np.full(len(z), b, np.int64)); sizes.append(len(z))
        boxes.append((z, p, c))
    return np.concatenate(zs), np.concatenate(ps), np.concatenate(cs), np.concatenate(bs), sizes, boxes


@pytest.mark.parametrize('parts', [((12, 0),), ((16, 0),), ((13, 0), (None, None), (13, 1))],
                         ids=['water_box12_2slices', 'water_box16_6slices', 'two_water_box13_and_empty_2slices'])
def test_sliced_system_sums_against_oracle(parts):
    """Energy, forces, virial and stress of nn_eval where the per-system sums run in slices, against the fp64 oracle.  The
    energy and virial bounds are checked here to be smaller than what dropping or double-counting one atom at a slice
    boundary would change."""
    from newtonnet_b200.compat import model_from_state_dict
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch, sizes, boxes = _water_boxes(parts)
    N = len(z)
    S, bnd = _slice_bounds(N, sizes)
    assert S == {5184: 2, 12288: 6, 13182: 2}[N]
    w = load_weights('seed0')
    model = model_from_state_dict({k: torch.tensor(v) for k, v in w.items()},
                                  output_properties=['energy', 'gradient_force', 'stress', 'virial']).to(DEV)
    model.eval()
    t = lambda a: torch.tensor(a, device=DEV)
    out = model(t(z), t(pos), t(cell), t(batch))
    E = out.energy.cpu().double().numpy()
    Fg = out.gradient_force.cpu().double().numpy()
    V = out.virial.cpu().double().numpy().reshape(-1, 3, 3)
    Sg = out.stress.cpu().double().numpy().reshape(-1, 3, 3)
    atom_node = out.atom_node.cpu().double()
    sd = O.as_torch_sd(w, torch.float64)
    first = np.concatenate([[0], np.cumsum(sizes)])
    e_self = O.atomic_energy(sd, atom_node, torch.as_tensor(z)).reshape(-1).numpy()
    for b, box in enumerate(boxes):
        if box is None:
            assert E[b] == 0.0 and np.all(V[b] == 0.0)
            continue
        zb, pb, cb = box
        ei, disp = O.radius_graph_cell_list(pb, cb, np.zeros(len(zb), np.int64))
        ref = O.forward_analytic(w, zb, pb, cb, np.zeros(len(zb), np.int64), edge_index=ei, disp=disp)
        lo, hi = first[b], first[b + 1]
        mine = (bnd >= lo) & (bnd < hi)
        # energy: the GPU head on its own final features, summed in fp64, against the per-system sum.  4 fp32 ulps of |E|
        # must stay below the smallest |e_atom| at a slice boundary (an atom dropped or counted twice)
        e_tol = 4 * np.spacing(np.float32(abs(E[b])))
        e_err = abs(E[b] - e_self[lo:hi].sum())
        # virial: each atom's half-share of its incident pairs (the per-pair terms of the oracle), at the boundaries
        pi, pj = ref['pairs']
        Mp = ref['M']
        Ms = 0.5 * (Mp + Mp.transpose(0, 2, 1))
        share = np.zeros((len(zb), 3, 3))
        np.add.at(share, pi, 0.5 * Ms)
        np.add.at(share, pj, 0.5 * Ms)
        v_ref = ref['virial'][0]
        v_tol = 1e-4 * np.abs(v_ref).max()                      # the stress tolerance of the parity tests
        v_err = np.abs(V[b] - v_ref).max()
        smallest = np.abs(share[bnd[mine] - lo]).reshape(-1, 9).max(1).min()
        s_ref = ref['stress'][0]
        det = abs(np.linalg.det(cb[0].astype(np.float64)))
        print(f'system {b}: {hi - lo} atoms, {S} slices; |dE| {e_err:.2e} (tol {e_tol:.2e}, smallest boundary |e_atom| '
              f'{np.abs(e_self[bnd[mine]]).min():.3f}; vs oracle {abs(E[b] - ref["energy"][0]):.2e}); |dV| {v_err:.2e} '
              f'(tol {v_tol:.2e}, smallest boundary share {smallest:.3e}, |V| {np.abs(v_ref).max():.3e}); '
              f'|dS| {np.abs(Sg[b] - s_ref).max() * det:.2e}; |dF| {np.abs(Fg[lo:hi] - ref["forces"]).max():.2e}')
        assert e_tol < 0.5 * np.abs(e_self[bnd[mine]]).min()
        assert e_err <= e_tol, (E[b], e_self[lo:hi].sum())
        assert abs(E[b] - ref['energy'][0]) <= 1e-5 * abs(ref['energy'][0])           # north-star energy tolerance
        assert np.abs(Fg[lo:hi] - ref['forces']).max() < 1e-4                         # north-star force tolerance
        assert v_tol < 0.5 * smallest, (v_tol, smallest)
        assert v_err <= v_tol, (v_err, v_tol)
        assert np.abs(Sg[b] - s_ref).max() <= v_tol / det

"""GPU parity tests: the CUDA path (through the C ABI / the public NewtonNet API) against the CPU oracle
and the committed golden vectors of the unmodified reference.

Tolerances are those of BASELINE.json north_star: neighbour edge sets bit-exact, energies within 1e-5
relative, forces within 1e-4 eV/A (fp32 kernels compared with the reference run in fp64).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_case, load_weights

pytestmark = pytest.mark.gpu

E_RTOL = 1e-5      # north_star: energies within 1e-5 relative
F_ATOL = 1e-4      # north_star: forces within 1e-4 eV/A
CASES_EF = ['aspirin1', 'aspirin100', 'mols24', 'mols_edge', 'mols256']
CASES_PBC = ['water375', 'water81_smallL', 'water1029', 'water192_ortho_unwrapped', 'water_batch2']


def dev():
    return torch.device('cuda:0')


@pytest.fixture(scope='module', params=[0, 1, 2], ids=['simt', 'tcgen05', 'tcgen05_ts'])
def backend(request):
    from newtonnet_b200 import _lib
    lib = _lib.load()
    if request.param >= 1:
        probe = torch.zeros(128, 128, device=dev())
        if not _tc_available(lib, probe):
            pytest.skip('tcgen05 backend not built')
    lib.nn_set_gemm_backend(request.param)
    yield request.param
    lib.nn_set_gemm_backend(2)


def _tc_available(lib, probe):
    from newtonnet_b200 import _lib as L
    a = L.GemmArgs()
    y = torch.empty_like(probe)
    img = torch.empty(L.NN_B_IMAGE_FLOATS, device=probe.device)
    lib.nn_gemm128_prepare_b(probe.data_ptr(), img.data_ptr(), torch.cuda.current_stream().cuda_stream)
    a.X, a.B, a.B_img, a.Y, a.m = probe.data_ptr(), probe.data_ptr(), img.data_ptr(), y.data_ptr(), 128
    lib.nn_set_gemm_backend(1)
    rc = lib.nn_gemm128(C.byref(a), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc == 0


def make_model(weights, props):
    from newtonnet_b200.compat import model_from_state_dict
    m = model_from_state_dict({k: torch.tensor(v) for k, v in weights.items()}, output_properties=props)
    m = m.to(dev())
    m.eval()
    return m


def run_model(model, d):
    t = lambda a, dt=None: torch.tensor(a, device=dev()) if dt is None else torch.tensor(a, device=dev(), dtype=dt)
    return model(t(d['z']), t(d['pos']), t(d['cell']), t(d['batch']))


# ----------------------------------------------------------------------------- neighbour list (R2)
@pytest.mark.parametrize('name', CASES_EF + CASES_PBC + ['water192_triclinic'])
def test_edge_set_bit_exact(name):
    """Same edges in the same order as the reference's dense search, and bit-identical displacements."""
    from newtonnet_b200.layers.representations import RadiusGraph
    from oracle import newtonnet_oracle as O
    d, _ = load_case(name)
    ei, disp = RadiusGraph(5.0)(torch.tensor(d['pos'], device=dev()), torch.tensor(d['cell'], device=dev()),
                                torch.tensor(d['batch'], device=dev()))
    assert ei.dtype == torch.int64
    if name == 'water192_triclinic':
        # general cells: same formula, fp32 inverse instead of LAPACK LU ("parity unpinned" in SURVEY 8a R2);
        # the edge SET still has to agree with the reference on this fixture.
        got = set(map(tuple, ei.cpu().numpy().T.tolist()))
        ref = set(map(tuple, d['ref32_edge_index'].T.tolist()))
        assert got == ref
        return
    assert np.array_equal(ei.cpu().numpy(), d['ref32_edge_index'])
    _, dref = O.radius_graph_dense(torch.tensor(d['pos']), torch.tensor(d['cell']), torch.tensor(d['batch']))
    assert np.array_equal(disp.cpu().numpy(), dref.numpy())


def test_edge_set_large_box_and_batch():
    """C3 (3,000-atom water box) and a 512-molecule C2-shaped batch against the cell-list oracle."""
    from newtonnet_b200.layers.representations import RadiusGraph
    from oracle import newtonnet_oracle as O
    for z, pos, cell, batch in (O.water_box(10), O.molecule_batch(512, seed=3)):
        ei, disp = RadiusGraph(5.0)(torch.tensor(pos, device=dev()), torch.tensor(cell, device=dev()),
                                    torch.tensor(batch, device=dev()))
        ref_ei, ref_d = O.radius_graph_cell_list(pos, cell, batch)
        assert np.array_equal(ei.cpu().numpy(), ref_ei)
        assert np.array_equal(disp.cpu().numpy(), ref_d)


def test_neighbor_list_errors():
    from newtonnet_b200.layers.representations import RadiusGraph
    pos = torch.rand(8, 3, device=dev())
    with pytest.raises(ValueError):      # unsorted batch
        RadiusGraph(5.0)(pos, torch.zeros(2, 3, 3, device=dev()), torch.tensor([0, 1, 0, 1, 0, 1, 0, 1], device=dev()))
    cell = torch.zeros(1, 3, 3, device=dev()); cell[0, 0, 0] = 10.0      # partially periodic -> singular
    with pytest.raises(RuntimeError, match='singular'):
        RadiusGraph(5.0)(pos, cell, torch.zeros(8, dtype=torch.long, device=dev()))


# ----------------------------------------------------------------------------- dense contraction
def _gemm(lib, X, B, pro=0, epi=0, bias=None, aux1=None, aux2=None, aux3=None, m_dev=None, mul=1, Y=None, aux_out=None,
          aux_tiled=0):
    from newtonnet_b200 import _lib as L
    a = L.GemmArgs()
    Y = torch.empty_like(X) if Y is None else Y
    img = torch.empty(L.NN_B_IMAGE_FLOATS, device=X.device)
    L.check(lib.nn_gemm128_prepare_b(B.data_ptr(), img.data_ptr(), torch.cuda.current_stream().cuda_stream), 'prepare_b')
    a.X, a.B, a.B_img, a.Y = X.data_ptr(), B.data_ptr(), img.data_ptr(), Y.data_ptr()
    a.bias, a.aux1, a.aux2, a.aux3, a.aux_out = L.ptr(bias), L.ptr(aux1), L.ptr(aux2), L.ptr(aux3), L.ptr(aux_out)
    a.m_dev, a.m_dev_mul, a.m, a.prologue, a.epilogue, a.aux_tiled = L.ptr(m_dev), mul, X.shape[0], pro, epi, aux_tiled
    L.check(lib.nn_gemm128(C.byref(a), torch.cuda.current_stream().cuda_stream), 'nn_gemm128')
    return Y


@pytest.mark.parametrize('M', [1, 127, 128, 300, 3 * 211, 4099, 148 * 128 * 3 + 77])
def test_gemm128_variants(backend, M):
    from newtonnet_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device='cpu').manual_seed(M)
    r = lambda *s: torch.randn(*s, generator=g).to(dev())
    X, B, bias, aux = r(M, 128), r(128, 128) / 11.3, r(128), r(M, 128)
    Xd, Bd = X.double(), B.double()
    silu = lambda t: t * torch.sigmoid(t)
    dsilu = lambda t: torch.sigmoid(t) * (1 + t * (1 - torch.sigmoid(t)))
    tol = dict(rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(_gemm(lib, X, B, bias=bias).double(), Xd @ Bd + bias.double(), **tol)
    torch.testing.assert_close(_gemm(lib, X, B).double(), Xd @ Bd, **tol)
    torch.testing.assert_close(_gemm(lib, X, B, pro=L.PRO_SILU, bias=bias).double(), silu(Xd) @ Bd + bias.double(), **tol)
    torch.testing.assert_close(_gemm(lib, X, B, epi=L.EPI_DSILU, aux1=aux).double(), (Xd @ Bd) * dsilu(aux.double()), **tol)
    torch.testing.assert_close(_gemm(lib, X, B, epi=L.EPI_ADD, aux1=aux).double(), Xd @ Bd + aux.double(), **tol)
    torch.testing.assert_close(_gemm(lib, X, B, epi=L.EPI_MUL, aux1=aux).double(), (Xd @ Bd) * aux.double(), **tol)
    # SILU_SAVE: product of silu(X) and, in place of X, silu'(X)
    xs = X.clone()
    got = _gemm(lib, xs, B, pro=L.PRO_SILU_SAVE, bias=bias, aux_out=xs)
    torch.testing.assert_close(got.double(), silu(Xd) @ Bd + bias.double(), **tol)
    torch.testing.assert_close(xs.double(), dsilu(Xd), rtol=1e-5, atol=1e-6)
    # in-place accumulate and in-place X == Y
    acc = aux.clone()
    _gemm(lib, X, B, epi=L.EPI_ADD, aux1=acc, Y=acc)
    torch.testing.assert_close(acc.double(), Xd @ Bd + aux.double(), **tol)
    xin = X.clone()
    _gemm(lib, xin, B, epi=L.EPI_DSILU, aux1=aux, Y=xin)
    torch.testing.assert_close(xin.double(), (Xd @ Bd) * dsilu(aux.double()), **tol)
    if M % 3 == 0:
        n = M // 3
        abar, fbar, gg = r(n, 128), r(M, 128), r(M, 128)
        want = (Xd * abar.double().repeat_interleave(3, 0)) @ Bd + fbar.double() + abar.double().repeat_interleave(3, 0) * gg.double()
        got = _gemm(lib, X, B, pro=L.PRO_ROWSCALE3, epi=L.EPI_EQUIV_BWD, aux1=fbar, aux2=abar, aux3=gg)
        torch.testing.assert_close(got.double(), want, **tol)
    # device-side row count smaller than the launch capacity: rows beyond it are untouched
    if M > 130:
        cnt = torch.tensor([M - 100], dtype=torch.int32, device=dev())
        Y = torch.full_like(X, 7.0)
        _gemm(lib, X, B, m_dev=cnt, Y=Y)
        torch.testing.assert_close(Y[:M - 100].double(), (Xd @ Bd)[:M - 100], **tol)
        assert bool((Y[M - 100:] == 7.0).all())


# ----------------------------------------------------------------------------- edge features (R3-R6)
def test_edge_embedding_matches_oracle():
    from newtonnet_b200.layers.representations import EdgeEmbedding
    from oracle import newtonnet_oracle as O
    d, w = load_case('water375')
    emb = EdgeEmbedding(5.0, 20).to(dev())
    rbf, unit, ei = emb(torch.tensor(d['pos'], device=dev()), torch.tensor(d['cell'], device=dev()),
                        torch.tensor(d['batch'], device=dev()))
    sd = O.as_torch_sd(w, torch.float64)
    r64, u64, e64 = O.edge_embedding(sd, torch.tensor(d['pos']).double(), torch.tensor(d['cell']).double(),
                                     torch.tensor(d['batch']))
    assert np.array_equal(ei.cpu().numpy(), e64.numpy())
    # fp32 rounding of the argument f_n * x (up to 63 rad) alone is ~4e-6 on a value of magnitude ~5
    assert np.abs(rbf.cpu().double().numpy() - r64.numpy()).max() < 5e-5
    assert np.abs(unit.cpu().double().numpy() - u64.numpy()).max() < 1e-6


# ----------------------------------------------------------------------------- full path (R0-R10, B)
@pytest.mark.parametrize('name', CASES_EF)
def test_energy_forces_match_reference(backend, name):
    d, w = load_case(name)
    out = run_model(make_model(w, ['energy', 'gradient_force']), d)
    e = out.energy.cpu().double().numpy(); f = out.gradient_force.cpu().double().numpy()
    assert np.abs(e - d['ref64_energy']).max() <= E_RTOL * max(1.0, np.abs(d['ref64_energy']).max())
    np.testing.assert_allclose(e, d['ref64_energy'], rtol=E_RTOL, atol=1e-4)
    assert np.abs(f - d['ref64_forces']).max() < F_ATOL
    assert np.array_equal(out.edge_index.cpu().numpy(), d['ref32_edge_index'])
    if 'ref64_atom_node' in d:
        assert np.abs(out.atom_node.cpu().double().numpy() - d['ref64_atom_node']).max() < 1e-4
        assert np.abs(out.force_node.cpu().double().numpy() - d['ref64_force_node']).max() < 1e-4


@pytest.mark.parametrize('name', CASES_PBC + ['water192_triclinic'])
def test_periodic_energy_forces_stress_match_reference(backend, name):
    d, w = load_case(name)
    out = run_model(make_model(w, ['energy', 'gradient_force', 'stress', 'virial']), d)
    e = out.energy.cpu().double().numpy(); f = out.gradient_force.cpu().double().numpy()
    np.testing.assert_allclose(e, d['ref64_energy'], rtol=E_RTOL, atol=1e-4)
    assert np.abs(f - d['ref64_forces']).max() < F_ATOL
    s = out.stress.cpu().double().numpy(); v = out.virial.cpu().double().numpy()
    assert np.abs(v - d['ref64_virial']).max() < 1e-4 * max(1.0, np.abs(d['ref64_virial']).max())
    assert np.abs(s - d['ref64_stress']).max() < 1e-4 * np.abs(d['ref64_stress']).max() + 1e-8


def test_known_answer_md_traj(backend):
    """The reference's own trajectory scripts/md17_md/md.traj (201 frames, fp32 calculator on CUDA)."""
    kat = np.load(f'{GOLDEN}/md17_kat.npz')
    w = load_weights('md17')
    nf = kat['positions'].shape[0]
    d = dict(z=np.tile(kat['numbers'], nf), pos=kat['positions'].reshape(-1, 3).astype(np.float32),
             cell=np.zeros((nf, 3, 3), np.float32), batch=np.repeat(np.arange(nf), 21))
    out = run_model(make_model(w, ['energy', 'gradient_force']), d)
    e = out.energy.cpu().double().numpy(); f = out.gradient_force.cpu().double().numpy().reshape(nf, 21, 3)
    assert abs(e[0] - (-17591.8262)) < 0.02            # scripts/md17_md/md.log:2
    assert np.abs(e / kat['energy'] - 1).max() < E_RTOL
    assert np.abs(e - kat['energy']).max() < 8e-3      # a few fp32 ulps at 1.76e4 eV
    assert np.abs(f - kat['forces']).max() < F_ATOL


def test_c3_water_box_against_oracle(backend):
    """3,000-atom periodic water box (config 3): edges from the cell-list oracle, E/F/stress from the
    analytic fp64 oracle."""
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch = O.water_box(10)
    w = load_weights('seed0')
    ei, disp = O.radius_graph_cell_list(pos, cell, batch)
    ref = O.forward_analytic(w, z, pos, cell, batch, edge_index=ei, disp=disp)
    out = run_model(make_model(w, ['energy', 'gradient_force', 'stress']), dict(z=z, pos=pos, cell=cell, batch=batch))
    assert np.array_equal(out.edge_index.cpu().numpy(), ei)
    np.testing.assert_allclose(out.energy.cpu().double().numpy(), ref['energy'], rtol=E_RTOL)
    assert np.abs(out.gradient_force.cpu().double().numpy() - ref['forces']).max() < F_ATOL
    assert np.abs(out.stress.cpu().double().numpy() - ref['stress']).max() < 1e-4 * np.abs(ref['stress']).max()


def test_full_size_batch_properties(backend):
    """Config 2 at full size (4,096 molecules, ~140k atoms): size-independent properties -
    determinism, zero net force per molecule, invariance under a per-molecule rigid translation and
    under molecule reordering, and agreement with the oracle on a 64-molecule sample."""
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch = O.molecule_batch(4096, seed=1)
    w = load_weights('seed0')
    model = make_model(w, ['energy', 'gradient_force'])
    d = dict(z=z, pos=pos, cell=cell, batch=batch)
    o1 = run_model(model, d); e1 = o1.energy.clone(); f1 = o1.gradient_force.clone()
    o2 = run_model(model, d)
    assert torch.equal(e1, o2.energy) and torch.equal(f1, o2.gradient_force)        # deterministic
    net = torch.zeros(4096, 3, device=dev(), dtype=torch.float64).index_add_(0, torch.tensor(batch, device=dev()), f1.double())
    assert float(net.abs().max()) < 1e-3
    shift = np.random.default_rng(0).uniform(-3, 3, (4096, 3)).astype(np.float32)
    o3 = run_model(model, dict(z=z, pos=pos + shift[batch], cell=cell, batch=batch))
    assert float((o3.energy - e1).abs().max()) < 1e-3 and float((o3.gradient_force - f1).abs().max()) < 2e-4
    # oracle on the first 64 molecules
    n = int((batch < 64).sum())
    ref = O.forward(w, z[:n], pos[:n], cell[:64], batch[:n], dtype=torch.float64)
    np.testing.assert_allclose(e1[:64].cpu().double().numpy(), ref['energy'], rtol=E_RTOL, atol=1e-4)
    assert np.abs(f1[:n].cpu().double().numpy() - ref['forces']).max() < F_ATOL


def test_capacity_regrow_and_reuse():
    """Same atom count, denser second call: the cached capacity overflows and is regrown transparently."""
    from oracle import newtonnet_oracle as O
    w = load_weights('seed0')
    model = make_model(w, ['energy', 'gradient_force'])
    z, pos, cell, batch = O.water_box(6)
    o1 = run_model(model, dict(z=z, pos=pos, cell=cell, batch=batch))
    n1 = o1.edge_index.shape[1]
    pos2 = (pos * 0.8).astype(np.float32); cell2 = (cell * 0.8).astype(np.float32)
    o2 = run_model(model, dict(z=z, pos=pos2, cell=cell2, batch=batch))
    ei, disp2 = O.radius_graph_cell_list(pos2, cell2, batch)
    assert o2.edge_index.shape[1] == ei.shape[1] > 1.5 * n1
    assert np.array_equal(o2.edge_index.cpu().numpy(), ei)
    ref = O.forward_analytic(w, z, pos2, cell2, batch, edge_index=ei, disp=disp2)
    assert np.abs(o2.gradient_force.cpu().double().numpy() - ref['forces']).max() < F_ATOL


def test_other_hyperparameters_against_oracle():
    """2 interaction layers, cutoff 4.2 A, fp64 model and inputs (cast at the boundary), an empty system in the
    batch - against the oracle directly (no golden fixture needed: the oracle is pinned to the reference)."""
    from newtonnet_b200.models import NewtonNet
    from oracle import newtonnet_oracle as O
    torch.manual_seed(5)
    model = NewtonNet(cutoff=4.2, n_interactions=2, output_properties=['energy', 'gradient_force', 'stress']).double()
    with torch.no_grad():
        model.scalers[0].scale.weight.uniform_(0.5, 1.5); model.scalers[0].shift.weight.normal_()
    sd = {k: v.detach().float().numpy() for k, v in model.state_dict().items()}   # fp32-rounded weights for both sides
    model.load_state_dict({k: torch.tensor(v).double() for k, v in sd.items()})
    model = model.to(dev()); model.eval()
    z1, p1, c1, b1 = O.water_box(4, seed=8)
    z2, p2, c2, b2 = O.water_box(5, seed=9)
    z = np.concatenate([z1, z2]); pos = np.concatenate([p1, p2])
    cell = np.concatenate([c1, np.eye(3, dtype=np.float32)[None] * 20.0, c2])          # system 1 has no atoms
    batch = np.concatenate([b1, b2 + 2])
    out = model(torch.tensor(z, device=dev()), torch.tensor(pos, device=dev()).double(),
                torch.tensor(cell, device=dev()).double(), torch.tensor(batch, device=dev()))
    assert out.energy.dtype == torch.float64 and out.energy.shape == (3,)
    ref = O.forward(sd, z, pos, cell, batch, dtype=torch.float64, stress=True, cutoff=4.2)
    assert float(out.energy[1]) == 0.0 and ref['energy'][1] == 0.0
    np.testing.assert_allclose(out.energy.cpu().numpy(), ref['energy'], rtol=E_RTOL, atol=1e-4)
    assert np.abs(out.gradient_force.cpu().numpy() - ref['forces']).max() < F_ATOL
    assert np.array_equal(out.edge_index.cpu().numpy(), ref['edge_index'])
    s_ref = ref['stress'][[0, 2]]; s_got = out.stress.cpu().numpy()[[0, 2]]
    assert np.abs(s_got - s_ref).max() < 1e-4 * np.abs(s_ref).max()


@pytest.mark.parametrize('name', ['mols_edge', 'water81'])
def test_layer_norm_and_direct_force(backend, name):
    """layer_norm=True and the direct_force head (SURVEY 8f rank 2) against the unmodified reference; also the
    training-mode (autograd-composed) forward of the same model."""
    from newtonnet_b200.models import NewtonNet
    d = dict(np.load(f'{GOLDEN}/wide_{name}.npz'))
    w = load_weights('seed0')
    w.update({k[6:]: v for k, v in d.items() if k.startswith('extra.')})
    model = NewtonNet(layer_norm=True, output_properties=['energy', 'gradient_force', 'direct_force'])
    model.load_state_dict({k: torch.tensor(v) for k, v in w.items()}, strict=True)
    model = model.to(dev()); model.eval()
    out = run_model(model, d)
    np.testing.assert_allclose(out.energy.cpu().double().numpy(), d['ref64_energy'], rtol=E_RTOL, atol=1e-4)
    assert np.abs(out.gradient_force.cpu().double().numpy() - d['ref64_forces']).max() < F_ATOL
    assert np.abs(out.direct_force.cpu().double().numpy() - d['ref64_direct_force']).max() < F_ATOL
    assert np.abs(out.atom_node.cpu().numpy() - d['ref64_atom_node']).max() < 1e-4
    model.train()
    t = lambda a: torch.tensor(a, device=dev())
    tr = model(t(d['z']), t(d['pos']).requires_grad_(True), t(d['cell']), t(d['batch']))
    assert np.abs(tr.gradient_force.detach().cpu().double().numpy() - d['ref64_forces']).max() < F_ATOL
    assert np.abs(tr.direct_force.detach().cpu().double().numpy() - d['ref64_direct_force']).max() < F_ATOL


def test_head_order_and_energy_only():
    d, w = load_case('aspirin1')
    out = run_model(make_model(w, ['energy']), d)
    assert not hasattr(out, 'gradient_force')
    np.testing.assert_allclose(out.energy.cpu().double().numpy(), d['ref64_energy'], rtol=E_RTOL)
    m = make_model(w, ['energy', 'gradient_force'])
    m.output_properties = ['gradient_force', 'energy']      # heads are evaluated in list order, as in the reference
    with pytest.raises(AttributeError):
        run_model(m, d)


# ----------------------------------------------------------------------------- training step (row T)
@pytest.mark.parametrize('name', ['mols24', 'water81'])
def test_training_step_gradients_match_reference(name):
    """Loss and parameter gradients of one training step (double backward through the forces, composed by
    autograd from the C-ABI primitives) against the unmodified reference in train mode, fp64."""
    d = dict(np.load(f'{GOLDEN}/train_{name}.npz'))
    w = load_weights('seed0')
    model = make_model(w, ['energy', 'gradient_force'])
    model.train()
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    pos = t(d['pos']).requires_grad_(True)
    out = model(t(d['z']), pos, t(d['cell']), t(d['batch']))
    assert out.gradient_force.requires_grad
    loss = torch.nn.functional.mse_loss(out.energy, t(d['e_target'], torch.float32)) + \
        float(d['force_weight']) * torch.nn.functional.mse_loss(out.gradient_force, t(d['f_target'], torch.float32))
    loss.backward()
    assert abs(loss.item() - float(d['loss'])) < 1e-4 * abs(float(d['loss']))
    worst = 0.0
    for k, p in model.named_parameters():
        ref = d['grad.' + k]
        got = np.zeros(ref.shape) if p.grad is None else p.grad.cpu().double().numpy()
        scale = max(np.abs(ref).max(), 1e-3 * max(np.abs(d[kk]).max() for kk in d if kk.startswith('grad.')))
        err = np.abs(got - ref).max() / scale
        worst = max(worst, err)
        assert err < 1e-4, (k, err)       # measured: 7e-6 (tcgen05 3xTF32), 7e-7 (fp32 SIMT)
    assert model.interaction_layers[0].equiv_message2[0].weight.grad.abs().max().item() == 0.0
    # eval mode afterwards takes the fused inference path again and agrees with the training-mode forward
    model.eval()
    o2 = model(t(d['z']), t(d['pos']), t(d['cell']), t(d['batch']))
    assert float((o2.gradient_force - out.gradient_force.detach()).abs().max()) < 5e-5
    assert float((o2.energy - out.energy.detach()).abs().max()) < 1e-3


def test_training_primitives_double_backward():
    """Gemm / GemmTN / Gather / SegmentSum composed twice by autograd against torch-native fp64."""
    import torch.nn.functional as Fn
    from newtonnet_b200.train import Gather, SegmentSum, Segments, linear

    def mlp(M, mine, dt):
        g = torch.Generator().manual_seed(1)
        r = lambda *sh: torch.randn(*sh, generator=g)
        x0, W1, b1, W2, b2, tgt = r(M, 128), r(128, 128) / 11, r(128), r(128, 128) / 11, r(128), r(M, 128)
        x = x0.to(dev(), dt).requires_grad_(True)
        P = [t.to(dev(), dt).requires_grad_(True) for t in (W1, b1, W2, b2)]
        lin = linear if mine else Fn.linear
        y = lin(Fn.silu(lin(x, P[0], P[1])), P[2], P[3])
        e = (y * y).sum()
        gx, = torch.autograd.grad(e, x, create_graph=True)
        loss = ((gx - tgt.to(dev(), dt)) ** 2).mean() + e * 1e-3
        return [t.double().cpu() for t in torch.autograd.grad(loss, P)]

    for M in (64, 914):
        for a, b in zip(mlp(M, True, torch.float32), mlp(M, False, torch.float64)):
            assert float((a - b).abs().max() / b.abs().max()) < 5e-5

    def graph(mine, dt):
        g = torch.Generator().manual_seed(2)
        N, E = 300, 4000
        idx = torch.randint(0, N, (E,), generator=g).sort().values.to(dev())
        idx2 = idx[torch.randperm(E, generator=g).to(dev())]
        rows = torch.randn(N, 128, generator=g).to(dev(), dt).requires_grad_(True)
        w = torch.randn(E, 128, generator=g).to(dev(), dt).requires_grad_(True)
        tgt = torch.randn(N, 128, generator=g).to(dev(), dt)
        if mine:
            s1, s2 = Segments(idx, N), Segments(idx2, N)
            out = SegmentSum.apply(Gather.apply(rows, s1) * Gather.apply(rows, s2) * w, s1)
        else:
            out = torch.zeros(N, 128, dtype=dt, device=dev()).index_add(0, idx, rows[idx] * rows[idx2] * w)
        gr, = torch.autograd.grad((out ** 3).sum(), rows, create_graph=True)
        return [t.double().cpu() for t in torch.autograd.grad(((gr - tgt) ** 2).mean(), [rows, w])]

    for a, b in zip(graph(True, torch.float32), graph(False, torch.float64)):
        assert float((a - b).abs().max() / b.abs().max()) < 1e-5


def test_gathered_products_double_backward():
    """GMul (the message product reading node rows through the edge index) feeding a segment product, composed twice by
    autograd against torch-native fp64 indexing."""
    from newtonnet_b200.train import GMul, SegMulBG, Segments, SegmentSum

    def run(mine, dt):
        g = torch.Generator().manual_seed(3)
        N, E = 200, 3000
        i1 = torch.randint(0, N, (E,), generator=g).sort().values.to(dev())
        i2 = i1[torch.randperm(E, generator=g).to(dev())]
        r = lambda *sh: torch.randn(*sh, generator=g).to(dev(), dt)
        me, mn, f3, e2, tgt = r(E, 128).requires_grad_(True), r(N, 128).requires_grad_(True), r(N, 3, 128).requires_grad_(True), \
            r(E, 128).requires_grad_(True), r(N, 128)
        if mine:
            s1, s2 = Segments(i1, N), Segments(i2, N)
            m = GMul.apply(me, None, mn, s1, mn, s2)
            out = SegmentSum.apply(m, s1) + SegMulBG.apply(e2 * m, f3, s1, s2).sum(1)
        else:
            m = me * mn[i1] * mn[i2]
            v = (e2 * m).unsqueeze(1) * f3[i2]
            out = torch.zeros(N, 128, dtype=dt, device=dev()).index_add(0, i1, m) + \
                torch.zeros(N, 3, 128, dtype=dt, device=dev()).index_add(0, i1, v).sum(1)
        first = torch.autograd.grad((out ** 2).sum(), [mn, f3], create_graph=True)
        loss = ((first[0] - tgt) ** 2).mean() + (first[1] ** 2).mean()
        return [t.double().cpu() for t in torch.autograd.grad(loss, [me, mn, f3, e2])]

    for a, b in zip(run(True, torch.float32), run(False, torch.float64)):
        assert float((a - b).abs().max() / b.abs().max()) < 2e-5


def test_segment_products_double_backward():
    """SegOuter / SegMulBG and their gradient family (ContractCG, RowDotG, SumMulCGG): delta f_i = sum_{e->i} e1_e u_e + e2_e f_j
    (reference models/newtonnet.py:219-226) composed twice by autograd against torch-native fp64 indexing; the second index is
    grouped through a permutation, as the source-atom segments of the neighbour list are."""
    from newtonnet_b200.train import SegMulBG, SegOuter, Segments

    def run(mine, dt):
        g = torch.Generator().manual_seed(5)
        N, E = 150, 2500
        i1 = torch.randint(0, N, (E,), generator=g).sort().values.to(dev())
        i2 = i1[torch.randperm(E, generator=g).to(dev())]
        r = lambda *sh: torch.randn(*sh, generator=g).to(dev(), dt)
        e1, e2, u, f3, tgt = r(E, 128).requires_grad_(True), r(E, 128).requires_grad_(True), r(E, 3).requires_grad_(True), \
            r(N, 3, 128).requires_grad_(True), r(N, 3, 128)
        if mine:
            s1, s2 = Segments(i1, N), Segments(i2, N)
            out = SegOuter.apply(e1, u, s1) + SegMulBG.apply(e2, f3, s1, s2)
            out = out + SegMulBG.apply(e1, out, s1, s2)           # a second layer reading the first one's output
        else:
            z = lambda: torch.zeros(N, 3, 128, dtype=dt, device=dev())
            out = z().index_add(0, i1, e1.unsqueeze(1) * u.unsqueeze(2)) + z().index_add(0, i1, e2.unsqueeze(1) * f3[i2])
            out = out + z().index_add(0, i1, e1.unsqueeze(1) * out[i2])
        first = torch.autograd.grad((out ** 2).sum(), [u, f3, e1], create_graph=True)
        loss = ((first[1] - tgt) ** 2).mean() + (first[0] ** 2).mean() + (first[2] ** 2).mean()
        return [t.double().cpu() for t in torch.autograd.grad(loss, [e1, e2, u, f3])]

    for a, b in zip(run(True, torch.float32), run(False, torch.float64)):
        assert float((a - b).abs().max() / b.abs().max()) < 5e-5


def test_training_step_runs_and_reduces_loss():
    from newtonnet_b200.train import training_step
    d = dict(np.load(f'{GOLDEN}/train_mols24.npz'))
    model = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    args = (t(d['z']), t(d['pos']), t(d['cell']), t(d['batch']), t(d['e_target'], torch.float32), t(d['f_target'], torch.float32))
    losses = [training_step(model, opt, *args).item() for _ in range(5)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]


def test_weight_gradient_sink_matches_autograd(monkeypatch):
    """training_step with the weight gradients accumulated on the side stream (WeightGradSink) against the same step
    with every gradient returned to autograd: same sums, different order of the additions only."""
    from newtonnet_b200 import train
    d = dict(np.load(f'{GOLDEN}/train_mols24.npz'))
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    args = (t(d['z']), t(d['pos']), t(d['cell']), t(d['batch']), t(d['e_target'], torch.float32), t(d['f_target'], torch.float32))
    grads = {}
    for sink in ('1', '0'):
        monkeypatch.setenv('NN_TRAIN_SINK', sink)
        m = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
        opt = torch.optim.SGD(m.parameters(), lr=0.0)
        before = train.weight_grad_sink(dev()).launched if sink == '1' else 0
        for _ in range(2):                                 # the second step overwrites, it does not add to the first
            train.training_step(m, opt, *args, force_weight=float(d['force_weight']), clip_grad=0.0)
        if sink == '1':
            assert train.weight_grad_sink(dev()).launched - before >= 2 * 30
        torch.cuda.synchronize()
        grads[sink] = {k: (None if p.grad is None else p.grad.double().cpu()) for k, p in m.named_parameters()}
    assert train._weight_grad_mode == 'autograd'
    scale_all = max(float(g.abs().max()) for g in grads['0'].values() if g is not None)
    for k, ref in grads['0'].items():
        got = grads['1'][k]
        assert (got is None) == (ref is None), k
        if ref is not None:
            assert float((got - ref).abs().max()) <= 2e-6 * max(float(ref.abs().max()), 1e-3 * scale_all), k


@pytest.mark.parametrize('name', ['mols24', 'water81'])
def test_graphed_training_step_matches_eager(name):
    """forward + double backward replayed as one CUDA graph over a padded, static-shape edge list: same loss, same
    gradients (checked against the reference golden like the eager path), same parameters after Adam steps."""
    import os
    from newtonnet_b200.train import GraphedTrainingStep, training_step
    if not os.path.exists(f'{GOLDEN}/train_{name}.npz'):
        pytest.skip('no such fixture')
    d = dict(np.load(f'{GOLDEN}/train_{name}.npz'))
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    args = (t(d['z']), t(d['pos']), t(d['cell']), t(d['batch']), t(d['e_target'], torch.float32), t(d['f_target'], torch.float32))
    fw = float(d['force_weight'])
    m_e = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    m_g = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    o_e, o_g = torch.optim.SGD(m_e.parameters(), lr=0.0), torch.optim.SGD(m_g.parameters(), lr=0.0)
    step = GraphedTrainingStep(m_g, o_g, *args, force_weight=fw, clip_grad=0.0)
    assert step.nl.cap_edges >= step.check()[4]
    loss_g = step(*args)
    loss_e = training_step(m_e, o_e, *args, force_weight=fw, clip_grad=0.0)
    assert abs(loss_g.item() - float(d['loss'])) < 1e-4 * abs(float(d['loss']))
    assert abs(loss_g.item() - loss_e.item()) < 1e-5 * abs(loss_e.item())
    scale_all = max(np.abs(d[kk]).max() for kk in d if kk.startswith('grad.'))
    for (k, pe), (_, pg) in zip(m_e.named_parameters(), m_g.named_parameters()):
        ref = d['grad.' + k]
        got = np.zeros(ref.shape) if pg.grad is None else pg.grad.cpu().double().numpy()
        scale = max(np.abs(ref).max(), 1e-3 * scale_all)
        assert np.abs(got - ref).max() / scale < 1e-4, k
        if pe.grad is not None:
            assert np.abs(got - pe.grad.cpu().double().numpy()).max() / scale < 2e-5, k
    # new positions through the same graph; Adam steps follow the eager trajectory
    o_e, o_g = torch.optim.Adam(m_e.parameters(), lr=1e-3), torch.optim.Adam(m_g.parameters(), lr=1e-3)
    step.optimizer = o_g
    rng = np.random.default_rng(0)
    for _ in range(3):
        pos = args[1] + t(rng.normal(0, 0.02, d['pos'].shape), args[1].dtype)
        a2 = (args[0], pos) + args[2:]
        lg, le = step(*a2), training_step(m_e, o_e, *a2, force_weight=fw, clip_grad=0.0)
        assert abs(lg.item() - le.item()) < 1e-4 * abs(le.item())
    step.check()
    for (k, pe), (_, pg) in zip(m_e.named_parameters(), m_g.named_parameters()):
        assert float((pe - pg).abs().max()) < 1e-4 * max(float(pe.abs().max()), 1e-3), k


# ----------------------------------------------------------------------------- calculator (R0 caller)
class FakeAtoms:
    """Duck-typed ase.Atoms (ase is not installed in the image)."""

    def __init__(self, numbers, positions, cell=None, pbc=False):
        self.numbers = np.asarray(numbers); self.positions = np.asarray(positions, dtype=np.float64)
        self.cell = np.zeros((3, 3)) if cell is None else np.asarray(cell, dtype=np.float64)
        self.pbc = np.array([pbc] * 3 if isinstance(pbc, bool) else pbc)

    def __len__(self):
        return len(self.numbers)

    def copy(self):
        return FakeAtoms(self.numbers.copy(), self.positions.copy(), self.cell.copy(), self.pbc.copy())

    def get_atomic_numbers(self):
        return self.numbers

    def get_positions(self, wrap=False):
        if wrap and self.pbc.any():
            frac = np.linalg.solve(self.cell.T, self.positions.T).T
            frac[:, self.pbc] %= 1.0
            return frac @ self.cell
        return self.positions

    def get_cell(self):
        return self.cell

    def get_pbc(self):
        return self.pbc


def test_ase_calculator(tmp_path):
    from newtonnet_b200.compat import model_from_state_dict
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    kat = np.load(f'{GOLDEN}/md17_kat.npz')
    w = load_weights('md17')
    path = tmp_path / 'best_model.pt'
    torch.save(model_from_state_dict({k: torch.tensor(v).double() for k, v in w.items()}), path)   # fp64 pickle like the shipped one
    calc = MLAseCalculator(str(path), properties=['energy', 'forces'], device='cuda:0', precision='single')
    for k in (0, 100, 200):
        atoms = FakeAtoms(kat['numbers'], kat['positions'][k])
        calc.calculate(atoms)
        assert calc.results['energy'].shape == () and calc.results['forces'].shape == (21, 3)
        assert abs(float(calc.results['energy']) / kat['energy'][k] - 1) < E_RTOL
        assert np.abs(calc.results['forces'] - kat['forces'][k]).max() < F_ATOL
    calc.calculate([FakeAtoms(kat['numbers'], kat['positions'][k]) for k in range(4)])
    assert calc.results['energy'].shape == (4,) and calc.results['forces'].shape == (4, 21, 3)
    # periodic system with stress, Voigt order [xx,yy,zz,yz,xz,xy]
    d, ws = load_case('water375')
    torch.save(model_from_state_dict({k: torch.tensor(v) for k, v in ws.items()}), path)
    calc = MLAseCalculator(str(path), properties=['energy', 'forces', 'stress'], device='cuda:0')
    calc.calculate(FakeAtoms(d['z'], d['pos'], d['cell'][0], True))
    s = d['ref64_stress'][0]
    voigt = np.array([s[0, 0], s[1, 1], s[2, 2], s[1, 2], s[0, 2], s[0, 1]])
    assert calc.results['stress'].shape == (6,)
    assert np.abs(calc.results['stress'] - voigt).max() < 1e-4 * np.abs(voigt).max()
    assert np.abs(calc.results['forces'] - d['ref64_forces']).max() < F_ATOL


def test_hessian_through_the_calculator(tmp_path):
    """hessian head (SURVEY 8f rank 2) via MLAseCalculator, against the unmodified reference (fp64 golden)."""
    from newtonnet_b200.compat import model_from_state_dict
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    d = np.load(f'{GOLDEN}/hessian_aspirin1.npz')
    w = load_weights('md17')
    path = tmp_path / 'm.pt'
    torch.save(model_from_state_dict({k: torch.tensor(v) for k, v in w.items()}), path)
    calc = MLAseCalculator(str(path), properties=['energy', 'forces', 'hessian'], device='cuda:0')
    calc.calculate(FakeAtoms(d['z'], d['pos']))
    h = calc.results['hessian']
    assert h.shape == (21, 3, 21, 3)
    assert np.abs(h - d['hessian']).max() < 2e-3 and np.abs(d['hessian']).max() > 50
    assert np.abs(calc.results['forces'] - d['forces']).max() < F_ATOL


def test_training_path_regrows_neighbour_capacity():
    """Same atom count, denser second batch through the differentiable (training) path and through RadiusGraph: the
    cached edge capacity overflows and must be regrown, not truncated (round-1 advisor finding)."""
    from newtonnet_b200.layers.representations import RadiusGraph
    from oracle import newtonnet_oracle as O
    model = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    model.train()
    z, pos, cell, batch = O.water_box(5)
    t = lambda a: torch.tensor(a, device=dev())
    o1 = model(t(z), t(pos).requires_grad_(True), t(cell), t(batch))
    pos2 = (pos * 0.8).astype(np.float32); cell2 = (cell * 0.8).astype(np.float32)
    ei, _ = O.radius_graph_cell_list(pos2, cell2, batch)
    p2 = t(pos2).requires_grad_(True)
    o2 = model(t(z), p2, t(cell2), t(batch))
    assert o2.edge_index.shape[1] == ei.shape[1] > 1.5 * o1.edge_index.shape[1]
    (o2.energy.sum() + o2.gradient_force.square().sum()).backward()
    ref = O.forward(load_weights('seed0'), z, pos2, cell2, batch, dtype=torch.float64)
    assert np.abs(o2.gradient_force.detach().cpu().double().numpy() - ref['forces']).max() < F_ATOL
    rg = RadiusGraph(5.0)
    rg(t(pos), t(cell), t(batch))
    e2, d2 = rg(t(pos2), t(cell2), t(batch))
    assert np.array_equal(e2.cpu().numpy(), ei) and d2.shape[0] == ei.shape[1]


def test_graphed_training_step_refuses_overflowing_batch():
    """A replay whose batch outgrew the captured edge capacity must raise BEFORE the optimizer moves (advisor finding)."""
    from newtonnet_b200.train import GraphedTrainingStep
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch = O.water_box(4)
    rng = np.random.default_rng(0)
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    args = (t(z), t(pos), t(cell), t(batch), t(rng.standard_normal(1), torch.float32), t(rng.standard_normal(pos.shape), torch.float32))
    model = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    opt = torch.optim.SGD(model.parameters(), lr=1e-2)
    step = GraphedTrainingStep(model, opt, *args, regrow=False)
    step(*args)
    before = [p.detach().clone() for p in model.parameters()]
    dense = (args[0], t((pos * 0.7).astype(np.float32)), t((cell * 0.7).astype(np.float32))) + args[3:]
    with pytest.raises(RuntimeError, match='overflow'):
        step(*dense)
    assert all(torch.equal(a, b.detach()) for a, b in zip(before, model.parameters()))


def test_graphed_training_step_regrows_on_overflow():
    """Default behaviour: the edge capacity is tight (probed count + 5 %), and a batch that outgrows it is re-captured with
    more room and applied - same loss and same parameters as the eager step on the same batches."""
    from newtonnet_b200.train import GraphedTrainingStep, training_step
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch = O.water_box(4)
    rng = np.random.default_rng(0)
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    args = (t(z), t(pos), t(cell), t(batch), t(rng.standard_normal(1), torch.float32), t(rng.standard_normal(pos.shape), torch.float32))
    dense = (args[0], t((pos * 0.7).astype(np.float32)), t((cell * 0.7).astype(np.float32))) + args[3:]
    m_g = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    m_e = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    o_g, o_e = torch.optim.SGD(m_g.parameters(), lr=1e-3), torch.optim.SGD(m_e.parameters(), lr=1e-3)
    step = GraphedTrainingStep(m_g, o_g, *args)
    cap0 = step.nl.cap_edges
    assert cap0 < 1.2 * step.check()[4]
    for a in (args, dense, args):
        lg, le = step(*a), training_step(m_e, o_e, *a)
        assert abs(lg.item() - le.item()) < 1e-4 * abs(le.item())
    assert step.recaptures == 1 and step.nl.cap_edges > 1.5 * cap0
    for (k, pe), (_, pg) in zip(m_e.named_parameters(), m_g.named_parameters()):
        assert float((pe.detach() - pg.detach()).abs().max()) < 1e-4 * max(float(pe.detach().abs().max()), 1e-3), k


def test_graphed_training_step_deferred_overflow_check():
    """Fused Adam: no host synchronisation per step - the overflowing batch is skipped ON THE DEVICE (optimizer skip flag),
    found by the next call's settle(), re-captured and applied then.  Parameters follow the eager trajectory exactly."""
    from newtonnet_b200.train import GraphedTrainingStep, training_step
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch = O.water_box(4)
    rng = np.random.default_rng(0)
    t = lambda a, dt=None: torch.tensor(a, device=dev(), dtype=dt)
    args = (t(z), t(pos), t(cell), t(batch), t(rng.standard_normal(1), torch.float32), t(rng.standard_normal(pos.shape), torch.float32))
    dense = (args[0], t((pos * 0.7).astype(np.float32)), t((cell * 0.7).astype(np.float32))) + args[3:]
    m_g = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    m_e = make_model(load_weights('seed0'), ['energy', 'gradient_force'])
    o_g = torch.optim.Adam(m_g.parameters(), lr=1e-3, fused=True)
    o_e = torch.optim.Adam(m_e.parameters(), lr=1e-3, fused=True)
    step = GraphedTrainingStep(m_g, o_g, *args)
    assert step._device_skip()
    for k, a in enumerate((args, dense, args, dense)):
        before = [p.detach().clone() for p in m_g.parameters()]
        step(*a)
        training_step(m_e, o_e, *a)
        if k == 1:          # the dense batch did not fit: skipped on the device, nothing moved yet, one step pending
            torch.cuda.synchronize()
            assert step._pending and step.recaptures == 0
            assert all(torch.equal(x, y.detach()) for x, y in zip(before, m_g.parameters()))
    step.settle()
    assert step.recaptures == 1 and not step._pending
    assert int(o_g.state[next(iter(m_g.parameters()))]['step']) == 4
    for (k, pe), (_, pg) in zip(m_e.named_parameters(), m_g.named_parameters()):
        assert float((pe.detach() - pg.detach()).abs().max()) < 2e-4 * max(float(pe.detach().abs().max()), 1e-3), k


def test_reference_module_pickle_evaluates_like_the_reference():
    """Whole-module pickle of the current reference (with its les.Les aggregator member) -> load_model -> CUDA path;
    outputs against the reference's own outputs saved next to the pickle (tests/golden/make_pickle_golden.py)."""
    from newtonnet_b200.compat import load_model
    d = np.load(f'{GOLDEN}/ref_module_pickle.npz')
    model = load_model(f'{GOLDEN}/ref_module_pickle.pt', map_location=dev())
    model.eval()
    n = len(d['z'])
    out = model(torch.tensor(d['z'], device=dev()), torch.tensor(d['pos'], device=dev()), torch.zeros(1, 3, 3, device=dev()),
                torch.zeros(n, dtype=torch.long, device=dev()))
    assert abs(out.energy.item() - d['energy'][0]) <= 1e-5 * abs(d['energy'][0]) + 1e-5
    assert np.abs(out.gradient_force.cpu().numpy() - d['forces']).max() < F_ATOL


def test_training_mode_energy_only_head_gets_gradients():
    """model.train() with output_properties=['energy'] (trainable in the reference, train/loss.py) must produce outputs
    with a grad_fn (advisor finding: the inference path returned constants)."""
    model = make_model(load_weights('seed0'), ['energy'])
    model.train()
    from oracle import newtonnet_oracle as O
    z, pos, cell, batch = O.molecule_batch(4, seed=3)
    t = lambda a: torch.tensor(a, device=dev())
    out = model(t(z), t(pos), t(cell), t(batch))
    assert out.energy.grad_fn is not None
    out.energy.sum().backward()
    assert model.interaction_layers[0].message_nodepart[0].weight.grad is not None


@pytest.mark.parametrize('kind', ['tilted', 'strongly_tilted', 'unwrapped', 'far_outside', 'symmetric', 'batch_of_two'])
def test_general_cells_grid_search_matches_dense_reference_search(kind):
    """Non-diagonal cells are searched through a Cartesian grid + lattice-image enumeration (csrc/nbr.cu, mode 2) instead of
    all pairs; the result must equal the reference's dense search (layers/representations.py:86-98, incl. its `cell @ n`
    shift): same edges in the same order, displacements equal to fp32 rounding (the reference solves with LAPACK, here an
    fp32 inverse - SURVEY 8a R2 'unpinned')."""
    from newtonnet_b200.layers.representations import RadiusGraph
    from oracle import newtonnet_oracle as O
    rng = np.random.default_rng({'tilted': 1, 'strongly_tilted': 2, 'unwrapped': 3, 'far_outside': 4, 'symmetric': 5, 'batch_of_two': 6}[kind])
    def system(n, L, tilt):
        cell = np.diag(L).astype(np.float64)
        cell[1, 0], cell[2, 0], cell[2, 1] = tilt
        if kind == 'symmetric':
            cell = cell + np.tril(cell, -1).T
        frac = rng.random((n, 3))
        if kind == 'unwrapped':
            frac += rng.integers(-1, 2, (n, 3))
        if kind == 'far_outside':
            frac += rng.integers(-4, 5, (n, 3))
        return (frac @ cell).astype(np.float32), cell.astype(np.float32)
    tilt = {'tilted': (2.0, -1.5, 3.0), 'strongly_tilted': (7.0, 6.0, -8.0)}.get(kind, (1.5, 2.5, -2.0))
    if kind == 'batch_of_two':
        p1, c1 = system(150, (13.0, 15.0, 14.0), tilt)
        p2, c2 = system(90, (16.0, 11.0, 12.0), (0.0, 0.0, 0.0))
        pos, cell, batch = np.concatenate([p1, p2]), np.stack([c1, c2]), np.concatenate([np.zeros(150, np.int64), np.ones(90, np.int64)])
    else:
        pos, c, = system(260, (16.0, 14.0, 18.0), tilt)
        cell, batch = c[None], np.zeros(260, np.int64)
    ei, disp = RadiusGraph(5.0)(torch.tensor(pos, device=dev()), torch.tensor(cell, device=dev()), torch.tensor(batch, device=dev()))
    ref_ei, ref_d = O.radius_graph_dense(torch.tensor(pos), torch.tensor(cell), torch.tensor(batch))
    assert ref_ei.shape[1] > 1000
    assert np.array_equal(ei.cpu().numpy(), ref_ei.numpy())
    assert np.abs(disp.cpu().numpy() - ref_d.numpy()).max() < 2e-5


def test_ase_calculator_resident_md_path(tmp_path):
    """The calculator's steady-state path (device-resident z / cell / batch, one CUDA graph, one synchronisation): the same
    numbers as the general path, step after step; it follows changes of the cell, of the atomic numbers and of the model
    parameters, and it survives a capacity overflow (denser positions)."""
    from newtonnet_b200.compat import model_from_state_dict
    from newtonnet_b200.utils.ase_interface import MLAseCalculator
    d, ws = load_case('water375')
    model = model_from_state_dict({k: torch.tensor(v) for k, v in ws.items()})
    calc = MLAseCalculator(model, properties=['energy', 'forces', 'stress'], device='cuda:0')
    ref = MLAseCalculator(model_from_state_dict({k: torch.tensor(v) for k, v in ws.items()}), properties=['energy', 'forces', 'stress'],
                          device='cuda:0')
    import newtonnet_b200.engine as E
    rng = np.random.default_rng(0)
    pos, cell, z = d['pos'].astype(np.float64), d['cell'][0].astype(np.float64), d['z'].copy()

    def both(z_, pos_, cell_):
        calc.calculate(FakeAtoms(z_, pos_, cell_, True))
        ref._resident = None                                   # general path every time
        ref.calculate(FakeAtoms(z_, pos_, cell_, True))
        for k in ('energy', 'forces', 'stress'):
            assert np.array_equal(np.asarray(calc.results[k]), np.asarray(ref.results[k])), k

    for step in range(5):
        both(z, pos + rng.normal(0, 0.02, pos.shape), cell)
    assert calc._resident is not None and calc._resident['key'] is not None     # the resident path is active
    both(z, pos * 1.01, cell * 1.01)                           # cell change
    z2 = z.copy(); z2[::7] = 6
    both(z2, pos, cell)                                        # other atomic numbers
    both(z, pos * 0.85, cell * 0.85)                           # much denser: capacity overflow -> general path regrows
    both(z, pos * 0.85 + rng.normal(0, 0.01, pos.shape), cell * 0.85)
    with torch.no_grad():
        for m in (calc.model, ref.model):
            m.scalers[0].shift.weight.add_(0.5)
    both(z, pos, cell)                                         # parameter update is picked up


def test_fused_row_products_double_backward():
    """Mul3 / Outer / ContractC / RowDot / MulB / SumMulC (csrc/train_ops.cu): values, gradients and gradients of gradients
    against the broadcasting torch expressions they replace, in fp64."""
    from newtonnet_b200.train import ContractC, Mul3, MulB, Outer, RowDot, SumMulC

    def run(mine, dt):
        g = torch.Generator().manual_seed(3)
        n = 257
        r = lambda *sh: torch.randn(*sh, generator=g).to(dev(), dt).requires_grad_(True)
        a, b, c, x, u, y3, z3, tgt = r(n, 128), r(n, 128), r(n, 128), r(n, 128), r(n, 3), r(n, 3, 128), r(n, 3, 128), r(n, 128)
        if mine:
            m = Mul3.apply(a, b, c)
            vec = Outer.apply(x, u) + MulB.apply(m, y3)
            s = SumMulC.apply(vec, z3) + ContractC.apply(vec, u)
            d = RowDot.apply(vec, m)
        else:
            m = a * b * c
            vec = x.unsqueeze(1) * u.unsqueeze(2) + m.unsqueeze(1) * y3
            s = (vec * z3).sum(1) + (vec * u.unsqueeze(2)).sum(1)
            d = (vec * m.unsqueeze(1)).sum(-1)
        e = (s * s).sum() + (d ** 3).sum() * 1e-3
        leaves = [a, b, c, x, u, y3, z3]
        g1 = torch.autograd.grad(e, [x, u, y3], create_graph=True)
        loss = ((g1[0] - tgt) ** 2).mean() + (g1[1] ** 2).mean() + (g1[2] ** 2).mean() * 1e-2
        g2 = torch.autograd.grad(loss, leaves, allow_unused=True)
        outs = [s, d] + list(g1) + [t for t in g2 if t is not None]
        return [t.detach().double().cpu() for t in outs]

    for got, ref in zip(run(True, torch.float32), run(False, torch.float64)):
        assert got.shape == ref.shape
        assert float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)) < 2e-5


def test_fused_radial_basis_and_silu_double_backward():
    """RbfScale / RbfDot (env(x) sin(f x)/x with two x-derivatives) and Silu / SiluB against the torch expressions in fp64:
    value, gradient, gradient of the gradient; exact zeros at x = 1 (padding rows)."""
    import math
    from newtonnet_b200.train import RbfScale, silu
    freq32 = torch.tensor([np.float32(n * math.pi) for n in range(1, 21)], device=dev())

    def env(x):
        p = torch.zeros_like(x) + 45.0
        for c in (36.0, 28.0, 21.0, 15.0, 10.0, 6.0, 3.0, 1.0):
            p = p * x + c
        return (1.0 - x) ** 3 * p

    def run(mine, dt):
        g = torch.Generator().manual_seed(9)
        n = 333
        x = (torch.rand(n, 1, generator=g) * 0.9 + 0.08).to(dev(), dt).requires_grad_(True)
        w = torch.randn(n, 20, generator=g).to(dev(), dt).requires_grad_(True)
        h = torch.randn(n, 128, generator=g).to(dev(), dt).requires_grad_(True)
        f = freq32.to(dt)
        rbf = RbfScale.apply(torch.ones_like(x), x, freq32, 0) if mine else env(x) * torch.sin(f * x) / x
        act = silu(h) if mine else torch.nn.functional.silu(h)
        e = (rbf * w).sum() + (rbf ** 2).sum() + (act ** 2).sum()
        gx, gh = torch.autograd.grad(e, [x, h], create_graph=True)
        loss = (gx ** 2).sum() + (gh ** 3).sum()
        g2 = torch.autograd.grad(loss, [x, w, h])
        return [t.detach().double().cpu() for t in (rbf, act, gx, gh) + tuple(g2)]

    for got, ref in zip(run(True, torch.float32), run(False, torch.float64)):
        assert float((got - ref).abs().max() / ref.abs().max()) < 5e-5
    one = torch.ones(4, 1, device=dev(), requires_grad=True)
    r = RbfScale.apply(torch.ones_like(one), one, freq32, 0)
    g1, = torch.autograd.grad(r.sum(), one, create_graph=True)
    g2, = torch.autograd.grad(g1.sum(), one)
    assert float(r.abs().max()) == 0.0 and float(g1.abs().max()) == 0.0 and float(g2.abs().max()) == 0.0

"""The reverse-sweep operators of the C ABI, one by one, against fp64 torch restatements of their formulas
(SURVEY.md section 8a row B; oracle.forward_analytic is the end-to-end specification, checked in test_gpu_parity.py)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_case

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = dict(rtol=2e-5, atol=2e-5)


def _nl(name='mols24'):
    from newtonnet_b200.engine import get_engine
    d, _ = load_case(name)
    t = lambda a: torch.tensor(a, device=DEV)
    nl = get_engine(torch.device(DEV)).neighbor_list(t(d['pos']), t(d['cell']), t(d['batch']), 5.0)
    st = nl.check()
    P = st[5]
    return nl, nl.n_atoms, P


def _rand(g, *shape):
    return torch.randn(*shape, generator=g).to(DEV)


def _mat(W, keep):
    from newtonnet_b200 import _lib as L
    lib = L.load()
    s = torch.cuda.current_stream().cuda_stream
    m = L.Mat()
    w, wt = W.contiguous(), W.t().contiguous()
    imgs = [torch.empty(L.NN_B_IMAGE_FLOATS, device=DEV) for _ in range(2)]
    L.check(lib.nn_gemm128_prepare_b(w.data_ptr(), imgs[0].data_ptr(), s), 'prepare')
    L.check(lib.nn_gemm128_prepare_b(wt.data_ptr(), imgs[1].data_ptr(), s), 'prepare')
    m.w, m.wt, m.w_img, m.wt_img = w.data_ptr(), wt.data_ptr(), imgs[0].data_ptr(), imgs[1].data_ptr()
    keep += [w, wt] + imgs
    return m


@pytest.mark.parametrize('M,pair_level', [(300, False), (5000, True)])
def test_mlp_fwd_bwd(M, pair_level):
    from newtonnet_b200 import _lib as L
    lib = L.load(); lib.nn_set_gemm_backend(2)
    s = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(M)
    X, W1, W2, b1, b2, G, acc0 = _rand(g, M, 128), _rand(g, 128, 128) / 11, _rand(g, 128, 128) / 11, _rand(g, 128), _rand(g, 128), \
        _rand(g, M, 128), _rand(g, M, 128)
    keep = []
    M1, M2 = _mat(W1, keep), _mat(W2, keep)
    cnt = torch.tensor([M], dtype=torch.int32, device=DEV) if pair_level else None
    # `mid` is what nn_mlp_bwd consumes: whole tiles of 128 rows, tile-transposed when the chained kernel runs (NN_TILED_INDEX)
    Mp = (M + 127) // 128 * 128
    mid, Y = torch.zeros(Mp, 128, device=DEV), torch.empty_like(X)
    L.check(lib.nn_mlp_fwd(X.data_ptr(), C.byref(M1), b1.data_ptr(), mid.data_ptr(), C.byref(M2), b2.data_ptr(), Y.data_ptr(), M,
                           L.ptr(cnt), 1, s), 'nn_mlp_fwd')
    Xd = X.double().requires_grad_(True)
    pre = Xd @ W1.double().t() + b1.double()
    sig = torch.sigmoid(pre)
    want = (pre * sig) @ W2.double().t() + b2.double()
    torch.testing.assert_close(Y.double(), want.detach(), **TOL)
    mid_rows = mid
    if lib.nn_mlp_mid_tiled(M, int(pair_level)):
        mid_rows = mid.view(Mp // 128, 32, 128, 4).permute(0, 2, 1, 3).reshape(Mp, 128)      # [tile][chunk][row][4] -> rows
    torch.testing.assert_close(mid_rows[:M].double(), (sig * (1 + pre * (1 - sig))).detach(), rtol=2e-5, atol=2e-6)
    gX, = torch.autograd.grad(want, Xd, G.double())
    for accumulate in (0, 1):
        out = acc0.clone()
        tmp = torch.empty_like(X)
        L.check(lib.nn_mlp_bwd(G.data_ptr(), C.byref(M2), mid.data_ptr(), tmp.data_ptr(), C.byref(M1), out.data_ptr(), M, L.ptr(cnt),
                               accumulate, s), 'nn_mlp_bwd')
        torch.testing.assert_close(out.double(), gX + (acc0.double() if accumulate else 0), **TOL)


def test_energy_head_bwd():
    from newtonnet_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(3)
    N = 77
    h2, w3, scale = _rand(g, N, 128), _rand(g, 128), torch.rand(119, generator=g).to(DEV) + 0.5
    z = torch.randint(1, 9, (N,), generator=g).to(DEV)
    out = torch.empty_like(h2)
    L.check(lib.nn_energy_head_bwd(h2.data_ptr(), w3.data_ptr(), scale.data_ptr(), z.data_ptr(), N, out.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream), 'nn_energy_head_bwd')
    hd = h2.double().requires_grad_(True)
    e = ((torch.nn.functional.silu(hd) * w3.double()).sum(1) * scale.double()[z]).sum()
    want, = torch.autograd.grad(e, hd)
    torch.testing.assert_close(out.double(), want, rtol=2e-5, atol=2e-6)


def test_pair_gather_bwd():
    from newtonnet_b200 import _lib as L
    lib = L.load()
    nl, N, P = _nl()
    g = torch.Generator().manual_seed(5)
    cap = nl.cap_pairs
    dfb, f_in, unit, e1, ubar0 = _rand(g, N, 3, 128), _rand(g, N, 3, 128), _rand(g, cap, 3), _rand(g, cap, 128), _rand(g, cap, 3)
    i, j = nl.pair_i[:P].long(), nl.pair_j[:P].long()
    s = torch.cuda.current_stream().cuda_stream
    for first in (False, True):
        e1_io, e2bar, ubar = e1.clone(), torch.zeros(cap, 128, device=DEV), ubar0.clone()
        L.check(lib.nn_pair_gather_bwd(C.byref(nl.struct), dfb.data_ptr(), None if first else f_in.data_ptr(), unit.data_ptr(),
                                       e1_io.data_ptr(), None if first else e2bar.data_ptr(), ubar.data_ptr(), s), 'nn_pair_gather_bwd')
        D, F, U, E1 = dfb.double(), f_in.double(), unit.double()[:P], e1.double()[:P]
        w = D[i] - D[j]                                                   # [P,3,128]
        torch.testing.assert_close(e1_io.double()[:P], (w * U[:, :, None]).sum(1), **TOL)
        torch.testing.assert_close(ubar.double()[:P], ubar0.double()[:P] + (w * E1[:, None, :]).sum(2), rtol=2e-5, atol=2e-4)
        if not first:
            torch.testing.assert_close(e2bar.double()[:P], (D[i] * F[j] + D[j] * F[i]).sum(1), **TOL)


@pytest.mark.parametrize('backend', [0, 2])
def test_edge_message_bwd(backend):
    from newtonnet_b200 import _lib as L
    lib = L.load(); lib.nn_set_gemm_backend(backend)
    nl, N, P = _nl()
    g = torch.Generator().manual_seed(7)
    cap = nl.cap_pairs
    abar, mn, rbf, drbf, We, mbar = _rand(g, N, 128), _rand(g, N, 128), _rand(g, cap, 20), _rand(g, cap, 20), _rand(g, 128, 20) / 4, \
        _rand(g, cap, 128)
    Wet = We.t().contiguous()
    img = torch.empty(2 * 128 * 32, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    L.check(lib.nn_message_prepare_b(We.data_ptr(), img.data_ptr(), s), 'prepare')
    io, x_part = mbar.clone(), torch.zeros(2, cap, device=DEV)
    L.check(lib.nn_edge_message_bwd(C.byref(nl.struct), abar.data_ptr(), mn.data_ptr(), rbf.data_ptr(), drbf.data_ptr(), Wet.data_ptr(),
                                    img.data_ptr() if backend else None, io.data_ptr(), x_part.data_ptr(), s), 'nn_edge_message_bwd')
    lib.nn_set_gemm_backend(2)
    i, j = nl.pair_i[:P].long(), nl.pair_j[:P].long()
    A, MN, W = abar.double(), mn.double(), We.double()
    mt = mbar.double()[:P] + A[i] + A[j]
    y = mt * MN[i] * MN[j]
    torch.testing.assert_close(x_part.double().sum(0)[:P], (y * (drbf.double()[:P] @ W.t())).sum(1), rtol=2e-5, atol=2e-3)
    torch.testing.assert_close(io.double()[:P], mt * (rbf.double()[:P] @ W.t()), rtol=2e-5, atol=2e-4)


def test_node_aggregate_bwd():
    from newtonnet_b200 import _lib as L
    lib = L.load()
    nl, N, P = _nl()
    g = torch.Generator().manual_seed(9)
    cap = nl.cap_pairs
    t_, mn, e2, dfb = _rand(g, cap, 128), _rand(g, N, 128), _rand(g, cap, 128), _rand(g, N, 3, 128)
    ei = nl.edge_index()                                                    # [2,E]: destination k, source i
    E = ei.shape[1]
    pair = (nl.edge_pair[:E].long() & 0x7fffffff)
    k, i = ei[0], ei[1]
    s = torch.cuda.current_stream().cuda_stream
    for first in (False, True):
        mnbar, fbar = torch.empty(N, 128, device=DEV), torch.empty(N, 3, 128, device=DEV)
        L.check(lib.nn_node_aggregate_bwd(C.byref(nl.struct), t_.data_ptr(), mn.data_ptr(), None if first else e2.data_ptr(),
                                          None if first else dfb.data_ptr(), mnbar.data_ptr(), None if first else fbar.data_ptr(), s),
                'nn_node_aggregate_bwd')
        want_mn = torch.zeros(N, 128, dtype=torch.float64, device=DEV).index_add_(0, k, t_.double()[pair] * mn.double()[i])
        torch.testing.assert_close(mnbar.double(), want_mn, **TOL)
        if not first:
            want_f = dfb.double().clone().index_add_(0, k, dfb.double()[i] * e2.double()[pair][:, None, :])
            torch.testing.assert_close(fbar.double(), want_f, **TOL)


@pytest.mark.parametrize('m', [1, 31, 32, 100, 4097, 30230, 200001])
def test_gemm128_tn_tensor_core(m):
    """X^T Y (weight gradients) on the tensor cores, 3xTF32, against fp64; row counts around the 32-row K block and the
    per-CTA row split; deterministic (fixed partition, fixed-order reduction)."""
    import ctypes as C
    from newtonnet_b200 import _lib as L
    lib = L.load()
    dev = torch.device('cuda:0')
    g = torch.Generator().manual_seed(m)
    X = torch.randn(m, 128, generator=g).to(dev)
    Y = torch.randn(m, 128, generator=g).to(dev)
    s = torch.cuda.current_stream().cuda_stream

    def run():
        out = torch.empty(128, 128, device=dev)
        ws = torch.empty(lib.nn_gemm128_tn_workspace_bytes(m), dtype=torch.uint8, device=dev)
        L.check(lib.nn_gemm128_tn(X.data_ptr(), Y.data_ptr(), m, out.data_ptr(), ws.data_ptr(), s), 'nn_gemm128_tn')
        return out
    a, b = run(), run()
    assert torch.equal(a, b)
    ref = X.double().t() @ Y.double()
    scale = float(ref.abs().max())
    # fp32 accumulation over m rows (TMEM accumulator per CTA, then a fixed-order sum of the partials)
    assert float((a.double() - ref).abs().max()) / scale < 3e-6 * max(1.0, (m / 1024) ** 0.5)


def test_gemm128_tn_accumulate():
    """nn_gemm128_tn_acc: out (+)= X^T Y - the form the training step's weight-gradient sink uses (newtonnet_b200/train.py)."""
    from newtonnet_b200 import _lib as L
    lib = L.load()
    dev = torch.device('cuda:0')
    g = torch.Generator().manual_seed(11)
    s = torch.cuda.current_stream().cuda_stream
    ws = torch.empty(lib.nn_gemm128_tn_workspace_bytes(1 << 20), dtype=torch.uint8, device=dev)
    out = torch.full((128, 128), 7.0, device=dev)
    want = torch.zeros(128, 128, dtype=torch.float64, device=dev)
    for k, m in enumerate((5000, 37, 30230)):
        X, Y = torch.randn(m, 128, generator=g).to(dev), torch.randn(m, 128, generator=g).to(dev)
        L.check(lib.nn_gemm128_tn_acc(X.data_ptr(), Y.data_ptr(), m, out.data_ptr(), ws.data_ptr(), int(k > 0), s), 'nn_gemm128_tn_acc')
        want += X.double().t() @ Y.double()
    assert float((out.double() - want).abs().max()) / float(want.abs().max()) < 2e-5
    before = out.clone()
    L.check(lib.nn_gemm128_tn_acc(out.data_ptr(), out.data_ptr(), 0, out.data_ptr(), ws.data_ptr(), 1, s), 'nn_gemm128_tn_acc')
    assert torch.equal(out, before)                      # no rows, accumulate: unchanged

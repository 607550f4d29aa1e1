"""Chained two-CTA contraction (csrc/gemm_chain.cu) against two single launches (bit-identical) and fp64."""
import ctypes as C

import pytest
import torch

from test_gpu_parity import _gemm, dev

pytestmark = pytest.mark.gpu


def _tile(t):
    """[M,128] rows -> the tile-transposed layout of include/newtonnet_b200.h (NN_TILED_INDEX), padded to whole tiles."""
    M = t.shape[0]
    Mp = (M + 127) // 128 * 128
    p = torch.zeros(Mp, 128, dtype=t.dtype, device=t.device)
    p[:M] = t
    return p.view(Mp // 128, 128, 32, 4).permute(0, 2, 1, 3).contiguous().view(Mp, 128)


def _untile(t, M):
    Mp = t.shape[0]
    return t.view(Mp // 128, 32, 128, 4).permute(0, 2, 1, 3).reshape(Mp, 128)[:M]


def _chain(lib, X, B1, B2, mid, out, bias1=None, bias2=None, aux1=None, aux2=None, aux_out=None, Y=None, m_dev=None):
    """One chained launch; aux_out / aux1 are tile-transposed (_tile)."""
    from newtonnet_b200 import _lib as L
    s = torch.cuda.current_stream().cuda_stream
    imgs = []
    for B in (B1, B2):
        img = torch.empty(L.NN_B_IMAGE_FLOATS, device=X.device)
        L.check(lib.nn_gemm128_prepare_b(B.data_ptr(), img.data_ptr(), s), 'prepare_b')
        imgs.append(img)
    Y = torch.empty_like(X) if Y is None else Y
    a = L.GemmChainArgs()
    a.X, a.B1_img, a.B2_img, a.Y = X.data_ptr(), imgs[0].data_ptr(), imgs[1].data_ptr(), Y.data_ptr()
    a.bias1, a.bias2, a.aux1, a.aux2, a.aux_out = L.ptr(bias1), L.ptr(bias2), L.ptr(aux1), L.ptr(aux2), L.ptr(aux_out)
    a.m_dev, a.m_dev_mul, a.m, a.mid, a.out = L.ptr(m_dev), 1, X.shape[0], mid, out
    L.check(lib.nn_gemm128_chain(C.byref(a), s), 'nn_gemm128_chain')
    torch.cuda.synchronize()
    return Y


def _tiled_like(X, fill):
    """A tile-transposed buffer for the rows of X: whole tiles of 128 rows."""
    return torch.full(((X.shape[0] + 127) // 128 * 128, 128), fill, device=X.device)


@pytest.mark.parametrize('M', [1, 127, 128, 129, 300, 4099, 74 * 128 * 3 + 77, 148 * 128 * 5 + 1])
def test_tiled_chain_matches_two_launches(M):
    """The chain with silu' tile-transposed (aux_out forward, aux1 reverse) against two launches: bit-identical."""
    from newtonnet_b200 import _lib as L
    lib = L.load()
    lib.nn_set_gemm_backend(2)
    g = torch.Generator(device='cpu').manual_seed(M)
    r = lambda *s: torch.randn(*s, generator=g).to(dev())
    X, B1, B2, b1, b2, aux, acc0 = r(M, 128), r(128, 128) / 11.3, r(128, 128) / 11.3, r(128), r(128), r(M, 128), r(M, 128)
    silu = lambda t: t * torch.sigmoid(t)
    dsilu = lambda t: torch.sigmoid(t) * (1 + t * (1 - torch.sigmoid(t)))
    Mp = (M + 127) // 128 * 128
    # forward MLP: two launches (pre-activation, then SILU_SAVE in place) vs one chained launch writing silu' tile-transposed
    pre = _gemm(lib, X, B1, bias=b1)
    want_mid = pre.clone()
    want = _gemm(lib, want_mid, B2, pro=L.PRO_SILU_SAVE, bias=b2, aux_out=want_mid)
    mid_t = _tiled_like(X, 9.0)
    got = _chain(lib, X, B1, B2, 0, 0, bias1=b1, bias2=b2, aux_out=mid_t)
    mid = _untile(mid_t, M)
    assert torch.equal(got, want) and torch.equal(mid, want_mid)
    ref = silu(X.double() @ B1.double() + b1.double()) @ B2.double() + b2.double()
    torch.testing.assert_close(got.double(), ref, rtol=3e-5, atol=3e-5)
    torch.testing.assert_close(mid.double(), dsilu(X.double() @ B1.double() + b1.double()), rtol=2e-5, atol=2e-6)
    # no biases
    assert torch.equal(_chain(lib, X, B1, B2, 0, 0, aux_out=mid_t),
                       _gemm(lib, _gemm(lib, X, B1), B2, pro=L.PRO_SILU))
    # reverse MLP: (X @ B1) * aux @ B2 [+ acc], aux tile-transposed in the chain
    aux_t = _tile(aux)
    t = _gemm(lib, X, B1, epi=L.EPI_MUL, aux1=aux)
    assert torch.equal(_gemm(lib, X, B1, epi=L.EPI_MUL, aux1=aux_t, aux_tiled=1), t)      # two launches, tiled factor
    assert torch.equal(_chain(lib, X, B1, B2, 1, 0, aux1=aux_t), _gemm(lib, t, B2))
    want_acc = acc0.clone(); _gemm(lib, t, B2, epi=L.EPI_ADD, aux1=want_acc, Y=want_acc)
    got_acc = acc0.clone(); _chain(lib, X, B1, B2, 1, 1, aux1=aux_t, aux2=got_acc, Y=got_acc)
    assert torch.equal(got_acc, want_acc)
    # device-side row count below the launch capacity: rows beyond it are untouched
    if M > 130:
        cnt = torch.tensor([M - 100], dtype=torch.int32, device=dev())
        Y = torch.full_like(X, 7.0); mid_t = _tiled_like(X, 5.0)
        _chain(lib, X, B1, B2, 0, 0, bias1=b1, bias2=b2, aux_out=mid_t, Y=Y, m_dev=cnt)
        assert torch.equal(Y[:M - 100], want[:M - 100]) and bool((Y[M - 100:] == 7.0).all())
        assert torch.equal(_untile(mid_t, M)[:M - 100], want_mid[:M - 100]) and bool((_untile(mid_t, Mp)[M - 100:] == 5.0).all())


def test_chain_argument_errors():
    from newtonnet_b200 import _lib as L
    lib = L.load()
    a = L.GemmChainArgs()
    assert lib.nn_gemm128_chain(C.byref(a), None) != 0
    assert b'null' in lib.nn_last_error()


@pytest.mark.parametrize('M', [1, 128, 129, 4099, 74 * 128 * 3 + 77, 148 * 128 * 5 + 1])
def test_tiled_dual_chain_matches_two_single_chains(M):
    """Two forward MLPs over the same input in ONE launch (odd / even clusters, X fetched from HBM once): Y and the
    tile-transposed silu' bit-identical to two chained launches; device-side row count honoured."""
    from newtonnet_b200 import _lib as L
    lib = L.load()
    lib.nn_set_gemm_backend(2)
    g = torch.Generator(device='cpu').manual_seed(1000 + M)
    r = lambda *s: torch.randn(*s, generator=g).to(dev())
    X = r(M, 128)
    A1, A2, B1, B2 = (r(128, 128) / 11.3 for _ in range(4))
    s = torch.cuda.current_stream().cuda_stream
    imgs = []
    for B in (A1, A2, B1, B2):
        img = torch.empty(L.NN_B_IMAGE_FLOATS, device=X.device)
        L.check(lib.nn_gemm128_prepare_b(B.data_ptr(), img.data_ptr(), s), 'prepare_b')
        imgs.append(img)
    Mp = (M + 127) // 128 * 128
    midA, midB = _tiled_like(X, 0.0), _tiled_like(X, 0.0)
    wantA = _chain(lib, X, A1, A2, 0, 0, aux_out=midA)
    wantB = _chain(lib, X, B1, B2, 0, 0, aux_out=midB)
    midA, midB = _untile(midA, M), _untile(midB, M)
    cnt = torch.tensor([max(M - 50, 1)], dtype=torch.int32, device=dev())
    for m_dev in (None, cnt):
        n = M if m_dev is None else int(cnt.item())
        YA, YB = torch.full_like(X, 3.0), torch.full_like(X, 3.0)
        mA_t, mB_t = _tiled_like(X, 3.0), _tiled_like(X, 3.0)
        a = L.GemmChainArgs()
        a.X, a.B1_img, a.B2_img, a.Y, a.aux_out = X.data_ptr(), imgs[0].data_ptr(), imgs[1].data_ptr(), YA.data_ptr(), mA_t.data_ptr()
        a.B1_img_b, a.B2_img_b, a.Y_b, a.aux_out_b = imgs[2].data_ptr(), imgs[3].data_ptr(), YB.data_ptr(), mB_t.data_ptr()
        a.m_dev, a.m_dev_mul, a.m, a.mid, a.out = L.ptr(m_dev), 1, M, 0, 0
        L.check(lib.nn_gemm128_chain(C.byref(a), s), 'nn_gemm128_chain(dual)')
        torch.cuda.synchronize()
        mA, mB = _untile(mA_t, Mp), _untile(mB_t, Mp)
        assert torch.equal(YA[:n], wantA[:n]) and torch.equal(YB[:n], wantB[:n])
        assert torch.equal(mA[:n], midA[:n]) and torch.equal(mB[:n], midB[:n])
        assert bool((YA[n:] == 3.0).all()) and bool((mB[n:] == 3.0).all())

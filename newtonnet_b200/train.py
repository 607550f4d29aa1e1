"""Differentiable (create_graph) evaluation and the data-parallel training step - SURVEY.md section 8a row T.

The inference path (csrc/eval.cu) uses a hand-derived reverse sweep and is not differentiable with respect
to the parameters.  Training needs d(loss)/d(parameters) THROUGH the forces (reference
models/newtonnet.py:106-113 sets create_graph=True; train/trainer.py:303-313 calls loss.backward()).  Here
the forward is composed from a closed set of primitives whose derivatives are again those primitives, so
autograd builds the double backward:

    X @ B         nn_gemm128 (tcgen05 3xTF32)     dX = dY @ B^T  (same op)      dB = X^T dY  (nn_gemm128_tn)
    X^T Y         nn_gemm128_tn                   dX = Y @ G^T                  dY = X @ G   (nn_gemm128)
    rows[idx]     nn_halo_pack (gather)           d rows = segment sum
    segment sum   nn_segment_sum (deterministic)  d src = rows[idx]

i.e. every 128-wide contraction (98 % of the FLOPs) and every gather / scatter of feature rows runs in the
CUDA library; element-wise glue (SiLU, products, the radial basis) is left to autograd's own element-wise
kernels in this round.  Edges come from the same cell-list kernel as inference (directed edges in the
reference's order).  NewtonNet.forward routes here when a derivative head has create_graph=True.
"""
import ctypes as C
import os

import torch
import torch.distributed as dist
import torch.nn.functional as Fn

from . import _lib as L
from .engine import NeighborList, all_pairs_bound, capture, count_edges, edge_capacity, get_engine, stream, warm_up


# ----------------------------------------------------------------------------- raw kernel calls
# Operand images of the model's weights, valid for ONE training step: every nn.Linear weight is multiplied in both
# orientations several times per step (forward, backward, double backward).  Only views of leaf parameters are cached
# (temporaries can reuse an address), keyed by storage address, version and strides; differentiable_forward clears the
# cache when a step begins, so a CUDA-graph capture always records the prepare kernels of its own step.
_image_cache = {}


def _image_key(B):
    base = B._base if B._base is not None else B
    if base.is_leaf and isinstance(base, torch.nn.Parameter):
        return (B.data_ptr(), base._version, tuple(B.shape), tuple(B.stride()))
    return None


def prepare_weight_images(model):
    """Both operand images (W and W^T) of every 128x128 weight of the model in ONE launch, registered in the step's
    cache under the keys the GEMM calls of forward / backward / double backward will ask for.  Replaces ~58 single
    prepare launches and as many transposed-copy kernels per training step."""
    lib = L.load()
    mats = [p for p in model.parameters() if p.dim() == 2 and tuple(p.shape) == (128, 128) and p.is_cuda
            and p.dtype == torch.float32 and p.is_contiguous()]
    if not mats:
        return
    n = 2 * len(mats)
    imgs = torch.empty(n, L.NN_B_IMAGE_FLOATS, dtype=torch.float32, device=mats[0].device)
    src = (C.c_void_p * n)(); img = (C.c_void_p * n)(); tr = (C.c_int32 * n)()
    for i, p in enumerate(mats):
        for t in (0, 1):                       # t = 0: operand B = W ([K,N] = W as stored); t = 1: operand B = W^T (view p.t())
            k = 2 * i + t
            src[k], img[k], tr[k] = p.data_ptr(), imgs[k].data_ptr(), t
            _image_cache[_image_key(p.t() if t else p)] = imgs[k]
    L.check(lib.nn_gemm128_prepare_b_batch(src, tr, img, n, stream()), 'nn_gemm128_prepare_b_batch')


def _operand_image(B):
    """Operand image of B [128,128] (any strides): from the step's cache, else prepared now from a contiguous copy."""
    key = _image_key(B)
    if key is not None:
        img = _image_cache.get(key)
        if img is not None:
            return img
    Bc = _c(B)
    img = torch.empty(L.NN_B_IMAGE_FLOATS, dtype=torch.float32, device=Bc.device)
    L.check(L.load().nn_gemm128_prepare_b(Bc.data_ptr(), img.data_ptr(), stream()), 'nn_gemm128_prepare_b')
    if key is not None:
        _image_cache[key] = img
    return img


def _gemm_raw(X, B):
    lib = L.load()
    M = X.shape[0]
    Y = torch.empty(M, 128, dtype=torch.float32, device=X.device)
    if M == 0:
        return Y
    img = _operand_image(B)
    a = L.GemmArgs()
    # the row-major matrix itself is read by the SIMT back-end only; the tensor-core back-ends take the image
    Bm = _c(B) if lib.nn_get_gemm_backend() == 0 else B
    a.X, a.B, a.B_img, a.Y, a.m = X.data_ptr(), Bm.data_ptr(), img.data_ptr(), Y.data_ptr(), M
    L.check(lib.nn_gemm128(C.byref(a), stream()), 'nn_gemm128')
    return Y


def _gemm_tn_raw(X, Y):
    lib = L.load()
    M = X.shape[0]
    out = torch.empty(128, 128, dtype=torch.float32, device=X.device)
    ws = torch.empty(max(lib.nn_gemm128_tn_workspace_bytes(M), 4), dtype=torch.uint8, device=X.device)
    L.check(lib.nn_gemm128_tn(X.data_ptr(), Y.data_ptr(), M, out.data_ptr(), ws.data_ptr(), stream()), 'nn_gemm128_tn')
    return out


def _c(t):
    return t.contiguous()


# ----------------------------------------------------------------------------- where weight gradients go
# A custom Function's backward computes every input gradient its ctx.needs_input_grad names, whether or not the running
# autograd call asked for it.  Two consequences for the training step, handled by a module-level mode (the engine runs
# backward nodes on its own device thread, so this is a plain global, not a thread-local):
#   'skip'     while the forces are being derived (autograd.grad(energy, pos, create_graph=True) inside
#              differentiable_forward): only d/d pos is wanted there, yet every linear would also form its X^T dY and throw
#              it away (~25 contractions + reductions per config-5 step);
#   'sink'     during the loss.backward() of a training step: X^T dY of a 128x128 nn.Linear weight is a LEAF of the backward
#              graph - nothing but the optimizer reads it - so it is launched on a side stream and accumulated straight
#              into weight.grad (nn_gemm128_tn_acc), off the critical path of the ~900-kernel chain and without autograd's
#              AccumulateGrad add / copy kernels;
#   'autograd' (default) returns the gradient to autograd like any Function.
_weight_grad_mode = 'autograd'
_weight_grad_sink = None


class WeightGradSink:
    """Side stream + workspace that receive the weight gradients of a training step's loss.backward().

        with sink.step():            # mode 'sink'; joins the side stream on exit
            loss.backward()

    Gradients are written into p.grad (allocated on first use, overwritten by the first contribution of a step, summed
    in launch order after it - deterministic).  Works eagerly and under CUDA-graph capture (the fork / join become graph
    edges); operands are marked with record_stream so the caching allocator does not hand their memory to a later
    main-stream kernel while the side stream still reads them."""

    def __init__(self, device):
        self.device = device
        self.stream = torch.cuda.Stream(device=device)
        self.workspace = torch.empty(L.load().nn_gemm128_tn_workspace_bytes(1 << 30), dtype=torch.uint8, device=device)
        self._touched = set()
        self.launched = 0

    def accumulate(self, W, A, Bm):
        """W.grad (+)= A^T @ Bm."""
        A, Bm = _c(A), _c(Bm)                      # on the main stream, before the fork
        first = id(W) not in self._touched
        if first:
            self._touched.add(id(W))
            if W.grad is None:
                W.grad = torch.empty_like(W, memory_format=torch.contiguous_format)
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        L.check(L.load().nn_gemm128_tn_acc(A.data_ptr(), Bm.data_ptr(), A.shape[0], W.grad.data_ptr(), self.workspace.data_ptr(),
                                           0 if first else 1, self.stream.cuda_stream), 'nn_gemm128_tn_acc')
        A.record_stream(self.stream); Bm.record_stream(self.stream)
        self.launched += 1

    def step(self):
        return _SinkStep(self)


class _SinkStep:
    def __init__(self, sink):
        self.sink = sink

    def __enter__(self):
        global _weight_grad_mode, _weight_grad_sink
        self.prev = (_weight_grad_mode, _weight_grad_sink)
        self.sink._touched.clear()
        _weight_grad_mode, _weight_grad_sink = 'sink', self.sink
        return self.sink

    def __exit__(self, *exc):
        global _weight_grad_mode, _weight_grad_sink
        _weight_grad_mode, _weight_grad_sink = self.prev
        torch.cuda.current_stream(self.sink.device).wait_stream(self.sink.stream)      # join
        return False


class _skip_weight_grads:
    def __enter__(self):
        global _weight_grad_mode
        self.prev = _weight_grad_mode
        _weight_grad_mode = 'skip'

    def __exit__(self, *exc):
        global _weight_grad_mode
        _weight_grad_mode = self.prev
        return False


def _weight_grad(W, A, Bm):
    """d/dW of a contraction with W: A^T @ Bm, routed by the mode above."""
    if _weight_grad_mode == 'skip':
        return None
    if (_weight_grad_mode == 'sink' and not torch.is_grad_enabled() and isinstance(W, torch.nn.Parameter) and W.is_leaf
            and W.is_contiguous() and A.shape[0] > 0):
        _weight_grad_sink.accumulate(W, A, Bm)
        return None
    return GemmTN.apply(A, Bm)


class Gemm(torch.autograd.Function):
    """Y[M,128] = X[M,128] @ B[128,128]."""

    @staticmethod
    def forward(ctx, X, B):
        # save the inputs themselves: a contiguous copy made here would be cut off from the graph, and
        # the double backward needs d(dX)/dB through them
        ctx.save_for_backward(X, B)
        return _gemm_raw(_c(X), B)

    @staticmethod
    def backward(ctx, dY):
        X, B = ctx.saved_tensors
        dX = Gemm.apply(dY, B.t()) if ctx.needs_input_grad[0] else None
        dB = GemmTN.apply(X, dY) if ctx.needs_input_grad[1] and _weight_grad_mode != 'skip' else None
        return dX, dB


class Linear(torch.autograd.Function):
    """Y[M,128] = X[M,128] @ W[128,128]^T with W as stored by nn.Linear (reference models/newtonnet.py:181-199)."""

    @staticmethod
    def forward(ctx, X, W):
        ctx.save_for_backward(X, W)
        ctx.weight = W
        return _gemm_raw(_c(X), W.t())

    @staticmethod
    def backward(ctx, dY):
        X, W = ctx.saved_tensors
        dX = LinearT.apply(dY, ctx.weight) if ctx.needs_input_grad[0] else None
        dW = _weight_grad(ctx.weight, dY, X) if ctx.needs_input_grad[1] else None          # dY^T X
        return dX, dW


class LinearT(torch.autograd.Function):
    """Y[M,128] = X[M,128] @ W[128,128]: the input gradient of Linear, a Function of its own so that the weight it was
    called with stays identifiable in the double backward."""

    @staticmethod
    def forward(ctx, X, W):
        ctx.save_for_backward(X, W)
        ctx.weight = W
        return _gemm_raw(_c(X), W)

    @staticmethod
    def backward(ctx, dY):
        X, W = ctx.saved_tensors
        dX = Linear.apply(dY, ctx.weight) if ctx.needs_input_grad[0] else None
        dW = _weight_grad(ctx.weight, X, dY) if ctx.needs_input_grad[1] else None          # X^T dY
        return dX, dW


class GemmTN(torch.autograd.Function):
    """G[128,128] = X[M,128]^T @ Y[M,128]."""

    @staticmethod
    def forward(ctx, X, Y):
        ctx.save_for_backward(X, Y)
        return _gemm_tn_raw(_c(X), _c(Y))

    @staticmethod
    def backward(ctx, G):
        X, Y = ctx.saved_tensors
        dX = Linear.apply(Y, G) if ctx.needs_input_grad[0] else None          # Y @ G^T
        dY = LinearT.apply(X, G) if ctx.needs_input_grad[1] else None         # X @ G
        return dX, dY


class Segments:
    """Index structure of one gather / segment-sum pair: idx[k] = target row of source row k."""

    def __init__(self, idx, n_rows, grouped=None, valid=None):
        """grouped: True = idx is non-decreasing, False = it is not, None = look (one host synchronisation; not
        allowed while a CUDA graph is being captured).  valid: mask of the real rows of a padded list; padding must
        come last - it is gathered (harmless) but belongs to no segment, so sums neither see it nor pay for it."""
        self.idx = idx.to(torch.int32).contiguous()
        self.n_rows = int(n_rows)
        ones = torch.ones(idx.shape[0], dtype=torch.int64, device=idx.device) if valid is None else valid.to(torch.int64)
        counts = torch.zeros(n_rows, dtype=torch.int64, device=idx.device).index_add_(0, idx.long(), ones)   # no host sync
        self.row_ptr = torch.zeros(n_rows + 1, dtype=torch.int32, device=idx.device)
        self.row_ptr[1:] = torch.cumsum(counts, 0)
        if grouped is None:
            grouped = bool((idx[1:] >= idx[:-1]).all()) if idx.numel() > 1 else True
        if grouped:
            self.perm = None                      # already grouped (destination-sorted edges)
        else:
            self.perm = torch.sort(idx, stable=True).indices.to(torch.int32).contiguous()

    @classmethod
    def from_csr(cls, idx, n_rows, row_ptr, perm=None):
        """Segments whose grouping is already known (the neighbour list's CSR): no counting pass, no sort."""
        self = cls.__new__(cls)
        self.idx = idx.to(torch.int32).contiguous()
        self.n_rows = int(n_rows)
        self.row_ptr = row_ptr
        self.perm = perm
        return self


class Gather(torch.autograd.Function):
    """out[k,:] = rows[idx[k],:]  (width % 4 == 0)."""

    @staticmethod
    def forward(ctx, rows, seg):
        rows = _c(rows)
        ctx.seg = seg
        n, width = seg.idx.shape[0], rows.shape[1]
        out = torch.empty(n, width, dtype=torch.float32, device=rows.device)
        if n:
            L.check(L.load().nn_halo_pack(rows.data_ptr(), seg.idx.data_ptr(), n, width, out.data_ptr(), stream()),
                    'nn_halo_pack')
        return out

    @staticmethod
    def backward(ctx, d_out):
        return SegmentSum.apply(d_out, ctx.seg), None


class SegmentSum(torch.autograd.Function):
    """out[i,:] = sum_{k: idx[k] = i} src[k,:], fixed summation order."""

    @staticmethod
    def forward(ctx, src, seg):
        src = _c(src)
        ctx.seg = seg
        width = src.shape[1]
        # the kernel writes every output row (empty segments get zeros): no fill kernel in front of it
        out = (torch.empty if src.shape[0] else torch.zeros)(seg.n_rows, width, dtype=torch.float32, device=src.device)
        if src.shape[0]:
            L.check(L.load().nn_segment_sum(src.data_ptr(), L.ptr(seg.perm), seg.row_ptr.data_ptr(), seg.n_rows, width,
                                            out.data_ptr(), stream()), 'nn_segment_sum')
        return out

    @staticmethod
    def backward(ctx, d_out):
        return Gather.apply(d_out, ctx.seg), None


# ----------------------------------------------------------------------------- fused row products (csrc/train_ops.cu)
# Six kernels that are closed under differentiation: every backward below is again one of these Functions, so the graph
# of the double backward consists of them (and of Gemm / GemmTN / Gather / SegmentSum) instead of broadcasting ATen ops.
def _rows(mode, p, q3, u, out_shape):
    ref = p if p is not None else q3
    out = torch.empty(out_shape, dtype=torch.float32, device=ref.device)
    n = out_shape[0]
    if n:
        L.check(L.load().nn_ew_rows(mode, L.ptr(p), L.ptr(q3), L.ptr(u), out.data_ptr(), n, stream()), 'nn_ew_rows')
    return out


class Mul3(torch.autograd.Function):
    """a * b * c (same shapes)."""

    @staticmethod
    def forward(ctx, a, b, c):
        ctx.save_for_backward(a, b, c)
        a, b, c = _c(a), _c(b), _c(c)
        out = torch.empty_like(a)
        if a.numel():
            L.check(L.load().nn_ew_mul3(a.data_ptr(), b.data_ptr(), c.data_ptr(), out.data_ptr(), a.numel(), stream()), 'nn_ew_mul3')
        return out

    @staticmethod
    def backward(ctx, g):
        a, b, c = ctx.saved_tensors
        ni = ctx.needs_input_grad
        return (Mul3.apply(g, b, c) if ni[0] else None, Mul3.apply(g, a, c) if ni[1] else None,
                Mul3.apply(g, a, b) if ni[2] else None)


class Outer(torch.autograd.Function):
    """out[e,c,:] = x[e,:] * u[e,c];  x [n,F], u [n,3] -> [n,3,F]."""

    @staticmethod
    def forward(ctx, x, u):
        ctx.save_for_backward(x, u)
        return _rows(0, _c(x), None, _c(u), (x.shape[0], 3, x.shape[1]))

    @staticmethod
    def backward(ctx, g):
        x, u = ctx.saved_tensors
        return (ContractC.apply(g, u) if ctx.needs_input_grad[0] else None, RowDot.apply(g, x) if ctx.needs_input_grad[1] else None)


class ContractC(torch.autograd.Function):
    """out[e,:] = sum_c x3[e,c,:] * u[e,c];  x3 [n,3,F], u [n,3] -> [n,F]."""

    @staticmethod
    def forward(ctx, x3, u):
        ctx.save_for_backward(x3, u)
        return _rows(1, None, _c(x3), _c(u), (x3.shape[0], x3.shape[2]))

    @staticmethod
    def backward(ctx, g):
        x3, u = ctx.saved_tensors
        return (Outer.apply(g, u) if ctx.needs_input_grad[0] else None, RowDot.apply(x3, g) if ctx.needs_input_grad[1] else None)


class RowDot(torch.autograd.Function):
    """out[e,c] = <x3[e,c,:], x[e,:]>;  x3 [n,3,F], x [n,F] -> [n,3]."""

    @staticmethod
    def forward(ctx, x3, x):
        ctx.save_for_backward(x3, x)
        return _rows(2, _c(x), _c(x3), None, (x3.shape[0], 3))

    @staticmethod
    def backward(ctx, g):
        x3, x = ctx.saved_tensors
        return (Outer.apply(x, g) if ctx.needs_input_grad[0] else None, ContractC.apply(x3, g) if ctx.needs_input_grad[1] else None)


class MulB(torch.autograd.Function):
    """out[e,c,:] = x[e,:] * y3[e,c,:];  x [n,F], y3 [n,3,F] -> [n,3,F]."""

    @staticmethod
    def forward(ctx, x, y3):
        ctx.save_for_backward(x, y3)
        return _rows(3, _c(x), _c(y3), None, tuple(y3.shape))

    @staticmethod
    def backward(ctx, g):
        x, y3 = ctx.saved_tensors
        return (SumMulC.apply(g, y3) if ctx.needs_input_grad[0] else None, MulB.apply(x, g) if ctx.needs_input_grad[1] else None)


class SumMulC(torch.autograd.Function):
    """out[e,:] = sum_c x3[e,c,:] * y3[e,c,:];  [n,3,F] x [n,3,F] -> [n,F]."""

    @staticmethod
    def forward(ctx, x3, y3):
        ctx.save_for_backward(x3, y3)
        return _rows(4, _c(y3), _c(x3), None, (x3.shape[0], x3.shape[2]))

    @staticmethod
    def backward(ctx, g):
        x3, y3 = ctx.saved_tensors
        return (MulB.apply(g, y3) if ctx.needs_input_grad[0] else None, MulB.apply(g, x3) if ctx.needs_input_grad[1] else None)


# Product with gathered operands (csrc/train_ops.cu k_ew_gmul): the node rows are read through the segments' indices inside
# the product, so neither forward nor the two backward sweeps materialise [E,F] copies of them.
def _gmul_raw(a, b, r1, seg1, r2, seg2):
    a = _c(a)
    out = torch.empty_like(a)
    n = a.shape[0]
    if n:
        b = None if b is None else _c(b)
        r1 = _c(r1)
        r2 = None if r2 is None else _c(r2)
        L.check(L.load().nn_ew_gmul(a.data_ptr(), L.ptr(b), r1.data_ptr(), seg1.idx.data_ptr(), L.ptr(r2),
                                    None if r2 is None else seg2.idx.data_ptr(), out.data_ptr(), n, stream()), 'nn_ew_gmul')
    return out


class GMul(torch.autograd.Function):
    """out[e,:] = a[e,:] * (b[e,:]) * r1[seg1.idx[e],:] * (r2[seg2.idx[e],:]);  b and r2 are optional, not both present.
    m_e = me_e * mn_i * mn_j (reference models/newtonnet.py:211) is GMul(me, None, mn, seg_dst, mn, seg_src)."""

    @staticmethod
    def forward(ctx, a, b, r1, seg1, r2, seg2):
        if b is not None and r2 is not None:
            raise NotImplementedError('GMul: at most three factors')
        ctx.save_for_backward(a, r1, *([b] if b is not None else []), *([r2] if r2 is not None else []))
        ctx.has_b, ctx.has_r2, ctx.seg1, ctx.seg2 = b is not None, r2 is not None, seg1, seg2
        return _gmul_raw(a, b, r1, seg1, r2, seg2)

    @staticmethod
    def backward(ctx, g):
        saved = list(ctx.saved_tensors)
        a, r1 = saved[0], saved[1]
        b = saved[2] if ctx.has_b else None
        r2 = saved[-1] if ctx.has_r2 else None
        seg1, seg2 = ctx.seg1, ctx.seg2
        ni = ctx.needs_input_grad
        da = GMul.apply(g, b, r1, seg1, r2, seg2) if ni[0] else None
        db = GMul.apply(g, a, r1, seg1, None, None) if (b is not None and ni[1]) else None
        dr1 = dr2 = None
        if ni[2]:               # everything but r1[i1], summed over the edges of each row
            if r2 is not None:
                rest = GMul.apply(g, a, r2, seg2, None, None)
            else:
                rest = Mul3.apply(g, a, b) if b is not None else g * a
            dr1 = SegmentSum.apply(rest, seg1)
        if r2 is not None and ni[4]:
            dr2 = SegmentSum.apply(GMul.apply(g, a, r1, seg1, None, None), seg2)
        return da, db, dr1, None, dr2, None


# Equivariant aggregation without [E,3,F] tensors (csrc/train_ops.cu k_seg_prod / k_ew_g3).  Five Functions, each gradient
# another member:   SegOuter(x,u;s)      d_x = ContractCG(go,u;s)          d_u = RowDotG(go,x;s)
#                   SegMulBG(x,r;so,si)  d_x = SumMulCGG(go,so,r,si)       d_r = SegMulBG(x,go;si,so)
#                   ContractCG(r,u;s)    d_r = SegOuter(go,u;s)            d_u = RowDotG(r,go;s)
#                   RowDotG(r,x;s)       d_r = SegOuter(x,go;s)            d_x = ContractCG(r,go;s)
#                   SumMulCGG(a,sa,b,sb) d_a = SegMulBG(go,b;sa,sb)        d_b = SegMulBG(go,a;sb,sa)
def _seg_prod_raw(x, u, rows3, seg_in, seg_out):
    x = _c(x)
    out = (torch.empty if x.shape[0] else torch.zeros)(seg_out.n_rows, 3, x.shape[1], dtype=torch.float32, device=x.device)
    if x.shape[0]:
        L.check(L.load().nn_seg_prod(x.data_ptr(), None if u is None else _c(u).data_ptr(), None if rows3 is None else _c(rows3).data_ptr(),
                                     None if seg_in is None else seg_in.idx.data_ptr(), L.ptr(seg_out.perm), seg_out.row_ptr.data_ptr(),
                                     seg_out.n_rows, out.data_ptr(), stream()), 'nn_seg_prod')
    return out


def _g3_raw(mode, rows3, seg, p, rowsb, segb, out_shape):
    out = torch.empty(out_shape, dtype=torch.float32, device=rows3.device)
    if out_shape[0]:
        L.check(L.load().nn_ew_g3(mode, _c(rows3).data_ptr(), seg.idx.data_ptr(), None if p is None else _c(p).data_ptr(),
                                  None if rowsb is None else _c(rowsb).data_ptr(), None if segb is None else segb.idx.data_ptr(),
                                  out.data_ptr(), out_shape[0], stream()), 'nn_ew_g3')
    return out


class SegOuter(torch.autograd.Function):
    """out[k,c,:] = sum_{e in seg(k)} x[e,:] * u[e,c];  x [E,F], u [E,3] -> [N,3,F]."""

    @staticmethod
    def forward(ctx, x, u, seg):
        ctx.save_for_backward(x, u)
        ctx.seg = seg
        return _seg_prod_raw(x, u, None, None, seg)

    @staticmethod
    def backward(ctx, go):
        x, u = ctx.saved_tensors
        ni = ctx.needs_input_grad
        return (ContractCG.apply(go, u, ctx.seg) if ni[0] else None, RowDotG.apply(go, x, ctx.seg) if ni[1] else None, None)


class SegMulBG(torch.autograd.Function):
    """out[k,c,:] = sum_{e in seg_out(k)} x[e,:] * rows3[seg_in.idx[e],c,:];  x [E,F], rows3 [N,3,F] -> [N,3,F]."""

    @staticmethod
    def forward(ctx, x, rows3, seg_out, seg_in):
        ctx.save_for_backward(x, rows3)
        ctx.seg_out, ctx.seg_in = seg_out, seg_in
        return _seg_prod_raw(x, None, rows3, seg_in, seg_out)

    @staticmethod
    def backward(ctx, go):
        x, rows3 = ctx.saved_tensors
        ni = ctx.needs_input_grad
        dx = SumMulCGG.apply(go, ctx.seg_out, rows3, ctx.seg_in) if ni[0] else None
        dr = SegMulBG.apply(x, go, ctx.seg_in, ctx.seg_out) if ni[1] else None
        return dx, dr, None, None


class ContractCG(torch.autograd.Function):
    """out[e,:] = sum_c u[e,c] * rows3[seg.idx[e],c,:]."""

    @staticmethod
    def forward(ctx, rows3, u, seg):
        ctx.save_for_backward(rows3, u)
        ctx.seg = seg
        return _g3_raw(0, rows3, seg, u, None, None, (u.shape[0], rows3.shape[2]))

    @staticmethod
    def backward(ctx, go):
        rows3, u = ctx.saved_tensors
        ni = ctx.needs_input_grad
        return (SegOuter.apply(go, u, ctx.seg) if ni[0] else None, RowDotG.apply(rows3, go, ctx.seg) if ni[1] else None, None)


class RowDotG(torch.autograd.Function):
    """out[e,c] = < rows3[seg.idx[e],c,:], x[e,:] >."""

    @staticmethod
    def forward(ctx, rows3, x, seg):
        ctx.save_for_backward(rows3, x)
        ctx.seg = seg
        return _g3_raw(1, rows3, seg, x, None, None, (x.shape[0], 3))

    @staticmethod
    def backward(ctx, go):
        rows3, x = ctx.saved_tensors
        ni = ctx.needs_input_grad
        return (SegOuter.apply(x, go, ctx.seg) if ni[0] else None, ContractCG.apply(rows3, go, ctx.seg) if ni[1] else None, None)


class SumMulCGG(torch.autograd.Function):
    """out[e,:] = sum_c a3[seg_a.idx[e],c,:] * b3[seg_b.idx[e],c,:]."""

    @staticmethod
    def forward(ctx, a3, seg_a, b3, seg_b):
        ctx.save_for_backward(a3, b3)
        ctx.seg_a, ctx.seg_b = seg_a, seg_b
        return _g3_raw(2, a3, seg_a, None, b3, seg_b, (seg_a.idx.shape[0], a3.shape[2]))

    @staticmethod
    def backward(ctx, go):
        a3, b3 = ctx.saved_tensors
        ni = ctx.needs_input_grad
        da = SegMulBG.apply(go, b3, ctx.seg_a, ctx.seg_b) if ni[0] else None
        db = SegMulBG.apply(go, a3, ctx.seg_b, ctx.seg_a) if ni[2] else None
        return da, None, db, None


def _rbf_raw(op, k, a, x, freq):
    if k > 2:
        raise NotImplementedError('third-order differentiation through the radial basis is not implemented by the fused training kernels')
    x = _c(x)
    n = x.shape[0]
    out = torch.empty((n, L.NN_NB) if op == 0 else (n, 1), dtype=torch.float32, device=x.device)
    if n:
        L.check(L.load().nn_ew_rbf(op, k, L.ptr(None if a is None else _c(a)), x.data_ptr(), freq.data_ptr(), out.data_ptr(), n, stream()),
                'nn_ew_rbf')
    return out


class RbfScale(torch.autograd.Function):
    """out[e,n] = s[e] * R^k_n(x[e]);  s, x [E,1] -> [E,20]  (R^k = k-th x-derivative of env(x) sin(f_n x) / x)."""

    @staticmethod
    def forward(ctx, s, x, freq, k):
        ctx.save_for_backward(s, x, freq)
        ctx.k = k
        return _rbf_raw(0, k, s, x, freq)

    @staticmethod
    def backward(ctx, g):
        s, x, freq = ctx.saved_tensors
        ds = RbfDot.apply(g, x, freq, ctx.k) if ctx.needs_input_grad[0] else None
        dx = s * RbfDot.apply(g, x, freq, ctx.k + 1) if ctx.needs_input_grad[1] else None
        return ds, dx, None, None


class RbfDot(torch.autograd.Function):
    """out[e] = sum_n g[e,n] R^k_n(x[e]);  g [E,20], x [E,1] -> [E,1]."""

    @staticmethod
    def forward(ctx, g, x, freq, k):
        ctx.save_for_backward(g, x, freq)
        ctx.k = k
        return _rbf_raw(1, k, g, x, freq)

    @staticmethod
    def backward(ctx, go):
        g, x, freq = ctx.saved_tensors
        dg = RbfScale.apply(go, x, freq, ctx.k) if ctx.needs_input_grad[0] else None
        dx = go * RbfDot.apply(g, x, freq, ctx.k + 1) if ctx.needs_input_grad[1] else None
        return dg, dx, None, None


def _silu_raw(mode, x, a=None, b=None):
    x = _c(x)
    out = torch.empty_like(x)
    if x.numel():
        L.check(L.load().nn_ew_silu(mode, x.data_ptr(), L.ptr(None if a is None else _c(a)), L.ptr(None if b is None else _c(b)),
                                    out.data_ptr(), x.numel(), stream()), 'nn_ew_silu')
    return out


class Silu(torch.autograd.Function):
    """silu(x); backward SiluB, whose backward is SiluB again and one silu'' kernel (never differentiated further)."""

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return _silu_raw(0, x)

    @staticmethod
    def backward(ctx, g):
        x, = ctx.saved_tensors
        return SiluB.apply(g, x)


class SiluB(torch.autograd.Function):
    """g * silu'(x)."""

    @staticmethod
    def forward(ctx, g, x):
        ctx.save_for_backward(g, x)
        return _silu_raw(1, x, g)

    @staticmethod
    def backward(ctx, go):
        g, x = ctx.saved_tensors
        if torch.is_grad_enabled() and ctx.needs_input_grad[1]:
            # this backward is itself being recorded (create_graph in the SECOND backward): third derivatives of the
            # activation would be needed - the reference's training step never asks for them (trainer.py:303-313)
            raise NotImplementedError('third-order differentiation through SiLU is not implemented by the fused training kernels')
        dg = SiluB.apply(go, x) if ctx.needs_input_grad[0] else None
        dx = _silu_raw(2, x, go, g) if ctx.needs_input_grad[1] else None       # go * g * silu''(x)
        return dg, dx


def silu(x):
    return Silu.apply(x)


def linear(x, weight, bias=None):
    """x @ weight^T (+ bias) through the tensor-core GEMM."""
    y = Linear.apply(x, weight)
    return y if bias is None else y + bias


# ----------------------------------------------------------------------------- forward (training mode)
def _edges(nl, pos, N, static):
    """Directed edges (reference order) and their minimum-image displacements as a function of pos.

    static = False: exactly E edges (one host synchronisation to read E).
    static = True : cap_edges rows, no host synchronisation (CUDA-graph capturable).  Rows beyond E are padding: a
    self edge of the last atom with the CONSTANT displacement (cutoff, 0, 0).  There x = 1, and the envelope
    (1-x)^3 p(x) vanishes together with its first and second derivative, so value, gradient and double backward of a
    padded row are exactly zero (the edge MLPs have no bias) and no gradient reaches pos through it."""
    if not static:
        nl.check()
        ei = nl.edge_index()
        dst, src = ei[0], ei[1]
        ep = nl.edge_pair[:nl.n_edges].long()
        valid = None
    else:
        E = nl.cap_edges
        ei = torch.zeros(2, E, dtype=torch.int64, device=pos.device)
        L.check(L.load().nn_nbr_edge_index(C.byref(nl.struct), ei.data_ptr(), E, stream()), 'nn_nbr_edge_index')
        # a list that outgrew its capacity was not (re)written: expose NO valid rows (the step then computes exact zeros from
        # padding instead of indexing with stale / uninitialised entries) - the caller reads the overflow flag afterwards
        n_valid = torch.where(nl.status[L.ST_EDGE_OVERFLOW] != 0, torch.zeros_like(nl.status[L.ST_N_EDGES]), nl.status[L.ST_N_EDGES])
        valid = torch.arange(E, device=pos.device) < n_valid
        dst = torch.where(valid, ei[0], N - 1)
        src = torch.where(valid, ei[1], N - 1)
        ep = torch.where(valid, nl.edge_pair[:E].long(), 0)
        ei = torch.stack([dst, src])
    sign = torch.where(ep < 0, -1.0, 1.0).to(torch.float32).unsqueeze(1)
    disp0 = nl.pair_disp[(ep & 0x7fffffff)] * sign
    return ei, dst, src, disp0, valid


def _displacements(pos, seg_dst, seg_src, disp0):
    """disp_e = pos_i - pos_j - (constant lattice shift), differentiable in pos.  The rows are fetched with Gather, whose
    backward is the deterministic segment sum over the neighbour list's CSR: ATen's pos[idx] backward is an index_put
    with a radix sort per call (4 x 35 us + 8 sort passes per config-5 step, tools/train_profile.py)."""
    pos4 = Fn.pad(pos, (0, 1))                              # rows of 4 floats: one 16-byte piece per row
    dd = (Gather.apply(pos4, seg_dst) - Gather.apply(pos4, seg_src))[:, :3]
    return dd - (dd.detach() - disp0)                       # minimum image with a constant lattice shift


def _table(emb, onehot):
    """emb(z) [N,1] of an nn.Embedding(119, 1, padding_idx=0) (layers/scalers.py: per-element scale / shift) as a matrix -
    vector product with the one-hot matrix of z: exact (entries 1.0 / 0.0), and its gradient is a gemv instead of ATen's
    embedding_dense_backward (2 x 82 us per config-5 step).  Row 0 is padding: read, never given a gradient."""
    w = emb.weight.reshape(-1).to(torch.float32)
    first = torch.arange(w.shape[0], device=w.device) == 0           # built by kernels: no H2D copy while capturing
    w = torch.where(first, w.detach(), w)
    return torch.mv(onehot[:, :w.shape[0]] if w.shape[0] <= onehot.shape[1] else onehot, w).unsqueeze(1)


def hessian_rows(pos_grad, pos):
    """d pos_grad / d pos [N,3,N,3] with one reverse pass per row of the 3N x 3N matrix (reference models/output.py:141-152
    batches the same rows with vmap).  pos_grad must carry a graph to pos (create_graph=True).  Every row's pass walks the
    whole batch: 3N passes over N atoms.  The rows themselves carry no graph: a third derivative through the fused SiLU and
    radial-basis kernels is not implemented (SiluB.backward, _rbf_raw)."""
    flat = pos_grad.reshape(-1)
    with _skip_weight_grads():
        rows = [torch.autograd.grad(flat[r], pos, retain_graph=True, create_graph=False)[0] for r in range(flat.numel())]
    N = pos.shape[0]
    return torch.stack(rows).reshape(N, 3, N, 3)


def differentiable_forward(model, z, pos, cell, batch, static_nl=None, properties=None):
    """NewtonNet.forward with create_graph semantics (reference models/newtonnet.py:74-104 in train mode).
    static_nl: a NeighborList of fixed capacity already rebuilt for `pos` on the current stream -> the whole forward
    has static shapes and no host synchronisation (GraphedTrainingStep).
    properties: the outputs to form (default: model.output_properties; heads are looked up in the model's own list)."""
    from newtonnet_b200.models.output import CustomOutputSet
    own = list(model.output_properties)
    props = own if properties is None else list(properties)
    if 'energy' not in props:
        raise RuntimeError("output_properties must contain 'energy'")
    for key in props:
        if key not in ('energy', 'gradient_force', 'direct_force', 'hessian'):
            raise NotImplementedError(f"the differentiable path supports energy, gradient_force, direct_force and hessian, not '{key}'")
    if not pos.is_cuda:
        raise RuntimeError('newtonnet_b200: inputs must be CUDA tensors - there is no CPU fallback')
    if pos.dtype != torch.float32 or next(model.parameters()).dtype != torch.float32:
        raise NotImplementedError('the training path computes in fp32: cast the model and inputs to float32')
    dev = pos.device
    cutoff = model.cutoff
    N, F = pos.shape[0], L.NN_F
    _image_cache.clear()                                    # operand images live for one step
    prepare_weight_images(model)
    if model.embedding_layers.requires_dr and pos.is_leaf and not pos.requires_grad:
        pos.requires_grad = True
    # ---- edges (reference order) from the cell-list kernel; image shifts are constants of the graph
    static = static_nl is not None
    nl = static_nl if static else get_engine(dev).checked_neighbor_list(pos, cell, batch, cutoff)   # regrows on overflow
    ei, dst, src, disp0, valid = _edges(nl, pos, N, static)
    # segments straight from the neighbour list: rows of the destination-sorted CSR, and - the edge set being symmetric -
    # the same rows read through the reversed-edge map for the grouping by source atom (no counting pass, no sort); a
    # list that outgrew its capacity exposes empty segments
    rev = torch.zeros(nl.cap_edges if static else max(nl.n_edges, 1), dtype=torch.int32, device=dev)
    L.check(L.load().nn_nbr_edge_reverse(C.byref(nl.struct), rev.data_ptr(), stream()), 'nn_nbr_edge_reverse')
    row_ptr = torch.where(nl.status[L.ST_EDGE_OVERFLOW] != 0, torch.zeros_like(nl.row_ptr), nl.row_ptr)
    seg_dst = Segments.from_csr(dst, N, row_ptr)
    seg_src = Segments.from_csr(src, N, row_ptr, perm=rev)
    disp = _displacements(pos, seg_dst, seg_src, disp0)
    if static:
        pad = torch.cat([torch.full((1, 1), float(cutoff), dtype=torch.float32, device=dev),
                         torch.zeros(1, 2, dtype=torch.float32, device=dev)], 1)      # fill kernels: no H2D copy while capturing
        disp = torch.where(valid.unsqueeze(1), disp, pad)
    d = disp.norm(dim=1, keepdim=True)
    u = disp / d
    x = d / cutoff
    emb = model.embedding_layers
    freq = emb.edge_embedding.embedding.frequencies
    rbf = RbfScale.apply(torch.ones_like(x), x, freq.detach().to(torch.float32).contiguous(), 0)
    rbf_pad = Fn.pad(rbf, (0, F - rbf.shape[1]))
    # nn.Embedding(119, F, padding_idx=0) (models/newtonnet.py:131,142) as a one-hot contraction through the same GEMM: its
    # weight gradient is then X^T dY on the tensor cores (deterministic) instead of ATen's atomic embedding backward
    # (3 x 104 us per step).  Exact: one-hot entries are 1.0 / 0.0 and B = B_hi + B_lo is summed exactly in fp32.
    w_emb = emb.node_embedding.weight
    if w_emb.shape[0] > F:
        raise NotImplementedError('embedding tables with more than 128 rows')
    keep = torch.ones(w_emb.shape[0], 1, dtype=torch.float32, device=dev)
    keep[0] = 0.0                                            # padding_idx = 0: row 0 neither contributes nor receives a gradient
    onehot = (z.unsqueeze(1) == torch.arange(F, device=dev).unsqueeze(0)).to(torch.float32)   # no host sync (graph capture)
    a = Gemm.apply(onehot, Fn.pad(w_emb * keep, (0, 0, 0, F - w_emb.shape[0])))
    f = torch.zeros(N, 3 * F, dtype=torch.float32, device=dev)
    for layer in model.interaction_layers:
        n0, n2 = layer.message_nodepart[0], layer.message_nodepart[2]
        mn = linear(silu(linear(a, n0.weight, n0.bias)), n2.weight, n2.bias)
        # K = 20 contraction through the same fp32-faithful GEMM (zero-padded to K = 128): a library matmul may
        # silently run in single-pass TF32 (TORCH_ALLOW_TF32_CUBLAS_OVERRIDE), which breaks gradient parity
        me = Gemm.apply(rbf_pad, Fn.pad(layer.message_edgepart.weight.t(), (0, 0, 0, F - rbf.shape[1])))
        m = GMul.apply(me, None, mn, seg_dst, mn, seg_src)
        a = a + SegmentSum.apply(m, seg_dst)
        e1 = linear(silu(linear(m, layer.equiv_message1[0].weight)), layer.equiv_message1[2].weight)
        e2 = linear(silu(linear(m, layer.equiv_message2[0].weight)), layer.equiv_message2[2].weight)
        # delta f_i = sum_{e->i} (e1_e u_e + e2_e * f_j): two segment products, no [E,3,F] tensor anywhere in the step
        f = f + (SegOuter.apply(e1, u, seg_dst) + SegMulBG.apply(e2, f.view(N, 3, F), seg_dst, seg_src)).reshape(N, 3 * F)
        g = linear(f.view(3 * N, F), layer.equiv_update.weight).view(N, 3, F)
        a = a + SumMulC.apply(f.view(N, 3, F), g)
        if layer.layer_norm is not None:
            a = Fn.layer_norm(a, (F,), layer.layer_norm.weight, layer.layer_norm.bias, layer.layer_norm.eps)
    k = own.index('energy')
    head, scaler = model.output_layers[k].layers, model.scalers[k]
    h = silu(linear(a, head[0].weight, head[0].bias))
    h = silu(linear(h, head[2].weight, head[2].bias))
    o = (h * head[4].weight).sum(1, keepdim=True) + head[4].bias           # 128 -> 1: exact fp32 reduction
    e_atom = o * _table(scaler.scale, onehot) + _table(scaler.shift, onehot)
    energy = torch.zeros(cell.shape[0], dtype=torch.float32, device=dev).index_add(0, batch, e_atom.reshape(-1))
    out = CustomOutputSet(z=z, pos=pos, cell=cell, batch=batch, edge_index=ei, atom_node=a, force_node=f.view(N, 3, F),
                          displacement=torch.eye(3, device=dev).repeat(cell.shape[0], 1, 1))
    for key in props:
        if key == 'energy':
            out.energy = energy
        elif key == 'direct_force':
            kd = own.index(key)
            dl, ds = model.output_layers[kd].layers, model.scalers[kd]
            hd = silu(linear(a, dl[0].weight, dl[0].bias))
            hd = linear(silu(linear(hd, dl[2].weight, dl[2].bias)), dl[4].weight, dl[4].bias)
            out.direct_force = RowDot.apply(f.view(N, 3, F), hd) * _table(ds.scale, onehot)
        elif key == 'hessian':
            # reference models/output.py:141-152 (vmap over unit vectors)
            if not hasattr(out, 'pos_grad') or not out.pos_grad.requires_grad:
                raise RuntimeError("'hessian' needs 'gradient_force' evaluated before it with create_graph=True "
                                   "(MLAseCalculator sets this, reference utils/ase_interface.py:125-128)")
            # training with create_graph heads (NewtonNet.train()) keeps the per-row loop; otherwise - MLAseCalculator, which
            # sets create_graph on every derivative head as the reference does, evaluates in eval mode - rows in batched blocks
            if model.training and bool(model.output_layers[own.index(key)].create_graph):
                out.hessian = hessian_rows(out.pos_grad, pos)
            else:
                from newtonnet_b200.hessian import hessian_blocks     # rows in batched blocks (newtonnet_b200/hessian.py)
                out.hessian = hessian_blocks(model, z, pos.detach(), cell, batch)
        else:
            create = bool(model.output_layers[own.index(key)].create_graph) or 'hessian' in props
            with _skip_weight_grads():              # only d/d pos is asked for: no X^T dY products in this sweep
                out.pos_grad, = torch.autograd.grad(energy, pos, torch.ones_like(energy), create_graph=create,
                                                    retain_graph=create)
            out.gradient_force = -out.pos_grad
    return out


# ----------------------------------------------------------------------------- training step (config 5)
def allreduce_gradients(params, group=None, flags=None):
    """Data-parallel gradient averaging: ONE all-reduce of a flat fp32 bucket (401,155 floats = 1.6 MB for
    the default model) instead of one per tensor; missing gradients (the dead layer-0 equiv_message2,
    the frozen frequencies) travel as zeros so every rank reduces the same layout.
    flags: optional 1-D float tensor of per-rank condition flags appended to the bucket; on return it holds their
    SUM over ranks (so every rank takes the same decision on a condition raised by one of them)."""
    params = [p for p in params if p.requires_grad]
    if not params:
        return None
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:                       # nothing to average: leave the gradients (and the flags) where they are
        return None
    parts = [(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params]
    n_flags = 0 if flags is None else flags.numel()
    if n_flags:
        parts.append(flags.reshape(-1).to(parts[0].dtype))
    flat = torch.cat(parts)
    dist.all_reduce(flat, group=group)
    if n_flags:
        flags.copy_(flat[-n_flags:].reshape(flags.shape))
        flat = flat[:-n_flags]
    flat /= world
    # one fused copy back into the parameters' gradient tensors
    views, off = [], 0
    for p in params:
        n = p.numel()
        views.append(flat[off:off + n].view_as(p))
        off += n
    missing = [i for i, p in enumerate(params) if p.grad is None]
    for i in missing:
        params[i].grad = torch.empty_like(params[i])
    torch._foreach_copy_([p.grad for p in params], views)
    return flat


_sinks = {}


class _NoSink:
    def step(self):
        import contextlib
        return contextlib.nullcontext()


def weight_grad_sink(device):
    """The device's WeightGradSink (NN_TRAIN_SINK=0: weight gradients go through autograd on the main stream)."""
    import os
    if os.environ.get('NN_TRAIN_SINK', '1') == '0':
        return _NoSink()
    device = torch.device(device)
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _sinks:
        _sinks[key] = WeightGradSink(device)
    return _sinks[key]


def training_step(model, optimizer, z, pos, cell, batch, e_target, f_target, force_weight=50.0, clip_grad=1.0,
                  group=None):
    """One step of reference train/trainer.py:303-313: forward (create_graph), loss = MSE(E) + w MSE(F)
    (train/loss.py:48), backward, gradient all-reduce across the data-parallel group, clip, optimizer step."""
    model.train()
    optimizer.zero_grad(set_to_none=True)
    pos = pos.detach().clone().requires_grad_(True)
    out = model(z, pos, cell, batch)
    loss = Fn.mse_loss(out.energy, e_target) + force_weight * Fn.mse_loss(out.gradient_force, f_target)
    with weight_grad_sink(pos.device).step():
        loss.backward()
    allreduce_gradients(model.parameters(), group)
    if clip_grad and clip_grad > 0:
        torch.nn.utils.clip_grad_norm_(model.parameters(), clip_grad)
    optimizer.step()
    return loss.detach()


class GraphedTrainingStep:
    """training_step with neighbour rebuild + forward + double backward replayed as ONE CUDA graph (static batch shape).

    Removes every host synchronisation and all Python / autograd dispatch from the captured part; the weight gradients
    form a parallel branch of the graph (WeightGradSink).  Shapes are made static by padding the edge list to the
    neighbour list's capacity (see `_edges`): every edge-level kernel of the step processes `cap_edges` rows, so the
    capacity is kept TIGHT - the probed edge count + 5 % + 256, never more than the all-pairs bound sum n_b (n_b - 1) of a
    non-periodic batch (config 5: 33.5k rows instead of the bound's 42k, for 30.2k real edges).  A replay whose batch
    outgrew the capacity is detected BEFORE the optimizer moves (the flag travels with the gradient bucket, so every
    rank sees it); with regrow=True (default) the step is then re-captured with more room and run again, with
    regrow=False it raises.  Gradient all-reduce, clipping and the optimizer step stay outside the graph.

    Host synchronisation: with an optimizer that can skip its step on a device flag (torch's fused Adam / AdamW / SGD,
    `fused=True`) and deferred_check=True (default) a call never waits for the GPU: the overflow flag is handed to the
    optimizer as its skip flag and read by the NEXT call (`settle()`), which re-captures and applies the skipped batch
    before it goes on - parameters are the same as with the strict path; only the loss RETURNED by the overflowing call
    is that of the empty padded graph.  Any other optimizer (or deferred_check=False) reads the flag every step."""

    HEADROOM = (1.05, 256)         # tight edge capacity: factor and slack over the counted edges

    def __init__(self, model, optimizer, z, pos, cell, batch, e_target, f_target, force_weight=50.0, clip_grad=1.0,
                 group=None, cap_edges=None, regrow=True, deferred_check=True):
        dev = pos.device
        self.model, self.optimizer, self.group = model, optimizer, group
        self.force_weight, self.clip_grad, self.regrow = float(force_weight), clip_grad, bool(regrow)
        self.z, self.batch = z.clone().to(torch.int64), batch.clone().to(torch.int64)
        self.pos = pos.detach().clone().to(torch.float32).contiguous()
        self.cell = cell.detach().clone().to(torch.float32).reshape(-1, 3, 3).contiguous()
        self.e_target, self.f_target = e_target.detach().clone(), f_target.detach().clone()
        self.engine = get_engine(dev)
        self.sink = weight_grad_sink(dev)
        self.recaptures = 0
        self.deferred_check = bool(deferred_check)
        self._pending = False
        self._flag_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        self._flag_event = torch.cuda.Event()
        if cap_edges is None:
            cap_edges = self._capacity(count_edges(self.engine, self.pos, self.cell, self.batch, model.cutoff).n_edges)
        else:
            cap_edges = edge_capacity(cap_edges, 1, 0)      # a given capacity is only made even
        self._capture(cap_edges)
        self.replays = 0

    def _capacity(self, n_edges):
        return edge_capacity(n_edges, *self.HEADROOM, all_pairs_bound(self.cell, self.batch))

    def _capture(self, cap_edges):
        dev = self.pos.device
        self.graph = None                                   # a previous capture's memory pool goes first
        self.nl = NeighborList(self.engine, self.pos, self.cell, self.batch, cap_edges=cap_edges)
        self.model.train()

        def zeroed_step():
            self.optimizer.zero_grad(set_to_none=True)
            self._forward_backward()
        warm_up(zeroed_step, dev, 2)
        self.optimizer.zero_grad(set_to_none=True)
        # kernels_per_replay: this library's kernels recorded in the graph
        self.graph, self.loss, self.kernels_per_replay = capture(self._forward_backward, dev)

    def _forward_backward(self):
        self.nl.rebuild(self.model.cutoff)
        pos = self.pos.clone().requires_grad_(True)
        out = differentiable_forward(self.model, self.z, pos, self.cell, self.batch, static_nl=self.nl)
        loss = Fn.mse_loss(out.energy, self.e_target) + self.force_weight * Fn.mse_loss(out.gradient_force, self.f_target)
        with self.sink.step():                  # weight gradients on a side stream: a parallel branch of the captured graph
            loss.backward()
        return loss.detach()

    def _device_skip(self):
        return self.deferred_check and bool(getattr(self.optimizer, '_step_supports_amp_scaling', False))

    def _apply(self, found_inf=None):
        """Clip + optimizer step; found_inf (device flag, exactly 1.0 = skip) makes a fused optimizer leave the parameters
        and its step count untouched without a host round trip (the mechanism torch.amp.GradScaler uses)."""
        if self.clip_grad and self.clip_grad > 0:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.clip_grad)
        if found_inf is None:
            self.optimizer.step()
            return
        self.optimizer.grad_scale, self.optimizer.found_inf = None, found_inf
        try:
            self.optimizer.step()
        finally:
            del self.optimizer.grad_scale, self.optimizer.found_inf

    def _replay(self):
        self.graph.replay()
        self.replays += 1
        # a batch that outgrew the captured edge capacity leaves padding-only rows in the replayed graph: the flag travels
        # with the gradient bucket so that every rank sees it, and it is looked at BEFORE the optimizer moves
        flag = (self.nl.status[L.ST_EDGE_OVERFLOW:L.ST_EDGE_OVERFLOW + 1] != 0).to(torch.float32)
        allreduce_gradients(self.model.parameters(), self.group, flags=flag)
        return flag

    def _run_strict(self, overflowed=False):
        """Replay, read the overflow flag on the host (one small D2H copy per step), re-capture with more room while it is set,
        then clip + step.  overflowed=True: the batch in the static buffers is already known not to fit."""
        for attempt in range(4):
            if not overflowed:
                if float(self._replay().item()) == 0:
                    break
            overflowed = False
            need = int(self.nl.status[L.ST_EDGE_OVERFLOW].item())            # 0 on a rank whose own list still fits
            if not self.regrow or attempt == 3:
                self.optimizer.zero_grad(set_to_none=False)      # in place: the captured graph keeps writing these tensors
                raise RuntimeError(f'edge capacity {self.nl.cap_edges} of the captured training graph overflowed on some rank '
                                   f'(this rank needs {need}): the step was NOT applied; rebuild GraphedTrainingStep with a larger cap_edges')
            if need:                             # this rank re-captures with room for the batch that did not fit; all ranks run the step again
                self._capture(max(self._capacity(need), self.nl.cap_edges + 2))
                self.recaptures += 1
        self._apply()

    def settle(self):
        """Deferred overflow check of the previous call (device-skip mode): waits for that call's flag; if its batch did
        not fit, the optimizer skipped it on the device - the step is re-captured with more room and the batch, still in the
        static buffers, is applied now.  Called at the start of every call and by check(); call it after the last step."""
        if not self._pending:
            return
        self._pending = False
        self._flag_event.synchronize()
        if float(self._flag_host[0]) != 0:
            self._run_strict(overflowed=True)

    def __call__(self, z, pos, cell, batch, e_target, f_target):
        if pos.shape != self.pos.shape or cell.reshape(-1, 3, 3).shape != self.cell.shape:
            raise ValueError('GraphedTrainingStep was captured for a different batch shape')
        self.settle()
        self.z.copy_(z); self.batch.copy_(batch); self.pos.copy_(pos.detach()); self.cell.copy_(cell.detach().reshape(-1, 3, 3))
        self.e_target.copy_(e_target); self.f_target.copy_(f_target)
        if not self._device_skip():
            self._run_strict()
            return self.loss.clone()
        # no host synchronisation in the step: the flag goes to pinned memory for the next call's settle(), and to the fused
        # optimizer as its skip flag
        flag = self._replay()
        self._flag_host.copy_(flag, non_blocking=True)
        self._flag_event.record()
        self._pending = True
        self._apply(found_inf=(flag > 0).to(torch.float32).reshape(()))      # 0-dim, as torch.amp.GradScaler passes it
        return self.loss.clone()

    def check(self):
        """Status words of the last replay (one host synchronisation): raises when the edge capacity overflowed."""
        self.settle()
        st = self.nl.check()
        if st[L.ST_EDGE_OVERFLOW]:
            raise RuntimeError(f'edge capacity {self.nl.cap_edges} overflowed ({st[L.ST_EDGE_OVERFLOW]} needed)')
        return st

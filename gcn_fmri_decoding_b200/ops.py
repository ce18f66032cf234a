"""PyTorch custom ops (``torch.library``, namespace ``gcn_b200``) over the C ABI.

PyTorch is plumbing here: it owns device memory (outputs and workspaces come from
the caching allocator), the current stream, and autograd bookkeeping.  All
arithmetic is done by ``libgcnb200.so``; there is no fallback of any kind.

Op                       replaces (``/root/reference/lib_new/models_gcn.py``)
-----------------------  ------------------------------------------------------
``cheb_fwd / cheb_bwd``   chebyshev5 ``:587-617`` / chebyshev2 ``:558-585`` + b1relu/b2relu
                          ``:619-629`` + mpool1 ``:631-639`` and their tf.gradients ``:298-303``
``spectral_fwd / _bwd``   fourier + filter_in_fourier ``:512-539`` (+ same epilogue)
``brelu_fwd / _bwd``      b1relu / b2relu stand-alone
``mpool_fwd / _bwd``      mpool1 stand-alone (tf.nn.max_pool SAME)
``perm_gather``           coarsening.perm_data_3d (``lib_new/coarsening.py:244-265``)
``mean_f_fwd / _bwd``     tf.reduce_mean(x, -1) of ``_inference`` ``:673``
``cheb_dx``               input gradient of a ChebyNet layer alone (saliency maps, ``saliency.py``; no reference
                          counterpart)
``cheb_dL``               gradient of a ChebyNet layer w.r.t. its operator's entries (edge saliency maps,
                          ``saliency.GraphGradient``; no reference counterpart)
``adjacency_grad``        chain rule from the operator gradients to the edge weights of the adjacency (edge saliency
                          maps in ROI coordinates, ``saliency.AdjacencyGradient``; no reference counterpart)
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib
from .plan import csr_struct

BIAS_NONE, BIAS_PER_FILTER, BIAS_PER_VERTEX = _lib.BIAS_NONE, _lib.BIAS_PER_FILTER, _lib.BIAS_PER_VERTEX
ALGO_AUTO, ALGO_GENERAL, ALGO_FUSED = _lib.ALGO_AUTO, _lib.ALGO_GENERAL, _lib.ALGO_FUSED


def _stream(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t):
    return None if t is None or t.numel() == 0 else C.c_void_p(t.data_ptr())


def _workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _check_x(x, name="x"):
    if x.dim() != 3:
        raise ValueError("%s must be [B, M, F] (got %d dims)" % (name, x.dim()))
    if x.dtype != torch.float32:
        raise ValueError("%s must be float32 (the reference placeholder is tf.float32, models_gcn.py:202)" % name)
    if not x.is_cuda:
        raise ValueError("%s must be a CUDA tensor: this package has no CPU path" % name)


def _pooled(M, p):
    return -(-M // p)


# ------------------------------------------------------------------------------------------ ChebyNet layer
@torch.library.custom_op("gcn_b200::cheb_fwd", mutates_args=(), device_types="cuda")
def cheb_fwd(x: Tensor, perm: Optional[Tensor], rowptr: Tensor, col: Tensor, val: Tensor, rowptr_t: Tensor,
             col_t: Tensor, val_t: Tensor, W: Tensor, bias: Optional[Tensor], K: int, p: int, bias_mode: int,
             relu: bool, want_argmax: bool, algo: int) -> Tuple[Tensor, Tensor]:
    _check_x(x)
    x = x.contiguous()
    W = W.contiguous()
    B, M_in, Fin = x.shape
    M = rowptr.numel() - 1
    if W.dim() != 2 or W.shape[0] != Fin * K:
        raise ValueError("W must be [Fin*K, Fout] = [%d, Fout], got %s" % (Fin * K, tuple(W.shape)))
    if perm is None and M_in != M:
        raise ValueError("x has %d vertices but the Laplacian has %d" % (M_in, M))
    if perm is not None and (perm.dtype != torch.int32 or perm.numel() != M):
        raise ValueError("perm must be int32 with one entry per (padded) vertex")
    Fout = W.shape[1]
    if bias_mode != BIAS_NONE:
        want = Fout if bias_mode == BIAS_PER_FILTER else M * Fout
        if bias is None or bias.numel() != want:
            raise ValueError("bias has the wrong number of elements for bias_mode=%d" % bias_mode)
        bias = bias.contiguous()
    Mo = _pooled(M, p)
    y = torch.empty((B, Mo, Fout), dtype=torch.float32, device=x.device)
    argmax = torch.empty((B, Mo, Fout) if (want_argmax and p > 1) else (0,), dtype=torch.uint8, device=x.device)
    L = _lib.lib()
    nbytes = L.gcnb_cheb_workspace_bytes(B, M, val.numel(), Fin, Fout, K, p, 0, 0, algo)
    ws = _workspace(nbytes, x.device)
    csr = csr_struct(rowptr, col, val, (B, Fin, Fout, K, p))
    rc = L.gcnb_cheb_fwd_f32(_ptr(x), _ptr(perm), M_in, C.byref(csr), _ptr(W), _ptr(bias), _ptr(y), _ptr(argmax), None,
                             None, B, Fin, Fout, K, p, bias_mode, int(relu), algo, _ptr(ws), ws.numel(), _stream(x))
    _lib.check(rc, "gcnb_cheb_fwd_f32")
    return y, argmax


def cheb_stack_supported(rowptr: Tensor, col: Tensor, val: Tensor, B: int, F: int, K: int, nlayers: int) -> bool:
    """Whether ``cheb_stack_fwd`` can run ``nlayers`` identical F -> F layers (p = 1) on this operator in one launch."""
    if nlayers < 1 or nlayers > 8 or F != 32 or not val.is_cuda:
        return False
    csr = csr_struct(rowptr, col, val, (B, F, F, K, 1))
    return bool(_lib.lib().gcnb_cheb_stack_supported(C.byref(csr), B, F, K, nlayers))


def cheb_tap_image(W: Tensor, Fin: int, K: int) -> Optional[Tensor]:
    """Pre-split tap image of a layer's weights ``W [Fin*K, Fout]`` as a device byte tensor (``gcnb_cheb_tap_image_build``
    on the host, then uploaded), or None for widths the tcgen05 kernel does not take.  Valid for these weight VALUES."""
    L = _lib.lib()
    Fout = int(W.shape[1])
    n = L.gcnb_cheb_tap_image_bytes(Fin, Fout, K)
    if not n:
        return None
    host_w = np.ascontiguousarray(W.detach().to("cpu", torch.float32).numpy())
    img = np.zeros(n, np.uint8)
    _lib.check(L.gcnb_cheb_tap_image_build(host_w.ctypes.data, Fin, Fout, K, img.ctypes.data, n), "gcnb_cheb_tap_image_build")
    return torch.from_numpy(img).to(W.device)


def cheb_stack_fwd(x: Tensor, rowptr: Tensor, col: Tensor, val: Tensor, Ws, biases, K: int, bias_mode: int,
                   relu: bool, tap_images=None) -> Tensor:
    """A run of identical ChebyNet layers (same operator, p = 1, 32 -> 32, same K) as ONE launch of the tcgen05 kernel
    (``gcnb_cheb_stack_fwd_f32``): activations stay on the SM between the layers.  Inference only (no autograd);
    bit-identical to calling ``cheb_fwd`` layer by layer."""
    _check_x(x)
    x = x.contiguous()
    B, M, F = x.shape
    n = len(Ws)
    Ws = [w.contiguous() for w in Ws]
    for w in Ws:
        if w.shape != (F * K, F):
            raise ValueError("every W of the stack must be [F*K, F] = [%d, %d], got %s" % (F * K, F, tuple(w.shape)))
    if bias_mode != BIAS_NONE:
        want = F if bias_mode == BIAS_PER_FILTER else M * F
        biases = [b.contiguous() for b in biases]
        if len(biases) != n or any(b.numel() != want for b in biases):
            raise ValueError("one bias per layer with %d elements is required for bias_mode=%d" % (want, bias_mode))
    y = torch.empty_like(x)
    wp = (C.c_void_p * n)(*[w.data_ptr() for w in Ws])
    bp = (C.c_void_p * n)(*[b.data_ptr() for b in biases]) if bias_mode != BIAS_NONE else None
    tp = None
    if tap_images is not None:
        if len(tap_images) != n:
            raise ValueError("tap_images must have one entry (tensor or None) per layer")
        tp = (C.c_void_p * n)(*[None if t is None else t.data_ptr() for t in tap_images])
    csr = csr_struct(rowptr, col, val, (B, F, F, K, 1))
    rc = _lib.lib().gcnb_cheb_stack_fwd_f32(_ptr(x), C.byref(csr), wp, bp, tp, _ptr(y), n, B, F, K, bias_mode, int(relu),
                                            _stream(x))
    _lib.check(rc, "gcnb_cheb_stack_fwd_f32")
    return y


@cheb_fwd.register_fake
def _(x, perm, rowptr, col, val, rowptr_t, col_t, val_t, W, bias, K, p, bias_mode, relu, want_argmax, algo):
    B = x.shape[0]
    Mo = _pooled(rowptr.numel() - 1, p)
    y = x.new_empty((B, Mo, W.shape[1]))
    am = x.new_empty((B, Mo, W.shape[1]) if (want_argmax and p > 1) else (0,), dtype=torch.uint8)
    return y, am


@torch.library.custom_op("gcn_b200::cheb_bwd", mutates_args=(), device_types="cuda")
def cheb_bwd(x: Tensor, perm: Optional[Tensor], y: Tensor, argmax: Tensor, dy: Tensor, rowptr: Tensor, col: Tensor,
             val: Tensor, rowptr_t: Tensor, col_t: Tensor, val_t: Tensor, W: Tensor, K: int, p: int, bias_mode: int,
             relu: bool, need_dx: bool, algo: int) -> Tuple[Tensor, Tensor, Tensor]:
    x = x.contiguous()
    dy = dy.contiguous()
    B, M_in, Fin = x.shape
    M = rowptr.numel() - 1
    Fout = W.shape[1]
    dx = torch.empty((B, M, Fin) if need_dx else (0,), dtype=torch.float32, device=x.device)
    dW = torch.empty_like(W)
    nb = 0 if bias_mode == BIAS_NONE else (Fout if bias_mode == BIAS_PER_FILTER else M * Fout)
    db = torch.empty((nb,), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    nbytes = L.gcnb_cheb_workspace_bytes(B, M, val.numel(), Fin, Fout, K, p, 1, int(need_dx), algo)
    ws = _workspace(nbytes, x.device)
    csr = csr_struct(rowptr, col, val)
    csr_t = csr_struct(rowptr_t, col_t, val_t, (B, Fin, Fout, K, p))
    rc = L.gcnb_cheb_bwd_f32(_ptr(x), _ptr(perm), M_in, _ptr(y), _ptr(argmax), _ptr(dy), 0, None, C.byref(csr),
                             C.byref(csr_t), _ptr(W), _ptr(dx), _ptr(dW), _ptr(db), B, Fin, Fout, K, p, bias_mode,
                             int(relu), algo, _ptr(ws), ws.numel(), _stream(x))
    _lib.check(rc, "gcnb_cheb_bwd_f32")
    return dx, dW, db


@cheb_bwd.register_fake
def _(x, perm, y, argmax, dy, rowptr, col, val, rowptr_t, col_t, val_t, W, K, p, bias_mode, relu, need_dx, algo):
    M = rowptr.numel() - 1
    Fout = W.shape[1]
    nb = 0 if bias_mode == BIAS_NONE else (Fout if bias_mode == BIAS_PER_FILTER else M * Fout)
    return (x.new_empty((x.shape[0], M, x.shape[2]) if need_dx else (0,)), torch.empty_like(W), x.new_empty((nb,)))


# Variants used by the explicit training schedule (train.FusedTrainer): the last conv layer also emits the mean over
# its filters (the head's input, models_gcn.py:673) and its backward takes the gradient of that mean; weight and bias
# gradients are written straight into caller-provided views of the flat gradient buffer.
@torch.library.custom_op("gcn_b200::cheb_fwd_mean", mutates_args=(), device_types="cuda")
def cheb_fwd_mean(x: Tensor, perm: Optional[Tensor], rowptr: Tensor, col: Tensor, val: Tensor, W: Tensor,
                  bias: Optional[Tensor], K: int, p: int, bias_mode: int, relu: bool, algo: int,
                  want_stack: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    _check_x(x)
    x = x.contiguous()
    B, M_in, Fin = x.shape
    M = rowptr.numel() - 1
    Fout = W.shape[1]
    Mo = _pooled(M, p)
    y = torch.empty((B, Mo, Fout), dtype=torch.float32, device=x.device)
    argmax = torch.empty((B, Mo, Fout) if p > 1 else (0,), dtype=torch.uint8, device=x.device)
    ymean = torch.empty((B, Mo), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    FP = L.gcnb_cheb_stack_width(B, M, val.numel(), Fin, Fout, K, p) if (want_stack and algo != ALGO_GENERAL) else 0
    stack = torch.empty((K, B, M, FP) if FP else (0,), dtype=torch.float32, device=x.device)
    ws = _workspace(L.gcnb_cheb_workspace_bytes(B, M, val.numel(), Fin, Fout, K, p, 0, 0, algo), x.device)
    csr = csr_struct(rowptr, col, val, (B, Fin, Fout, K, p))
    rc = L.gcnb_cheb_fwd_f32(_ptr(x), _ptr(perm), M_in, C.byref(csr), _ptr(W), _ptr(bias), _ptr(y), _ptr(argmax),
                             _ptr(ymean), _ptr(stack), B, Fin, Fout, K, p, bias_mode, int(relu), algo, _ptr(ws), ws.numel(),
                             _stream(x))
    _lib.check(rc, "gcnb_cheb_fwd_f32")
    return y, argmax, ymean, stack


@cheb_fwd_mean.register_fake
def _(x, perm, rowptr, col, val, W, bias, K, p, bias_mode, relu, algo, want_stack=False):
    B = x.shape[0]
    Mo = _pooled(rowptr.numel() - 1, p)
    return (x.new_empty((B, Mo, W.shape[1])), x.new_empty((B, Mo, W.shape[1]) if p > 1 else (0,), dtype=torch.uint8),
            x.new_empty((B, Mo)), x.new_empty((0,)))


@torch.library.custom_op("gcn_b200::cheb_bwd_into", mutates_args=("dW_out", "db_out"), device_types="cuda")
def cheb_bwd_into(x: Tensor, perm: Optional[Tensor], y: Tensor, argmax: Tensor, dy: Tensor, dy_is_mean: bool,
                  rowptr: Tensor, col: Tensor, val: Tensor, rowptr_t: Tensor, col_t: Tensor, val_t: Tensor, W: Tensor,
                  dW_out: Tensor, db_out: Tensor, K: int, p: int, bias_mode: int, relu: bool, need_dx: bool,
                  algo: int, stack: Optional[Tensor] = None) -> Tensor:
    x = x.contiguous()
    dy = dy.contiguous()
    B, M_in, Fin = x.shape
    M = rowptr.numel() - 1
    Fout = W.shape[1]
    if not (dW_out.is_contiguous() and db_out.is_contiguous() and dW_out.numel() == W.numel()):
        raise ValueError("dW_out / db_out must be contiguous views of the right size")
    dx = torch.empty((B, M, Fin) if need_dx else (0,), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    ws = _workspace(L.gcnb_cheb_workspace_bytes(B, M, val.numel(), Fin, Fout, K, p, 1, int(need_dx), algo), x.device)
    csr = csr_struct(rowptr, col, val)
    csr_t = csr_struct(rowptr_t, col_t, val_t, (B, Fin, Fout, K, p))
    rc = L.gcnb_cheb_bwd_f32(_ptr(x), _ptr(perm), M_in, _ptr(y), _ptr(argmax), _ptr(dy), int(dy_is_mean), _ptr(stack),
                             C.byref(csr),
                             C.byref(csr_t), _ptr(W), _ptr(dx), _ptr(dW_out), _ptr(db_out), B, Fin, Fout, K, p, bias_mode,
                             int(relu), algo, _ptr(ws), ws.numel(), _stream(x))
    _lib.check(rc, "gcnb_cheb_bwd_f32")
    return dx


@cheb_bwd_into.register_fake
def _(x, perm, y, argmax, dy, dy_is_mean, rowptr, col, val, rowptr_t, col_t, val_t, W, dW_out, db_out, K, p, bias_mode,
      relu, need_dx, algo, stack=None):
    return x.new_empty((x.shape[0], rowptr.numel() - 1, x.shape[2]) if need_dx else (0,))


@torch.library.custom_op("gcn_b200::cheb_dx", mutates_args=(), device_types="cuda")
def cheb_dx(x: Optional[Tensor], perm: Optional[Tensor], M_in: int, y: Tensor, argmax: Tensor, dy: Tensor,
            dy_is_mean: bool, rowptr: Tensor, col: Tensor, val: Tensor, rowptr_t: Tensor, col_t: Tensor, val_t: Tensor,
            W: Tensor, K: int, p: int, relu: bool, algo: int) -> Tensor:
    """Input gradient of a ChebyNet layer alone (``gcnb_cheb_dx_f32``: no dW, no db).  With ``perm`` (a Graclus
    permutation of the layer's vertices) it is the gradient w.r.t. the raw windows ``[B, M_in, Fin]``, un-permuted in the
    kernel's store; without, w.r.t. the layer input ``[B, M, Fin]``.  ``x`` (the layer input) may be None on the tcgen05
    route, which never reads it (``_lib.describe_dx`` names the route)."""
    dy = dy.contiguous()
    B = y.shape[0]
    M = rowptr.numel() - 1
    Fout = W.shape[1]
    Fin = W.shape[0] // K
    if perm is None and M_in != M:
        raise ValueError("without perm the layer input has M = %d vertices (got M_in = %d)" % (M, M_in))
    if perm is not None and (perm.dtype != torch.int32 or perm.numel() != M):
        raise ValueError("perm must be int32 with one entry per (padded) vertex")
    if x is not None:
        x = x.contiguous()
        if tuple(x.shape) != (B, M_in, Fin):
            raise ValueError("x must be [B, M_in, Fin] = %s, got %s" % ((B, M_in, Fin), tuple(x.shape)))
    dx = torch.empty((B, M_in, Fin), dtype=torch.float32, device=y.device)
    L = _lib.lib()
    _, nbytes = _lib.describe_dx(B, M, val.numel(), Fin, Fout, K, p, algo)
    ws = _workspace(nbytes, y.device)
    csr = csr_struct(rowptr, col, val)
    csr_t = csr_struct(rowptr_t, col_t, val_t, (B, Fin, Fout, K, p))
    rc = L.gcnb_cheb_dx_f32(_ptr(x), _ptr(perm), M_in, _ptr(y), _ptr(argmax), _ptr(dy), int(dy_is_mean), C.byref(csr),
                            C.byref(csr_t), _ptr(W.contiguous()), _ptr(dx), B, Fin, Fout, K, p, int(relu), algo, _ptr(ws),
                            ws.numel(), _stream(y))
    _lib.check(rc, "gcnb_cheb_dx_f32")
    return dx


@cheb_dx.register_fake
def _(x, perm, M_in, y, argmax, dy, dy_is_mean, rowptr, col, val, rowptr_t, col_t, val_t, W, K, p, relu, algo):
    return y.new_empty((y.shape[0], M_in, W.shape[0] // K))


@torch.library.custom_op("gcn_b200::cheb_dL", mutates_args=("dval", "ddiag"), device_types="cuda")
def cheb_dL(x: Tensor, perm: Optional[Tensor], M_in: int, y: Tensor, argmax: Tensor, dy: Tensor, dy_is_mean: bool,
            rowptr: Tensor, col: Tensor, val: Tensor, rowptr_t: Tensor, col_t: Tensor, val_t: Tensor, W: Tensor,
            dval: Tensor, ddiag: Tensor, accumulate: bool, K: int, p: int, relu: bool, need_dx: bool) -> Tensor:
    """Gradient of a ChebyNet layer w.r.t. the entries of its operator (``gcnb_cheb_dL_f32``), per window: into
    ``dval [B, nnz]`` (L~'s CSR entries) and ``ddiag [B, M]`` (the diagonal ``(i, i)``), both contiguous float32;
    ``accumulate`` adds onto them (layers that share an operator).  Returns the layer's input gradient with ``need_dx``
    (bit for bit ``cheb_dx`` on the general path, un-permuted through ``perm``), else an empty tensor."""
    dy = dy.contiguous()
    x = x.contiguous()
    B, M = y.shape[0], rowptr.numel() - 1
    Fout = W.shape[1]
    Fin = W.shape[0] // K
    nnz = val.numel()
    if perm is None and M_in != M:
        raise ValueError("without perm the layer input has M = %d vertices (got M_in = %d)" % (M, M_in))
    if perm is not None and (perm.dtype != torch.int32 or perm.numel() != M):
        raise ValueError("perm must be int32 with one entry per (padded) vertex")
    if tuple(x.shape) != (B, M_in, Fin):
        raise ValueError("x must be [B, M_in, Fin] = %s, got %s" % ((B, M_in, Fin), tuple(x.shape)))
    for name, t, shape in (("dval", dval, (B, nnz)), ("ddiag", ddiag, (B, M))):
        if tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("%s must be a contiguous float32 %s tensor" % (name, shape))
    dx = torch.empty((B, M_in, Fin) if need_dx else (0,), dtype=torch.float32, device=y.device)
    L = _lib.lib()
    _, nbytes = _lib.describe_dL(B, M, nnz, Fin, Fout, K, p)
    ws = _workspace(nbytes, y.device)
    csr = csr_struct(rowptr, col, val)
    csr_t = csr_struct(rowptr_t, col_t, val_t)
    rc = L.gcnb_cheb_dL_f32(_ptr(x), _ptr(perm), M_in, _ptr(y), _ptr(argmax), _ptr(dy), int(dy_is_mean), C.byref(csr),
                            C.byref(csr_t), _ptr(W.contiguous()), _ptr(dval), _ptr(ddiag), int(accumulate), _ptr(dx), B,
                            Fin, Fout, K, p, int(relu), _ptr(ws), ws.numel(), _stream(y))
    _lib.check(rc, "gcnb_cheb_dL_f32")
    return dx


@cheb_dL.register_fake
def _(x, perm, M_in, y, argmax, dy, dy_is_mean, rowptr, col, val, rowptr_t, col_t, val_t, W, dval, ddiag, accumulate, K,
      p, relu, need_dx):
    return y.new_empty((y.shape[0], M_in, W.shape[0] // K) if need_dx else (0,))


def adjacency_grad(levels, edges: Tensor, absolute: bool) -> Tensor:
    """Gradient w.r.t. the undirected edge weights of the adjacency, per window (``gcnb_adjacency_grad_f32``): float32
    ``[B, E]``.  ``levels``, finest first: one ``(dval [B, nnz], rowptr, val, rowptr_t, tpos, ss, hinv, parent)`` per
    level, ``dval`` the level's operator gradient (``cheb_dL``'s, contiguous float32), ``rowptr / val / rowptr_t`` its
    plan's CSR arrays, ``tpos`` (int32 [nnz]) the position in ``val`` of each entry of the transpose's CSR order,
    ``ss`` (float32 [nnz]) ``s_a s_b``, ``hinv`` (float32 [M]) ``1 / (2 d)``, ``parent`` (int32 [nnz]) the entry of the next
    level in the list or -1, None for the last.  ``edges`` (int32 [E, 2]): the level-0 entries ``(a, b)`` and ``(b, a)`` of
    each edge.  ``absolute``: ``|.|`` per window.  No host synchronisation (CUDA-graph capturable)."""
    dev = edges.device
    B = levels[0][0].shape[0]
    structs = (_lib.GcnbAdjLevel * len(levels))()
    for l, (dval, rowptr, val, rowptr_t, tpos, ss, hinv, parent) in enumerate(levels):
        M, nnz = rowptr.numel() - 1, val.numel()
        if tuple(dval.shape) != (B, nnz) or dval.dtype != torch.float32 or not dval.is_contiguous():
            raise ValueError("level %d: dval must be a contiguous float32 %s tensor" % (l, (B, nnz)))
        for name, t, n, dt in (("rowptr_t", rowptr_t, M + 1, torch.int32), ("tpos", tpos, nnz, torch.int32),
                               ("ss", ss, nnz, torch.float32), ("hinv", hinv, M, torch.float32)):
            if t.numel() != n or t.dtype != dt or t.device != dev:
                raise ValueError("level %d: %s must be %s with %d entries on %s" % (l, name, dt, n, dev))
        if (parent is None) != (l == len(levels) - 1) or (parent is not None and parent.numel() != nnz):
            raise ValueError("level %d: parent must be int32 [nnz] on every level but the last, None there" % l)
        addr = lambda t: None if t is None or t.numel() == 0 else t.data_ptr()
        structs[l] = _lib.GcnbAdjLevel(addr(dval), addr(rowptr), addr(val), addr(rowptr_t), addr(tpos), addr(ss),
                                       addr(hinv), addr(parent), M, nnz)
    if edges.dim() != 2 or edges.shape[1] != 2 or edges.dtype != torch.int32:
        raise ValueError("edges must be int32 [E, 2]")
    E = edges.shape[0]
    out = torch.empty((B, E), dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = _workspace(L.gcnb_adjacency_grad_workspace_bytes(structs, len(levels), B), dev)
    rc = L.gcnb_adjacency_grad_f32(structs, len(levels), _ptr(edges), E, _ptr(out), B, int(absolute), _ptr(ws),
                                   ws.numel(), _stream(out))
    _lib.check(rc, "gcnb_adjacency_grad_f32")
    return out


def unpermute(dx: Tensor, perm: Tensor, M_in: int) -> Tensor:
    """Gradient w.r.t. the raw windows ``[B, M_in, F]`` from the gradient ``dx [B, M, F]`` w.r.t. the input permuted by
    ``perm`` (the adjoint of ``perm_gather``): row m goes back to raw row ``perm[m]``; fake vertices (``perm[m] >= M_in``)
    are dropped.  No host synchronisation (CUDA-graph capturable): fake vertices land in one extra row, cut off."""
    gx = dx.new_zeros((dx.shape[0], M_in + 1, dx.shape[2]))
    gx.index_copy_(1, torch.where(perm < M_in, perm, M_in).long(), dx)
    return gx[:, :M_in]


def _cheb_setup(ctx, inputs, output):
    (x, perm, rowptr, col, val, rowptr_t, col_t, val_t, W, bias, K, p, bias_mode, relu, want_argmax, algo) = inputs
    y, argmax = output
    if p > 1 and not want_argmax:
        raise ValueError("cheb_fwd needs want_argmax=True to be differentiable when p > 1")
    ctx.save_for_backward(x, perm, rowptr, col, val, rowptr_t, col_t, val_t, W, y, argmax)
    ctx.meta = (K, p, bias_mode, relu, algo, None if bias is None else tuple(bias.shape))


def _cheb_backward(ctx, dy, _dargmax):
    x, perm, rowptr, col, val, rowptr_t, col_t, val_t, W, y, argmax = ctx.saved_tensors
    K, p, bias_mode, relu, algo, bshape = ctx.meta
    need_dx = ctx.needs_input_grad[0]
    dx, dW, db = torch.ops.gcn_b200.cheb_bwd(x, perm, y, argmax, dy, rowptr, col, val, rowptr_t, col_t, val_t, W, K, p,
                                             bias_mode, relu, need_dx, algo)
    gx = None
    if need_dx:
        gx = dx if perm is None else unpermute(dx, perm, x.shape[1])
    gb = db.reshape(bshape) if (bshape is not None and ctx.needs_input_grad[9]) else None
    return (gx, None, None, None, None, None, None, None, dW if ctx.needs_input_grad[8] else None, gb,
            None, None, None, None, None, None)


cheb_fwd.register_autograd(_cheb_backward, setup_context=_cheb_setup)


# ------------------------------------------------------------------------------------------ spectral layer
@torch.library.custom_op("gcn_b200::spectral_fwd", mutates_args=(), device_types="cuda")
def spectral_fwd(x: Tensor, Ut: Tensor, W: Tensor, bias: Optional[Tensor], p: int, bias_mode: int, relu: bool,
                 want_argmax: bool) -> Tuple[Tensor, Tensor]:
    _check_x(x)
    x = x.contiguous()
    W = W.contiguous()
    B, M, Fin = x.shape
    if Ut.shape != (M, M):
        raise ValueError("Ut must be [M, M] with M = x.shape[1]")
    if W.dim() != 3 or W.shape[0] != M or W.shape[2] != Fin:
        raise ValueError("W must be [M, Fout, Fin] (models_gcn.py:538), got %s" % (tuple(W.shape),))
    Fout = W.shape[1]
    if bias_mode != BIAS_NONE:
        bias = bias.contiguous()
    Mo = _pooled(M, p)
    y = torch.empty((B, Mo, Fout), dtype=torch.float32, device=x.device)
    argmax = torch.empty((B, Mo, Fout) if (want_argmax and p > 1) else (0,), dtype=torch.uint8, device=x.device)
    L = _lib.lib()
    ws = _workspace(L.gcnb_spectral_workspace_bytes(B, M, Fin, Fout, p, 0), x.device)
    rc = L.gcnb_spectral_fwd_f32(_ptr(x), _ptr(Ut), _ptr(W), _ptr(bias), _ptr(y), _ptr(argmax), B, M, Fin, Fout, p,
                                 bias_mode, int(relu), _ptr(ws), ws.numel(), _stream(x))
    _lib.check(rc, "gcnb_spectral_fwd_f32")
    return y, argmax


@spectral_fwd.register_fake
def _(x, Ut, W, bias, p, bias_mode, relu, want_argmax):
    B, M, _ = x.shape
    Mo = _pooled(M, p)
    return (x.new_empty((B, Mo, W.shape[1])),
            x.new_empty((B, Mo, W.shape[1]) if (want_argmax and p > 1) else (0,), dtype=torch.uint8))


@torch.library.custom_op("gcn_b200::spectral_bwd", mutates_args=(), device_types="cuda")
def spectral_bwd(x: Tensor, y: Tensor, argmax: Tensor, dy: Tensor, Ut: Tensor, W: Tensor, p: int, bias_mode: int,
                 relu: bool, need_dx: bool) -> Tuple[Tensor, Tensor, Tensor]:
    x = x.contiguous()
    dy = dy.contiguous()
    B, M, Fin = x.shape
    Fout = W.shape[1]
    dx = torch.empty((B, M, Fin) if need_dx else (0,), dtype=torch.float32, device=x.device)
    dW = torch.empty_like(W)
    nb = 0 if bias_mode == BIAS_NONE else (Fout if bias_mode == BIAS_PER_FILTER else M * Fout)
    db = torch.empty((nb,), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    ws = _workspace(L.gcnb_spectral_workspace_bytes(B, M, Fin, Fout, p, 1), x.device)
    rc = L.gcnb_spectral_bwd_f32(_ptr(x), _ptr(y), _ptr(argmax), _ptr(dy), _ptr(Ut), _ptr(W), _ptr(dx), _ptr(dW),
                                 _ptr(db), B, M, Fin, Fout, p, bias_mode, int(relu), _ptr(ws), ws.numel(), _stream(x))
    _lib.check(rc, "gcnb_spectral_bwd_f32")
    return dx, dW, db


@spectral_bwd.register_fake
def _(x, y, argmax, dy, Ut, W, p, bias_mode, relu, need_dx):
    M, Fout = x.shape[1], W.shape[1]
    nb = 0 if bias_mode == BIAS_NONE else (Fout if bias_mode == BIAS_PER_FILTER else M * Fout)
    return (x.new_empty(tuple(x.shape) if need_dx else (0,)), torch.empty_like(W), x.new_empty((nb,)))


def _spectral_setup(ctx, inputs, output):
    x, Ut, W, bias, p, bias_mode, relu, want_argmax = inputs
    y, argmax = output
    if p > 1 and not want_argmax:
        raise ValueError("spectral_fwd needs want_argmax=True to be differentiable when p > 1")
    ctx.save_for_backward(x, Ut, W, y, argmax)
    ctx.meta = (p, bias_mode, relu, None if bias is None else tuple(bias.shape))


def _spectral_backward(ctx, dy, _dargmax):
    x, Ut, W, y, argmax = ctx.saved_tensors
    p, bias_mode, relu, bshape = ctx.meta
    need_dx = ctx.needs_input_grad[0]
    dx, dW, db = torch.ops.gcn_b200.spectral_bwd(x, y, argmax, dy, Ut, W, p, bias_mode, relu, need_dx)
    gb = db.reshape(bshape) if (bshape is not None and ctx.needs_input_grad[3]) else None
    return (dx if need_dx else None, None, dW if ctx.needs_input_grad[2] else None, gb, None, None, None, None)


spectral_fwd.register_autograd(_spectral_backward, setup_context=_spectral_setup)


# ------------------------------------------------------------------------------------------ stand-alone pieces
@torch.library.custom_op("gcn_b200::brelu_fwd", mutates_args=(), device_types="cuda")
def brelu_fwd(x: Tensor, bias: Tensor, bias_mode: int) -> Tensor:
    _check_x(x)
    x = x.contiguous()
    bias = bias.contiguous()
    B, M, F = x.shape
    if bias.numel() != (F if bias_mode == BIAS_PER_FILTER else M * F):
        raise ValueError("bias has the wrong number of elements for bias_mode=%d" % bias_mode)
    y = torch.empty_like(x)
    rc = _lib.lib().gcnb_brelu_fwd_f32(_ptr(x), _ptr(bias), _ptr(y), B, M, F, bias_mode, _stream(x))
    _lib.check(rc, "gcnb_brelu_fwd_f32")
    return y


@brelu_fwd.register_fake
def _(x, bias, bias_mode):
    return torch.empty_like(x)


@torch.library.custom_op("gcn_b200::brelu_bwd", mutates_args=(), device_types="cuda")
def brelu_bwd(dy: Tensor, y: Tensor, bias_mode: int) -> Tuple[Tensor, Tensor]:
    dy = dy.contiguous()
    B, M, F = y.shape
    dx = torch.empty_like(y)
    db = torch.empty((F if bias_mode == BIAS_PER_FILTER else M * F,), dtype=torch.float32, device=y.device)
    ws = _workspace(M * F * 4 + 256, y.device)
    rc = _lib.lib().gcnb_brelu_bwd_f32(_ptr(dy), _ptr(y), _ptr(dx), _ptr(db), B, M, F, bias_mode, _ptr(ws), ws.numel(),
                                       _stream(y))
    _lib.check(rc, "gcnb_brelu_bwd_f32")
    return dx, db


@brelu_bwd.register_fake
def _(dy, y, bias_mode):
    B, M, F = y.shape
    return torch.empty_like(y), y.new_empty((F if bias_mode == BIAS_PER_FILTER else M * F,))


def _brelu_setup(ctx, inputs, output):
    _, bias, bias_mode = inputs
    ctx.save_for_backward(output)
    ctx.meta = (bias_mode, tuple(bias.shape))


def _brelu_backward(ctx, dy):
    (y,) = ctx.saved_tensors
    bias_mode, bshape = ctx.meta
    dx, db = torch.ops.gcn_b200.brelu_bwd(dy, y, bias_mode)
    return dx, db.reshape(bshape), None


brelu_fwd.register_autograd(_brelu_backward, setup_context=_brelu_setup)


@torch.library.custom_op("gcn_b200::mpool_fwd", mutates_args=(), device_types="cuda")
def mpool_fwd(x: Tensor, p: int) -> Tuple[Tensor, Tensor]:
    _check_x(x)
    x = x.contiguous()
    B, M, F = x.shape
    Mo = _pooled(M, p)
    y = torch.empty((B, Mo, F), dtype=torch.float32, device=x.device)
    am = torch.empty((B, Mo, F), dtype=torch.uint8, device=x.device)
    rc = _lib.lib().gcnb_mpool_fwd_f32(_ptr(x), _ptr(y), _ptr(am), B, M, F, p, _stream(x))
    _lib.check(rc, "gcnb_mpool_fwd_f32")
    return y, am


@mpool_fwd.register_fake
def _(x, p):
    B, M, F = x.shape
    return x.new_empty((B, _pooled(M, p), F)), x.new_empty((B, _pooled(M, p), F), dtype=torch.uint8)


@torch.library.custom_op("gcn_b200::mpool_bwd", mutates_args=(), device_types="cuda")
def mpool_bwd(dy: Tensor, argmax: Tensor, M: int, p: int) -> Tensor:
    dy = dy.contiguous()
    B, Mo, F = dy.shape
    dx = torch.empty((B, M, F), dtype=torch.float32, device=dy.device)
    rc = _lib.lib().gcnb_mpool_bwd_f32(_ptr(dy), _ptr(argmax), _ptr(dx), B, M, F, p, _stream(dy))
    _lib.check(rc, "gcnb_mpool_bwd_f32")
    return dx


@mpool_bwd.register_fake
def _(dy, argmax, M, p):
    return dy.new_empty((dy.shape[0], M, dy.shape[2]))


def _mpool_setup(ctx, inputs, output):
    x, p = inputs
    ctx.save_for_backward(output[1])
    ctx.meta = (x.shape[1], p)


def _mpool_backward(ctx, dy, _dam):
    (am,) = ctx.saved_tensors
    M, p = ctx.meta
    return torch.ops.gcn_b200.mpool_bwd(dy, am, M, p), None


mpool_fwd.register_autograd(_mpool_backward, setup_context=_mpool_setup)


@torch.library.custom_op("gcn_b200::perm_gather", mutates_args=(), device_types="cuda")
def perm_gather(x: Tensor, perm: Tensor) -> Tensor:
    _check_x(x)
    x = x.contiguous()
    if perm.dtype != torch.int32:
        raise ValueError("perm must be int32")
    B, M_in, F = x.shape
    M_out = perm.numel()
    if M_out < M_in:
        raise ValueError("the ordering is shorter than the data (coarsening.py:254)")
    y = torch.empty((B, M_out, F), dtype=torch.float32, device=x.device)
    rc = _lib.lib().gcnb_perm_gather_f32(_ptr(x), _ptr(perm), _ptr(y), B, M_in, M_out, F, _stream(x))
    _lib.check(rc, "gcnb_perm_gather_f32")
    return y


@perm_gather.register_fake
def _(x, perm):
    return x.new_empty((x.shape[0], perm.numel(), x.shape[2]))


@torch.library.custom_op("gcn_b200::mean_f_fwd", mutates_args=(), device_types="cuda")
def mean_f_fwd(x: Tensor) -> Tensor:
    x = x.contiguous()
    F = x.shape[-1]
    rows = x.numel() // F
    y = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device)
    rc = _lib.lib().gcnb_mean_f_fwd_f32(_ptr(x), _ptr(y), rows, F, _stream(x))
    _lib.check(rc, "gcnb_mean_f_fwd_f32")
    return y


@mean_f_fwd.register_fake
def _(x):
    return x.new_empty(x.shape[:-1])


@torch.library.custom_op("gcn_b200::mean_f_bwd", mutates_args=(), device_types="cuda")
def mean_f_bwd(dy: Tensor, F: int) -> Tensor:
    dy = dy.contiguous()
    dx = torch.empty(tuple(dy.shape) + (F,), dtype=torch.float32, device=dy.device)
    rc = _lib.lib().gcnb_mean_f_bwd_f32(_ptr(dy), _ptr(dx), dy.numel(), F, _stream(dy))
    _lib.check(rc, "gcnb_mean_f_bwd_f32")
    return dx


@mean_f_bwd.register_fake
def _(dy, F):
    return dy.new_empty(tuple(dy.shape) + (F,))


def _mean_setup(ctx, inputs, output):
    ctx.F = inputs[0].shape[-1]


def _mean_backward(ctx, dy):
    return torch.ops.gcn_b200.mean_f_bwd(dy, ctx.F)


mean_f_fwd.register_autograd(_mean_backward, setup_context=_mean_setup)

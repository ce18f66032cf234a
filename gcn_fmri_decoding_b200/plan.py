"""Device-resident operator plans: what the kernels need of a Laplacian, uploaded once.

``GraphPlan`` is the replacement of the graph-build-time block of the reference's
``chebyshev5`` (``/root/reference/lib_new/models_gcn.py:590-596``: csr copy ->
``graph.rescale_L(L, lmax=2)`` -> COO -> ``tf.SparseTensor`` -> ``sparse_reorder``).
``SpectralPlan`` replaces ``models_gcn.py:535-536`` (``graph.fourier`` -> ``U.T`` constant).
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib, graphs


class GraphPlan:
    """Rescaled Laplacian ``L~`` (CSR) and its explicit transpose on the device, fp32/int32.

    ``L`` is the *un-rescaled* normalised Laplacian exactly as ``graph.laplacian`` returns it
    (fp32 or fp64, any SciPy sparse format); values are cast to fp32 once here (SURVEY D8).
    The transpose is stored explicitly because ``L~`` is not bit-symmetric (SURVEY A.4).
    """

    def __init__(self, L, device="cuda", lmax=2, rescale=True):
        if not sp.issparse(L):
            raise ValueError("L must be a scipy sparse matrix")
        if L.shape[0] != L.shape[1]:
            raise ValueError("L must be square")
        Lt = graphs.rescale_L(L, lmax=lmax) if rescale else sp.csr_matrix(L)
        self.M = int(Lt.shape[0])
        self.device = torch.device(device)
        rp, ci, v = graphs.csr_arrays(Lt)
        rpt, cit, vt = graphs.csr_arrays(Lt, transpose=True)
        self.nnz = int(v.shape[0])
        self.max_degree = int(np.diff(rp).max()) if self.M > 0 else 0
        t = lambda a: torch.from_numpy(a).to(self.device)
        self.rowptr, self.col, self.val = t(rp), t(ci), t(v)
        self.rowptr_t, self.col_t, self.val_t = t(rpt), t(cit), t(vt)
        # host copies for the operator images (built lazily per layer shape, see image())
        self._host = {False: (rp, ci, v), True: (rpt, cit, vt)}
        self._images = {}
        if self.device.type == "cuda":
            _PLANS[self.val.data_ptr()] = (weakref.ref(self), False, self.val._version)
            _PLANS[self.val_t.data_ptr()] = (weakref.ref(self), True, self.val_t._version)
            weakref.finalize(self, _forget, self.val.data_ptr(), self.val_t.data_ptr())

    def tensors(self):
        return self.rowptr, self.col, self.val, self.rowptr_t, self.col_t, self.val_t

    def image(self, shape, transposed=False):
        """Device tensor holding the operator image of layer ``shape = (B, Fin, Fout, K, p)`` (``gcnb_cheb_image_build``),
        or ``None`` when the library has no image-based kernel for it.  ``transposed``: the image of ``L~^T`` that serves
        the input gradient of the same layer.  Built once per shape and cached."""
        key = (tuple(int(a) for a in shape), bool(transposed))
        if key not in self._images:
            B, Fin, Fout, K, p = key[0]
            rp, ci, v = self._host[key[1]]
            L = _lib.lib()
            args = (B, self.M, self.nnz, Fin, Fout, K, p, int(key[1]))
            n = L.gcnb_cheb_image_bytes(rp.ctypes.data, ci.ctypes.data, *args)
            img = None
            if n:
                host = np.zeros(n, np.uint8)
                _lib.check(L.gcnb_cheb_image_build(rp.ctypes.data, ci.ctypes.data, v.ctypes.data, *args, host.ctypes.data, n),
                           "gcnb_cheb_image_build")
                img = torch.from_numpy(host).to(self.device)
            self._images[key] = img
        return self._images[key]


# plan.USE_IMAGES = False: never attach operator images -- the kernels then build their own CSR-ordered work lists in
# every launch (the tests that cover callers passing no image set it)
USE_IMAGES = True

# device address of a plan's value array -> (plan, is-transpose, tensor version at upload); lets csr_struct find the
# plan (hence the cached operator images) behind the raw tensors the custom ops are called with
_PLANS = {}


def _forget(*ptrs):
    for p in ptrs:
        _PLANS.pop(p, None)


def csr_struct(rowptr, col, val, shape=None):
    """``gcnb_csr`` for three device tensors (kept alive by the caller for the duration of the call).

    With ``shape = (B, Fin, Fout, K, p)`` of the layer about to run, the operator image of the owning ``GraphPlan``
    is attached when these are a plan's (unmodified) tensors; otherwise the kernels derive their work lists themselves.
    """
    csr = _lib.GcnbCsr(rowptr.data_ptr(), col.data_ptr(), val.data_ptr(), rowptr.numel() - 1, val.numel(), None, 0)
    if shape is not None and USE_IMAGES:
        ent = _PLANS.get(val.data_ptr())
        plan = ent[0]() if ent else None
        if plan is not None and val._version == ent[2]:
            t = (plan.rowptr_t, plan.col_t) if ent[1] else (plan.rowptr, plan.col)
            if t[0].data_ptr() == rowptr.data_ptr() and t[1].data_ptr() == col.data_ptr():
                img = plan.image(shape, ent[1])
                if img is not None:
                    csr.image, csr.image_bytes = img.data_ptr(), img.numel()
    return csr


class SpectralPlan:
    """``Ut`` = transposed eigenvector matrix of ``L`` as an fp32 device tensor ``[M, M]``."""

    def __init__(self, L=None, device="cuda", Ut=None):
        if Ut is None:
            _, U = graphs.fourier(L)
            Ut = np.ascontiguousarray(U.T).astype(np.float32)
        Ut = np.ascontiguousarray(Ut, dtype=np.float32)
        if Ut.ndim != 2 or Ut.shape[0] != Ut.shape[1]:
            raise ValueError("Ut must be [M, M]")
        self.M = int(Ut.shape[0])
        self.Ut = torch.from_numpy(Ut).to(device)

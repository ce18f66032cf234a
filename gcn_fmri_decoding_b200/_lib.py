"""ctypes binding of ``libgcnb200.so`` (the C ABI declared in ``include/gcnb200.h``).

There is no CPU fallback: if the shared library is missing the import of any
compute entry point raises, loudly.  The library is built in-tree by
``csrc/build.sh`` (``__graft_entry__.build()`` calls it).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GCNB_LIB_PATH: load another build of the same library (e.g. the -DGCNB_TRACE debug build of tools/build_trace.sh)
LIB_PATH = os.environ.get("GCNB_LIB_PATH") or os.path.join(_HERE, "libgcnb200.so")

GCNB_OK = 0
BIAS_NONE, BIAS_PER_FILTER, BIAS_PER_VERTEX = 0, 1, 2
ALGO_AUTO, ALGO_GENERAL, ALGO_FUSED = 0, 1, 2
EPI_NONE, EPI_RELU_DROPOUT, EPI_MASK = 0, 1, 2


class GcnbCsr(C.Structure):
    """``struct gcnb_csr`` -- device pointers of a rescaled Laplacian in CSR."""

    _fields_ = [("rowptr", C.c_void_p), ("col", C.c_void_p), ("val", C.c_void_p), ("M", C.c_int32), ("nnz", C.c_int32),
                ("image", C.c_void_p), ("image_bytes", C.c_size_t)]


class GcnbAdjLevel(C.Structure):
    """``struct gcnb_adj_level`` -- one coarsening level of ``gcnb_adjacency_grad_f32`` (device pointers)."""

    _fields_ = [("dval", C.c_void_p), ("rowptr", C.c_void_p), ("val", C.c_void_p), ("rowptr_t", C.c_void_p),
                ("tpos", C.c_void_p), ("ss", C.c_void_p), ("hinv", C.c_void_p), ("parent", C.c_void_p),
                ("M", C.c_int32), ("nnz", C.c_int32)]


_i, _p, _z = C.c_int, C.c_void_p, C.c_size_t
_CSRP = C.POINTER(GcnbCsr)
_ADJP = C.POINTER(GcnbAdjLevel)

# name -> (restype, argtypes); must list every symbol include/gcnb200.h declares
SIGNATURES = {
    "gcnb_version": (_i, []),
    "gcnb_last_error_string": (C.c_char_p, []),
    "gcnb_launch_count": (C.c_ulonglong, []),
    "gcnb_cheb_fused_supported": (_i, [_i] * 9),
    "gcnb_cheb_workspace_bytes": (_z, [_i] * 10),
    "gcnb_cheb_describe": (_i, [_i] * 11 + [C.c_char_p, _z, C.POINTER(_z)]),
    "gcnb_cheb_stack_width": (_i, [_i] * 7),
    "gcnb_cheb_image_bytes": (_z, [_p, _p] + [_i] * 8),
    "gcnb_cheb_image_build": (_i, [_p, _p, _p] + [_i] * 8 + [_p, _z]),
    "gcnb_cheb_stack_supported": (_i, [_CSRP, _i, _i, _i, _i]),
    "gcnb_cheb_stack_fwd_f32": (_i, [_p, _CSRP, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p]),
    "gcnb_cheb_tap_image_bytes": (_z, [_i, _i, _i]),
    "gcnb_cheb_tap_image_build": (_i, [_p, _i, _i, _i, _p, _z]),
    "gcnb_cheb_fwd_f32": (_i, [_p, _p, _i, _CSRP, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _z, _p]),
    "gcnb_cheb_bwd_f32": (_i, [_p, _p, _i, _p, _p, _p, _i, _p, _CSRP, _CSRP, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _z, _p]),
    "gcnb_cheb_dx_describe": (_i, [_i] * 8 + [C.c_char_p, _z, C.POINTER(_z)]),
    "gcnb_cheb_dx_f32": (_i, [_p, _p, _i, _p, _p, _p, _i, _CSRP, _CSRP, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _z, _p]),
    "gcnb_cheb_dL_describe": (_i, [_i] * 7 + [C.c_char_p, _z, C.POINTER(_z)]),
    "gcnb_cheb_dL_f32": (_i, [_p, _p, _i, _p, _p, _p, _i, _CSRP, _CSRP, _p, _p, _p, _i, _p, _i, _i, _i, _i, _i, _i, _p,
                              _z, _p]),
    "gcnb_adjacency_grad_workspace_bytes": (_z, [_ADJP, _i, _i]),
    "gcnb_adjacency_grad_f32": (_i, [_ADJP, _i, _p, _i, _p, _i, _i, _p, _z, _p]),
    "gcnb_spectral_workspace_bytes": (_z, [_i] * 6),
    "gcnb_spectral_fwd_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _z, _p]),
    "gcnb_spectral_bwd_f32": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _z, _p]),
    "gcnb_brelu_fwd_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "gcnb_brelu_bwd_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _z, _p]),
    "gcnb_mpool_fwd_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "gcnb_mpool_bwd_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "gcnb_perm_gather_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "gcnb_mean_f_fwd_f32": (_i, [_p, _p, _i, _i, _p]),
    "gcnb_mean_f_bwd_f32": (_i, [_p, _p, _i, _i, _p]),
    "gcnb_softmax_xent_f32": (_i, [_p, _p, _p, _p, _p, _i, _i, _p, C.c_float, C.c_float, C.c_float, _p]),
    "gcnb_head_step_workspace_bytes": (_z, [_i] * 5),
    "gcnb_head_step_f32": (_i, [_p] * 17 + [_i] * 5 + [C.c_float, C.c_uint, C.c_uint, _p, C.c_float, C.c_float, C.c_float,
                                 _i, _p, _z, _p]),
    "gcnb_relu_dropout_fwd_f32": (_i, [_p, C.c_longlong, _i, _i, C.c_float, C.c_uint, _p, _p]),
    "gcnb_relu_dropout_bwd_f32": (_i, [_p, _p, C.c_longlong, _i, _i, _i, C.c_float, _p]),
    "gcnb_colsum_multi_f32": (_i, [_p, _p, _p, _p, _i, _p]),
    "gcnb_group_colsum_f32": (_i, [_p, _i, _i, _p, _i, _i, _p, _p]),
    "gcnb_gemm_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "gcnb_gemm_epilogue_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, C.c_float, C.c_uint, _p,
                                    _p]),
    "gcnb_adam_allreduce_flag_bytes": (_z, []),
    "gcnb_adam_tf_allreduce_f32": (_i, [_p, _p, _p, _p, _p, C.c_longlong, C.c_float, C.c_float, C.c_float, C.c_float,
                                        _p, _p, _i, _i, _p]),
    "gcnb_nadam_tf_allreduce_f32": (_i, [_p, _p, _p, _p, _p, C.c_longlong, C.c_float, C.c_float, C.c_float, C.c_float,
                                         _p, _p, _i, _i, _p]),
    "gcnb_adam_tf_f32": (_i, [_p, _p, _p, _p, _p, _p, C.c_longlong, C.c_float, C.c_float, C.c_float, C.c_float,
                              C.c_float, C.c_float, _i, _p]),
    "gcnb_nadam_tf_f32": (_i, [_p, _p, _p, _p, _p, _p, C.c_longlong, C.c_float, C.c_float, C.c_float, C.c_float,
                               C.c_float, _i, _p]),
}

_lib = None


class GcnbError(RuntimeError):
    pass


def lib():
    """The loaded library (loads on first use; raises if it was never built)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise GcnbError(
                "libgcnb200.so not found at %s -- build it with gcn_fmri_decoding_b200/csrc/build.sh "
                "(or python -c 'import __graft_entry__ as g; g.build()'); there is no CPU fallback" % LIB_PATH
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def describe(B, M, nnz, Fin, Fout, K, p, backward=False, need_dx=False, saved_basis=False, algo=ALGO_AUTO):
    """The route a Chebyshev layer call takes, as ``("<route>: <its kernels>", workspace bytes of that route)``."""
    buf, nbytes = C.create_string_buffer(512), _z()
    check(lib().gcnb_cheb_describe(B, M, nnz, Fin, Fout, K, p, int(backward), int(need_dx), int(saved_basis), algo, buf,
                                   512, C.byref(nbytes)), "gcnb_cheb_describe")
    return buf.value.decode(), nbytes.value


def describe_dx(B, M, nnz, Fin, Fout, K, p, algo=ALGO_AUTO):
    """The route of the input-gradient-only call ``gcnb_cheb_dx_f32``, as ``("<route>: <its kernels>", workspace bytes)``."""
    buf, nbytes = C.create_string_buffer(512), _z()
    check(lib().gcnb_cheb_dx_describe(B, M, nnz, Fin, Fout, K, p, algo, buf, 512, C.byref(nbytes)), "gcnb_cheb_dx_describe")
    return buf.value.decode(), nbytes.value


def describe_dL(B, M, nnz, Fin, Fout, K, p):
    """The kernels of the operator-gradient call ``gcnb_cheb_dL_f32`` and the workspace it takes, as a pair."""
    buf, nbytes = C.create_string_buffer(512), _z()
    check(lib().gcnb_cheb_dL_describe(B, M, nnz, Fin, Fout, K, p, buf, 512, C.byref(nbytes)), "gcnb_cheb_dL_describe")
    return buf.value.decode(), nbytes.value


def describe_fwd(B, M, nnz, Fin, Fout, K, p):
    """Which forward kernel AUTO dispatch picks for this layer shape, and its tile geometry."""
    return describe(B, M, nnz, Fin, Fout, K, p)[0]


def last_error():
    return lib().gcnb_last_error_string().decode("utf-8", "replace")


def check(rc, what):
    """Translate a return code: argument/workspace problems -> ValueError, CUDA failures -> RuntimeError."""
    if rc == GCNB_OK:
        return
    msg = "%s failed (%d): %s" % (what, rc, last_error())
    if rc in (-1, -2):
        raise ValueError(msg)
    raise GcnbError(msg)

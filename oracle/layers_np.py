"""CPU oracle of the graph-convolution hot path -- TEST INFRASTRUCTURE, NOT PRODUCT.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this package; nothing under
``gcn_fmri_decoding_b200/`` does.

What it is: a NumPy/SciPy restatement, op for op, of the reference's
TensorFlow-1.x layer code in ``/root/reference/lib_new/models_gcn.py`` and of
the host recursion in ``/root/reference/lib_new/graph.py``.  Every function
cites the lines it follows.  The arithmetic of the reference executes inside
TensorFlow 1.x (un-vendored, un-pinned, not installable here: Python 3.12, no
wheel), so:

    PARITY UNPINNED at the TF boundary -- no reference test or golden vector
    pins the TF-executed results (SURVEY.md section 8c).

What narrows that gap: the reference's own layer code (``cgcnn.__init__``,
``chebyshev5/2``, ``fourier``, ``b1relu/b2relu``, ``mpool1``, ``fc``,
``_inference``, ``loss``) is compiled from ``models_gcn.py`` with ``tf`` bound to
a NumPy stand-in for the ~25 ops it calls (``oracle/tf_shim.py``) and compared
with this module bit for bit (``tests/test_reference_on_shim.py``, build
container only) -- so the TRANSCRIPTION (op order, transposes, reshapes, weight
row order, variable names, L2 list) is pinned to the reference source, and the
backward functions below agree with torch.autograd run over that same source
(torch-backed stand-in); only TensorFlow's implementation of those ops is not.

What *is* pinned: (i) the Chebyshev recursion against the reference's own
NumPy implementation ``graph.chebyshev`` (``graph.py:155-172``, literally the
body of ``chebyshev2``) executed in the build container, (ii) ``rescale_L`` /
``laplacian`` / ``fourier`` / ``coarsen`` / ``perm_data_3d`` against the
reference functions executed in the build container, (iii) ``compute_perm``
against the reference's known-answer vector (``coarsening.py:217-218``).  The
outputs of those runs are committed under ``tests/golden/`` by
``oracle/make_golden.py``.

All functions take ``dtype``: ``np.float32`` reproduces the reference "as run"
(fp32 SpMM, fp32 sgemm), ``np.float64`` is the truth the CUDA path is measured
against (tolerance in the tests).
"""
from __future__ import annotations

import numpy as np
import scipy.sparse


# ----------------------------------------------------------------------------- graph operators
def rescale_L(L, lmax=2):
    """graph.py:146-152 -- ``L/(lmax/2) - I`` (on a copy; the reference mutates a shallow copy)."""
    L = scipy.sparse.csr_matrix(L, copy=True)
    M, M = L.shape
    I = scipy.sparse.identity(M, format="csr", dtype=L.dtype)
    L /= lmax / 2
    L -= I
    return L


def chebyshev_basis(L, X, K):
    """graph.py:155-172 -- ``Xt[k] = T_k(L) X`` for ``X [M, N]``; returns ``[K, M, N]``."""
    M, N = X.shape
    assert L.dtype == X.dtype
    Xt = np.empty((K, M, N), L.dtype)
    Xt[0, ...] = X
    if K > 1:
        Xt[1, ...] = L.dot(X)
    for k in range(2, K):
        Xt[k, ...] = 2 * L.dot(Xt[k - 1, ...]) - Xt[k - 2, ...]
    return Xt


def _rescaled(L, dtype):
    """models_gcn.py:590-596 -- csr copy, rescale with lmax=2, row-major sorted entries."""
    Lt = rescale_L(scipy.sparse.csr_matrix(L), lmax=2)
    Lt = scipy.sparse.csr_matrix(Lt, dtype=dtype)
    Lt.sort_indices()
    return Lt


# ----------------------------------------------------------------------------- filters (forward)
def chebyshev_stack(x, L, K, dtype=np.float32):
    """models_gcn.py:598-613 -- the ``[N*M, Fin*K]`` matrix fed to the dense filter.

    ``x [N, M, Fin]`` -> transpose ``[1,2,0]`` -> ``[M, Fin*N]`` -> recursion with
    ``sparse_tensor_dense_matmul`` -> ``[K, M, Fin, N]`` -> transpose ``[3,1,2,0]`` ->
    ``[N*M, Fin*K]`` (column ``f*K + k``).
    """
    x = np.asarray(x, dtype)
    N, M, Fin = x.shape
    Lt = _rescaled(L, dtype)
    x0 = np.transpose(x, (1, 2, 0)).reshape(M, Fin * N)
    xs = [x0]
    if K > 1:
        x1 = Lt.dot(x0)
        xs.append(x1)
    for _ in range(2, K):
        x2 = 2 * Lt.dot(x1) - x0
        xs.append(x2)
        x0, x1 = x1, x2
    xs = np.stack(xs, 0).reshape(K, M, Fin, N)
    xs = np.transpose(xs, (3, 1, 2, 0))
    return np.ascontiguousarray(xs).reshape(N * M, Fin * K)


def chebyshev5(x, L, W, K, dtype=np.float32):
    """models_gcn.py:587-617 -- ``y [N, M, Fout]`` with ``W [Fin*K, Fout]``."""
    N, M, Fin = x.shape
    W = np.asarray(W, dtype)
    assert W.shape[0] == Fin * K
    X = chebyshev_stack(x, L, K, dtype)
    return (X @ W).reshape(N, M, W.shape[1])


def chebyshev2(x, L, W, K, dtype=np.float32):
    """models_gcn.py:558-585 -- same filter with the recursion done by ``graph.chebyshev`` on the host."""
    x = np.asarray(x, dtype)
    N, M, Fin = x.shape
    W = np.asarray(W, dtype)
    Lt = _rescaled(L, dtype)
    x0 = np.transpose(x, (1, 2, 0)).reshape(M, Fin * N)
    xt = chebyshev_basis(Lt, np.ascontiguousarray(x0), K)
    xt = xt.reshape(K, M, Fin, N)
    xt = np.transpose(xt, (3, 1, 2, 0)).reshape(N * M, Fin * K)
    return (xt @ W).reshape(N, M, W.shape[1])


def fourier_basis(L, dtype=np.float32):
    """models_gcn.py:535-536 + graph.py:110-128 -- ``U^T`` of ``eigh(L.toarray())``, cast like ``tf.constant``."""
    _, U = np.linalg.eigh(L.toarray())
    return np.ascontiguousarray(U.T).astype(dtype)


def filter_in_fourier(x, Ut, W, dtype=np.float32):
    """models_gcn.py:512-528 with ``U := Ut`` (the reference passes ``U.T`` as ``U``).

    ``x [N,M,Fin]``, ``W [M,Fout,Fin]`` -> ``[N,M,Fout]``; ``tf.transpose(x)`` at ``:523`` reverses all axes.
    """
    x = np.asarray(x, dtype)
    W = np.asarray(W, dtype)
    Ut = np.asarray(Ut, dtype)
    N, M, Fin = x.shape
    Fout = W.shape[1]
    x = np.transpose(x, (1, 2, 0)).reshape(M, Fin * N)
    x = Ut @ x
    x = x.reshape(M, Fin, N)
    x = np.matmul(W, x)  # [M, Fout, N]
    x = np.transpose(x)  # [N, Fout, M]
    x = x.reshape(N * Fout, M)
    x = x @ Ut
    x = x.reshape(N, Fout, M)
    return np.ascontiguousarray(np.transpose(x, (0, 2, 1)))


def fourier(x, L, W, K=None, dtype=np.float32):
    """models_gcn.py:530-539 -- ``K`` is ignored by the reference (SURVEY D4)."""
    return filter_in_fourier(x, fourier_basis(L, dtype), W, dtype)


# ----------------------------------------------------------------------------- bias / relu / pooling
def b1relu(x, b):
    """models_gcn.py:619-623 -- ``relu(x + b)``, ``b [1,1,F]``."""
    b = np.asarray(b, x.dtype).reshape(1, 1, -1)
    return np.maximum(x + b, 0)


def b2relu(x, b):
    """models_gcn.py:625-629 -- ``relu(x + b)``, ``b [1,M,F]``."""
    b = np.asarray(b, x.dtype).reshape(1, x.shape[1], x.shape[2])
    return np.maximum(x + b, 0)


def mpool1(x, p, with_argmax=False):
    """models_gcn.py:631-639 -- ``tf.nn.max_pool(ksize=[1,p,1,1], strides=[1,p,1,1], 'SAME')`` over the vertex axis.

    Output length ``ceil(M/p)``; SAME padding (split ``pad//2`` before) never wins the max.
    ``argmax`` is the offset of the first maximum inside the (unpadded) window start
    ``j*p - pad_before``, uint8 -- the index ``MaxPoolGrad`` routes to.
    """
    if p <= 1:
        return (x, np.zeros(x.shape, np.uint8)) if with_argmax else x
    N, M, F = x.shape
    Mo = -(-M // p)
    pad = Mo * p - M
    before = pad // 2
    xp = np.full((N, Mo * p, F), -np.inf, x.dtype)
    xp[:, before : before + M, :] = x
    win = xp.reshape(N, Mo, p, F)
    y = win.max(axis=2)
    if not with_argmax:
        return y
    return y, win.argmax(axis=2).astype(np.uint8)  # np.argmax returns the first maximum


# ----------------------------------------------------------------------------- conv stack + head
def conv_stack(x, Ls, params, filter="chebyshev5", brelu="b1relu", pool="mpool1", dtype=np.float32,
               keep=False):
    """models_gcn.py:658-668 -- ``filter -> brelu -> pool`` per layer.

    ``Ls[i]`` is the Laplacian layer ``i`` uses (already selected as ``cgcnn.__init__:462-469`` does);
    ``params[i] = dict(W=..., b=..., K=..., p=...)``.  With ``keep`` returns the per-layer intermediates too.
    """
    x = np.asarray(x, dtype)
    trace = []
    for L, pr in zip(Ls, params):
        if filter == "chebyshev5":
            z = chebyshev5(x, L, pr["W"], pr["K"], dtype)
        elif filter == "chebyshev2":
            z = chebyshev2(x, L, pr["W"], pr["K"], dtype)
        elif filter == "fourier":
            z = fourier(x, L, pr["W"], pr["K"], dtype)
        else:
            raise ValueError(filter)
        a = b1relu(z, pr["b"]) if brelu == "b1relu" else b2relu(z, pr["b"])
        y, am = mpool1(a, pr["p"], with_argmax=True)
        trace.append(dict(x=x, z=z, a=a, y=y, argmax=am))
        x = y
    return (x, trace) if keep else x


def select_laplacians(L, p):
    """models_gcn.py:462-469 -- layer ``i`` uses ``L[sum_{q<i} log2 p_q]``."""
    out, j = [], 0
    for pp in p:
        out.append(L[j])
        j += int(np.log2(pp)) if pp > 1 else 0
    return out


def head(x, fcs, dtype=np.float32):
    """models_gcn.py:670-682 -- mean over F, FC+ReLU hidden layers (dropout keep-prob 1), linear logits.

    ``fcs = [(W, b), ...]``; the last pair is the logits layer (no ReLU).
    """
    x = np.asarray(x, dtype).mean(axis=-1, dtype=dtype)
    for i, (W, b) in enumerate(fcs):
        x = x @ np.asarray(W, dtype) + np.asarray(b, dtype)
        if i < len(fcs) - 1:
            x = np.maximum(x, 0)
    return x


def loss(logits, labels, regularized, regularization):
    """models_gcn.py:253-262 -- mean sparse-softmax CE + ``regularization * sum(l2_loss(v))``, ``l2_loss = sum(v^2)/2``."""
    z = logits - logits.max(axis=1, keepdims=True)
    logp = z - np.log(np.exp(z).sum(axis=1, keepdims=True))
    ce = -logp[np.arange(len(labels)), labels].mean()
    reg = sum(0.5 * float((np.asarray(v, np.float64) ** 2).sum()) for v in regularized)
    return ce + regularization * reg


# ----------------------------------------------------------------------------- backward (what tf.gradients computes, SURVEY A.2)
def mpool1_bwd(dy, argmax, p, M):
    """MaxPoolGrad: route ``dy [N, ceil(M/p), F]`` to the first maximum of each window."""
    if p <= 1:
        return dy
    N, Mo, F = dy.shape
    pad = Mo * p - M
    before = pad // 2
    d = np.zeros((N, Mo, p, F), dy.dtype)
    n, j, f = np.meshgrid(np.arange(N), np.arange(Mo), np.arange(F), indexing="ij")
    d[n, j, argmax, f] = dy
    return d.reshape(N, Mo * p, F)[:, before : before + M, :]


def brelu_bwd(da, a, per_vertex):
    """ReluGrad ``dz = da * [a > 0]`` and the bias gradient (sum over N, and over M for b1relu)."""
    dz = da * (a > 0)
    db = dz.sum(axis=0) if per_vertex else dz.sum(axis=(0, 1))
    return dz, db


def chebyshev5_bwd(x, L, W, K, dz, dtype=np.float32, need_dx=True):
    """Gradient of ``chebyshev5`` w.r.t. ``W`` and ``x`` (adjoint of models_gcn.py:598-617).

    ``dW = X^T dZ`` with ``X`` the ``[N*M, Fin*K]`` stack; ``dx`` through the transposed recursion
    ``g_{k-1} += 2 L~^T g_k``, ``g_{k-2} -= g_k``, ``g_0 += L~^T g_1``.
    """
    x = np.asarray(x, dtype)
    W = np.asarray(W, dtype)
    dz = np.asarray(dz, dtype)
    N, M, Fin = x.shape
    Fout = W.shape[1]
    X = chebyshev_stack(x, L, K, dtype)
    dZ = dz.reshape(N * M, Fout)
    dW = X.T @ dZ
    if not need_dx:
        return None, dW
    dX = dZ @ W.T  # [N*M, Fin*K]
    g = np.transpose(dX.reshape(N, M, Fin, K), (3, 1, 2, 0)).reshape(K, M, Fin * N).copy()
    LtT = scipy.sparse.csr_matrix(_rescaled(L, dtype).T)
    for k in range(K - 1, 1, -1):
        g[k - 1] += 2 * LtT.dot(g[k])
        g[k - 2] -= g[k]
    if K > 1:
        g[0] += LtT.dot(g[1])
    dx = np.transpose(g[0].reshape(M, Fin, N), (2, 0, 1))
    return np.ascontiguousarray(dx), dW


def fourier_bwd(x, Ut, W, dz, dtype=np.float32):
    """Gradient of ``filter_in_fourier``: ``dyh = U^T dz``, ``dW[m] = dyh[m] xh[m]^T``, ``dx = U (W[m]^T dyh[m])``."""
    x = np.asarray(x, dtype)
    W = np.asarray(W, dtype)
    Ut = np.asarray(Ut, dtype)
    dz = np.asarray(dz, dtype)
    xh = np.einsum("mn,bnf->bmf", Ut, x)
    dyh = np.einsum("mn,bno->bmo", Ut, dz)
    dW = np.einsum("bmo,bmf->mof", dyh, xh)
    dxh = np.einsum("mof,bmo->bmf", W, dyh)
    dx = np.einsum("mn,bmf->bnf", Ut, dxh)
    return dx, dW


def conv_stack_bwd(trace, Ls, params, dy, filter="chebyshev5", brelu="b1relu", dtype=np.float32,
                   first_needs_dx=False, decisions=None):
    """Back-propagate ``dy`` through the layers recorded by ``conv_stack(..., keep=True)``.

    ``decisions`` (optional, one ``dict(argmax=uint8, relu=bool)`` per layer, both at pooled resolution
    ``[N, ceil(M/p), F]``) routes the gradient the way another implementation decided: ``argmax`` replaces the
    first-maximum bytes of the trace and ``relu`` (that implementation's ``y > 0``) replaces the ReLU mask.  Where a
    window maximum or a pre-activation sits within rounding of a tie, an fp32 run may decide the other way and move a
    whole gradient element; conditioning on its decisions keeps the comparison about the arithmetic.  Passing the
    trace's own decisions gives bit for bit what passing none gives.

    Returns ``(dx_or_None, [dict(dW, db), ...])``.
    """
    grads = [None] * len(params)
    for i in range(len(params) - 1, -1, -1):
        t, pr, L = trace[i], params[i], Ls[i]
        M = t["a"].shape[1]
        am, live = t["argmax"], t["a"]
        if decisions is not None:
            am = np.asarray(decisions[i]["argmax"], np.uint8).reshape(t["argmax"].shape)
            # the routed element of a window is live iff the pooled value is: (a > 0) at the arg-max is (y > 0)
            live = mpool1_bwd(np.asarray(decisions[i]["relu"], dtype).reshape(t["y"].shape), am, pr["p"], M)
        da = mpool1_bwd(np.asarray(dy, dtype), am, pr["p"], M)
        dz, db = brelu_bwd(da, live, per_vertex=(brelu == "b2relu"))
        need_dx = i > 0 or first_needs_dx
        if filter == "fourier":
            dx, dW = fourier_bwd(t["x"], fourier_basis(L, dtype), pr["W"], dz, dtype)
        else:
            dx, dW = chebyshev5_bwd(t["x"], L, pr["W"], pr["K"], dz, dtype, need_dx=need_dx)
        grads[i] = dict(dW=dW, db=db)
        dy = dx
    return dy, grads


# ----------------------------------------------------------------------------- whole training step (CPU baseline)
def counter_dropout_mask(rows, cols, keep, seed, step):
    """The 0/1 mask the CUDA path draws for a ``[rows, cols]`` activation (``dropout_keeps`` in ``csrc/common.cuh``:
    murmur3-finaliser hash of the element index, keyed by a layer seed and the optimiser step count).  Exists so that the
    oracle can be run with the SAME mask as the device when ``tf.nn.dropout`` (models_gcn.py:677) is active."""
    def mix32(x):
        x = np.asarray(x, np.uint64) & 0xFFFFFFFF
        x ^= x >> 16
        x = (x * 0x85EBCA6B) & 0xFFFFFFFF
        x ^= x >> 13
        x = (x * 0xC2B2AE35) & 0xFFFFFFFF
        x ^= x >> 16
        return x

    if keep >= 1.0:
        return np.ones((rows, cols), np.float64)
    key = mix32(np.uint64(seed) ^ mix32((np.uint64(int(step)) + 0x9E3779B9) & 0xFFFFFFFF))
    thresh = np.uint64(int(np.float32(keep) * 4294967296.0))
    idx = np.arange(rows * cols, dtype=np.uint64)
    h = mix32((idx * 0x9E3779B1 + key) & 0xFFFFFFFF)
    return (h < thresh).astype(np.float64).reshape(rows, cols)


def network_step(x, labels, Ls, params, fcs, regularization, filter="chebyshev5", brelu="b1relu", dtype=np.float32,
                 dropout_masks=None, keep=1.0, conv_decisions=None):
    """Forward + loss + backward of the whole network (conv stack, mean over F, FC head, CE + L2).

    What one ``sess.run([op_train, ...])`` computes up to the optimiser update (models_gcn.py:146, :298-303).
    ``dropout_masks`` (one 0/1 array per hidden FC layer) with keep-probability ``keep`` reproduces ``tf.nn.dropout``
    (models_gcn.py:677: kept activations scaled by 1/keep) for a GIVEN mask.  ``conv_decisions`` routes the conv
    backward through given pooling / ReLU decisions (``conv_stack_bwd(decisions=...)``).
    Returns ``(loss, conv_grads, fc_grads)``.  Used as the CPU baseline and by the gradient parity test.
    """
    h, trace = conv_stack(x, Ls, params, filter=filter, brelu=brelu, dtype=dtype, keep=True)
    F_last = h.shape[-1]
    acts = [h.mean(axis=-1, dtype=dtype)]
    for i, (W, b) in enumerate(fcs):
        z = acts[-1] @ np.asarray(W, dtype) + np.asarray(b, dtype)
        if i < len(fcs) - 1:
            z = np.maximum(z, 0)
            if dropout_masks is not None:
                z = (z * np.asarray(dropout_masks[i], dtype) / dtype(keep)).astype(dtype)
        acts.append(z)
    logits = acts[-1]
    regs = [np.asarray(p["W"]) for p in params if filter != "chebyshev2"] + [v for Wb in fcs for v in Wb]
    value = loss(logits.astype(np.float64), labels, regs, regularization)
    B = x.shape[0]
    pz = np.exp(logits - logits.max(axis=1, keepdims=True))
    pz /= pz.sum(axis=1, keepdims=True)
    pz[np.arange(B), labels] -= 1
    d = (pz / B).astype(dtype)
    fc_grads = [None] * len(fcs)
    for i in range(len(fcs) - 1, -1, -1):
        W, b = fcs[i]
        if i < len(fcs) - 1:
            d = d * (acts[i + 1] > 0)
            if dropout_masks is not None:
                d = (d / dtype(keep)).astype(dtype)  # acts > 0 already implies "kept"
        fc_grads[i] = (acts[i].T @ d + regularization * np.asarray(W, dtype), d.sum(0) + regularization * np.asarray(b, dtype))
        d = d @ np.asarray(W, dtype).T
    dh = np.repeat(d[:, :, None], F_last, axis=2) / dtype(F_last)
    _, conv_grads = conv_stack_bwd(trace, Ls, params, dh, filter=filter, brelu=brelu, dtype=dtype,
                                   decisions=conv_decisions)
    if filter != "chebyshev2":
        for g, p in zip(conv_grads, params):
            g["dW"] = g["dW"] + regularization * np.asarray(p["W"], dtype)
    return value, conv_grads, fc_grads

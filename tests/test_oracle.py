"""The oracle against the reference-generated golden vectors and against itself (CPU only)."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import GOLDEN, rel_inf
from oracle import layers_np as O
from oracle import ref_loader


def test_rescale_matches_reference_vectors(graph_l4):
    for L, Lt in zip(graph_l4["L"], graph_l4["Lt"]):
        mine = O.rescale_L(L, 2)
        mine.sort_indices()
        assert mine.dtype == Lt.dtype == np.float32
        assert np.array_equal(mine.indptr, Lt.indptr) and np.array_equal(mine.indices, Lt.indices)
        assert np.array_equal(mine.data, Lt.data)
        assert abs(mine.diagonal()).max() == 0  # lmax=2 => zero diagonal, SURVEY A.4


def test_chebyshev_recursion_matches_reference_graph_chebyshev(graph_l4):
    """graph.chebyshev (graph.py:155-172) ran in the build container; bit-exact restatement."""
    z = np.load(os.path.join(GOLDEN, "ref_chebyshev.npz"))
    for name in "abcde":
        lvl, K = (int(v) for v in z["meta_" + name])
        Xt = O.chebyshev_basis(graph_l4["Lt"][lvl], z["X_" + name], K)
        assert Xt.dtype == np.float32
        assert np.array_equal(Xt, z["Xt_" + name]), name


def test_chebyshev5_equals_chebyshev2_and_einsum(graph_l4):
    """The TF-op transcription (chebyshev5) and the py_func route (chebyshev2) are the same filter,
    and the W row order is f*K + k (SURVEY A.1)."""
    rng = np.random.RandomState(0)
    L = graph_l4["L"][2]
    x = rng.randn(3, 100, 6).astype(np.float32)
    W = rng.randn(6 * 4, 5).astype(np.float32)
    y5 = O.chebyshev5(x, L, W, 4, np.float64)
    y2 = O.chebyshev2(x, L, W, 4, np.float64)
    assert rel_inf(y5, y2) < 1e-13
    Lt = graph_l4["Lt"][2].astype(np.float64)
    T = [x.astype(np.float64)]
    T.append(np.einsum("mn,bnf->bmf", Lt.toarray(), T[0]))
    for _ in range(2, 4):
        T.append(2 * np.einsum("mn,bnf->bmf", Lt.toarray(), T[-1]) - T[-2])
    T = np.stack(T, -1)  # [B, M, Fin, K]
    ref = np.einsum("bmfk,fko->bmo", T, W.astype(np.float64).reshape(6, 4, 5))
    assert rel_inf(y5, ref) < 1e-13
    # K = 1 is a per-vertex dense layer: no neighbour mixing (SURVEY D1)
    W1 = rng.randn(6, 5).astype(np.float32)
    assert rel_inf(O.chebyshev5(x, L, W1, 1, np.float64), x.astype(np.float64) @ W1) < 1e-14


def test_fourier_is_U_W_Ut(graph_l4):
    rng = np.random.RandomState(1)
    L = graph_l4["L"][3]
    M = L.shape[0]
    x = rng.randn(2, M, 3)
    W = rng.randn(M, 4, 3)
    lamb, U = np.linalg.eigh(L.toarray().astype(np.float64))
    xh = np.einsum("nm,bnf->bmf", U, x)
    yh = np.einsum("mof,bmf->bmo", W, xh)
    ref = np.einsum("nm,bmo->bno", U, yh)
    got = O.filter_in_fourier(x, U.T, W, np.float64)
    assert rel_inf(got, ref) < 1e-12


def test_mpool_same_padding_and_first_max():
    x = np.array([[[1.0], [3.0], [3.0], [2.0], [5.0], [0.0]]])  # M = 6
    y, a = O.mpool1(x, 4, with_argmax=True)  # ceil(6/4)=2, pad 2 -> one before, one after
    assert y[0, :, 0].tolist() == [3.0, 5.0]
    assert a[0, :, 0].tolist() == [2, 1]  # window 0 = [pad, x0, x1, x2]: first max (x1) at offset 2
    y, a = O.mpool1(x, 2, with_argmax=True)
    assert y[0, :, 0].tolist() == [3.0, 3.0, 5.0] and a[0, :, 0].tolist() == [1, 0, 0]
    dy = np.ones((1, 3, 1))
    assert O.mpool1_bwd(dy, a, 2, 6)[0, :, 0].tolist() == [0, 1, 1, 0, 1, 0]
    assert O.mpool1(x, 1) is x


def test_backward_against_finite_differences(graph_l4):
    rng = np.random.RandomState(3)
    for filt, brelu, lvl, Fin, Fout, K, p in (("chebyshev5", "b1relu", 3, 3, 4, 4, 2),
                                               ("chebyshev5", "b2relu", 4, 2, 3, 3, 1),
                                               ("fourier", "b1relu", 4, 2, 3, 0, 1)):
        L = graph_l4["L"][lvl]
        M = L.shape[0]
        x = rng.randn(2, M, Fin)
        W = rng.randn(M, Fout, Fin) if filt == "fourier" else rng.randn(Fin * K, Fout)
        b = rng.randn(M, Fout) if brelu == "b2relu" else rng.randn(Fout)
        dy = rng.randn(2, M // p, Fout)
        pr = [dict(W=W, b=b, K=K, p=p)]

        def f(x_, W_, b_):
            y = O.conv_stack(x_, [L], [dict(W=W_, b=b_, K=K, p=p)], filter=filt, brelu=brelu, dtype=np.float64)
            return float((y * dy).sum())

        _, tr = O.conv_stack(x, [L], pr, filter=filt, brelu=brelu, dtype=np.float64, keep=True)
        dx, g = O.conv_stack_bwd(tr, [L], pr, dy, filter=filt, brelu=brelu, dtype=np.float64, first_needs_dx=True)
        eps = 1e-6
        for arr, grad, which in ((x, dx, 0), (W, g[0]["dW"], 1), (b, g[0]["db"], 2)):
            for _ in range(6):
                idx = tuple(rng.randint(0, s) for s in arr.shape)
                hi, lo = arr.copy(), arr.copy()
                hi[idx] += eps
                lo[idx] -= eps
                args_hi = [x, W, b]
                args_lo = [x, W, b]
                args_hi[which], args_lo[which] = hi, lo
                num = (f(*args_hi) - f(*args_lo)) / (2 * eps)
                assert abs(num - grad[idx]) < 1e-5 * max(1.0, abs(num)), (filt, which, idx)


def test_layer_cases_reproduce(graph_l4, layer_cases):
    """The committed oracle vectors are reproduced by the oracle as it stands."""
    for name, c in layer_cases.items():
        lvl, B, Fin, Fout, K, p = (int(v) for v in c["meta"])
        filt, brelu = str(c["kind"]).split("/")
        L = graph_l4["L"][lvl]
        pr = [dict(W=c["W"], b=c["b"], K=K, p=p)]
        y, tr = O.conv_stack(c["x"], [L], pr, filter=filt, brelu=brelu, dtype=np.float64, keep=True)
        if filt == "fourier":
            # eigenvectors of a degenerate spectrum are host-BLAS dependent: rebuild with the stored basis
            z = O.filter_in_fourier(c["x"], c["Ut"], c["W"], np.float64)
            a = O.b1relu(z, c["b"]) if brelu == "b1relu" else O.b2relu(z, c["b"])
            y, am = O.mpool1(a, p, with_argmax=True)
            assert rel_inf(y, c["y64"]) < 1e-5, name
            continue
        assert rel_inf(y, c["y64"]) < 1e-12, name
        assert np.array_equal(tr[0]["argmax"], c["argmax"]), name
        # as-run fp32 oracle vs fp64 truth: the noise floor the 1e-4 bar sits above
        assert rel_inf(c["y32"], c["y64"]) < 2e-5, name


def test_select_laplacians_and_head():
    assert O.select_laplacians(list("abcde"), [4, 4]) == ["a", "c"]
    assert O.select_laplacians(list("ab"), [1, 1, 1, 1, 1, 1]) == ["a"] * 6
    assert O.select_laplacians(list("abcdefg"), [1, 4, 1, 4, 1, 4]) == ["a", "a", "c", "c", "e", "e"]
    rng = np.random.RandomState(5)
    x = rng.randn(4, 25, 32)
    fcs = [(rng.randn(25, 8), rng.randn(8)), (rng.randn(8, 22), rng.randn(22))]
    out = O.head(x, fcs, np.float64)
    assert out.shape == (4, 22)
    ref = np.maximum(x.mean(-1) @ fcs[0][0] + fcs[0][1], 0) @ fcs[1][0] + fcs[1][1]
    assert rel_inf(out, ref) < 1e-14
    lab = np.array([0, 5, 20, 3])
    l = O.loss(out, lab, [fcs[0][0]], 5e-4)
    p = np.exp(out - out.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    assert abs(l - (-np.log(p[np.arange(4), lab]).mean() + 5e-4 * 0.5 * (fcs[0][0] ** 2).sum())) < 1e-12


@pytest.mark.skipif(not ref_loader.available(), reason="reference sources only exist in the build container")
def test_oracle_against_live_reference(graph_l4):
    """Container-only: the reference's functions executed now agree with the oracle bit for bit."""
    graph, coarsening = ref_loader.load()
    rng = np.random.RandomState(21)
    for lvl, K in ((0, 5), (2, 8), (4, 3)):
        L = graph_l4["L"][lvl]
        Lt_ref = graph.rescale_L(sp.csr_matrix(L, copy=True), lmax=2)
        X = rng.randn(L.shape[0], 9).astype(np.float32)
        assert np.array_equal(graph.chebyshev(Lt_ref, X, K), O.chebyshev_basis(O.rescale_L(L), X, K))


# --------------------------------------------------------------------------------------------------------------------
# A second, independent transcription of the TF graph -- the reference's ops replaced one for one by their torch (CPU,
# fp64) counterparts IN THE REFERENCE'S ORDER (transpose -> reshape -> sparse matmul -> concat -> transpose -> matmul),
# differentiated by torch.autograd where the reference calls tf.gradients (models_gcn.py:298).  TF 1.x cannot run here,
# so this is the closest stand-in for "the graph as executed": the NumPy oracle's hand-written forward AND backward must
# agree with an autograd engine that never saw the oracle's formulas.
def _torch_network(x, labels, Ls, params, fcs, regularization, filt, brelu, masks=None, keep=1.0):
    import torch
    import torch.nn.functional as TF

    t = lambda a: torch.tensor(np.asarray(a, np.float64), requires_grad=True)  # noqa: E731
    x = torch.tensor(np.asarray(x, np.float64))
    leaves = dict(W=[t(p["W"]) for p in params], b=[t(p["b"]) for p in params], fcW=[t(W) for W, _ in fcs],
                  fcb=[t(b) for _, b in fcs])
    for i, (L, pr) in enumerate(zip(Ls, params)):
        N, M, Fin = x.shape
        K, p, W, b = pr["K"], pr["p"], leaves["W"][i], leaves["b"][i]
        if filt == "fourier":  # models_gcn.py:512-539
            _, U = np.linalg.eigh(L.toarray())  # graph.fourier (graph.py:110-128), algo 'eigh', in L's own dtype
            U = torch.tensor(np.ascontiguousarray(U.T).astype(np.float64))
            xf = torch.matmul(U, x.permute(1, 2, 0).reshape(M, Fin * N)).reshape(M, Fin, N)
            xf = torch.matmul(W, xf)                                     # [M, Fout, Fin] x [M, Fin, N]
            xf = xf.permute(2, 1, 0).reshape(N * W.shape[1], M)
            z = torch.matmul(xf, U).reshape(N, W.shape[1], M).permute(0, 2, 1)
        else:  # models_gcn.py:587-617 (chebyshev5); chebyshev2 (:558-585) is the same arithmetic
            Lr = sp.csr_matrix(L, dtype=np.float64)
            Lr = (Lr / (2 / 2) - sp.identity(M, format="csr", dtype=np.float64)).tocoo()  # graph.rescale_L, lmax = 2
            Lt = torch.sparse_coo_tensor(np.vstack((Lr.row, Lr.col)), Lr.data, Lr.shape, check_invariants=True).coalesce()
            x0 = x.permute(1, 2, 0).reshape(M, Fin * N)
            xs = [x0]
            if K > 1:
                x1 = torch.sparse.mm(Lt, x0)
                xs.append(x1)
            for _ in range(2, K):
                x2 = 2 * torch.sparse.mm(Lt, x1) - x0
                xs.append(x2)
                x0, x1 = x1, x2
            xk = torch.stack(xs, 0).reshape(K, M, Fin, N).permute(3, 1, 2, 0).reshape(N * M, Fin * K)
            z = torch.matmul(xk, W).reshape(N, M, W.shape[1])
        a = torch.relu(z + (b.reshape(1, 1, -1) if brelu == "b1relu" else b.reshape(1, M, -1)))  # :619-629
        if p > 1:  # :631-639, SAME: ceil(M/p) windows, padding split pad//2 in front, never the maximum
            Mo = -(-M // p)
            pad = Mo * p - M
            a = TF.pad(a.permute(0, 2, 1), (pad // 2, pad - pad // 2), value=float("-inf"))
            a = TF.max_pool1d(a, p, p).permute(0, 2, 1)
        x = a
    h = x.mean(-1)  # :673
    for i in range(len(fcs)):
        h = torch.matmul(h, leaves["fcW"][i]) + leaves["fcb"][i]
        if i < len(fcs) - 1:
            h = torch.relu(h)
            if masks is not None:  # tf.nn.dropout(x, keep_prob): kept values scaled by 1/keep (:677)
                h = h * torch.tensor(masks[i]) / keep
    ce = TF.cross_entropy(h, torch.tensor(np.asarray(labels, np.int64)))  # :255-257
    regs = ([] if filt == "chebyshev2" else leaves["W"]) + leaves["fcW"] + leaves["fcb"]  # :253-262, _weight/_bias_variable
    loss = ce + regularization * sum((v ** 2).sum() / 2 for v in regs)
    flat = leaves["W"] + leaves["b"] + leaves["fcW"] + leaves["fcb"]
    grads = torch.autograd.grad(loss, flat)
    n, m = len(params), len(fcs)
    g = [v.numpy() for v in grads]
    return float(loss.detach()), h.detach().numpy(), g[:n], g[n:2 * n], g[2 * n:2 * n + m], g[2 * n + m:]


@pytest.mark.parametrize("filt,brelu,lvls,ps,K,keep", [("chebyshev5", "b1relu", (0, 2), (4, 4), 5, 0.5),   # config 2
                                                        ("chebyshev5", "b2relu", (3, 3), (1, 1), 3, 1.0),   # config 1 style
                                                        ("chebyshev2", "b1relu", (2, 3), (2, 4), 2, 1.0),   # config 3a
                                                        ("fourier", "b1relu", (3, 4), (2, 1), 0, 0.5)])     # config 3b
def test_network_step_against_torch_autograd_twin(graph_l4, filt, brelu, lvls, ps, K, keep):
    rng = np.random.RandomState(11)
    Ls = [graph_l4["L"][l] for l in lvls]
    B, Fs, widths = 5, (3, 6, 4), (7, 5, 4)
    params = []
    for i, L in enumerate(Ls):
        M, Fin, Fout = L.shape[0], Fs[i], Fs[i + 1]
        W = rng.randn(M, Fout, Fin) * 0.3 if filt == "fourier" else rng.randn(Fin * K, Fout) * 0.3
        b = rng.randn(M, Fout) * 0.1 if brelu == "b2relu" else rng.randn(Fout) * 0.1
        params.append(dict(W=W, b=b, K=K, p=ps[i]))
    x = rng.randn(B, Ls[0].shape[0], Fs[0])
    labels = rng.randint(0, widths[-1], B)
    M_last = -(-Ls[-1].shape[0] // ps[-1])  # SAME pooling: ceil (the chebyshev2 case pools 50 vertices by 4 -> 13)
    dims = (M_last,) + widths
    fcs = [(rng.randn(dims[i], dims[i + 1]) * 0.2, rng.randn(dims[i + 1]) * 0.1) for i in range(len(widths))]
    masks = None if keep == 1.0 else [(rng.rand(B, w) < keep).astype(np.float64) for w in widths[:-1]]
    val, cg, fg = O.network_step(x, labels, Ls, params, fcs, 5e-4, filter=filt, brelu=brelu, dtype=np.float64,
                                 dropout_masks=masks, keep=keep)
    tval, tlogits, tW, tb, tfW, tfb = _torch_network(x, labels, Ls, params, fcs, 5e-4, filt, brelu, masks, keep)
    assert abs(val - tval) <= 1e-12 * abs(tval)
    for i in range(len(Ls)):
        assert rel_inf(cg[i]["dW"], tW[i]) <= 1e-11, (i, "dW")
        assert rel_inf(np.asarray(cg[i]["db"]).reshape(tb[i].shape), tb[i]) <= 1e-11, (i, "db")
    for i in range(len(fcs)):
        assert rel_inf(fg[i][0], tfW[i]) <= 1e-11 and rel_inf(fg[i][1], tfb[i]) <= 1e-11, i
    # inference path of the oracle (conv_stack + head, no dropout) against the twin's logits
    if masks is None:
        logits = O.head(O.conv_stack(x, Ls, params, filter=filt, brelu=brelu, dtype=np.float64), fcs, np.float64)
        assert rel_inf(logits, tlogits) <= 1e-12


@pytest.mark.parametrize("M,p", [(10, 4), (7, 2), (9, 8), (16, 4), (5, 1)])
def test_mpool1_ragged_against_torch_same_padding(M, p):
    """SAME max-pooling of a ragged vertex axis and the MaxPoolGrad routing (oracle mpool1 / mpool1_bwd, models_gcn.py:
    631-639) against torch's max_pool1d + autograd over an explicit -inf padding; values are distinct, so no ties."""
    import torch
    import torch.nn.functional as TF

    rng = np.random.RandomState(M * 10 + p)
    x = rng.permutation(3 * M * 4).reshape(3, M, 4).astype(np.float64)
    y, am = O.mpool1(x, p, with_argmax=True)
    dy = rng.randn(*y.shape)
    dx = O.mpool1_bwd(dy, am, p, M) if p > 1 else dy
    xt = torch.tensor(x, requires_grad=True)
    if p > 1:
        Mo = -(-M // p)
        pad = Mo * p - M
        yt = TF.max_pool1d(TF.pad(xt.permute(0, 2, 1), (pad // 2, pad - pad // 2), value=float("-inf")), p, p).permute(0, 2, 1)
    else:
        yt = xt * 1
    (gx,) = torch.autograd.grad((yt * torch.tensor(dy)).sum(), xt)
    assert np.array_equal(y, yt.detach().numpy()) and np.array_equal(dx, gx.numpy())


def test_oracle_reproduces_the_vectors_of_the_reference_source(graph_l1, graph_l4):
    """tests/golden/ref_source_steps.npz was produced by the reference's OWN layer and loss source (models_gcn.py) run on
    the NumPy / torch stand-ins for ``tf`` in the build container (oracle/make_golden_ref_source.py; live version:
    tests/test_reference_on_shim.py).  The fixture carries that pin to machines without /root/reference: fp32 logits to
    fp32 rounding, fp64 loss to 1e-12 and every gradient ``tf.gradients`` would return to 1e-10."""
    import ast

    z = np.load(os.path.join(GOLDEN, "ref_source_steps.npz"))
    cases = sorted({k.split(".")[0] for k in z.files})
    assert cases == ["config1", "config2", "config3a"]
    for name in cases:
        filt, brelu, fixture, F, K, p, Mfc, keep = z[name + ".meta"]
        F, K, p, Mfc, keep = (ast.literal_eval(str(v)) for v in (F, K, p, Mfc, keep))
        L = (graph_l1 if "l1" in str(fixture) else graph_l4)["L"]
        Ls = O.select_laplacians(L, p)
        var = {k[len(name) + 5:].replace("__", "/"): z[k] for k in z.files if k.startswith(name + ".var.")}
        grad = {k[len(name) + 6:].replace("__", "/"): z[k] for k in z.files if k.startswith(name + ".grad.")}
        params = [dict(W=var["conv%d/weights" % (i + 1)], b=var["conv%d/bias" % (i + 1)].reshape(
            (-1, F[i]) if brelu == "b2relu" else (F[i],)), K=K[i], p=p[i]) for i in range(len(p))]
        fc_names = ["fc%d" % (i + 1) for i in range(len(Mfc) - 1)] + ["logits"]
        fcs = [(var[s + "/weights"], var[s + "/bias"]) for s in fc_names]
        x, labels = z[name + ".x"], z[name + ".labels"]
        logits = O.head(O.conv_stack(x, Ls, params, filter=str(filt), brelu=str(brelu), dtype=np.float32), fcs, np.float32)
        # bit for bit where it was generated (the live test asserts exactly that); another host's BLAS may sum the
        # fp32 GEMMs in another order, so the travelling check allows fp32 rounding
        assert rel_inf(logits, z[name + ".logits32"]) <= 2e-6, name
        masks = [z[name + ".mask%d" % i].astype(np.float64) for i in range(len(Mfc) - 1)] if keep < 1 else None
        L64 = [l.astype(np.float64) for l in Ls]
        val, cg, fg = O.network_step(x.astype(np.float64), labels, L64, params, fcs, 5e-4, filter=str(filt), brelu=str(brelu),
                                     dtype=np.float64, dropout_masks=masks, keep=keep)
        assert abs(val - float(z[name + ".loss64"])) <= 1e-12 * abs(val), name

        def close(a, b):
            return np.abs(np.asarray(a).reshape(b.shape) - b).max() <= 1e-10 * np.abs(b).max()

        for i, s in enumerate(fc_names):
            assert close(fg[i][0], grad[s + "/weights"]) and close(fg[i][1], grad[s + "/bias"]), (name, s)
        for i in range(len(p)):
            key = "conv%d/weights" % (i + 1)
            if key not in grad:                          # chebyshev2: no gradient below a py_func in the reference
                assert str(filt) == "chebyshev2" and i < len(p) - 1
                continue
            assert close(cg[i]["dW"], grad[key]) and close(cg[i]["db"], grad["conv%d/bias" % (i + 1)]), (name, i)


# --------------------------------------------------------------------------------------------------------------------
# Backward conditioned on given pooling / ReLU decisions (what the GPU tests use to compare with an fp32 run whose
# near-tie decisions went the other way).
def _own_decisions(trace):
    return [dict(argmax=t["argmax"], relu=t["y"] > 0) for t in trace]


@pytest.mark.parametrize("brelu,lvls,ps", [("b1relu", (0, 2), (4, 4)), ("b2relu", (3, 3), (1, 2)), ("b1relu", (2, 3), (2, 8))])
def test_backward_with_its_own_decisions_is_bit_identical(graph_l4, brelu, lvls, ps):
    """Passing the oracle's own arg-max bytes and ReLU mask changes nothing, bit for bit: conv_stack_bwd and
    network_step.  (lvl 3 pooled by 8: 50 vertices, a ragged SAME window.)"""
    rng = np.random.RandomState(17)
    Ls = [graph_l4["L"][l] for l in lvls]
    B, Fs, K = 6, (5, 8, 6), 3
    params = []
    for i, L in enumerate(Ls):
        M = L.shape[0]
        b = rng.randn(M, Fs[i + 1]) * 0.3 if brelu == "b2relu" else rng.randn(Fs[i + 1]) * 0.3
        params.append(dict(W=rng.randn(Fs[i] * K, Fs[i + 1]) * 0.3, b=b, K=K, p=ps[i]))
    x = rng.randn(B, Ls[0].shape[0], Fs[0])
    y, tr = O.conv_stack(x, Ls, params, brelu=brelu, dtype=np.float64, keep=True)
    assert 0.1 < np.mean([t["y"] > 0 for t in tr][-1]) < 0.9          # both branches of the ReLU are taken
    dy = rng.randn(*y.shape)
    dx0, g0 = O.conv_stack_bwd(tr, Ls, params, dy, brelu=brelu, dtype=np.float64, first_needs_dx=True)
    dx1, g1 = O.conv_stack_bwd(tr, Ls, params, dy, brelu=brelu, dtype=np.float64, first_needs_dx=True,
                               decisions=_own_decisions(tr))
    assert np.array_equal(dx0, dx1)
    for a, b in zip(g0, g1):
        assert np.array_equal(a["dW"], b["dW"]) and np.array_equal(a["db"], b["db"])
    labels = rng.randint(0, 4, B)
    M_last = y.shape[1]
    fcs = [(rng.randn(M_last, 7) * 0.2, rng.randn(7) * 0.1), (rng.randn(7, 4) * 0.2, rng.randn(4) * 0.1)]
    masks = [(rng.rand(B, 7) < 0.5).astype(np.float64)]
    r0 = O.network_step(x, labels, Ls, params, fcs, 5e-4, brelu=brelu, dtype=np.float64, dropout_masks=masks, keep=0.5)
    r1 = O.network_step(x, labels, Ls, params, fcs, 5e-4, brelu=brelu, dtype=np.float64, dropout_masks=masks, keep=0.5,
                        conv_decisions=_own_decisions(tr))
    assert r0[0] == r1[0]
    for a, b in zip(r0[1], r1[1]):
        assert np.array_equal(a["dW"], b["dW"]) and np.array_equal(a["db"], b["db"])
    for a, b in zip(r0[2], r1[2]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_flipped_argmax_byte_moves_exactly_that_gradient(graph_l4):
    """One arg-max byte sent to another vertex of its window moves that one dz element there: dW changes by
    dy * (X[new row] - X[old row]) in that one column, the per-vertex bias gradient moves between the two vertices,
    everything else stays put.  A dead ReLU decision removes the element instead."""
    rng = np.random.RandomState(23)
    L = graph_l4["L"][2]
    M, B, Fin, Fout, K, p = L.shape[0], 3, 4, 5, 3, 4
    pr = [dict(W=rng.randn(Fin * K, Fout) * 0.3, b=rng.randn(M, Fout) * 0.3, K=K, p=p)]
    x = rng.randn(B, M, Fin)
    y, tr = O.conv_stack(x, [L], pr, brelu="b2relu", dtype=np.float64, keep=True)
    dy = rng.randn(*y.shape)
    live = np.argwhere(tr[0]["y"] > 0)
    n, j, f = live[len(live) // 2]
    old = int(tr[0]["argmax"][n, j, f])
    new = (old + 1) % p
    dec = _own_decisions(tr)
    dec[0]["argmax"] = dec[0]["argmax"].copy()
    dec[0]["argmax"][n, j, f] = new
    _, g0 = O.conv_stack_bwd(tr, [L], pr, dy, brelu="b2relu", dtype=np.float64)
    _, g1 = O.conv_stack_bwd(tr, [L], pr, dy, brelu="b2relu", dtype=np.float64, decisions=dec)
    X = O.chebyshev_stack(x, L, K, np.float64).reshape(B, M, Fin * K)
    r_old, r_new = j * p + old, j * p + new
    expect = g0[0]["dW"].copy()
    expect[:, f] += dy[n, j, f] * (X[n, r_new] - X[n, r_old])
    assert np.allclose(g1[0]["dW"], expect, rtol=0, atol=1e-12 * np.abs(expect).max())
    assert not np.allclose(g1[0]["dW"][:, f], g0[0]["dW"][:, f], rtol=0, atol=1e-6 * np.abs(expect).max())
    ddb = g1[0]["db"] - g0[0]["db"]
    want = np.zeros_like(ddb)
    want[r_old, f], want[r_new, f] = -dy[n, j, f], dy[n, j, f]
    assert np.allclose(ddb, want, rtol=0, atol=1e-12)
    # the same element declared dead: its gradient disappears from the bias gradient of its vertex
    dec2 = _own_decisions(tr)
    dec2[0]["relu"] = dec2[0]["relu"].copy()
    dec2[0]["relu"][n, j, f] = False
    _, g2 = O.conv_stack_bwd(tr, [L], pr, dy, brelu="b2relu", dtype=np.float64, decisions=dec2)
    want = np.zeros_like(ddb)
    want[r_old, f] = -dy[n, j, f]
    assert np.allclose(g2[0]["db"] - g0[0]["db"], want, rtol=0, atol=1e-12)

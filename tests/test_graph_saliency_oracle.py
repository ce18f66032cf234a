"""Edge saliency maps without a GPU: the fp64 oracle of a ChebyNet layer's gradient w.r.t. the entries of its operator
(``chebyshev5_dL`` below) against central finite differences and torch autograd, the network-level graph gradient
(``network_graph_gradient``) against finite differences of the target logit, and the host-side mapping of the level-0
matrix to input-ROI order.  The GPU tests import the oracle from here."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import layers_np as O
from test_saliency_oracle import permute_rows


# ---- the fp64 oracle -----------------------------------------------------------------------------------------------
def chebyshev5_dL(x, L, W, K, dz, chunk=32):
    """Gradient of ``<dz, chebyshev5(x, L, W, K)>`` w.r.t. the entries of the rescaled operator ``L~ = L - I``, per
    window, in fp64: ``(dval [N, nnz], ddiag [N, M])``, ``dval`` in the CSR order of ``L~`` (``O._rescaled``: rows sorted
    by column) and ``ddiag`` the diagonal ``(i, i)`` whether or not ``L~`` stores it.  With the basis ``X_k`` and the
    Clenshaw states ``b_{K-1} = G_{K-1}``, ``b_k = G_k + 2 L~^T b_{k+1} - b_{k+2}`` of the seeds ``G_k = dz W_k^T``:
    ``dL~[i, j] = sum_f b_1[i, f] X_0[j, f] + sum_{k=2}^{K-1} 2 sum_f b_k[i, f] X_{k-1}[j, f]``.  ``L~ = L - I``, so these
    are also the gradients w.r.t. the entries of ``L``.  K = 1: zeros."""
    x = np.asarray(x, np.float64)
    dz = np.asarray(dz, np.float64)
    W = np.asarray(W, np.float64)
    N, M, Fin = x.shape
    Lt = O._rescaled(L, np.float64)
    rows = np.repeat(np.arange(M), np.diff(Lt.indptr))
    cols = Lt.indices
    LtT = sp.csr_matrix(Lt.T)
    dval = np.zeros((N, Lt.nnz))
    ddiag = np.zeros((N, M))
    if K == 1:
        return dval, ddiag
    apply = lambda A, Y: np.einsum("ij,njf->nif", A, Y) if not sp.issparse(A) else np.stack([A @ y for y in Y])
    for s in range(0, N, chunk):
        xs, dzs = x[s:s + chunk], dz[s:s + chunk]
        X = [xs, apply(Lt, xs)]
        for _ in range(2, K):
            X.append(2 * apply(Lt, X[-1]) - X[-2])
        G = [dzs @ W[k::K].T for k in range(K)]  # W row f*K + k is the tap of order k
        b = [None] * (K + 1)
        b[K - 1] = G[K - 1]
        for k in range(K - 2, 0, -1):
            b[k] = G[k] + 2 * apply(LtT, b[k + 1]) - (b[k + 2] if k + 2 <= K - 1 else 0)
        for k in range(1, K):
            c = 1.0 if k == 1 else 2.0
            dval[s:s + chunk] += c * np.einsum("nef,nef->ne", b[k][:, rows], X[k - 1][:, cols])
            ddiag[s:s + chunk] += c * np.einsum("nif,nif->ni", b[k], X[k - 1])
    return dval, ddiag


def network_graph_gradient(x, Ls, params, fcs, target, perm, M_in, levels, brelu="b1relu", conv_decisions=None,
                           head_masks=None):
    """Gradient of ``logits[b, target[b]]`` w.r.t. the entries of every level's Laplacian, per window, in fp64:
    ``{level: (dval [N, nnz], ddiag [N, M])}`` with layer ``i`` on ``Ls[i]`` of level ``levels[i]`` (layers of one level
    add up).  Built like ``network_input_gradient``: ``conv_stack`` on the windows permuted by ``perm`` (None: already
    in the first layer's order), the head, the one-hot seed, the head backward, then per layer from the top the
    MaxPoolGrad / ReluGrad of ``conv_stack_bwd`` (routed through ``conv_decisions`` when given), ``chebyshev5_dL`` and
    ``chebyshev5_bwd``'s dx for the layer below."""
    x = np.asarray(x, np.float64)
    xp = permute_rows(x, perm, M_in) if perm is not None else x
    h, trace = O.conv_stack(xp, Ls, params, brelu=brelu, dtype=np.float64, keep=True)
    F_last = h.shape[-1]
    acts = [h.mean(axis=-1)]
    for i, (W, b) in enumerate(fcs):
        z = acts[-1] @ np.asarray(W, np.float64) + np.asarray(b, np.float64)
        acts.append(np.maximum(z, 0) if i < len(fcs) - 1 else z)
    N = x.shape[0]
    d = np.zeros_like(acts[-1])
    d[np.arange(N), np.asarray(target)] = 1
    for i in range(len(fcs) - 1, -1, -1):
        if i < len(fcs) - 1:
            d = d * (np.asarray(head_masks[i], bool) if head_masks is not None else acts[i + 1] > 0)
        d = d @ np.asarray(fcs[i][0], np.float64).T
    dy = np.repeat(d[:, :, None], F_last, axis=2) / F_last
    out = {}
    for i in range(len(params) - 1, -1, -1):
        t, pr, L = trace[i], params[i], Ls[i]
        M = t["a"].shape[1]
        am, live = t["argmax"], t["a"]
        if conv_decisions is not None:
            am = np.asarray(conv_decisions[i]["argmax"], np.uint8).reshape(t["argmax"].shape)
            live = O.mpool1_bwd(np.asarray(conv_decisions[i]["relu"], np.float64).reshape(t["y"].shape), am, pr["p"], M)
        dz = O.mpool1_bwd(dy, am, pr["p"], M) * (live > 0)
        dval, ddiag = chebyshev5_dL(t["x"], L, pr["W"], pr["K"], dz)
        if levels[i] in out:
            out[levels[i]] = (out[levels[i]][0] + dval, out[levels[i]][1] + ddiag)
        else:
            out[levels[i]] = (dval, ddiag)
        if i > 0:
            dy, _ = O.chebyshev5_bwd(t["x"], L, pr["W"], pr["K"], dz, np.float64)
    return out


# ---- the layer -----------------------------------------------------------------------------------------------------
def _small_graph(M, seed):
    """A normalised Laplacian (stored diagonal of ones) of a random symmetric graph with a few isolated edges."""
    rng = np.random.RandomState(seed)
    A = sp.random(M, M, density=0.25, random_state=rng)
    A = sp.triu(A, 1)
    A = (A + A.T).tocsr()
    d = np.asarray(A.sum(1)).ravel() + 1e-3
    D = sp.diags(1 / np.sqrt(d))
    return sp.csr_matrix(sp.identity(M) - D @ A @ D)


def _layer_loss(x, L, W, b, K, p, brelu, dy):
    z = O.chebyshev5(x, L, W, K, np.float64)
    a = O.b1relu(z, b) if brelu == "b1relu" else O.b2relu(z, b)
    return (O.mpool1(a, p) * dy).sum(axis=(1, 2))  # per window


def _layer_case(K, p, brelu, seed, N=2, M=12, Fin=3, Fout=4):
    rng = np.random.RandomState(seed)
    L = _small_graph(M, seed)
    x = rng.randn(N, M, Fin)
    W = rng.randn(Fin * K, Fout) * 0.5
    b = rng.randn(Fout) * 0.1 if brelu == "b1relu" else rng.randn(M, Fout) * 0.1
    dy = rng.randn(N, -(-M // p), Fout)
    z = O.chebyshev5(x, L, W, K, np.float64)
    a = O.b1relu(z, b) if brelu == "b1relu" else O.b2relu(z, b)
    _, am = O.mpool1(a, p, with_argmax=True)
    dz = O.mpool1_bwd(dy, am, p, M) * (a > 0)
    return L, x, W, b, dy, dz


@pytest.mark.parametrize("K", [1, 2, 3, 5])
@pytest.mark.parametrize("p", [1, 4])
@pytest.mark.parametrize("brelu", ["b1relu", "b2relu"])
def test_layer_dL_matches_finite_differences(K, p, brelu):
    """Every stored entry of L~ and every diagonal entry, per window, against central differences of the layer's
    ``<dy, layer(x)>`` in L (``L~ = L - I``: the same entry)."""
    L, x, W, b, dy, dz = _layer_case(K, p, brelu, seed=10 * K + p)
    dval, ddiag = chebyshev5_dL(x, L, W, K, dz)
    Lt = O._rescaled(L, np.float64)
    M = L.shape[0]
    rows = np.repeat(np.arange(M), np.diff(Lt.indptr))
    entries = [(r, c, dval[:, e]) for e, (r, c) in enumerate(zip(rows, Lt.indices))]
    entries += [(i, i, ddiag[:, i]) for i in range(M)]
    Ld = L.toarray()
    h = 1e-6
    for r, c, an in entries:
        Lp, Lm = Ld.copy(), Ld.copy()
        Lp[r, c] += h
        Lm[r, c] -= h
        fd = (_layer_loss(x, sp.csr_matrix(Lp), W, b, K, p, brelu, dy)
              - _layer_loss(x, sp.csr_matrix(Lm), W, b, K, p, brelu, dy)) / (2 * h)
        assert np.allclose(an, fd, rtol=1e-6, atol=1e-7), (r, c, an, fd)
    if K == 1:
        assert not dval.any() and not ddiag.any()


@pytest.mark.parametrize("K,p,brelu", [(2, 1, "b1relu"), (3, 4, "b2relu"), (5, 4, "b1relu"), (5, 1, "b2relu")])
def test_layer_dL_matches_torch_autograd(K, p, brelu):
    """Against torch fp64 autograd through a dense L~ leaf (one copy per window) to 1e-10."""
    torch = pytest.importorskip("torch")
    L, x, W, b, dy, dz = _layer_case(K, p, brelu, seed=7 + K, N=3, M=16)
    N, M, Fin = x.shape
    Lt = O._rescaled(L, np.float64)
    leaf = torch.tensor(np.repeat(Lt.toarray()[None], N, 0), requires_grad=True)
    X = [torch.tensor(x)]
    if K > 1:
        X.append(torch.einsum("nij,njf->nif", leaf, X[0]))
    for _ in range(2, K):
        X.append(2 * torch.einsum("nij,njf->nif", leaf, X[-1]) - X[-2])
    Wt = torch.tensor(W)
    z = sum(X[k] @ Wt[k::K] for k in range(K))
    a = torch.relu(z + torch.tensor(b).reshape((1, 1, -1) if brelu == "b1relu" else (1, M, -1)))
    Mo = -(-M // p)
    pad = Mo * p - M
    ap = torch.nn.functional.pad(a, (0, 0, pad // 2, pad - pad // 2), value=-np.inf)
    y = ap.reshape(N, Mo, p, -1).amax(2)
    (y * torch.tensor(dy)).sum().backward()
    g = leaf.grad.numpy() if K > 1 else np.zeros((N, M, M))
    dval, ddiag = chebyshev5_dL(x, L, W, K, dz)
    rows = np.repeat(np.arange(M), np.diff(Lt.indptr))
    ref_val = g[:, rows, Lt.indices]
    ref_diag = g[:, np.arange(M), np.arange(M)]
    scale = max(np.abs(g).max(), 1.0)
    assert np.abs(dval - ref_val).max() <= 1e-10 * scale
    assert np.abs(ddiag - ref_diag).max() <= 1e-10 * scale


# ---- the network ---------------------------------------------------------------------------------------------------
def _network(graph, p, nlayers, seed, Fin=3, F=5, K=3, fc=(7, 4)):
    """A small seeded network on the 400-vertex test graph: ``nlayers`` layers with pooling ``p`` (levels from
    ``select_laplacians``; p = 1 puts every layer on the same Laplacian object)."""
    rng = np.random.RandomState(seed)
    Ls = O.select_laplacians(graph["L"], [p] * nlayers)
    levels, j = [], 0
    for _ in range(nlayers):
        levels.append(j)
        j += int(np.log2(p)) if p > 1 else 0
    params, fin = [], Fin
    for L in Ls:
        W = rng.randn(fin * K, F) * (0.8 / np.sqrt(fin * K))
        params.append(dict(W=W, b=rng.randn(F) * 0.1, K=K, p=p))
        fin = F
    width = -(-Ls[-1].shape[0] // p)
    fcs = []
    for n in fc:
        fcs.append((rng.randn(width, n) * (1.0 / np.sqrt(width)), rng.randn(n) * 0.1))
        width = n
    return Ls, levels, params, fcs


@pytest.mark.parametrize("p,nlayers", [(1, 3), (4, 2)])
def test_network_graph_gradient_matches_finite_differences(graph_l4, p, nlayers):
    """Directional derivatives of the summed target logits along random perturbations of each level's Laplacian (on
    its pattern and diagonal), by central differences, against <gradient, direction>: three layers sharing one
    Laplacian, and a pooled two-level network."""
    perm, M_in, N = graph_l4["perm"], 360, 2
    Ls, levels, params, fcs = _network(graph_l4, p, nlayers, seed=p + nlayers)
    rng = np.random.RandomState(5)
    x = rng.randn(N, M_in, 3)
    target = rng.randint(0, fcs[-1][0].shape[1], N)
    g = network_graph_gradient(x, Ls, params, fcs, target, perm, M_in, levels)
    assert sorted(g) == sorted(set(levels))

    def logit(Lmod):
        h = O.conv_stack(permute_rows(x, perm, M_in), Lmod, params, dtype=np.float64)
        return O.head(h, fcs, np.float64)[np.arange(N), target].sum()

    h = 1e-6
    for lvl in sorted(g):
        L = Ls[levels.index(lvl)]
        M = L.shape[0]
        Lt = O._rescaled(L, np.float64)
        rows = np.repeat(np.arange(M), np.diff(Lt.indptr))
        for _ in range(3):
            v_val, v_diag = rng.randn(Lt.nnz), rng.randn(M)
            V = sp.csr_matrix((v_val, (rows, Lt.indices)), shape=(M, M)) + sp.diags(v_diag)
            pert = lambda s: [Li + s * V if lv == lvl else Li for Li, lv in zip(Ls, levels)]
            fd = (logit(pert(h)) - logit(pert(-h))) / (2 * h)
            an = float((g[lvl][0].sum(0) * v_val).sum() + (g[lvl][1].sum(0) * v_diag).sum())
            assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (lvl, fd, an)


def test_edge_matrix_and_input_order(graph_l4):
    """The level-0 matrix in input-ROI order: every real entry of the pattern (diagonal included) lands exactly once
    at (perm[i], perm[j]) with its value, entries that touch a fake vertex are dropped; the model-order matrix has the
    pattern of L."""
    torch = pytest.importorskip("torch")  # noqa: F841
    from gcn_fmri_decoding_b200.plan import GraphPlan
    from gcn_fmri_decoding_b200.saliency import edge_matrix, to_input_order

    L = graph_l4["L"][0]
    perm, M_in = np.asarray(graph_l4["perm"]), 360
    pl = GraphPlan(L, "cpu")
    M, nnz = pl.M, pl.nnz
    g = np.arange(1, nnz + M + 1, dtype=np.float64)
    G = edge_matrix(pl, g)
    pattern = (sp.csr_matrix(L) != 0).astype(int) + sp.identity(M, dtype=int)
    assert ((G != 0).astype(int) != (pattern > 0).astype(int)).nnz == 0
    rp, ci, _ = pl._host[False]
    rows = np.repeat(np.arange(M), np.diff(rp))
    Gd = G.toarray()
    for e in range(nnz):
        if rows[e] != ci[e]:
            assert Gd[rows[e], ci[e]] == g[e]
    assert np.array_equal(np.diag(Gd), g[nnz:])
    R = to_input_order(G, perm, M_in)
    assert R.shape == (M_in, M_in)
    Gc = sp.coo_matrix(G)
    real = (perm[Gc.row] < M_in) & (perm[Gc.col] < M_in)
    assert R.nnz == real.sum() and real.sum() < Gc.nnz  # the test graph has fake vertices with entries
    Rd = R.toarray()
    seen = np.zeros((M_in, M_in), int)
    for r, c, v in zip(Gc.row[real], Gc.col[real], Gc.data[real]):
        assert Rd[perm[r], perm[c]] == v
        seen[perm[r], perm[c]] += 1
    assert seen.max() == 1 and seen.sum() == R.nnz
    fake_vals = set(Gc.data[~real].tolist())
    assert not fake_vals & set(R.data.tolist())

"""Edge saliency maps w.r.t. the adjacency, without a GPU: the fp64 chain rule from the per-level operator gradients to
the undirected edge weights of ``A`` (``adjacency_chain`` below: each level's degree normalisation, the Graclus
coarsening, the level-0 permutation) and the network-level ``network_adjacency_gradient`` against central differences
of the target logit along symmetric perturbations of ``A`` and against torch fp64 autograd through a dense ``A``; the
host maps of ``saliency.AdjacencyMaps`` against a brute-force construction; and the refusals of ``AdjacencyMaps``.
The GPU tests import the oracle from here."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import layers_np as O
from test_graph_saliency_oracle import _network, network_graph_gradient
from test_saliency_oracle import permute_rows


# ---- the fp64 oracle -----------------------------------------------------------------------------------------------
def coarsening(A, nlevels):
    """``graclus.coarsen(A, nlevels)`` -> ``(graphs, perm)``, leaving NumPy's global generator as it was."""
    from gcn_fmri_decoding_b200 import graclus

    state = np.random.get_state()
    try:
        return graclus.coarsen(sp.csr_matrix(A), nlevels)
    finally:
        np.random.set_state(state)


def _index(M, rows, cols):
    idx = -np.ones((M, M), np.int64)
    idx[rows, cols] = np.arange(len(rows))
    return idx


def edges_of(A):
    """The undirected edges ``(i, j)``, ``i < j``, of ``A``: the upper triangle in CSR order (``AdjacencyMaps``')."""
    U = sp.triu(sp.csr_matrix(A), 1).tocsr()
    U.eliminate_zeros()
    return np.repeat(np.arange(U.shape[0]), np.diff(U.indptr)), U.indices.copy()


def adjacency_chain(g, graphs, perm, A, Ls):
    """``{level: G [N, nnz]}`` (the gradient w.r.t. the entries of ``L~`` of that level, in ``O._rescaled(Ls[level])``'s
    CSR order) -> the gradient w.r.t. the undirected edge weights of ``A``, ``[N, E]`` in ``edges_of(A)``'s order, fp64.
    ``graphs`` / ``perm``: ``coarsening(A, ...)``.  Per level, top-down: ``T_l[(a, b)] = -G_ab s_a s_b - (r_b + c_b) /
    (2 d_b) + T_{l+1}[(a >> 1, b >> 1)]`` (the last term only across clusters); then ``S_ij = T_0[(a, b)] + T_0[(b, a)]``
    with ``a, b`` the model rows of ROIs ``i, j``."""
    T_next, idx_next = None, None
    for lvl in range(max(g), -1, -1):
        Al = sp.coo_matrix(graphs[lvl])
        a, b, w = Al.row.astype(np.int64), Al.col.astype(np.int64), Al.data.astype(np.float64)
        M = Al.shape[0]
        d = np.bincount(b, w, M)
        s = np.where(d > 0, 1 / np.sqrt(np.where(d > 0, d, 1)), 0)
        N = next(iter(g.values())).shape[0]
        T = np.zeros((N, len(a)))
        if lvl in g:
            Lt = O._rescaled(Ls[lvl], np.float64)
            idx = _index(M, np.repeat(np.arange(M), np.diff(Lt.indptr)), Lt.indices)
            assert (idx[a, b] >= 0).all()
            G = np.asarray(g[lvl], np.float64)[:, idx[a, b]]
            GL = G * (-s[a] * w * s[b])
            onehot = lambda v: sp.csr_matrix((np.ones(len(v)), (np.arange(len(v)), v)), shape=(len(v), M))
            r, c = GL @ onehot(a), GL @ onehot(b)
            T = -G * (s[a] * s[b]) - 0.5 * ((r + c) / np.where(d > 0, d, 1))[:, b]
        if T_next is not None:
            cross = (a >> 1) != (b >> 1)
            par = idx_next[a[cross] >> 1, b[cross] >> 1]
            assert (par >= 0).all()
            T[:, cross] += T_next[:, par]
        T_next, idx_next = T, _index(M, a, b)
    i, j = edges_of(A)
    inv = np.arange(graphs[0].shape[0])
    if perm is not None:
        inv[np.asarray(perm)] = np.arange(len(perm))
    return T_next[:, idx_next[inv[i], inv[j]]] + T_next[:, idx_next[inv[j], inv[i]]]


def network_adjacency_gradient(x, A, graphs, perm, Ls, params, fcs, target, M_in, levels, **kw):
    """Gradient of ``logits[b, target[b]]`` w.r.t. every undirected edge weight of ``A``, per window, fp64 ``[N, E]``:
    ``network_graph_gradient`` (layer ``i`` on ``Ls[levels[i]]``) followed by ``adjacency_chain``."""
    g = network_graph_gradient(x, [Ls[lv] for lv in levels], params, fcs, target, perm, M_in, levels, **kw)
    return adjacency_chain({lv: dval for lv, (dval, _) in g.items()}, graphs, perm, A, Ls)


# ---- the network, with the Laplacians rebuilt from A through the frozen coarsening -------------------------------
def laplacians_from(A, perm, sizes):
    """fp64 Laplacians of every level from ``A`` (dense or sparse), the matching frozen: level 0 is ``A`` permuted by
    ``perm``, level ``l + 1`` is ``P^T A_l P`` (vertices ``2J, 2J + 1`` merge into ``J``) with its diagonal zeroed."""
    from gcn_fmri_decoding_b200 import graphs

    A = sp.csr_matrix(A, dtype=np.float64)
    n = A.shape[0]
    if perm is not None:
        real = np.asarray(perm) < n
        Pm = sp.csr_matrix((np.ones(real.sum()), (np.arange(len(perm))[real], np.asarray(perm)[real])),
                           shape=(len(perm), n))
        A = sp.csr_matrix(Pm @ A @ Pm.T)
    out = []
    for lvl, M in enumerate(sizes):
        if lvl:
            P = sp.csr_matrix((np.ones(2 * M), (np.arange(2 * M), np.arange(2 * M) // 2)), shape=(2 * M, M))
            A = sp.lil_matrix(P.T @ A @ P)
            A.setdiag(0)
            A = sp.csr_matrix(A)
            A.eliminate_zeros()
        out.append(graphs.laplacian(A))
    return out


def _setup(graph, p, nlayers, seed, N=2):
    A = sp.csr_matrix(graph["A"], dtype=np.float64)
    sizes = [int(v) for v in graph["sizes"]]
    graphs_, perm = coarsening(graph["A"], len(sizes) - 1)
    perm = np.asarray(perm)
    assert np.array_equal(perm, graph["perm"])
    Ls = laplacians_from(A, perm, sizes)
    _, levels, params, fcs = _network(dict(L=Ls), p, nlayers, seed)
    rng = np.random.RandomState(seed + 1)
    x = rng.randn(N, A.shape[0], 3)
    target = rng.randint(0, fcs[-1][0].shape[1], N)
    return A, graphs_, perm, sizes, Ls, levels, params, fcs, x, target


def _logit(x, A, perm, sizes, levels, params, fcs, target):
    Ls = laplacians_from(A, perm, sizes)
    h = O.conv_stack(permute_rows(x, perm, x.shape[1]), [Ls[lv] for lv in levels], params, dtype=np.float64)
    return O.head(h, fcs, np.float64)[np.arange(x.shape[0]), target].sum()


@pytest.mark.parametrize("name,p,nlayers", [("graph_l4", 4, 2), ("graph_l1", 1, 3)])
def test_network_adjacency_gradient_matches_finite_differences(request, name, p, nlayers):
    """Directional derivatives of the summed target logits along random symmetric perturbations of ``A`` on its
    pattern, the Laplacians of every level rebuilt through the frozen coarsening, by central differences: a pooled
    two-level network (levels 0 and 2, level 1 only on the chain) and three layers on level 0 with fake vertices."""
    graph = request.getfixturevalue(name)
    A, graphs_, perm, sizes, Ls, levels, params, fcs, x, target = _setup(graph, p, nlayers, seed=3 + p)
    S = network_adjacency_gradient(x, A, graphs_, perm, Ls, params, fcs, target, A.shape[0], levels)
    i, j = edges_of(A)
    assert S.shape == (x.shape[0], len(i))
    rng = np.random.RandomState(11)
    h = 1e-6
    for _ in range(3):
        v = rng.randn(len(i))
        V = sp.csr_matrix((np.concatenate([v, v]), (np.concatenate([i, j]), np.concatenate([j, i]))), shape=A.shape)
        fd = (_logit(x, A + h * V, perm, sizes, levels, params, fcs, target)
              - _logit(x, A - h * V, perm, sizes, levels, params, fcs, target)) / (2 * h)
        an = float((S.sum(0) * v).sum())
        assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (fd, an)


def test_network_adjacency_gradient_matches_torch_autograd(graph_l4):
    """Against torch fp64 autograd through a dense ``A`` leaf (both orientations of each edge are separate entries of
    the leaf, so the edge gradient is ``grad[i, j] + grad[j, i]``) to 1e-10."""
    torch = pytest.importorskip("torch")
    A, graphs_, perm, sizes, Ls, levels, params, fcs, x, target = _setup(graph_l4, 2, 3, seed=21)
    S = network_adjacency_gradient(x, A, graphs_, perm, Ls, params, fcs, target, A.shape[0], levels)
    leaf = torch.tensor(A.toarray(), requires_grad=True)
    n, M0 = A.shape[0], sizes[0]
    Pm = torch.zeros(M0, n, dtype=torch.float64)
    real = perm < n
    Pm[np.arange(M0)[real], perm[real]] = 1
    Al = Pm @ leaf @ Pm.T
    Lt = []
    for lvl, M in enumerate(sizes):
        if lvl:
            P = torch.zeros(2 * M, M, dtype=torch.float64)
            P[np.arange(2 * M), np.arange(2 * M) // 2] = 1
            Al = (P.T @ Al @ P) * (1 - torch.eye(M, dtype=torch.float64))
        d = Al.sum(0)
        s = torch.where(d > 0, torch.where(d > 0, d, torch.ones_like(d)).rsqrt(), torch.zeros_like(d))
        Lt.append(-(s[:, None] * Al * s[None, :]))  # L - I: the diagonal of L is 1
    h = torch.tensor(permute_rows(x, perm, n))
    for lv, pr in zip(levels, params):
        K, W = pr["K"], torch.tensor(pr["W"])
        X = [h, Lt[lv] @ h]
        for _ in range(2, K):
            X.append(2 * (Lt[lv] @ X[-1]) - X[-2])
        z = sum(X[k] @ W[k::K] for k in range(K))
        a = torch.relu(z + torch.tensor(pr["b"]))
        Mo = -(-a.shape[1] // pr["p"])
        pad = Mo * pr["p"] - a.shape[1]
        a = torch.nn.functional.pad(a, (0, 0, pad // 2, pad - pad // 2), value=-np.inf)
        h = a.reshape(a.shape[0], Mo, pr["p"], -1).amax(2)
    out = h.mean(-1)
    for k, (W, b) in enumerate(fcs):
        out = out @ torch.tensor(W) + torch.tensor(b)
        if k < len(fcs) - 1:
            out = torch.relu(out)
    out[np.arange(len(target)), target].sum().backward()
    g = leaf.grad.numpy()
    i, j = edges_of(A)
    ref = g[i, j] + g[j, i]
    assert np.abs(S.sum(0) - ref).max() <= 1e-10 * max(np.abs(ref).max(), 1.0)


# ---- the host maps -------------------------------------------------------------------------------------------------
def _model(graph, p, nlayers=2, filt="chebyshev5", L=None, perm="graph"):
    torch = pytest.importorskip("torch")  # noqa: F841
    from gcn_fmri_decoding_b200.models import cgcnn

    return cgcnn(L=graph["L"] if L is None else L, F=[8] * nlayers, K=[3] * nlayers, p=[p] * nlayers, M=[16, 22],
                 filter=filt, channel=15, device="cpu", seed=1, perm=graph["perm"] if isinstance(perm, str) else perm,
                 n_input_vertices=360)


@pytest.mark.parametrize("name,p,nlayers", [("graph_l4", 4, 2), ("graph_l4", 2, 3), ("graph_l1", 1, 3)])
def test_adjacency_maps_match_brute_force(request, name, p, nlayers):
    """Every map of ``AdjacencyMaps`` against a per-entry construction from the recomputed coarsening: the transposed
    positions, ``s_a s_b`` and ``1 / (2 d)`` in fp64 rounded to fp32, the parent entries across one or more levels,
    and the two level-0 entries of every ROI edge."""
    from gcn_fmri_decoding_b200.saliency import AdjacencyMaps

    graph = request.getfixturevalue(name)
    model = _model(graph, p, nlayers)
    maps = AdjacencyMaps(model, graph["A"])
    graphs_, perm = coarsening(graph["A"], len(graph["sizes"]) - 1)
    used = sorted(set(model._graph_levels))
    assert maps.levels == used
    entries = {}
    for lvl in range(used[-1] + 1):
        pl = model._plan(graph["L"][lvl]) if lvl in used else None
        G = sp.csr_matrix(graphs_[lvl])
        G.sort_indices()
        rows = np.repeat(np.arange(G.shape[0]), np.diff(G.indptr))
        entries[lvl] = {(int(a), int(b)): e for e, (a, b) in enumerate(zip(rows, G.indices))}
        if pl is None:
            continue
        rp, ci, v = pl._host[False]
        rpt, cit, vt = pl._host[True]
        assert np.array_equal(v[maps.tpos[lvl]], vt)
        trow = np.repeat(np.arange(pl.M), np.diff(rpt))
        for t, e in enumerate(maps.tpos[lvl]):
            assert (rows[e], G.indices[e]) == (cit[t], trow[t])
        d = np.asarray(G.astype(np.float64).sum(0)).ravel()
        for e, (a, b) in enumerate(zip(rows, G.indices)):
            assert maps.ss[lvl][e] == np.float32(1 / np.sqrt(d[a] * d[b])) or \
                abs(maps.ss[lvl][e] - 1 / np.sqrt(d[a]) / np.sqrt(d[b])) <= 1e-7 * maps.ss[lvl][e]
        for b in range(pl.M):
            assert maps.hinv[lvl][b] == (np.float32(0.5 / d[b]) if d[b] > 0 else 0)
    for k, lvl in enumerate(used):
        if k + 1 == len(used):
            assert maps.parent[lvl] is None
            continue
        q = used[k + 1] - lvl
        for (a, b), e in entries[lvl].items():
            want = entries[used[k + 1]].get((a >> q, b >> q), -1) if (a >> q) != (b >> q) else -1
            if (a >> q) != (b >> q):
                assert want >= 0
            assert maps.parent[lvl][e] == want
    inv = {int(m): r for r, m in enumerate(perm)} if perm is not None else None
    ri, rj = edges_of(graph["A"])
    assert np.array_equal(maps.rows, ri) and np.array_equal(maps.cols, rj)
    for k, (i, j) in enumerate(zip(ri, rj)):
        a, b = (inv[i], inv[j]) if inv else (i, j)
        assert tuple(maps.edges[k]) == (entries[0][(a, b)], entries[0][(b, a)])
    Mx = maps.matrix(np.arange(1, len(ri) + 1))
    assert (Mx != Mx.T).nnz == 0 and ((Mx != 0) != (sp.csr_matrix(graph["A"]) != 0)).nnz == 0


def test_adjacency_maps_without_perm():
    """A single-level graph with no coarsening: no ``perm``, the level-0 entries are ``A``'s own."""
    torch = pytest.importorskip("torch")  # noqa: F841
    from gcn_fmri_decoding_b200 import graphs
    from gcn_fmri_decoding_b200.models import cgcnn
    from gcn_fmri_decoding_b200.saliency import AdjacencyMaps

    A = small_adjacency(40, seed=3)
    model = cgcnn(L=[graphs.laplacian(A)], F=[8], K=[3], p=[1], M=[22], channel=5, device="cpu", seed=1)
    maps = AdjacencyMaps(model, A)
    i, j = edges_of(A)
    G = sp.csr_matrix(A)
    idx = _index(40, np.repeat(np.arange(40), np.diff(G.indptr)), G.indices)
    assert np.array_equal(maps.edges[:, 0], idx[i, j]) and np.array_equal(maps.edges[:, 1], idx[j, i])
    assert maps.parent == {0: None}


def small_adjacency(n, seed, dtype=np.float32):
    """A random symmetric weighted graph with a zero diagonal and one isolated vertex."""
    rng = np.random.RandomState(seed)
    A = sp.triu(sp.random(n, n, density=0.15, random_state=rng), 1).tocsr()
    A = sp.lil_matrix(A + A.T, dtype=dtype)
    A[n - 1, :] = 0
    A[:, n - 1] = 0
    A = sp.csr_matrix(A)
    A.eliminate_zeros()
    return A


# ---- the refusals --------------------------------------------------------------------------------------------------
def test_adjacency_maps_refusals(graph_l4):
    from gcn_fmri_decoding_b200.saliency import AdjacencyMaps

    model = _model(graph_l4, 4)
    A = sp.csr_matrix(graph_l4["A"])
    with pytest.raises(ValueError, match="square"):
        AdjacencyMaps(model, A[:, :359])
    Aa = A.tolil()
    i, j = edges_of(A)
    Aa[i[0], j[0]] *= 2
    with pytest.raises(ValueError, match="symmetric"):
        AdjacencyMaps(model, Aa)
    Ad = A.tolil()
    Ad[5, 5] = 1
    with pytest.raises(ValueError, match="diagonal"):
        AdjacencyMaps(model, Ad)
    perm = np.array(graph_l4["perm"])
    perm[[0, 1]] = perm[[1, 0]]
    with pytest.raises(ValueError, match="perm"):
        AdjacencyMaps(_model(graph_l4, 4, perm=perm), A)
    with pytest.raises(ValueError, match="perm"):
        AdjacencyMaps(_model(graph_l4, 4, perm=None), A)
    L = list(graph_l4["L"])
    L2 = sp.csr_matrix(L[2], copy=True)
    L2.data[L2.data != 1] *= np.float32(1 + 1e-6)
    L[2] = L2
    with pytest.raises(ValueError, match="level 2"):
        AdjacencyMaps(_model(graph_l4, 4, L=L), A)
    L[2] = graph_l4["L"][2]
    L[1] = L2  # level 1 is used by no layer: only the used levels are compared
    AdjacencyMaps(_model(graph_l4, 4, L=L), A)
    with pytest.raises(ValueError, match="fourier"):
        AdjacencyMaps(_model(graph_l4, 4, filt="fourier"), A)
    state = np.random.get_state()
    AdjacencyMaps(model, A)
    assert np.array_equal(np.random.get_state()[1], state[1])  # the coarsening leaves the global generator alone

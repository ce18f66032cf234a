"""Saliency maps without a GPU: the fp64 oracle of a network's input gradient (``network_input_gradient`` below)
against central finite differences, the un-permutation of the Graclus ordering, and the host-side queries the
input-gradient call relies on (its route planner, the operator image of the transposed first-layer operator)."""
import numpy as np
import pytest

from oracle import layers_np as O


# ---- the fp64 oracle of a saliency map, built from oracle.layers_np (the GPU tests import it from here) ----
def permute_rows(x, perm, M_in):
    """coarsening.perm_data_3d: ``x [N, M_in, F]`` -> ``[N, len(perm), F]``, row ``m`` = raw row ``perm[m]``, zero for a
    fake vertex (``perm[m] >= M_in``)."""
    perm = np.asarray(perm)
    out = np.zeros((x.shape[0], len(perm), x.shape[2]), x.dtype)
    real = perm < M_in
    out[:, real] = x[:, perm[real]]
    return out


def unpermute_rows(g, perm, M_in):
    """Adjoint of ``permute_rows``: ``g [N, M, F]`` -> ``[N, M_in, F]``, row ``m`` added to raw row ``perm[m]``, fake
    vertices dropped."""
    perm = np.asarray(perm)
    out = np.zeros((g.shape[0], M_in, g.shape[2]), g.dtype)
    real = perm < M_in
    np.add.at(out, (slice(None), perm[real]), g[:, real])
    return out


def network_input_gradient(x, Ls, params, fcs, target, perm, M_in, filter="chebyshev5", brelu="b1relu",
                           conv_decisions=None, head_masks=None, dtype=np.float64):
    """Gradient of ``logits[b, target[b]]`` w.r.t. the raw windows ``x [N, M_in, F]`` (a gradient saliency map).

    ``conv_stack`` (on the windows permuted by ``perm``; ``perm=None``: ``x`` is already in the first layer's order) ->
    mean over F -> ``head`` with every activation kept, the one-hot seed of ``target`` on the logits, the head backward,
    ``conv_stack_bwd(first_needs_dx=True, decisions=conv_decisions)`` and the un-permutation through ``perm``.
    ``head_masks`` (one boolean ``[N, width]`` per hidden FC layer, another implementation's ``activation > 0``) routes
    the head backward the way that implementation decided, as ``conv_decisions`` does for pooling and the conv ReLUs;
    passing the oracle's own masks gives bit for bit what passing none gives.  Returns ``[N, M_in, F]`` (``[N, M, F]``
    without ``perm``).
    """
    x = np.asarray(x, dtype)
    xp = permute_rows(x, perm, M_in) if perm is not None else x
    h, trace = O.conv_stack(xp, Ls, params, filter=filter, brelu=brelu, dtype=dtype, keep=True)
    F_last = h.shape[-1]
    acts = [h.mean(axis=-1, dtype=dtype)]
    for i, (W, b) in enumerate(fcs):
        z = acts[-1] @ np.asarray(W, dtype) + np.asarray(b, dtype)
        acts.append(np.maximum(z, 0) if i < len(fcs) - 1 else z)
    N = x.shape[0]
    d = np.zeros_like(acts[-1])
    d[np.arange(N), np.asarray(target)] = 1
    for i in range(len(fcs) - 1, -1, -1):
        if i < len(fcs) - 1:
            d = d * (np.asarray(head_masks[i], bool) if head_masks is not None else acts[i + 1] > 0)
        d = d @ np.asarray(fcs[i][0], dtype).T
    dh = np.repeat(d[:, :, None], F_last, axis=2) / dtype(F_last)
    g, _ = O.conv_stack_bwd(trace, Ls, params, dh, filter=filter, brelu=brelu, dtype=dtype, first_needs_dx=True,
                          decisions=conv_decisions)
    return unpermute_rows(g, perm, M_in) if perm is not None else g


def _network(graph, filt, brelu, p, seed, Fin=3, F=(6, 5), K=(3, 2), fc=(7, 4)):
    """A small seeded two-layer network on the 400-vertex test graph (levels chosen by the pooling sizes)."""
    rng = np.random.RandomState(seed)
    Ls = O.select_laplacians(graph["L"], [p, p])
    params, fin = [], Fin
    for i, L in enumerate(Ls):
        M = L.shape[0]
        W = rng.randn(M, F[i], fin) * 0.5 if filt == "fourier" else rng.randn(fin * K[i], F[i]) * (0.8 / np.sqrt(fin * K[i]))
        b = rng.randn(F[i]) * 0.1 if brelu == "b1relu" else rng.randn(M, F[i]) * 0.1
        params.append(dict(W=W, b=b, K=K[i], p=p))
        fin = F[i]
    width = -(-Ls[-1].shape[0] // p)
    fcs = []
    for n in fc:
        fcs.append((rng.randn(width, n) * (1.0 / np.sqrt(width)), rng.randn(n) * 0.1))
        width = n
    return Ls, params, fcs


def _margin(x, perm, M_in, Ls, params, fcs, filt, brelu):
    """Smallest distance of any ReLU pre-activation from zero and of any pooled maximum from its runner-up (relative to
    the largest magnitude): the network is smooth within that distance.  Ties within rounding are left out: they are
    between values that do not depend on the input (fake vertices), whose gradient is zero whichever way they go."""
    nz = lambda a: a[a > 1e-12 * a.max()].min()
    xp = permute_rows(x, perm, M_in)
    h, trace = O.conv_stack(xp, Ls, params, filter=filt, brelu=brelu, dtype=np.float64, keep=True)
    gaps = []
    for t, pr in zip(trace, params):
        b = np.asarray(pr["b"]).reshape((1, 1, -1) if brelu == "b1relu" else (1,) + t["z"].shape[1:])
        pre = t["z"] + b
        gaps.append(nz(np.abs(pre)) / np.abs(pre).max())
        p = pr["p"]
        if p > 1:
            N, M, F = pre.shape
            Mo = -(-M // p)
            pad = np.full((N, Mo * p, F), -np.inf)
            pad[:, (Mo * p - M) // 2:(Mo * p - M) // 2 + M] = np.maximum(pre, 0)
            win = np.sort(pad.reshape(N, Mo, p, F), axis=2)
            live = win[:, :, -1] > 0
            gaps.append(nz((win[:, :, -1] - win[:, :, -2])[live]) / np.abs(pre).max())
    a = h.mean(-1)
    for i, (W, b) in enumerate(fcs[:-1]):
        a = a @ W + b
        gaps.append(nz(np.abs(a)) / np.abs(a).max())
        a = np.maximum(a, 0)
    return min(gaps)


def _logit(x, perm, M_in, Ls, params, fcs, filt, brelu, target):
    h = O.conv_stack(permute_rows(x, perm, M_in), Ls, params, filter=filt, brelu=brelu, dtype=np.float64)
    lg = O.head(h, fcs, np.float64)
    return lg[np.arange(len(target)), target].sum()


@pytest.mark.parametrize("filt,brelu,p", [("chebyshev5", "b1relu", 1), ("chebyshev5", "b2relu", 2),
                                          ("chebyshev5", "b1relu", 4), ("chebyshev5", "b2relu", 4),
                                          ("fourier", "b1relu", 2)])
def test_input_gradient_matches_finite_differences(graph_l4, filt, brelu, p):
    """Directional derivatives of the summed target logits, by central differences, against <gradient, direction>, at
    points whose ReLU and arg-max decisions are at least 2e-5 (relative) away from a tie."""
    perm, M_in, N = graph_l4["perm"], 360, 3
    Ls, params, fcs = _network(graph_l4, filt, brelu, p, seed=p)
    for seed in range(20):
        rng = np.random.RandomState(100 + seed)
        x = rng.randn(N, M_in, 3)
        if _margin(x, perm, M_in, Ls, params, fcs, filt, brelu) > 2e-5:
            break
    else:
        pytest.fail("no seed gives a point away from ties")
    target = rng.randint(0, fcs[-1][0].shape[1], N)
    g = network_input_gradient(x, Ls, params, fcs, target, perm, M_in, filter=filt, brelu=brelu)
    assert g.shape == x.shape
    h = 1e-7
    for _ in range(4):
        v = rng.randn(*x.shape)
        fd = (_logit(x + h * v, perm, M_in, Ls, params, fcs, filt, brelu, target)
              - _logit(x - h * v, perm, M_in, Ls, params, fcs, filt, brelu, target)) / (2 * h)
        an = float((g * v).sum())
        assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (fd, an)


def test_unpermutation_drops_fake_vertices_and_writes_every_raw_vertex_once(graph_l4):
    """The adjoint of the first layer's gather: every raw row receives exactly the row its vertex has in the layer's
    order, and the rows of fake vertices (perm >= M_in) reach no raw row -- in the oracle and in ops.unpermute."""
    torch = pytest.importorskip("torch")
    from gcn_fmri_decoding_b200 import ops

    perm, M_in = graph_l4["perm"], 360
    M = len(perm)
    assert (perm >= M_in).sum() == M - M_in and sorted(perm) == list(range(M))
    g = (np.arange(2 * M * 3, dtype=np.float64).reshape(2, M, 3) + 1)
    raw = unpermute_rows(g, perm, M_in)
    hits = np.zeros(M_in, int)
    for m in range(M):
        if perm[m] < M_in:
            hits[perm[m]] += 1
            assert np.array_equal(raw[:, perm[m]], g[:, m])
    assert (hits == 1).all()
    fake_vals = set(g[:, perm >= M_in].ravel().tolist())
    assert not fake_vals & set(raw.ravel().tolist())
    got = ops.unpermute(torch.as_tensor(g), torch.as_tensor(perm, dtype=torch.int32), M_in).numpy()
    assert np.array_equal(got, raw)
    # the adjoint of permute_rows: <P x, g> = <x, P^T g>
    x = np.random.RandomState(0).randn(2, M_in, 3)
    assert np.isclose((permute_rows(x, perm, M_in) * g).sum(), (x * raw).sum(), rtol=1e-12)


@pytest.mark.parametrize("filt,brelu", [("chebyshev5", "b1relu"), ("chebyshev5", "b2relu")])
def test_own_decisions_and_masks_are_bit_identical(graph_l4, filt, brelu):
    perm, M_in = graph_l4["perm"], 360
    Ls, params, fcs = _network(graph_l4, filt, brelu, 4, seed=9)
    rng = np.random.RandomState(3)
    x = rng.randn(4, M_in, 3)
    target = rng.randint(0, 4, 4)
    xp = permute_rows(x, perm, M_in)
    h, trace = O.conv_stack(xp, Ls, params, filter=filt, brelu=brelu, dtype=np.float64, keep=True)
    dec = [dict(argmax=t["argmax"], relu=t["y"] > 0) for t in trace]
    a = h.mean(-1)
    masks = []
    for W, b in fcs[:-1]:
        a = np.maximum(a @ W + b, 0)
        masks.append(a > 0)
    plain = network_input_gradient(x, Ls, params, fcs, target, perm, M_in, filter=filt, brelu=brelu)
    given = network_input_gradient(x, Ls, params, fcs, target, perm, M_in, filter=filt, brelu=brelu,
                                     conv_decisions=dec, head_masks=masks)
    assert np.array_equal(plain, given)


# the benchmarked layer shapes: (graph, level of conv 1, level of conv 2, channel, F, K, p, B)
PLANNER_CASES = [("config2", "l4", 0, 2, 15, 32, 5, 4, 512), ("config3a-K2", "l4", 0, 2, 15, 32, 2, 4, 512),
                 ("config3a-K1", "l4", 0, 2, 15, 32, 1, 4, 512), ("config1", "l1", 0, 0, 15, 32, 5, 1, 128)]


@pytest.mark.parametrize("name,graph,l1,l2,C,F,K,p,B", PLANNER_CASES)
def test_dx_planner_takes_the_tcgen05_adjoint_for_benchmarked_layers(graph_l4, graph_l1, name, graph, l1, l2, C, F, K, p,
                                                                      B):
    """gcnb_cheb_dx_describe: conv 1 (Fin = 15, not a multiple of 4) and conv 2 take the tcgen05 adjoint under AUTO; the
    workspace it returns covers the route it names -- nothing for the adjoint, and for ALGO_FUSED / ALGO_GENERAL at
    least what the same route needs inside the full backward."""
    from gcn_fmri_decoding_b200 import _lib

    g = graph_l4 if graph == "l4" else graph_l1
    for lvl, Fin in ((l1, C), (l2, F)):
        Lr = g["L"][lvl]
        shape = (B, Lr.shape[0], g["Lt"][lvl].nnz, Fin, F, K, p)
        text, ws = _lib.describe_dx(*shape)
        assert text.startswith("tcgen05 adjoint only: k_cheb_fwd_umma"), (name, lvl, text)
        assert ws == 0
        for algo, route in ((_lib.ALGO_FUSED, "fused dx"), (_lib.ALGO_GENERAL, "general path")):
            text, ws = _lib.describe_dx(*shape, algo)
            if algo == _lib.ALGO_FUSED and not _lib.lib().gcnb_cheb_fused_supported(*shape, 1, 1):
                route = "unsupported"  # the fused backward with dx does not hold this graph (conv 1 of config 2)
            assert text.split(":")[0] == route, text
            if route == "unsupported":
                continue
            _, full = _lib.describe(*shape, True, True, False, algo)
            assert ws % 256 == 0 and ws >= (full if algo == _lib.ALGO_GENERAL else 0) + B * Lr.shape[0] * Fin * 4, (text, ws)


def test_dx_planner_leaves_the_full_backward_alone(graph_l4):
    """The widened adjoint serves the input-gradient-only call alone: the training backward of a Fin = 15 layer with dx
    keeps its route."""
    from gcn_fmri_decoding_b200 import _lib

    shape = (512, 400, graph_l4["Lt"][0].nnz, 15, 32, 5, 4)
    for saved in (True, False):
        assert "tcgen05" not in _lib.describe(*shape, True, True, saved)[0]
    assert _lib.describe_dx(*shape)[0].startswith("tcgen05 adjoint only")


def test_adjoint_image_of_the_first_layer_decodes_to_the_transpose(graph_l4):
    """The operator image of L~^T for the Fin = 15 layer shape (the input gradient of conv 1), as test_image checks the
    other shapes."""
    from test_image import _decode

    from gcn_fmri_decoding_b200 import _lib, graphs

    Lr = graphs.rescale_L(graph_l4["L"][0], lmax=2)
    rp, ci, v = graphs.csr_arrays(Lr, transpose=True)
    M, nnz = Lr.shape[0], len(v)
    lib = _lib.lib()
    args = (512, M, nnz, 15, 32, 5, 4, 1)
    n = lib.gcnb_cheb_image_bytes(rp.ctypes.data, ci.ctypes.data, *args)
    assert n > 0 and n % 16 == 0
    img = np.zeros(n, np.uint8)
    _lib.check(lib.gcnb_cheb_image_build(rp.ctypes.data, ci.ctypes.data, v.ctypes.data, *args, img.ctypes.data, n), "build")
    assert np.array_equal(_decode(img, M, 1), np.asarray(Lr.T.todense(), np.float32))

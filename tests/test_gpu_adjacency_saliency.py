"""Edge saliency maps w.r.t. the adjacency on the B200 against the fp64 oracle: the chain-rule call
(``ops.adjacency_grad``: ``k_adjacency_level`` per level, ``k_adjacency_edges``) and the whole schedule
(``saliency.AdjacencyGradient`` / ``cgcnn.adjacency_saliency``).  Run on the B200 box: -m gpu.

As in test_gpu_graph_saliency, the oracle is routed through the device's pooling, ReLU and FC-mask decisions.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import rel_inf
from test_adjacency_saliency_oracle import (adjacency_chain, coarsening, edges_of, network_adjacency_gradient,
                                            small_adjacency)
from test_gpu_parity import build_model
from test_gpu_saliency import T, _device_decisions, _params

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _coarsening(graph):
    graphs_, perm = coarsening(graph["A"], len(graph["sizes"]) - 1)
    return graphs_, np.asarray(perm)


# ------------------------------------------------------------------------------------------ the call
@pytest.mark.parametrize("name,p,nlayers", [("graph_l4", 4, 2), ("graph_l4", 2, 3), ("graph_l1", 1, 2)])
@pytest.mark.parametrize("absolute", [False, True])
def test_adjacency_grad_matches_fp64_chain(dev, request, name, p, nlayers, absolute):
    """ops.adjacency_grad on random operator gradients at B = 37 against the fp64 chain: levels 0 and 2 (level 1 on
    the chain only), levels 0, 1 and 2, and one level with fake vertices; then bit-identical repeats."""
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.saliency import AdjacencyMaps

    graph = request.getfixturevalue(name)
    model = build_model(graph, [8] * nlayers, [3] * nlayers, [p] * nlayers, [64, 22], "chebyshev5", "b1relu", dev,
                        perm=graph["perm"])
    maps = AdjacencyMaps(model, graph["A"])
    per_level, edges = maps.device(dev)
    B = 37
    rng = np.random.RandomState(7 + p)
    G, levels = {}, []
    for lvl in maps.levels:
        pl = model._plan(graph["L"][lvl])
        G[lvl] = rng.randn(B, pl.nnz).astype(np.float32)
        levels.append((T(G[lvl], dev), pl.rowptr, pl.val, pl.rowptr_t) + per_level[lvl])
    got = ops.adjacency_grad(levels, edges, absolute)
    graphs_, perm = _coarsening(graph)
    ref = adjacency_chain(G, graphs_, perm, graph["A"], graph["L"])
    if absolute:
        ref = np.abs(ref)
    assert got.shape == ref.shape
    assert rel_inf(got.cpu().numpy(), ref) <= TOL, rel_inf(got.cpu().numpy(), ref)
    assert torch.equal(got, ops.adjacency_grad(levels, edges, absolute))


# ------------------------------------------------------------------------------------------ the network
def _reference(model, graph, xraw, target, dec, masks, absolute, chunk=128):
    """The oracle's edge vector, through the device's decisions, summed over windows (|.| per window)."""
    params, fcs = _params(model)
    graphs_, perm = _coarsening(graph)
    total = 0.0
    for s in range(0, xraw.shape[0], chunk):
        sl = slice(s, min(xraw.shape[0], s + chunk))
        S = network_adjacency_gradient(xraw[sl], graph["A"], graphs_, perm, graph["L"], params, fcs, target[sl],
                                       xraw.shape[1], model._graph_levels, brelu=model.brelu_name,
                                       conv_decisions=[{k: v[sl] for k, v in d.items()} for d in dec],
                                       head_masks=[m_[sl] for m_ in masks])
        total = total + (np.abs(S) if absolute else S).sum(0)
    return total


def _decisions(model, xraw, gather):
    """The device's conv decisions and FC masks, batch by batch as the schedule pads them."""
    from gcn_fmri_decoding_b200.saliency import InputGradient

    n, bs = xraw.shape[0], model.batch_size
    ig = InputGradient(model)
    ig(model._padded_batch(xraw, 0), gather=gather)  # sets up the dropout counter the head's GEMM call takes
    decs, maskss = [], []
    for s in range(0, n, bs):
        d, m_ = _device_decisions(model, ig, model._padded_batch(xraw, s), gather)
        k = min(bs, n - s)
        decs.append([{a: v[:k] for a, v in di.items()} for di in d])
        maskss.append([mm[:k] for mm in m_])
    dec = [{a: np.concatenate([dd[i][a] for dd in decs]) for a in decs[0][i]} for i in range(len(model.p))]
    masks = [np.concatenate([mm[i] for mm in maskss]) for i in range(len(model.M) - 1)]
    return dec, masks


def _check_network(dev, model, graph, xraw):
    """cgcnn.adjacency_saliency on raw windows against the oracle, signed and absolute: a symmetric float64 CSR on
    the pattern of A in ROI order."""
    target = model.predict(xraw).astype(np.int64)
    dec, masks = _decisions(model, xraw, True)
    A = sp.csr_matrix(graph["A"])
    i, j = edges_of(A)
    for absolute in (False, True):
        got = model.adjacency_saliency(xraw, A, absolute=absolute)
        assert isinstance(got, sp.csr_matrix) and got.dtype == np.float64 and got.shape == A.shape
        assert (got != got.T).nnz == 0
        ref = _reference(model, graph, xraw, target, dec, masks, absolute)
        vals = np.asarray(got[i, j]).ravel()
        assert rel_inf(vals, ref) <= TOL, (absolute, rel_inf(vals, ref))
        nz = got.tocoo()
        assert np.asarray(A[nz.row, nz.col]).all()  # nothing off the pattern of A
        if absolute:
            assert got.data.min() >= 0


def test_config2_network_matches_oracle(dev, graph_l4):
    """The benchmark's config-2 network (two levels, 0 and 2, with level 1 on the chain) at B = 512 over 889 windows:
    the last batch is zero-padded and its padding contributes nothing."""
    from gcn_fmri_decoding_b200 import synth

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    model.batch_size = 512
    _check_network(dev, model, graph_l4, synth.bold_windows(889, seed=41))


def test_config1_network_matches_oracle(dev, graph_l1):
    """Config 1: six b2relu layers on level 0 (with fake vertices) at B = 128."""
    from gcn_fmri_decoding_b200 import synth

    model = build_model(graph_l1, [32] * 6, [5] * 6, [1] * 6, [512, 256, 22], "chebyshev5", "b2relu", dev,
                        perm=graph_l1["perm"])
    model.batch_size = 128
    _check_network(dev, model, graph_l1, synth.bold_windows(128, seed=42))


def test_signed_output_is_the_chain_of_graph_gradient(dev, graph_l4):
    """The map is linear: the signed adjacency gradient equals the fp64 chain applied to GraphGradient's per-level sums
    over the same batches."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.saliency import AdjacencyGradient, AdjacencyMaps, GraphGradient

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    maps = AdjacencyMaps(model, graph_l4["A"])
    gg, ag = GraphGradient(model), AdjacencyGradient(model, maps)
    sums, got = {}, 0.0
    for seed in (1, 2, 3):
        x = T(synth.bold_windows(256, seed=seed), dev)
        for lvl, v in gg(x, gather=True)[0].items():
            nnz = model._plan(graph_l4["L"][lvl]).nnz
            sums[lvl] = sums.get(lvl, 0.0) + v[:nnz].cpu().numpy().astype(np.float64)
        got = got + ag(x, gather=True)[0].cpu().numpy().astype(np.float64)
    graphs_, perm = _coarsening(graph_l4)
    ref = adjacency_chain({lvl: v[None] for lvl, v in sums.items()}, graphs_, perm, graph_l4["A"], graph_l4["L"])[0]
    assert rel_inf(got, ref) <= TOL, rel_inf(got, ref)


def test_repeats_and_graph_replay_are_bit_identical(dev, graph_l4):
    """Two calls give the same bits, the CUDA-graph replay equals the eager schedule bit for bit, a given target is
    honoured, and padding rows (valid < B) contribute nothing."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.saliency import AdjacencyGradient, AdjacencyMaps

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    maps = AdjacencyMaps(model, graph_l4["A"])
    x = T(synth.bold_windows(64, seed=8), dev)
    ag = AdjacencyGradient(model, maps)
    for absolute in (False, True):
        a, _, t = ag(x, gather=True, absolute=absolute)
        a = a.clone()
        b = ag(x, gather=True, absolute=absolute)[0]
        e = AdjacencyGradient(model, maps, use_cuda_graph=False)(x, gather=True, absolute=absolute)[0]
        assert torch.equal(a, b) and torch.equal(a, e)
        assert torch.equal(ag(x, target=t, gather=True, absolute=absolute)[0], a)
    part = ag(x, gather=True, valid=40)[0].clone()
    only = AdjacencyGradient(model, maps, use_cuda_graph=False)(x[:40], gather=True)[0]
    assert rel_inf(part.cpu().numpy(), only.cpu().numpy()) <= 1e-6


def test_single_level_graph_without_perm(dev):
    """A 60-vertex graph with one isolated vertex, one level, no perm: windows in the graph's own order."""
    from gcn_fmri_decoding_b200 import graphs
    from gcn_fmri_decoding_b200.models import cgcnn

    A = small_adjacency(60, seed=5)
    L = [graphs.laplacian(A)]
    model = cgcnn(L=L, F=[16, 16], K=[4, 3], p=[1, 1], M=[64, 22], channel=15, device=dev, seed=3, batch_size=32)
    rng = np.random.RandomState(9)
    x = rng.randn(50, 60, 15).astype(np.float32)
    target = rng.randint(0, 22, 50)
    got = model.adjacency_saliency(x, A, target=target)
    params, fcs = _params(model)
    dec, masks = _decisions(model, x, False)
    ref = network_adjacency_gradient(x, A, [A], None, L, params, fcs, target, 60, [0, 0], brelu=model.brelu_name,
                                     conv_decisions=dec, head_masks=masks).sum(0)
    i, j = edges_of(A)
    assert rel_inf(np.asarray(got[i, j]).ravel(), ref) <= TOL
    assert model.adjacency_saliency(x, A, target=target)[i, j].tolist() == got[i, j].tolist()

"""Edge saliency maps on the B200 against the fp64 oracle: the operator-gradient layer call (``ops.cheb_dL``: the general
path's stacks and ``k_sddmm_tma``) and the whole schedule (``saliency.GraphGradient`` / ``cgcnn.graph_saliency``).
Run on the B200 box: -m gpu.

As in test_gpu_saliency, the oracle is routed through the device's pooling, ReLU and FC-mask decisions.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import rel_inf
from oracle import layers_np as O
from test_gpu_parity import build_model
from test_gpu_saliency import T, _device_decisions, _params, _perm_with_fakes
from test_graph_saliency_oracle import chebyshev5_dL, network_graph_gradient
from test_saliency_oracle import permute_rows, unpermute_rows

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------ the layer
# (level, Fin, Fout, K, p, brelu, dy_is_mean, with_perm, B): every Fin x K, each other value at least twice; B = 37 makes
# B * Fin a non-multiple of 4 for the odd widths (unaligned row chunks)
LAYER_CASES = [
    (0, 9, 16, 1, 4, "b1relu", True, True, 37),
    (0, 9, 32, 2, 1, "b2relu", False, False, 64),
    (0, 9, 16, 5, 4, "b2relu", False, True, 37),
    (2, 15, 32, 1, 1, "b1relu", False, True, 37),
    (0, 15, 32, 2, 4, "b1relu", True, True, 37),
    (2, 15, 16, 5, 1, "b2relu", True, False, 37),
    (0, 15, 32, 5, 4, "b1relu", True, True, 300),
    (0, 32, 32, 1, 4, "b2relu", False, False, 37),
    (2, 32, 16, 2, 4, "b2relu", True, True, 37),
    (0, 32, 32, 5, 1, "b1relu", False, True, 37),
    (2, 32, 32, 5, 4, "b1relu", True, True, 129),
]


@pytest.mark.parametrize("lvl,Fin,Fout,K,p,brelu,dy_is_mean,with_perm,B", LAYER_CASES)
def test_cheb_dL_matches_oracle(dev, graph_l4, lvl, Fin, Fout, K, p, brelu, dy_is_mean, with_perm, B):
    """ops.cheb_dL against chebyshev5_dL (dval, ddiag) and chebyshev5_bwd (dx); dx bit for bit cheb_dx on the general
    path; accumulate onto zeros bit for bit the overwrite, and onto a previous result its sum."""
    from gcn_fmri_decoding_b200 import _lib, ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    L = graph_l4["L"][lvl]
    M = L.shape[0]
    pl = GraphPlan(L, dev)
    assert "k_sddmm_tma" in _lib.describe_dL(B, M, pl.nnz, Fin, Fout, K, p)[0] or K == 1
    if with_perm:
        perm = graph_l4["perm"].astype(np.int32) if lvl == 0 else _perm_with_fakes(M, 10, Fin)
        M_in = 360 if lvl == 0 else M - 10
    else:
        perm, M_in = None, M
    rng = np.random.RandomState(100 * Fin + 10 * K + p)
    x = rng.randn(B, M_in, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * (0.4 / np.sqrt(Fin * K))).astype(np.float32)
    bshape = (Fout,) if brelu == "b1relu" else (M, Fout)
    b = (rng.randn(*bshape) * 0.1).astype(np.float32)
    mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
    Mo = -(-M // p)
    dy = rng.randn(B, Mo).astype(np.float32) if dy_is_mean else rng.randn(B, Mo, Fout).astype(np.float32)
    pt = T(perm, dev, torch.int32) if perm is not None else None
    y, am, _, _ = ops.cheb_fwd_mean(T(x, dev), pt, pl.rowptr, pl.col, pl.val, T(W, dev), T(b, dev), K, p, mode, True,
                                    _lib.ALGO_AUTO, False)
    dval, ddiag = torch.empty((B, pl.nnz), device=dev), torch.empty((B, M), device=dev)
    args = (T(x, dev), pt, M_in, y, am, T(dy, dev), dy_is_mean, *pl.tensors(), T(W, dev))
    dx = ops.cheb_dL(*args, dval, ddiag, False, K, p, True, True)
    # the oracle, through the device's decisions
    ya, ama = y.cpu().numpy().astype(np.float64), am.cpu().numpy() if p > 1 else np.zeros(y.shape, np.uint8)
    dyf = np.repeat(dy[:, :, None].astype(np.float64), Fout, 2) / Fout if dy_is_mean else dy.astype(np.float64)
    dz = O.mpool1_bwd(dyf * (ya > 0), ama, p, M)
    xp = permute_rows(x.astype(np.float64), perm, M_in) if perm is not None else x.astype(np.float64)
    ref_val, ref_diag = chebyshev5_dL(xp, L, W, K, dz)
    g, _ = O.chebyshev5_bwd(xp, L, W, K, dz, np.float64)
    ref_dx = unpermute_rows(g, perm, M_in) if perm is not None else g
    if K == 1:
        assert not dval.any() and not ddiag.any()
    else:
        assert rel_inf(dval.cpu().numpy(), ref_val) <= TOL, rel_inf(dval.cpu().numpy(), ref_val)
        assert rel_inf(ddiag.cpu().numpy(), ref_diag) <= TOL, rel_inf(ddiag.cpu().numpy(), ref_diag)
    assert rel_inf(dx.cpu().numpy(), ref_dx) <= TOL, rel_inf(dx.cpu().numpy(), ref_dx)
    # dx: the general route of the input-gradient-only call, bit for bit
    dx_g = ops.cheb_dx(*args, K, p, True, _lib.ALGO_GENERAL)
    assert torch.equal(dx, dx_g)
    # accumulate onto zeros = overwrite; onto the previous result = twice it (one rounding: x + x is exact)
    v0, d0 = torch.zeros_like(dval), torch.zeros_like(ddiag)
    ops.cheb_dL(*args, v0, d0, True, K, p, True, False)
    assert torch.equal(v0, dval) and torch.equal(d0, ddiag)
    ops.cheb_dL(*args, v0, d0, True, K, p, True, False)
    assert torch.equal(v0, 2 * dval) and torch.equal(d0, 2 * ddiag)


# ------------------------------------------------------------------------------------------ the network
def _reference(model, xraw, target, dec, masks, absolute, chunk=128):
    """{level: dense [M, M]} of the oracle, through the device's decisions, summed over windows (|.| per window)."""
    params, fcs = _params(model)
    perm = model.perm.cpu().numpy()
    levels = model._graph_levels
    out = {}
    for s in range(0, xraw.shape[0], chunk):
        sl = slice(s, min(xraw.shape[0], s + chunk))
        g = network_graph_gradient(xraw[sl], model.L, params, fcs, target[sl], perm, xraw.shape[1], levels,
                                   brelu=model.brelu_name, conv_decisions=[{k: v[sl] for k, v in d.items()} for d in dec],
                                   head_masks=[m_[sl] for m_ in masks])
        for lvl, (dval, ddiag) in g.items():
            if absolute:
                dval, ddiag = np.abs(dval), np.abs(ddiag)
            acc = out.setdefault(lvl, [0.0, 0.0])
            acc[0] = acc[0] + dval.sum(0)
            acc[1] = acc[1] + ddiag.sum(0)
    dense = {}
    for lvl, (v, d) in out.items():
        L = model.L[levels.index(lvl)]
        Lt = O._rescaled(L, np.float64)
        M = L.shape[0]
        rows = np.repeat(np.arange(M), np.diff(Lt.indptr))
        off = rows != Lt.indices
        D = np.zeros((M, M))
        D[rows[off], Lt.indices[off]] = v[off]
        D[np.arange(M), np.arange(M)] = d
        dense[lvl] = D
    return dense


def _check_network(dev, model, xraw):
    """cgcnn.graph_saliency on raw windows (level 0 in ROI order, coarser levels in the model's order) against the
    oracle, signed and absolute."""
    from gcn_fmri_decoding_b200.saliency import InputGradient

    n = xraw.shape[0]
    perm = model.perm.cpu().numpy()
    target = model.predict(xraw).astype(np.int64)
    # the device's decisions, batch by batch as graph_saliency pads them
    bs = model.batch_size
    ig = InputGradient(model)
    ig(model._padded_batch(xraw, 0), gather=True)  # sets up the dropout counter the head's GEMM call takes
    decs, maskss = [], []
    for s in range(0, n, bs):
        g = model._padded_batch(xraw, s)
        d, m_ = _device_decisions(model, ig, g, True)
        k = min(bs, n - s)
        decs.append([{a: v[:k] for a, v in di.items()} for di in d])
        maskss.append([mm[:k] for mm in m_])
    dec = [{a: np.concatenate([dd[i][a] for dd in decs]) for a in decs[0][i]} for i in range(len(model.p))]
    masks = [np.concatenate([mm[i] for mm in maskss]) for i in range(len(model.M) - 1)]
    for absolute in (False, True):
        got = model.graph_saliency(xraw, absolute=absolute)
        ref = _reference(model, xraw, target, dec, masks, absolute)
        assert sorted(got) == sorted(ref) == sorted(set(model._graph_levels))
        for lvl, G in got.items():
            assert isinstance(G, sp.csr_matrix) and G.dtype == np.float64
            R = ref[lvl]
            if lvl == 0:  # raw windows: ROI order, fake vertices dropped
                M_in = xraw.shape[1]
                assert G.shape == (M_in, M_in)
                real = perm < M_in
                Rr = np.zeros((M_in, M_in))
                Rr[np.ix_(perm[real], perm[real])] = R[np.ix_(real, real)]
                R = Rr
            assert rel_inf(G.toarray(), R) <= TOL, (lvl, absolute, rel_inf(G.toarray(), R))
            if absolute:
                assert G.data.min() >= 0
    return target


def test_config2_network_matches_oracle(dev, graph_l4):
    """The benchmark's config-2 network (360 ROIs -> 400 -> 100 vertices, 15 TRs, two levels) at B = 512 over 889
    windows: the last batch is zero-padded and its padding contributes nothing."""
    from gcn_fmri_decoding_b200 import synth

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    model.batch_size = 512
    assert model._graph_levels == [0, 2]
    _check_network(dev, model, synth.bold_windows(889, seed=31))


def test_config1_network_matches_oracle(dev, graph_l1):
    """Config 1: six b2relu layers on L[0] (one Laplacian, six contributions per window) at B = 128."""
    from gcn_fmri_decoding_b200 import synth

    model = build_model(graph_l1, [32] * 6, [5] * 6, [1] * 6, [512, 256, 22], "chebyshev5", "b2relu", dev,
                        perm=graph_l1["perm"])
    model.batch_size = 128
    assert model._graph_levels == [0] * 6
    _check_network(dev, model, synth.bold_windows(128, seed=32))


def test_repeats_and_graph_replay_are_bit_identical(dev, graph_l4):
    """Two calls give the same bits, the CUDA-graph replay equals the eager schedule bit for bit, a given target is
    honoured, and padding rows (valid < B) contribute exactly nothing."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.saliency import GraphGradient

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    x = T(synth.bold_windows(64, seed=8), dev)
    gg = GraphGradient(model)
    for absolute in (False, True):
        a, _, t = gg(x, gather=True, absolute=absolute)
        a = {k: v.clone() for k, v in a.items()}
        b = gg(x, gather=True, absolute=absolute)[0]
        e = GraphGradient(model, use_cuda_graph=False)(x, gather=True, absolute=absolute)[0]
        for k in a:
            assert torch.equal(a[k], b[k]) and torch.equal(a[k], e[k])
        given = gg(x, target=t, gather=True, absolute=absolute)[0]
        for k in a:
            assert torch.equal(given[k], a[k])
    part = {k: v.clone() for k, v in gg(x, gather=True, valid=40)[0].items()}
    only = GraphGradient(model, use_cuda_graph=False)(x[:40], gather=True)[0]
    for k in part:
        assert rel_inf(part[k].cpu().numpy(), only[k].cpu().numpy()) <= 1e-6


def test_refusals_and_zeros(dev, graph_l4):
    """A fourier network is refused; a K = 1 network returns all zeros on the pattern of each level's L."""
    from gcn_fmri_decoding_b200 import synth

    four = build_model(graph_l4, [16, 16], [0, 0], [4, 4], [64, 22], "fourier", "b1relu", dev, perm=graph_l4["perm"])
    with pytest.raises(ValueError, match="fourier"):
        four.graph_saliency(synth.bold_windows(8, seed=1))
    k1 = build_model(graph_l4, [32, 32], [1, 1], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                     perm=graph_l4["perm"])
    out = k1.graph_saliency(synth.bold_windows(20, seed=2), absolute=True)
    assert sorted(out) == [0, 2]
    for lvl, G in out.items():
        assert G.nnz > 0 and not G.data.any()

"""Group saliency maps on the B200: the grouped column sum (``gcnb_group_colsum_f32`` / ``k_group_colsum``) against NumPy
fp64, the grouped mode of ``InputGradient`` against the device's own per-window gradients, every grouped public call
against the fp64 oracle, and the grouped edge maps against the ungrouped calls on each group's windows.  Run on the
B200 box: -m gpu.
"""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import rel_inf
from test_gpu_adjacency_saliency import _decisions
from test_gpu_adjacency_saliency import _reference as _adjacency_reference
from test_gpu_graph_saliency import _reference as _graph_reference
from test_gpu_parity import build_model
from test_gpu_saliency import T, _params
from test_saliency_oracle import network_input_gradient

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SENTINEL = -12345.0


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _colsum(X, group, n_groups, absolute, out):
    from gcn_fmri_decoding_b200 import _lib

    rc = _lib.lib().gcnb_group_colsum_f32(C.c_void_p(X.data_ptr()), X.shape[0], X.shape[1], C.c_void_p(group.data_ptr()),
                                         n_groups, int(absolute), C.c_void_p(out.data_ptr()),
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "gcnb_group_colsum_f32")
    return out


def _patterns(rows, rng):
    """(name, group [rows] int32, n_groups): the group patterns of the kernel test."""
    runs = np.arange(rows) // 48
    minus = rng.randint(0, max(1, rows // 4), rows)
    minus[rng.rand(rows) < 0.2] = -1
    return [("one", np.zeros(rows), 1),
            ("distinct", rng.permutation(rows), rows),
            ("gaps", rng.choice(rng.choice(rows, max(1, rows // 7), replace=False), rows), rows),
            ("runs", runs, int(runs.max()) + 1),
            ("minus_one", minus, max(1, rows // 4)),
            ("beyond", rng.randint(0, rows, rows), max(1, rows // 2))]


def _reference(X64, group, n_groups):
    """fp64 sums and sums of |X| per group, and the groups present."""
    ok = (group >= 0) & (group < n_groups)
    order = np.argsort(group[ok], kind="stable")
    rows = np.flatnonzero(ok)[order]
    g = group[rows]
    present, starts = np.unique(g, return_index=True)
    if len(rows) == 0:
        return present, np.zeros((0, X64.shape[1])), np.zeros((0, X64.shape[1]))
    Xs = X64[rows]
    return present, np.add.reduceat(Xs, starts, axis=0), np.add.reduceat(np.abs(Xs), starts, axis=0)


# ------------------------------------------------------------------------------------------ the kernel
@pytest.mark.parametrize("cols", [1, 33, 4084, 5400])
@pytest.mark.parametrize("rows", [1, 37, 512, 4096, 8192])
def test_group_colsum_matches_fp64(dev, rows, cols):
    """Every group pattern, signed and absolute: each present group within 1e-5 * sum |X| of the fp64 sum, absent
    groups keep the sentinel, repeats are bit-identical."""
    gen = torch.Generator(device=dev).manual_seed(rows * 7919 + cols)
    X = torch.randn((rows, cols), generator=gen, device=dev)
    X64 = X.cpu().numpy().astype(np.float64)
    rng = np.random.RandomState(rows + cols)
    for name, group, n_groups in _patterns(rows, rng):
        group = group.astype(np.int32)
        g = torch.as_tensor(group, device=dev)
        present, ref, ref_abs = _reference(X64, group, n_groups)
        absent = np.setdiff1d(np.arange(n_groups), present)
        for absolute in (False, True):
            out = torch.full((n_groups, cols), SENTINEL, device=dev)
            got = _colsum(X, g, n_groups, absolute, out).cpu().numpy()
            want = ref_abs if absolute else ref
            err = np.abs(got[present] - want) - 1e-5 * ref_abs
            assert err.max(initial=-1.0) <= 0, (name, absolute, err.max())
            assert (got[absent] == SENTINEL).all(), (name, absolute)
            again = _colsum(X, g, n_groups, absolute, torch.full_like(out, SENTINEL))
            assert torch.equal(again, out), (name, absolute)


def test_group_colsum_graph_replay_and_refusals(dev):
    """Captured in a CUDA graph the call replays bit for bit what the eager call gives; bad shapes are refused with
    the reason in the message."""
    from gcn_fmri_decoding_b200 import _lib

    rng = np.random.RandomState(3)
    X = T(rng.randn(512, 5400), dev)
    g = torch.as_tensor(rng.randint(-1, 22, 512).astype(np.int32), device=dev)
    eager = _colsum(X, g, 512, True, torch.full((512, 5400), SENTINEL, device=dev)).clone()
    out = torch.full((512, 5400), SENTINEL, device=dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _colsum(X, g, 512, True, out)
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
    # buffers large enough for every shape below, so that only the argument checks stand between a bad shape and a run
    big = torch.zeros((8193, 33), device=dev)
    gbig = torch.zeros(8193, dtype=torch.int32, device=dev)
    obig = torch.zeros((8193, 33), device=dev)
    lib = _lib.lib()
    for (rows, cols, n_groups), msg in (((8193, 33, 1), "rows = 8193"), ((0, 33, 1), "rows = 0"),
                                        ((4, 0, 1), "cols = 0"), ((4, 33, 5), "n_groups = 5"),
                                        ((4, 33, 0), "n_groups = 0")):
        rc = lib.gcnb_group_colsum_f32(C.c_void_p(big.data_ptr()), rows, cols, C.c_void_p(gbig.data_ptr()), n_groups, 0,
                                       C.c_void_p(obig.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        with pytest.raises(ValueError, match=msg):
            _lib.check(rc, "gcnb_group_colsum_f32")


# ------------------------------------------------------------------------------------------ InputGradient, grouped
def _per_window_sums(model, xraw, ids, G, target=None, absolute=False):
    """The device's per-window saliency maps (the ungrouped call) summed per group in fp64."""
    grads, targets = model.saliency(xraw, target=target)
    g64 = grads.astype(np.float64)
    if absolute:
        g64 = np.abs(g64)
    ids = targets if ids is None else ids
    out = np.zeros((G,) + grads.shape[1:])
    np.add.at(out, ids, g64)
    return out, targets


def _check_grouped_input(model, xraw, groups, G, target=None, absolute=False):
    sums, counts, targets = model.saliency(xraw, target=target, groups=groups, absolute=absolute)
    ids = None if isinstance(groups, str) else groups
    ref, ref_targets = _per_window_sums(model, xraw, ids, G, target, absolute)
    assert sums.dtype == np.float64 and sums.shape == ref.shape
    assert counts.dtype == np.int64 and counts.tolist() == np.bincount(
        ref_targets if ids is None else ids, minlength=G).tolist()
    assert np.array_equal(targets, ref_targets)
    assert rel_inf(sums, ref) <= 1e-5, rel_inf(sums, ref)
    return sums


def _config2(graph, dev, B, **kw):
    model = build_model(graph, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph["perm"], **kw)
    model.batch_size = B
    return model


def test_input_gradient_grouped_config2(dev, graph_l4):
    """Config 2 at B = 512 over 889 windows (a padded last batch): groups = labels, by target with target=None, and runs
    of 48 windows per id; absolute by labels."""
    from gcn_fmri_decoding_b200 import synth

    model = _config2(graph_l4, dev, 512)
    xraw = synth.bold_windows(889, seed=51)
    labels = synth.labels(889, seed=51)
    _check_grouped_input(model, xraw, labels, int(labels.max()) + 1)
    _check_grouped_input(model, xraw, "target", 22)
    runs = np.arange(889) // 48
    _check_grouped_input(model, xraw, runs, int(runs.max()) + 1)
    _check_grouped_input(model, xraw, labels, int(labels.max()) + 1, absolute=True)
    _check_grouped_input(model, xraw, "target", 22, target=labels, absolute=True)


def test_input_gradient_grouped_config1_and_fourier(dev, graph_l1, graph_l4):
    """Config 1 at B = 128 (300 windows), and a two-layer fourier network (the sum runs after ops.unpermute)."""
    from gcn_fmri_decoding_b200 import synth

    m1 = build_model(graph_l1, [32] * 6, [5] * 6, [1] * 6, [512, 256, 22], "chebyshev5", "b2relu", dev,
                     perm=graph_l1["perm"])
    m1.batch_size = 128
    x1 = synth.bold_windows(300, seed=52)
    ids = np.random.RandomState(1).randint(0, 9, 300)
    _check_grouped_input(m1, x1, ids, int(ids.max()) + 1)
    _check_grouped_input(m1, x1, "target", 22, absolute=True)
    four = build_model(graph_l4, [16, 16], [0, 0], [4, 4], [64, 22], "fourier", "b1relu", dev, perm=graph_l4["perm"])
    x4 = synth.bold_windows(40, seed=53)
    ids = np.random.RandomState(2).randint(0, 5, 40)
    _check_grouped_input(four, x4, ids, int(ids.max()) + 1)
    _check_grouped_input(four, x4, ids, int(ids.max()) + 1, absolute=True)


def test_capacity_does_not_change_the_sums(dev, graph_l4):
    """512 windows in 4 groups: capacity n_groups = 512 gives bit for bit the sums of n_groups = 4; an ungrouped call
    returns the same bytes before and after grouped calls on the same object (separate graph-cache keys)."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.saliency import GraphGradient, InputGradient

    model = _config2(graph_l4, dev, 512)
    x = T(synth.bold_windows(512, seed=54), dev)
    g = torch.as_tensor(np.random.RandomState(4).randint(0, 4, 512).astype(np.int32), device=dev)
    ig = InputGradient(model)
    before = ig(x, gather=True)[0].clone()
    small = ig(x, gather=True, group=g, n_groups=4)[0].clone()
    large = ig(x, gather=True, group=g, n_groups=512)[0]
    assert torch.equal(small, large[:4])
    assert torch.equal(ig(x, gather=True)[0], before)
    eager = InputGradient(model, use_cuda_graph=False)(x, gather=True, group=g, n_groups=4)[0]
    assert torch.equal(eager, small)
    gg = GraphGradient(model)
    before = {k: v.clone() for k, v in gg(x, gather=True)[0].items()}
    small = {k: tuple(a.clone() for a in v) for k, v in gg(x, gather=True, group=g, n_groups=4)[0].items()}
    large = gg(x, gather=True, group=g, n_groups=512)[0]
    for k, (a, b) in small.items():
        assert torch.equal(a, large[k][0][:4]) and torch.equal(b, large[k][1][:4])
    for k, v in gg(x, gather=True)[0].items():
        assert torch.equal(v, before[k])


# ------------------------------------------------------------------------------------------ end to end vs the oracle
def _oracle_setup(dev, graph_l4):
    from gcn_fmri_decoding_b200 import synth

    model = _config2(graph_l4, dev, 64)
    xraw = synth.bold_windows(150, seed=55)
    ids = np.random.RandomState(5).choice([0, 2, 5], 150)
    target = model.predict(xraw).astype(np.int64)
    dec, masks = _decisions(model, xraw, True)
    return model, xraw, ids, target, dec, masks


def _subset(dec, masks, sel):
    return [{k: v[sel] for k, v in d.items()} for d in dec], [m_[sel] for m_ in masks]


def test_grouped_saliency_matches_oracle(dev, graph_l4):
    model, xraw, ids, target, dec, masks = _oracle_setup(dev, graph_l4)
    params, fcs = _params(model)
    perm = model.perm.cpu().numpy()
    for absolute in (False, True):
        sums, counts, targets = model.saliency(xraw, groups=ids, absolute=absolute)
        assert np.array_equal(targets, target) and counts.tolist() == np.bincount(ids, minlength=6).tolist()
        ref = np.zeros_like(sums)
        g = network_input_gradient(xraw, model.L, params, fcs, target, perm, xraw.shape[1], filter=model.filter_name,
                                   brelu=model.brelu_name, conv_decisions=dec, head_masks=masks)
        np.add.at(ref, ids, np.abs(g) if absolute else g)
        assert rel_inf(sums, ref) <= 1e-4, (absolute, rel_inf(sums, ref))


def test_grouped_graph_saliency_matches_oracle(dev, graph_l4):
    model, xraw, ids, target, dec, masks = _oracle_setup(dev, graph_l4)
    perm = model.perm.cpu().numpy()
    got, counts = model.graph_saliency(xraw, groups=ids, absolute=True)
    assert counts.tolist() == np.bincount(ids, minlength=6).tolist()
    for g in range(6):
        sel = ids == g
        if not sel.any():
            for mats in got.values():
                assert mats[g].nnz == 0 or not mats[g].data.any()
            continue
        ref = _graph_reference(model, xraw[sel], target[sel], *_subset(dec, masks, sel), True)
        for lvl, mats in got.items():
            R = ref[lvl]
            if lvl == 0:
                M_in = xraw.shape[1]
                real = perm < M_in
                Rr = np.zeros((M_in, M_in))
                Rr[np.ix_(perm[real], perm[real])] = R[np.ix_(real, real)]
                R = Rr
            assert rel_inf(mats[g].toarray(), R) <= 1e-4, (g, lvl, rel_inf(mats[g].toarray(), R))


def test_grouped_adjacency_saliency_matches_oracle(dev, graph_l4):
    from test_adjacency_saliency_oracle import edges_of

    model, xraw, ids, target, dec, masks = _oracle_setup(dev, graph_l4)
    A = sp.csr_matrix(graph_l4["A"])
    i, j = edges_of(A)
    got, counts = model.adjacency_saliency(xraw, A, groups=ids)
    assert len(got) == 6 and counts.tolist() == np.bincount(ids, minlength=6).tolist()
    for g in (0, 2, 5):
        sel = ids == g
        ref = _adjacency_reference(model, graph_l4, xraw[sel], target[sel], *_subset(dec, masks, sel), False)
        assert (got[g] != got[g].T).nnz == 0
        assert rel_inf(np.asarray(got[g][i, j]).ravel(), ref) <= 1e-4


# ------------------------------------------------------------------------------------------ grouped vs ungrouped
def test_grouped_edge_maps_match_ungrouped_calls(dev, graph_l4):
    """Each group's map equals the ungrouped call on that group's windows; signed, the sum over groups equals the
    ungrouped call on all windows; by target the groups are the predicted classes."""
    from gcn_fmri_decoding_b200 import synth

    model = _config2(graph_l4, dev, 512)
    xraw = synth.bold_windows(889, seed=56)
    labels = synth.labels(889, seed=56)
    A = sp.csr_matrix(graph_l4["A"])
    for absolute in (False, True):
        got, counts = model.graph_saliency(xraw, groups=labels, absolute=absolute)
        adj, _ = model.adjacency_saliency(xraw, A, groups=labels, absolute=absolute)
        for g in np.unique(labels):
            sel = labels == g
            one = model.graph_saliency(xraw[sel], absolute=absolute)
            for lvl, mats in got.items():
                assert rel_inf(mats[g].toarray(), one[lvl].toarray()) <= 1e-5, (g, lvl, absolute)
            ref = model.adjacency_saliency(xraw[sel], A, absolute=absolute)
            assert (adj[g] != adj[g].T).nnz == 0
            assert rel_inf(adj[g].toarray(), ref.toarray()) <= 1e-5, (g, absolute)
        if not absolute:
            whole = model.graph_saliency(xraw)
            for lvl, mats in got.items():
                assert rel_inf(sum(m_.toarray() for m_ in mats), whole[lvl].toarray()) <= 1e-5
            whole = model.adjacency_saliency(xraw, A)
            assert rel_inf(sum(m_.toarray() for m_ in adj), whole.toarray()) <= 1e-5
    pred = model.predict(xraw).astype(np.int64)
    by_target, counts = model.adjacency_saliency(xraw, A, groups="target")
    assert len(by_target) == 22 and counts.tolist() == np.bincount(pred, minlength=22).tolist()
    for g in np.unique(pred)[:3]:
        ref = model.adjacency_saliency(xraw[pred == g], A, target=pred[pred == g])
        assert rel_inf(by_target[g].toarray(), ref.toarray()) <= 1e-5

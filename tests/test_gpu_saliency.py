"""Saliency maps on the B200 against the fp64 oracle: the input-gradient-only layer call (``ops.cheb_dx``: the tcgen05
adjoint of any input width, un-permuting in its store, and its fallbacks) and the whole schedule
(``saliency.InputGradient`` / ``cgcnn.saliency``).  Run on the B200 box: -m gpu.

The fp32 kernels decide every max-pool arg-max and every ReLU (conv and FC) on their own; the oracle is routed through
the device's decisions (``decisions`` / ``head_masks``) so that near-ties at large batches do not decide the comparison.
"""
import ctypes as C
import re

import numpy as np
import pytest

from conftest import rel_inf
from oracle import layers_np as O
from test_gpu_parity import build_model
from test_gpu_saved_basis import run_images
from test_saliency_oracle import network_input_gradient, permute_rows, unpermute_rows

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def T(a, dev, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)


def _perm_with_fakes(M, n_fake, seed):
    """A permutation of [0, M) whose entries >= M - n_fake are fake vertices (as Graclus pads a graph)."""
    return np.random.RandomState(seed).permutation(M).astype(np.int32)


# ------------------------------------------------------------------------------------------ the layer
# (level of the 400-vertex test graph, Fin, algo): the tcgen05 adjoint under AUTO, k_cheb_bwd_fused on a graph it holds,
# the general path on the benchmark's first-layer graph
_A, _F, _G = 0, 2, 1
LAYER_CASES = [(0, Fin, _A) for Fin in (9, 13, 15, 16, 31)] + [(2, Fin, _F) for Fin in (9, 15, 16)] + \
              [(0, Fin, _G) for Fin in (15, 31)]


@pytest.mark.parametrize("lvl,Fin,algo", LAYER_CASES)
@pytest.mark.parametrize("with_perm", [False, True])
def test_cheb_dx_matches_oracle(dev, graph_l4, lvl, Fin, algo, with_perm):
    """ops.cheb_dx against oracle.chebyshev5_bwd's dx (K = 5, p = 4, ReLU, 32 filters), with and without a permutation
    with fake vertices, with and without operator images; un-permuted through that permutation by the oracle."""
    from gcn_fmri_decoding_b200 import _lib, ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    L = graph_l4["L"][lvl]
    M, Fout, K, p = L.shape[0], 32, 5, 4
    pl = GraphPlan(L, dev)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    text, _ = _lib.describe_dx(1, M, pl.nnz, Fin, Fout, K, p, algo)
    route = text.split(":")[0]
    assert route == {_A: "tcgen05 adjoint only", _F: "fused dx", _G: "general path"}[algo], text
    if algo == _A:  # at least 3 tiles per CTA of the persistent adjoint kernel
        wpt = int(re.search(r"(\d+) windows/tile", text).group(1))
        B = 3 * sms * wpt + wpt // 2 + 1
        tiles = int(re.search(r"(\d+) tiles$", _lib.describe_dx(B, M, pl.nnz, Fin, Fout, K, p, algo)[0]).group(1))
        assert tiles // sms >= 3, tiles
    else:
        B = 67
    if with_perm:
        perm = graph_l4["perm"].astype(np.int32) if lvl == 0 else _perm_with_fakes(M, 10, Fin)
        M_in = 360 if lvl == 0 else M - 10
    else:
        perm, M_in = None, M
    rng = np.random.RandomState(10 * Fin + lvl)
    x = rng.randn(B, M_in, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * (0.4 / np.sqrt(Fin * K))).astype(np.float32)
    b = (rng.randn(Fout) * 0.1).astype(np.float32)
    dy = rng.randn(B, M // p, Fout).astype(np.float32)
    pt = T(perm, dev, torch.int32) if perm is not None else None
    y, am, _, _ = ops.cheb_fwd_mean(T(x, dev), pt, pl.rowptr, pl.col, pl.val, T(W, dev), T(b, dev), K, p,
                                    ops.BIAS_PER_FILTER, True, _lib.ALGO_AUTO, False)
    # the oracle, routed through the device's decisions, in chunks of windows
    ya, ama = y.cpu().numpy(), am.cpu().numpy()
    ref = np.empty((B, M_in, Fin))
    for s in range(0, B, 256):
        sl = slice(s, min(B, s + 256))
        xp = permute_rows(x[sl].astype(np.float64), perm, M_in) if perm is not None else x[sl].astype(np.float64)
        dz = O.mpool1_bwd(dy[sl].astype(np.float64) * (ya[sl] > 0), ama[sl], p, M)
        g, _ = O.chebyshev5_bwd(xp, L, W, K, dz, np.float64)
        ref[sl] = unpermute_rows(g, perm, M_in) if perm is not None else g
    for use in (True, False):
        args = (pt, M_in, y, am, T(dy, dev), False, *pl.tensors(), T(W, dev), K, p, True, algo)
        got = run_images(use, lambda: ops.cheb_dx(T(x, dev), *args)).cpu().numpy()
        assert got.shape == ref.shape
        assert rel_inf(got, ref) <= TOL, (route, use, rel_inf(got, ref))
        if algo != _G:  # these routes never read x
            again = run_images(use, lambda: ops.cheb_dx(None, *args)).cpu().numpy()
            assert np.array_equal(again, got)
    if algo == _G:
        with pytest.raises(ValueError, match="general path"):
            ops.cheb_dx(None, pt, M_in, y, am, T(dy, dev), False, *pl.tensors(), T(W, dev), K, p, True, algo)


# ------------------------------------------------------------------------------------------ the network
def _device_decisions(model, ig, x, gather):
    """The device's conv decisions (pooled arg-max, y > 0) and FC masks (activation > 0) of InputGradient's forward: the
    same launches with the same arguments (deterministic kernels)."""
    from gcn_fmri_decoding_b200 import _lib, ops

    lib = _lib.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr())
    dec, h, h0 = [], x, None
    with torch.no_grad():
        for i in range(len(model.p)):
            perm = model.perm if (gather and i == 0) else None
            if model.filter_name == "fourier":
                hin = ops.perm_gather(h, perm) if perm is not None else h
                sp = model._spectral_plan(model.L[i])
                y, am = ops.spectral_fwd(hin, sp.Ut, model.conv_weights[i], model.conv_bias[i], model.p[i],
                                         model._bias_mode(), True, True)
            else:
                pl = model._plan(model.L[i])
                y, am, h0, _ = ops.cheb_fwd_mean(h, perm, pl.rowptr, pl.col, pl.val, model.conv_weights[i],
                                                 model.conv_bias[i], model.K[i], model.p[i], model._bias_mode(), True,
                                                 model.algo, False)
            dec.append(dict(argmax=am.cpu().numpy() if model.p[i] > 1 else np.zeros(y.shape, np.uint8),
                            relu=(y > 0).cpu().numpy()))
            h = y
        if model.filter_name == "fourier":
            h0 = ops.mean_f_fwd(h)
        masks, a = [], h0
        for i in range(len(model.M) - 1):
            W = model.fc_weights[i]
            out = torch.empty((a.shape[0], W.shape[1]), device=x.device)
            _lib.check(lib.gcnb_gemm_epilogue_f32(vp(a), vp(W), vp(out), vp(model.fc_bias[i]), a.shape[0], W.shape[1],
                                                  W.shape[0], a.shape[1], W.shape[1], W.shape[1], 0, 0,
                                                  _lib.EPI_RELU_DROPOUT, None, 0, 1.0, 0, vp(ig._step), stream), "gemm")
            masks.append((out > 0).cpu().numpy())
            a = out
    return dec, masks


def _params(model):
    sd = {k: v.astype(np.float64) for k, v in model.state_dict_tf().items()}
    n = len(model.p)
    params = [dict(W=sd["conv%d/weights" % (i + 1)], b=sd["conv%d/bias" % (i + 1)].reshape(
        (-1, model.F[i]) if model.brelu_name == "b2relu" else (model.F[i],)), K=model.K[i], p=model.p[i]) for i in range(n)]
    names = ["fc%d" % (i + 1) for i in range(len(model.M) - 1)] + ["logits"]
    return params, [(sd[s + "/weights"], sd[s + "/bias"]) for s in names]


def _check_network(dev, model, xraw, chunk=256):
    """InputGradient (CUDA graph) on raw windows against network_input_gradient with the device's decisions."""
    from gcn_fmri_decoding_b200.saliency import InputGradient

    ig = InputGradient(model)
    x = T(xraw, dev)
    grad, logits, target = ig(x, gather=True)
    grad, target = grad.cpu().numpy(), target.cpu().numpy()
    assert grad.shape == xraw.shape
    assert np.array_equal(target, logits.argmax(1).cpu().numpy())
    dec, masks = _device_decisions(model, ig, x, True)
    params, fcs = _params(model)
    perm = model.perm.cpu().numpy()
    err, ref_max = 0.0, 0.0
    for s in range(0, xraw.shape[0], chunk):
        sl = slice(s, min(xraw.shape[0], s + chunk))
        ref = network_input_gradient(xraw[sl], model.L, params, fcs, target[sl], perm, xraw.shape[1],
                                       filter=model.filter_name, brelu=model.brelu_name,
                                       conv_decisions=[{k: v[sl] for k, v in d.items()} for d in dec],
                                       head_masks=[m_[sl] for m_ in masks])
        err = max(err, float(np.abs(grad[sl] - ref).max()))
        ref_max = max(ref_max, float(np.abs(ref).max()))
    assert err / ref_max <= TOL, err / ref_max
    return ig, x, grad


@pytest.mark.parametrize("B", [512, 2048, 889])
def test_config2_network_matches_oracle(dev, graph_l4, B):
    """The benchmark's config-2 network (360 ROIs -> 400 -> 100 -> 25 vertices, 15 TRs) at B = 512, 2048 and a ragged
    889; conv 1's input gradient through the tcgen05 adjoint with the Graclus un-permutation fused into its store."""
    from gcn_fmri_decoding_b200 import _lib, synth

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    for i, Fin in ((0, 15), (1, 32)):
        pl = model._plan(model.L[i])
        assert _lib.describe_dx(B, pl.M, pl.nnz, Fin, 32, 5, 4)[0].startswith("tcgen05 adjoint only")
    _check_network(dev, model, synth.bold_windows(B, seed=B))


def test_config1_and_fourier_networks_match_oracle(dev, graph_l1, graph_l4):
    """The config-1 six-layer b2relu ChebyNet (372 vertices, p = 1) at B = 128, and a two-layer fourier network."""
    from gcn_fmri_decoding_b200 import synth

    m1 = build_model(graph_l1, [32] * 6, [5] * 6, [1] * 6, [512, 256, 22], "chebyshev5", "b2relu", dev,
                     perm=graph_l1["perm"])
    _check_network(dev, m1, synth.bold_windows(128, seed=3))
    m2 = build_model(graph_l4, [16, 16], [0, 0], [4, 4], [64, 22], "fourier", "b1relu", dev, perm=graph_l4["perm"])
    _check_network(dev, m2, synth.bold_windows(40, seed=4))


def test_agrees_with_autograd_and_replays_bit_identically(dev, graph_l4):
    """Against torch.autograd.grad through cgcnn.forward (the same forward kernels, hence the same decisions) to 1e-5; the
    CUDA-graph replay equals the eager schedule bit for bit, and two runs are bit-identical."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.saliency import InputGradient

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    x = T(synth.bold_windows(64, seed=8), dev)
    ig = InputGradient(model)
    g1, lg, t = (a.clone() for a in ig(x, gather=True))
    g2 = ig(x, gather=True)[0].clone()
    eager = InputGradient(model, use_cuda_graph=False)(x, gather=True)[0]
    assert torch.equal(g1, g2) and torch.equal(g1, eager)
    given = ig(x, target=t, gather=True)[0]
    assert torch.equal(given, g1)
    xa = x.clone().requires_grad_(True)
    logits = model(xa)
    (ga,) = torch.autograd.grad(logits.gather(1, t.view(-1, 1)).sum(), xa)
    assert rel_inf(g1.cpu().numpy(), ga.cpu().numpy()) <= 1e-5, rel_inf(g1.cpu().numpy(), ga.cpu().numpy())


def test_cgcnn_saliency_batches_like_predict(dev, graph_l4):
    """cgcnn.saliency: batches of batch_size with a zero-padded last one, target=None = prediction(), a given target is
    honoured, the ambiguous input layout is refused and so is a perm that is not a permutation."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.saliency import InputGradient

    model = build_model(graph_l4, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev,
                        perm=graph_l4["perm"])
    model.batch_size = 512
    data = synth.bold_windows(889, seed=21)
    grad, target = model.saliency(data)
    assert grad.shape == data.shape and grad.dtype == np.float32 and target.dtype == np.int64
    assert np.array_equal(target, model.predict(data).astype(np.int64))
    padded = np.zeros((512,) + data.shape[1:], np.float32)
    padded[:889 - 512] = data[512:]
    g_last = InputGradient(model)(T(padded, dev), gather=True)[0].cpu().numpy()
    assert np.array_equal(grad[512:], g_last[:889 - 512])
    other = (target + 1) % 22
    g_other, t_other = model.saliency(data[:100], target=other[:100])
    assert np.array_equal(t_other, other[:100]) and not np.array_equal(g_other, grad[:100])
    model.n_input_vertices = model.L[0].shape[0]
    with pytest.raises(ValueError, match="gather"):
        model.saliency(np.zeros((4, 400, 15), np.float32))
    model.n_input_vertices = 360
    bad = model.perm.clone()
    bad[0] = bad[1]
    model.perm = bad
    with pytest.raises(ValueError, match="permutation"):
        model.saliency(data[:4])

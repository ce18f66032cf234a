"""Parity of the CUDA path (through the C ABI) against the oracle.  Run on the B200 box: -m gpu.

Bars (BASELINE.md section 4):
* integer work -- permutation/padding, pooled arg-max bytes: bit-exact;
* floating point -- ||y - y_ref||_inf / ||y_ref||_inf <= 1e-4 against the fp64 oracle
  (TOL below); the as-run fp32 oracle's own distance to fp64 is the noise floor.
Arg-max note: where the fp64 window maximum leads the runner-up by less than fp32 rounding
noise (ARGMAX_GAP, relative to the tensor's max), either index is a correct fp32 answer; such
windows are counted, required to be rare, and excluded from the exact comparison.
"""
import numpy as np
import pytest

from conftest import rel_inf
from oracle import layers_np as O

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-4
ARGMAX_GAP = 2e-5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def T(a, dev, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)


def algos_for(B, M, nnz, Fin, Fout, K, p, backward=False, need_dx=True):
    from gcn_fmri_decoding_b200 import _lib

    out = [_lib.ALGO_GENERAL]
    if _lib.lib().gcnb_cheb_fused_supported(B, M, nnz, Fin, Fout, K, p, int(backward), int(need_dx)):
        out.append(_lib.ALGO_FUSED)
    return out


def check_argmax(got, a64, p, name=""):
    """got: uint8 [B, Mo, F]; a64: fp64 pre-pool activation [B, M, F] (M % p == 0)."""
    B, M, F = a64.shape
    win = a64.reshape(B, M // p, p, F)
    ref = win.argmax(2)
    srt = np.sort(win, axis=2)
    gap = srt[:, :, -1, :] - srt[:, :, -2, :]
    scale = np.abs(a64).max()
    bad = got.astype(np.int64) != ref
    # a disagreement is only admissible on a (near-)tie that is not an exact tie
    assert not np.any(bad & (gap > ARGMAX_GAP * scale)), name
    assert not np.any(bad & (gap == 0)), name  # exact ties (e.g. all-zero after ReLU): first index, bit-exact
    assert bad.mean() < 1e-3, name


def run_layer(dev, L, x, W, b, K, p, brelu, algo, perm=None, dy=None, need_dx=True):
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    pl = GraphPlan(L, dev)
    mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
    xt = T(x, dev).requires_grad_(need_dx)
    Wt = T(W, dev).requires_grad_(True)
    bt = T(b, dev).requires_grad_(True)
    pt = None if perm is None else T(perm, dev, torch.int32)
    y, am = ops.cheb_fwd(xt, pt, *pl.tensors(), Wt, bt, K, p, mode, True, True, algo)
    out = dict(y=y.detach().cpu().numpy(), argmax=am.cpu().numpy())
    if dy is not None:
        y.backward(T(dy, dev))
        out.update(dW=Wt.grad.cpu().numpy(), db=bt.grad.cpu().numpy().reshape(np.shape(b)))
        if need_dx:
            out["dx"] = xt.grad.cpu().numpy()
    return out


# ------------------------------------------------------------------------------------------ golden cases
def test_golden_layer_cases(dev, graph_l4, layer_cases):
    for name, c in layer_cases.items():
        filt, brelu = str(c["kind"]).split("/")
        if filt == "fourier":
            continue
        lvl, B, Fin, Fout, K, p = (int(v) for v in c["meta"])
        L = graph_l4["L"][lvl]
        for algo in algos_for(B, L.shape[0], graph_l4["Lt"][lvl].nnz, Fin, Fout, K, p, True, True):
            r = run_layer(dev, L, c["x"], c["W"], c["b"], K, p, brelu, algo, dy=c["dy"])
            tag = "%s algo=%d" % (name, algo)
            assert rel_inf(r["y"], c["y64"]) <= TOL, tag
            assert rel_inf(r["dW"], c["dW64"]) <= TOL, tag
            assert rel_inf(r["db"], c["db64"]) <= TOL, tag
            assert rel_inf(r["dx"], c["dx64"]) <= TOL, tag
            if p > 1:
                # the fp64 pre-activation from the oracle (test_oracle.py pins it to the stored y64 and argmax)
                _, tr = O.conv_stack(c["x"], [L], [dict(W=c["W"], b=c["b"], K=K, p=p)], filter=filt, brelu=brelu,
                                     dtype=np.float64, keep=True)
                z64 = tr[0]["z"]
                a64 = O.b1relu(z64, c["b"]) if brelu == "b1relu" else O.b2relu(z64, c["b"])
                check_argmax(r["argmax"], a64, p, tag)


def test_golden_spectral_cases(dev, layer_cases):
    from gcn_fmri_decoding_b200 import ops

    for name, c in layer_cases.items():
        filt, brelu = str(c["kind"]).split("/")
        if filt != "fourier":
            continue
        lvl, B, Fin, Fout, K, p = (int(v) for v in c["meta"])
        mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
        xt, Wt, bt = (T(c[k], dev).requires_grad_(True) for k in ("x", "W", "b"))
        y, am = ops.spectral_fwd(xt, T(c["Ut"], dev), Wt, bt, p, mode, True, True)
        y.backward(T(c["dy"], dev))
        # reference values recomputed in fp64 from the stored fp32 basis (eigenvectors are host-BLAS dependent)
        pr = dict(W=c["W"], b=c["b"], K=K, p=p)
        z = O.filter_in_fourier(c["x"], c["Ut"], c["W"], np.float64)
        a = O.b1relu(z, c["b"]) if brelu == "b1relu" else O.b2relu(z, c["b"])
        yref, amref = O.mpool1(a, p, with_argmax=True)
        dz, db = O.brelu_bwd(O.mpool1_bwd(c["dy"].astype(np.float64), amref, p, a.shape[1]), a, brelu == "b2relu")
        dx, dW = O.fourier_bwd(c["x"], c["Ut"], c["W"], dz, np.float64)
        assert rel_inf(y.detach().cpu().numpy(), yref) <= TOL, name
        assert rel_inf(xt.grad.cpu().numpy(), dx) <= TOL, name
        assert rel_inf(Wt.grad.cpu().numpy(), dW) <= TOL, name
        assert rel_inf(bt.grad.cpu().numpy().reshape(db.shape), db) <= TOL, name
        if p > 1:
            check_argmax(am.cpu().numpy(), a, p, name)


# ------------------------------------------------------------------------------------------ live oracle sweeps
SWEEP = [
    # lvl, B, Fin, Fout, K, p, brelu
    (0, 6, 15, 32, 5, 4, "b1relu"),   # config 2, layer 1 shape
    (2, 9, 32, 32, 5, 4, "b1relu"),   # config 2, layer 2 shape
    (0, 3, 15, 32, 5, 1, "b2relu"),   # production-like b2relu, no pooling
    (0, 4, 15, 32, 2, 4, "b1relu"),   # config 3a, K=2
    (0, 4, 15, 32, 1, 4, "b1relu"),   # K=1 "firstorder" (SURVEY D1)
    (2, 5, 32, 32, 2, 4, "b2relu"),
    (1, 3, 7, 24, 10, 2, "b1relu"),
    (3, 5, 32, 16, 20, 2, "b2relu"),
    (4, 7, 3, 8, 25, 1, "b1relu"),
    (2, 1, 1, 1, 3, 1, "b1relu"),     # degenerate widths
    (2, 2, 33, 40, 3, 2, "b1relu"),   # widths that are not multiples of 8
    (1, 2, 64, 64, 3, 8, "b1relu"),
    (3, 40, 32, 32, 3, 2, "b1relu"),  # vertex-major rows wider than one TMA column chunk (B*Fin = 1280 floats)
    (1, 8, 16, 32, 12, 1, "b2relu"),  # general path: TMA SpMM + all three tensor-core contractions, K=12
]


@pytest.mark.parametrize("lvl,B,Fin,Fout,K,p,brelu", SWEEP)
def test_cheb_layer_vs_oracle(dev, graph_l4, lvl, B, Fin, Fout, K, p, brelu):
    rng = np.random.RandomState(100 + lvl * 7 + K)
    L = graph_l4["L"][lvl]
    M = L.shape[0]
    x = rng.randn(B, M, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * 0.2).astype(np.float32)
    b = (0.2 + 0.1 * rng.randn(*((M, Fout) if brelu == "b2relu" else (Fout,)))).astype(np.float32)
    dy = rng.randn(B, M // p, Fout).astype(np.float32)
    pr = [dict(W=W, b=b, K=K, p=p)]
    y64, tr = O.conv_stack(x, [L], pr, brelu=brelu, dtype=np.float64, keep=True)
    dx64, g64 = O.conv_stack_bwd(tr, [L], pr, dy, brelu=brelu, dtype=np.float64, first_needs_dx=True)
    y32 = O.conv_stack(x, [L], pr, brelu=brelu, dtype=np.float32)
    for algo in algos_for(B, M, graph_l4["Lt"][lvl].nnz, Fin, Fout, K, p, True, True):
        r = run_layer(dev, L, x, W, b, K, p, brelu, algo, dy=dy)
        tag = "algo=%d" % algo
        err = rel_inf(r["y"], y64)
        assert err <= TOL, (tag, err, "fp32 oracle noise floor", rel_inf(y32, y64))
        assert rel_inf(r["dW"], g64[0]["dW"]) <= TOL, tag
        assert rel_inf(r["db"], g64[0]["db"]) <= TOL, tag
        assert rel_inf(r["dx"], dx64) <= TOL, tag
        if p > 1:
            check_argmax(r["argmax"], tr[0]["a"], p, tag)
        # no-dx variant (layer 1 of a network): same dW/db (the tile geometry, hence the summation order, may differ)
        r2 = run_layer(dev, L, x, W, b, K, p, brelu, algo, dy=dy, need_dx=False)
        assert rel_inf(r2["dW"], r["dW"]) <= 1e-5 and rel_inf(r2["db"], r["db"]) <= 1e-5, tag
        # and the backward is run-to-run deterministic (no float atomics anywhere)
        r3 = run_layer(dev, L, x, W, b, K, p, brelu, algo, dy=dy)
        assert np.array_equal(r3["dW"], r["dW"]) and np.array_equal(r3["db"], r["db"]) and np.array_equal(r3["dx"], r["dx"]), tag


@pytest.mark.parametrize("levels", [0, 1, 2, 4])
def test_fused_perm_gather_all_graph_sizes(dev, levels):
    """M in {360, 372, 384, 400}: raw [B,360,15] windows, perm_data_3d fused into the layer-1 load."""
    from gcn_fmri_decoding_b200 import graclus, synth

    A, gs, perm, L = synth.brain_graph(levels)
    M = L[0].shape[0]
    rng = np.random.RandomState(5)
    xraw = synth.bold_windows(5, seed=3)
    W = (rng.randn(15 * 5, 32) * 0.2).astype(np.float32)
    b = np.full(32, 0.2, np.float32)
    p = 2 if levels else 1
    xp = graclus.perm_data_3d(xraw, perm).astype(np.float32) if perm is not None else xraw
    y64, tr = O.conv_stack(xp, [L[0]], [dict(W=W, b=b, K=5, p=p)], dtype=np.float64, keep=True)
    for algo in algos_for(5, M, 3684, 15, 32, 5, p):
        if perm is None:
            r = run_layer(dev, L[0], xraw, W, b, 5, p, "b1relu", algo)
        else:
            r = run_layer(dev, L[0], xraw, W, b, 5, p, "b1relu", algo, perm=np.asarray(perm))
        assert rel_inf(r["y"], y64) <= TOL, (levels, algo)
        if p > 1:
            check_argmax(r["argmax"], tr[0]["a"], p)


def test_perm_gather_bit_exact(dev, graph_l4):
    import os

    from conftest import GOLDEN
    from gcn_fmri_decoding_b200 import ops

    z = np.load(os.path.join(GOLDEN, "ref_fourier_perm.npz"))
    got = ops.perm_gather(T(z["x"], dev), T(graph_l4["perm"], dev, torch.int32)).cpu().numpy()
    assert got.dtype == np.float32 and np.array_equal(got, z["x_perm"].astype(np.float32))
    with pytest.raises(ValueError):
        ops.perm_gather(T(z["x"], dev), T(np.arange(10), dev, torch.int32))


@pytest.mark.parametrize("M,p", [(10, 4), (7, 2), (16, 8), (5, 1), (33, 16)])
def test_standalone_brelu_mpool_ragged(dev, M, p):
    """b1relu/b2relu and mpool1 one by one, including ragged M (tf SAME padding)."""
    from gcn_fmri_decoding_b200 import ops

    rng = np.random.RandomState(M * 10 + p)
    x = rng.randn(3, M, 6).astype(np.float32)
    b1 = rng.randn(6).astype(np.float32)
    b2 = rng.randn(M, 6).astype(np.float32)
    for b, mode, per_vertex in ((b1, ops.BIAS_PER_FILTER, False), (b2, ops.BIAS_PER_VERTEX, True)):
        xt, bt = T(x, dev).requires_grad_(True), T(b, dev).requires_grad_(True)
        a = ops.brelu_fwd(xt, bt, mode)
        y, am = ops.mpool_fwd(a, p)
        a_ref = O.b2relu(x, b) if per_vertex else O.b1relu(x, b)
        y_ref, am_ref = O.mpool1(a_ref, p, with_argmax=True)
        assert np.array_equal(a.detach().cpu().numpy(), a_ref)  # one add and one max: bit-exact
        assert np.array_equal(y.detach().cpu().numpy(), y_ref)
        if p > 1:
            assert np.array_equal(am.cpu().numpy(), am_ref)
        dy = rng.randn(*y_ref.shape).astype(np.float32)
        y.backward(T(dy, dev))
        da = O.mpool1_bwd(dy, am_ref, p, M) if p > 1 else dy
        dz, db = O.brelu_bwd(da.astype(np.float64), a_ref, per_vertex)
        assert rel_inf(xt.grad.cpu().numpy(), dz) <= 1e-6
        assert rel_inf(bt.grad.cpu().numpy(), db) <= 1e-5


def test_error_behaviour(dev, graph_l4):
    """Shape/dtype/arity violations raise ValueError, like the reference's asserts."""
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    pl = GraphPlan(graph_l4["L"][4], dev)
    x = torch.zeros(2, 25, 3, device=dev)
    W = torch.zeros(9, 4, device=dev)
    b = torch.zeros(4, device=dev)
    with pytest.raises(ValueError):  # W rows != Fin*K
        ops.cheb_fwd(x, None, *pl.tensors(), W, b, 2, 1, ops.BIAS_PER_FILTER, True, False, 0)
    with pytest.raises(ValueError):  # wrong vertex count
        ops.cheb_fwd(torch.zeros(2, 24, 3, device=dev), None, *pl.tensors(), W, b, 3, 1, ops.BIAS_PER_FILTER, True, False, 0)
    with pytest.raises(ValueError):  # pooling size not a power of two
        ops.cheb_fwd(x, None, *pl.tensors(), W, b, 3, 3, ops.BIAS_PER_FILTER, True, False, 0)
    with pytest.raises(ValueError):  # float64 input
        ops.cheb_fwd(x.double(), None, *pl.tensors(), W, b, 3, 1, ops.BIAS_PER_FILTER, True, False, 0)
    with pytest.raises(ValueError):  # K < 1
        ops.cheb_fwd(x, None, *pl.tensors(), torch.zeros(0, 4, device=dev), b, 0, 1, ops.BIAS_PER_FILTER, True, False, 0)
    y, _ = ops.cheb_fwd(x, None, *pl.tensors(), W, b, 3, 1, ops.BIAS_PER_FILTER, True, False, 0)
    assert y.shape == (2, 25, 4) and float(y.abs().sum()) == 0.0


# ------------------------------------------------------------------------------------------ whole model
def build_model(graph, F, K, p, Mfc, filt, brelu, dev, fused=True, perm=None, algo=0):
    from gcn_fmri_decoding_b200.models import cgcnn

    return cgcnn(L=graph["L"], F=F, K=K, p=p, M=Mfc, filter=filt, brelu=brelu, channel=15, device=dev, seed=7,
                 regularization=5e-4, batch_size=16, perm=perm, n_input_vertices=360, fused=fused, algo=algo)


def oracle_logits(model, xperm, dtype=np.float64):
    sd = model.state_dict_tf()
    n = len(model.p)
    params = [dict(W=sd["conv%d/weights" % (i + 1)], b=sd["conv%d/bias" % (i + 1)].reshape(
        (-1, model.F[i]) if model.brelu_name == "b2relu" else (model.F[i],)), K=model.K[i], p=model.p[i]) for i in range(n)]
    h = O.conv_stack(xperm, model.L, params, filter=model.filter_name, brelu=model.brelu_name, dtype=dtype)
    names = ["fc%d" % (i + 1) for i in range(len(model.M) - 1)] + ["logits"]
    return O.head(h, [(sd[s + "/weights"], sd[s + "/bias"]) for s in names], dtype)


@pytest.mark.parametrize("cfg", ["config2", "config1_b2", "config1_b1", "config3_k2", "config3_k1"])
def test_model_logits_and_argmax(dev, graph_l1, graph_l4, cfg):
    """Whole network (conv stack + head) against the oracle: logits within TOL, identical arg-max over 22 columns."""
    from gcn_fmri_decoding_b200 import graclus, synth

    if cfg == "config2":
        g, F, K, p, filt, brelu = graph_l4, [32, 32], [5, 5], [4, 4], "chebyshev5", "b1relu"
    elif cfg.startswith("config1"):
        g, F, K, p, filt = graph_l1, [32] * 6, [5] * 6, [1] * 6, "chebyshev5"
        brelu = "b2relu" if cfg.endswith("b2") else "b1relu"
    elif cfg == "config3_k2":
        g, F, K, p, filt, brelu = graph_l4, [32, 32], [2, 2], [4, 4], "chebyshev2", "b1relu"
    else:
        g, F, K, p, filt, brelu = graph_l4, [32, 32], [1, 1], [4, 4], "chebyshev5", "b1relu"
    xraw = synth.bold_windows(16, seed=11)
    xperm = graclus.perm_data_3d(xraw, g["perm"]).astype(np.float32)
    model = build_model(g, F, K, p, [512, 256, 22], filt, brelu, dev, perm=g["perm"])
    ref = oracle_logits(model, xperm)
    with torch.no_grad():
        fused_from_raw = model(T(xraw, dev)).cpu().numpy()          # gather fused into layer 1
        fused_from_perm = model(T(xperm, dev), gather=False).cpu().numpy()
        model.fused = False
        unfused = model(T(xperm, dev), gather=False).cpu().numpy()   # filter / brelu / pool one by one
    for got in (fused_from_raw, fused_from_perm, unfused):
        assert got.shape == (16, 22)
        assert rel_inf(got, ref) <= TOL
        assert np.array_equal(got.argmax(1), ref.argmax(1))
    assert np.array_equal(fused_from_raw, fused_from_perm)


def test_model_spectral(dev, graph_l4):
    from gcn_fmri_decoding_b200 import graclus, synth

    g = graph_l4
    xraw = synth.bold_windows(8, seed=12)
    xperm = graclus.perm_data_3d(xraw, g["perm"]).astype(np.float32)
    model = build_model(g, [32, 32], [0, 0], [4, 4], [512, 256, 22], "fourier", "b1relu", dev, perm=g["perm"])
    sd = model.state_dict_tf()
    # oracle with the very basis the model uses
    h = xperm
    for i in range(2):
        Ut = model._spectral_plan(model.L[i]).Ut.cpu().numpy()
        z = O.filter_in_fourier(h, Ut, sd["conv%d/weights" % (i + 1)], np.float64)
        h = O.mpool1(O.b1relu(z, sd["conv%d/bias" % (i + 1)]), 4)
    ref = O.head(h, [(sd[s + "/weights"], sd[s + "/bias"]) for s in ("fc1", "fc2", "logits")], np.float64)
    with torch.no_grad():
        got = model(T(xraw, dev)).cpu().numpy()
    assert rel_inf(got, ref) <= TOL and np.array_equal(got.argmax(1), ref.argmax(1))


def test_training_step_gradients_match_oracle(dev, graph_l4):
    """Full backward through both conv layers and the head: dW/db of every conv layer against the oracle."""
    from gcn_fmri_decoding_b200 import graclus, synth

    g = graph_l4
    B = 12
    xraw = synth.bold_windows(B, seed=13)
    labels = synth.labels(B, seed=13)
    xperm = graclus.perm_data_3d(xraw, g["perm"]).astype(np.float32)
    model = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
    logits = model(T(xraw, dev))
    loss = model.loss(logits, T(labels, dev, torch.long))
    loss.backward()
    # oracle: forward in fp64, softmax-CE gradient, head backward, conv backward
    sd = {k: v.astype(np.float64) for k, v in model.state_dict_tf().items()}
    params = [dict(W=sd["conv%d/weights" % (i + 1)], b=sd["conv%d/bias" % (i + 1)].reshape(32), K=5, p=4) for i in range(2)]
    h, tr = O.conv_stack(xperm, model.L, params, dtype=np.float64, keep=True)
    hm = h.mean(-1)
    a1 = np.maximum(hm @ sd["fc1/weights"] + sd["fc1/bias"], 0)
    a2 = np.maximum(a1 @ sd["fc2/weights"] + sd["fc2/bias"], 0)
    lg = a2 @ sd["logits/weights"] + sd["logits/bias"]
    regs = [sd["conv1/weights"], sd["conv2/weights"]] + [sd[s + t] for s in ("fc1", "fc2", "logits") for t in ("/weights", "/bias")]
    assert abs(float(loss) - O.loss(lg, labels, regs, 5e-4)) <= 1e-4 * abs(float(loss))
    pz = np.exp(lg - lg.max(1, keepdims=True))
    pz /= pz.sum(1, keepdims=True)
    pz[np.arange(B), labels] -= 1
    dlg = pz / B
    da2 = (dlg @ sd["logits/weights"].T) * (a2 > 0)
    da1 = (da2 @ sd["fc2/weights"].T) * (a1 > 0)
    dhm = da1 @ sd["fc1/weights"].T
    dh = np.repeat(dhm[:, :, None], 32, 2) / 32
    _, grads = O.conv_stack_bwd(tr, model.L, params, dh, dtype=np.float64)
    for i in range(2):
        gW = grads[i]["dW"] + 5e-4 * sd["conv%d/weights" % (i + 1)]
        assert rel_inf(model.conv_weights[i].grad.cpu().numpy(), gW) <= TOL, i
        assert rel_inf(model.conv_bias[i].grad.cpu().numpy().reshape(32), grads[i]["db"]) <= TOL, i


def test_fused_trainer_matches_autograd_trainer(dev, graph_l4):
    """The explicit few-launch training step (FusedTrainer: fused mean, custom xent, flat TF-Adam with the L2 term
    folded in) produces the gradients of the autograd step, and the same parameters after a few Adam steps wherever
    the gradient is not numerically zero (Adam's m/sqrt(v) amplifies rounding noise on those)."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.train import FusedTrainer, Trainer

    g = graph_l4
    x = T(synth.bold_windows(32, seed=21), dev)
    y = T(synth.labels(32, seed=21), dev, torch.long)
    for graph, own in ((False, False), (True, False), (False, True)):
        a = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
        b = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
        ta = Trainer(a, distributed=False)
        tb = FusedTrainer(b, distributed=False, use_cuda_graph=graph, dropout=1.0, own_gemm=own)
        p0 = tb.flat_p.clone()
        la, _ = ta.step(x, y)
        lb, _ = tb.step(x, y)
        torch.cuda.synchronize()
        reg_before = 5e-4 * 0.5 * float((p0 * p0 * tb.decay).sum())
        assert abs(float(la) - (float(lb) + reg_before)) <= 1e-4 * abs(float(la))
        g_auto = ta.flat_grad                                   # d(CE + L2)/dp
        g_fused = tb.flat_g + 5e-4 * p0 * tb.decay              # the update kernel adds the L2 term itself
        scale = float(g_auto.abs().max())
        assert float((g_auto - g_fused).abs().max()) <= 1e-4 * scale, (graph, own)
        big = g_auto.abs() > 1e-3 * scale
        for _ in range(2):
            ta.step(x, y)
            tb.step(x, y)
            big &= ta.flat_grad.abs() > 1e-3 * scale            # ... at every one of the steps
        torch.cuda.synchronize()
        pa = torch.cat([p.detach().reshape(-1) for p in a.parameters()])
        assert int(big.sum()) > 1000
        assert float((pa - tb.flat_p)[big].abs().max()) <= 2e-4, (graph, own)  # three steps of size 1e-3


@pytest.mark.parametrize("lvl,B,Fin,Fout,K,p,brelu", [(0, 7, 15, 32, 5, 4, "b1relu"), (0, 3, 15, 32, 3, 1, "b2relu"),
                                                     (2, 9, 32, 32, 5, 4, "b1relu"), (3, 5, 6, 16, 2, 2, "b2relu"),
                                                     (1, 4, 8, 24, 4, 2, "b1relu")])
def test_saved_basis_weight_gradient(dev, graph_l4, lvl, B, Fin, Fout, K, p, brelu):
    """Training path of a first layer: the forward keeps X_k, the backward contracts it with dZ in one streamed GEMM.
    dW / db must match the fp64 oracle and the recompute path; the saved basis must equal the oracle's recursion."""
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    rng = np.random.RandomState(77 + lvl)
    L = graph_l4["L"][lvl]
    M = L.shape[0]
    x = rng.randn(B, M, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * 0.2).astype(np.float32)
    b = (0.2 + 0.1 * rng.randn(*((M, Fout) if brelu == "b2relu" else (Fout,)))).astype(np.float32)
    dy = rng.randn(B, M // p, Fout).astype(np.float32)
    pr = [dict(W=W, b=b, K=K, p=p)]
    y64, tr = O.conv_stack(x, [L], pr, brelu=brelu, dtype=np.float64, keep=True)
    dx64, g64 = O.conv_stack_bwd(tr, [L], pr, dy, brelu=brelu, dtype=np.float64, first_needs_dx=True)
    pl = GraphPlan(L, dev)
    mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
    xt, Wt, bt = T(x, dev), T(W, dev), T(b, dev)
    y, am, _, stack = ops.cheb_fwd_mean(xt, None, pl.rowptr, pl.col, pl.val, Wt, bt, K, p, mode, True, ops.ALGO_FUSED, True)
    assert stack.numel() > 0 and stack.shape[:3] == (K, B, M)
    basis = O.chebyshev_stack(x, L, K, np.float64).reshape(B, M, Fin, K)          # [b, m, f, k]
    got = stack.cpu().numpy()[..., :Fin].transpose(1, 2, 3, 0)                      # [k,b,m,f] -> [b,m,f,k]
    assert rel_inf(got, basis) <= 1e-5
    assert float(stack[..., Fin:].abs().max()) == 0.0 if stack.shape[-1] > Fin else True
    gW, gb = torch.empty_like(Wt), torch.empty(b.size, device=dev)
    ops.cheb_bwd_into(xt, None, y, am, T(dy, dev), False, *pl.tensors(), Wt, gW, gb, K, p, mode, True, False, ops.ALGO_FUSED, stack)
    assert rel_inf(gW.cpu().numpy(), g64[0]["dW"]) <= TOL
    assert rel_inf(gb.cpu().numpy().reshape(b.shape), g64[0]["db"]) <= TOL
    gW2, gb2 = torch.empty_like(Wt), torch.empty(b.size, device=dev)
    ops.cheb_bwd_into(xt, None, y, am, T(dy, dev), False, *pl.tensors(), Wt, gW2, gb2, K, p, mode, True, False, ops.ALGO_FUSED, None)
    assert rel_inf(gW.cpu().numpy(), gW2.cpu().numpy()) <= 1e-5 and rel_inf(gb.cpu().numpy(), gb2.cpu().numpy()) <= 1e-5
    gW3, gb3 = torch.empty_like(Wt), torch.empty(b.size, device=dev)
    ops.cheb_bwd_into(xt, None, y, am, T(dy, dev), False, *pl.tensors(), Wt, gW3, gb3, K, p, mode, True, False, ops.ALGO_FUSED, stack)
    assert torch.equal(gW, gW3) and torch.equal(gb, gb3)  # deterministic
    # a layer that also needs dx: dW/db from the saved basis, dx from the adjoint recursion alone
    gW4, gb4 = torch.empty_like(Wt), torch.empty(b.size, device=dev)
    dx = ops.cheb_bwd_into(xt, None, y, am, T(dy, dev), False, *pl.tensors(), Wt, gW4, gb4, K, p, mode, True, True, ops.ALGO_AUTO, stack)
    assert rel_inf(dx.cpu().numpy(), dx64) <= TOL
    assert rel_inf(gW4.cpu().numpy(), g64[0]["dW"]) <= TOL and rel_inf(gb4.cpu().numpy().reshape(b.shape), g64[0]["db"]) <= TOL


def test_saved_basis_vertex_level_graph(dev):
    """Graphs the fused kernels cannot hold keep the basis in the general path's vertex-major layout: the backward
    then skips the K-1 sparse steps and must give exactly what the recompute path gives."""
    from gcn_fmri_decoding_b200 import _lib, ops, synth
    from gcn_fmri_decoding_b200.plan import GraphPlan

    M, B, Fin, Fout, K = 3000, 4, 15, 32, 9
    L = synth.fibonacci_sphere_graph(M, 6)
    pl = GraphPlan(L, dev)
    if _lib.lib().gcnb_cheb_fused_supported(B, M, pl.nnz, Fin, Fout, K, 1, 0, 0):
        pytest.skip("this shape fits the fused kernels")
    assert _lib.lib().gcnb_cheb_stack_width(B, M, pl.nnz, Fin, Fout, K, 1) == Fin
    rng = np.random.RandomState(5)
    x = rng.randn(B, M, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * 0.1).astype(np.float32)
    b = np.full(Fout, 0.2, np.float32)
    dy = rng.randn(B, M, Fout).astype(np.float32)
    xt, Wt, bt, dyt = T(x, dev), T(W, dev), T(b, dev), T(dy, dev)
    y, am, ymean, stack = ops.cheb_fwd_mean(xt, None, pl.rowptr, pl.col, pl.val, Wt, bt, K, 1, ops.BIAS_PER_FILTER, True,
                                            ops.ALGO_AUTO, True)
    assert tuple(stack.shape) == (K, B, M, Fin)
    basis = O.chebyshev_stack(x, L, K, np.float64).reshape(B, M, Fin, K)           # [b, m, f, k]
    got = stack.cpu().numpy().reshape(K, M, B, Fin).transpose(2, 1, 3, 0)            # [k,m,b,f] -> [b,m,f,k]
    assert rel_inf(got, basis) <= 1e-5
    assert rel_inf(ymean.cpu().numpy(), y.cpu().numpy().mean(-1)) <= 1e-6
    out = []
    for st in (stack, None):
        gW, gb = torch.empty_like(Wt), torch.empty(Fout, device=dev)
        dx = ops.cheb_bwd_into(xt, None, y, am, dyt, False, *pl.tensors(), Wt, gW, gb, K, 1, ops.BIAS_PER_FILTER, True, True,
                               ops.ALGO_AUTO, st)
        out.append((dx, gW, gb))
    for a, c in zip(*out):
        assert torch.equal(a, c)


def test_head_pieces(dev, graph_l4):
    """Fused mean over filters (forward) / mean-form dy (backward), ReLU+dropout, column sums, xent -- against NumPy."""
    import ctypes as C

    from gcn_fmri_decoding_b200 import _lib, ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    lib = _lib.lib()
    vp = lambda t: C.c_void_p(t.data_ptr())
    rng = np.random.RandomState(4)
    L = graph_l4["L"][2]
    pl = GraphPlan(L, dev)
    x = T(rng.randn(6, 100, 32).astype(np.float32), dev)
    W = T((rng.randn(160, 32) * 0.2).astype(np.float32), dev)
    b = T(np.full(32, 0.2, np.float32), dev)
    for algo in algos_for(6, 100, pl.nnz, 32, 32, 5, 4, True, True):
        y, am, ym, _ = ops.cheb_fwd_mean(x, None, pl.rowptr, pl.col, pl.val, W, b, 5, 4, ops.BIAS_PER_FILTER, True, algo)
        y2, am2 = ops.cheb_fwd(x, None, *pl.tensors(), W, b, 5, 4, ops.BIAS_PER_FILTER, True, True, algo)
        assert torch.equal(y, y2) and torch.equal(am, am2)
        assert float((ym - y.mean(-1)).abs().max()) <= 1e-5 * float(y.abs().max())
        dm = T(rng.randn(6, 25).astype(np.float32), dev)
        full = (dm / 32).unsqueeze(-1).expand(6, 25, 32).contiguous()
        ref = torch.ops.gcn_b200.cheb_bwd(x, None, y, am, full, *pl.tensors(), W, 5, 4, ops.BIAS_PER_FILTER, True, True, algo)
        gW, gb = torch.empty_like(W), torch.empty(32, device=dev)
        dx = ops.cheb_bwd_into(x, None, y, am, dm, True, *pl.tensors(), W, gW, gb, 5, 4, ops.BIAS_PER_FILTER, True, True, algo)
        for got, want in ((dx, ref[0]), (gW, ref[1]), (gb, ref[2])):
            assert float((got - want).abs().max()) <= 1e-5 * float(want.abs().max()), algo
    # ReLU + dropout: kept fraction, scaling, fresh mask per step, deterministic for a given step
    a = T(rng.randn(512, 512).astype(np.float32), dev)
    state = torch.tensor([1.0, 1.0, 0.0, 3.0], device=dev)
    o1, o2 = a.clone(), a.clone()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.gcnb_relu_dropout_fwd_f32(vp(o1), 512, 512, 512, 0.5, 7, vp(state), stream) == 0
    assert lib.gcnb_relu_dropout_fwd_f32(vp(o2), 512, 512, 512, 0.5, 7, vp(state), stream) == 0
    assert torch.equal(o1, o2)
    pos = a > 0
    kept = (o1 > 0) & pos
    assert abs(float(kept.sum()) / float(pos.sum()) - 0.5) < 0.01
    assert torch.allclose(o1[kept], 2 * a[kept]) and float(o1[~pos].abs().max()) == 0.0
    state[3] = 4.0
    o3 = a.clone()
    lib.gcnb_relu_dropout_fwd_f32(vp(o3), 512, 512, 512, 0.5, 7, vp(state), stream)
    assert not torch.equal(o1, o3)
    d = T(rng.randn(512, 512).astype(np.float32), dev)
    d0 = d.clone()
    lib.gcnb_relu_dropout_bwd_f32(vp(d), vp(o1), 512, 512, 512, 512, 0.5, stream)
    assert torch.equal(d, torch.where(o1 > 0, 2 * d0, torch.zeros_like(d0)))
    o4 = a.clone()
    lib.gcnb_relu_dropout_fwd_f32(vp(o4), 512, 512, 512, 1.0, 7, vp(state), stream)
    assert torch.equal(o4, torch.relu(a))
    # column sums of several matrices in one launch
    ms = [T(rng.randn(512, n).astype(np.float32), dev) for n in (512, 256, 22)]
    outs = [torch.empty(n, device=dev) for n in (512, 256, 22)]
    rc = lib.gcnb_colsum_multi_f32((C.c_void_p * 3)(*[t.data_ptr() for t in ms]), (C.c_void_p * 3)(*[t.data_ptr() for t in outs]),
                                   (C.c_int * 3)(512, 512, 512), (C.c_int * 3)(512, 256, 22), 3, stream)
    assert rc == 0
    for mm_, oo in zip(ms, outs):
        assert float((oo - mm_.double().sum(0).float()).abs().max()) <= 1e-4
    # tensor-core GEMM (3xTF32): all four transpose combinations, ragged sizes, bias
    for (Mg, Ng, Kg, ta, tb) in ((512, 256, 512, 0, 0), (25, 512, 512, 1, 0), (512, 25, 512, 0, 1), (67, 45, 33, 1, 1), (400, 7680, 400, 1, 0)):
        A = T(rng.randn(*((Kg, Mg) if ta else (Mg, Kg))).astype(np.float32), dev)
        Bm = T(rng.randn(*((Ng, Kg) if tb else (Kg, Ng))).astype(np.float32), dev)
        bias = T(rng.randn(Ng).astype(np.float32), dev)
        Cc = torch.empty(Mg, Ng, device=dev)
        rc = lib.gcnb_gemm_f32(vp(A), vp(Bm), vp(Cc), vp(bias), Mg, Ng, Kg, A.shape[1], Bm.shape[1], Ng, ta, tb, stream)
        assert rc == 0
        ref = (A.double().t() if ta else A.double()) @ (Bm.double().t() if tb else Bm.double()) + bias.double()
        assert float((Cc.double() - ref).abs().max()) <= 1e-5 * float(ref.abs().max()), (Mg, Ng, Kg, ta, tb)
    # fused FC epilogues: bit-identical to the GEMM followed by the stand-alone ReLU/dropout kernels (same mask, same step)
    for (Mg, Ng, Kg) in ((512, 512, 25), (512, 256, 512), (70, 45, 33), (512, 4096, 64)):
        A = T(rng.randn(Mg, Kg).astype(np.float32), dev)
        Bm = T(rng.randn(Kg, Ng).astype(np.float32), dev)
        bias = T(rng.randn(Ng).astype(np.float32), dev)
        stp = torch.tensor([0.0, 0.0, 0.0, 5.0], device=dev)
        for keep in (0.5, 1.0):
            two, one = torch.empty(Mg, Ng, device=dev), torch.empty(Mg, Ng, device=dev)
            assert lib.gcnb_gemm_f32(vp(A), vp(Bm), vp(two), vp(bias), Mg, Ng, Kg, Kg, Ng, Ng, 0, 0, stream) == 0
            assert lib.gcnb_relu_dropout_fwd_f32(vp(two), Mg, Ng, Ng, keep, 11, vp(stp), stream) == 0
            assert lib.gcnb_gemm_epilogue_f32(vp(A), vp(Bm), vp(one), vp(bias), Mg, Ng, Kg, Kg, Ng, Ng, 0, 0, _lib.EPI_RELU_DROPOUT,
                                              None, 0, keep, 11, vp(stp), stream) == 0
            assert torch.equal(one, two), (Mg, Ng, Kg, keep)
            # adjoint: d W^T masked by the activation
            dd = T(rng.randn(Mg, Ng).astype(np.float32), dev)
            Wt_ = T(rng.randn(Kg, Ng).astype(np.float32), dev)           # dx[Mg x Kg] = dd[Mg x Ng] Wt_^T
            act = T(np.maximum(rng.randn(Mg, Kg), 0).astype(np.float32), dev)
            two, one = torch.empty(Mg, Kg, device=dev), torch.empty(Mg, Kg, device=dev)
            assert lib.gcnb_gemm_f32(vp(dd), vp(Wt_), vp(two), None, Mg, Kg, Ng, Ng, Ng, Kg, 0, 1, stream) == 0
            assert lib.gcnb_relu_dropout_bwd_f32(vp(two), vp(act), Mg, Kg, Kg, Kg, keep, stream) == 0
            assert lib.gcnb_gemm_epilogue_f32(vp(dd), vp(Wt_), vp(one), None, Mg, Kg, Ng, Ng, Ng, Kg, 0, 1, _lib.EPI_MASK, vp(act), Kg,
                                              keep, 0, None, stream) == 0
            assert torch.equal(one, two), (Mg, Ng, Kg, keep)
    assert lib.gcnb_gemm_epilogue_f32(vp(A), vp(Bm), vp(one), None, 4, 4, 4, 4, 4, 4, 0, 0, _lib.EPI_MASK, None, 0, 0.5, 0, None, stream) != 0
    # cross-entropy forward+backward and the optimiser clock
    lg = T(rng.randn(512, 22).astype(np.float32) * 3, dev)
    lab = T(rng.randint(0, 21, 512), dev, torch.long)
    loss, dl, rows = torch.zeros((), device=dev), torch.empty_like(lg), torch.empty(512, device=dev)
    st2 = torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev)
    assert lib.gcnb_softmax_xent_f32(vp(lg), vp(lab), vp(loss), vp(dl), vp(rows), 512, 22, vp(st2), 1e-3, 0.9, 0.999, stream) == 0
    lgr = lg.clone().double().requires_grad_(True)
    ref = torch.nn.functional.cross_entropy(lgr, lab)
    ref.backward()
    assert abs(float(loss) - float(ref)) <= 1e-5 * float(ref)
    assert float((dl.double() - lgr.grad).abs().max()) <= 1e-7
    assert np.allclose(st2.cpu().numpy(), [0.9, 0.999, 1e-3 * np.sqrt(1 - 0.999) / (1 - 0.9), 1.0], rtol=1e-5)


# ------------------------------------------------------------------------------------------ full-size properties
def test_full_size_properties(dev, graph_l4):
    """BASELINE config-2 sizes (B=512): determinism, batch independence, linearity of the filter,
    agreement of the two kernel families, pooled output = max over the un-pooled output."""
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    rng = np.random.RandomState(0)
    torch.manual_seed(1234)
    B = 512
    for lvl, Fin in ((0, 15), (2, 32)):
        L = graph_l4["L"][lvl]
        M = L.shape[0]
        pl = GraphPlan(L, dev)
        x1 = torch.randn(B, M, Fin, device=dev)
        x2 = torch.randn(B, M, Fin, device=dev)
        W = T((rng.randn(Fin * 5, 32) * 0.2).astype(np.float32), dev)
        b = torch.full((32,), 0.2, device=dev)
        outs = {}
        for algo in algos_for(B, M, pl.nnz, Fin, 32, 5, 4):
            y, am = ops.cheb_fwd(x1, None, *pl.tensors(), W, b, 5, 4, ops.BIAS_PER_FILTER, True, True, algo)
            y_again, am_again = ops.cheb_fwd(x1, None, *pl.tensors(), W, b, 5, 4, ops.BIAS_PER_FILTER, True, True, algo)
            assert torch.equal(y, y_again) and torch.equal(am, am_again)  # deterministic
            ysub, _ = ops.cheb_fwd(x1[100:103].contiguous(), None, *pl.tensors(), W, b, 5, 4, ops.BIAS_PER_FILTER, True,
                                   True, algo)
            assert torch.allclose(ysub, y[100:103], rtol=0, atol=2e-5 * float(y.abs().max()))  # batch independence
            # un-pooled activation, pooled by hand, must give the same values and arg-max
            a, _ = ops.cheb_fwd(x1, None, *pl.tensors(), W, b, 5, 1, ops.BIAS_PER_FILTER, True, False, algo)
            win = a.view(B, M // 4, 4, 32)
            assert torch.equal(win.max(2).values, y)
            # FIRST maximum of the window (MaxPoolGrad's rule; torch.argmax does not promise it on ties), bit-exact.
            # All-zero windows after the ReLU included: there the first vertex is the arg-max.
            hit = win == win.max(2, keepdim=True).values
            first = torch.where(hit, torch.arange(4, device=dev).view(1, 1, 4, 1), torch.full((), 4, device=dev)).min(2).values
            assert torch.equal(first.to(torch.uint8), am)
            # linearity of the bare filter: f(2 x1 - 3 x2) = 2 f(x1) - 3 f(x2)
            f = lambda t: ops.cheb_fwd(t, None, *pl.tensors(), W, None, 5, 1, ops.BIAS_NONE, False, False, algo)[0]
            lhs, rhs = f(2 * x1 - 3 * x2), 2 * f(x1) - 3 * f(x2)
            assert float((lhs - rhs).abs().max()) <= 1e-4 * float(rhs.abs().max())
            outs[algo] = y
        ys = list(outs.values())
        for other in ys[1:]:
            assert float((other - ys[0]).abs().max()) <= 1e-4 * float(ys[0].abs().max())


@pytest.mark.parametrize("n,B", [(3000, 3), (3000, 4), (32492, 8)])
def test_large_graph_general_path(dev, n, B):
    """Vertex-level graph (config 5 family): HBM-resident operator, K=25.  B=4 makes the vertex-major rows 16-byte
    multiples (TMA-staged SpMM) and leaves ragged last tiles in the tensor-core contractions; (32492, 8) is BASELINE
    config 5's own graph size (the sphere kNN graph bench.py --config 5 runs on) at a batch the fp64 oracle finishes
    in seconds -- forward and backward (dx, dW, db)."""
    from gcn_fmri_decoding_b200 import synth

    L = synth.fibonacci_sphere_graph(n, 6)
    rng = np.random.RandomState(9)
    x = rng.randn(B, n, 15).astype(np.float32)
    W = (rng.randn(15 * 25, 32) * 0.05).astype(np.float32)
    b = np.full(32, 0.2, np.float32)
    dy = rng.randn(B, n, 32).astype(np.float32)
    pr = [dict(W=W, b=b, K=25, p=1)]
    y64, tr = O.conv_stack(x, [L], pr, dtype=np.float64, keep=True)
    # A pre-activation within fp32 rounding of zero makes the ReLU mask (hence the gradient routed through that one
    # element) a coin toss between fp32 and the fp64 oracle: take those elements out of dy.  (With this seed there
    # is exactly such an element.)
    pre = tr[0]["z"] + b
    dy[np.abs(pre) < 1e-5 * np.abs(pre).max()] = 0.0
    dx64, g64 = O.conv_stack_bwd(tr, [L], pr, dy, dtype=np.float64, first_needs_dx=True)
    from gcn_fmri_decoding_b200 import _lib

    r = run_layer(dev, L, x, W, b, 25, 1, "b1relu", _lib.ALGO_GENERAL, dy=dy)
    assert rel_inf(r["y"], y64) <= TOL
    assert rel_inf(r["dW"], g64[0]["dW"]) <= TOL
    assert rel_inf(r["db"], g64[0]["db"]) <= TOL
    assert rel_inf(r["dx"], dx64) <= TOL


# ------------------------------------------------------------------------------------------ round 2
def _head_oracle(a0, labels, Ws, bs, masks, keep):
    """fp64 head forward + backward for given dropout masks (models_gcn.py:650-656, :674-681, :253-259, :298-303)."""
    a0 = a0.astype(np.float64)
    h1 = np.maximum(a0 @ Ws[0] + bs[0], 0) * masks[0] / keep
    h2 = np.maximum(h1 @ Ws[1] + bs[1], 0) * masks[1] / keep
    lg = h2 @ Ws[2] + bs[2]
    z = lg - lg.max(1, keepdims=True)
    logp = z - np.log(np.exp(z).sum(1, keepdims=True))
    B = len(labels)
    loss = -logp[np.arange(B), labels].mean()
    d3 = np.exp(logp)
    d3[np.arange(B), labels] -= 1
    d3 /= B
    d2 = (d3 @ Ws[2].T) * (h2 > 0) / keep
    d1 = (d2 @ Ws[1].T) * (h1 > 0) / keep
    return dict(logits=lg, loss=loss, gW=[a0.T @ d1, h1.T @ d2, h2.T @ d3], gb=[d1.sum(0), d2.sum(0), d3.sum(0)],
                d0=d1 @ Ws[0].T)


@pytest.mark.parametrize("B,widths,keep", [(512, (25, 512, 256, 22), 1.0), (512, (25, 512, 256, 22), 0.5),
                                           (37, (25, 512, 256, 22), 0.5), (130, (7, 100, 50, 5), 0.75),
                                           (64, (32, 129, 67, 32), 1.0), (2048, (25, 512, 256, 22), 0.5),
                                           (4096, (25, 512, 256, 22), 0.5)])
def test_head_step_kernel_matches_oracle(dev, B, widths, keep):
    """gcnb_head_step_f32 (one cooperative launch: FC x3, cross-entropy, full backward) against the fp64 oracle run with
    the SAME dropout masks (the counter-based mask is mirrored in oracle.counter_dropout_mask)."""
    import ctypes as C

    from gcn_fmri_decoding_b200 import _lib

    lib = _lib.lib()
    rng = np.random.RandomState(B + widths[1])
    n0, n1, n2, nc = widths
    a0 = np.abs(rng.randn(B, n0)).astype(np.float32)
    labels = rng.randint(0, nc, size=B).astype(np.int64)
    Ws = [(rng.randn(a, b) * 0.2).astype(np.float32) for a, b in ((n0, n1), (n1, n2), (n2, nc))]
    bs = [(rng.randn(b) * 0.1 + 0.1).astype(np.float32) for b in (n1, n2, nc)]
    step = 3.0
    state = T(np.array([0.9 ** 3, 0.999 ** 3, 0.0, step], np.float32), dev)
    masks = [O.counter_dropout_mask(B, n1, keep, 0x5eed, step), O.counter_dropout_mask(B, n2, keep, 0x5eed + 1, step)]
    ref = _head_oracle(a0, labels, [w.astype(np.float64) for w in Ws], [b.astype(np.float64) for b in bs], masks, keep)
    ta0, tl = T(a0, dev), T(labels, dev, torch.long)
    tW, tb = [T(w, dev) for w in Ws], [T(b, dev) for b in bs]
    gW, gb = [torch.empty_like(w) for w in tW], [torch.empty_like(b) for b in tb]
    logits = torch.empty(B, nc, device=dev)
    loss = torch.zeros((), device=dev)
    d0 = torch.empty(B, n0, device=dev)
    nbytes = lib.gcnb_head_step_workspace_bytes(B, n0, n1, n2, nc)
    assert nbytes > 0
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    vp = lambda t: C.c_void_p(t.data_ptr())
    outs = []
    for rep in range(2):  # twice: bit-reproducible
        state.copy_(T(np.array([0.9 ** 3, 0.999 ** 3, 0.0, step], np.float32), dev))
        rc = lib.gcnb_head_step_f32(vp(ta0), vp(tl), vp(tW[0]), vp(tb[0]), vp(tW[1]), vp(tb[1]), vp(tW[2]), vp(tb[2]),
                                    vp(logits), vp(loss), vp(gW[0]), vp(gb[0]), vp(gW[1]), vp(gb[1]), vp(gW[2]), vp(gb[2]),
                                    vp(d0), B, n0, n1, n2, nc, keep, 0x5eed, 0x5eed + 1, vp(state), 1e-3, 0.9, 0.999, 1,
                                    vp(ws), ws.numel(), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _lib.check(rc, "gcnb_head_step_f32")
        torch.cuda.synchronize()
        outs.append([t.clone() for t in (logits, loss, d0, *gW, *gb)])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert float(state[3]) == step + 1  # the optimiser clock advanced once
    assert rel_inf(logits.cpu().numpy(), ref["logits"]) <= TOL
    assert np.array_equal(logits.cpu().numpy().argmax(1), ref["logits"].argmax(1))
    assert abs(float(loss) - ref["loss"]) <= TOL * abs(ref["loss"])
    assert rel_inf(d0.cpu().numpy(), ref["d0"]) <= TOL
    for i in range(3):
        assert rel_inf(gW[i].cpu().numpy(), ref["gW"][i]) <= TOL, i
        assert rel_inf(gb[i].cpu().numpy(), ref["gb"][i]) <= TOL, i


@pytest.mark.parametrize("graph", [False, True])
def test_fused_trainer_with_dropout_matches_oracle(dev, graph_l4, graph):
    """The benched configuration -- FusedTrainer(dropout=0.5, own_gemm=True), fused head, tcgen05 forward, saved basis --
    against oracle.network_step run with the device's dropout masks: every gradient of the step."""
    from gcn_fmri_decoding_b200 import graclus, synth
    from gcn_fmri_decoding_b200.train import FusedTrainer

    g = graph_l4
    # A small batch: every pooled window / ReLU whose fp64 decision margin is below fp32 rounding is a coin toss that
    # reroutes one gradient element (see test_large_graph_general_path); with 16 windows this seed has none.
    B = 16
    xraw = synth.bold_windows(B, seed=31)
    labels = synth.labels(B, seed=31)
    model = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
    tr = FusedTrainer(model, distributed=False, use_cuda_graph=graph, dropout=0.5, own_gemm=True)
    sd = {k: v.astype(np.float64) for k, v in model.state_dict_tf().items()}
    p0 = tr.flat_p.clone()
    loss, logits = tr.step(T(xraw, dev), T(labels, dev, torch.long))
    torch.cuda.synchronize()
    # the first step draws its masks with the optimiser step count 0
    masks = [O.counter_dropout_mask(B, 512, 0.5, tr.dropout_seed, 0), O.counter_dropout_mask(B, 256, 0.5, tr.dropout_seed + 1, 0)]
    xperm = graclus.perm_data_3d(xraw, g["perm"])
    params = [dict(W=sd["conv%d/weights" % i], b=sd["conv%d/bias" % i].reshape(32), K=5, p=4) for i in (1, 2)]
    fcs = [(sd[s + "/weights"], sd[s + "/bias"]) for s in ("fc1", "fc2", "logits")]
    ref_loss, conv_g, fc_g = O.network_step(xperm, labels, model.L, params, fcs, 0.0, dtype=np.float64,
                                            dropout_masks=masks, keep=0.5)
    assert abs(float(loss) - ref_loss) <= TOL * abs(ref_loss)       # CE only (regularization=0 in the oracle call)
    for i in range(2):
        assert rel_inf(tr.gview[id(model.conv_weights[i])].cpu().numpy(), conv_g[i]["dW"]) <= TOL, i
        assert rel_inf(tr.gview[id(model.conv_bias[i])].cpu().numpy().reshape(32), conv_g[i]["db"]) <= TOL, i
    for i in range(3):
        assert rel_inf(tr.gview[id(model.fc_weights[i])].cpu().numpy(), fc_g[i][0]) <= TOL, i
        assert rel_inf(tr.gview[id(model.fc_bias[i])].cpu().numpy(), fc_g[i][1]) <= TOL, i
    # one TF-Adam step from p0 with g + reg * p on the regularised tensors (models_gcn.py:260-262, :294)
    gfull = tr.flat_g + 5e-4 * p0 * tr.decay
    m = 0.1 * gfull
    v = 0.001 * gfull * gfull
    lr_t = 1e-3 * np.sqrt(1 - 0.999) / (1 - 0.9)
    expect = p0 - lr_t * m / (v.sqrt() + 1e-8)
    assert float((expect - tr.flat_p).abs().max()) <= 1e-6


def test_benched_shapes_run_on_tcgen05(dev):
    """The forward kernel AUTO dispatch picks for the BASELINE config shapes is the tcgen05/TMEM one."""
    from gcn_fmri_decoding_b200 import _lib

    for shape in ((512, 400, 3684, 15, 32, 5, 4), (512, 100, 898, 32, 32, 5, 4), (128, 372, 3684, 32, 32, 5, 1)):
        assert "tcgen05" in _lib.describe_fwd(*shape), shape


@pytest.mark.parametrize("lvl,Fin,p,brelu", [(0, 15, 4, "b1relu"), (2, 32, 4, "b1relu"), (1, 15, 2, "b2relu"), (2, 32, 2, "b2relu"),
                                             (1, 15, 8, "b1relu")])
def test_fused_argmax_bit_exact_against_own_activations(dev, graph_l4, lvl, Fin, p, brelu):
    """mpool1 inside the fused kernel is bit-exact: the pooled values and the arg-max bytes equal the first-maximum
    pooling (MaxPoolGrad's rule, ties included) of the SAME kernel's un-pooled activations (p = 1 launch)."""
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    from gcn_fmri_decoding_b200 import _lib

    L = graph_l4["L"][lvl]
    M = L.shape[0]
    assert M % p == 0
    pl = GraphPlan(L, dev)
    torch.manual_seed(lvl * 10 + p)
    B = 33
    # both launches must run the same kernel family for the bit-for-bit comparison to mean anything
    assert "tcgen05" in _lib.describe_fwd(B, M, pl.nnz, Fin, 32, 5, p) and "tcgen05" in _lib.describe_fwd(B, M, pl.nnz, Fin, 32, 5, 1)
    x = torch.randn(B, M, Fin, device=dev)
    W = torch.randn(Fin * 5, 32, device=dev) * 0.2
    mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
    b = torch.randn(32 if brelu == "b1relu" else M * 32, device=dev) * 0.3
    y, am = ops.cheb_fwd(x, None, *pl.tensors(), W, b, 5, p, mode, True, True, ops.ALGO_FUSED)
    a, _ = ops.cheb_fwd(x, None, *pl.tensors(), W, b, 5, 1, mode, True, False, ops.ALGO_FUSED)
    win = a.view(B, M // p, p, 32)
    mx = win.max(2, keepdim=True).values
    first = torch.where(win == mx, torch.arange(p, device=dev).view(1, 1, p, 1), torch.full((), p, device=dev)).min(2).values
    assert torch.equal(mx.squeeze(2), y)
    assert torch.equal(first.to(torch.uint8), am)


@pytest.mark.parametrize("lvl,B,Fin,Fout,K,p,brelu", [(0, 9, 15, 32, 5, 4, "b1relu"), (2, 11, 32, 32, 5, 4, "b1relu"),
                                                      (1, 5, 16, 32, 3, 2, "b2relu"), (2, 6, 12, 8, 2, 1, "b1relu"),
                                                      (0, 300, 15, 32, 5, 4, "b1relu")])
def test_operator_image_kernels_match_the_self_built_ones(dev, graph_l4, lvl, B, Fin, Fout, K, p, brelu):
    """The row-blocked kernels fed by a host-built operator image (gcnb_cheb_image_build) add every row's terms in the
    same (ascending column) order as the kernels that derive their work lists from the CSR arrays -- zero-weight terms
    of sibling rows in between are exact no-ops -- so outputs and gradients must be IDENTICAL, not just close."""
    from gcn_fmri_decoding_b200 import _lib, plan

    L = graph_l4["L"][lvl]
    M = L.shape[0]
    rng = np.random.RandomState(lvl * 10 + B)
    x = rng.randn(B, M, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * 0.2).astype(np.float32)
    b = (rng.randn(Fout) * 0.1).astype(np.float32) if brelu == "b1relu" else (rng.randn(M, Fout) * 0.1).astype(np.float32)
    dy = rng.randn(B, M // p, Fout).astype(np.float32)
    gp = plan.GraphPlan(L, dev)
    assert gp.image((B, Fin, Fout, K, p)) is not None, "no image-based kernel for a benched shape family"
    outs = []
    for use in (True, False):
        old = plan.USE_IMAGES
        plan.USE_IMAGES = use
        try:
            outs.append(run_layer(dev, L, x, W, b, K, p, brelu, _lib.ALGO_AUTO, dy=dy))
        finally:
            plan.USE_IMAGES = old
    for key in ("y", "argmax", "dx", "dW", "db"):
        assert np.array_equal(outs[0][key], outs[1][key]), key
    y64, tr = O.conv_stack(x, [L], [dict(W=W, b=b, K=K, p=p)], brelu=brelu, dtype=np.float64, keep=True)
    assert rel_inf(outs[0]["y"], y64) <= TOL


def test_input_pipeline_and_bound_inputs_equal_plain_steps(dev, graph_l4):
    """train.InputPipeline (pinned host -> device slots on a copy stream, slots bound with FusedTrainer.bind_inputs so the
    captured step reads them in place) must train exactly like plain step() calls on device tensors: same kernels, same
    dropout stream, deterministic reductions -> bit-identical losses and parameters."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.train import FusedTrainer, InputPipeline

    g = graph_l4
    B, steps = 16, 5
    xs = [synth.bold_windows(B, seed=40 + i) for i in range(steps)]
    ys = [synth.labels(B, seed=40 + i) for i in range(steps)]

    def make():
        model = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
        return FusedTrainer(model, distributed=False, use_cuda_graph=True, dropout=0.5, dropout_seed=77)

    plain, piped = make(), make()
    ref = [float(plain.step(T(x, dev), T(y, dev, torch.long))[0]) for x, y in zip(xs, ys)]
    pipe = InputPipeline(piped, (B, 360, 15))
    got = []
    pipe.feed(xs[0], ys[0])
    for i in range(steps):
        if i + 1 < steps:
            pipe.feed(xs[i + 1], ys[i + 1])      # the copy of the next batch overlaps this step
        got.append(float(pipe.step()[0]))         # (the returned tensors are the graph's static outputs: read them now)
    assert got == ref
    assert torch.equal(plain.flat_p, piped.flat_p)
    with pytest.raises(RuntimeError):
        pipe.step()                               # nothing queued


def _random_tcgen05_cases(n=14, seed=2026):
    rng = np.random.RandomState(seed)
    cases = []
    while len(cases) < n:
        lvl = int(rng.randint(0, 4))                    # M = 400, 200, 100, 50
        p = int(rng.choice([1, 2, 4, 8]))
        Fin, Fout = int(rng.randint(9, 33)), int(4 * rng.randint(1, 9))
        K, B = int(rng.randint(1, 8)), int(rng.choice([1, 2, 5, 37, 130]))
        brelu = str(rng.choice(["b1relu", "b2relu"]))
        M = 400 >> lvl
        if M % p:
            continue
        cases.append((lvl, B, Fin, Fout, K, p, brelu))
    return cases


@pytest.mark.parametrize("lvl,B,Fin,Fout,K,p,brelu", _random_tcgen05_cases())
def test_layer_random_shapes(dev, graph_l4, lvl, B, Fin, Fout, K, p, brelu):
    """Seeded random layer shapes around the tcgen05 kernel's domain (9 <= Fin <= 32, Fout a multiple of 4, any K, p in
    {1,2,4,8}, ragged batches): forward (y, arg-max) and the autograd backward against the fp64 oracle, with and without
    the host-built operator image where the shape has one.  Autograd keeps no basis, so the backward recomputes it
    (k_cheb_bwd_fused or the general path); the saved-basis backward of the training step is swept in
    test_gpu_saved_basis.py."""
    from gcn_fmri_decoding_b200 import _lib, plan

    L = graph_l4["L"][lvl]
    M = L.shape[0]
    rng = np.random.RandomState(1000 * lvl + 10 * B + K)
    x = rng.randn(B, M, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * (0.4 / np.sqrt(Fin * K))).astype(np.float32)
    b = (rng.randn(Fout) * 0.1).astype(np.float32) if brelu == "b1relu" else (rng.randn(M, Fout) * 0.1).astype(np.float32)
    dy = rng.randn(B, M // p, Fout).astype(np.float32)
    pr = [dict(W=W, b=b, K=K, p=p)]
    y64, tr = O.conv_stack(x, [L], pr, brelu=brelu, dtype=np.float64, keep=True)
    # elements whose ReLU / pooling decision sits within fp32 rounding of a tie are coin tosses (see
    # test_large_graph_general_path): take them out of dy
    a64 = tr[0]["a"]
    pre = tr[0]["z"] + b                                     # pre-activation; max-pool(relu(.)) = relu(max(.))
    win = np.sort(pre.reshape(B, M // p, p, Fout), axis=2)
    eps = 1e-5 * np.abs(pre).max()
    tie = np.abs(win[:, :, -1]) < eps                        # the ReLU of the window maximum
    if p > 1:
        tie |= ((win[:, :, -1] - win[:, :, -2]) < eps) & (win[:, :, -1] > -eps)   # which vertex is the maximum
    dy[tie] = 0.0
    dx64, g64 = O.conv_stack_bwd(tr, [L], pr, dy, brelu=brelu, dtype=np.float64, first_needs_dx=True)
    # (AUTO dispatch: all but the shapes whose tables do not fit beside two state buffers run k_cheb_fwd_umma)
    for use_images in (True, False):
        old = plan.USE_IMAGES
        plan.USE_IMAGES = use_images
        try:
            r = run_layer(dev, L, x, W, b, K, p, brelu, _lib.ALGO_AUTO, dy=dy)
        finally:
            plan.USE_IMAGES = old
        tag = "images=%s" % use_images
        assert rel_inf(r["y"], y64) <= TOL, tag
        check_argmax(r["argmax"], a64, p, tag) if p > 1 else None
        assert rel_inf(r["dW"], g64[0]["dW"]) <= TOL, tag
        assert rel_inf(r["db"], g64[0]["db"]) <= TOL, tag
        assert rel_inf(r["dx"], dx64) <= TOL, tag


@pytest.mark.parametrize("brelu,nlayers,B", [("b2relu", 5, 19), ("b1relu", 3, 150), ("b2relu", 8, 2), ("b1relu", 4, 445)])
def test_layer_stack_is_bit_identical_to_layer_by_layer(dev, graph_l1, brelu, nlayers, B):
    """gcnb_cheb_stack_fwd_f32: a run of identical p = 1, 32 -> 32 layers in one launch (the production network's
    layers 2-6, model.py:271-274) gives bit for bit what the same layers give one launch at a time -- and hence the
    oracle's result within the layer tolerance; cgcnn.conv_stack picks it by itself under no_grad."""
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    L = graph_l1["L"][0]
    M = L.shape[0]
    pl = GraphPlan(L, dev)
    rng = np.random.RandomState(nlayers)
    x = rng.randn(B, M, 32).astype(np.float32)
    Ws = [(rng.randn(32 * 5, 32) * (0.5 / np.sqrt(160))).astype(np.float32) for _ in range(nlayers)]
    bs = [(rng.randn(32) * 0.1).astype(np.float32) if brelu == "b1relu" else (rng.randn(M, 32) * 0.1).astype(np.float32)
          for _ in range(nlayers)]
    mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
    xt, Wt, bt = T(x, dev), [T(w, dev) for w in Ws], [T(b, dev) for b in bs]
    assert ops.cheb_stack_supported(pl.rowptr, pl.col, pl.val, B, 32, 5, nlayers)
    y = ops.cheb_stack_fwd(xt, pl.rowptr, pl.col, pl.val, Wt, bt, 5, mode, True)
    h = xt
    for w, b in zip(Wt, bt):
        h = ops.cheb_fwd(h, None, *pl.tensors(), w, b, 5, 1, mode, True, False, ops.ALGO_AUTO)[0]
    assert torch.equal(y, h)
    # pre-split tap images (one TMA bulk copy per layer instead of the in-kernel split): bit for bit the same taps
    imgs = [ops.cheb_tap_image(w, 32, 5) for w in Wt]
    assert all(i is not None and i.numel() == 51200 for i in imgs)
    assert torch.equal(ops.cheb_stack_fwd(xt, pl.rowptr, pl.col, pl.val, Wt, bt, 5, mode, True, tap_images=imgs), y)
    mixed = [img if q % 2 == 0 else None for q, img in enumerate(imgs)]
    assert torch.equal(ops.cheb_stack_fwd(xt, pl.rowptr, pl.col, pl.val, Wt, bt, 5, mode, True, tap_images=mixed), y)
    y64 = O.conv_stack(x, [L] * nlayers, [dict(W=w, b=b, K=5, p=1) for w, b in zip(Ws, bs)], brelu=brelu, dtype=np.float64)
    assert rel_inf(y.cpu().numpy(), y64) <= TOL * nlayers


def test_model_uses_the_layer_stack_under_no_grad(dev, graph_l1):
    """config 1 (six p = 1 layers): the model's inference path takes layers 2-6 in one launch and returns the same
    logits as the layer-by-layer path that autograd uses."""
    from gcn_fmri_decoding_b200 import _lib

    g = graph_l1
    model = build_model(g, [32] * 6, [5] * 6, [1] * 6, [512, 256, 22], "chebyshev5", "b2relu", dev, perm=g["perm"])
    x = T(np.random.RandomState(3).randn(9, 360, 15).astype(np.float32), dev)
    lib = _lib.lib()
    c0 = lib.gcnb_launch_count()
    with torch.no_grad():
        a = model(x)
    torch.cuda.synchronize()
    launches = lib.gcnb_launch_count() - c0
    b = model(x)          # grad enabled: one launch per layer
    assert torch.equal(a, b.detach())
    assert launches <= 4, launches   # layer 1, the stack of layers 2-6, mean over filters (+ nothing else from this library)


def test_fit_runs_through_the_input_pipeline(dev, graph_l4):
    """train.fit (the reference's training loop, models_gcn.py:112-184) with a FusedTrainer feeds the batches through
    train.InputPipeline: the loss history is finite, reproducible, and the parameters move."""
    from gcn_fmri_decoding_b200 import synth
    from gcn_fmri_decoding_b200.train import FusedTrainer, fit

    g = graph_l4
    data = synth.bold_windows(64, seed=9)
    labels = synth.labels(64, seed=9)

    def run():
        model = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
        model.batch_size, model.num_epochs, model.eval_frequency, model.dropout = 16, 2, 10 ** 9, 0.5
        tr = FusedTrainer(model, distributed=False, use_cuda_graph=True, dropout_seed=5)
        p0 = tr.flat_p.clone()
        losses = fit(model, data, labels, trainer=tr, seed=3, verbose=False)
        return losses, float((tr.flat_p - p0).abs().max())

    a, moved = run()
    b, _ = run()
    assert len(a) == 8 and np.all(np.isfinite(a)) and moved > 0
    assert a == b

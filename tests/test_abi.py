"""CPU-side checks of the boundary: the C-ABI library loads and exports every declared symbol;
host-side validation raises like the reference's asserts.  No compute calls (no GPU here)."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_library_exports_every_declared_symbol():
    from gcn_fmri_decoding_b200 import _lib

    header = open(os.path.join(ROOT, "include", "gcnb200.h")).read()
    declared = set(re.findall(r"GCNB_API\s+[\w\s\*]+?\b(gcnb_\w+)\s*\(", header))
    assert len(declared) >= 15
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.lib()  # raises if the .so is missing: the product has no fallback
    for name in declared:
        assert hasattr(lib, name)
    assert lib.gcnb_version() >= 100
    assert isinstance(_lib.last_error(), str)


def test_workspace_queries_are_pure_host_calls():
    from gcn_fmri_decoding_b200 import _lib

    lib = _lib.lib()
    fwd = lib.gcnb_cheb_workspace_bytes(512, 400, 3684, 15, 32, 5, 4, 0, 0, _lib.ALGO_GENERAL)
    bwd = lib.gcnb_cheb_workspace_bytes(512, 400, 3684, 15, 32, 5, 4, 1, 1, _lib.ALGO_GENERAL)
    assert fwd >= 4 * (5 * 400 * 512 * 15 + 400 * 512 * 32)
    assert bwd > fwd
    assert lib.gcnb_spectral_workspace_bytes(8, 100, 8, 16, 4, 1) > lib.gcnb_spectral_workspace_bytes(8, 100, 8, 16, 4, 0)
    # vertex-level graph (BASELINE config 5): the general path needs the whole K-order stack (+ the G stack for dx)
    B, M, nnz, Fin, Fout, K = 64, 32492, 196396, 15, 32, 25
    slab = 4 * B * M * Fin
    fwd5 = lib.gcnb_cheb_workspace_bytes(B, M, nnz, Fin, Fout, K, 1, 0, 0, _lib.ALGO_AUTO)
    bwd5 = lib.gcnb_cheb_workspace_bytes(B, M, nnz, Fin, Fout, K, 1, 1, 1, _lib.ALGO_AUTO)
    assert K * slab < fwd5 < K * slab + 8 * B * M * (Fout + 8)
    assert 2 * K * slab < bwd5 < 2 * K * slab + 16 * B * M * (Fout + 8)
    # saved-basis width: padded feature count for graphs the fused kernels hold, Fin (vertex-major stack) otherwise
    assert lib.gcnb_cheb_stack_width(512, 400, 3684, 15, 32, 5, 4) == 16
    assert lib.gcnb_cheb_stack_width(B, M, nnz, Fin, Fout, K, 1) == Fin
    assert lib.gcnb_cheb_fused_supported(B, M, nnz, Fin, Fout, K, 1, 0, 0) == 0


def test_missing_library_fails_loudly(monkeypatch):
    from gcn_fmri_decoding_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libgcnb200.so")
    with pytest.raises(_lib.GcnbError, match="no CPU fallback"):
        _lib.lib()


def test_constructor_checks_mirror_reference(graph_l4):
    """cgcnn.__init__ validation (models_gcn.py:452-460) -- raised before any device work."""
    from gcn_fmri_decoding_b200.models import cgcnn

    L = graph_l4["L"]
    with pytest.raises(ValueError, match="len"):
        cgcnn(L=L, F=[32, 32], K=[5], p=[4, 4], M=[22], device="cpu")
    with pytest.raises(ValueError, match="powers of 2"):
        cgcnn(L=L, F=[32], K=[5], p=[3], M=[22], device="cpu")
    with pytest.raises(ValueError, match="coarsening levels"):
        cgcnn(L=L[:2], F=[32, 32], K=[5, 5], p=[4, 4], M=[22], device="cpu")
    with pytest.raises(ValueError, match="filter"):
        cgcnn(L=L, F=[32], K=[5], p=[4], M=[22], filter="spline", device="cpu")
    with pytest.raises(ValueError, match="pool"):
        cgcnn(L=L, F=[32], K=[5], p=[4], M=[22], pool="apool1", device="cpu")


def test_model_parameter_layout_and_tf_names(graph_l4):
    """Shapes and names a reference checkpoint maps onto (SURVEY 8a row a11); host tensors only."""
    from gcn_fmri_decoding_b200.models import cgcnn

    m = cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu")
    assert [l.shape[0] for l in m.L] == [400, 100]  # L[0] and L[2] (models_gcn.py:462-469)
    sd = m.state_dict_tf()
    assert list(sd) == ["conv1/weights", "conv1/bias", "conv2/weights", "conv2/bias", "fc1/weights", "fc1/bias",
                        "fc2/weights", "fc2/bias", "logits/weights", "logits/bias"]
    assert sd["conv1/weights"].shape == (75, 32) and sd["conv2/weights"].shape == (160, 32)
    assert sd["conv1/bias"].shape == (1, 1, 32) and sd["fc1/weights"].shape == (25, 512)
    assert sum(v.size for v in sd.values()) == 157878  # SURVEY 8e message size
    assert np.all(sd["conv1/bias"] == np.float32(0.2)) and abs(sd["conv1/weights"]).max() <= 0.4 + 1e-6
    m2 = cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu", seed=3)
    m2.load_state_dict_tf(sd)
    assert all(np.array_equal(a, b) for a, b in zip(sd.values(), m2.state_dict_tf().values()))
    b2 = cgcnn(L=graph_l4["L"][:2], F=[32] * 6, K=[5] * 6, p=[1] * 6, M=[512, 256, 22], channel=15,
               brelu="b2relu", device="cpu")
    assert b2.state_dict_tf()["conv3/bias"].shape == (1, 400, 32)
    four = cgcnn(L=graph_l4["L"][2:], F=[8], K=[100], p=[2], M=[22], channel=4, filter="fourier", device="cpu")
    assert four.state_dict_tf()["conv1/weights"].shape == (100, 8, 4)


def test_layers_refuse_cpu_tensors(graph_l4):
    import torch

    from gcn_fmri_decoding_b200.models import cgcnn

    m = cgcnn(L=graph_l4["L"][4:], F=[4], K=[2], p=[1], M=[3], channel=2, device="cpu")
    with pytest.raises((ValueError, NotImplementedError, RuntimeError)):
        m(torch.zeros(2, 25, 2))


def test_checkpoints_roundtrip_and_best_k(graph_l4, tmp_path):
    """checkpoints.py: parameters survive a save / load under the reference's TF variable names, and BestCheckpoints
    keeps the best k by value with the reference's replacement rule (checkmat.py:43-84)."""
    import json
    import os

    from gcn_fmri_decoding_b200 import checkpoints
    from gcn_fmri_decoding_b200.models import cgcnn

    def make(seed):
        return cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu", seed=seed)

    a, b = make(1), make(2)
    f = checkpoints.save_checkpoint(a, str(tmp_path / "model"), step=7)
    assert f.endswith("model-7.npz") and checkpoints.latest_checkpoint(str(tmp_path)) == f
    with np.load(f) as z:
        assert "conv1__weights" in z.files and z["conv1__weights"].shape == (75, 32) and "logits__bias" in z.files
    checkpoints.load_checkpoint(b, f)
    for k, v in a.state_dict_tf().items():
        assert np.array_equal(v, b.state_dict_tf()[k]), k
    keep = checkpoints.BestCheckpoints(str(tmp_path / "best"), num_to_keep=2, maximize=True)
    assert keep.handle(0.50, a, 1) and keep.handle(0.70, a, 2)
    assert keep.handle(0.40, a, 3) is None                    # worse than everything kept
    assert keep.handle(0.60, a, 4)                            # replaces the 0.50 checkpoint
    index = json.load(open(os.path.join(str(tmp_path / "best"), "best_checkpoints")))
    assert sorted(index.values()) == [0.60, 0.70] and not os.path.exists(str(tmp_path / "best" / "best.ckpt-1.npz"))
    assert keep.best().endswith("best.ckpt-2.npz")
    s, acc, f1 = checkpoints.classification_summary([0, 1, 1, 2], [0, 1, 2, 2], loss=0.5)
    assert abs(acc - 75.0) < 1e-9 and "3 / 4" in s
    try:
        import sklearn.metrics

        assert abs(f1 - 100 * sklearn.metrics.f1_score([0, 1, 1, 2], [0, 1, 2, 2], average="weighted")) < 1e-9
    except ImportError:
        pass


def test_legacy_pooled_six_layer_configuration():
    """The reference's older six-layer network (HCP_task_fmri_gcn_test8.py:1633-1636): F=[32,32,64,64,128,128],
    p=[1,4,1,4,1,4], K=[20,10,10,10,5,5] on a 6-level coarsening.  Host side only: Laplacian selection
    (models_gcn.py:462-469: layers 1-2 use L[0], 3-4 L[2], 5-6 L[4]), parameter shapes under the TF names, and the oracle
    running the same configuration (narrower filters) against the torch-autograd twin."""
    from gcn_fmri_decoding_b200 import graclus, synth
    from gcn_fmri_decoding_b200.models import cgcnn
    from oracle import layers_np as O
    from test_oracle import _torch_network

    _, gs, perm, L = synth.brain_graph(6)
    sizes = [l.shape[0] for l in L]
    assert len(L) == 7 and all(a == 2 * b for a, b in zip(sizes, sizes[1:]))
    F, p, K = [32, 32, 64, 64, 128, 128], [1, 4, 1, 4, 1, 4], [20, 10, 10, 10, 5, 5]
    m = cgcnn(L=L, F=F, K=K, p=p, M=[512, 256, 22], channel=15, device="cpu", perm=perm, n_input_vertices=360)
    assert [l.shape[0] for l in m.L] == [sizes[0], sizes[0], sizes[2], sizes[2], sizes[4], sizes[4]]
    sd = m.state_dict_tf()
    fin = [15] + F[:-1]
    for i in range(6):
        assert sd["conv%d/weights" % (i + 1)].shape == (fin[i] * K[i], F[i])
        assert sd["conv%d/bias" % (i + 1)].shape == (1, 1, F[i])
    assert sd["fc1/weights"].shape == (sizes[6], 512)  # mean over the 128 filters leaves one value per coarsest vertex
    # the oracle on this layer pattern (filters scaled down 8x to keep the CPU test short) against the autograd twin
    rng = np.random.RandomState(5)
    Fs = [15] + [f // 8 for f in F]
    params = [dict(W=rng.randn(Fs[i] * K[i], Fs[i + 1]) * (0.5 / np.sqrt(Fs[i] * K[i])), b=rng.randn(Fs[i + 1]) * 0.1,
                   K=K[i], p=p[i]) for i in range(6)]
    Ls = O.select_laplacians(L, p)
    assert [l.shape[0] for l in Ls] == [l.shape[0] for l in m.L]
    x = graclus.perm_data_3d(synth.bold_windows(3, seed=9), perm).astype(np.float64)
    labels = synth.labels(3, seed=9)
    dims = (sizes[6], 6, 5, 22)
    fcs = [(rng.randn(dims[i], dims[i + 1]) * 0.3, rng.randn(dims[i + 1]) * 0.1) for i in range(3)]
    val, cg, fg = O.network_step(x, labels, Ls, params, fcs, 5e-4, dtype=np.float64)
    tval, _, tW, tb, tfW, tfb = _torch_network(x, labels, Ls, params, fcs, 5e-4, "chebyshev5", "b1relu")
    assert np.isfinite(val) and abs(val - tval) <= 1e-11 * abs(tval)
    for i in range(6):
        # T_19 of the recursion amplifies rounding: gradients agree to 1e-9 of their largest entry
        assert np.abs(cg[i]["dW"] - tW[i]).max() <= 1e-9 * np.abs(tW[i]).max(), i
        assert np.abs(np.asarray(cg[i]["db"]).reshape(tb[i].shape) - tb[i]).max() <= 1e-9 * np.abs(tb[i]).max(), i
    for i in range(3):
        assert np.abs(fg[i][0] - tfW[i]).max() <= 1e-9 * np.abs(tfW[i]).max(), i


def test_classification_report_and_confusion_matrix_match_sklearn():
    """checkpoints.classification_report / confusion_matrix (what the reference's evaluate prints with target_name,
    models_gcn.py:94-101) against scikit-learn, including a class that is never predicted and one without support."""
    import sklearn.metrics

    from gcn_fmri_decoding_b200 import checkpoints

    rng = np.random.RandomState(4)
    names = ["task%d" % i for i in range(6)]
    y = rng.randint(0, 5, 300)                      # class 5 has no support
    pred = np.where(rng.rand(300) < 0.7, y, rng.randint(0, 6, 300))
    pred[pred == 3] = 2                             # class 3 is never predicted
    text, rows = checkpoints.classification_report(y, pred, names)
    ref = sklearn.metrics.classification_report(y, pred, labels=range(6), target_names=names, output_dict=True,
                                                zero_division=0)
    for name in names + ["macro avg", "weighted avg"]:
        for got, key in zip(rows[name], ("precision", "recall", "f1-score", "support")):
            assert abs(got - ref[name][key]) <= 1e-12, (name, key)
    assert abs(rows["accuracy"][0] - sklearn.metrics.accuracy_score(y, pred)) <= 1e-12
    assert all(n in text for n in names) and "weighted avg" in text
    C = checkpoints.confusion_matrix(y, pred, 6)
    assert np.array_equal(C, sklearn.metrics.confusion_matrix(y, pred, labels=range(6)))
    s, acc, f1 = checkpoints.classification_summary(y, pred)
    assert abs(f1 - 100 * sklearn.metrics.f1_score(y, pred, average="weighted")) <= 1e-9
    assert abs(acc - 100 * sklearn.metrics.accuracy_score(y, pred)) <= 1e-9


def test_he_initialiser_follows_tf_contrib_variance_scaling(graph_l4):
    """initial='he' (models_gcn.py:334-337, the production setting of model.py): truncated normal of stddev
    sqrt(1.3 * 2 / fan_in) with tf.contrib's fan_in = shape[-2] * prod(shape[:-2]); nothing beyond two stddev."""
    from gcn_fmri_decoding_b200.models import cgcnn

    m = cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu", initial="he")
    sd = m.state_dict_tf()
    for name, fan_in in (("conv1/weights", 75), ("conv2/weights", 160), ("fc1/weights", 25), ("fc2/weights", 512)):
        s = np.sqrt(1.3 * 2.0 / fan_in)
        w = sd[name]
        assert abs(w).max() <= 2 * s * (1 + 1e-6), name
        assert abs(w.std() / (0.87962566 * s) - 1) < 0.05, (name, w.std(), s)   # std of a 2-sigma truncated normal
    assert np.all(sd["conv1/bias"] == np.float32(0.2))
    f = cgcnn(L=graph_l4["L"][2:], F=[8], K=[0], p=[2], M=[22], channel=4, filter="fourier", device="cpu", initial="he")
    w = f.state_dict_tf()["conv1/weights"]          # [M=100, Fout=8, Fin=4]: fan_in = 8 * 100
    s = np.sqrt(2.6 / 800)
    assert w.shape == (100, 8, 4) and abs(w).max() <= 2 * s * (1 + 1e-6) and abs(w.std() / (0.87962566 * s) - 1) < 0.05


def test_reference_style_fit_and_small_methods(graph_l4, tmp_path, monkeypatch, capsys):
    """cgcnn.fit / get_var / probabilities / prediction with the reference's signatures and return values
    (models_gcn.py:112-191, :241-251).  Host logic only: the step and the evaluation are stubbed (they need the GPU and
    are covered by the GPU tests); checked here: step count, evaluation points, best-3 checkpoint bookkeeping, the
    (accuracies, losses, t_step) tuple."""
    import json
    import os

    import torch

    from gcn_fmri_decoding_b200.models import cgcnn

    m = cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu",
              batch_size=8, num_epochs=3, eval_frequency=4, dropout=0.5, dir_name="run1")
    assert np.array_equal(m.get_var("conv1/weights:0"), m.state_dict_tf()["conv1/weights"])
    assert m.get_var("logits/bias").shape == (22,)
    with pytest.raises(KeyError):
        m.get_var("conv7/weights")
    lg = torch.tensor([[0.0, 2.0, 1.0], [3.0, 0.0, 0.0]])
    assert m.prediction(lg).tolist() == [1, 0] and torch.allclose(m.probabilities(lg).sum(1), torch.ones(2))

    seen = []

    class StubTrainer:
        def step(self, x, y, dropout=None):
            assert tuple(x.shape) == (8, 360, 15) and x.dtype == torch.float32 and y.dtype == torch.long and dropout == 0.5
            seen.append(y.clone())
            return torch.tensor(1.0 / len(seen)), None

    accs = iter([40.0, 55.0, 50.0, 60.0, 45.0, 58.0])
    monkeypatch.setattr(m, "evaluate", lambda d, l, **kw: ("accuracy: stub", next(accs), 0.0, 0.25))
    data = np.zeros((32, 360, 15), np.float32)
    labels = np.arange(32) % 21
    np.random.seed(0)
    accuracies, losses, t_step = m.fit(data, labels, data[:8], labels[:8], best_checkpoint_dir=str(tmp_path / "best"),
                                       trainer=StubTrainer())
    assert len(seen) == 12                                   # int(3 epochs * 32 / 8)
    assert accuracies == [40.0, 55.0, 50.0] and losses == [0.25] * 3 and t_step > 0      # evaluated at steps 4, 8, 12
    # every window is used once per pass before any is used twice (the reference's deque of permutations)
    first_pass = torch.cat(seen[:4]).numpy()
    assert sorted(first_pass.tolist()) == sorted(labels.tolist())
    index = json.load(open(tmp_path / "best" / "best_checkpoints"))
    assert index == {"best.ckpt-4.npz": 40.0, "best.ckpt-8.npz": 55.0, "best.ckpt-12.npz": 50.0}
    assert all(os.path.exists(tmp_path / "best" / k) for k in index)
    out = capsys.readouterr().out
    assert "training with 12 steps in total with batch_size=8 and epochs=3 for training_set=32:" in out
    assert "validation accuracy: peak = 55.00, mean = 48.33" in out and "step 12 / 12 (epoch 3.00 / 3):" in out


def test_model_perf_harness(graph_l4, tmp_path, monkeypatch, capsys):
    """perf.model_perf (models_gcn.py:936-1075): test() book-keeping and predict()'s checkpoint choice, reports and
    per-subject / per-time-point tables against scikit-learn.  The network itself is stubbed (GPU code)."""
    import sklearn.metrics

    from gcn_fmri_decoding_b200 import checkpoints, tf_bundle
    from gcn_fmri_decoding_b200.models import cgcnn
    from gcn_fmri_decoding_b200.perf import model_perf

    def make(seed):
        return cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 6], channel=15, device="cpu", seed=seed)

    trained, m = make(1), make(2)
    run = tmp_path / "run"
    # a run directory as the reference's BestCheckpointSaver leaves it: the state file lists the kept checkpoints best first
    tf_bundle.save_tf_checkpoint(make(5), str(run / "model" / "best.ckpt"), step=100)
    tf_bundle.save_tf_checkpoint(trained, str(run / "model" / "best.ckpt"), step=300)
    (run / "model" / "checkpoint").write_text('model_checkpoint_path: "best.ckpt-300"\n'
                                              'all_model_checkpoint_paths: "best.ckpt-300"\n'
                                              'all_model_checkpoint_paths: "best.ckpt-100"\n')
    rng = np.random.RandomState(2)
    n_sub, per_sub, names = 4, 34, ["t%d" % i for i in range(6)]
    y = rng.randint(0, 6, n_sub * per_sub)
    pred = np.where(rng.rand(len(y)) < 0.6, y, rng.randint(0, 6, len(y))).astype(np.float64)
    logits = rng.randn(len(y), 6).astype(np.float32)
    calls = {}

    def fake_predict(data, labels=None, return_logits=False):
        calls["bs"] = m.batch_size
        return pred, 0.125, logits

    monkeypatch.setattr(m, "predict", fake_predict)
    perf = model_perf()
    lg, pl, loss, acc = perf.predict(run, np.zeros((len(y), 360, 15), np.float32), y, target_name=names, batch_size=64, model=m)
    assert calls["bs"] == 64 and m.batch_size != 64                      # the harness' batch size, then restored
    assert all(np.array_equal(v, m.state_dict_tf()[k]) for k, v in trained.state_dict_tf().items())   # best.ckpt-300
    assert lg is logits and np.array_equal(pl, pred) and loss == 0.125 * len(y) / 64       # the SUM of the batch losses
    assert abs(acc[0] - 100 * sklearn.metrics.accuracy_score(y, pred)) < 1e-9
    out = capsys.readouterr().out
    assert "Confusion Matrix:" in out and "f1 (weighted):" in out and "best.ckpt-300" in out
    _, _, _, table = perf.predict(run, None, y, target_name=names, model=m, sub_name=["s%d" % i for i in range(n_sub)])
    assert table.shape == (n_sub, 7)
    ys, ps = y.reshape(n_sub, -1), pred.reshape(n_sub, -1)
    for si in range(n_sub):
        assert abs(table[si, -1] - sklearn.metrics.f1_score(ys[si], ps[si], average="weighted")) < 1e-12
        for li in range(6):
            mask = ys[si] == li
            assert abs(table[si, li] - sklearn.metrics.f1_score(ys[si, mask], ps[si, mask], average="weighted")) < 1e-12
    _, _, _, per_t = perf.predict(run, None, y, target_name=names, model=m, trial_dura=17, flag_starttr=True)
    yt, pt = y.reshape(-1, 17), pred.reshape(-1, 17)
    assert per_t.shape == (6, 17)
    mask = yt[:, 3] == 2
    assert abs(per_t[2, 3] - 100 * sklearn.metrics.accuracy_score(yt[mask, 3], pt[mask, 3])) < 1e-9
    with pytest.raises(ValueError, match="model="):
        perf.predict(run, None, y, target_name=names)
    # without TensorFlow's state file: the best of a BestCheckpoints index
    run2 = tmp_path / "run2"
    keep = checkpoints.BestCheckpoints(str(run2 / "model"), num_to_keep=3)
    keep.handle(0.4, make(7), 10), keep.handle(0.9, trained, 20), keep.handle(0.5, make(8), 30)
    m2 = make(9)
    monkeypatch.setattr(m2, "predict", fake_predict)
    perf.predict(run2, None, y, model=m2)
    assert all(np.array_equal(v, m2.state_dict_tf()[k]) for k, v in trained.state_dict_tf().items())
    # test(): fit + two evaluations, figures stored under the experiment's name
    monkeypatch.setattr(m, "fit", lambda *a, **k: ([50.0, 60.0], [1.0, 0.8], 0.01))
    monkeypatch.setattr(m, "evaluate", lambda d, l, target_name=None: ("accuracy: stub", float(len(l)), 1.0, 0.5))
    perf.test(m, "cheby", dict(K=5), None, [0] * 7, None, None, None, [0] * 3)
    assert perf.names == {"cheby"} and perf.fit_accuracies["cheby"] == [50.0, 60.0] and perf.fit_time["cheby"] == 0.01
    assert perf.train_accuracy["cheby"] == 7.0 and perf.test_accuracy["cheby"] == 3.0 and perf.params["cheby"] == dict(K=5)


def test_fused_trainer_refuses_ambiguous_input_layout(graph_l4):
    """perm set and no fake vertices added: raw and permuted batches have the same shape -- the trainer asks (as
    cgcnn.forward does) instead of guessing.  Raised before any device work."""
    from gcn_fmri_decoding_b200.models import cgcnn
    from gcn_fmri_decoding_b200.train import FusedTrainer

    m = cgcnn(L=graph_l4["L"][4:], F=[4], K=[2], p=[1], M=[3], channel=2, device="cpu", perm=np.arange(25),
              n_input_vertices=25)
    with pytest.raises(ValueError, match="gather=True"):
        FusedTrainer(m, distributed=False)
    import torch

    with pytest.raises(ValueError, match="gather=True"):
        m.inference(torch.zeros(2, 25, 2))


def test_c_abi_from_plain_c(tmp_path):
    """include/gcnb200.h is a C header (C99, -pedantic -Werror) and the library links and answers from plain C exactly
    as through ctypes -- the boundary a cgo / JNI / N-API binding would use.  Host-only calls, no GPU."""
    import shutil
    import subprocess

    from gcn_fmri_decoding_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    libdir = os.path.dirname(_lib.LIB_PATH)
    exe = str(tmp_path / "abi_host_calls")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "abi_c", "abi_host_calls.c"), "-o", exe, "-L", libdir,
                    "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir], check=True)
    out = dict(line.split(" ", 1) for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())
    lib = _lib.lib()
    assert int(out["version"]) == lib.gcnb_version()
    assert int(out["tap_bytes"]) == lib.gcnb_cheb_tap_image_bytes(32, 32, 5) == 2 * 5 * 32 * 32 * 4 + 5 * 32 * 32 * 2
    assert int(out["tap_bytes_unsupported"]) == 0
    M = 8
    rows = [[j for j in (i - 1, i + 1) if 0 <= j < M] for i in range(M)]
    rp = np.cumsum([0] + [len(r) for r in rows]).astype(np.int32)
    ci = np.array([j for r in rows for j in r], np.int32)
    v = np.full(len(ci), -0.5, np.float32)
    n = lib.gcnb_cheb_image_bytes(rp.ctypes.data, ci.ctypes.data, 4, M, len(ci), 16, 8, 3, 2, 0)
    img = np.zeros(n, np.uint8)
    _lib.check(lib.gcnb_cheb_image_build(rp.ctypes.data, ci.ctypes.data, v.ctypes.data, 4, M, len(ci), 16, 8, 3, 2, 0,
                                         img.ctypes.data, n), "image")
    f = out["image_bytes"].split()
    assert int(f[0]) == n > 0 and int(f[2]) == 0 and int(f[4]) == int(img.astype(np.uint64).sum())
    assert out["wrong_size"].split() == ["rc", "-1", "error_set", "1"]


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under gcn_fmri_decoding_b200/ may import it (only tests/,
    __graft_entry__.smoke() and bench.py's CPU legs do), and the package has no CPU compute fallback to route through."""
    import ast
    import glob

    pkg = os.path.join(ROOT, "gcn_fmri_decoding_b200")
    for path in glob.glob(os.path.join(pkg, "**", "*.py"), recursive=True):
        tree = ast.parse(open(path).read())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            assert not any(n == "oracle" or n.startswith("oracle.") for n in names), path
    # bench.py imports the oracle only inside its CPU-baseline functions
    tree = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    for node in tree.body:
        if isinstance(node, (ast.Import, ast.ImportFrom)):
            mod = node.module if isinstance(node, ast.ImportFrom) else ",".join(a.name for a in node.names)
            assert "oracle" not in (mod or ""), "bench.py must not import the oracle at module level"


def test_planner_queries_over_random_shapes():
    """The host-side planners (dispatch / workspace / basis-width / describe queries) over 400 seeded random layer shapes,
    including degenerate and oversized ones: they never fail, answer deterministically, and agree with each other --
    every call (saved basis or not, with or without dx, each algo) takes one of the enumerated routes and the workspace
    query covers that route, the AUTO workspace is no larger than the larger of the two kernel families', sizes are
    multiples of 256 bytes, the saved-basis width is 0, Fin, or Fin padded to a power of two, and the forward
    description names a kernel."""
    from gcn_fmri_decoding_b200 import _lib

    lib = _lib.lib()
    rng = np.random.RandomState(77)
    routes = {0: ("k_cheb_fwd_umma<FP=16>", "k_cheb_fwd_umma<FP=32>", "k_cheb_fwd_fused", "general path", "unsupported"),
              1: ("stack-dW", "stack-dW + tcgen05 adjoint", "stack-dW + fused dx", "fused recompute", "general path",
                  "unsupported")}
    seen_fused = seen_general = 0
    for _ in range(400):
        B = int(rng.choice([1, 2, 7, 16, 64, 128, 512, 600]))
        M = int(rng.choice([4, 24, 25, 100, 372, 400, 1000, 2048, 4096, 32492]))
        p = int(rng.choice([1, 2, 4, 8]))
        Fin, Fout = int(rng.randint(1, 65)), int(rng.randint(1, 65))
        K = int(rng.randint(1, 31))
        nnz = int(M * rng.randint(0, 20))
        shape = (B, M, nnz, Fin, Fout, K, p)
        fused = [lib.gcnb_cheb_fused_supported(*shape, bwd, dx) for bwd, dx in ((0, 0), (1, 0), (1, 1))]
        assert all(f in (0, 1) for f in fused)
        assert fused == [lib.gcnb_cheb_fused_supported(*shape, bwd, dx) for bwd, dx in ((0, 0), (1, 0), (1, 1))]
        for (bwd, dx), f in zip(((0, 0), (1, 0), (1, 1)), fused):
            auto = lib.gcnb_cheb_workspace_bytes(*shape, bwd, dx, _lib.ALGO_AUTO)
            general = lib.gcnb_cheb_workspace_bytes(*shape, bwd, dx, _lib.ALGO_GENERAL)
            fused_ws = lib.gcnb_cheb_workspace_bytes(*shape, bwd, dx, _lib.ALGO_FUSED)
            assert 0 <= auto < 2 ** 48 and 0 <= general < 2 ** 48 and 0 <= fused_ws < 2 ** 48
            assert auto <= max(fused_ws, general), (shape, bwd, dx, auto, fused_ws, general)
            assert auto % 256 == 0 and general % 256 == 0
            for algo, query in ((_lib.ALGO_AUTO, auto), (_lib.ALGO_GENERAL, general), (_lib.ALGO_FUSED, fused_ws)):
                for saved in (False, True):
                    text, need = _lib.describe(*shape, bwd, dx, saved, algo)
                    assert text.split(":")[0] in routes[bwd], (shape, bwd, dx, saved, algo, text)
                    assert need <= query and need % 256 == 0, (shape, bwd, dx, saved, algo, text, need, query)
        width = lib.gcnb_cheb_stack_width(*shape)
        assert width == 0 or (width >= Fin and width in (Fin, 8, 16, 32, 64)), (shape, width)
        text = _lib.describe_fwd(*shape)
        assert text and ("k_" in text or "general" in text.lower() or "unsupported" in text.lower()), text
        seen_fused += fused[0]
        seen_general += 1 - fused[0]
    assert seen_fused > 20 and seen_general > 20


def test_predict_pads_the_last_batch_and_returns_what_the_reference_returns(graph_l4, monkeypatch):
    """cgcnn.predict (models_gcn.py:31-71) with the network stubbed: zero-padded last batch, predictions cropped to the
    data set, loss = sum of batch losses * batch_size / size, and the three return forms."""
    import torch

    from gcn_fmri_decoding_b200.models import cgcnn

    m = cgcnn(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu", batch_size=8)
    batches = []

    def fake_forward(x, dropout=1.0, gather=None):
        batches.append(x.clone())
        lg = torch.zeros(x.shape[0], 22)
        lg[torch.arange(x.shape[0]), (x[:, 0, 0].long() % 22)] = 5.0     # class = first value of the window
        return lg

    monkeypatch.setattr(m, "forward", fake_forward)
    data = np.zeros((19, 360, 15), np.float32)
    data[:, 0, 0] = np.arange(19) + 1
    labels = (np.arange(19) + 1) % 22
    preds = m.predict(data)
    assert isinstance(preds, np.ndarray) and preds.shape == (19,) and np.array_equal(preds, labels)
    assert [tuple(b.shape) for b in batches] == [(8, 360, 15)] * 3 and float(batches[2][3:].abs().sum()) == 0.0   # padding
    preds, loss = m.predict(data, labels)
    per_batch = []
    for b in range(3):
        lab = np.zeros(8, np.int64)
        chunk = labels[8 * b:8 * b + 8]
        lab[:len(chunk)] = chunk
        per_batch.append(float(m.loss(fake_forward(torch.as_tensor(np.pad(data[8 * b:8 * b + 8], ((0, 8 - len(chunk)), (0, 0), (0, 0))))),
                                     torch.as_tensor(lab))))
    assert abs(loss - sum(per_batch) * 8 / 19) < 1e-6
    preds2, loss2, logits = m.predict(data, labels, return_logits=True)
    assert np.array_equal(preds2, preds) and loss2 == loss and logits.shape == (19, 22) and np.array_equal(logits.argmax(1), labels)
    preds3, logits3 = m.predict(data, return_logits=True)
    assert np.array_equal(preds3, preds) and np.array_equal(logits3, logits)

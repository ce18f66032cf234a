"""Fine-tuning on the host: the fp64 references of the head step and of TF Nadam (``head_step``, ``nadam_tf``, built from
``oracle.layers_np`` and imported by the GPU tests), the ``finetuning_cgcnn`` constructor (conv variables from a
``cgcnn``, an ``.npz`` checkpoint or a TF V2 checkpoint, copied and frozen) and the batches its ``fit`` draws.
The device side is in ``test_gpu_finetune.py``."""
import numpy as np
import pytest

from oracle import layers_np as O

torch = pytest.importorskip("torch")


def _conv_params(Ls, F, K, p, Fin, rng):
    out = []
    for Fo, k, pp in zip(F, K, p):
        out.append(dict(W=(rng.randn(Fin * k, Fo) * 0.3).astype(np.float32), b=(rng.randn(Fo) * 0.1).astype(np.float32),
                        K=k, p=pp))
        Fin = Fo
    return out


def _fcs(widths, rng):
    return [((rng.randn(a, b) * 0.3).astype(np.float32), (rng.randn(b) * 0.1).astype(np.float32))
            for a, b in zip(widths[:-1], widths[1:])]


def head_step(a0, labels, fcs, regularization, dropout_masks=None, keep=1.0, dtype=np.float32):
    """Reference of the fine-tuning step's head, the head half of ``oracle.layers_np.network_step``: forward, loss and
    backward of the FC layers on ``a0 [B, n0]`` (the mean over the last conv layer's filters), with the same op order --
    so the FC gradients equal ``network_step``'s bit for bit on the same trace.  The loss's L2 term covers the FC variables only (the conv layers are frozen when fine-tuning,
    models_gcn.py:685-933).  Returns ``(loss, fc_grads)``."""
    acts = [np.asarray(a0, dtype)]
    for i, (W, b) in enumerate(fcs):
        z = acts[-1] @ np.asarray(W, dtype) + np.asarray(b, dtype)
        if i < len(fcs) - 1:
            z = np.maximum(z, 0)
            if dropout_masks is not None:
                z = (z * np.asarray(dropout_masks[i], dtype) / dtype(keep)).astype(dtype)
        acts.append(z)
    logits = acts[-1]
    value = O.loss(logits.astype(np.float64), labels, [v for Wb in fcs for v in Wb], regularization)
    B = acts[0].shape[0]
    pz = np.exp(logits - logits.max(axis=1, keepdims=True))
    pz /= pz.sum(axis=1, keepdims=True)
    pz[np.arange(B), labels] -= 1
    d = (pz / B).astype(dtype)
    fc_grads = [None] * len(fcs)
    for i in range(len(fcs) - 1, -1, -1):
        W, b = fcs[i]
        if i < len(fcs) - 1:
            d = d * (acts[i + 1] > 0)
            if dropout_masks is not None:
                d = (d / dtype(keep)).astype(dtype)
        fc_grads[i] = (acts[i].T @ d + regularization * np.asarray(W, dtype), d.sum(0) + regularization * np.asarray(b, dtype))
        d = d @ np.asarray(W, dtype).T
    return value, fc_grads


def nadam_tf(p, g, m, v, t, lr, b1, b2, eps, reg, decay):
    """Reference of ``gcnb_nadam_tf_f32``: one ``tf.contrib.opt.NadamOptimizer`` step in fp64 (TF's ``ApplyAdam`` with
    ``use_nesterov=True``), with the L2 term folded in where ``decay`` is set; ``t`` is the step's 1-based count.
        g' = g + reg p;  m = m + (1-b1)(g' - m);  v = v + (1-b2)(g'^2 - v)
        p = p - lr sqrt(1-b2^t)/(1-b1^t) (b1 m + (1-b1) g') / (sqrt(v) + eps)
    Not the momentum schedule of Keras' Nadam or ``torch.optim.NAdam``.  Returns ``(p, m, v)``."""
    p, g, m, v = (np.asarray(a, np.float64) for a in (p, g, m, v))
    g = g + reg * p * (np.asarray(decay) != 0)
    m = m + (1 - b1) * (g - m)
    v = v + (1 - b2) * (g * g - v)
    lr_t = lr * np.sqrt(1 - b2 ** t) / (1 - b1 ** t)
    return p - lr_t * (b1 * m + (1 - b1) * g) / (np.sqrt(v) + eps), m, v


@pytest.mark.parametrize("keep", [1.0, 0.5])
def test_head_step_is_the_head_half_of_network_step(graph_l4, keep):
    """head_step on the mean of the conv stack's output gives network_step's FC gradients bit for bit."""
    rng = np.random.RandomState(3)
    Ls = O.select_laplacians(graph_l4["L"], [4, 4])
    params = _conv_params(Ls, [8, 8], [3, 3], [4, 4], 4, rng)
    B = 6
    x = rng.randn(B, Ls[0].shape[0], 4).astype(np.float32)
    labels = rng.randint(0, 5, B)
    fcs = _fcs([25, 16, 12, 5], rng)
    masks = None if keep == 1.0 else [O.counter_dropout_mask(B, 16, keep, 11, 0), O.counter_dropout_mask(B, 12, keep, 12, 0)]
    _, _, want = O.network_step(x, labels, Ls, params, fcs, 5e-4, dropout_masks=masks, keep=keep)
    h = O.conv_stack(x, Ls, params)
    value, got = head_step(h.mean(axis=-1, dtype=np.float32), labels, fcs, 5e-4, dropout_masks=masks, keep=keep)
    for (gw, gb), (ww, wb) in zip(got, want):
        assert np.array_equal(gw, ww) and np.array_equal(gb, wb)
    assert np.isfinite(value)


def test_head_step_matches_central_differences():
    rng = np.random.RandomState(4)
    B, widths, reg, keep = 5, [6, 9, 7, 4], 3e-2, 0.5
    a0 = rng.rand(B, widths[0])
    labels = rng.randint(0, widths[-1], B)
    fcs = [(W.astype(np.float64), b.astype(np.float64)) for W, b in _fcs(widths, rng)]
    masks = [O.counter_dropout_mask(B, w, keep, 21 + i, 0) for i, w in enumerate(widths[1:-1])]
    f = lambda fc: head_step(a0, labels, fc, reg, dropout_masks=masks, keep=keep, dtype=np.float64)
    _, grads = f(fcs)
    eps = 1e-6
    for layer in range(len(fcs)):
        for which in (0, 1):
            g = grads[layer][which]
            for idx in list(np.ndindex(g.shape))[::3]:
                plus = [(W.copy(), b.copy()) for W, b in fcs]
                minus = [(W.copy(), b.copy()) for W, b in fcs]
                plus[layer][which][idx] += eps
                minus[layer][which][idx] -= eps
                fd = (f(plus)[0] - f(minus)[0]) / (2 * eps)
                assert abs(fd - g[idx]) <= 1e-6 * max(1.0, abs(fd)), (layer, which, idx, fd, g[idx])


def test_nadam_first_step_known_answer():
    """From zero moments the first Nadam step moves p by lr (1 + b1) g / (|g| + eps / sqrt(1 - b2)); Adam's has no
    (1 + b1) factor."""
    rng = np.random.RandomState(5)
    p, g = rng.randn(50), rng.randn(50)
    lr, b1, b2, eps = 1e-3, 0.9, 0.999, 1e-8
    z = np.zeros(50)
    p1, m1, v1 = nadam_tf(p, g, z, z, 1, lr, b1, b2, eps, 0.0, np.zeros(50))
    want = lr * (1 + b1) * g / (np.abs(g) + eps / np.sqrt(1 - b2))
    np.testing.assert_allclose(p - p1, want, rtol=1e-12, atol=0)
    np.testing.assert_allclose(m1, (1 - b1) * g, rtol=1e-15)
    np.testing.assert_allclose(v1, (1 - b2) * g * g, rtol=1e-15)
    adam = lr * g / (np.abs(g) + eps / np.sqrt(1 - b2))
    assert np.all(np.abs((p - p1) / adam - (1 + b1)) < 1e-6)


def test_nadam_with_zero_beta1_is_adam():
    rng = np.random.RandomState(6)
    n, lr, b2, eps, reg = 40, 1e-2, 0.99, 1e-8, 0.1
    decay = rng.rand(n) < 0.5
    p = q = rng.randn(n)
    m = v = np.zeros(n)
    ma, va = m, v
    for t in range(1, 6):
        g = rng.randn(n)
        p, m, v = nadam_tf(p, g, m, v, t, lr, 0.0, b2, eps, reg, decay)
        ga = g + reg * q * decay          # TF Adam with the same L2 fold, b1 = 0
        ma = ga
        va = va + (1 - b2) * (ga * ga - va)
        q = q - lr * np.sqrt(1 - b2 ** t) * ma / (np.sqrt(va) + eps)
        np.testing.assert_allclose(p, q, rtol=1e-13, atol=1e-15)


# ------------------------------------------------------------------------------------------------ the model, on the host
def _args(graph_l4, **kw):
    a = dict(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device="cpu", seed=1,
             perm=graph_l4["perm"], n_input_vertices=360, regularization=5e-4)
    a.update(kw)
    return a


def _check_conv(ft, base):
    for i in range(len(base.p)):
        for mine, theirs in ((ft.conv_weights[i], base.conv_weights[i]), (ft.conv_bias[i], base.conv_bias[i])):
            assert torch.equal(mine, theirs.to(mine.device))
            assert mine.data_ptr() != theirs.data_ptr() and not mine.requires_grad


@pytest.mark.parametrize("source", ["cgcnn", "npz", "tf"])
def test_constructor_copies_and_freezes_the_conv_layers(graph_l4, tmp_path, source):
    from gcn_fmri_decoding_b200 import checkpoints, tf_bundle
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    base = cgcnn(**_args(graph_l4, seed=9))
    pretrained = base
    if source == "npz":
        pretrained = checkpoints.save_checkpoint(base, str(tmp_path / "pre"))
    elif source == "tf":
        pretrained = tf_bundle.write_tf_checkpoint(str(tmp_path / "pre_tf"), base.state_dict_tf())
    ft = finetuning_cgcnn(**_args(graph_l4, M=[64, 7]), pretrained=pretrained)
    _check_conv(ft, base)
    with torch.no_grad():
        base.conv_weights[0].add_(1.0)              # copied, not shared
    assert not torch.equal(ft.conv_weights[0], base.conv_weights[0])
    # the head: shapes and TF names from the new M, initialised from the seed as cgcnn does
    sd = ft.state_dict_tf()
    assert [k for k in sd if not k.startswith("conv")] == ["fc1/weights", "fc1/bias", "logits/weights", "logits/bias"]
    assert sd["fc1/weights"].shape == (25, 64) and sd["logits/weights"].shape == (64, 7) and sd["logits/bias"].shape == (7,)
    plain = cgcnn(**_args(graph_l4, M=[64, 7]))
    for k in ("fc1/weights", "fc1/bias", "logits/weights", "logits/bias"):
        assert np.array_equal(sd[k], plain.state_dict_tf()[k])
    assert all(p.requires_grad for p in list(ft.fc_weights) + list(ft.fc_bias))


def test_constructor_names_a_mismatched_conv_variable(graph_l4, tmp_path):
    from gcn_fmri_decoding_b200 import checkpoints
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    other = cgcnn(**_args(graph_l4, K=[5, 3]))
    with pytest.raises(ValueError, match="conv2/weights"):
        finetuning_cgcnn(**_args(graph_l4, M=[64, 7]), pretrained=other)
    one_layer = checkpoints.save_checkpoint(cgcnn(**_args(graph_l4, F=[32], K=[5], p=[4])), str(tmp_path / "one"))
    with pytest.raises(ValueError, match="conv2/weights"):
        finetuning_cgcnn(**_args(graph_l4, M=[64, 7]), pretrained=one_layer)


def test_fit_draws_the_batches_cgcnn_fit_draws(graph_l4, tmp_path, monkeypatch, capsys):
    """finetuning_cgcnn.fit on stubbed trunk features and a stub trainer: the same index batches as cgcnn.fit under the
    same np.random.seed, the same evaluation points and prints; the validation table it evaluates is padded."""
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    kw = dict(batch_size=8, num_epochs=3, eval_frequency=4, dropout=0.5)
    n, n_val = 36, 11
    data = np.zeros((n, 360, 15), np.float32)
    data[:, 0, 0] = np.arange(n)
    labels = np.arange(n) % 7
    val = np.zeros((n_val, 360, 15), np.float32)

    def run(model, width):
        seen = []

        class StubTrainer:
            def step(self, x, y, dropout=None):
                assert tuple(x.shape[:2]) == (8, width) and x.dtype == torch.float32 and dropout == 0.5
                seen.append(x.reshape(8, -1)[:, 0].numpy().astype(np.int64))
                return torch.tensor(1.0), None

        np.random.seed(0)
        out = model.fit(data, labels, val, labels[:n_val], best_checkpoint_dir=str(tmp_path / str(width)),
                        trainer=StubTrainer())
        return seen, out

    base = cgcnn(**_args(graph_l4, **kw))
    monkeypatch.setattr(base, "evaluate", lambda d, l, **k: ("accuracy: stub", 50.0, 0.0, 0.25))
    want, want_out = run(base, 360)

    ft = finetuning_cgcnn(**_args(graph_l4, M=[64, 7], **kw), pretrained=base)
    tables = []

    def fake_trunk(d, gather=None, padded=False):
        rows = -(-len(d) // 8) * 8 if padded else len(d)
        t = np.full((rows, 25), -1.0, np.float32)
        t[:len(d)] = d[:, :1, 0]
        return t

    def fake_eval(table, l):
        tables.append(table.shape)
        return "accuracy: stub", 50.0, 0.0, 0.25

    monkeypatch.setattr(ft, "trunk_features", fake_trunk)
    monkeypatch.setattr(ft, "evaluate_features", fake_eval)
    capsys.readouterr()
    got, got_out = run(ft, 25)
    assert len(got) == len(want) == int(3 * n / 8)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    assert got_out[:2] == want_out[:2] and tables == [(16, 25)] * 4     # steps 4, 8, 12, 13
    out = capsys.readouterr().out
    assert "training with 13 steps in total with batch_size=8 and epochs=3 for training_set=36:" in out
    assert "step 12 / 13 (epoch 2.67 / 3):" in out


def test_fit_refuses_a_cpu_model(graph_l4):
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    ft = finetuning_cgcnn(**_args(graph_l4, M=[64, 7]), pretrained=cgcnn(**_args(graph_l4)))
    with pytest.raises(ValueError, match="CUDA only"):
        ft.fit(np.zeros((4, 360, 15), np.float32), np.zeros(4, np.int64), np.zeros((2, 360, 15), np.float32),
               np.zeros(2, np.int64))

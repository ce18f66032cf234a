"""Fine-tuning on the B200: ``gcnb_nadam_tf_f32`` against ``nadam_tf``, the trunk pass against the calls
``predict`` makes, one ``HeadTrainer`` step against ``head_step`` (with the device's dropout masks), graph replay
and the input pipeline against eager steps, and ``finetuning_cgcnn.fit`` end to end.  Run on the B200 box: -m gpu."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from conftest import rel_inf
from oracle import layers_np as O
from test_finetune import head_step, nadam_tf

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def T(a, dev, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)


def _cfg2(graph_l4, dev, **kw):
    a = dict(L=graph_l4["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device=dev, seed=1,
             perm=graph_l4["perm"], n_input_vertices=360, regularization=5e-4)
    a.update(kw)
    return a


def _cfg1(graph_l1, dev, **kw):
    a = dict(L=graph_l1["L"], F=[32] * 6, K=[5] * 6, p=[1] * 6, M=[512, 256, 22], channel=15, device=dev, seed=1,
             perm=graph_l1["perm"], n_input_vertices=360, regularization=5e-4)
    a.update(kw)
    return a


def _f32(x):
    return float(np.float32(x))


def _windows(n, seed):
    from gcn_fmri_decoding_b200 import synth

    return synth.bold_windows(n, seed=seed)


# ------------------------------------------------------------------------------------------------ the kernel
def test_nadam_kernel_matches_oracle(dev):
    from gcn_fmri_decoding_b200 import _lib

    lib = _lib.lib()
    # the kernel takes fp32 hyper-parameters: the oracle gets the same values (1 - 0.999f is 1.3e-5 off 0.001)
    n, lr, b1, b2, eps, reg = 157878, *(_f32(h) for h in (1e-3, 0.9, 0.999, 1e-8, 5e-4))
    rng = np.random.RandomState(0)
    p0 = rng.randn(n).astype(np.float32)
    decay = (rng.rand(n) < 0.6).astype(np.uint8)
    grads = [(rng.randn(n) * 10.0 ** rng.uniform(-3, 1, n)).astype(np.float32) for _ in range(5)]
    vp = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def run(check):
        p, m, v = T(p0, dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)
        state = torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev)
        dk = T(decay, dev, torch.uint8)
        for t, g in enumerate(grads, 1):
            before = [a.cpu().numpy() for a in (p, m, v)]
            _lib.check(lib.gcnb_nadam_tf_f32(vp(p), vp(T(g, dev)), vp(m), vp(v), vp(dk), vp(state), n, lr, b1, b2, eps,
                                             reg, 1, stream), "gcnb_nadam_tf_f32")
            torch.cuda.synchronize()
            if check:
                want = nadam_tf(*before[:1], g, *before[1:], t, lr, b1, b2, eps, reg, decay)
                for got, w in zip((p, m, v), want):
                    assert rel_inf(got.cpu().numpy(), w) <= 1e-6, (t, rel_inf(got.cpu().numpy(), w))
                assert state[3].item() == t
        return p.cpu().numpy(), m.cpu().numpy(), v.cpu().numpy()

    first, again = run(True), run(False)
    assert all(np.array_equal(a, b) for a, b in zip(first, again))


# ------------------------------------------------------------------------------------------------ the trunk pass
@pytest.mark.parametrize("config", ["2", "1"])
def test_trunk_features_are_the_head_input_of_predict(dev, graph_l4, graph_l1, config):
    from gcn_fmri_decoding_b200 import ops
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    if config == "2":
        args, n = _cfg2(graph_l4, dev, batch_size=512), 1000
    else:
        args, n = _cfg1(graph_l1, dev, batch_size=128), 300
    base = cgcnn(**args)
    ft = finetuning_cgcnn(**args, pretrained=base)
    data = _windows(n, 7)
    got = ft.trunk_features(data)
    table = ft.trunk_features(data, padded=True)
    bs = args["batch_size"]
    assert got.shape == (n, base.fc_weights[0].shape[0]) and table.shape[0] == -(-n // bs) * bs
    assert np.array_equal(table[:n], got)
    with torch.no_grad():
        for begin in range(0, n, bs):
            batch = torch.zeros((bs, 360, 15), device=dev)
            batch[: min(bs, n - begin)] = T(data[begin:begin + bs], dev)
            want = ops.mean_f_fwd(base.conv_stack(batch, gather=True)).cpu().numpy()
            assert np.array_equal(table[begin:begin + bs], want), begin
    # the head on the cached features gives predict's logits bit for bit
    _, logits = ft.predict(data, return_logits=True)
    with torch.no_grad():
        head = np.concatenate([ft._head(T(table[b:b + bs], dev)).cpu().numpy() for b in range(0, n, bs)])[:n]
    assert np.array_equal(head, logits)


# ------------------------------------------------------------------------------------------------ one step
STEP_CASES = [("cfg2", [512, 256, 7], 512, "fused"), ("cfg2", [512, 256, 7], 2048, "fused"),
              ("wide", [512, 256, 22], 512, "layers"), ("cfg2", [64, 7], 512, "layers")]


def _head_model(graph_l4, graph_l1, dev, kind, M, bs=512):
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    if kind == "cfg2":
        args = _cfg2(graph_l4, dev, M=M, batch_size=bs, dropout=0.5)
    else:  # one conv layer on the 372-vertex graph: the head's input is 372 wide
        args = _cfg1(graph_l1, dev, F=[32], K=[5], p=[1], M=M, batch_size=bs, dropout=0.5)
    return finetuning_cgcnn(**args, pretrained=cgcnn(**dict(args, M=[8, 3], seed=3)))


@pytest.mark.parametrize("kind,M,B,path", STEP_CASES)
def test_head_step_matches_oracle(dev, graph_l4, graph_l1, kind, M, B, path):
    from gcn_fmri_decoding_b200 import _lib
    from gcn_fmri_decoding_b200.train import HeadTrainer

    ft = _head_model(graph_l4, graph_l1, dev, kind, M)
    n0 = ft.fc_weights[0].shape[0]
    widths = [n0] + list(M)
    fused = len(M) == 3 and _lib.lib().gcnb_head_step_workspace_bytes(B, *widths) > 0
    assert fused == (path == "fused")
    conv = [t.detach().clone() for t in list(ft.conv_weights) + list(ft.conv_bias)]
    sd = ft.state_dict_tf()
    names = ["fc%d" % (i + 1) for i in range(len(M) - 1)] + ["logits"]
    fcs = [(sd[s + "/weights"].astype(np.float64), sd[s + "/bias"].astype(np.float64)) for s in names]
    rng = np.random.RandomState(B + n0)
    a0 = (rng.rand(B, n0) * 0.5).astype(np.float32)
    labels = rng.randint(0, M[-1], B).astype(np.int64)
    tr = HeadTrainer(ft, use_cuda_graph=False)
    p_before = tr.flat_p.cpu().numpy().astype(np.float64)
    loss, logits = tr.step(T(a0, dev), T(labels, dev, torch.long))
    torch.cuda.synchronize()
    masks = [O.counter_dropout_mask(B, w, 0.5, tr.dropout_seed + i, 0) for i, w in enumerate(M[:-1])]
    want_loss, want = head_step(a0.astype(np.float64), labels, fcs, 0.0, dropout_masks=masks, keep=0.5,
                                  dtype=np.float64)
    assert abs(float(loss) - want_loss) <= 1e-4 * abs(want_loss)
    for i in range(len(M)):
        assert rel_inf(tr.gview[id(ft.fc_weights[i])].cpu().numpy(), want[i][0]) <= 1e-4, i
        assert rel_inf(tr.gview[id(ft.fc_bias[i])].cpu().numpy(), want[i][1]) <= 1e-4, i
    # the update: TF Nadam on the device's own gradient, L2 folded in over the whole head
    g = tr.flat_g.cpu().numpy().astype(np.float64)
    z = np.zeros_like(g)
    p_want, _, _ = nadam_tf(p_before, g, z, z, 1, *(_f32(h) for h in (tr.lr, tr.b1, tr.b2, tr.eps, ft.regularization)),
                              np.ones_like(g))
    assert rel_inf(tr.flat_p.cpu().numpy(), p_want) <= 1e-6
    assert tr.decay.all() and tr.n == sum(W.numel() + b.numel() for W, b in zip(ft.fc_weights, ft.fc_bias))
    assert tr.state.cpu().tolist()[3] == 1.0 and abs(tr.state[0].item() - tr.b1) < 1e-7   # the clock ticked once
    assert all(torch.equal(a, b) for a, b in zip(conv, list(ft.conv_weights) + list(ft.conv_bias)))
    reg_term = 0.5 * ft.regularization * float((tr.flat_p.double() ** 2).sum())   # the head's L2 term only
    assert abs(tr.regularization_term() - reg_term) <= 1e-5 * reg_term


@pytest.mark.parametrize("M", [[512, 256, 7], [64, 7]])
def test_graph_replay_and_pipeline_are_bit_identical_to_eager(dev, graph_l4, graph_l1, M):
    from gcn_fmri_decoding_b200.train import HeadTrainer, InputPipeline

    B = 512
    rng = np.random.RandomState(1)
    batches = [((rng.rand(B, 25) * 0.5).astype(np.float32), rng.randint(0, M[-1], B).astype(np.int64))
               for _ in range(20)]
    models = [_head_model(graph_l4, graph_l1, dev, "cfg2", M) for _ in range(3)]
    eager = HeadTrainer(models[0], use_cuda_graph=False)
    graph = HeadTrainer(models[1])
    piped = HeadTrainer(models[2])
    pipe = InputPipeline(piped, (B, 25))
    pipe.feed(*batches[0])
    for i, (x, y) in enumerate(batches):
        le, _ = eager.step(T(x, dev), T(y, dev, torch.long))
        lg, _ = graph.step(T(x, dev), T(y, dev, torch.long))
        if i + 1 < len(batches):
            pipe.feed(*batches[i + 1])
        lp, _ = pipe.step()
        assert float(le) == float(lg) == float(lp), i
    torch.cuda.synchronize()
    assert torch.equal(eager.flat_p, graph.flat_p) and torch.equal(eager.flat_p, piped.flat_p)
    assert torch.equal(eager.flat_m, graph.flat_m) and torch.equal(eager.state, graph.state)
    assert eager.state[3].item() == 20


# ------------------------------------------------------------------------------------------------ end to end
E2E_MIN_ACCURACY = 60.0   # chance is 14.3 %; the first run on a B200 reached 87.9 %


def test_fit_end_to_end(dev, graph_l4, tmp_path, capsys):
    from gcn_fmri_decoding_b200 import checkpoints
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    base = cgcnn(**_cfg2(graph_l4, dev, batch_size=256))
    args = _cfg2(graph_l4, dev, M=[512, 256, 7], batch_size=256, num_epochs=40, eval_frequency=160)
    ft = finetuning_cgcnn(**args, pretrained=base)
    n, n_val = 4096, 1000
    data, val = _windows(n, 11), _windows(n_val, 12)
    # a 7-class task the frozen features can express: labels = argmax(standardised features @ R)
    f_tr, f_val = ft.trunk_features(data), ft.trunk_features(val)
    mu, sd = f_tr.mean(0), f_tr.std(0) + 1e-12
    R = np.random.RandomState(5).randn(f_tr.shape[1], 7)
    labels = np.argmax(((f_tr - mu) / sd) @ R, 1).astype(np.int64)
    val_labels = np.argmax(((f_val - mu) / sd) @ R, 1).astype(np.int64)
    np.random.seed(0)
    best_dir = str(tmp_path / "best")
    accuracies, losses, t_step = ft.fit(data, labels, val, val_labels, best_checkpoint_dir=best_dir)
    with capsys.disabled():
        print("\n[fine-tuning end to end] validation accuracy %.2f %% (peak %.2f %%), loss %.4f -> %.4f"
              % (accuracies[-1], max(accuracies), losses[0], losses[-1]))
    assert len(accuracies) == 4 and losses[-1] < losses[0]
    assert max(accuracies) >= E2E_MIN_ACCURACY
    for i in range(2):
        assert torch.equal(ft.conv_weights[i], base.conv_weights[i]) and torch.equal(ft.conv_bias[i], base.conv_bias[i])
    index = json.load(open(os.path.join(best_dir, "best_checkpoints")))
    assert 1 <= len(index) <= 3 and len([f for f in os.listdir(best_dir) if f.endswith(".npz")]) == len(index)
    # evaluating the cached validation table is evaluate() on the windows
    assert ft.evaluate_features(ft.trunk_features(val, padded=True), val_labels) == ft.evaluate(val, val_labels)
    # the best checkpoint loads into a plain cgcnn with the new head and predicts the same logits
    best = checkpoints.BestCheckpoints(best_dir).best()
    plain = cgcnn(**args)
    checkpoints.load_checkpoint(plain, best)
    checkpoints.load_checkpoint(ft, best)
    assert np.array_equal(plain.predict(val, return_logits=True)[1], ft.predict(val, return_logits=True)[1])
    # saliency of the fine-tuned model against autograd through forward
    x = T(val[:256], dev).requires_grad_(True)
    lg = ft(x, gather=True)
    target = lg.argmax(1)
    want = torch.autograd.grad(lg.gather(1, target.view(-1, 1)).sum(), x)[0]
    got, tg = ft.saliency(val[:256])
    assert np.array_equal(tg, target.cpu().numpy())
    assert rel_inf(got, want.cpu().numpy()) <= 1e-5

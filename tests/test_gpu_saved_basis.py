"""The training path of a ChebyNet layer against the fp64 oracle: forward with a saved Chebyshev basis, then the
backward ``FusedTrainer`` runs -- dW/db streamed from the basis (``k_dw_from_stack``) and dx through the tcgen05 adjoint
(``k_cheb_fwd_umma`` on L~^T), ``k_cheb_bwd_fused`` or the general path.  Run on the B200 box: -m gpu.

The fp32 kernels decide every max-pool arg-max and every ReLU on their own.  Where the fp64 decision margin is below
fp32 rounding, either decision is correct, and the one taken moves a whole gradient element.  So each test checks that
the device's decisions are admissible (``check_decisions``, built on ``check_argmax``) and then compares the gradients
with the oracle routed through those same decisions (``conv_stack_bwd(decisions=...)``).
"""
import os
import re
import time

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import rel_inf
from oracle import layers_np as O
from test_gpu_parity import build_model, check_argmax

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-4
RELU_GAP = 1e-5   # a ReLU decision may differ from fp64 only where |window-max pre-activation| < RELU_GAP * max|pre|
# every CTA of k_dw_from_stack runs at least 4 rounds of its ring when B*M >= 4 * 128 * 296: chunks of at most 128 rows,
# at most 296 CTAs (stack_dw.cu), at most 3 stages
RING_ROWS = 128 * 296

STACK_DW, STACK_ADJ, STACK_FUSED, GENERAL = "stack-dW", "stack-dW + tcgen05 adjoint", "stack-dW + fused dx", "general"


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def T(a, dev, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)


def backward_route(B, M, nnz, Fin, Fout, K, p, need_dx, algo):
    """Which backward ``gcnb_cheb_bwd_f32`` runs after ``cheb_fwd_mean(..., want_stack=True)``, from the library's own
    dispatch queries (the conditions of its saved-basis branch, api.cu)."""
    from gcn_fmri_decoding_b200 import _lib

    lib = _lib.lib()
    if algo == _lib.ALGO_GENERAL:
        return GENERAL                          # cheb_fwd_mean keeps no basis for the general path
    width = lib.gcnb_cheb_stack_width(B, M, nnz, Fin, Fout, K, p)
    if width == 0:
        return "fused recompute"                # no basis kept at all: not a saved-basis route
    saved = lib.gcnb_cheb_fused_supported(B, M, nnz, Fin, Fout, K, p, 0, 0)   # else the general path's vertex-major basis
    if saved and not need_dx:
        return STACK_DW
    if saved and lib.gcnb_cheb_fused_supported(B, M, nnz, Fin, Fout, K, p, 1, 1):
        if (K > 1 and algo == _lib.ALGO_AUTO and Fin % 4 == 0 and Fout % 4 == 0 and os.environ.get("GCNB_UMMA_ADJ", "1")[:1] != "0"
                and "tcgen05" in _lib.describe_fwd(B, M, nnz, Fout, Fin, K, 1)):
            return STACK_ADJ
        return STACK_FUSED
    return GENERAL


def tiles(B, M, nnz, Fin, Fout, K, p):
    """Tiles of the k_cheb_fwd_umma launch for this shape (the last number of gcnb_cheb_fwd_describe)."""
    from gcn_fmri_decoding_b200 import _lib

    d = _lib.describe_fwd(B, M, nnz, Fin, Fout, K, p)
    assert "tcgen05" in d, d
    return int(re.search(r"(\d+) tiles$", d).group(1))


def saved_basis_layer(dev, pl, x, W, b, K, p, brelu, dy, need_dx, dy_is_mean, algo):
    """One layer the way FusedTrainer runs it: cheb_fwd_mean(want_stack=True), then cheb_bwd_into with that basis."""
    from gcn_fmri_decoding_b200 import ops

    mode = ops.BIAS_PER_FILTER if brelu == "b1relu" else ops.BIAS_PER_VERTEX
    xt, Wt, bt = T(x, dev), T(W, dev), T(b, dev)
    y, am, _, stack = ops.cheb_fwd_mean(xt, None, pl.rowptr, pl.col, pl.val, Wt, bt, K, p, mode, True, algo, True)
    gW, gb = torch.empty_like(Wt), torch.empty(b.size, device=dev)
    dx = ops.cheb_bwd_into(xt, None, y, am, T(dy, dev), dy_is_mean, *pl.tensors(), Wt, gW, gb, K, p, mode, True, need_dx,
                           algo, stack if stack.numel() else None)
    out = dict(y=y.cpu().numpy(), argmax=am.cpu().numpy(), dW=gW.cpu().numpy(), db=gb.cpu().numpy().reshape(np.shape(b)))
    if need_dx:
        out["dx"] = dx.cpu().numpy()
    return out


def full_dy(dy, Fout, dy_is_mean):
    """The gradient of y that a mean-form dy [B, Mo] stands for (dy / Fout on every filter)."""
    dy = np.asarray(dy, np.float64)
    return np.repeat(dy[:, :, None], Fout, axis=2) / Fout if dy_is_mean else dy


def check_decisions(dec, pre64, p, name=""):
    """The device's decisions (pooled arg-max bytes, ReLU mask y > 0) are admissible for the fp64 pre-activation
    [B, M, F]: the ReLU decision may differ from fp64 only where the window maximum of the pre-activation is within
    RELU_GAP * max|pre| of zero, and the arg-max follows check_argmax.  A window that fp64 finds all-dead but the device
    finds live is an exact tie of zeros for check_argmax; there the device's pick must be a near-maximum instead."""
    B, M, F = pre64.shape
    win = pre64.reshape(B, M // p, p, F)
    wmax = win.max(2)
    scale = np.abs(pre64).max()
    bad = dec["relu"] != (wmax > 0)
    assert not np.any(bad & (np.abs(wmax) >= RELU_GAP * scale)), name
    if p > 1:
        am = np.asarray(dec["argmax"])
        flip = dec["relu"] & ~(wmax > 0)
        picked = np.take_along_axis(win, am[:, :, None, :].astype(np.int64), 2)[:, :, 0]
        assert np.all(wmax[flip] - picked[flip] < RELU_GAP * scale), name
        a64 = np.maximum(pre64, 0)
        check_argmax(np.where(flip, a64.reshape(win.shape).argmax(2), am), a64, p, name)


class Worst:
    """||got - ref||_inf / ||ref||_inf accumulated over chunks of windows."""

    def __init__(self):
        self.err, self.ref = 0.0, 0.0

    def add(self, got, ref):
        self.err = max(self.err, float(np.abs(np.asarray(got, np.float64) - ref).max()))
        self.ref = max(self.ref, float(np.abs(ref).max()))

    def rel(self):
        return self.err / (self.ref if self.ref > 0 else 1.0)


def oracle_compare(r, L, x, W, b, K, p, brelu, dy, need_dx, dy_is_mean, name="", chunk=512):
    """Check the device's decisions and compare y, dW, db (and dx) of one layer with the decision-conditioned fp64
    oracle, computed in chunks of windows (y and dx per window, dW and db summed over the chunks)."""
    B = x.shape[0]
    Fout = W.shape[1]
    pr = [dict(W=W, b=b, K=K, p=p)]
    wy, wdx = Worst(), Worst()
    dW, db = 0.0, 0.0
    for s in range(0, B, chunk):
        sl = slice(s, min(B, s + chunk))
        y64, tr = O.conv_stack(x[sl], [L], pr, brelu=brelu, dtype=np.float64, keep=True)
        wy.add(r["y"][sl], y64)
        pre = tr[0]["z"] + (b.reshape(1, 1, -1) if brelu == "b1relu" else b[None])
        dec = dict(argmax=r["argmax"][sl] if p > 1 else np.zeros(y64.shape, np.uint8), relu=r["y"][sl] > 0)
        check_decisions(dec, pre, p, name)
        dx64, g = O.conv_stack_bwd(tr, [L], pr, full_dy(dy[sl], Fout, dy_is_mean), brelu=brelu, dtype=np.float64,
                                   first_needs_dx=need_dx, decisions=[dec])
        dW, db = dW + g[0]["dW"], db + g[0]["db"]
        if need_dx:
            wdx.add(r["dx"][sl], dx64)
    assert wy.rel() <= TOL, (name, "y", wy.rel())
    assert rel_inf(r["dW"], dW) <= TOL, (name, "dW", rel_inf(r["dW"], dW))
    assert rel_inf(r["db"], db) <= TOL, (name, "db", rel_inf(r["db"], db))
    if need_dx:
        assert wdx.rel() <= TOL, (name, "dx", wdx.rel())


def layer_inputs(rng, B, M, Fin, Fout, K, p, brelu, dy_is_mean):
    x = rng.randn(B, M, Fin).astype(np.float32)
    W = (rng.randn(Fin * K, Fout) * (0.4 / np.sqrt(Fin * K))).astype(np.float32)
    b = (rng.randn(Fout) * 0.1).astype(np.float32) if brelu == "b1relu" else (rng.randn(M, Fout) * 0.1).astype(np.float32)
    dy = rng.randn(*((B, M // p) if dy_is_mean else (B, M // p, Fout))).astype(np.float32)
    return x, W, b, dy


def run_images(use, fn):
    from gcn_fmri_decoding_b200 import plan

    old = plan.USE_IMAGES
    plan.USE_IMAGES = use
    try:
        return fn()
    finally:
        plan.USE_IMAGES = old


# ------------------------------------------------------------------------------------------ seeded sweep
def _random_saved_basis_cases(n=28, seed=4257):
    rng = np.random.RandomState(seed)
    cases = []
    while len(cases) < n:
        lvl = int(rng.randint(0, 4))                    # M = 400, 200, 100, 50
        p = int(rng.choice([1, 2, 4, 8]))
        K = int(rng.randint(1, 6))                      # plan_stack keeps a basis of at most 5 orders
        if rng.rand() < 0.5:                            # both widths multiples of 4 (the tcgen05 adjoint's domain) ...
            Fin, Fout = 4 * int(rng.randint(3, 9)), 4 * int(rng.randint(1, 9))
        else:                                           # ... or neither
            Fin, Fout = int(rng.choice([9, 10, 11, 13, 15, 18, 21, 27, 31])), int(rng.choice([3, 5, 6, 10, 13, 18, 25, 30]))
        B = int(rng.choice([1, 2, 5, 37, 130]))
        brelu = str(rng.choice(["b1relu", "b2relu"]))
        need_dx = bool(rng.rand() < 0.7)
        dy_is_mean = bool(rng.rand() < 0.5)
        if (400 >> lvl) % p:
            continue
        cases.append((lvl, B, Fin, Fout, K, p, brelu, need_dx, dy_is_mean))
    return cases


SWEEP = _random_saved_basis_cases()


@pytest.mark.parametrize("lvl,B,Fin,Fout,K,p,brelu,need_dx,dy_is_mean", SWEEP)
def test_saved_basis_layer_sweep(dev, graph_l4, lvl, B, Fin, Fout, K, p, brelu, need_dx, dy_is_mean):
    """Seeded random layer shapes around the tcgen05 domain through the saved-basis backward (ALGO_AUTO), with and without
    the host-built operator images: y, dW, db and dx against the decision-conditioned fp64 oracle."""
    from gcn_fmri_decoding_b200 import _lib
    from gcn_fmri_decoding_b200.plan import GraphPlan

    L = graph_l4["L"][lvl]
    M = L.shape[0]
    pl = GraphPlan(L, dev)
    route = backward_route(B, M, pl.nnz, Fin, Fout, K, p, need_dx, _lib.ALGO_AUTO)
    assert route in (STACK_DW, STACK_ADJ, STACK_FUSED, GENERAL), route
    rng = np.random.RandomState(1000 * lvl + 10 * B + K + Fin)
    x, W, b, dy = layer_inputs(rng, B, M, Fin, Fout, K, p, brelu, dy_is_mean)
    # without dx the saved basis takes stack_dw under ALGO_FUSED too, also where the fused backward does not fit
    for algo in (_lib.ALGO_AUTO, _lib.ALGO_FUSED) if route == STACK_DW else (_lib.ALGO_AUTO,):
        for use in (True, False):
            r = run_images(use, lambda: saved_basis_layer(dev, pl, x, W, b, K, p, brelu, dy, need_dx, dy_is_mean, algo))
            oracle_compare(r, L, x, W, b, K, p, brelu, dy, need_dx, dy_is_mean, "%s algo=%d images=%s" % (route, algo, use))


def test_saved_basis_sweep_covers_every_route(dev, graph_l4):
    """The sweep above takes each of the four backward routes several times."""
    from gcn_fmri_decoding_b200 import _lib

    count = {}
    for lvl, B, Fin, Fout, K, p, brelu, need_dx, dy_is_mean in SWEEP:
        r = backward_route(B, 400 >> lvl, graph_l4["Lt"][lvl].nnz, Fin, Fout, K, p, need_dx, _lib.ALGO_AUTO)
        count[r] = count.get(r, 0) + 1
    print("saved-basis sweep routes:", count)
    for r in (STACK_DW, STACK_ADJ, STACK_FUSED, GENERAL):
        assert count.get(r, 0) >= 3, count


# ------------------------------------------------------------------------------------------ benchmark-sized cases
ODD_B = 889   # conv 1: 445 tiles of 2 windows, the last one half full; conv 2: 889 tiles -- 3+ tiles per CTA on 148 SMs

BENCH_CASES = [
    # name, lvl, Fin, Fout, K, need_dx, dy_is_mean, B
    *[("config2-conv1", 0, 15, 32, 5, False, False, B) for B in (512, 2048, 4096, ODD_B)],
    *[("config2-conv2", 2, 32, 32, 5, True, True, B) for B in (512, 2048, 4096, ODD_B)],
    ("config3a-conv2", 2, 32, 32, 2, True, True, 512),
    ("config3a1-conv2", 2, 32, 32, 1, True, True, 512),
]


@pytest.mark.parametrize("name,lvl,Fin,Fout,K,need_dx,dy_is_mean,B", BENCH_CASES)
def test_saved_basis_at_benchmark_batch_sizes(dev, graph_l4, name, lvl, Fin, Fout, K, need_dx, dy_is_mean, B):
    """The benched layers at the batch sizes of bench.py (512 per GPU, 2048 / 4096 for --strong) and one odd batch:
    persistent loops that wrap -- several tiles per CTA of k_cheb_fwd_umma (forward and adjoint) and several rounds of
    k_dw_from_stack's stage ring -- against the fp64 oracle in chunks of windows."""
    from gcn_fmri_decoding_b200 import _lib
    from gcn_fmri_decoding_b200.plan import GraphPlan

    L = graph_l4["L"][lvl]
    M, p, brelu = L.shape[0], 4, "b1relu"
    pl = GraphPlan(L, dev)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    route = backward_route(B, M, pl.nnz, Fin, Fout, K, p, need_dx, _lib.ALGO_AUTO)
    assert route == (STACK_DW if not need_dx else STACK_ADJ if K > 1 else STACK_FUSED), route
    per_cta = [tiles(B, M, pl.nnz, Fin, Fout, K, p) // sms]
    if route == STACK_ADJ:
        per_cta.append(tiles(B, M, pl.nnz, Fout, Fin, K, 1) // sms)
    rounds = B * M // RING_ROWS
    print("%s B=%d: tiles per CTA (forward%s) >= %s, k_dw_from_stack rounds per CTA >= %d"
          % (name, B, ", adjoint" if len(per_cta) > 1 else "", per_cta, rounds))
    if B >= 2048 or B % 2:
        assert min(per_cta) >= 3, per_cta
    if (lvl == 0 and B >= 512) or B >= 2048:
        assert rounds >= 4, rounds
    rng = np.random.RandomState(B + K)
    x, W, b, dy = layer_inputs(rng, B, M, Fin, Fout, K, p, brelu, dy_is_mean)
    t0 = time.time()
    r = saved_basis_layer(dev, pl, x, W, b, K, p, brelu, dy, need_dx, dy_is_mean, _lib.ALGO_AUTO)
    oracle_compare(r, L, x, W, b, K, p, brelu, dy, need_dx, dy_is_mean, "%s B=%d" % (name, B))
    print("%s B=%d: device + fp64 oracle %.1f s" % (name, B, time.time() - t0))


# ------------------------------------------------------------------------------------------ the benched step
def test_benched_step_at_512_matches_oracle(dev, graph_l4):
    """FusedTrainer(dropout=0.5, own_gemm=True) replayed as a CUDA graph (bench.py's configuration) for one step at
    B = 512, against oracle.network_step run with the device's dropout masks and the device's conv decisions: the loss,
    every gradient and the Adam update."""
    from gcn_fmri_decoding_b200 import graclus, ops, synth
    from gcn_fmri_decoding_b200.train import FusedTrainer

    g = graph_l4
    B = 512
    xraw = synth.bold_windows(B, seed=51)
    labels = synth.labels(B, seed=51)
    model = build_model(g, [32, 32], [5, 5], [4, 4], [512, 256, 22], "chebyshev5", "b1relu", dev, perm=g["perm"])
    tr = FusedTrainer(model, distributed=False, use_cuda_graph=True, dropout=0.5, own_gemm=True)
    sd = {k: v.astype(np.float64) for k, v in model.state_dict_tf().items()}
    p0 = tr.flat_p.clone()
    xt = T(xraw, dev)
    # the trainer's two forward launches with the arguments of its step (deterministic kernels): the decisions the
    # step's backward routes its gradients by
    dec = []
    with torch.no_grad():
        h = xt
        for i in range(2):
            pl = model._plan(model.L[i])
            y, am, _, _ = ops.cheb_fwd_mean(h, model.perm if i == 0 else None, pl.rowptr, pl.col, pl.val,
                                            model.conv_weights[i], model.conv_bias[i], model.K[i], model.p[i],
                                            model._bias_mode(), True, model.algo, tr.save_basis)
            dec.append(dict(argmax=am.cpu().numpy(), relu=(y > 0).cpu().numpy()))
            h = y
    loss, logits = tr.step(xt, T(labels, dev, torch.long))
    torch.cuda.synchronize()
    masks = [O.counter_dropout_mask(B, 512, 0.5, tr.dropout_seed, 0), O.counter_dropout_mask(B, 256, 0.5, tr.dropout_seed + 1, 0)]
    xperm = graclus.perm_data_3d(xraw, g["perm"])
    params = [dict(W=sd["conv%d/weights" % i], b=sd["conv%d/bias" % i].reshape(32), K=5, p=4) for i in (1, 2)]
    fcs = [(sd[s + "/weights"], sd[s + "/bias"]) for s in ("fc1", "fc2", "logits")]
    _, trace = O.conv_stack(xperm, model.L, params, dtype=np.float64, keep=True)
    for i in range(2):
        check_decisions(dec[i], trace[i]["z"] + params[i]["b"], 4, "conv%d" % (i + 1))
    ref_loss, conv_g, fc_g = O.network_step(xperm, labels, model.L, params, fcs, 0.0, dtype=np.float64,
                                            dropout_masks=masks, keep=0.5, conv_decisions=dec)
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


# ------------------------------------------------------------------------------------------ non-symmetric operator
def directed_hub_graph(M=100, seed=3):
    """L = I - D^-1 A of a weighted directed graph: every vertex points at its ring neighbours (some reverse edges
    dropped) and at a hub, vertex 0, which points at only two vertices.  L~ = L - I has rows of at most 5 entries,
    L~^T has a hub row of M - 1: an operator whose transpose differs from it far beyond rounding."""
    rng = np.random.RandomState(seed)
    rows, cols = [], []
    for i in range(1, M):
        for d in (-2, -1, 1, 2):
            j = (i + d) % M
            if j != 0 and not (d < 0 and rng.rand() < 0.4):
                rows.append(i)
                cols.append(j)
        rows.append(i)
        cols.append(0)
    rows += [0, 0]
    cols += [1, 2]
    A = sp.csr_matrix((rng.uniform(0.5, 2.0, len(rows)), (rows, cols)), shape=(M, M))
    A.sum_duplicates()
    d = np.asarray(A.sum(1)).ravel()
    L = sp.identity(M, format="csr") - sp.diags(1.0 / d) @ A
    return sp.csr_matrix(L, dtype=np.float32)


def test_non_symmetric_operator(dev):
    """A directed graph whose L~ and L~^T are far apart: the forward must apply L~, every backward L~^T -- the tcgen05
    adjoint (ALGO_AUTO), k_cheb_bwd_fused (ALGO_FUSED) and the general path's Clenshaw step (ALGO_GENERAL), with and
    without operator images, through the saved basis and through autograd (the recompute paths)."""
    from gcn_fmri_decoding_b200 import _lib, ops
    from gcn_fmri_decoding_b200.plan import GraphPlan

    L = directed_hub_graph()
    M = L.shape[0]
    Lr = O.rescale_L(L)
    assert abs(Lr - Lr.T).max() > 0.1 and np.diff(Lr.T.tocsr().indptr).max() >= M - 1 > 4 * np.diff(Lr.indptr).max()
    B, Fin, Fout, K, p, brelu = 37, 16, 32, 4, 2, "b1relu"
    pl = GraphPlan(L, dev)
    assert backward_route(B, M, pl.nnz, Fin, Fout, K, p, True, _lib.ALGO_AUTO) == STACK_ADJ
    assert backward_route(B, M, pl.nnz, Fin, Fout, K, p, True, _lib.ALGO_FUSED) == STACK_FUSED
    assert pl.image((B, Fin, Fout, K, p)) is not None and pl.image((B, Fin, Fout, K, p), transposed=True) is not None
    rng = np.random.RandomState(8)
    x, W, b, dy = layer_inputs(rng, B, M, Fin, Fout, K, p, brelu, False)
    mode = ops.BIAS_PER_FILTER
    for algo in (_lib.ALGO_AUTO, _lib.ALGO_FUSED, _lib.ALGO_GENERAL):
        for use in (True, False):
            tag = "algo=%d images=%s" % (algo, use)
            r = run_images(use, lambda: saved_basis_layer(dev, pl, x, W, b, K, p, brelu, dy, True, False, algo))
            oracle_compare(r, L, x, W, b, K, p, brelu, dy, True, False, "saved basis " + tag)

            def autograd():
                xt, Wt, bt = (T(a, dev).requires_grad_(True) for a in (x, W, b))
                y, am = ops.cheb_fwd(xt, None, *pl.tensors(), Wt, bt, K, p, mode, True, True, algo)
                y.backward(T(dy, dev))
                return dict(y=y.detach().cpu().numpy(), argmax=am.cpu().numpy(), dW=Wt.grad.cpu().numpy(),
                            db=bt.grad.cpu().numpy(), dx=xt.grad.cpu().numpy())

            oracle_compare(run_images(use, autograd), L, x, W, b, K, p, brelu, dy, True, False, "autograd " + tag)

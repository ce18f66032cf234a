"""Data parallelism through the model API on two GPUs (NCCL; skipped with fewer than two devices).

One spawned pair of ranks per way of averaging the gradients (the peer-memory exchange fused into the optimiser kernel,
and plain NCCL) runs, in one process group:
  * ``cgcnn.fit`` at config-2 shapes with dropout off (keep 1.0), batch 64 -- against one-GPU ``fit`` from the same NumPy
    state: the same evaluation steps, bit-identical replicas, final parameters within 2e-4 of one GPU's on the
    parameters whose gradient stayed large (as ``test_dp_nccl.py``), kept checkpoints written by rank 0 alone;
  * ``evaluate`` and ``predict(return_logits=True)`` -- bit for bit one GPU's, at 889 windows and below 2 x batch_size;
  * fine-tuning: ``trunk_features`` bit for bit one GPU's, three ``HeadTrainer`` steps on half batches against one rank
    on the full batch, ``finetuning_cgcnn.fit`` end to end;
  * ``gcnb_nadam_tf_allreduce_f32`` at world 2 against the fp64 ``nadam_tf`` on the averaged gradient.
The world-1 kernel test runs in this process.  Workers leave with ``os._exit`` (communicators live in captured graphs).
"""
import ctypes as C
import json
import os
import socket
import sys

import numpy as np
import pytest

from conftest import rel_inf
from test_finetune import nadam_tf

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORLD = 2
FIT_BS, N_TRAIN, N_VAL = 64, 256, 200
EVAL_SIZES, EVAL_BS = (889, 150), 128
FT_BS, N_TRUNK, HEAD_B = 128, 700, 256
N_KERNEL = 157878


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _cfg2(graph, dev, **kw):
    a = dict(L=graph["L"], F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device=dev, seed=1,
             perm=graph["perm"], n_input_vertices=360, regularization=5e-4, dropout=0)
    a.update(kw)
    return a


def _graph():
    from conftest import GOLDEN, load_csr

    z = np.load(os.path.join(GOLDEN, "ref_graph_l4.npz"))
    return dict(L=[load_csr(z, "L%d" % i) for i in range(len(z["sizes"]))], perm=z["perm"])


def _windows(n, seed):
    from gcn_fmri_decoding_b200 import synth

    return synth.bold_windows(n, seed=seed)


def _fit_data():
    rng = np.random.RandomState(4)
    return (_windows(N_TRAIN, 21), rng.randint(0, 22, N_TRAIN).astype(np.int64), _windows(N_VAL, 22),
            rng.randint(0, 22, N_VAL).astype(np.int64))


def _fit_model(graph, dev):
    from gcn_fmri_decoding_b200.models import cgcnn

    return cgcnn(**_cfg2(graph, dev, batch_size=FIT_BS, num_epochs=2, eval_frequency=3))


def _run_fit(model, best_dir, trainer):
    """``model.fit`` from NumPy state 3 (rank 0's; other ranks start elsewhere); returns its result, the steps the
    checkpoint keeper was called at, and the mask of parameters whose gradient stayed above 1e-3 x max every step."""
    from gcn_fmri_decoding_b200 import checkpoints

    calls, big = [], [None]
    handle = checkpoints.BestCheckpoints.handle

    def counted(self, value, m, step):
        calls.append(step)
        return handle(self, value, m, step)

    step = trainer.step

    def tracked(x, y, dropout=None):
        out = step(x, y, dropout)
        g = trainer.flat_g.abs()
        sel = g > 1e-3 * g.max()
        big[0] = sel if big[0] is None else (big[0] & sel)
        return out

    trainer.step = tracked
    checkpoints.BestCheckpoints.handle = counted
    try:
        res = model.fit(*_fit_data(), best_checkpoint_dir=best_dir, trainer=trainer)
    finally:
        checkpoints.BestCheckpoints.handle = handle
    return res, calls, big[0]


def _finetune_model(graph, dev, bs):
    from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn

    base = cgcnn(**_cfg2(graph, dev, batch_size=bs))
    return finetuning_cgcnn(**_cfg2(graph, dev, batch_size=bs, M=[512, 256, 7], num_epochs=2, eval_frequency=2),
                            pretrained=base)


def _head_batch():
    rng = np.random.RandomState(9)
    return (rng.rand(HEAD_B, 25) * 0.5).astype(np.float32), rng.randint(0, 7, HEAD_B).astype(np.int64)


def _kernel_inputs(rank):
    rng = np.random.RandomState(50)
    p0 = rng.randn(N_KERNEL).astype(np.float32)
    decay = (rng.rand(N_KERNEL) < 0.6).astype(np.uint8)
    grads = [[(np.random.RandomState(100 * r + t).randn(N_KERNEL) * 10.0 ** rng.uniform(-3, 1, N_KERNEL)).astype(np.float32)
              for r in range(WORLD)] for t in range(3)]
    return p0, decay, grads


def _hyper():
    return tuple(float(np.float32(h)) for h in (1e-3, 0.9, 0.999, 1e-8, 5e-4))


def _tick(lib, state, stream, dev):
    """Advance the optimiser clock ``state`` once (a one-element gcnb_nadam_tf_f32 with tick = 1)."""
    from gcn_fmri_decoding_b200 import _lib

    lr, b1, b2, eps, reg = _hyper()
    one = [torch.zeros(1, device=dev) for _ in range(4)]
    vp = lambda t: C.c_void_p(t.data_ptr())
    _lib.check(lib.gcnb_nadam_tf_f32(vp(one[0]), vp(one[1]), vp(one[2]), vp(one[3]), None, vp(state), 1, lr, b1, b2,
                                     eps, reg, 1, stream), "gcnb_nadam_tf_f32")


def _kernel_world2(rank, dev):
    """gcnb_nadam_tf_allreduce_f32 over symmetric memory at world 2: (p, m, v) after each step and the clock."""
    import torch.distributed as dist
    import torch.distributed._symmetric_memory as symm

    from gcn_fmri_decoding_b200 import _lib

    lib = _lib.lib()
    lr, b1, b2, eps, reg = _hyper()
    p0, decay, grads = _kernel_inputs(rank)
    n = N_KERNEL
    stride = (n + 3) & ~3
    nflag = int(lib.gcnb_adam_allreduce_flag_bytes()) // 4
    buf = symm.empty(2 * stride + nflag, dtype=torch.float32, device=dev)
    buf.zero_()
    hdl = symm.rendezvous(buf, dist.group.WORLD)
    ptrs = [int(q) for q in hdl.buffer_ptrs]
    torch.cuda.synchronize()
    dist.barrier()
    gtab = [(C.c_void_p * WORLD)(*[q + par * stride * 4 for q in ptrs]) for par in (0, 1)]
    ftab = (C.c_void_p * WORLD)(*[q + 2 * stride * 4 for q in ptrs])
    vp = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = torch.as_tensor(p0, device=dev)
    m, v = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    dk = torch.as_tensor(decay, device=dev)
    state = torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev)
    out = []
    for t, g in enumerate(grads):
        par = t % 2
        buf[par * stride:par * stride + n].copy_(torch.as_tensor(g[rank], device=dev))
        _tick(lib, state, stream, dev)
        _lib.check(lib.gcnb_nadam_tf_allreduce_f32(vp(p), vp(m), vp(v), vp(dk), vp(state), n, b1, b2, eps, reg,
                                                   gtab[par], ftab, rank, WORLD, stream), "gcnb_nadam_tf_allreduce_f32")
        torch.cuda.synchronize()
        out.append([a.cpu().numpy() for a in (p, m, v)])
    dist.barrier()
    return out


def _worker(rank, world, port, peer, out_dir):
    import torch.distributed as dist

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from gcn_fmri_decoding_b200 import train

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    graph = _graph()
    res = {}
    # ---- cgcnn.fit
    model = _fit_model(graph, dev)
    tr = train.FusedTrainer(model, peer_allreduce=peer)
    np.random.seed(3 if rank == 0 else 1234)
    best_dir = os.path.join(out_dir, "best")
    (acc, losses, t_step), calls, _ = _run_fit(model, best_dir, tr)
    torch.cuda.synchronize()
    every = [torch.empty_like(tr.flat_p) for _ in range(world)]
    dist.all_gather(every, tr.flat_p)
    res["fit"] = dict(acc=acc, losses=losses, t_step=t_step, calls=calls, kind=tr.allreduce_kind,
                      p=[q.cpu() for q in every])
    with open(os.path.join(best_dir, "best_checkpoints")) as f:
        index = json.load(f)
    best = os.path.join(best_dir, max(index, key=index.get))
    res["fit"]["restored"] = model.evaluate(_fit_data()[2], _fit_data()[3], checkpoint=best)
    # ---- evaluate / predict
    from gcn_fmri_decoding_b200.models import cgcnn

    ev = cgcnn(**_cfg2(graph, dev, batch_size=EVAL_BS, seed=5))
    res["eval"] = {}
    for size in EVAL_SIZES:
        data = _windows(size, 30 + size)
        labels = np.random.RandomState(size).randint(0, 22, size)
        res["eval"][size] = (ev.evaluate(data, labels), ev.predict(data, labels, return_logits=True))
    # ---- fine-tuning
    ft = _finetune_model(graph, dev, FT_BS)
    res["trunk"] = ft.trunk_features(_windows(N_TRUNK, 40), padded=True)
    a0, y = _head_batch()
    lo, hi = train.shard(HEAD_B, rank, world)
    ht = train.HeadTrainer(_finetune_model(graph, dev, HEAD_B), peer_allreduce=peer)
    xa, ya = torch.as_tensor(a0[lo:hi], device=dev), torch.as_tensor(y[lo:hi], device=dev)
    for _ in range(3):
        ht.step(xa, ya)
    torch.cuda.synchronize()
    every = [torch.empty_like(ht.flat_p) for _ in range(world)]
    dist.all_gather(every, ht.flat_p)
    res["head"] = dict(p=[q.cpu() for q in every], kind=ht.allreduce_kind)
    np.random.seed(8)
    data, val = _windows(512, 41), _windows(200, 42)
    labels, val_labels = np.random.RandomState(1).randint(0, 7, 512), np.random.RandomState(2).randint(0, 7, 200)
    res["ft_fit"] = ft.fit(data, labels, val, val_labels, best_checkpoint_dir=os.path.join(out_dir, "ft_best"))
    # ---- the kernel at world 2
    if peer:
        res["kernel"] = _kernel_world2(rank, dev)
    torch.save(res, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.barrier()
    os._exit(0)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def one_gpu(dev, tmp_path_factory):
    """One-GPU results of everything the workers run (computed once)."""
    from gcn_fmri_decoding_b200 import train
    from gcn_fmri_decoding_b200.models import cgcnn

    graph = _graph()
    out = {}
    model = _fit_model(graph, dev)
    tr = train.FusedTrainer(model, distributed=False)
    start = tr.flat_p.clone()
    np.random.seed(3)
    (acc, losses, _), calls, big = _run_fit(model, str(tmp_path_factory.mktemp("one") / "best"), tr)
    torch.cuda.synchronize()
    out["fit"] = dict(acc=acc, losses=losses, calls=calls, p=tr.flat_p.cpu(), big=big.cpu(),
                      moved=(tr.flat_p - start).abs().cpu())
    ev = cgcnn(**_cfg2(graph, dev, batch_size=EVAL_BS, seed=5))
    out["eval"] = {}
    for size in EVAL_SIZES:
        data = _windows(size, 30 + size)
        labels = np.random.RandomState(size).randint(0, 22, size)
        out["eval"][size] = (ev.evaluate(data, labels), ev.predict(data, labels, return_logits=True))
    ft = _finetune_model(graph, dev, FT_BS)
    out["trunk"] = ft.trunk_features(_windows(N_TRUNK, 40), padded=True)
    a0, y = _head_batch()
    ht = train.HeadTrainer(_finetune_model(graph, dev, HEAD_B), distributed=False)
    hbig = None
    for _ in range(3):
        ht.step(torch.as_tensor(a0, device=dev), torch.as_tensor(y, device=dev))
        torch.cuda.synchronize()
        g = ht.flat_g.abs()
        sel = g > 1e-3 * g.max()
        hbig = sel if hbig is None else (hbig & sel)
    out["head"] = dict(p=ht.flat_p.cpu(), big=hbig.cpu())
    return out


@pytest.mark.parametrize("peer", [True, False])
def test_model_api_on_two_ranks(dev, one_gpu, tmp_path, peer):
    import torch.multiprocessing as mp

    mp.spawn(_worker, args=(WORLD, _free_port(), peer, str(tmp_path)), nprocs=WORLD, join=True)
    got = [torch.load(str(tmp_path / ("rank%d.pt" % r)), weights_only=False) for r in range(WORLD)]
    # ---- cgcnn.fit
    want = one_gpu["fit"]
    f0, f1 = got[0]["fit"], got[1]["fit"]
    assert f0["kind"].startswith("peer-memory") if peer else f0["kind"] == "nccl", f0["kind"]
    p0, p1 = f0["p"]
    assert torch.equal(p0, p1) and torch.equal(p0, f1["p"][0])                   # bit-identical replicas
    assert f0["calls"] == want["calls"] == [3, 6, 8] and f1["calls"] == []       # same evaluation points; rank 0 keeps
    assert len(f0["acc"]) == len(f1["acc"]) == len(want["acc"]) == 3
    assert (f0["acc"], f0["losses"], f0["t_step"]) == (f1["acc"], f1["losses"], f1["t_step"])   # same on every rank
    big = want["big"]
    assert int(big.sum()) > 1000 and float(want["moved"][big].max()) > 1e-3
    assert float((want["p"] - p0)[big].abs().max()) <= 2e-4
    index = json.load(open(str(tmp_path / "best" / "best_checkpoints")))
    npz = sorted(f for f in os.listdir(str(tmp_path / "best")) if f.endswith(".npz"))
    assert 1 <= len(index) <= 3 and npz == sorted(index)
    assert f0["restored"] == f1["restored"]
    # ---- evaluate / predict: bit for bit one GPU's
    for size in EVAL_SIZES:
        (w_ev, (w_pred, w_loss, w_logits)) = one_gpu["eval"][size]
        for r in range(WORLD):
            g_ev, (g_pred, g_loss, g_logits) = got[r]["eval"][size]
            assert g_ev == w_ev, (r, size)
            assert np.array_equal(g_pred, w_pred) and g_loss == w_loss and np.array_equal(g_logits, w_logits), (r, size)
    # ---- fine-tuning
    for r in range(WORLD):
        assert np.array_equal(got[r]["trunk"], one_gpu["trunk"]), r
    h0, h1 = got[0]["head"]["p"]
    assert got[0]["head"]["kind"].startswith("peer-memory") if peer else got[0]["head"]["kind"] == "nccl"
    assert torch.equal(h0, h1)
    hbig = one_gpu["head"]["big"]
    assert int(hbig.sum()) > 1000
    assert float((one_gpu["head"]["p"] - h0)[hbig].abs().max()) <= 2e-4
    a0_, l0_, _ = got[0]["ft_fit"]
    a1_, l1_, _ = got[1]["ft_fit"]
    assert len(a0_) == 4 and a0_ == a1_ and l0_ == l1_ and all(np.isfinite(l0_))
    # ---- the kernel at world 2 against fp64 Nadam on the averaged gradient
    if peer:
        lr, b1, b2, eps, reg = _hyper()
        p_, decay, grads = _kernel_inputs(0)
        before = (p_, np.zeros(N_KERNEL), np.zeros(N_KERNEL))
        for t, g in enumerate(grads):
            gavg = (g[0].astype(np.float64) + g[1].astype(np.float64)) / WORLD
            want = nadam_tf(before[0], gavg, *before[1:], t + 1, lr, b1, b2, eps, reg, decay)
            before = got[0]["kernel"][t]
            for r in range(WORLD):
                for a, w in zip(got[r]["kernel"][t], want):
                    assert rel_inf(a, w) <= 1e-6, (r, t, rel_inf(a, w))
            assert all(np.array_equal(a, b) for a, b in zip(got[0]["kernel"][t], got[1]["kernel"][t]))


def test_nadam_allreduce_at_world_one_is_nadam_bit_for_bit():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gcn_fmri_decoding_b200 import _lib

    dev = torch.device("cuda:0")
    lib = _lib.lib()
    lr, b1, b2, eps, reg = _hyper()
    n = N_KERNEL
    rng = np.random.RandomState(0)
    p0 = rng.randn(n).astype(np.float32)
    decay = torch.as_tensor((rng.rand(n) < 0.6).astype(np.uint8), device=dev)
    grads = [torch.as_tensor((rng.randn(n) * 10.0 ** rng.uniform(-3, 1, n)).astype(np.float32), device=dev)
             for _ in range(5)]
    vp = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    a = [torch.as_tensor(p0, device=dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)]
    b = [t.clone() for t in a]
    sa, sb = torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev), torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev)
    gbufs = [torch.zeros(n, device=dev), torch.zeros(n, device=dev)]   # the two alternating gradient buffers
    flags = torch.zeros(int(lib.gcnb_adam_allreduce_flag_bytes()) // 4, dtype=torch.int32, device=dev)
    ftab = (C.c_void_p * 1)(flags.data_ptr())
    for t, g in enumerate(grads):
        _lib.check(lib.gcnb_nadam_tf_f32(vp(a[0]), vp(g), vp(a[1]), vp(a[2]), vp(decay), vp(sa), n, lr, b1, b2, eps, reg,
                                         1, stream), "gcnb_nadam_tf_f32")
        sb.copy_(sa)   # the fused kernel reads this step's clock; the tick is the caller's
        gbufs[t % 2].copy_(g)
        _lib.check(lib.gcnb_nadam_tf_allreduce_f32(vp(b[0]), vp(b[1]), vp(b[2]), vp(decay), vp(sb), n, b1, b2, eps, reg,
                                                   (C.c_void_p * 1)(gbufs[t % 2].data_ptr()), ftab, 0, 1, stream),
                   "gcnb_nadam_tf_allreduce_f32")
        torch.cuda.synchronize()
        for x, y in zip(a, b):
            assert torch.equal(x, y), t
    assert int(flags[63]) == 5   # one exchange per step

"""Data parallelism through the model API on CPU: world_size 2 over gloo.

``train.fit`` under a process group must draw the global batches one process draws from rank 0's NumPy state, hand each
rank's trainer only its own rows, end where one process on the full batches ends and return the global-batch loss
history; its refusals (``batch_size % world != 0``, different training data on the ranks) must be raised on every rank
before the first step.  ``cgcnn._predict`` deals its batches over the ranks and must return, on every rank, bit for bit
what one process returns.  A small stand-in network (as in ``test_dp_gloo.py``) and a CPU-built ``cgcnn`` with a stub
``logits_at`` keep the GPU out of it.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gcn_fmri_decoding_b200 import train

WORLD = 2


class FitNet(torch.nn.Module):
    """Stand-in network with the attributes ``train.fit`` reads from a ``cgcnn``."""

    def __init__(self, seed, batch_size=8):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.w1 = torch.nn.Parameter(torch.randn(6, 5, generator=g) * 0.3)
        self.b1 = torch.nn.Parameter(torch.full((5,), 0.2))
        self.w2 = torch.nn.Parameter(torch.randn(5, 3, generator=g) * 0.3)
        self.regularization = 5e-4
        self.batch_size, self.num_epochs, self.eval_frequency, self.dropout = batch_size, 2, 1000, 0
        self.dev = torch.device("cpu")

    def forward(self, x, dropout=1.0):
        return torch.relu(x.mean(-1) @ self.w1 + self.b1) @ self.w2

    def loss(self, logits, labels):
        return torch.nn.functional.cross_entropy(logits, labels) + self.regularization * 0.5 * (self.w1 ** 2).sum()


def _data(shift=0.0):
    rng = np.random.RandomState(321)
    return (rng.randn(44, 6, 4).astype(np.float32) + np.float32(shift)), rng.randint(0, 3, 44).astype(np.int64)


def _recording_fit(model, data, labels, trainer):
    """``train.fit`` with ``seed=None`` (``cgcnn.fit``'s path); returns (loss history, the rows every step received)."""
    seen = []
    step = trainer.step

    def recorded(x, y, dropout=1.0):
        seen.append((x.clone(), y.clone()))
        return step(x, y, dropout)

    trainer.step = recorded
    history = train.fit(model, data, labels, trainer=trainer, seed=None, verbose=False)
    return history, seen


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _spawn(target, *args):
    """Run ``target(rank, world, out, *args)`` on WORLD gloo ranks; returns ``out`` as a dict (every worker must exit)."""
    ctx = mp.get_context("spawn")
    with ctx.Manager() as mgr:
        out = mgr.dict()
        port = _free_port()
        procs = [ctx.Process(target=_run, args=(r, port, out, target) + args) for r in range(WORLD)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(150)
        alive = [p for p in procs if p.is_alive()]
        for p in alive:
            p.kill()
            p.join()
        assert not alive, "a rank did not finish"
        assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
        return dict(out)


def _run(rank, port, out, target, *args):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        target(rank, WORLD, out, *args)
    finally:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------- train.fit
def _fit_worker(rank, world, out):
    data, labels = _data()
    np.random.seed(5 if rank == 0 else 999)   # rank 1 starts from another state: fit must use rank 0's
    model = FitNet(seed=10 + rank)
    tr = train.Trainer(model)
    assert tr.world == world
    history, seen = _recording_fit(model, data, labels, tr)
    out[rank] = dict(history=history, x=[x for x, _ in seen], y=[y for _, y in seen],
                     params=[p.detach().clone() for p in model.parameters()])


@pytest.mark.timeout(200)
def test_fit_on_two_ranks_draws_the_batches_of_one_process_and_ends_where_it_ends():
    data, labels = _data()
    np.random.seed(5)
    single = FitNet(seed=10)
    want_history, want_seen = _recording_fit(single, data, labels, train.Trainer(single, distributed=False))
    want_params = [p.detach().clone() for p in single.parameters()]
    assert len(want_seen) == int(2 * 44 / 8) == 11

    got = _spawn(_fit_worker)
    r0, r1 = got[0], got[1]
    assert len(r0["x"]) == len(r1["x"]) == len(want_seen)
    for step, (wx, wy) in enumerate(want_seen):
        assert r0["x"][step].shape[0] == r1["x"][step].shape[0] == 4        # each rank gets only its half
        assert torch.equal(torch.cat([r0["x"][step], r1["x"][step]]), wx), step
        assert torch.equal(torch.cat([r0["y"][step], r1["y"][step]]), wy), step
    for a, b, w in zip(r0["params"], r1["params"], want_params):
        assert torch.equal(a, b)                                            # the replicas stay identical
        assert torch.allclose(a, w, rtol=0, atol=1e-6)
    for h in (r0["history"], r1["history"]):
        assert np.allclose(h, want_history, rtol=0, atol=1e-6)              # global-batch loss of every step
    assert r0["history"] == r1["history"]


def _refusal_worker(rank, world, out, case):
    data, labels = _data(shift=1.0 if (case == "data" and rank == 1) else 0.0)
    model = FitNet(seed=3, batch_size=7 if case == "batch" else 8)
    tr = train.Trainer(model)
    stepped = []
    tr.step = lambda *a, **k: stepped.append(1)
    try:
        train.fit(model, data, labels, trainer=tr, seed=None, verbose=False)
        out[rank] = ("no error", len(stepped))
    except ValueError as e:
        out[rank] = (str(e), len(stepped))


@pytest.mark.timeout(200)
@pytest.mark.parametrize("case, match", [("batch", "not a multiple"), ("data", "different training data")])
def test_fit_refuses_on_every_rank_before_the_first_step(case, match):
    got = _spawn(_refusal_worker, case)
    for rank in range(WORLD):
        msg, steps = got[rank]
        assert match in msg, (rank, msg)
        assert steps == 0


# ------------------------------------------------------------------------------------------------- cgcnn._predict
BS = 128
SIZES = (1, BS - 1, BS * WORLD + 1, 889)


def _model(graph_L):
    from gcn_fmri_decoding_b200.models import cgcnn

    return cgcnn(L=graph_L, F=[4], K=[2], p=[1], M=[3], channel=2, device="cpu", batch_size=BS)


def _logits_at(begin):
    """Stand-in forward: a fixed function of the batch's first window (ties included: rows repeat every 7)."""
    r = torch.arange(BS, dtype=torch.float32).remainder(7).reshape(BS, 1)
    c = torch.arange(3, dtype=torch.float32).reshape(1, 3)
    return torch.sin(r * 0.37 + c * 1.3 + float(begin) * 0.01) * 4.0


def _labels(size):
    return np.random.RandomState(size).randint(0, 3, size)


def _predict_all(model):
    res = {}
    for size in SIZES:
        res[size] = (model._predict(size, _logits_at, _labels(size), True), model._predict(size, _logits_at, None, False))
    return res


def _predict_worker(rank, world, out, graph_L):
    out[rank] = _predict_all(_model(graph_L))


@pytest.mark.timeout(200)
def test_predict_dealt_over_two_ranks_is_bit_identical(graph_l4):
    L = graph_l4["L"][4:]
    want = _predict_all(_model(L))
    got = _spawn(_predict_worker, L)
    for rank in range(WORLD):
        for size in SIZES:
            (wp, wl, wlog), wp_nolab = want[size]
            (gp, gl, glog), gp_nolab = got[rank][size]
            assert np.array_equal(gp, wp) and np.array_equal(gp_nolab, wp_nolab), (rank, size)
            assert np.array_equal(glog, wlog), (rank, size)
            assert gl == wl, (rank, size, gl, wl)

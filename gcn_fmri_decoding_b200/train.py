"""Training step, TF-style Adam and batch-sharded data parallelism.

* ``TFAdam`` -- ``tf.train.AdamOptimizer(learning_rate=0.001)`` as hard-coded by the reference
  (``/root/reference/lib_new/models_gcn.py:294``): ``lr_t = lr*sqrt(1-b2^t)/(1-b1^t)``,
  ``v -= lr_t * m / (sqrt(v) + eps)`` ("epsilon hat" form, which differs from ``torch.optim.Adam``).
* ``Trainer`` -- one training step = forward, loss (``:253-262``), backward, optimiser
  (``:298-305``); with ``world_size > 1`` every rank takes its slice of the global batch, the
  Laplacians and weights are replicated and ONE all-reduce of a flat gradient buffer averages
  the gradients (SURVEY 8e).  The reference has no distributed code; this is the only
  collective the path needs.
* ``fit`` -- the reference's step loop (``:112-184``) without sessions/checkpoints/summaries.
* ``FusedTrainer`` -- the same step with an explicit schedule, one CUDA graph; ``HeadTrainer`` -- its head alone on cached
  conv features with TF's Nadam, the step of the fine-tuning model (``:685-933``).
"""
from __future__ import annotations

import collections
import time

import numpy as np
import torch
import torch.distributed as dist


class TFAdam:
    """TensorFlow-1.x Adam on a flat parameter list (multi-tensor ``_foreach`` ops)."""

    def __init__(self, params, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8):
        self.params = [p for p in params]
        self.lr, self.b1, self.b2, self.eps = lr, beta1, beta2, eps
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        dev = self.params[0].device
        # step-dependent scalars live on the device so that a captured CUDA graph can replay the step
        self.b1_pow = torch.ones((), device=dev)
        self.b2_pow = torch.ones((), device=dev)

    @torch.no_grad()
    def step(self, grads=None):
        grads = [p.grad for p in self.params] if grads is None else grads
        self.b1_pow.mul_(self.b1)
        self.b2_pow.mul_(self.b2)
        lr_t = self.lr * torch.sqrt(1 - self.b2_pow) / (1 - self.b1_pow)
        torch._foreach_mul_(self.m, self.b1)
        torch._foreach_add_(self.m, grads, alpha=1 - self.b1)
        torch._foreach_mul_(self.v, self.b2)
        torch._foreach_addcmul_(self.v, grads, grads, value=1 - self.b2)
        denom = torch._foreach_sqrt(self.v)
        torch._foreach_add_(denom, self.eps)
        upd = torch._foreach_div(self.m, denom)
        torch._foreach_mul_(upd, -lr_t)
        torch._foreach_add_(self.params, upd)

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    def state(self):
        """Every tensor a warm-up before a graph capture must put back."""
        return self.m + self.v + [self.b1_pow, self.b2_pow]


class TFDecayedSGD:
    """The reference's ``momentum == 0`` branch (models_gcn.py:283-292): ``tf.train.GradientDescentOptimizer`` on
    ``tf.train.exponential_decay(learning_rate, global_step, decay_steps, decay_rate, staircase=True)`` --
    ``p -= lr * decay_rate ** floor(global_step / decay_steps) * g`` with ``global_step`` the number of updates applied
    so far (no decay when ``decay_rate == 1``, :284).  No script of the reference selects it (``momentum = 0.9``
    everywhere: model.py:172); it exists so that a ``cgcnn(momentum=0)`` trains as the reference would.  The step counter
    lives on the device (CUDA-graph replays advance it)."""

    def __init__(self, params, lr, decay_steps=None, decay_rate=1.0):
        self.params = [p for p in params]
        self.lr, self.decay_rate = float(lr), float(decay_rate)
        self.decay_steps = float(decay_steps) if decay_steps else None
        if self.decay_rate != 1.0 and not self.decay_steps:
            raise ValueError("decay_rate != 1 needs decay_steps (models_gcn.py:284-286)")
        self.global_step = torch.zeros((), dtype=torch.float64, device=self.params[0].device)

    @torch.no_grad()
    def step(self, grads=None):
        grads = [p.grad for p in self.params] if grads is None else grads
        if self.decay_rate != 1.0:
            lr = self.lr * torch.pow(torch.tensor(self.decay_rate, dtype=torch.float64, device=self.global_step.device),
                                     torch.floor(self.global_step / self.decay_steps))
            upd = torch._foreach_mul(grads, -lr.to(torch.float32))
            torch._foreach_add_(self.params, upd)
        else:
            torch._foreach_add_(self.params, grads, alpha=-self.lr)
        self.global_step.add_(1)

    def state(self):
        return [self.global_step]


class Trainer:
    """Forward + loss + backward + (all-reduce) + optimiser for a ``cgcnn``; optionally CUDA-graph captured.

    Optimiser as the reference picks it (models_gcn.py:291-296): Adam(0.001) unless the model says ``momentum == 0``,
    which selects plain SGD on the exponentially decayed ``learning_rate``."""

    def __init__(self, model, lr=1e-3, distributed=None, use_cuda_graph=False):
        self.model = model
        self.params = [p for p in model.parameters()]
        if getattr(model, "momentum", 0.9) == 0:
            self.opt = TFDecayedSGD(self.params, getattr(model, "learning_rate", lr), getattr(model, "decay_steps", None),
                                    getattr(model, "decay_rate", 1.0))
        else:
            self.opt = TFAdam(self.params, lr=lr)
        self.distributed = dist.is_available() and dist.is_initialized() if distributed is None else distributed
        self.world = dist.get_world_size() if self.distributed else 1
        sizes = [p.numel() for p in self.params]
        self.flat_grad = torch.zeros(sum(sizes), dtype=torch.float32, device=self.params[0].device)
        self.grad_views = []
        off = 0
        for p, n in zip(self.params, sizes):
            self.grad_views.append(self.flat_grad[off:off + n].view_as(p))
            off += n
        self.use_cuda_graph = use_cuda_graph
        self._graph = None
        self._static = None
        if self.distributed:  # start from identical weights on every rank
            for p in self.params:
                dist.broadcast(p.data, src=0)

    def _step_impl(self, x, labels, dropout):
        logits = self.model(x, dropout=dropout)
        loss = self.model.loss(logits, labels)
        grads = torch.autograd.grad(loss, self.params)
        torch._foreach_copy_(self.grad_views, grads)
        if self.world > 1:
            # gradients of the local-batch mean; the global-batch mean is their average over ranks.
            dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM)
            self.flat_grad.mul_(1.0 / self.world)
        self.opt.step(self.grad_views)
        return loss.detach(), logits.detach()

    def step(self, x, labels, dropout=1.0):
        """One optimisation step on the local shard ``x [b, M, channel]``; returns (loss, logits)."""
        if not self.use_cuda_graph:
            return self._step_impl(x, labels, dropout)
        if self._graph is None:
            self._static = (torch.empty_like(x), torch.empty_like(labels))
            self._static[0].copy_(x)
            self._static[1].copy_(labels)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            state = self._snapshot()
            with torch.cuda.stream(side):
                for _ in range(3):  # warm up allocator / lazy init outside the capture
                    self._step_impl(self._static[0], self._static[1], dropout)
            torch.cuda.current_stream().wait_stream(side)
            self._restore(state)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._out = self._step_impl(self._static[0], self._static[1], dropout)
            self._restore(state)
        self._static[0].copy_(x, non_blocking=True)
        self._static[1].copy_(labels, non_blocking=True)
        self._graph.replay()
        return self._out

    def _snapshot(self):
        return [p.detach().clone() for p in self.params], [t.clone() for t in self.opt.state()]

    def _restore(self, s):
        with torch.no_grad():
            for p, q in zip(self.params, s[0]):
                p.copy_(q)
            for a, b in zip(self.opt.state(), s[1]):
                a.copy_(b)


def shard(n, rank, world):
    """Contiguous slice of ``range(n)`` rank ``rank`` of ``world`` owns (windows [r*n/G, (r+1)*n/G)).

    The trainers average the ranks' gradients with equal weights (SUM / world), which is the gradient of the global-batch
    mean only for EQUAL shards: feed them batches with ``n % world == 0`` (config 4: 4096 over 2/4/8 GPUs), or drop the
    remainder -- uneven shards would weight the windows of the smaller ranks more."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def fit(model, train_data, train_labels, val_data=None, val_labels=None, trainer=None, seed=0, verbose=True,
        on_eval=None):
    """The reference's training loop (models_gcn.py:112-184): epochs of random batches from a deque of
    shuffled indices, dropout keep-prob ``model.dropout``, periodic validation.  Returns the loss history.

    ``seed=None`` draws the permutations from NumPy's global generator, as the reference does (:140);
    ``on_eval(step, num_steps, loss)`` replaces the built-in report at every evaluation point (``cgcnn.fit`` uses it
    for the reference's validation / best-checkpoint bookkeeping)."""
    trainer = trainer or Trainer(model)
    rng = np.random if seed is None else np.random.RandomState(seed)
    n = train_data.shape[0]
    num_steps = int(model.num_epochs * n / model.batch_size)
    indices = collections.deque()
    losses, t0 = [], time.time()
    dev = model.dev
    def draw():
        if len(indices) < model.batch_size:
            indices.extend(rng.permutation(n))
        idx = [indices.popleft() for _ in range(model.batch_size)]
        return (np.ascontiguousarray(train_data[idx], dtype=np.float32), np.ascontiguousarray(train_labels[idx]).astype(np.int64))

    # a FusedTrainer is fed through the asynchronous input pipeline: the copy of batch i+1 overlaps step i
    pipe = None
    if isinstance(trainer, FusedTrainer) and trainer.use_cuda_graph and torch.device(dev).type == "cuda":
        pipe = InputPipeline(trainer, (model.batch_size,) + tuple(train_data.shape[1:]))
        if num_steps > 0:
            pipe.feed(*draw())
    for step in range(1, num_steps + 1):
        if pipe is not None:
            if step < num_steps:
                pipe.feed(*draw())
            loss, _ = pipe.step()
        else:
            xb, yb = draw()
            x = torch.as_tensor(xb, dtype=torch.float32, device=dev)
            y = torch.as_tensor(yb, dtype=torch.long, device=dev)
            loss, _ = trainer.step(x, y, dropout=model.dropout if model.dropout else 1.0)
        losses.append(float(loss))
        if on_eval is not None:
            if step % model.eval_frequency == 0 or step == num_steps:
                on_eval(step, num_steps, losses[-1])
        elif verbose and (step % model.eval_frequency == 0 or step == num_steps):
            msg = "step %d / %d (epoch %.2f): loss %.4f" % (step, num_steps, step * model.batch_size / n, losses[-1])
            if val_data is not None:
                pred, vloss = model.predict(val_data, val_labels)
                msg += "  val acc %.2f%% loss %.4f" % (100.0 * float(np.mean(pred == np.asarray(val_labels))), vloss)
            print(msg + "  (%.1fs)" % (time.time() - t0))
    return losses


class FusedTrainer:
    """The training step with an explicit (autograd-free) schedule and as few launches as possible.

    forward : fused conv launches (``ops.cheb_fwd`` / ``spectral_fwd``) -> mean over F -> FC stack (cuBLAS) ->
              ``gcnb_softmax_xent_f32`` (loss and dlogits in one pass)
    backward: FC stack written straight into one flat gradient buffer -> fused conv backward launches
    update  : one all-reduce of the flat buffer (world > 1) -> ``gcnb_adam_tf_f32`` over the flat parameter buffer with
              the L2 term of ``models_gcn.py:260-262`` folded in (``g += reg * p`` on the regularised tensors).
    The whole step is captured once and replayed as a CUDA graph.  Parameters of the model become views into one flat
    buffer.  Gradients equal those of ``Trainer`` (autograd) -- see ``tests/test_gpu_parity.py``.
    """

    def __init__(self, model, lr=1e-3, distributed=None, use_cuda_graph=True, dropout=None, beta1=0.9, beta2=0.999,
                 eps=1e-8, own_gemm=True, save_basis=True, fused_head=True, peer_allreduce=True, dropout_seed=None,
                 gather=None):
        import ctypes as C

        from . import _lib, ops

        self.params = self._trained_parameters(model)
        self.model, self.lr, self.b1, self.b2, self.eps = model, lr, beta1, beta2, eps
        self.C, self._lib, self.ops = C, _lib, ops
        # keep-probability of the FC dropout: the model's own (what Trainer and the reference use, models_gcn.py:145,677)
        # unless the caller overrides it; it is baked into the captured graph.
        if dropout is None:
            dropout = getattr(model, "dropout", 1.0)
        self.keep = float(dropout) if dropout else 1.0
        self.own_gemm = own_gemm
        # dropout stream: layer i draws with seed (dropout_seed + i); data-parallel ranks and differently seeded models
        # draw different masks (the reference seeds tf.nn.dropout from the graph seed)
        rank = dist.get_rank() if (dist.is_available() and dist.is_initialized() and distributed is not False) else 0
        base = dropout_seed if dropout_seed is not None else 0x5eed + 0x9e3779b1 * rank + 7919 * int(getattr(model, "seed", 0) or 0)
        self.dropout_seed = int(base) & 0x7FFFFFFF
        self.fused_head = fused_head
        self.save_basis = save_basis
        # gather: True = the steps get raw [B, n_input_vertices, C] windows (permuted in the first layer's load), False =
        # already permuted input, None = tell by the shape -- refused when the two shapes coincide (as cgcnn.forward does)
        if gather is None and model.perm is not None and model.n_input_vertices == model.L[0].shape[0]:
            raise ValueError("FusedTrainer: with perm set and n_input_vertices == M_0 say gather=True (raw windows) or "
                             "gather=False (already permuted) -- the shapes are identical")
        self.gather = gather
        self.distributed = dist.is_available() and dist.is_initialized() if distributed is None else distributed
        self.world = dist.get_world_size() if self.distributed else 1
        dev = self.params[0].device
        sizes = [p.numel() for p in self.params]
        self.n = sum(sizes)
        self.flat_p = torch.empty(self.n, dtype=torch.float32, device=dev)
        self.flat_m = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.flat_v = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.decay = torch.zeros(self.n, dtype=torch.uint8, device=dev)
        self.state = torch.tensor([1.0, 1.0, 0.0, 0.0], dtype=torch.float32, device=dev)  # b1^t, b2^t, lr_t, t
        # world > 1: the gradient average is fused into the optimiser kernel (gcnb_adam_tf_allreduce_f32): the flat
        # gradient buffers then live in peer-mapped symmetric memory, two of them used on alternate steps (a peer may
        # still be reading the previous one).  Falls back to one NCCL all-reduce when symmetric memory is unavailable.
        self.allreduce_kind = "none"
        self._peer = None
        gbufs = None
        if self.world > 1:
            self.allreduce_kind = "nccl"
            if peer_allreduce and dev.type == "cuda":
                try:
                    self._peer, gbufs = self._setup_peer_buffers(dev)
                    self.allreduce_kind = "peer-memory (fused into the Adam kernel)"
                except Exception as e:  # no NVLink peer access / symmetric memory unsupported: NCCL it is
                    self._peer_error = repr(e)
        if gbufs is None:
            gbufs = [torch.zeros(self.n, dtype=torch.float32, device=dev)]
        self._gbufs = gbufs
        regularized = {id(p) for p in model._regularized}
        self._gviews = [dict() for _ in gbufs]
        off = 0
        with torch.no_grad():
            for p, n in zip(self.params, sizes):
                self.flat_p[off:off + n].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[off:off + n].view_as(p)
                for gv, gb in zip(self._gviews, gbufs):
                    gv[id(p)] = gb[off:off + n].view_as(p)
                if id(p) in regularized:
                    self.decay[off:off + n] = 1
                off += n
        self._par = self._cur_par = 0
        self.flat_g, self.gview = self._gbufs[0], self._gviews[0]   # the buffers of the step in flight / last run
        if self.distributed:
            dist.broadcast(self.flat_p, src=0)
        self.use_cuda_graph = use_cuda_graph
        self._graphs = {}   # (gradient-buffer parity, bound-input key or None) -> (graph, outputs)
        self._bound = {}    # (x.data_ptr(), labels.data_ptr()) -> tensors registered by bind_inputs
        self._sx = self._sl = None
        self._loss = torch.zeros((), dtype=torch.float32, device=dev)

    def _trained_parameters(self, model):
        """The parameters the step updates: all of them, with TF Adam."""
        if getattr(model, "momentum", 0.9) == 0:
            raise NotImplementedError("FusedTrainer implements the Adam branch of the reference's optimiser choice "
                                      "(models_gcn.py:294, what every reference script selects); momentum == 0 (decayed "
                                      "SGD, :291-292) trains through train.Trainer")
        return [p for p in model.parameters()]

    def _setup_peer_buffers(self, dev):
        """Symmetric (peer-mapped) memory of every rank: two flat gradient buffers + the flag array, zeroed; returns the
        per-parity pointer tables for the kernel and the two local gradient tensors."""
        import torch.distributed._symmetric_memory as symm

        C = self.C
        lib = self._lib.lib()
        stride = (self.n + 3) & ~3                      # parity buffers start 16-byte aligned
        nflag = int(lib.gcnb_adam_allreduce_flag_bytes()) // 4
        buf = symm.empty(2 * stride + nflag, dtype=torch.float32, device=dev)
        buf.zero_()
        hdl = symm.rendezvous(buf, dist.group.WORLD)
        ptrs = [int(p) for p in hdl.buffer_ptrs]
        if len(ptrs) != self.world or any(p == 0 for p in ptrs):
            raise RuntimeError("symmetric memory rendezvous returned %d pointers for %d ranks" % (len(ptrs), self.world))
        torch.cuda.synchronize()
        dist.barrier()  # every rank's buffer is zero before anybody can raise a flag
        grads = [(C.c_void_p * self.world)(*[p + par * stride * 4 for p in ptrs]) for par in (0, 1)]
        flags = (C.c_void_p * self.world)(*[p + 2 * stride * 4 for p in ptrs])
        peer = {"buf": buf, "hdl": hdl, "grads": grads, "flags": flags, "rank": dist.get_rank()}
        return peer, [buf[0:self.n], buf[stride:stride + self.n]]

    # -- one step, eagerly ---------------------------------------------------------------------------------------
    @torch.no_grad()
    def _step_impl(self, x, labels):
        m, ops, C = self.model, self.ops, self.C
        lib = self._lib.lib()
        stream = C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        vp = lambda t: C.c_void_p(t.data_ptr())
        nconv = len(m.p)
        mode = m._bias_mode()
        cheb = m.filter_name != "fourier"
        gather = self.gather
        if gather is None:
            gather = m.perm is not None and x.shape[1] == m.n_input_vertices != m.L[0].shape[0]
        gather = bool(gather) and m.perm is not None
        # ---- forward: conv stack (the last layer also emits the mean over its filters = the head's input) ----
        saved, h, h0 = [], x, None
        for i in range(nconv):
            perm = m.perm if (gather and i == 0) else None
            last = i == nconv - 1
            if cheb:
                pl = m._plan(m.L[i])
                # keep the Chebyshev basis: the weight gradient becomes one streamed GEMM and the backward kernel only runs
                # the adjoint recursion for dx (none at all for the first layer); last layer: also emit the mean over filters
                y, am, hm, stack = ops.cheb_fwd_mean(h, perm, pl.rowptr, pl.col, pl.val, m.conv_weights[i], m.conv_bias[i],
                                                     m.K[i], m.p[i], mode, True, m.algo, self.save_basis)
                if last:
                    h0 = hm
                saved.append((h, perm, y, am, pl, stack if stack.numel() else None))
            else:
                if perm is not None:
                    h = ops.perm_gather(h, perm)
                sp = m._spectral_plan(m.L[i])
                y, am = ops.spectral_fwd(h, sp.Ut, m.conv_weights[i], m.conv_bias[i], m.p[i], mode, True, True)
                saved.append((h, None, y, am, sp, None))
            h = y
        if h0 is None:
            h0 = ops.mean_f_fwd(h)
        logits, d = self._head(h0, labels, lib, vp, stream)
        # ---- backward: conv stack (d is the gradient of the mean over filters of the last layer) ----
        dy, dy_is_mean = d, True
        if not cheb:
            dy, dy_is_mean = torch.ops.gcn_b200.mean_f_bwd(d, h.shape[-1]), False
        for i in range(nconv - 1, -1, -1):
            hin, perm, y, am, pl, stack = saved[i]
            need_dx = i > 0
            gW, gb = self.gview[id(m.conv_weights[i])], self.gview[id(m.conv_bias[i])]
            if cheb:
                dx = ops.cheb_bwd_into(hin, perm, y, am, dy, dy_is_mean, *pl.tensors(), m.conv_weights[i], gW, gb, m.K[i],
                                       m.p[i], mode, True, need_dx, m.algo, stack)
            else:
                dx, dW, db = torch.ops.gcn_b200.spectral_bwd(hin, y, am, dy, pl.Ut, m.conv_weights[i], m.p[i], mode, True,
                                                             need_dx)
                gW.copy_(dW)
                gb.copy_(db.view_as(gb))
            dy, dy_is_mean = dx, False
        # ---- update ----
        if self._peer is not None:
            rc = lib.gcnb_adam_tf_allreduce_f32(vp(self.flat_p), vp(self.flat_m), vp(self.flat_v), vp(self.decay),
                                                vp(self.state), self.n, self.b1, self.b2, self.eps,
                                                float(m.regularization or 0.0), self._peer["grads"][self._cur_par],
                                                self._peer["flags"], self._peer["rank"], self.world, stream)
            self._lib.check(rc, "gcnb_adam_tf_allreduce_f32")
            return self._loss, logits
        if self.world > 1:
            dist.all_reduce(self.flat_g, op=dist.ReduceOp.SUM)
        rc = lib.gcnb_adam_tf_f32(vp(self.flat_p), vp(self.flat_g), vp(self.flat_m), vp(self.flat_v), vp(self.decay),
                                  vp(self.state), self.n, self.lr, self.b1, self.b2, self.eps,
                                  float(m.regularization or 0.0), 1.0 / self.world, 0, stream)
        self._lib.check(rc, "gcnb_adam_tf_f32")
        return self._loss, logits

    def _head(self, h0, labels, lib, vp, stream):
        """The classifier head of the step on ``h0`` (the mean over the last conv layer's filters): forward, loss and
        backward, the FC gradients written into the flat gradient buffer, the optimiser clock advanced.  Returns
        ``(logits, d)`` with ``d`` the gradient w.r.t. ``h0``."""
        m = self.model
        nfc = len(m.M)

        def gemm(A, Bm, out, bias, M_, N_, K_, ta, tb):
            rc = lib.gcnb_gemm_f32(vp(A), vp(Bm), vp(out), None if bias is None else vp(bias), M_, N_, K_, A.shape[1],
                                   Bm.shape[1], out.shape[1], ta, tb, stream)
            self._lib.check(rc, "gcnb_gemm_f32")
            return out

        # The FC GEMMs are plain library GEMMs (cuBLAS fp32): at B=512 they are a few microseconds each and launch
        # bound; the in-house 3xTF32 kernel (`gemm`, used by the spectral layer) pays off only for large operands.
        use_own_gemm = self.own_gemm

        def gemm_epi(A, Bm, out, bias, M_, N_, K_, ta, tb, epi, aux, seed):
            rc = lib.gcnb_gemm_epilogue_f32(vp(A), vp(Bm), vp(out), None if bias is None else vp(bias), M_, N_, K_,
                                            A.shape[1], Bm.shape[1], out.shape[1], ta, tb, epi,
                                            None if aux is None else vp(aux), 0 if aux is None else aux.shape[1],
                                            self.keep, seed, vp(self.state), stream)
            self._lib.check(rc, "gcnb_gemm_epilogue_f32")
            return out

        def fc_fwd(i, a_in, hidden):
            """FC layer i; hidden layers apply ReLU + dropout (fused into the GEMM store on the in-house path)."""
            W = m.fc_weights[i]
            if not use_own_gemm:
                a = torch.addmm(m.fc_bias[i], a_in, W)
                if hidden:
                    rc = lib.gcnb_relu_dropout_fwd_f32(vp(a), a.shape[0], a.shape[1], a.shape[1], self.keep, self.dropout_seed + i,
                                                       vp(self.state), stream)
                    self._lib.check(rc, "gcnb_relu_dropout_fwd_f32")
                return a
            out = torch.empty((a_in.shape[0], W.shape[1]), dtype=torch.float32, device=h0.device)
            if hidden:
                return gemm_epi(a_in, W, out, m.fc_bias[i], a_in.shape[0], W.shape[1], W.shape[0], 0, 0,
                                self._lib.EPI_RELU_DROPOUT, None, self.dropout_seed + i)
            return gemm(a_in, W, out, m.fc_bias[i], a_in.shape[0], W.shape[1], W.shape[0], 0, 0)

        B = h0.shape[0]
        widths = [h0.shape[1]] + [w.shape[1] for w in m.fc_weights]
        head_ws = lib.gcnb_head_step_workspace_bytes(B, *widths) if (self.fused_head and nfc == 3) else 0
        if head_ws:
            # the whole head -- three FC layers, cross-entropy, their backward pass, the optimiser clock -- in ONE launch
            logits = torch.empty((B, widths[3]), dtype=torch.float32, device=h0.device)
            d = torch.empty((B, widths[0]), dtype=torch.float32, device=h0.device)
            ws = torch.empty(head_ws, dtype=torch.uint8, device=h0.device)
            g = lambda t: vp(self.gview[id(t)])
            W1, W2, W3 = m.fc_weights
            b1, b2, b3 = m.fc_bias
            rc = lib.gcnb_head_step_f32(vp(h0), vp(labels), vp(W1), vp(b1), vp(W2), vp(b2), vp(W3), vp(b3), vp(logits),
                                        vp(self._loss), g(W1), g(b1), g(W2), g(b2), g(W3), g(b3), vp(d), B, *widths,
                                        self.keep, self.dropout_seed, self.dropout_seed + 1, vp(self.state), self.lr, self.b1, self.b2, 1,
                                        vp(ws), ws.numel(), stream)
            self._lib.check(rc, "gcnb_head_step_f32")
        else:
            logits, d = self._head_by_layers(h0, labels, gemm, gemm_epi, fc_fwd, lib, vp, stream)
        return logits, d

    def _head_by_layers(self, h0, labels, gemm, gemm_epi, fc_fwd, lib, vp, stream):
        """The head launch by launch (any number of FC layers): GEMM + fused ReLU/dropout per layer, cross-entropy,
        two GEMMs per layer backward, one multi-matrix column sum for the bias gradients."""
        m, C = self.model, self.C
        nfc = len(m.M)
        x = h0
        use_own_gemm = self.own_gemm
        acts = [h0]
        for i in range(nfc - 1):
            acts.append(fc_fwd(i, acts[-1], True))
        logits = fc_fwd(nfc - 1, acts[-1], False)
        B, ncls = logits.shape
        d = torch.empty_like(logits)
        rows = torch.empty(B, dtype=torch.float32, device=x.device)
        # loss, dlogits and the optimiser clock in one launch
        rc = lib.gcnb_softmax_xent_f32(vp(logits), vp(labels), vp(self._loss), vp(d), vp(rows), B, ncls, vp(self.state),
                                       self.lr, self.b1, self.b2, stream)
        self._lib.check(rc, "gcnb_softmax_xent_f32")
        # ---- backward: head; weight gradients land in the flat buffer, the bias gradients in one launch at the end ----
        ds = [None] * nfc
        for i in range(nfc - 1, -1, -1):
            ds[i] = d
            W = m.fc_weights[i]
            if use_own_gemm:
                gemm(acts[i], d, self.gview[id(W)], None, W.shape[0], W.shape[1], d.shape[0], 1, 0)   # dW = a^T d
                dn = torch.empty((d.shape[0], W.shape[0]), dtype=torch.float32, device=x.device)
                if i > 0:  # dx = d W^T through the ReLU/dropout mask of the activation it feeds, in the same launch
                    d = gemm_epi(d, W, dn, None, d.shape[0], W.shape[0], W.shape[1], 0, 1, self._lib.EPI_MASK, acts[i], 0)
                else:
                    d = gemm(d, W, dn, None, d.shape[0], W.shape[0], W.shape[1], 0, 1)
            else:
                torch.mm(acts[i].t(), d, out=self.gview[id(W)])
                d = torch.mm(d, W.t())
                if i > 0:
                    rc = lib.gcnb_relu_dropout_bwd_f32(vp(d), vp(acts[i]), d.shape[0], d.shape[1], d.shape[1], d.shape[1],
                                                       self.keep, stream)
                    self._lib.check(rc, "gcnb_relu_dropout_bwd_f32")
        for lo in range(0, nfc, 4):
            grp = list(range(lo, min(nfc, lo + 4)))
            n = len(grp)
            mats = (C.c_void_p * n)(*[ds[i].data_ptr() for i in grp])
            outs = (C.c_void_p * n)(*[self.gview[id(m.fc_bias[i])].data_ptr() for i in grp])
            rws = (C.c_int * n)(*[ds[i].shape[0] for i in grp])
            cls = (C.c_int * n)(*[ds[i].shape[1] for i in grp])
            rc = lib.gcnb_colsum_multi_f32(mats, outs, rws, cls, n, stream)
            self._lib.check(rc, "gcnb_colsum_multi_f32")
        return logits, d

    def regularization_term(self):
        """``regularization * sum_v ||v||^2 / 2`` over the regularised tensors (reported with the loss, not needed by the step)."""
        with torch.no_grad():
            return float(self.model.regularization or 0.0) * 0.5 * float((self.flat_p * self.flat_p * self.decay).sum())

    def step(self, x, labels, dropout=None):
        """One optimisation step on the local shard; returns (cross-entropy loss tensor, logits).  ``labels`` int64.

        The returned loss is the mean cross-entropy; ``regularization_term()`` gives the L2 term the reference adds to
        the reported loss (models_gcn.py:260-262) -- the update itself always includes it.  ``dropout`` must be None or
        the keep-probability this trainer was built with (it is part of the captured graph)."""
        if dropout is not None and abs(float(dropout if dropout else 1.0) - self.keep) > 1e-12:
            raise ValueError("FusedTrainer was built with dropout keep-probability %g; step(dropout=%g) would be ignored "
                             "-- construct the trainer with the value you want" % (self.keep, float(dropout)))
        par = self._cur_par = self._par
        self.flat_g, self.gview = self._gbufs[par], self._gviews[par]
        if len(self._gbufs) > 1:
            self._par ^= 1                      # the next step writes the other gradient buffer
        if not self.use_cuda_graph:
            return self._step_impl(x, labels)
        key = (x.data_ptr(), labels.data_ptr())
        if key in self._bound and self._bound[key][0].shape == x.shape:
            graph, out = self._graph_for(par, key, *self._bound[key])   # reads x / labels where they are: no copy
        else:
            if self._sx is None or self._sx.shape != x.shape:
                self._sx, self._sl = torch.empty_like(x), torch.empty_like(labels)
                self._graphs = {k: v for k, v in self._graphs.items() if k[1] is not None}
            self._sx.copy_(x, non_blocking=True)
            self._sl.copy_(labels, non_blocking=True)
            graph, out = self._graph_for(par, None, self._sx, self._sl)
        graph.replay()
        return out

    def bind_inputs(self, x, labels):
        """Register device tensors the caller refills IN PLACE (slots of an input ring): ``step(x, labels)`` on them
        replays a graph that reads them where they are, without the copy into the trainer's own static buffer
        (11 MB device-to-device per step at B = 512).  The tensors are kept alive by the trainer.  With data
        parallelism every rank must bind the same number of inputs in the same order (capturing runs collectives)."""
        if not self.use_cuda_graph:
            return
        key = (x.data_ptr(), labels.data_ptr())
        self._bound[key] = (x, labels)
        for par in range(len(self._gbufs)):
            self._graph_for(par, key, x, labels)

    def _graph_for(self, par, key, x, labels):
        """The captured step of gradient-buffer parity ``par`` reading ``x`` / ``labels`` (captured on first use:
        three eager warm-up steps on a side stream, then the capture; optimiser state restored afterwards)."""
        if (par, key) in self._graphs:
            return self._graphs[(par, key)]
        keep = (self.flat_g, self.gview)
        self.flat_g, self.gview = self._gbufs[par], self._gviews[par]
        snap = [t.clone() for t in (self.flat_p, self.flat_m, self.flat_v, self.state)]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                self._step_impl(x, labels)
                if self._peer is not None:
                    # warm-up steps reuse ONE gradient buffer back to back: let every peer finish reading it
                    torch.cuda.synchronize()
                    dist.barrier()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = self._step_impl(x, labels)
        self._graphs[(par, key)] = (graph, out)
        with torch.no_grad():
            for t, q in zip((self.flat_p, self.flat_m, self.flat_v, self.state), snap):
                t.copy_(q)
        if self._peer is not None:
            torch.cuda.synchronize()
            dist.barrier()
        self.flat_g, self.gview = keep
        return self._graphs[(par, key)]


class HeadTrainer(FusedTrainer):
    """Training step of a new classifier head on frozen graph convolutions (``finetune.finetuning_cgcnn``).

    ``step(a0, labels)`` takes ``a0 [B, n0]``, the mean over the last conv layer's filters of each window (what
    ``finetuning_cgcnn.trunk_features`` computes once per data set), and runs ``FusedTrainer``'s head on it -- one
    ``gcnb_head_step_f32`` launch for a three-layer head the kernel takes, the layer-by-layer launches otherwise, with the
    same dropout keep-probability, seeds and masks -- followed by ``gcnb_nadam_tf_f32`` (TF's ``NadamOptimizer``) over one
    flat buffer that holds only the FC weights and biases, all regularised.  The conv parameters are never written.
    Captured as one CUDA graph per batch shape; ``bind_inputs`` lets ``InputPipeline`` feed it."""

    def __init__(self, model, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, use_cuda_graph=True):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            raise NotImplementedError("HeadTrainer: data-parallel fine-tuning is not implemented")
        super().__init__(model, lr=lr, distributed=False, use_cuda_graph=use_cuda_graph, beta1=beta1, beta2=beta2,
                         eps=eps, gather=False)

    def _trained_parameters(self, model):
        """The head's weights and biases (updated with TF Nadam whatever ``model.momentum`` says)."""
        return [p for W, b in zip(model.fc_weights, model.fc_bias) for p in (W, b)]

    @torch.no_grad()
    def _step_impl(self, a0, labels):
        lib, C = self._lib.lib(), self.C
        stream = C.c_void_p(torch.cuda.current_stream(a0.device).cuda_stream)
        vp = lambda t: C.c_void_p(t.data_ptr())
        logits, _ = self._head(a0, labels, lib, vp, stream)
        rc = lib.gcnb_nadam_tf_f32(vp(self.flat_p), vp(self.flat_g), vp(self.flat_m), vp(self.flat_v), vp(self.decay),
                                   vp(self.state), self.n, self.lr, self.b1, self.b2, self.eps,
                                   float(self.model.regularization or 0.0), 0, stream)
        self._lib.check(rc, "gcnb_nadam_tf_f32")
        return self._loss, logits


class InputPipeline:
    """Asynchronous input feed of a ``FusedTrainer`` (SURVEY.md 8f row 3; the reference feeds ``feed_dict`` copies,
    models_gcn.py:142-146): batches go from (pinned) host memory to ``depth`` device slots on a copy stream while the
    previous step runs; the slots are bound to the trainer, so a step reads its batch in place.

        pipe = InputPipeline(trainer, (B, n_vertices, channel))
        pipe.feed(x0, y0)
        for x, y in batches:          # host arrays / tensors
            pipe.feed(x, y)           # H2D of the NEXT batch overlaps ...
            loss, logits = pipe.step()  # ... the step on the previous one
    """

    def __init__(self, trainer, x_shape, depth=2, label_dtype=torch.long):
        dev = trainer.flat_p.device
        self.trainer, self.depth = trainer, depth
        self.dx = [torch.empty(*x_shape, dtype=torch.float32, device=dev) for _ in range(depth)]
        self.dy = [torch.empty(x_shape[0], dtype=label_dtype, device=dev) for _ in range(depth)]
        self.hx = [torch.empty(*x_shape, dtype=torch.float32).pin_memory() for _ in range(depth)]
        self.hy = [torch.empty(x_shape[0], dtype=label_dtype).pin_memory() for _ in range(depth)]
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.ready = [torch.cuda.Event() for _ in range(depth)]    # slot filled
        self.freed = [torch.cuda.Event() for _ in range(depth)]    # slot consumed by its step
        self.staged = [torch.cuda.Event() for _ in range(depth)]   # pinned staging buffer of the slot copied out
        for s in range(depth):
            trainer.bind_inputs(self.dx[s], self.dy[s])
            self.freed[s].record(torch.cuda.current_stream())
            self.staged[s].record(self.copy_stream)
        self._head = self._tail = 0   # slots fed / stepped so far

    def feed(self, x, labels):
        """Queue one batch: asynchronous copy into the next free slot (pageable inputs are staged through a pinned
        buffer of the slot first)."""
        if self._head - self._tail >= self.depth:
            raise RuntimeError("InputPipeline: all %d slots are full -- call step() first" % self.depth)
        s = self._head % self.depth
        x, labels = torch.as_tensor(x), torch.as_tensor(labels)
        if not (x.is_cuda or x.is_pinned()):
            self.staged[s].synchronize()
            self.hx[s].copy_(x)
            x = self.hx[s]
        if not (labels.is_cuda or labels.is_pinned()):
            self.staged[s].synchronize()
            self.hy[s].copy_(labels)
            labels = self.hy[s]
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.freed[s])
            self.dx[s].copy_(x, non_blocking=True)
            self.dy[s].copy_(labels, non_blocking=True)
            self.staged[s].record(self.copy_stream)
            self.ready[s].record(self.copy_stream)
        self._head += 1

    def step(self):
        """Run the training step on the oldest queued batch; returns what ``FusedTrainer.step`` returns."""
        if self._tail >= self._head:
            raise RuntimeError("InputPipeline: nothing queued -- call feed() first")
        s = self._tail % self.depth
        main = torch.cuda.current_stream()
        main.wait_event(self.ready[s])
        out = self.trainer.step(self.dx[s], self.dy[s])
        self.freed[s].record(main)
        self._tail += 1
        return out

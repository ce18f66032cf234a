"""``cgcnn`` -- the reference's graph-CNN class, with the same constructor and layer methods.

Mirrors ``/root/reference/lib_new/models_gcn.py``: ``cgcnn.__init__ :445-510`` (argument
checks, Laplacian selection, layers bound by name), the layer methods ``chebyshev5 :587-617``,
``chebyshev2 :558-585``, ``fourier :530-539``, ``b1relu :619-623``, ``b2relu :625-629``,
``mpool1 :631-639``, ``fc :650-656``, ``_inference :658-682`` and the ``base_model`` pieces
``loss :253-276``, ``predict :31-71``, ``fit :112-184`` (loop structure only; there is no
TF session, checkpointing or TensorBoard here -- see DESIGN.md, out of scope).

Differences a reference user will notice:
* tensors are CUDA fp32 ``torch.Tensor``; ``L`` is still the list of SciPy Laplacians.
* parameters exist before the first call (TF creates them while building the graph); their
  names follow the TF variable scopes: ``conv{i}/weights``, ``conv{i}/bias``, ``fc{i}/...``,
  ``logits/...`` (``state_dict_tf()`` / ``load_state_dict_tf()``).
* ``conv(i, x)`` is the fast path: ONE fused kernel per layer (filter+bias+ReLU+pool).
  ``filter``/``brelu``/``pool`` called one by one (as ``_inference`` does in the reference) give
  the same numbers through three kernels.
"""
from __future__ import annotations

import math
from collections import OrderedDict

import numpy as np
import torch
import torch.nn as nn

from . import ops, synth
from .plan import GraphPlan, SpectralPlan


class cgcnn(nn.Module):
    """Graph CNN with Chebyshev / first-order / spectral filters (drop-in for the reference class)."""

    def __init__(self, config=None, L=None, F=None, K=None, p=None, M=None, filter="chebyshev5", brelu="b1relu",
                 pool="mpool1", initial="normal", channel=1, num_epochs=20, learning_rate=0.1, decay_rate=0.95,
                 decay_steps=None, momentum=0.9, regularization=0, dropout=0, batch_size=100, eval_frequency=200,
                 dir_name="", device="cuda", seed=0, perm=None, n_input_vertices=None, algo=ops.ALGO_AUTO,
                 fused=True, verbose=False):
        super().__init__()
        # ---- the reference's consistency checks (models_gcn.py:452-460) ----------------------------
        # The reference only *prints* when ``len(L) >= len(F) == len(K) == len(p)`` fails (:452-456), and its
        # shipped config depends on that: 6 layers with p=1 on 2 Laplacians (model.py:271-274).  Unequal
        # F/K/p lengths crash it a few lines later, so those are rejected here.
        if not (len(F) == len(K) == len(p)):
            raise ValueError("need len(F) == len(K) == len(p) (got %d, %d, %d)" % (len(F), len(K), len(p)))
        if not np.all(np.array(p) >= 1):
            raise ValueError("pooling sizes must be >= 1")
        p_log2 = np.where(np.array(p) > 1, np.log2(np.maximum(p, 1)), 0)
        if not np.all(np.mod(p_log2, 1) == 0):
            raise ValueError("pooling sizes must be powers of 2")
        if not len(L) >= np.sum(p_log2):
            raise ValueError("not enough coarsening levels for the pooling sizes")
        if filter not in ("chebyshev5", "chebyshev2", "fourier"):
            raise ValueError("filter must be 'chebyshev5', 'chebyshev2' or 'fourier' (spline is out of scope)")
        if brelu not in ("b1relu", "b2relu"):
            raise ValueError("brelu must be 'b1relu' or 'b2relu'")
        if pool != "mpool1":
            raise ValueError("pool must be 'mpool1' (apool1 is never selected by the reference, model.py:163)")
        if initial not in ("normal", "he"):
            raise ValueError("initial must be 'normal' or 'he'")

        # ---- keep the useful Laplacians only (models_gcn.py:462-469) ------------------------------
        M_0 = L[0].shape[0]
        j, used = 0, []
        for pp in p:
            used.append(L[j])
            j += int(np.log2(pp)) if pp > 1 else 0
        self.L, self.F, self.K, self.p, self.M = used, list(F), list(K), list(p), list(M)
        self.num_epochs, self.learning_rate = num_epochs, learning_rate
        self.decay_rate, self.decay_steps, self.momentum = decay_rate, decay_steps, momentum
        self.regularization, self.dropout = regularization, dropout
        self.batch_size, self.eval_frequency = batch_size, eval_frequency
        self.dir_name, self.initial, self.channel = dir_name, initial, channel
        self.filter_name, self.brelu_name, self.pool_name = filter, brelu, pool
        self.filter = getattr(self, filter)  # bound by name, like models_gcn.py:504-506
        self.brelu = getattr(self, brelu)
        self.pool = getattr(self, pool)
        self.algo, self.fused = algo, fused
        self.dev = torch.device(device)
        self._layer = None

        # ---- operator plans, uploaded once ---------------------------------------------------------
        self._plans, self._splans = {}, {}
        for Li in self.L:
            if filter == "fourier":
                self._spectral_plan(Li)
            else:
                self._plan(Li)
        self.perm = None
        if perm is not None:
            self.perm = torch.as_tensor(np.asarray(perm), dtype=torch.int32, device=self.dev)
            if self.perm.numel() != M_0:
                raise ValueError("perm must have one entry per vertex of L[0]")
        self.n_input_vertices = n_input_vertices if n_input_vertices is not None else M_0

        # ---- parameters (shapes/initialisers of models_gcn.py:330-355) ------------------------------
        self.seed = int(seed)
        rng = np.random.RandomState(seed)
        self.conv_weights, self.conv_bias = nn.ParameterList(), nn.ParameterList()
        self._regularized = []
        Fin = channel
        for i in range(len(self.p)):
            Mi = self.L[i].shape[0]
            if filter == "fourier":
                W = self._init_weight(rng, (Mi, self.F[i], Fin))
                regularize = True  # models_gcn.py:538
            else:
                W = self._init_weight(rng, (Fin * self.K[i], self.F[i]))
                regularize = filter == "chebyshev5"  # :615 regularised, chebyshev2 :583 not
            bshape = (1, 1, self.F[i]) if brelu == "b1relu" else (1, Mi, self.F[i])
            self.conv_weights.append(nn.Parameter(torch.from_numpy(W).to(self.dev)))
            self.conv_bias.append(nn.Parameter(torch.full(bshape, 0.2, dtype=torch.float32, device=self.dev)))
            if regularize:
                self._regularized.append(self.conv_weights[-1])
            Fin = self.F[i]
        # fully connected head: input width is the number of vertices left (mean over F, :671-673)
        # mpool1 is tf.nn.max_pool SAME: ceil(M / p) vertices survive (models_gcn.py:634-637)
        M_last = -(-self.L[-1].shape[0] // self.p[-1]) if len(self.p) else M_0
        self.fc_weights, self.fc_bias = nn.ParameterList(), nn.ParameterList()
        width = M_last
        for Mi in self.M:
            W = self._init_weight(rng, (width, Mi))
            self.fc_weights.append(nn.Parameter(torch.from_numpy(W).to(self.dev)))
            self.fc_bias.append(nn.Parameter(torch.full((Mi,), 0.2, dtype=torch.float32, device=self.dev)))
            self._regularized += [self.fc_weights[-1], self.fc_bias[-1]]  # fc: both regularised (:652-653)
            width = Mi
        if verbose:
            self.describe()

    # ------------------------------------------------------------------ helpers
    def _init_weight(self, rng, shape):
        if self.initial == "normal":  # tf.truncated_normal_initializer(0, 0.2), models_gcn.py:333
            return synth.truncated_normal(rng, shape, 0.2)
        # 'he' (models_gcn.py:334-337): tf.contrib.layers.variance_scaling_initializer(factor=2.0, mode='FAN_IN',
        # uniform=False) takes fan_in = shape[-2] * prod(shape[:-2]) -- Fin*K for a Chebyshev filter, M*Fout (sic) for
        # the [M, Fout, Fin] spectral weight -- and draws a truncated normal of stddev sqrt(1.3 * factor / fan_in)
        # (contrib's constant 1.3 ~ 1/0.8796^2 compensates the truncation at two standard deviations)
        fan_in = float(shape[-2] if len(shape) > 1 else shape[-1])
        for dim in shape[:-2]:
            fan_in *= float(dim)
        return synth.truncated_normal(rng, shape, math.sqrt(1.3 * 2.0 / fan_in))

    def _plan(self, L):
        key = id(L)
        if key not in self._plans:
            self._plans[key] = (GraphPlan(L, self.dev), L)
        return self._plans[key][0]

    def _spectral_plan(self, L):
        key = id(L)
        if key not in self._splans:
            self._splans[key] = (SpectralPlan(L, self.dev), L)
        return self._splans[key][0]

    def describe(self):
        print("NN architecture")
        print("  input: M_0 = %d" % self.L[0].shape[0])
        for i in range(len(self.p)):
            print("  layer %d: cgconv%d  M=%d F=%d K=%d p=%d  weights %s" % (
                i + 1, i + 1, self.L[i].shape[0], self.F[i], self.K[i], self.p[i], tuple(self.conv_weights[i].shape)))
        for i, Mi in enumerate(self.M):
            print("  layer %d: %s  M=%d" % (len(self.p) + i + 1, "logits" if i == len(self.M) - 1 else "fc%d" % (i + 1), Mi))

    def _bias_mode(self):
        return ops.BIAS_PER_FILTER if self.brelu_name == "b1relu" else ops.BIAS_PER_VERTEX

    def _weights_for(self, layer, W):
        if W is not None:
            return W
        layer = self._layer if layer is None else layer
        if layer is None:
            raise ValueError("call inside _inference, or pass layer=<index> / W=<tensor>")
        return self.conv_weights[layer]

    # ------------------------------------------------------------------ the reference's layer methods
    def chebyshev5(self, x, L, Fout, K, layer=None, W=None):
        """``filter(x, L, Fout, K) -> [B, M, Fout]`` (models_gcn.py:587-617)."""
        W = self._weights_for(layer, W)
        if W.shape[1] != Fout or W.shape[0] != x.shape[2] * K:
            raise ValueError("weights %s do not match Fin*K=%d, Fout=%d" % (tuple(W.shape), x.shape[2] * K, Fout))
        pl = self._plan(L)
        y, _ = ops.cheb_fwd(x, None, *pl.tensors(), W, None, K, 1, ops.BIAS_NONE, False, False, self.algo)
        return y

    def chebyshev2(self, x, L, Fout, K, layer=None, W=None):
        """Same filter; the reference computes the recursion with NumPy on the host (models_gcn.py:558-585)."""
        return self.chebyshev5(x, L, Fout, K, layer=layer, W=W)

    def fourier(self, x, L, Fout, K, layer=None, W=None):
        """Spectral filter; ``K`` is ignored exactly as in the reference (models_gcn.py:530-539, SURVEY D4)."""
        W = self._weights_for(layer, W)
        sp = self._spectral_plan(L)
        y, _ = ops.spectral_fwd(x, sp.Ut, W, None, 1, ops.BIAS_NONE, False, False)
        return y

    def b1relu(self, x, layer=None, b=None):
        """Bias and ReLU, one bias per filter (models_gcn.py:619-623)."""
        b = self.conv_bias[self._layer if layer is None else layer] if b is None else b
        return ops.brelu_fwd(x, b, ops.BIAS_PER_FILTER)

    def b2relu(self, x, layer=None, b=None):
        """Bias and ReLU, one bias per vertex per filter (models_gcn.py:625-629)."""
        b = self.conv_bias[self._layer if layer is None else layer] if b is None else b
        return ops.brelu_fwd(x, b, ops.BIAS_PER_VERTEX)

    def mpool1(self, x, p):
        """Max pooling of size p over the vertex axis (models_gcn.py:631-639)."""
        if p > 1:
            return ops.mpool_fwd(x, p)[0]
        return x

    def fc(self, x, layer, relu=True):
        """Fully connected layer (models_gcn.py:650-656)."""
        x = torch.addmm(self.fc_bias[layer], x, self.fc_weights[layer])
        return torch.relu(x) if relu else x

    # ------------------------------------------------------------------ fused fast path
    def conv(self, i, x, gather=False):
        """Layer ``i`` as ONE fused op: filter -> brelu -> pool.  ``gather`` fuses ``perm_data_3d`` into the load."""
        want_argmax = torch.is_grad_enabled() and self.p[i] > 1
        b = self.conv_bias[i]
        perm = self.perm if gather else None
        if self.filter_name == "fourier":
            if perm is not None:
                x = ops.perm_gather(x, perm)
            sp = self._spectral_plan(self.L[i])
            return ops.spectral_fwd(x, sp.Ut, self.conv_weights[i], b, self.p[i], self._bias_mode(), True, want_argmax)[0]
        pl = self._plan(self.L[i])
        return ops.cheb_fwd(x, perm, *pl.tensors(), self.conv_weights[i], b, self.K[i], self.p[i], self._bias_mode(),
                            True, want_argmax, self.algo)[0]

    # ------------------------------------------------------------------ model
    def conv_stack(self, x, gather=False):
        """The conv loop of ``_inference`` (models_gcn.py:661-668)."""
        if gather and not self.fused:
            x = ops.perm_gather(x, self.perm)
            gather = False
        i, n = 0, len(self.p)
        while i < n:
            if self.fused:
                j = self._stack_run(i, x) if not (gather and i == 0) else i + 1
                if j - i >= 2:
                    # a run of identical layers (the production network, model.py:271-274): ONE launch, the activations
                    # never leave the SM between the layers
                    pl = self._plan(self.L[i])
                    x = ops.cheb_stack_fwd(x, pl.rowptr, pl.col, pl.val, self.conv_weights[i:j], self.conv_bias[i:j],
                                           self.K[i], self._bias_mode(), True,
                                           tap_images=[self._tap_image(q) for q in range(i, j)])
                    i = j
                    continue
                x = self.conv(i, x, gather=gather and i == 0)
            else:
                self._layer = i
                try:
                    x = self.filter(x, self.L[i], self.F[i], self.K[i])
                    x = self.brelu(x)
                    x = self.pool(x, self.p[i])
                finally:
                    self._layer = None
            i += 1
        return x

    def _tap_image(self, i):
        """Pre-split tap image of conv layer ``i`` (cached per weight version: rebuilt when the weights change)."""
        W = self.conv_weights[i]
        key = (W.data_ptr(), W._version)
        cache = self.__dict__.setdefault("_tap_images", {})
        if cache.get(i, (None, None))[0] != key:
            cache[i] = (key, ops.cheb_tap_image(W, W.shape[0] // self.K[i], self.K[i]))
        return cache[i][1]

    def _stack_run(self, i, x):
        """End (exclusive) of the run of layers starting at ``i`` that ``ops.cheb_stack_fwd`` can take in one launch:
        inference, Chebyshev filter, no pooling, 32 -> 32 filters, same operator and K."""
        if torch.is_grad_enabled() or self.filter_name == "fourier" or self.algo == ops.ALGO_GENERAL or x.shape[2] != 32:
            return i + 1
        j = i
        while (j < len(self.p) and j - i < 8 and self.p[j] == 1 and self.F[j] == 32 and self.K[j] == self.K[i]
               and self.L[j] is self.L[i]):
            j += 1
        if j - i >= 2:
            pl = self._plan(self.L[i])
            if not ops.cheb_stack_supported(pl.rowptr, pl.col, pl.val, x.shape[0], 32, self.K[i], j - i):
                return i + 1
        return max(j, i + 1)

    def _inference(self, x, dropout=1.0, gather=False):
        """logits = head(conv_stack(x)); ``dropout`` is the keep probability, as in the reference."""
        x = self.conv_stack(x, gather=gather)
        x = ops.mean_f_fwd(x)  # tf.reduce_mean(x, -1), models_gcn.py:673
        return self._head(x, dropout)

    def _head(self, x, dropout=1.0):
        """The FC layers of ``_inference`` (models_gcn.py:674-682) on the mean over the last conv layer's filters."""
        for i in range(len(self.M) - 1):
            x = self.fc(x, i)
            if dropout < 1.0:
                x = torch.nn.functional.dropout(x, 1.0 - dropout, training=True)
        return self.fc(x, len(self.M) - 1, relu=False)

    def forward(self, x, dropout=1.0, gather=None):
        if gather is None:
            # raw [B, n_input_vertices, C] windows are permuted in the first layer's load; already permuted / padded
            # [B, M_0, C] input is not.  The two cannot be told apart by shape when coarsening added no fake vertices.
            if self.perm is not None and self.n_input_vertices == self.L[0].shape[0]:
                raise ValueError("cgcnn.forward: with perm set and n_input_vertices == M_0 say gather=True (raw windows) "
                                 "or gather=False (already permuted) -- the shapes are identical")
            gather = self.perm is not None and x.shape[1] == self.n_input_vertices != self.L[0].shape[0]
        return self._inference(x, dropout, gather)

    def loss(self, logits, labels, regularization=None):
        """mean sparse-softmax CE + regularization * sum_v ||v||^2/2 (models_gcn.py:253-262)."""
        reg = self.regularization if regularization is None else regularization
        ce = torch.nn.functional.cross_entropy(logits, labels)
        if reg:
            ce = ce + reg * sum(0.5 * (v * v).sum() for v in self._regularized)
        return ce

    @torch.no_grad()
    def predict(self, data, labels=None, return_logits=False):
        """Batched prediction with the reference's zero-padded last batch (models_gcn.py:31-71); with ``return_logits``
        the logits ``[size, n_classes]`` are returned as a third (second, without labels) value -- what
        ``model_perf.predict`` collects (:1012-1016)."""
        return self._predict(data.shape[0], lambda begin: self.forward(self._padded_batch(data, begin)), labels,
                             return_logits)

    def _padded_batch(self, data, begin):
        """Rows ``begin : begin + batch_size`` of ``data`` on the device, zero-padded past its end as ``predict`` pads."""
        bs = self.batch_size
        end = min(begin + bs, data.shape[0])
        batch = torch.zeros((bs,) + tuple(data.shape[1:]), dtype=torch.float32, device=self.dev)
        batch[: end - begin] = torch.as_tensor(np.asarray(data[begin:end]), dtype=torch.float32, device=self.dev)
        return batch

    def _predict(self, size, logits_at, labels, return_logits):
        """``predict`` over ``size`` windows with ``logits_at(begin)`` giving the logits of the batch that starts at window
        ``begin``: the batching, the cropping and the loss of the zero-padded last batch.  Under a process group the
        batches are dealt round-robin over the ranks (``train.deal``) and their logits and losses gathered to every
        rank, which assembles them in batch order: the forward pass is batch-independent, so every rank returns
        bit for bit what one process returns."""
        from . import train

        preds = np.empty(size)
        all_logits = np.empty((size, self.M[-1]), np.float32) if return_logits else None
        total = 0.0
        bs = self.batch_size
        nb = -(-size // bs)

        def one(j):
            begin, end = j * bs, min(j * bs + bs, size)
            logits = logits_at(begin)
            l = 0.0
            if labels is not None:
                lab = torch.zeros(bs, dtype=torch.long, device=self.dev)
                lab[: end - begin] = torch.as_tensor(np.asarray(labels[begin:end]), dtype=torch.long, device=self.dev)
                l = float(self.loss(logits, lab))
                if not np.isfinite(l):
                    l = 0.0
            return logits, l

        def one_as_tensors(j):
            logits, l = one(j)
            return logits, torch.tensor(l, dtype=torch.float64)

        if train.data_parallel()[1] > 1 and nb > 0:
            like = (torch.empty((bs, self.M[-1]), dtype=torch.float32, device=self.dev),
                    torch.empty((), dtype=torch.float64, device=self.dev))
            batches = ((lg, float(l)) for lg, l in train.deal(nb, one_as_tensors, like))
        else:
            batches = (one(j) for j in range(nb))
        for j, (logits, l) in enumerate(batches):
            begin, end = j * bs, min(j * bs + bs, size)
            total += l
            preds[begin:end] = logits.argmax(1)[: end - begin].cpu().numpy()
            if return_logits:
                all_logits[begin:end] = logits[: end - begin].detach().cpu().numpy()
        out = (preds, total * bs / size) if labels is not None else (preds,)
        if return_logits:
            out += (all_logits,)
        return out if len(out) > 1 else out[0]

    def saliency(self, data, target=None, gather=None):
        """Gradient saliency maps: ``(grad [n, n_input_vertices, channel] float32, target [n] int64)``, the gradient of
        the logit of class ``target[i]`` w.r.t. window ``i`` of ``data`` -- which ROIs and which TRs drive the decision.
        ``target=None`` takes the predicted class (the arg-max of the logits, as ``prediction()``).  Batched like
        ``predict``: batches of ``batch_size``, the last one zero-padded.  ``gather`` follows ``forward``: raw windows
        are permuted in the first layer's load and their gradient un-permuted in its store (with ``gather=False`` the
        data and the gradient are in the first layer's vertex order, ``[n, M_0, channel]``).  Runs on the GPU through
        ``saliency.InputGradient`` (one CUDA graph per batch shape)."""
        from .saliency import InputGradient

        M0 = self.L[0].shape[0]
        if gather is None:
            if self.perm is not None and self.n_input_vertices == M0:
                raise ValueError("cgcnn.saliency: with perm set and n_input_vertices == M_0 say gather=True (raw windows) "
                                 "or gather=False (already permuted) -- the shapes are identical")
            gather = self.perm is not None and data.shape[1] == self.n_input_vertices != M0
        gather = bool(gather) and self.perm is not None
        if gather:
            # the first layer writes each raw row's gradient exactly once: that needs a permutation of [0, M_0)
            perm = self.perm.cpu().numpy()
            if not np.array_equal(np.sort(perm), np.arange(M0)):
                raise ValueError("cgcnn.saliency: perm is not a permutation of [0, M_0 = %d)" % M0)
        params = tuple(p.data_ptr() for p in self.parameters())
        cached = self.__dict__.get("_saliency")
        if cached is None or cached[0] != params:
            cached = self.__dict__["_saliency"] = (params, InputGradient(self))
        ig = cached[1]
        size, bs = data.shape[0], self.batch_size
        grads = np.empty((size,) + tuple(data.shape[1:]), np.float32)
        targets = np.empty(size, np.int64)
        for begin in range(0, size, bs):
            end = min(begin + bs, size)
            batch = torch.zeros((bs,) + tuple(data.shape[1:]), dtype=torch.float32, device=self.dev)
            batch[: end - begin] = torch.as_tensor(np.asarray(data[begin:end]), dtype=torch.float32, device=self.dev)
            t = None
            if target is not None:
                t = torch.zeros(bs, dtype=torch.long, device=self.dev)
                t[: end - begin] = torch.as_tensor(np.asarray(target[begin:end]), dtype=torch.long, device=self.dev)
            g, _, tg = ig(batch, t, gather=gather)
            grads[begin:end] = g[: end - begin].cpu().numpy()
            targets[begin:end] = tg[: end - begin].cpu().numpy()
        return grads, targets

    # ------------------------------------------------------------------ base_model's small public methods
    def inference(self, data, dropout=1.0):
        """Logits of a batch (models_gcn.py:224-239); raw windows are permuted on the way in, as in ``forward``."""
        return self.forward(data, dropout)

    def probabilities(self, logits):
        """Class probabilities (models_gcn.py:241-245: ``tf.nn.softmax``)."""
        return torch.softmax(logits, dim=1)

    def prediction(self, logits):
        """Predicted classes (models_gcn.py:247-251: ``tf.argmax(logits, axis=1)``)."""
        return torch.argmax(logits, dim=1)

    def get_var(self, name):
        """Value of a variable by its TF name, e.g. ``'conv1/weights'`` (models_gcn.py:186-191)."""
        sd = self.state_dict_tf()
        key = name[:-2] if name.endswith(":0") else name
        if key not in sd:
            raise KeyError("no variable %r (have: %s)" % (name, ", ".join(sd)))
        return sd[key]

    def fit(self, train_data, train_labels, val_data, val_labels, best_checkpoint_dir=None, trainer=None):
        """The reference's ``fit`` (models_gcn.py:112-184): ``num_epochs * n / batch_size`` steps on random batches (NumPy's
        global generator, as there), every ``eval_frequency`` steps the validation set is evaluated and the three best
        checkpoints by validation accuracy are kept (checkmat.py, directory ``best_checkpoint_dir`` or
        ``checkpoints/<dir_name>/model``).  Returns ``(accuracies, losses, t_step)`` like the reference.  On a CUDA
        device the steps run through ``train.FusedTrainer`` fed by ``train.InputPipeline``."""
        from . import train

        if trainer is None:
            fused = self.dev.type == "cuda" and self.momentum != 0
            trainer = train.FusedTrainer(self) if fused else train.Trainer(self)
        return self._fit(train_data, train_labels, lambda: self.evaluate(val_data, val_labels), best_checkpoint_dir,
                         trainer)

    def _fit(self, train_data, train_labels, evaluate, best_checkpoint_dir, trainer):
        """The loop of ``fit`` on ``train_data`` with ``evaluate()`` giving ``evaluate``'s result at every evaluation.

        Under a process group (``train.fit`` shards the batches) every rank evaluates its share of the validation batches
        and gets the same figures; only rank 0 prints and keeps checkpoints, and every rank waits for it at a barrier
        after each evaluation, so that the kept files exist wherever ``evaluate(checkpoint=...)`` runs next.  Every rank
        returns the same ``(accuracies, losses, t_step)`` (rank 0's ``t_step``)."""
        import os
        import time

        import torch.distributed as dist

        from . import checkpoints, train

        rank, world = train.data_parallel()
        say = print if rank == 0 else (lambda *a, **k: None)
        path = best_checkpoint_dir or os.path.join("checkpoints", self.dir_name, "model")
        keeper = checkpoints.BestCheckpoints(path, num_to_keep=3, maximize=True) if rank == 0 else None
        n = train_data.shape[0]
        say("training with {} steps in total with batch_size={} and epochs={} for training_set={}:".format(
            int(self.num_epochs * n / self.batch_size), self.batch_size, self.num_epochs, n))
        accuracies, losses = [], []
        t_process, t_wall = time.process_time(), time.time()

        def on_eval(step, num_steps, loss_average):
            say("step {} / {} (epoch {:.2f} / {}):".format(step, num_steps, step * self.batch_size / n, self.num_epochs))
            say("  loss_average = {:.2e}".format(loss_average))
            string, accuracy, f1, loss = evaluate()
            accuracies.append(accuracy)
            losses.append(loss)
            say("  validation {}".format(string))
            say("  time: {:.0f}s (wall {:.0f}s)".format(time.process_time() - t_process, time.time() - t_wall))
            if keeper is not None:
                keeper.handle(accuracy, self, step)
            if world > 1:
                dist.barrier()

        history = train.fit(self, train_data, train_labels, trainer=trainer, seed=None, verbose=False, on_eval=on_eval)
        if accuracies:
            say("validation accuracy: peak = {:.2f}, mean = {:.2f}".format(max(accuracies), np.mean(accuracies[-10:])))
        t_step = (time.time() - t_wall) / max(len(history), 1)
        if world > 1:
            t_step = [t_step]
            dist.broadcast_object_list(t_step, src=0)
            t_step = t_step[0]
        return accuracies, losses, t_step

    def evaluate(self, data, labels, checkpoint=None, target_name=None):
        """``(summary string, accuracy %, weighted F1 %, loss)`` over a full data set, like the reference's ``evaluate``
        (models_gcn.py:72-110); ``checkpoint`` (a file written by ``checkpoints.save_checkpoint``) is restored first,
        as the reference restores the latest checkpoint.  With ``target_name`` (class names) the per-class report and
        the confusion matrix are printed first, as the reference does (:94-101)."""
        from . import checkpoints

        if checkpoint is not None:
            checkpoints.load_checkpoint(self, checkpoint)
        from .train import data_parallel

        predictions, loss = self.predict(data, labels)
        if target_name is not None and data_parallel()[0] == 0:   # under a process group rank 0 prints the report
            print(checkpoints.classification_report(labels, predictions, target_name)[0])
            print("Confusion Matrix:")
            print(checkpoints.confusion_matrix(labels, predictions, len(target_name)))
        string, accuracy, f1 = checkpoints.classification_summary(labels, predictions, loss)
        return string, accuracy, f1, loss

    # ------------------------------------------------------------------ TF-style names for checkpoints
    def state_dict_tf(self):
        """Parameters under the reference's TF variable names (models_gcn.py:662,343,351,675,680)."""
        out = OrderedDict()
        for i in range(len(self.p)):
            out["conv%d/weights" % (i + 1)] = self.conv_weights[i].detach().cpu().numpy()
            out["conv%d/bias" % (i + 1)] = self.conv_bias[i].detach().cpu().numpy()
        for i in range(len(self.M)):
            scope = "logits" if i == len(self.M) - 1 else "fc%d" % (i + 1)
            out[scope + "/weights"] = self.fc_weights[i].detach().cpu().numpy()
            out[scope + "/bias"] = self.fc_bias[i].detach().cpu().numpy()
        return out

    @torch.no_grad()
    def load_state_dict_tf(self, d):
        mine = OrderedDict()
        for i in range(len(self.p)):
            mine["conv%d/weights" % (i + 1)] = self.conv_weights[i]
            mine["conv%d/bias" % (i + 1)] = self.conv_bias[i]
        for i in range(len(self.M)):
            scope = "logits" if i == len(self.M) - 1 else "fc%d" % (i + 1)
            mine[scope + "/weights"] = self.fc_weights[i]
            mine[scope + "/bias"] = self.fc_bias[i]
        for k, v in mine.items():
            a = np.asarray(d[k], dtype=np.float32)
            if tuple(a.shape) != tuple(v.shape):
                raise ValueError("%s: shape %s does not match %s" % (k, a.shape, tuple(v.shape)))
            v.copy_(torch.from_numpy(a).to(v.device))


def __getattr__(name):
    # the fine-tuning model lives in finetune.py (it subclasses cgcnn) and is importable from here, next to cgcnn, as the
    # reference keeps both classes in models_gcn.py
    if name == "finetuning_cgcnn":
        from .finetune import finetuning_cgcnn

        return finetuning_cgcnn
    raise AttributeError("module %r has no attribute %r" % (__name__, name))

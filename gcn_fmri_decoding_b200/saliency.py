"""Gradient saliency maps of a trained ``cgcnn``: the gradient of one class's logit with respect to the raw input window
``[n_input_vertices (ROIs), channel (TRs)]`` -- which brain regions and which time points drive the decision.  The
reference ships no code for this; ``cgcnn.saliency`` is the public call.

``InputGradient`` runs an explicit schedule modelled on ``train.FusedTrainer._step_impl``, with nothing updated and no
dropout:

forward : ``cheb_fwd_mean`` per conv layer (no saved basis; y and the arg-max kept, the last layer emits the mean over
          its filters) -> the FC head through ``gcnb_gemm_epilogue_f32(EPI_RELU_DROPOUT, keep = 1)`` / ``gcnb_gemm_f32``,
          keeping the activations
seed    : the one-hot of the target class on the logits
backward: ``EPI_MASK`` GEMMs down to the gradient of the mean -> ``ops.cheb_dx`` per conv layer (input gradient only; the
          first layer un-permutes the Graclus ordering in its store)

The whole schedule is captured as one CUDA graph per batch shape.

``GraphGradient`` (``cgcnn.graph_saliency``) differentiates the same logit w.r.t. the entries of the graph Laplacians
instead: the same forward, seed and head backward, then ``ops.cheb_dL`` per conv layer (the operator gradient of
``k_sddmm_tma`` on the general path's stacks, and the input gradient that feeds the layer below).
``AdjacencyGradient`` (``cgcnn.adjacency_saliency``) carries those per-level gradients on to the edge weights of the
adjacency the Laplacians were built from (``ops.adjacency_grad``, with the host maps of ``AdjacencyMaps``).

Every class also has a grouped mode (``group=...``): instead of per-window values it returns, per group of windows (a
class, a subject, a run), the sum of the windows' gradients (or of their absolute values) -- the fixed-order grouped
column sum ``gcnb_group_colsum_f32`` inside the same CUDA graph, so only ``[n_groups, ...]`` leaves the device.

The ``fourier`` filter has no input-gradient-only kernel: its layers go through ``spectral_bwd(need_dx=True)``, which also
computes the weight and bias gradients that are then dropped, and the first layer is un-permuted by ``ops.unpermute``.
That path is correct but not optimised.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib, ops


class InputGradient:
    """``grad, logits, target = InputGradient(model)(x, target=None, gather=...)``: the gradient of
    ``logits[b, target[b]]`` w.r.t. ``x`` for every window ``b`` of the batch; ``target=None`` takes the predicted class
    (the arg-max of the logits).  ``gather``: ``x`` holds raw windows ``[B, n_input_vertices, channel]`` that the first
    layer permutes (``model.perm`` must then be a permutation of ``[0, M_0)``, which ``cgcnn.saliency`` checks); else
    ``x`` is already in the first layer's vertex order ``[B, M_0, channel]``.

    Grouped mode, ``group`` (int32 ``[B]`` on the device, or ``"target"``): ``(sums [n_groups, *x.shape[1:]], logits,
    target)`` with ``sums[g]`` the sum of the gradients of the windows ``b`` with ``group[b] == g`` (``absolute``: of
    their absolute values).  Rows with a group outside ``[0, n_groups)`` (-1 on padding rows) count nowhere, and rows of
    ``sums`` whose group occurs in no row are not written.  ``n_groups`` defaults to ``B``; the cost does not depend on
    it.  ``group="target"`` groups by the differentiated class: ``n_groups`` is the number of classes, the first
    ``valid`` rows (None: all) are windows, and ``sums`` is zeroed first.

    With ``use_cuda_graph`` the returned tensors belong to the captured graph of that batch shape and are overwritten by
    the next call with the same shape.  A graph reads the model's parameters where they are when it is captured: build a
    new ``InputGradient`` after the parameters are replaced (not merely updated in place).
    """

    def __init__(self, model, use_cuda_graph=True):
        if model.filter_name not in ("chebyshev5", "chebyshev2", "fourier"):
            raise ValueError("InputGradient: unsupported filter %r" % model.filter_name)
        self.model = model
        self.use_cuda_graph = use_cuda_graph
        self._graphs = {}  # (x shape, gather, target given, ..., grouping) -> (static inputs, outputs, graph)
        self._step = None  # device counter of the dropout generator: keep = 1 never reads a mask, but the call takes one

    # -- one run, eagerly --------------------------------------------------------------------------------------------
    @torch.no_grad()
    def _forward(self, x, target, gather, mask=None):
        """The forward pass, the seed and the head backward: ``(saved, d, logits, target)`` with ``saved[i] = (layer
        input, perm, y, argmax, plan)`` and ``d`` the gradient of the mean over the last conv layer's filters.  ``mask``
        (float32 [B] of 0 / 1, optional) zeroes the seed of the rows marked 0."""
        m = self.model
        lib = _lib.lib()
        stream = C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
        vp = lambda t: C.c_void_p(t.data_ptr())
        mode = m._bias_mode()
        cheb = m.filter_name != "fourier"
        nconv, nfc = len(m.p), len(m.M)
        if self._step is None or self._step.device != x.device:
            self._step = torch.zeros(4, dtype=torch.float32, device=x.device)
        # ---- forward: conv stack ----
        saved, h, h0 = [], x, None
        for i in range(nconv):
            perm = m.perm if (gather and i == 0) else None
            if cheb:
                pl = m._plan(m.L[i])
                y, am, hm, _ = ops.cheb_fwd_mean(h, perm, pl.rowptr, pl.col, pl.val, m.conv_weights[i], m.conv_bias[i],
                                                 m.K[i], m.p[i], mode, True, m.algo, False)
                if i == nconv - 1:
                    h0 = hm
                saved.append((h, perm, y, am, pl))
            else:
                hin = ops.perm_gather(h, perm) if perm is not None else h
                sp = m._spectral_plan(m.L[i])
                y, am = ops.spectral_fwd(hin, sp.Ut, m.conv_weights[i], m.conv_bias[i], m.p[i], mode, True, True)
                saved.append((hin, perm, y, am, sp))
            h = y
        if h0 is None:
            h0 = ops.mean_f_fwd(h)
        # ---- forward: head (hidden layers: ReLU fused into the GEMM store, keep-probability 1) ----
        def gemm(A, Bm, out, bias, ta, tb, M_, N_, K_, epi=None, aux=None):
            if epi is None:
                rc = lib.gcnb_gemm_f32(vp(A), vp(Bm), vp(out), None if bias is None else vp(bias), M_, N_, K_, A.shape[1],
                                       Bm.shape[1], out.shape[1], ta, tb, stream)
            else:
                rc = lib.gcnb_gemm_epilogue_f32(vp(A), vp(Bm), vp(out), None if bias is None else vp(bias), M_, N_, K_,
                                                A.shape[1], Bm.shape[1], out.shape[1], ta, tb, epi,
                                                None if aux is None else vp(aux), 0 if aux is None else aux.shape[1], 1.0,
                                                0, vp(self._step), stream)
            _lib.check(rc, "gcnb_gemm_f32" if epi is None else "gcnb_gemm_epilogue_f32")
            return out

        B = h0.shape[0]
        acts = [h0]
        for i in range(nfc):
            W = m.fc_weights[i]
            out = torch.empty((B, W.shape[1]), dtype=torch.float32, device=x.device)
            hidden = i < nfc - 1
            acts.append(gemm(acts[-1], W, out, m.fc_bias[i], 0, 0, B, W.shape[1], W.shape[0],
                             _lib.EPI_RELU_DROPOUT if hidden else None))
        logits = acts[-1]
        if target is None:
            target = logits.argmax(1)
        # ---- seed and head backward: d = one-hot(target); d <- (d W^T) masked by the activation it came from ----
        d = torch.zeros_like(logits)
        d.scatter_(1, target.view(-1, 1), 1.0)
        if mask is not None:
            d.mul_(mask.view(-1, 1))
        for i in range(nfc - 1, -1, -1):
            W = m.fc_weights[i]
            dn = torch.empty((B, W.shape[0]), dtype=torch.float32, device=x.device)
            if i > 0:
                d = gemm(d, W, dn, None, 0, 1, B, W.shape[0], W.shape[1], _lib.EPI_MASK, acts[i])
            else:
                d = gemm(d, W, dn, None, 0, 1, B, W.shape[0], W.shape[1])
        return saved, d, logits, target

    @torch.no_grad()
    def _impl(self, x, target, gather, group=None, mask=None, grouping=None):
        m = self.model
        mode = m._bias_mode()
        cheb = m.filter_name != "fourier"
        nconv = len(m.p)
        saved, d, logits, target = self._forward(x, target, gather)
        h = saved[-1][2]
        # ---- conv backward: input gradients only (d is the gradient of the mean over the last layer's filters) ----
        if cheb:
            dy, dy_is_mean = d, True
        else:
            dy, dy_is_mean = ops.mean_f_bwd(d, h.shape[-1]), False
        for i in range(nconv - 1, -1, -1):
            hin, perm, y, am, pl = saved[i]
            M_in = x.shape[1] if i == 0 else hin.shape[1]
            if cheb:
                dy = ops.cheb_dx(hin, perm, M_in, y, am, dy, dy_is_mean, *pl.tensors(), m.conv_weights[i], m.K[i], m.p[i],
                                 True, m.algo)
            else:
                # the spectral layer has no input-gradient-only kernel: spectral_bwd also computes dW / db, which are
                # dropped, and the first layer is un-permuted in a separate scatter.  Correct, not optimised.
                dy, _, _ = ops.spectral_bwd(hin, y, am, dy, pl.Ut, m.conv_weights[i], m.p[i], mode, True, True)
                if perm is not None:
                    dy = ops.unpermute(dy, perm, M_in)
            dy_is_mean = False
        if grouping is None:
            return dy, logits, target
        n_groups, absolute, _ = grouping
        B = x.shape[0]
        out = _grouped_out((n_groups,) + tuple(x.shape[1:]), grouping, x.device)
        _group_sums([(dy.reshape(B, -1), out.view(n_groups, -1))], _group_vector(group, target, mask), n_groups,
                    absolute)
        return out, logits, target

    def _grouping(self, x, group, n_groups, absolute, valid):
        """The grouped call's ``(group int32 [B] or None, mask or None, (n_groups, absolute, by target))`` (None:
        ungrouped)."""
        B = x.shape[0]
        if group is None:
            return None, None, None
        if isinstance(group, str):
            if group != "target":
                raise ValueError("%s: group must be an int32 tensor or 'target' (got %r)" % (type(self).__name__, group))
            valid = B if valid is None else int(valid)
            mask = (torch.arange(B, device=x.device) < valid).to(torch.float32)
            return None, mask, (int(self.model.M[-1]), bool(absolute), True)
        n_groups = B if n_groups is None else int(n_groups)
        if not 1 <= n_groups <= B:
            raise ValueError("%s: n_groups = %d outside [1, B = %d]" % (type(self).__name__, n_groups, B))
        group = torch.as_tensor(group, dtype=torch.int32, device=x.device)
        if tuple(group.shape) != (B,):
            raise ValueError("%s: group must have shape [%d] (got %s)" % (type(self).__name__, B, tuple(group.shape)))
        return group, None, (n_groups, bool(absolute), False)

    def _run(self, key, fn, *inputs):
        """``fn(*inputs)``; with ``use_cuda_graph`` replayed from the CUDA graph of ``key``, captured on static copies of
        the tensor ``inputs`` (a None input stays None) and fed by copies into them."""
        if not self.use_cuda_graph:
            return fn(*inputs)
        if key not in self._graphs:
            static = tuple(None if t is None else t.clone() for t in inputs)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):  # warm up: allocator, lazy library set-up, operator images
                    fn(*static)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = fn(*static)
            self._graphs[key] = (static, out, graph)
        static, out, graph = self._graphs[key]
        for s_, t in zip(static, inputs):
            if s_ is not None:
                s_.copy_(t, non_blocking=True)
        graph.replay()
        return out

    def __call__(self, x, target=None, gather=False, group=None, n_groups=None, absolute=False, valid=None):
        """``(grad [B, *x.shape[1:]], logits [B, C], target [B] int64)`` for the batch ``x`` (float32, on the model's
        device); ``target`` (int64 [B] or None) is the class whose logit is differentiated.  With ``group``: ``(sums
        [n_groups, *x.shape[1:]], logits, target)`` (see the class)."""
        gather = bool(gather) and self.model.perm is not None
        if target is not None:
            target = torch.as_tensor(target, dtype=torch.long, device=x.device)
        group, mask, grouping = self._grouping(x, group, n_groups, absolute, valid)
        if grouping is None and absolute:
            raise ValueError("InputGradient: absolute needs group (the per-window gradient is returned signed)")
        key = (tuple(x.shape), gather, target is not None, grouping)
        return self._run(key, lambda sx, st, sg, sm: self._impl(sx, st, gather, sg, sm, grouping), x, target, group,
                         mask)


class GraphGradient(InputGradient):
    """``grads, logits, target = GraphGradient(model)(x, target=None, gather=False, valid=None, absolute=False)``: the
    gradient of ``logits[b, target[b]]`` w.r.t. every entry of every graph Laplacian the network uses -- which
    connections of the graph the decision relies on -- summed over the windows ``b`` of the batch.

    ``grads[level]`` (float32 ``[nnz + M]``, ``level`` an index into the model's constructor ``L`` list) holds the
    entries of the rescaled operator's CSR pattern (``GraphPlan``'s order) followed by the diagonal ``(i, i)``.  The
    gradient w.r.t. ``L~ = L - I`` is the gradient w.r.t. ``L``.  ``valid``: the first ``valid`` rows are windows, the
    rest padding, whose seed is zero.  ``absolute``: ``sum_b |dL_b|`` instead of ``sum_b dL_b``, the absolute value taken
    per window after the contributions of every layer that uses the Laplacian are added up.

    Schedule: ``InputGradient``'s forward, seed and head backward, then from the top conv layer down one
    ``ops.cheb_dL`` per layer, accumulating into one ``[B, nnz + M]`` buffer per distinct Laplacian (its ``dx`` feeds the
    layer below), and a fixed-order sum over the windows per buffer (``gcnb_colsum_multi_f32``).  One CUDA graph per
    batch shape.  The ``fourier`` filter is refused: its operator is the eigenbasis, not ``L``.

    Grouped mode (``group``, ``n_groups`` as in ``InputGradient``): ``grads[level] = (sums [n_groups, nnz], sums
    [n_groups, M])``, the CSR-entry and diagonal blocks summed per group by ``gcnb_group_colsum_f32`` (with
    ``absolute`` the absolute value fused into that sum, still per window after all layers are added up).
    """

    def __init__(self, model, use_cuda_graph=True):
        if model.filter_name == "fourier":
            raise ValueError("GraphGradient: the fourier filter's operator is the eigenbasis U, not the Laplacian L")
        super().__init__(model, use_cuda_graph)

    @torch.no_grad()
    def _level_grads(self, x, target, gather, mask):
        """The forward pass, the seed and the ``cheb_dL`` loop: ``(bufs, logits, target)`` with ``bufs[level] = (buf,
        dval [B, nnz], ddiag [B, M])``, the per-window gradient w.r.t. that level's operator."""
        m = self.model
        nconv = len(m.p)
        saved, dy, logits, target = self._forward(x, target, gather, mask)
        B = x.shape[0]
        bufs = {}  # level -> (dL [B, nnz + M] as its dval [B, nnz] and ddiag [B, M] blocks)
        dy_is_mean = True
        for i in range(nconv - 1, -1, -1):
            hin, perm, y, am, pl = saved[i]
            lvl = m._graph_levels[i]
            accumulate = lvl in bufs
            if not accumulate:
                buf = torch.empty(B * (pl.nnz + pl.M), dtype=torch.float32, device=x.device)
                bufs[lvl] = (buf, buf[: B * pl.nnz].view(B, pl.nnz), buf[B * pl.nnz:].view(B, pl.M))
            _, dval, ddiag = bufs[lvl]
            M_in = x.shape[1] if i == 0 else hin.shape[1]
            dy = ops.cheb_dL(hin, perm, M_in, y, am, dy, dy_is_mean, *pl.tensors(), m.conv_weights[i], dval, ddiag,
                             accumulate, m.K[i], m.p[i], True, i > 0)
            dy_is_mean = False
        return bufs, logits, target

    @torch.no_grad()
    def _impl(self, x, target, gather, mask=None, absolute=False, group=None, grouping=None):
        bufs, logits, target = self._level_grads(x, target, gather, mask)
        if grouping is not None:
            n_groups, absolute, _ = grouping
            out, mats = {}, []
            for lvl, (buf, dval, ddiag) in sorted(bufs.items()):
                out[lvl] = tuple(_grouped_out((n_groups, a.shape[1]), grouping, x.device) for a in (dval, ddiag))
                mats += [(a, o) for a, o in zip((dval, ddiag), out[lvl]) if a.shape[1]]
            _group_sums(mats, _group_vector(group, target, mask), n_groups, absolute)
            return out, logits, target
        # ---- sum over the windows, fixed order: the dval and ddiag blocks of every buffer as column sums ----
        out, mats = {}, []
        for lvl, (buf, dval, ddiag) in sorted(bufs.items()):
            if absolute:
                buf.abs_()
            o = torch.empty(dval.shape[1] + ddiag.shape[1], dtype=torch.float32, device=x.device)
            out[lvl] = o
            if dval.shape[1]:
                mats.append((dval, o[: dval.shape[1]]))
            mats.append((ddiag, o[dval.shape[1]:]))
        _colsums(mats, x.device)
        return out, logits, target

    def __call__(self, x, target=None, gather=False, valid=None, absolute=False, group=None, n_groups=None):
        """``({level: float32 [nnz + M]}, logits [B, C], target [B] int64)`` for the batch ``x`` (float32, on the model's
        device); ``target`` (int64 [B] or None) is the class whose logit is differentiated, ``valid`` the number of
        leading rows that are windows (None: all).  With ``group``: ``({level: (sums [n_groups, nnz], sums [n_groups,
        M])}, logits, target)`` (see the class)."""
        gather = bool(gather) and self.model.perm is not None
        B = x.shape[0]
        valid = B if valid is None else int(valid)
        mask = (torch.arange(B, device=x.device) < valid).to(torch.float32)
        if target is not None:
            target = torch.as_tensor(target, dtype=torch.long, device=x.device)
        group, _, grouping = self._grouping(x, group, n_groups, absolute, valid)
        absolute = bool(absolute)
        key = (tuple(x.shape), gather, target is not None, absolute, grouping)
        return self._run(key, lambda sx, st, sm, sg: self._impl(sx, st, gather, sm, absolute, sg, grouping), x, target,
                         mask, group)


def _colsums(mats, device):
    """``out = a.sum(0)`` in a fixed order for every ``(a [R, C], out [C])`` of ``mats`` (``gcnb_colsum_multi_f32``, up
    to four matrices per launch)."""
    lib = _lib.lib()
    stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    for c in range(0, len(mats), 4):
        part = mats[c:c + 4]
        n = len(part)
        rc = lib.gcnb_colsum_multi_f32((C.c_void_p * n)(*[a.data_ptr() for a, _ in part]),
                                       (C.c_void_p * n)(*[o.data_ptr() for _, o in part]),
                                       (C.c_int * n)(*[a.shape[0] for a, _ in part]),
                                       (C.c_int * n)(*[a.shape[1] for a, _ in part]), n, stream)
        _lib.check(rc, "gcnb_colsum_multi_f32")


def _group_sums(mats, group, n_groups, absolute):
    """``out[g] = sum of the rows r of a with group[r] == g`` (``|a|`` with ``absolute``) in a fixed order for every
    ``(a [R, C], out [n_groups, C])`` of ``mats`` (``gcnb_group_colsum_f32``, one launch each); ``group`` int32 [R] on
    the device.  Rows of ``out`` whose group occurs in no row are not written."""
    lib = _lib.lib()
    stream = C.c_void_p(torch.cuda.current_stream(group.device).cuda_stream)
    for a, out in mats:
        a = a.contiguous()  # the kernel takes dense rows; ops.unpermute's gradient (fourier) is a strided view
        rc = lib.gcnb_group_colsum_f32(C.c_void_p(a.data_ptr()), a.shape[0], a.shape[1], C.c_void_p(group.data_ptr()),
                                       n_groups, int(absolute), C.c_void_p(out.data_ptr()), stream)
        _lib.check(rc, "gcnb_group_colsum_f32")


def _group_vector(group, target, mask):
    """The group of every row of a grouped call: ``group`` as given, or (``group`` None: by target) the target class,
    -1 on the padding rows (``mask`` 0)."""
    if group is not None:
        return group
    return torch.where(mask > 0, target, torch.full_like(target, -1)).to(torch.int32)


def _grouped_out(shape, grouping, device):
    """The float32 output of a grouped sum: zeroed when grouped by target (rows of absent classes are not written)."""
    return (torch.zeros if grouping[2] else torch.empty)(shape, dtype=torch.float32, device=device)


class AdjacencyMaps:
    """The host maps of the chain rule from the per-level operator gradients of ``GraphGradient`` to the undirected edge
    weights of the adjacency ``A`` the model's Laplacians were built from (``A -> graclus.coarsen -> graphs.laplacian``
    per level), built once per model and ``A``.

    The coarsening is recomputed from ``A`` with ``len(L) - 1`` levels of the constructor's ``L`` list; its vertex order
    must be ``model.perm`` and every Laplacian the network uses must come out, rescaled and cast to fp32, exactly as
    the model's operator.  Per used level (finest first): ``tpos`` (the position in the operator's CSR of each entry of
    the transpose's CSR order), ``ss = s_a s_b`` per entry and ``hinv = 1 / (2 d)`` per vertex (fp64, then fp32; 0 for
    an isolated vertex), and ``parent``, the entry of the next used level that entry ``(a, b)`` is summed into through
    the coarsening (``(a >> q, b >> q)``, q the levels in between; -1 for a pair inside one cluster).  ``edges [E, 2]``:
    the level-0 entries ``(a, b)``, ``(b, a)`` of every edge ``(rows[k], cols[k])``, ``rows < cols``, of ``A`` (the
    upper triangle in CSR order)."""

    def __init__(self, model, A):
        from . import graclus, graphs

        if model.filter_name == "fourier":
            raise ValueError("adjacency saliency: the fourier filter's operator is the eigenbasis U, not the Laplacian L")
        A = sp.csr_matrix(A, copy=True)
        if A.shape[0] != A.shape[1]:
            raise ValueError("adjacency saliency: A must be square (got %s)" % (A.shape,))
        if not np.issubdtype(A.dtype, np.floating):
            raise ValueError("adjacency saliency: A must hold floating-point weights (got %s)" % A.dtype)
        A.sum_duplicates()
        A.eliminate_zeros()
        if (A != A.T).nnz:
            raise ValueError("adjacency saliency: A must be symmetric")
        if A.diagonal().any():
            raise ValueError("adjacency saliency: A must have a zero diagonal")
        state = np.random.get_state()  # graclus.metis seeds the global generator, as the reference does
        try:
            gs, perm = graclus.coarsen(A, model._n_laplacians - 1)
        finally:
            np.random.set_state(state)
        mperm = None if model.perm is None else model.perm.cpu().numpy()
        if (perm is None) != (mperm is None) or (perm is not None and not np.array_equal(perm, mperm)):
            raise ValueError("adjacency saliency: the vertex order of A's coarsening differs from model.perm")
        used = sorted(set(model._graph_levels))
        self.n, self.levels, host = A.shape[0], used, []
        for lvl in range(used[-1] + 1):
            rp, ci, v = graphs.csr_arrays(graphs.rescale_L(graphs.laplacian(gs[lvl])))
            M = len(rp) - 1
            rows = np.repeat(np.arange(M), np.diff(rp)).astype(np.int64)
            if lvl in used:
                pl = model._plan(model.L[model._graph_levels.index(lvl)])
                if not all(np.array_equal(a, b) for a, b in zip((rp, ci, v), pl._host[False])):
                    raise ValueError("adjacency saliency: the Laplacian of level %d built from A (rescaled, fp32) is not "
                                     "the model's" % lvl)
            G = sp.csr_matrix(gs[lvl], dtype=np.float64)
            G.sum_duplicates()
            G.sort_indices()
            if not (np.array_equal(G.indptr, rp) and np.array_equal(G.indices, ci)):
                raise ValueError("adjacency saliency: level %d: the operator's pattern is not the adjacency's" % lvl)
            d = np.asarray(G.sum(axis=0)).ravel()
            s = np.where(d > 0, 1 / np.sqrt(np.where(d > 0, d, 1)), 0)
            host.append(dict(M=M, rows=rows, cols=ci.astype(np.int64), tpos=np.lexsort((rows, ci)),
                             ss=(s[rows] * s[ci]).astype(np.float32),
                             hinv=np.where(d > 0, 0.5 / np.where(d > 0, d, 1), 0).astype(np.float32)))
        # entry (a, b) of level l -> entry (a >> 1, b >> 1) of level l + 1, then composed across the unused levels
        for lvl in range(used[-1]):
            h, up = host[lvl], host[lvl + 1]
            pa, pb = h["rows"] >> 1, h["cols"] >> 1
            cross = pa != pb
            h["up"] = np.full(len(pa), -1, np.int64)
            h["up"][cross] = _entry_index(up, pa[cross], pb[cross])
        self.parent = {}
        for i, lvl in enumerate(used):
            if i + 1 == len(used):
                self.parent[lvl] = None
                continue
            par = host[lvl]["up"]
            for mid in range(lvl + 1, used[i + 1]):
                par = np.where(par >= 0, host[mid]["up"][np.maximum(par, 0)], -1)
            self.parent[lvl] = par.astype(np.int32)
        # the edges of A in ROI order -> their two level-0 entries in the model's vertex order
        U = sp.triu(A, 1).tocsr()
        self.rows = np.repeat(np.arange(self.n), np.diff(U.indptr))
        self.cols = U.indices.astype(np.int64)
        inv = np.arange(host[0]["M"])
        if perm is not None:
            inv[np.asarray(perm)] = np.arange(len(perm))
        a, b = inv[self.rows], inv[self.cols]
        self.edges = np.stack([_entry_index(host[0], a, b), _entry_index(host[0], b, a)], 1).astype(np.int32)
        self.tpos = {lvl: host[lvl]["tpos"].astype(np.int32) for lvl in used}
        self.ss = {lvl: host[lvl]["ss"] for lvl in used}
        self.hinv = {lvl: host[lvl]["hinv"] for lvl in used}
        self._dev = {}

    def device(self, device):
        """The maps as device tensors: ``({level: (tpos, ss, hinv, parent or None)}, edges)``."""
        device = torch.device(device)
        if device not in self._dev:
            t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(device)
            self._dev[device] = ({lvl: (t(self.tpos[lvl]), t(self.ss[lvl]), t(self.hinv[lvl]), t(self.parent[lvl]))
                                  for lvl in self.levels}, t(self.edges))
        return self._dev[device]

    def matrix(self, g):
        """Symmetric ``[n, n]`` float64 CSR on the pattern of ``A`` from an edge vector ``g [E]``."""
        g = np.asarray(g, np.float64)
        return sp.csr_matrix((np.concatenate([g, g]), (np.concatenate([self.rows, self.cols]),
                                                       np.concatenate([self.cols, self.rows]))), shape=(self.n, self.n))


def _entry_index(h, r, c):
    """Positions of the entries ``(r[k], c[k])`` in a level's CSR order (sorted rows); every entry must be stored."""
    key = h["rows"] * h["M"] + h["cols"]
    q = np.asarray(r, np.int64) * h["M"] + np.asarray(c, np.int64)
    pos = np.minimum(np.searchsorted(key, q), max(len(key) - 1, 0))
    if len(q) and (len(key) == 0 or (key[pos] != q).any()):
        raise ValueError("adjacency saliency: the coarsening maps an entry onto one its coarser level does not store")
    return pos


class AdjacencyGradient(GraphGradient):
    """``g, logits, target = AdjacencyGradient(model, maps)(x, target=None, gather=False, valid=None, absolute=False)``:
    the gradient of ``logits[b, target[b]]`` w.r.t. every undirected edge weight of the adjacency ``A`` behind the
    model's Laplacians (``maps = AdjacencyMaps(model, A)``), summed over the windows ``b`` of the batch: float32
    ``[E]`` in the order of ``maps.rows / maps.cols``.  ``absolute``: ``sum_b |dA_b|``, the absolute value taken per
    window after every path through which the weight reaches the network is added up.

    Schedule: ``GraphGradient``'s forward, seed and ``cheb_dL`` loop, then ``ops.adjacency_grad`` on the per-level
    buffers (the chain through each level's degree normalisation and the coarsening, into ``[B, E]``) and a
    fixed-order sum over the windows (``gcnb_colsum_multi_f32``).  One CUDA graph per batch shape.

    Grouped mode (``group``, ``n_groups`` as in ``InputGradient``): ``g [n_groups, E]``, the per-window edge gradients
    summed per group by ``gcnb_group_colsum_f32``."""

    def __init__(self, model, maps, use_cuda_graph=True):
        super().__init__(model, use_cuda_graph)
        self.maps = maps

    @torch.no_grad()
    def _impl(self, x, target, gather, mask=None, absolute=False, group=None, grouping=None):
        m = self.model
        bufs, logits, target = self._level_grads(x, target, gather, mask)
        per_level, edges = self.maps.device(x.device)
        levels = []
        for lvl in self.maps.levels:
            pl = m._plan(m.L[m._graph_levels.index(lvl)])
            levels.append((bufs[lvl][1], pl.rowptr, pl.val, pl.rowptr_t) + per_level[lvl])
        if grouping is not None:
            n_groups, absolute, _ = grouping
            S = ops.adjacency_grad(levels, edges, False)
            out = _grouped_out((n_groups, S.shape[1]), grouping, x.device)
            if S.shape[1]:
                _group_sums([(S, out)], _group_vector(group, target, mask), n_groups, absolute)
            return out, logits, target
        S = ops.adjacency_grad(levels, edges, absolute)
        out = torch.empty(S.shape[1], dtype=torch.float32, device=x.device)
        if S.shape[1]:
            _colsums([(S, out)], x.device)
        return out, logits, target


def edge_matrix(plan, g):
    """``[M, M]`` float64 CSR from a ``GraphGradient`` vector ``g [nnz + M]`` of ``plan``'s operator: the off-diagonal
    entries of its CSR pattern and the whole diagonal (the pattern of ``L``).  A diagonal entry the operator stores
    itself holds the same quantity as ``g[nnz + i]`` and is taken from there once."""
    rp, ci, _ = plan._host[False]
    M, nnz = plan.M, plan.nnz
    g = np.asarray(g, np.float64)
    rows = np.repeat(np.arange(M), np.diff(rp))
    off = rows != ci
    r = np.concatenate([rows[off], np.arange(M)])
    c = np.concatenate([ci[off], np.arange(M)])
    v = np.concatenate([g[:nnz][off], g[nnz:]])
    return sp.csr_matrix((v, (r, c)), shape=(M, M))


def to_input_order(G, perm, M_in):
    """A level-0 edge matrix in the model's vertex order -> input-ROI order ``[M_in, M_in]``: entry ``(i, j)`` goes to
    ``(perm[i], perm[j])``; entries that touch a fake vertex (``perm >= M_in``) are dropped."""
    perm = np.asarray(perm)
    G = sp.coo_matrix(G)
    keep = (perm[G.row] < M_in) & (perm[G.col] < M_in)
    return sp.csr_matrix((G.data[keep], (perm[G.row[keep]], perm[G.col[keep]])), shape=(M_in, M_in))

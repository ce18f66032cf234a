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

The ``fourier`` filter has no input-gradient-only kernel: its layers go through ``spectral_bwd(need_dx=True)``, which also
computes the weight and bias gradients that are then dropped, and the first layer is un-permuted by ``ops.unpermute``.
That path is correct but not optimised.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib, ops


class InputGradient:
    """``grad, logits, target = InputGradient(model)(x, target=None, gather=...)``: the gradient of
    ``logits[b, target[b]]`` w.r.t. ``x`` for every window ``b`` of the batch; ``target=None`` takes the predicted class
    (the arg-max of the logits).  ``gather``: ``x`` holds raw windows ``[B, n_input_vertices, channel]`` that the first
    layer permutes (``model.perm`` must then be a permutation of ``[0, M_0)``, which ``cgcnn.saliency`` checks); else
    ``x`` is already in the first layer's vertex order ``[B, M_0, channel]``.

    With ``use_cuda_graph`` the returned tensors belong to the captured graph of that batch shape and are overwritten by
    the next call with the same shape.  A graph reads the model's parameters where they are when it is captured: build a
    new ``InputGradient`` after the parameters are replaced (not merely updated in place).
    """

    def __init__(self, model, use_cuda_graph=True):
        if model.filter_name not in ("chebyshev5", "chebyshev2", "fourier"):
            raise ValueError("InputGradient: unsupported filter %r" % model.filter_name)
        self.model = model
        self.use_cuda_graph = use_cuda_graph
        self._graphs = {}  # (x shape, gather, target given) -> (static x, static target, outputs, graph)
        self._step = None  # device counter of the dropout generator: keep = 1 never reads a mask, but the call takes one

    # -- one run, eagerly --------------------------------------------------------------------------------------------
    @torch.no_grad()
    def _impl(self, x, target, gather):
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
        for i in range(nfc - 1, -1, -1):
            W = m.fc_weights[i]
            dn = torch.empty((B, W.shape[0]), dtype=torch.float32, device=x.device)
            if i > 0:
                d = gemm(d, W, dn, None, 0, 1, B, W.shape[0], W.shape[1], _lib.EPI_MASK, acts[i])
            else:
                d = gemm(d, W, dn, None, 0, 1, B, W.shape[0], W.shape[1])
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
        return dy, logits, target

    def __call__(self, x, target=None, gather=False):
        """``(grad [B, *x.shape[1:]], logits [B, C], target [B] int64)`` for the batch ``x`` (float32, on the model's
        device); ``target`` (int64 [B] or None) is the class whose logit is differentiated."""
        gather = bool(gather) and self.model.perm is not None
        if target is not None:
            target = torch.as_tensor(target, dtype=torch.long, device=x.device)
        if not self.use_cuda_graph:
            return self._impl(x, target, gather)
        key = (tuple(x.shape), gather, target is not None)
        if key not in self._graphs:
            sx = torch.empty_like(x)
            st = torch.zeros(x.shape[0], dtype=torch.long, device=x.device) if target is not None else None
            sx.copy_(x)
            if st is not None:
                st.copy_(target)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):  # warm up: allocator, lazy library set-up, operator images
                    self._impl(sx, st, gather)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self._impl(sx, st, gather)
            self._graphs[key] = (sx, st, out, graph)
        sx, st, out, graph = self._graphs[key]
        sx.copy_(x, non_blocking=True)
        if st is not None:
            st.copy_(target, non_blocking=True)
        graph.replay()
        return out

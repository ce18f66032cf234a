"""``finetuning_cgcnn`` -- move a trained decoder to a new task: its graph convolutions frozen, a new classifier head
trained with TensorFlow's Nadam (the reference's ``finetuning_cgcnn``, ``lib_new/models_gcn.py:685-933``, which imports
the trained meta-graph, freezes the conv layers, adds a new FC head and trains it with ``tf.contrib.opt.NadamOptimizer``).

The conv layers are frozen and have no dropout, so the head's input for a window -- the mean over the last conv layer's
filters, ``[n0]`` floats -- is a fixed function of the window.  ``fit`` therefore runs every training and validation
window through the conv stack once (``trunk_features``, the calls ``predict`` makes) and trains the head on that table:
each step is ``train.HeadTrainer``'s head launch(es) plus one ``gcnb_nadam_tf_f32`` launch, one CUDA graph, fed by
``train.InputPipeline``.  ``predict``, ``evaluate``, ``saliency``, ``state_dict_tf`` and the checkpoint functions are
``cgcnn``'s: a saved fine-tuned model loads into a plain ``cgcnn`` built with the same arguments.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import checkpoints, ops
from .models import cgcnn


def _pretrained_variables(pretrained, names):
    """``{name: ndarray}`` of the variables ``names`` of a ``cgcnn``, a ``save_checkpoint`` ``.npz`` file or a TensorFlow
    V2 checkpoint prefix."""
    if isinstance(pretrained, cgcnn):
        found = pretrained.state_dict_tf()
    elif isinstance(pretrained, (str, os.PathLike)):
        path = os.fspath(pretrained)
        if os.path.exists(path + ".index"):
            from . import tf_bundle

            return tf_bundle.read_tf_checkpoint(path, names=names)
        with np.load(path) as z:
            found = {k.replace("__", "/"): z[k] for k in z.files}
    else:
        raise TypeError("pretrained must be a cgcnn, a .npz checkpoint or a TF checkpoint prefix, not %s"
                        % type(pretrained).__name__)
    missing = [n for n in names if n not in found]
    if missing:
        raise ValueError("pretrained model has no variable %s (has: %s)" % (", ".join(missing), ", ".join(found)))
    return {n: found[n] for n in names}


class finetuning_cgcnn(cgcnn):
    """A ``cgcnn`` whose conv layers come from a trained model and stay fixed; only the new head ``M`` is trained.

    Takes ``cgcnn``'s constructor (``M`` = the new head's widths, its last entry the new task's class count) and the
    required keyword ``pretrained``: a ``cgcnn`` with the same conv layers, a file written by
    ``checkpoints.save_checkpoint`` or the prefix of a TensorFlow V2 checkpoint.  Its ``conv{i}/weights`` and
    ``conv{i}/bias`` are copied (``requires_grad=False``); FC variables in it are ignored, the head is initialised from
    ``seed`` as ``cgcnn`` does.  ``L`` must be the original Laplacian list (``cgcnn`` keeps only the levels it uses, so
    ``pretrained.L`` would be selected again wrongly when pooling): splat in the ``params`` of
    ``configs.build_chebyshev_graph_cnn`` with a new ``M``."""

    def __init__(self, *args, pretrained, **kwargs):
        super().__init__(*args, **kwargs)
        names = ["conv%d/%s" % (i + 1, v) for i in range(len(self.p)) for v in ("weights", "bias")]
        found = _pretrained_variables(pretrained, names)
        with torch.no_grad():
            for i in range(len(self.p)):
                for name, param in (("conv%d/weights" % (i + 1), self.conv_weights[i]),
                                    ("conv%d/bias" % (i + 1), self.conv_bias[i])):
                    a = np.asarray(found[name], np.float32)
                    if tuple(a.shape) != tuple(param.shape):
                        raise ValueError("%s: pretrained shape %s does not match %s" % (name, a.shape, tuple(param.shape)))
                    param.copy_(torch.from_numpy(a).to(param.device))
                    param.requires_grad_(False)

    @torch.no_grad()
    def trunk_features(self, data, gather=None, padded=False):
        """The head's input for every window of ``data``: ``mean_f_fwd(conv_stack(batch))`` over ``predict``'s batches,
        ``[n, n0]`` float32 -- bit for bit what ``predict`` and ``forward`` feed the head.  ``gather`` follows
        ``forward``.  ``padded=True`` also returns the rows of the zero windows that pad the last batch
        (``ceil(n / batch_size) * batch_size`` rows), what ``evaluate_features`` takes."""
        M0 = self.L[0].shape[0]
        if gather is None:
            if self.perm is not None and self.n_input_vertices == M0:
                raise ValueError("finetuning_cgcnn.trunk_features: with perm set and n_input_vertices == M_0 say "
                                 "gather=True (raw windows) or gather=False (already permuted) -- the shapes are identical")
            gather = self.perm is not None and data.shape[1] == self.n_input_vertices != M0
        size, bs = data.shape[0], self.batch_size
        table = np.empty((-(-size // bs) * bs, self.fc_weights[0].shape[0]), np.float32)
        for begin in range(0, size, bs):
            h = self.conv_stack(self._padded_batch(data, begin), gather=gather)
            table[begin:begin + bs] = ops.mean_f_fwd(h).cpu().numpy()
        return table if padded else table[:size]

    @torch.no_grad()
    def evaluate_features(self, table, labels):
        """``evaluate(data, labels)`` from ``table = trunk_features(data, padded=True)``: the same FC calls on the same
        batches, so the same ``(summary string, accuracy %, weighted F1 %, loss)``."""
        size, bs = len(labels), self.batch_size
        if table.shape[0] != -(-size // bs) * bs:
            raise ValueError("evaluate_features: %d rows for %d labels -- pass trunk_features(data, padded=True)"
                             % (table.shape[0], size))
        logits_at = lambda begin: self._head(torch.as_tensor(table[begin:begin + bs], device=self.dev))
        predictions, loss = self._predict(size, logits_at, labels, False)
        string, accuracy, f1 = checkpoints.classification_summary(labels, predictions, loss)
        return string, accuracy, f1, loss

    def fit(self, train_data, train_labels, val_data, val_labels, best_checkpoint_dir=None, trainer=None):
        """``cgcnn.fit``'s signature, prints and ``(accuracies, losses, t_step)``, training the head only: the trunk
        features of both sets are computed once, the steps draw the batches ``cgcnn.fit`` draws (NumPy's global
        generator) from the training table and run ``train.HeadTrainer`` (CUDA only), the validation set is evaluated
        from its table (``evaluate_features``) and the three best checkpoints of the whole model are kept."""
        from . import train

        if trainer is None and self.dev.type != "cuda":
            raise ValueError("finetuning_cgcnn.fit: fine-tuning runs on CUDA only (device is %s)" % self.dev)
        features = self.trunk_features(train_data)
        val_table = self.trunk_features(val_data, padded=True)
        if trainer is None:
            trainer = train.HeadTrainer(self)
        return self._fit(features, train_labels, lambda: self.evaluate_features(val_table, val_labels),
                         best_checkpoint_dir, trainer)

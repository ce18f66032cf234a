"""``model_perf`` -- the reference's experiment harness around a model (``/root/reference/lib_new/models_gcn.py:936-1075``,
used by ``HCP_task_fmri_gcn_test8.py:1741-1821, 1900-2002``): ``test`` trains and evaluates a model and keeps the figures
per experiment name; ``predict`` restores the newest checkpoint of a run and reports on a data set.  Host code
(SURVEY.md 8f row 4); the arithmetic is ``cgcnn.fit`` / ``evaluate`` / ``predict``.

Difference from the reference: TensorFlow rebuilds the network from the ``.meta`` graph next to the checkpoint; here the
caller passes the ``cgcnn`` whose architecture the checkpoint has (``model=``).
"""
from __future__ import annotations

import os
import sys

import numpy as np

from . import checkpoints
from .train import data_parallel


def _checkpoint_of_run(ckp_path):
    """The checkpoint ``model_perf.predict`` restores.  With TensorFlow's ``checkpoint`` state file in ``<ckp_path>/model/``:
    literally what the reference reads (models_gcn.py:968-970) -- the file's SECOND line, i.e. the first
    ``all_model_checkpoint_paths`` entry; ``BestCheckpointSaver`` re-registers its kept checkpoints best first before every
    save (checkmat.py:95-100), so that entry is the best one by validation accuracy.  (First line when the file has only
    one.)  Without a state file: the best of a ``BestCheckpoints`` index, else the highest step."""
    d = os.path.join(str(ckp_path), "model")
    state = os.path.join(d, "checkpoint")
    if os.path.exists(state):
        with open(state) as f:
            lines = [line.rstrip("\n") for line in f if line.strip()]
        line = lines[1] if len(lines) > 1 else lines[0]
        return os.path.join(d, line.replace('"', "").split(" ")[-1].split("/")[-1])
    best = checkpoints.BestCheckpoints(d).best() if os.path.exists(os.path.join(d, checkpoints.INDEX_NAME)) else None
    found = best or checkpoints.latest_checkpoint(d, "best.ckpt") or checkpoints.latest_checkpoint(d, "model")
    if found is None:
        raise FileNotFoundError("no checkpoint under %s" % d)
    return found


class model_perf(object):
    """Figures of a series of experiments, keyed by experiment name (same attributes as the reference's class)."""

    def __init__(s):
        s.names, s.params = set(), {}
        s.fit_accuracies, s.fit_losses, s.fit_time = {}, {}, {}
        s.train_accuracy, s.train_f1, s.train_loss = {}, {}, {}
        s.test_accuracy, s.test_f1, s.test_loss = {}, {}, {}

    def test(s, model, name, params, train_data, train_labels, val_data, val_labels, test_data, test_labels,
             target_name=None):
        """Train ``model``, then evaluate it on the training and the test set (models_gcn.py:944-958).  Under a process
        group every rank trains its shards and gets the same figures; rank 0 prints."""
        say = print if data_parallel()[0] == 0 else (lambda *a, **k: None)   # under a process group: rank 0 prints
        s.params[name] = params
        s.fit_accuracies[name], s.fit_losses[name], s.fit_time[name] = model.fit(train_data, train_labels, val_data, val_labels)
        string, s.train_accuracy[name], s.train_f1[name], s.train_loss[name] = model.evaluate(
            train_data, train_labels, target_name=target_name)
        say("\ntrain {}\n".format(string))
        string, s.test_accuracy[name], s.test_f1[name], s.test_loss[name] = model.evaluate(
            test_data, test_labels, target_name=target_name)
        say("\ntest  {}\n".format(string))
        sys.stdout.flush()
        s.names.add(name)
        return s

    def predict(s, ckp_path, test_data, test_labels, target_name=None, batch_size=128, trial_dura=17, flag_starttr=False,
                sub_name=None, model=None):
        """Restore the newest checkpoint under ``<ckp_path>/model/`` into ``model`` and predict ``test_data`` in zero-padded
        batches of ``batch_size`` (models_gcn.py:960-1037).  Prints the per-class report, the confusion matrix and the
        summary line; returns ``(logits, predictions, loss, accuracy figures)`` as the reference does (``loss`` is the sum
        of the batch losses, as there; ``logits`` is the full ``[size, n_classes]`` array -- the reference flattens and
        crops it to ``size`` values, :1019, which no caller uses):
        ``[accuracy]``, or with ``sub_name`` the per-subject weighted F1 table ``[n_subjects, n_classes + 1]`` (last column:
        all classes; :1039-1057, without the CSV side effect), or with ``flag_starttr`` the accuracy per class and time point
        ``[n_classes, trial_dura]`` (:1066-1075)."""
        if model is None:
            raise ValueError("model_perf.predict needs model=<cgcnn with the checkpoint's architecture> "
                             "(there is no TensorFlow meta-graph to rebuild it from)")
        ckpt = _checkpoint_of_run(ckp_path)
        print(ckpt)
        checkpoints.load_checkpoint(model, ckpt)
        keep_bs, model.batch_size = model.batch_size, int(batch_size)
        try:
            pred_labels, pred_loss, pred_logits = model.predict(test_data, test_labels, return_logits=True)
        finally:
            model.batch_size = keep_bs
        # model_perf.predict reports the plain SUM of the batch losses (models_gcn.py:1016), not base_model.predict's
        # sum * batch_size / size (:69)
        test_labels = np.asarray(test_labels)
        pred_loss = pred_loss * len(test_labels) / int(batch_size)
        if target_name is not None:
            print(checkpoints.classification_report(test_labels, pred_labels, target_name)[0])
            print("Confusion Matrix:")
            print(checkpoints.confusion_matrix(test_labels, pred_labels, len(target_name)))
        string, accuracy, f1 = checkpoints.classification_summary(test_labels, pred_labels, pred_loss)
        print(string)
        test_acc = [accuracy]
        sys.stdout.flush()
        n_classes = len(target_name) if target_name is not None else int(model.M[-1])
        if sub_name is not None:
            n_sub = len(sub_name)
            used = pred_labels.shape[0] // n_sub * n_sub
            y_pred = pred_labels[:used].reshape(n_sub, -1)
            y_label = test_labels[:used].reshape(n_sub, -1)
            test_acc = np.zeros((n_sub, n_classes + 1))
            for si in range(n_sub):
                for li in range(n_classes):
                    mask = y_label[si] == li
                    test_acc[si, li] = checkpoints.classification_summary(y_label[si, mask], y_pred[si, mask])[2] / 100.0
                test_acc[si, -1] = checkpoints.classification_summary(y_label[si], y_pred[si])[2] / 100.0
        if flag_starttr:
            y_pred = pred_labels.reshape(-1, trial_dura)
            y_label = test_labels.reshape(-1, trial_dura)
            test_acc = np.zeros((n_classes, trial_dura))
            for li in range(n_classes):
                for ti in range(trial_dura):
                    mask = y_label[:, ti] == li
                    test_acc[li, ti] = 100.0 * float((y_pred[mask, ti] == li).mean()) if mask.any() else 0.0
        return pred_logits, pred_labels, pred_loss, test_acc

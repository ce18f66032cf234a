"""Fine-tuning speed at config 2 (360 ROIs x 15 TRs -> 400 -> 100 -> 25 vertices, 32 filters, K = 5), B = 512, new head
25-512-256-7, dropout keep 0.5:
  * the trunk pass (``mean_f_fwd(conv_stack(batch))`` under no_grad, what ``finetuning_cgcnn.trunk_features`` runs per
    batch) in windows/s, over a ring of device inputs larger than the 126 MB L2, and ``trunk_features`` on host windows
    (with the copies to and from the device);
  * the ``train.HeadTrainer`` step (head + TF Nadam) as a CUDA graph reading bound inputs, in ms/step and windows/s;
  * for comparison, a step that recomputes the frozen trunk every time (the same trunk forward, then the same head step)
    -- the cost the cached features remove.
The outputs are checked first: the ring's trunk pass against ``trunk_features``, and a few cached-feature steps against
the same steps on recomputed features (bit for bit).  Every timed region is warmed up and timed with CUDA events.

    python tools/time_finetune.py [--steps 24]
"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from gcn_fmri_decoding_b200 import ops, synth
from gcn_fmri_decoding_b200.models import cgcnn, finetuning_cgcnn
from gcn_fmri_decoding_b200.train import HeadTrainer


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def events(fn, n, reps=3):
    """Mean ms of fn(i) over reps passes of i = 0..n-1, after one warm pass."""
    for i in range(n):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        for i in range(n):
            fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / (reps * n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=24, help="inputs in the ring (each 11 MB at B = 512)")
    ap.add_argument("--batch", type=int, default=512)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    B, n = args.batch, max(args.steps, 12)
    A, gs, perm, L = synth.brain_graph(4)
    kw = dict(L=L, F=[32, 32], K=[5, 5], p=[4, 4], channel=15, device=dev, seed=1, perm=perm, n_input_vertices=360,
              batch_size=B, regularization=5e-4, dropout=0.5)
    base = cgcnn(M=[512, 256, 22], **kw)

    def make():
        return finetuning_cgcnn(M=[512, 256, 7], pretrained=base, **kw)

    model = make()
    host = [synth.bold_windows(B, seed=100 + i) for i in range(n)]
    ring = [torch.as_tensor(h, device=dev) for h in host]
    ring_mb = n * ring[0].numel() * 4 / 2 ** 20
    labels = [torch.as_tensor(np.random.RandomState(i).randint(0, 7, B), device=dev) for i in range(n)]

    def trunk(i):
        with torch.no_grad():
            return ops.mean_f_fwd(model.conv_stack(ring[i], gather=True))

    # outputs first: the ring's trunk pass is trunk_features, and cached-feature steps equal recomputed-feature steps
    table = model.trunk_features(np.concatenate(host))
    feats = [torch.as_tensor(table[i * B:(i + 1) * B], device=dev) for i in range(n)]
    for i in range(n):
        if not torch.equal(trunk(i), feats[i]):
            sys.exit("the trunk pass on input %d differs from trunk_features" % i)
    cached, recomputed = HeadTrainer(model), HeadTrainer(make())
    a0 = torch.empty(B, 25, device=dev)
    for i in range(n):
        cached.bind_inputs(feats[i], labels[i])
        recomputed.bind_inputs(a0, labels[i])
    for i in range(3):
        lc, _ = cached.step(feats[i], labels[i])
        a0.copy_(trunk(i))
        lr, _ = recomputed.step(a0, labels[i])
        if float(lc) != float(lr):
            sys.exit("step %d: loss %r on cached features, %r on recomputed ones" % (i, float(lc), float(lr)))
    if not torch.equal(cached.flat_p, recomputed.flat_p):
        sys.exit("cached-feature and recomputed-feature steps reached different weights")

    def recompute_step(i):
        a0.copy_(trunk(i))
        recomputed.step(a0, labels[i])

    t_trunk = events(trunk, n)
    t_step = events(lambda i: cached.step(feats[i], labels[i]), n, reps=20)
    t_recompute = events(recompute_step, n)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.trunk_features(np.concatenate(host))
    torch.cuda.synchronize()
    t_host = (time.perf_counter() - t0) * 1e3 / n
    name, power = card()
    print("card: %s, power limit %s" % (name, power))
    print("config 2, B = %d, head 25-512-256-7, keep 0.5, ring of %d inputs (%.0f MB); outputs agree bit for bit"
          % (B, n, ring_mb))
    print("trunk pass (device inputs): %.3f ms/batch = %.0f windows/s" % (t_trunk, B / t_trunk * 1e3))
    print("trunk_features (host windows, with copies): %.3f ms/batch = %.0f windows/s" % (t_host, B / t_host * 1e3))
    print("HeadTrainer step (CUDA graph, bound inputs): %.4f ms/step = %.0f windows/s" % (t_step, B / t_step * 1e3))
    print("step recomputing the frozen trunk (trunk forward + the same head step): %.4f ms/step = %.0f windows/s"
          % (t_recompute, B / t_recompute * 1e3))


if __name__ == "__main__":
    main()

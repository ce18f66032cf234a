"""Windows/s of gradient saliency maps at config 2 (360 ROIs x 15 TRs -> 400 -> 100 -> 25 vertices, 32 filters, K = 5,
head 512-256-22), B = 512: saliency.InputGradient (one CUDA graph per batch) against the autograd path
(torch.autograd.grad through cgcnn.forward) on the same inputs.  The inputs are a ring larger than the 126 MB L2; every
timed region is warmed up first and measured with CUDA events.  The two paths' outputs are checked against each other
before any rate is printed.  Also prints the per-launch time of conv 1's input gradient: the tcgen05 adjoint launch
(ops.cheb_dx) next to the backward the autograd path runs for that layer (ops.cheb_bwd with dx, the route the library
names).

    python tools/time_saliency.py [--steps 20]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from gcn_fmri_decoding_b200 import _lib, ops, synth
from gcn_fmri_decoding_b200.models import cgcnn
from gcn_fmri_decoding_b200.saliency import InputGradient


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
    ap.add_argument("--steps", type=int, default=20, help="inputs in the ring (each 11 MB at B = 512)")
    ap.add_argument("--batch", type=int, default=512)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    B, n = args.batch, max(args.steps, 12)
    A, gs, perm, L = synth.brain_graph(4)
    model = cgcnn(L=L, F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device=dev, seed=1, perm=perm,
                  n_input_vertices=360, batch_size=B)
    ring = [torch.as_tensor(synth.bold_windows(B, seed=100 + i), device=dev) for i in range(n)]
    ring_mb = n * ring[0].numel() * 4 / 2 ** 20
    ig = InputGradient(model)

    def autograd(i):
        x = ring[i].clone().requires_grad_(True)
        logits = model(x, gather=True)
        t = logits.argmax(1)
        return torch.autograd.grad(logits.gather(1, t.view(-1, 1)).sum(), x)[0], t

    # outputs first: both paths on the same inputs
    worst = 0.0
    for i in range(3):
        g, _, t = ig(ring[i], gather=True)
        ga, ta = autograd(i)
        if not torch.equal(t, ta):
            sys.exit("targets differ between InputGradient and autograd on input %d" % i)
        worst = max(worst, float((g - ga).abs().max() / ga.abs().max()))
    if worst > 1e-5:
        sys.exit("InputGradient and autograd disagree: max rel err %.2e" % worst)
    t_ig = events(lambda i: ig(ring[i], gather=True), n)
    t_ag = events(autograd, n)
    # conv 1's input gradient alone: the adjoint launch vs the backward autograd runs for the layer
    pl = model._plan(model.L[0])
    permt, W, b = model.perm, model.conv_weights[0], model.conv_bias[0]
    fw = [ops.cheb_fwd(ring[i], permt, *pl.tensors(), W, b, 5, 4, 1, True, True, model.algo) for i in range(n)]
    dys = [torch.randn_like(fw[i][0]) for i in range(n)]
    t_dx = events(lambda i: ops.cheb_dx(ring[i], permt, 360, fw[i][0], fw[i][1], dys[i], False, *pl.tensors(), W, 5, 4,
                                        True, model.algo), n)
    t_bwd = events(lambda i: torch.ops.gcn_b200.cheb_bwd(ring[i], permt, fw[i][0], fw[i][1], dys[i], *pl.tensors(), W, 5, 4,
                                                         1, True, True, model.algo), n)
    name, power = card()
    print("card: %s, power limit %s" % (name, power))
    print("config 2, B = %d, ring of %d inputs (%.0f MB), outputs agree to %.1e" % (B, n, ring_mb, worst))
    print("InputGradient (CUDA graph): %.3f ms/batch = %.0f windows/s" % (t_ig, B / t_ig * 1e3))
    print("autograd through cgcnn.forward: %.3f ms/batch = %.0f windows/s" % (t_ag, B / t_ag * 1e3))
    print("conv 1 input gradient: %s  %.1f us" % (_lib.describe_dx(B, pl.M, pl.nnz, 15, 32, 5, 4)[0].split(",")[0],
                                                  t_dx * 1e3))
    print("conv 1 full backward with dx (autograd's): %s  %.1f us" % (
        _lib.describe(B, pl.M, pl.nnz, 15, 32, 5, 4, True, True, False)[0].split(":")[0], t_bwd * 1e3))


if __name__ == "__main__":
    main()

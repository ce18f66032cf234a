"""Edge saliency maps: time per batch of saliency.GraphGradient (one CUDA graph per batch) next to saliency.InputGradient
in the same run, at config 2 (360 ROIs x 15 TRs -> 400 -> 100 vertices, 32 filters, K = 5, head 512-256-22, B = 512)
and config 1 (six 32-filter K = 5 layers on the 372-vertex graph, p = 1, B = 128); then the time per launch of
k_sddmm_tma for each conv layer (torch.profiler over graph replays, a run of its own), its algorithmic bytes and the
resulting rate.  Inputs are a ring larger than the 126 MB L2; every timed region is warmed up first and measured with
CUDA events.  GraphGradient's eager and replayed outputs are compared before any time is printed.

Bytes of one k_sddmm_tma launch (layer of M vertices, nnz stored entries, B windows, Fin features, order K):
  gathered  (K-1) * 4 * B * Fin * (nnz + M + groups)   every entry's X_{k-1} row chunk and, once per group of 8
                                                        entries, b_k[i]: what the kernel moves from L2 to the SMs
  distinct  2 * (K-1) * 4 * M * B * Fin                 each stack slab it reads, once (the HBM lower bound)
  written   4 * B * (nnz + M)                           (read too where a layer accumulates)

    python tools/time_graph_saliency.py [--steps 20]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from gcn_fmri_decoding_b200 import synth
from gcn_fmri_decoding_b200.models import cgcnn
from gcn_fmri_decoding_b200.saliency import GraphGradient, InputGradient


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


def sddmm_bytes(plan, B, Fin, K, accumulate):
    rp = plan._host[False][0]
    deg = np.diff(rp)
    groups = int(((deg + 1 + 7) // 8).sum())
    gathered = (K - 1) * 4 * B * Fin * (plan.nnz + plan.M + groups)
    distinct = 2 * (K - 1) * 4 * plan.M * B * Fin
    written = 4 * B * (plan.nnz + plan.M) * (2 if accumulate else 1)
    return gathered, distinct, written


def model_for(cfg, B, dev):
    if cfg == "config2":
        A, gs, perm, L = synth.brain_graph(4)
        return cgcnn(L=L, F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device=dev, seed=1, perm=perm,
                     n_input_vertices=360, batch_size=B)
    A, gs, perm, L = synth.brain_graph(1)
    return cgcnn(L=L, F=[32] * 6, K=[5] * 6, p=[1] * 6, M=[512, 256, 22], channel=15, brelu="b2relu", device=dev, seed=1,
                 perm=perm, n_input_vertices=360, batch_size=B)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="inputs in the ring")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    name, power = card()
    print("card: %s, power limit %s" % (name, power))
    for cfg, B in (("config2", 512), ("config1", 128)):
        model = model_for(cfg, B, dev)
        n = max(args.steps, 12) * (512 // B)
        ring = [torch.as_tensor(synth.bold_windows(B, seed=100 + i), device=dev) for i in range(n)]
        ring_mb = n * ring[0].numel() * 4 / 2 ** 20
        gg, ig = GraphGradient(model), InputGradient(model)
        eager = GraphGradient(model, use_cuda_graph=False)(ring[0], gather=True)[0]
        replay = gg(ring[0], gather=True)[0]
        for k in eager:
            if not torch.equal(eager[k], replay[k]):
                sys.exit("%s: GraphGradient replay differs from the eager schedule" % cfg)
        t_gg = events(lambda i: gg(ring[i], gather=True), n)
        t_ga = events(lambda i: gg(ring[i], gather=True, absolute=True), n)
        t_ig = events(lambda i: ig(ring[i], gather=True), n)
        print("%s, B = %d, ring of %d inputs (%.0f MB)" % (cfg, B, n, ring_mb))
        print("  GraphGradient (CUDA graph): %.3f ms/batch = %.0f windows/s; absolute: %.3f ms/batch" % (
            t_gg, B / t_gg * 1e3, t_ga))
        print("  InputGradient (CUDA graph): %.3f ms/batch = %.0f windows/s" % (t_ig, B / t_ig * 1e3))
        # k_sddmm_tma per launch: kernels of a few replays, the i-th launch of a replay serving conv layer nconv-1-i
        nconv, reps = len(model.p), 10
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for i in range(reps):
                gg(ring[i], gather=True)
            torch.cuda.synchronize()
        ks = sorted((e for e in prof.events() if "k_sddmm_tma" in e.name), key=lambda e: e.time_range.start)
        if len(ks) != reps * nconv:
            sys.exit("%s: expected %d k_sddmm_tma launches, the profile has %d" % (cfg, reps * nconv, len(ks)))
        seen = set()
        for layer in range(nconv - 1, -1, -1):
            pos = nconv - 1 - layer
            us = float(np.mean([ks[r * nconv + pos].time_range.elapsed_us() for r in range(reps)]))
            pl = model._plan(model.L[layer])
            lvl = model._graph_levels[layer]
            Fin = 15 if layer == 0 else model.F[layer - 1]
            g, d, w = sddmm_bytes(pl, B, Fin, model.K[layer], accumulate=lvl in seen)
            seen.add(lvl)
            print("  k_sddmm_tma conv %d (M = %d, nnz = %d, Fin = %d): %.1f us; gathered %.1f MB -> %.0f GB/s, distinct "
                  "%.1f MB -> %.0f GB/s, written %.2f MB" % (layer + 1, pl.M, pl.nnz, Fin, us, g / 1e6, g / us / 1e3,
                                                             d / 1e6, d / us / 1e3, w / 1e6))


if __name__ == "__main__":
    main()

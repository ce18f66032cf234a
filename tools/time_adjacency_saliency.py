"""Edge saliency maps w.r.t. the adjacency: time per batch of saliency.AdjacencyGradient (one CUDA graph per batch) next
to saliency.GraphGradient in the same run, at config 2 (360 ROIs x 15 TRs -> 400 -> 100 vertices, 32 filters, K = 5,
head 512-256-22, B = 512) and config 1 (six 32-filter K = 5 layers on the 372-vertex graph, p = 1, B = 128).  Inputs are
a ring larger than the 126 MB L2; every timed region is warmed up first and measured with CUDA events, the two schedules
alternating pass by pass.  AdjacencyGradient's eager and replayed outputs are compared before any time is printed.

With --profile (a run of its own: tracing slows the host) the time per launch of the chain's kernels instead, from
torch.profiler over graph replays, with their algorithmic bytes:
  k_adjacency_level  per level: reads G twice (its row and its column sums, 8 B per entry each with the value) and
                     once more for the entry pass with ss, tpos and parent (16 B), writes T_l (4 B), reads T_{l+1} at
                     the parent entries (4 B): about 40 * B * nnz bytes
  k_adjacency_edges  reads two T_0 entries and the edge pair (8 B + 8 B per edge and window), writes 4 B

    python tools/time_adjacency_saliency.py [--steps 20] [--profile]
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
from gcn_fmri_decoding_b200.saliency import AdjacencyGradient, AdjacencyMaps, GraphGradient


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def model_for(cfg, B, dev):
    if cfg == "config2":
        A, gs, perm, L = synth.brain_graph(4)
        return A, cgcnn(L=L, F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device=dev, seed=1,
                        perm=perm, n_input_vertices=360, batch_size=B)
    A, gs, perm, L = synth.brain_graph(1)
    return A, cgcnn(L=L, F=[32] * 6, K=[5] * 6, p=[1] * 6, M=[512, 256, 22], channel=15, brelu="b2relu", device=dev,
                    seed=1, perm=perm, n_input_vertices=360, batch_size=B)


def alternate(fns, n, reps=3):
    """Mean ms per call of each fn(i), i = 0..n-1, after one warm pass; the functions take turns pass by pass."""
    for fn in fns:
        for i in range(n):
            fn(i)
    torch.cuda.synchronize()
    total = [0.0] * len(fns)
    for _ in range(reps):
        for k, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n):
                fn(i)
            b.record()
            torch.cuda.synchronize()
            total[k] += a.elapsed_time(b)
    return [t / (reps * n) for t in total]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="inputs in the ring")
    ap.add_argument("--profile", action="store_true", help="time the chain's kernels with torch.profiler instead")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    name, power = card()
    print("card: %s, power limit %s" % (name, power))
    for cfg, B in (("config2", 512), ("config1", 128)):
        A, model = model_for(cfg, B, dev)
        maps = AdjacencyMaps(model, A)
        n = max(args.steps, 12) * (512 // B)
        ring = [torch.as_tensor(synth.bold_windows(B, seed=100 + i), device=dev) for i in range(n)]
        ring_mb = n * ring[0].numel() * 4 / 2 ** 20
        ag, gg = AdjacencyGradient(model, maps), GraphGradient(model)
        eager = AdjacencyGradient(model, maps, use_cuda_graph=False)(ring[0], gather=True)[0]
        if not torch.equal(eager, ag(ring[0], gather=True)[0]):
            sys.exit("%s: AdjacencyGradient replay differs from the eager schedule" % cfg)
        print("%s, B = %d, ring of %d inputs (%.0f MB), %d edges" % (cfg, B, n, ring_mb, len(maps.rows)))
        if not args.profile:
            for absolute in (False, True):
                t_ag, t_gg = alternate([lambda i: ag(ring[i], gather=True, absolute=absolute),
                                        lambda i: gg(ring[i], gather=True, absolute=absolute)], n)
                print("  absolute=%d: AdjacencyGradient %.3f ms/batch (%.0f windows/s), GraphGradient %.3f ms/batch: "
                      "%+.1f%%" % (absolute, t_ag, B / t_ag * 1e3, t_gg, 100 * (t_ag / t_gg - 1)))
            continue
        reps = 10
        for i in range(reps):
            ag(ring[i], gather=True)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for i in range(reps):
                ag(ring[i], gather=True)
            torch.cuda.synchronize()
        kern = list(prof.events())  # device activity only (CUDA activities)
        levels = [model._plan(model.L[model._graph_levels.index(lv)]) for lv in maps.levels]
        lv_us = sorted((e for e in kern if "k_adjacency_level" in e.name), key=lambda e: e.time_range.start)
        ed_us = [e.time_range.elapsed_us() for e in kern if "k_adjacency_edges" in e.name]
        if len(lv_us) != reps * len(levels) or len(ed_us) != reps:
            sys.exit("%s: expected %d k_adjacency_level and %d k_adjacency_edges launches, the profile has %d and %d" % (
                cfg, reps * len(levels), reps, len(lv_us), len(ed_us)))
        for pos, pl in enumerate(reversed(levels)):  # launched from the coarsest level down
            us = float(np.mean([lv_us[r * len(levels) + pos].time_range.elapsed_us() for r in range(reps)]))
            nbytes = 40 * B * pl.nnz
            print("  k_adjacency_level (M = %d, nnz = %d): %.1f us, %.1f MB -> %.0f GB/s" % (
                pl.M, pl.nnz, us, nbytes / 1e6, nbytes / us / 1e3))
        E = len(maps.rows)
        us = float(np.mean(ed_us))
        print("  k_adjacency_edges (E = %d): %.1f us, %.1f MB -> %.0f GB/s" % (E, us, 20 * B * E / 1e6,
                                                                           20 * B * E / us / 1e3))


if __name__ == "__main__":
    main()

"""Group saliency maps: time per batch of the grouped schedules next to the ungrouped ones in the same run, at config 2
(360 ROIs x 15 TRs -> 400 -> 100 vertices, 32 filters, K = 5, head 512-256-22, B = 512) and config 1 (six 32-filter
K = 5 layers on the 372-vertex graph, p = 1, B = 128): InputGradient and GraphGradient ungrouped, grouped by target,
and in 4 groups with capacity n_groups = B and n_groups = 4.  Inputs are a ring larger than the 126 MB L2; every timed
region is warmed up first and measured with CUDA events, the schedules alternating pass by pass.  Then cgcnn.saliency
end to end over 32 768 host windows, per-window against groups=labels (host clock; the call ends in its device-to-host
copies).

With --profile (a run of its own: tracing slows the host) the time per launch of k_group_colsum instead, from
torch.profiler over graph replays of InputGradient with 4 groups at capacity B, with its algorithmic bytes
rows x cols x 4 (each element of the per-window maps read once; the [n_groups, cols] output is small next to it).

    python tools/time_group_saliency.py [--steps 20] [--profile]
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from gcn_fmri_decoding_b200 import synth
from gcn_fmri_decoding_b200.saliency import GraphGradient, InputGradient
from time_adjacency_saliency import alternate, card, model_for


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="inputs in the ring")
    ap.add_argument("--profile", action="store_true", help="time k_group_colsum with torch.profiler instead")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    name, power = card()
    print("card: %s, power limit %s" % (name, power))
    for cfg, B in (("config2", 512), ("config1", 128)):
        _, model = model_for(cfg, B, dev)
        n = max(args.steps, 12) * (512 // B)
        ring = [torch.as_tensor(synth.bold_windows(B, seed=100 + i), device=dev) for i in range(n)]
        g4 = torch.as_tensor(np.random.RandomState(0).randint(0, 4, B).astype(np.int32), device=dev)
        ig, gg = InputGradient(model), GraphGradient(model)
        cap = ig(ring[0], gather=True, group=g4)[0][:4].clone()
        if not torch.equal(cap, ig(ring[0], gather=True, group=g4, n_groups=4)[0]):
            sys.exit("%s: the sums at capacity %d differ from those at n_groups = 4" % (cfg, B))
        print("%s, B = %d, ring of %d inputs (%.0f MB)" % (cfg, B, n, n * ring[0].numel() * 4 / 2 ** 20))
        if args.profile:
            reps = 10
            for i in range(reps):
                ig(ring[i], gather=True, group=g4)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for i in range(reps):
                    ig(ring[i], gather=True, group=g4)
                torch.cuda.synchronize()
            us = [e.time_range.elapsed_us() for e in prof.events() if "k_group_colsum" in e.name]
            if len(us) != reps:
                sys.exit("%s: expected %d k_group_colsum launches, the profile has %d" % (cfg, reps, len(us)))
            nbytes = ring[0].numel() * 4
            print("  k_group_colsum (rows = %d, cols = %d): %.1f us, %.1f MB -> %.0f GB/s" % (
                B, ring[0][0].numel(), float(np.mean(us)), nbytes / 1e6, nbytes / float(np.mean(us)) / 1e3))
            continue
        for label, cls in (("InputGradient", ig), ("GraphGradient", gg)):
            t = alternate([lambda i: cls(ring[i], gather=True),
                           lambda i: cls(ring[i], gather=True, group="target"),
                           lambda i: cls(ring[i], gather=True, group=g4),
                           lambda i: cls(ring[i], gather=True, group=g4, n_groups=4)], n)
            print("  %s: ungrouped %.3f ms/batch, by target %.3f ms (%+.1f%%), 4 groups at capacity %d %.3f ms "
                  "(%+.1f%%), 4 groups at n_groups = 4 %.3f ms (%+.1f%%)" % (
                      label, t[0], t[1], 100 * (t[1] / t[0] - 1), B, t[2], 100 * (t[2] / t[0] - 1), t[3],
                      100 * (t[3] / t[0] - 1)))
    if args.profile:
        return
    _, model = model_for("config2", 512, dev)
    n = 32768
    data = synth.bold_windows(n, seed=7)
    labels = synth.labels(n, seed=7)
    model.saliency(data[:1024])  # capture both graphs
    model.saliency(data[:1024], groups=labels[:1024])
    times = {"per-window": [], "groups=labels": []}
    for _ in range(2):
        for key, kw in (("per-window", {}), ("groups=labels", dict(groups=labels))):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.saliency(data, **kw)
            times[key].append(time.perf_counter() - t0)
    for key, ts in times.items():
        print("cgcnn.saliency over %d host windows (config 2, B = 512), %s: %.3f s (best of %d: %.0f windows/s)" % (
            n, key, min(ts), len(ts), n / min(ts)))


if __name__ == "__main__":
    main()

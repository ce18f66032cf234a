"""``cgcnn.fit`` under data parallelism at config 2 (360 ROIs x 15 TRs -> 400 -> 100 -> 25 vertices, 32 filters, K = 5,
head 25-512-256-22, dropout keep 0.5), 512 windows per GPU (global batch 512 N), from a host training set larger than the
126 MB L2.  For each N it spawns N ranks (NCCL process group, peer-memory gradient exchange) and reports
  * windows/s of the step loop alone: ``train.fit`` without evaluations, from the first step to the last (the input
    pipeline's graphs are captured before the first step and not counted);
  * windows/s of ``cgcnn.fit`` as a user runs it, with its evaluations of the validation set (``eval_frequency`` =
    steps / 4), the best-checkpoint files and the graph captures -- wall time over all steps;
  * the cost of the per-step loss all-reduce ``fit`` makes: one float64 scalar all-reduce plus the host read, mean
    of 200, in ms, next to the mean step time.
The outputs are checked first: after fit the replicas are bit-identical.

    python tools/time_fit_dp.py [--gpus 1 2 4 8] [--steps 48]
"""
import argparse
import os
import socket
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

PER_GPU = 512


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, steps, n_train, out_dir):
    import torch.distributed as dist

    from gcn_fmri_decoding_b200 import synth, train
    from gcn_fmri_decoding_b200.models import cgcnn

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    B = PER_GPU * world
    A, gs, perm, L = synth.brain_graph(4)
    data = synth.bold_windows(n_train, seed=5)                       # the same host set on every rank
    labels = synth.labels(n_train, seed=5)
    val, val_labels = synth.bold_windows(2048, seed=6), synth.labels(2048, seed=6)

    def model():
        return cgcnn(L=L, F=[32, 32], K=[5, 5], p=[4, 4], M=[512, 256, 22], channel=15, device=dev, seed=1, perm=perm,
                     n_input_vertices=360, regularization=5e-4, dropout=0.5, batch_size=B,
                     num_epochs=steps * B / n_train, eval_frequency=max(1, steps // 4))

    # ---- the step loop alone
    m = model()
    tr = train.FusedTrainer(m)
    t = {}
    step = tr.step

    def timed(x, y, dropout=None):
        if "first" not in t:
            torch.cuda.synchronize()
            t["first"] = time.perf_counter()
        return step(x, y, dropout)

    tr.step = timed
    np.random.seed(0)
    history = train.fit(m, data, labels, trainer=tr, seed=None, verbose=False)
    torch.cuda.synchronize()
    loop = time.perf_counter() - t["first"]
    n_loop = len(history)
    every = [torch.empty_like(tr.flat_p) for _ in range(world)]
    dist.all_gather(every, tr.flat_p)
    identical = all(torch.equal(every[0], e) for e in every)
    # ---- cgcnn.fit with its evaluations
    m2 = model()
    np.random.seed(0)
    dist.barrier()
    t0 = time.perf_counter()
    acc, _, _ = m2.fit(data, labels, val, val_labels, best_checkpoint_dir=os.path.join(out_dir, "best%d" % world))
    torch.cuda.synchronize()
    full = time.perf_counter() - t0
    # ---- the per-step loss all-reduce
    x = torch.ones((), dtype=torch.float64, device=dev)
    for _ in range(20):
        dist.all_reduce(x)
        float(x)
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(200):
        y = torch.ones(1, dtype=torch.float64, device=dev)
        dist.all_reduce(y)
        float(y)
    t_ar = (time.perf_counter() - t0) / 200
    if rank == 0:
        torch.save(dict(loop=loop, n_loop=n_loop, full=full, steps=len(history), evals=len(acc), t_ar=t_ar,
                        identical=identical, kind=tr.allreduce_kind, B=B), os.path.join(out_dir, "n%d.pt" % world))
    dist.barrier()
    os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--train-windows", type=int, default=8192, help="host training set (8192 windows = 177 MB)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs CUDA devices"
    import torch.multiprocessing as mp

    name, power = card()
    out_dir = tempfile.mkdtemp()
    mb = args.train_windows * 360 * 15 * 4 / 1e6
    print("card: %s, power limit %s" % (name, power))
    print("config 2, %d windows per GPU, keep 0.5, %d steps, host training set %d windows (%.0f MB)"
          % (PER_GPU, args.steps, args.train_windows, mb))
    for n in args.gpus:
        if n > torch.cuda.device_count():
            print("N = %d: only %d devices, skipped" % (n, torch.cuda.device_count()))
            continue
        mp.spawn(_worker, args=(n, _free_port(), args.steps, args.train_windows, out_dir), nprocs=n, join=True)
        r = torch.load(os.path.join(out_dir, "n%d.pt" % n))
        per_step = r["loop"] / r["n_loop"]
        print("N = %d (global batch %d, %s): step loop %.0f windows/s (%.3f ms/step); cgcnn.fit with %d evaluations "
              "%.0f windows/s; loss all-reduce %.3f ms/step (%.1f %% of a step); replicas identical: %s"
              % (n, r["B"], r["kind"], r["n_loop"] * r["B"] / r["loop"], per_step * 1e3, r["evals"],
                 r["steps"] * r["B"] / r["full"], r["t_ar"] * 1e3, 100.0 * r["t_ar"] / per_step, r["identical"]))
        sys.stdout.flush()


if __name__ == "__main__":
    main()

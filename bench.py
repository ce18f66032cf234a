#!/usr/bin/env python
"""Benchmark of the graph-convolution hot path (BASELINE.json metric: ChebyNet windows/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3a|3a1|3b|5] [--strong]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workloads (BASELINE.json ``configs``; SURVEY.md 8d pins the shapes):
  2   (default; the configuration the metric is quoted on) ChebyNet K=5 training step (forward + backward + Adam),
      2 conv layers F=[32,32] K=[5,5] p=[4,4] on the pinned 360-ROI graph coarsened 4 levels (M=400->100->25), head
      25->512->256->22, 512 windows of [360 ROI x 15 TR] per GPU, fp32.  N>1: weak scaling (N=8 = config 4's global
      batch 4096) -- or, with ``--strong``, config 4 as written: global batch 4096 split over the N GPUs.
  3a  the same step with the ``chebyshev2`` entry at K=2;  3a1: K=1 (the repo's "firstorder");  3b: ``fourier``.
  1   ChebyNet K=5 predict (predict_states path): 6 conv layers F=32 K=5 p=1 b2relu on M=372, head 372-512-256-22,
      batch 128, forward only.
  5   vertex-level ChebyNet K=25 on a 32 492-vertex sphere graph (HBM-resident operator), 15->32, batch 64,
      forward + backward of the layer.

One JSON line on stdout (rank 0).  ``value`` = windows/s with inputs resident in HBM (a ring of distinct batches
larger than 2x L2, so every step reads HBM); ``e2e`` = the same step fed from pinned host memory with the H2D copy and
a D2H read of the result inside the timed region; ``roofline`` = algorithmic bytes (or FLOPs) / CUDA-event time of
the dominant kernel against the measured peak; ``cpu_baseline`` = the NumPy/SciPy oracle of the same step on the
host cores (bounded sample).  ``--impl reference`` times that CPU implementation alone (the reference's TF-1.x stack
cannot be installed; see BASELINE.md section 2).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

REG = 5e-4
MFC = [512, 256, 22]

CONFIGS = {
    "2": dict(kind="train", filter="chebyshev5", K=[5, 5], batch=512,
              metric="ChebyNet K=5 training windows/sec (fwd+bwd+update, 2 conv layers + Graclus mpool, batch 512/GPU)",
              workload="config2: ChebyNet K=5 train step, F=[32,32] K=[5,5] p=[4,4], M=400->100->25, head 25-512-256-22, "
                       "B=512/GPU, 15-TR windows"),
    "3a": dict(kind="train", filter="chebyshev2", K=[2, 2], batch=512,
               metric="1stGCN (chebyshev2, K=2) training windows/sec (fwd+bwd+update, config-2 shape, batch 512/GPU)",
               workload="config3a: chebyshev2 K=2 train step at the config-2 shape (F=[32,32] p=[4,4], M=400->100->25, "
                        "head 25-512-256-22), B=512/GPU"),
    "3a1": dict(kind="train", filter="chebyshev5", K=[1, 1], batch=512,
                metric="first-order ChebyNet (K=1) training windows/sec (fwd+bwd+update, config-2 shape, batch 512/GPU)",
                workload="config3a/K=1: chebyshev5 K=1 ('firstorder', model.py:263) train step at the config-2 shape, B=512/GPU"),
    "3b": dict(kind="train", filter="fourier", K=[0, 0], batch=512,
               metric="spectral GCN (fourier) training windows/sec (fwd+bwd+update, config-2 shape, batch 512/GPU)",
               workload="config3b: fourier (Laplacian eigenbasis) train step at the config-2 shape, B=512/GPU"),
    "1": dict(kind="predict", batch=128,
              metric="ChebyNet K=5 predict windows/sec (6 conv layers M=372 b2relu + head, batch 128, forward)",
              workload="config1: ChebyNet K=5 predict, 6 conv layers F=32 K=5 p=1 b2relu on M=372, head 372-512-256-22, B=128"),
    "5": dict(kind="vertex", batch=64,
              metric="vertex-level ChebyNet K=25 windows/sec (32 492-vertex graph, 15->32, batch 64, layer fwd+bwd)",
              workload="config5: ChebyNet K=25 layer on a 32492-vertex sphere kNN graph (nnz ~1.96e5), 15->32, B=64, "
                       "forward + backward (dx, dW, db)"),
}
F2, P2 = [32, 32], [4, 4]


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ CPU side (oracle port)
CPU_MODE_TEXT = {"pool": "thread pool over window chunks, BLAS pinned to 1 thread per worker",
                 "blas": "one chunk, BLAS on all cores"}


def _cpu_problem(cfg, n_windows):
    """(step(chunk_indices), n_windows, chunk size) of the oracle for this config; data and weights seeded."""
    from gcn_fmri_decoding_b200 import graclus, synth
    from oracle import layers_np as O

    rng = np.random.RandomState(7)
    if cfg["kind"] == "train":
        A, gs, perm, L = synth.brain_graph(4)
        Ls = O.select_laplacians(L, P2)
        params, fin = [], 15
        for li, (f, k, p) in enumerate(zip(F2, cfg["K"], P2)):
            M = Ls[li].shape[0]
            shape = (M, f, fin) if cfg["filter"] == "fourier" else (fin * k, f)
            params.append(dict(W=synth.truncated_normal(rng, shape, 0.2), b=np.full(f, 0.2, np.float32), K=k, p=p))
            fin = f
        fcs, width = [], Ls[-1].shape[0] // P2[-1]
        for m in MFC:
            fcs.append((synth.truncated_normal(rng, (width, m), 0.2), np.full(m, 0.2, np.float32)))
            width = m
        x = graclus.perm_data_3d(synth.bold_windows(n_windows, seed=2024), perm).astype(np.float32)
        lab = synth.labels(n_windows)
        return (lambda c: O.network_step(x[c], lab[c], Ls, params, fcs, REG, filter=cfg["filter"], dtype=np.float32)), 32
    if cfg["kind"] == "predict":
        A, gs, perm, L = synth.brain_graph(1)
        Ls = [L[0]] * 6
        params, fin = [], 15
        for _ in range(6):
            params.append(dict(W=synth.truncated_normal(rng, (fin * 5, 32), 0.2), b=np.full((372, 32), 0.2, np.float32), K=5, p=1))
            fin = 32
        fcs, width = [], 372
        for m in MFC:
            fcs.append((synth.truncated_normal(rng, (width, m), 0.2), np.full(m, 0.2, np.float32)))
            width = m
        x = graclus.perm_data_3d(synth.bold_windows(n_windows, seed=30), perm).astype(np.float32)
        return (lambda c: O.head(O.conv_stack(x[c], Ls, params, brelu="b2relu", dtype=np.float32), fcs, np.float32)), 16
    L = synth.fibonacci_sphere_graph(32492, 6)
    W = (rng.randn(15 * 25, 32) * 0.05).astype(np.float32)
    pr = [dict(W=W, b=np.full(32, 0.2, np.float32), K=25, p=1)]
    x = rng.randn(n_windows, 32492, 15).astype(np.float32)
    dy = rng.randn(n_windows, 32492, 32).astype(np.float32)

    def step(c):
        y, tr = O.conv_stack(x[c], [L], pr, dtype=np.float32, keep=True)
        O.conv_stack_bwd(tr, [L], pr, dy[c], dtype=np.float32, first_needs_dx=True)

    return step, 1


def cpu_step_times(cfg, n_windows, reps, warm, cores, mode=None):
    """Seconds per oracle step over ``n_windows`` windows on ``cores`` host threads; returns (times, mode).

    SciPy's CSR x dense product is single-threaded, so the step is parallelised over window chunks by a thread pool
    with BLAS pinned to ONE thread per worker (cores x cores oversubscription made the round-1 number 5x too slow);
    mode "blas" = no pool, BLAS on all cores; None = time both once and keep the faster."""
    from concurrent.futures import ThreadPoolExecutor

    from threadpoolctl import threadpool_limits

    step, chunk = _cpu_problem(cfg, n_windows)
    chunks = [c for c in np.array_split(np.arange(n_windows), max(1, n_windows // chunk)) if len(c)]

    def one_pool():
        with threadpool_limits(limits=1):
            with ThreadPoolExecutor(cores) as ex:
                list(ex.map(step, chunks))

    def one_blas():
        with threadpool_limits(limits=cores):
            step(np.arange(n_windows))

    def clock(fn):
        t = time.perf_counter()
        fn()
        return time.perf_counter() - t

    if mode is None:
        tp, tb = clock(one_pool), clock(one_blas)
        mode = "pool" if min(tp, clock(one_pool)) <= min(tb, clock(one_blas)) else "blas"
    one = one_pool if mode == "pool" else one_blas
    for _ in range(warm):
        one()
    return [clock(one) for _ in range(reps)], mode


CPU_PROBE = {"train": 128, "predict": 64, "vertex": 2}


def cpu_model():
    """Host CPU model string (SURVEY 8d: printed with every CPU number)."""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args, cfg):
    """--impl reference: the CPU implementation of the path (oracle port), all host threads, bounded sample."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = os.cpu_count() or 1
    n0 = CPU_PROBE[cfg["kind"]]
    probe, mode = cpu_step_times(cfg, n0, 1, 0, cores)
    rate = n0 / probe[0]
    budget = 100.0 / max(1, args.steps + args.warmup)
    gran = 32 if cfg["kind"] == "train" else (16 if cfg["kind"] == "predict" else 1)
    n = int(min(cfg["batch"], max(gran, (rate * budget) // gran * gran)))
    times, mode = cpu_step_times(cfg, n, args.steps, args.warmup, cores, mode)
    total = float(np.sum(times))
    value = n * args.steps / total
    what = {"train": "training step (fwd+loss+bwd, no optimiser update)", "predict": "forward pass",
            "vertex": "layer forward+backward"}[cfg["kind"]]
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": "windows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": cfg["workload"], "sample": "%d windows per step" % n},
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": cores, "kind": "port", "cpu": cpu_model(),
                         "sample": "%d-window %s of the NumPy/SciPy oracle, %d steps, %s"
                                   % (n, what, args.steps, CPU_MODE_TEXT[mode])},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU side
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.file,
                                         stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None
        self.marks = []

    def mark(self):
        self.marks.append(self._lines())

    def _lines(self):
        self.file.flush()
        try:
            with open(self.file.name) as f:
                return sum(1 for _ in f)
        except OSError:
            return 0

    def stop(self, lo=None, hi=None):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        rows = []
        try:
            with open(self.file.name) as f:
                for ln in f:
                    parts = [p.strip() for p in ln.split(",")]
                    if len(parts) >= 8:
                        rows.append(parts)
            os.unlink(self.file.name)
        except OSError:
            pass
        sel = rows[lo:hi] if (lo is not None and hi is not None and hi > lo) else rows
        if not sel:
            sel = rows
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        sm = []
        for r in sel:
            try:
                sm.append(float(r[0]))
            except ValueError:
                pass
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in sel for i in range(4) if r[4 + i].lower().startswith("active")})
        try:
            mx = float(sel[0][1])
        except ValueError:
            mx = None
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(sel)}


def layer_bytes(B, M_read, M, Fin, Fout, Kk, p, nnz, nb, backward, need_dx):
    """ALGORITHMIC bytes of one conv-layer launch (SURVEY.md 8d)."""
    Mo = -(-M // p)
    csr = 8 * nnz + 4 * (M + 1)
    w = 4 * (Fin * Kk * Fout + nb)
    if not backward:
        return 4 * B * M_read * Fin + 4 * B * Mo * Fout + csr + w
    return 4 * B * M_read * Fin + 2 * 4 * B * Mo * Fout + (4 * B * M * Fin if need_dx else 0) + csr + 2 * w


def graph_timed(torch, lib, fn, n, reps=3):
    """GPU seconds per call: the n calls (one per ring slot) are captured into a CUDA graph and the replays are
    bracketed by CUDA events on the launching stream, so host launch overhead is not counted as kernel time.
    Returns (seconds per call, launches of this library per call)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(3):
            fn(i % n)
    torch.cuda.current_stream().wait_stream(side)
    c0 = lib.gcnb_launch_count()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(n):
            fn(i)
    per_call = (lib.gcnb_launch_count() - c0) / n
    g.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3 / (reps * n), per_call


class TrainWorkload:
    """Configs 2 / 3a / 3a1 / 3b: one optimisation step of the two-conv-layer network (train.FusedTrainer)."""

    def __init__(self, cfg, args, torch, dev, rank, world):
        from gcn_fmri_decoding_b200 import _lib, ops, synth
        from gcn_fmri_decoding_b200.models import cgcnn
        from gcn_fmri_decoding_b200.train import FusedTrainer

        self.cfg, self.args, self.torch, self.dev, self.ops, self.lib = cfg, args, torch, dev, ops, _lib.lib()
        self._lib = _lib
        self.batch = cfg["batch"] if not args.strong else max(1, 4096 // world)
        B = self.batch
        A, gs, perm, L = synth.brain_graph(4)
        self.model = cgcnn(L=L, F=F2, K=cfg["K"], p=P2, M=MFC, filter=cfg["filter"], channel=15, device=dev, seed=7,
                           regularization=REG, batch_size=B, perm=perm, n_input_vertices=360, algo=args.algo)
        # dropout keep-probability 0.5 on the FC layers, as the reference trains (model.py:169, models_gcn.py:145)
        self.trainer = FusedTrainer(self.model, use_cuda_graph=not args.no_graph, dropout=0.5, own_gemm=not args.cublas_fc,
                                    fused_head=not args.no_fused_head, peer_allreduce=not args.nccl_allreduce)
        # ring of distinct resident batches: more than 2 x 126 MB of raw windows
        per = B * 360 * 15 * 4
        self.R = R = max(4, int(np.ceil(276e6 / per)))
        self.host = synth.bold_windows(min(B * 4, 4096), seed=2024 + rank)
        nh = self.host.shape[0] // B if self.host.shape[0] >= B else 1
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        base = [torch.as_tensor(self.host[(i % nh) * B:(i % nh + 1) * B], device=dev) for i in range(nh)]
        self.ring_x = [base[i % nh] + 0.01 * torch.randn(B, 360, 15, device=dev, generator=gen) for i in range(R)]
        self.ring_y = [torch.as_tensor(synth.labels(B, seed=i + 100 * rank), device=dev) for i in range(R)]
        self.l2_policy = "inputs rotate through a ring of %d distinct batches (%.0f MB > 2x L2)" % (R, R * per / 1e6)
        self.h2d = per + B * 8
        self.d2h = 4
        self.nh = nh
        # the ring slots are bound inputs: a step reads its batch in place (no copy into a static graph buffer)
        for xb, yb in zip(self.ring_x, self.ring_y):
            self.trainer.bind_inputs(xb, yb)

    def count_launches(self):
        tr = self.trainer
        snap = [t.clone() for t in (tr.flat_p, tr.flat_m, tr.flat_v, tr.state)]
        c0 = self.lib.gcnb_launch_count()
        tr._step_impl(self.ring_x[0], self.ring_y[0])
        self.torch.cuda.synchronize()
        n = int(self.lib.gcnb_launch_count() - c0)
        with self.torch.no_grad():
            for t, q in zip((tr.flat_p, tr.flat_m, tr.flat_v, tr.state), snap):
                t.copy_(q)
        return n

    def step(self, i):
        self.out = self.trainer.step(self.ring_x[i % self.R], self.ring_y[i % self.R])
        self.last = self.out[0]

    def outputs(self):
        """The last step's loss and logits, the gradient it computed and the parameters after its update."""
        loss, logits = self.out
        return {"loss": loss.reshape(1), "logits": logits, "grads": self.trainer.flat_g, "params": self.trainer.flat_p}

    def result_ok(self):
        v = float(self.last)
        assert np.isfinite(v), "training diverged"
        return {"final_loss": v, "allreduce": self.trainer.allreduce_kind}

    def e2e_setup(self):
        torch, B, dev = self.torch, self.batch, self.dev
        from gcn_fmri_decoding_b200 import synth

        self.pin_x = [torch.as_tensor(self.host[(i % self.nh) * B:(i % self.nh + 1) * B]).pin_memory() for i in range(4)]
        self.pin_y = [torch.as_tensor(synth.labels(B, seed=i)).pin_memory() for i in range(4)]
        self.dbuf_x = [torch.empty(B, 360, 15, device=dev) for _ in range(2)]
        self.dbuf_y = [torch.empty(B, dtype=torch.long, device=dev) for _ in range(2)]
        for s in range(2):  # what train.InputPipeline does with its slots
            self.trainer.bind_inputs(self.dbuf_x[s], self.dbuf_y[s])

    def e2e_copy(self, i, s):
        self.dbuf_x[s].copy_(self.pin_x[i % 4], non_blocking=True)
        self.dbuf_y[s].copy_(self.pin_y[i % 4], non_blocking=True)

    def e2e_step(self, i, s, out_host):
        l, _ = self.trainer.step(self.dbuf_x[s], self.dbuf_y[s])
        if out_host is not None:
            out_host[i].copy_(l, non_blocking=True)

    def roofline(self):
        torch, ops, lib, model, B, dev = self.torch, self.ops, self.lib, self.model, self.batch, self.dev
        hbm, tflops, src = measured_peaks()
        kernels = []
        if self.cfg["filter"] == "fourier":
            sp1, sp2 = model._spectral_plan(model.L[0]), model._spectral_plan(model.L[1])
            W1, W2, b1, b2 = model.conv_weights[0], model.conv_weights[1], model.conv_bias[0], model.conv_bias[1]
            mode = ops.BIAS_PER_FILTER
            with torch.no_grad():
                n1 = min(self.R, 12)
                x1 = [ops.perm_gather(self.ring_x[i], model.perm) for i in range(n1)]
                f1 = lambda i: ops.spectral_fwd(x1[i], sp1.Ut, W1, b1, 4, mode, True, True)
                ys1 = [f1(i) for i in range(n1)]
                f2 = lambda i: ops.spectral_fwd(ys1[i][0], sp2.Ut, W2, b2, 4, mode, True, True)
                ys2 = [f2(i) for i in range(n1)]
                dy2 = [torch.randn_like(ys2[i][0]) for i in range(n1)]
                dy1 = [torch.randn_like(ys1[i][0]) for i in range(n1)]
                fl = lambda M, Fi, Fo: 2.0 * M * M * Fi * B + 2.0 * M * Fo * Fi * B + 2.0 * M * M * Fo * B
                specs = [
                    ("conv1 fwd: spectral (U^T x, per-frequency mix, U y) 15->32 + b1relu + mpool4, M=400", f1, fl(400, 15, 32)),
                    ("conv2 fwd: spectral 32->32 + b1relu + mpool4, M=100", f2, fl(100, 32, 32)),
                    ("conv2 bwd: spectral backward (dx, dW, db)", lambda i: torch.ops.gcn_b200.spectral_bwd(
                        ys1[i][0], ys2[i][0], ys2[i][1], dy2[i], sp2.Ut, W2, 4, mode, True, True), 2 * fl(100, 32, 32)),
                    ("conv1 bwd: spectral backward (dW, db)", lambda i: torch.ops.gcn_b200.spectral_bwd(
                        x1[i], ys1[i][0], ys1[i][1], dy1[i], sp1.Ut, W1, 4, mode, True, False), 1.5 * fl(400, 15, 32)),
                ]
                for name, fn, flops in specs:
                    sec, per_call = graph_timed(torch, lib, fn, n1)
                    kernels.append({"op": name, "launches_per_op": per_call, "us": sec * 1e6, "algorithmic_flops": flops,
                                    "achieved_tflops": flops / sec * 1e-12, "frac": flops / sec * 1e-12 / tflops})
            top = max(kernels, key=lambda k: k["us"])
            return {"bound": "tensor", "kernel": top["op"], "achieved": top["achieved_tflops"], "peak": tflops,
                    "unit": "TFLOP/s", "frac": top["frac"], "traffic": None, "peak_source": src + ", dense bf16 burst",
                    "note": "spectral GEMMs run 3-pass TF32 mma.sync for fp32-level accuracy; FLOPs are algorithmic "
                            "(one pass)", "kernels": kernels}
        K1, K2 = self.cfg["K"]
        pl1, pl2 = model._plan(model.L[0]), model._plan(model.L[1])
        W1, W2, b1, b2 = model.conv_weights[0], model.conv_weights[1], model.conv_bias[0], model.conv_bias[1]
        mode = ops.BIAS_PER_FILTER
        n1 = min(self.R, 25)
        with torch.no_grad():
            # the same launches the training step issues (train.FusedTrainer): forward keeps the Chebyshev basis,
            # backward = streamed dW GEMM from the basis (+ the adjoint recursion for dx in layer 2)
            f1 = lambda i: ops.cheb_fwd_mean(self.ring_x[i], model.perm, pl1.rowptr, pl1.col, pl1.val, W1, b1, K1, 4, mode,
                                             True, self.args.algo, True)
            ys1 = [f1(i) for i in range(n1)]
            n2 = min(40, max(n1, int(40 * 512 / B)))
            y1s = [ys1[i % n1][0] + 0.0 * i for i in range(n2)]
            f2 = lambda i: ops.cheb_fwd_mean(y1s[i], None, pl2.rowptr, pl2.col, pl2.val, W2, b2, K2, 4, mode, True,
                                             self.args.algo, True)
            ys2 = [f2(i) for i in range(n2)]
            dm2 = [torch.randn_like(ys2[i][2]) for i in range(n2)]   # gradient of the mean over filters
            dy1 = [torch.randn_like(ys1[i][0]) for i in range(n1)]
            gW1, gb1 = torch.empty_like(W1), torch.empty(32, device=dev)
            gW2, gb2 = torch.empty_like(W2), torch.empty(32, device=dev)
            st = lambda t: t[3] if t[3].numel() else None
            k1 = self._lib.describe_fwd(B, 400, pl1.nnz, 15, 32, K1, 4).split(":")[0]
            k2 = self._lib.describe_fwd(B, 100, pl2.nnz, 32, 32, K2, 4).split(":")[0]
            specs = [
                ("conv1 fwd: %s (gather+cheb K=%d 15->32+b1relu+mpool4, M=400, keeps basis)" % (k1, K1), n1, f1,
                 layer_bytes(B, 360, 400, 15, 32, K1, 4, pl1.nnz, 32, False, False)),
                ("conv2 fwd: %s (cheb K=%d 32->32+b1relu+mpool4+mean, M=100, keeps basis)" % (k2, K2), n2, f2,
                 layer_bytes(B, 100, 100, 32, 32, K2, 4, pl2.nnz, 32, False, False)),
                ("conv2 bwd: k_dw_from_stack + k_dw_from_partials (dW,db from basis) + %s in adjoint mode (dx)" % k2, n2,
                 lambda i: ops.cheb_bwd_into(y1s[i], None, ys2[i][0], ys2[i][1], dm2[i], True, *pl2.tensors(), W2, gW2, gb2,
                                             K2, 4, mode, True, True, self.args.algo, st(ys2[i])),
                 layer_bytes(B, 100, 100, 32, 32, K2, 4, pl2.nnz, 32, True, True)),
                ("conv1 bwd: k_dw_from_stack + k_dw_from_partials (dW,db from basis)", n1,
                 lambda i: ops.cheb_bwd_into(self.ring_x[i], model.perm, ys1[i][0], ys1[i][1], dy1[i], False, *pl1.tensors(),
                                             W1, gW1, gb1, K1, 4, mode, True, False, self.args.algo, st(ys1[i])),
                 layer_bytes(B, 360, 400, 15, 32, K1, 4, pl1.nnz, 32, True, False)),
            ]
            traffic = {}
            tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
            if os.path.isfile(tpath):
                with open(tpath) as f:
                    traffic = json.load(f)
            for name, n, fn, nbytes in specs:
                sec, per_call = graph_timed(torch, lib, fn, n)
                key = name.split(":")[0] + ("" if self.cfg is CONFIGS["2"] and B == 512 else " (other config)")
                kernels.append({"op": name, "launches_per_op": per_call, "us": sec * 1e6, "algorithmic_bytes": nbytes,
                                "achieved_gbs": nbytes / sec * 1e-9, "frac": nbytes / sec * 1e-9 / hbm,
                                "traffic": traffic.get(key)})
        # the dominant KERNEL: ops that are one launch compete with their own time, multi-launch ops with their mean
        top = max(kernels, key=lambda k: k["us"] / max(k["launches_per_op"], 1.0))
        total_bytes = sum(k["algorithmic_bytes"] for k in kernels)
        total_us = sum(k["us"] for k in kernels)
        return {"bound": "hbm", "kernel": top["op"], "achieved": top["achieved_gbs"], "peak": hbm, "unit": "GB/s",
                "frac": top["frac"], "traffic": top["traffic"], "peak_source": src,
                "note": "algorithmic bytes per SURVEY 8d (no basis stack); the training path also writes/reads the "
                        "K-order basis -- see traffic and DESIGN.md section 3",
                "conv_stack_fwd_bwd": {"algorithmic_bytes": total_bytes, "us": total_us,
                                       "achieved": total_bytes / total_us * 1e-3,
                                       "frac": total_bytes / total_us * 1e-3 / hbm},
                "kernels": kernels}

    cpu_what = "training step (fwd+loss+bwd, no optimiser update)"


class PredictWorkload:
    """Config 1: forward pass of the production 6-layer network (predict_states path, models_gcn.py:998-1020)."""

    def __init__(self, cfg, args, torch, dev, rank, world):
        from gcn_fmri_decoding_b200 import _lib, ops, synth
        from gcn_fmri_decoding_b200.models import cgcnn

        self.cfg, self.args, self.torch, self.dev, self.ops, self.lib, self._lib = cfg, args, torch, dev, ops, _lib.lib(), _lib
        self.batch = B = cfg["batch"]
        A, gs, perm, L = synth.brain_graph(1)
        self.model = cgcnn(L=L, F=[32] * 6, K=[5] * 6, p=[1] * 6, M=MFC, filter="chebyshev5", brelu="b2relu", channel=15,
                           device=dev, seed=7, batch_size=B, perm=perm, n_input_vertices=360, algo=args.algo)
        per = B * 360 * 15 * 4
        self.R = R = 100  # 100 x 2.76 MB = 276 MB > 2 x L2
        self.host = synth.bold_windows(B * 4, seed=30 + rank)
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        self.ring_x = [torch.as_tensor(self.host[(i % 4) * B:(i % 4 + 1) * B], device=dev)
                       + 0.01 * torch.randn(B, 360, 15, device=dev, generator=gen) for i in range(R)]
        self.l2_policy = "inputs rotate through a ring of %d distinct batches (%.0f MB > 2x L2)" % (R, R * per / 1e6)
        self.h2d, self.d2h = per, B * 8
        # one CUDA graph of the forward pass over a static input buffer
        self.static_x = torch.empty(B, 360, 15, device=dev)
        self.static_x.copy_(self.ring_x[0])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(3):
                self.model(self.static_x)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = None
        if not args.no_graph:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph), torch.no_grad():
                self.logits = self.model(self.static_x)
                self.pred = self.logits.argmax(1)

    def count_launches(self):
        c0 = self.lib.gcnb_launch_count()
        with self.torch.no_grad():
            self.model(self.static_x)
        self.torch.cuda.synchronize()
        return int(self.lib.gcnb_launch_count() - c0)

    def _run(self, x):
        if self.graph is not None:
            self.static_x.copy_(x, non_blocking=True)
            self.graph.replay()
        else:
            with self.torch.no_grad():
                self.logits = self.model(x)
                self.pred = self.logits.argmax(1)

    def step(self, i):
        self._run(self.ring_x[i % self.R])

    def outputs(self):
        return {"logits": self.logits, "pred": self.pred.double()}

    def result_ok(self):
        assert bool(self.torch.isfinite(self.logits).all()), "non-finite logits"
        return {}

    def e2e_setup(self):
        torch, B = self.torch, self.batch
        self.pin_x = [torch.as_tensor(self.host[(i % 4) * B:(i % 4 + 1) * B]).pin_memory() for i in range(4)]
        self.dbuf_x = [torch.empty(B, 360, 15, device=self.dev) for _ in range(2)]
        self.pred_host = torch.zeros(B, dtype=torch.long).pin_memory()

    def e2e_copy(self, i, s):
        self.dbuf_x[s].copy_(self.pin_x[i % 4], non_blocking=True)

    def e2e_step(self, i, s, out_host):
        self._run(self.dbuf_x[s])
        self.pred_host.copy_(self.pred, non_blocking=True)

    def roofline(self):
        torch, ops, lib, model, B, dev = self.torch, self.ops, self.lib, self.model, self.batch, self.dev
        hbm, tflops, src = measured_peaks()
        pl = model._plan(model.L[0])
        mode = ops.BIAS_PER_VERTEX
        n = 25
        kernels = []
        with torch.no_grad():
            f1 = lambda i: ops.cheb_fwd(self.ring_x[i], model.perm, *pl.tensors(), model.conv_weights[0], model.conv_bias[0], 5,
                                        1, mode, True, False, self.args.algo)
            hs = [f1(i)[0] for i in range(n)]
            f2 = lambda i: ops.cheb_fwd(hs[i], None, *pl.tensors(), model.conv_weights[1], model.conv_bias[1], 5, 1, mode,
                                        True, False, self.args.algo)
            for name, fn, nbytes in (
                    ("layer 1: %s (gather+cheb K=5 15->32+b2relu, M=372)" % self._lib.describe_fwd(B, 372, pl.nnz, 15, 32, 5, 1).split(":")[0],
                     f1, layer_bytes(B, 360, 372, 15, 32, 5, 1, pl.nnz, 372 * 32, False, False)),
                    ("layers 2-6 (each): %s (cheb K=5 32->32+b2relu, M=372)" % self._lib.describe_fwd(B, 372, pl.nnz, 32, 32, 5, 1).split(":")[0],
                     f2, layer_bytes(B, 372, 372, 32, 32, 5, 1, pl.nnz, 372 * 32, False, False))):
                sec, per_call = graph_timed(torch, lib, fn, n)
                kernels.append({"op": name, "launches_per_op": per_call, "us": sec * 1e6, "algorithmic_bytes": nbytes,
                                "achieved_gbs": nbytes / sec * 1e-9, "frac": nbytes / sec * 1e-9 / hbm, "traffic": None})
            top = kernels[1]
            if ops.cheb_stack_supported(pl.rowptr, pl.col, pl.val, B, 32, 5, 5):
                # what the model's inference path launches for layers 2-6: ONE kernel, activations stay on the SM
                taps = [model._tap_image(q) for q in range(1, 6)]   # pre-split tap images, as the model's own path uses
                f3 = lambda i: ops.cheb_stack_fwd(hs[i], pl.rowptr, pl.col, pl.val, model.conv_weights[1:6], model.conv_bias[1:6],
                                                  5, mode, True, tap_images=taps)
                one = layer_bytes(B, 372, 372, 32, 32, 5, 1, pl.nnz, 372 * 32, False, False)
                nbytes = one + 4 * (4 * (32 * 5 * 32 + 372 * 32))   # + the weights and biases of four more layers
                sec, per_call = graph_timed(torch, lib, f3, n)
                kernels.append({"op": "layers 2-6 in one launch: k_cheb_fwd_umma<FP=32> layer stack (5 x cheb K=5 32->32+b2relu, M=372)",
                                "launches_per_op": per_call, "us": sec * 1e6, "algorithmic_bytes": nbytes,
                                "achieved_gbs": nbytes / sec * 1e-9, "frac": nbytes / sec * 1e-9 / hbm, "traffic": None})
                top = kernels[2]
        return {"bound": "hbm", "kernel": top["op"], "achieved": top["achieved_gbs"], "peak": hbm, "unit": "GB/s",
                "frac": top["frac"], "traffic": None, "peak_source": src, "kernels": kernels}

    cpu_what = "forward pass"


class VertexWorkload:
    """Config 5: one ChebyNet K=25 layer on a 32 492-vertex graph, forward + backward (general HBM-resident path)."""

    def __init__(self, cfg, args, torch, dev, rank, world):
        from gcn_fmri_decoding_b200 import _lib, ops, synth
        from gcn_fmri_decoding_b200.plan import GraphPlan

        self.cfg, self.args, self.torch, self.dev, self.ops, self.lib, self._lib = cfg, args, torch, dev, ops, _lib.lib(), _lib
        self.batch = B = cfg["batch"] if not args.strong else max(1, cfg["batch"] // world)
        self.M, self.K = 32492, 25
        self.pl = GraphPlan(synth.fibonacci_sphere_graph(self.M, 6), dev)
        gen = torch.Generator(device=dev).manual_seed(5 + rank)
        self.R = 3  # 3 x 125 MB of input windows > 2 x L2; the state itself (3 GB) streams through HBM anyway
        self.ring_x = [torch.randn(B, self.M, 15, device=dev, generator=gen) for _ in range(self.R)]
        self.W = torch.randn(15 * self.K, 32, device=dev, generator=gen) * 0.05
        self.bias = torch.full((32,), 0.2, device=dev)
        self.dy = torch.randn(B, self.M, 32, device=dev, generator=gen)
        self.l2_policy = "3 distinct input batches of %.0f MB; the K-order state (%.1f GB) exceeds L2 by itself" % (
            B * self.M * 15 * 4 / 1e6, self.K * B * self.M * 15 * 4 / 1e9)
        self.h2d, self.d2h = B * self.M * 15 * 4, 4

    def _fwd_bwd(self, x):
        ops, pl = self.ops, self.pl
        with self.torch.no_grad():
            y, am = ops.cheb_fwd(x, None, *pl.tensors(), self.W, self.bias, self.K, 1, ops.BIAS_PER_FILTER, True, True, self.args.algo)
            dx, dW, db = self.torch.ops.gcn_b200.cheb_bwd(x, None, y, am, self.dy, *pl.tensors(), self.W, self.K, 1,
                                                          ops.BIAS_PER_FILTER, True, True, self.args.algo)
        self.last = dW
        if self.args.dump_outputs:      # otherwise the step's 390 MB of outputs are freed as at any other step
            self.out = (y, dx, dW, db)
        return y

    def count_launches(self):
        c0 = self.lib.gcnb_launch_count()
        self._fwd_bwd(self.ring_x[0])
        self.torch.cuda.synchronize()
        return int(self.lib.gcnb_launch_count() - c0)

    def step(self, i):
        self._fwd_bwd(self.ring_x[i % self.R])

    def outputs(self):
        """y and dx (266 MB and 125 MB at B=64) on a fixed sample of 2048 vertices, dW and db whole."""
        y, dx, dW, db = self.out
        idx = self.torch.as_tensor(np.sort(np.random.RandomState(0).choice(self.M, 2048, replace=False)), device=self.dev)
        return {"y": y[:, idx], "dx": dx[:, idx], "dW": dW, "db": db}

    def result_ok(self):
        assert bool(self.torch.isfinite(self.last).all()), "non-finite gradient"
        return {}

    def e2e_setup(self):
        torch = self.torch
        self.pin_x = [self.ring_x[i].cpu().pin_memory() for i in range(2)]
        self.dbuf_x = [torch.empty_like(self.ring_x[0]) for _ in range(2)]
        self.sum_host = torch.zeros((), dtype=torch.float32).pin_memory()

    def e2e_copy(self, i, s):
        self.dbuf_x[s].copy_(self.pin_x[i % 2], non_blocking=True)

    def e2e_step(self, i, s, out_host):
        self._fwd_bwd(self.dbuf_x[s])
        self.sum_host.copy_(self.last.sum(), non_blocking=True)

    def roofline(self):
        torch, ops, lib, pl, B = self.torch, self.ops, self.lib, self.pl, self.batch
        hbm, tflops, src = measured_peaks()
        with torch.no_grad():
            f = lambda i: ops.cheb_fwd(self.ring_x[i % self.R], None, *pl.tensors(), self.W, self.bias, self.K, 1,
                                       ops.BIAS_PER_FILTER, True, False, self.args.algo)
            sec, per_call = graph_timed(torch, lib, f, self.R, reps=2)
        ideal = 4.0 * B * self.M * (15 + 32) + 8 * pl.nnz + 4 * (self.M + 1) + 4 * (15 * self.K * 32 + 32)
        stream = (self.K - 1) * 3 * 4.0 * B * self.M * 15 + 4.0 * B * self.M * (15 + 32)
        return {"bound": "hbm", "kernel": "forward: k_tile_swap + 24 x k_spmm_tma + k_stack_contract (whole layer forward)",
                "achieved": ideal / sec * 1e-9, "peak": hbm, "unit": "GB/s", "frac": ideal / sec * 1e-9 / hbm, "traffic": None,
                "peak_source": src, "us": sec * 1e6, "launches_per_op": per_call, "algorithmic_bytes": ideal,
                "note": "algorithmic = state-on-chip ideal (SURVEY 8d); the state cannot be on chip (one order = %.0f MB): "
                        "against the streaming model ((K-1) x 3 slabs + x + y = %.2f GB) the forward runs at %.2f of the "
                        "measured HBM peak" % (4.0 * B * self.M * 15 / 1e6, stream / 1e9, stream / sec * 1e-9 / hbm)}

    cpu_what = "layer forward+backward"


DUMP_LIMIT = 64 << 20


def dump_outputs(outputs, dirname):
    """Write each device tensor as ``dirname/<name>.npy`` (float64 stays float64, everything else becomes float32)."""
    arrays = {}
    for name, t in outputs.items():
        a = t.detach().cpu().numpy()
        arrays[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS))
    ap.add_argument("--strong", action="store_true", help="config 4 as written: global batch 4096 split over the GPUs")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--algo", type=int, default=0, help="0 auto, 1 general (HBM) kernels, 2 fused kernels")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fused-head", action="store_true", help="head launch by launch instead of k_head_step")
    ap.add_argument("--nccl-allreduce", action="store_true", help="N>1: plain NCCL all-reduce instead of the peer-memory "
                    "reduction fused into the Adam kernel")
    ap.add_argument("--cublas-fc", action="store_true", help="(with --no-fused-head) FC GEMMs through cuBLAS fp32")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed "
                    "(rank 0) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    if args.steps is None:
        args.steps = {"train": 200, "predict": 200, "vertex": 10}[cfg["kind"]]
    if args.warmup is None:
        args.warmup = {"train": 20, "predict": 20, "vertex": 3}[cfg["kind"]]
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    wl = {"train": TrainWorkload, "predict": PredictWorkload, "vertex": VertexWorkload}[cfg["kind"]](
        cfg, args, torch, dev, rank, world)
    B = wl.batch

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # launches of this library per step (counted on an eager step outside the timed region; a CUDA graph replays
    # exactly these launches)
    launches_per_step = wl.count_launches()

    sampler = ClockSampler(local) if rank == 0 else None
    for i in range(args.warmup):
        wl.step(i)
    barrier()
    if sampler:
        sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        wl.step(i)
    ev1.record()
    barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    value = world * B * args.steps / (ms_total * 1e-3)
    # copied on the device now, written once the clock-sampling window below has closed
    dumped = {k: t.detach().clone() for k, t in wl.outputs().items()} if args.dump_outputs and rank == 0 else None
    if sampler:
        sampler.mark()
    # keep the GPU under the same load for >= 1.5 s so that nvidia-smi (100 ms period) sees the clocks.
    # Every rank runs the same number of extra steps (a training step contains a collective).
    if ms_total < 1500:
        extra = int(min(20000, np.ceil(1500.0 / max(ms_total / args.steps, 1e-3))))
        for i in range(extra):
            wl.step(i)
            if i % 50 == 49:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        if sampler:
            sampler.marks[-1] = sampler._lines()
    if dumped is not None:
        dump_outputs(dumped, args.dump_outputs)
    extra_cfg = wl.result_ok()

    # ---- end to end: pinned host ring -> H2D -> step -> D2H result, all inside the timed region --------------------
    wl.e2e_setup()
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    # --steps sets every timed region: over few steps the one un-overlapped copy that fills the pipeline is a visible
    # share of the end-to-end time (4 % at 20 steps)
    n_e2e = args.steps
    out_host = torch.zeros(max(n_e2e, 1), dtype=torch.float32).pin_memory()

    def e2e_loop(n, record):
        main_stream = torch.cuda.current_stream()
        for s in range(2):
            freed[s].record(main_stream)
        for i in range(n):
            s = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[s])
                wl.e2e_copy(i, s)
                ready[s].record(copy_stream)
            main_stream.wait_event(ready[s])
            wl.e2e_step(i, s, out_host if record else None)
            freed[s].record(main_stream)

    e2e_loop(max(3, args.warmup // 2), False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    e2e_loop(n_e2e, True)
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    ms2 = torch.tensor([max(e0.elapsed_time(e1), 0.0)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * n_e2e / (float(ms2) * 1e-3)
    assert np.all(np.isfinite(out_host.numpy()))

    clocks = sampler.stop(*sampler.marks[-2:]) if sampler else None
    roofline = wl.roofline() if rank == 0 else None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        n0 = CPU_PROBE[cfg["kind"]]
        probe, mode = cpu_step_times(cfg, n0, 1, 0, cores)
        gran = 32 if cfg["kind"] == "train" else (16 if cfg["kind"] == "predict" else 1)
        n = int(min(cfg["batch"], max(gran, (n0 / probe[0] * 4.0) // gran * gran)))   # ~4 s of CPU work per step
        times, mode = cpu_step_times(cfg, n, 5, 1, cores, mode)
        cpu = {"value": n / float(np.median(times)), "unit": "windows/s", "cores": cores, "kind": "port", "cpu": cpu_model(),
               "sample": "%d-window %s of the NumPy/SciPy oracle, median of 5 after 1 warm-up, %s"
                         % (n, wl.cpu_what, CPU_MODE_TEXT[mode])}

    if rank == 0:
        config = {"workload": cfg["workload"], "global_batch": B * world, "parallelism": "dp%d" % world,
                  "l2_policy": wl.l2_policy, "cuda_graph": not args.no_graph, "algo": args.algo}
        if cfg["kind"] == "train":
            config["dropout_keep"] = 0.5
        config.update(extra_cfg)
        line = {
            "metric": cfg["metric"], "value": value, "unit": "windows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "windows/s", "h2d_bytes_per_step": wl.h2d, "d2h_bytes_per_step": wl.d2h,
                    "steps": n_e2e, "wall_s": wall},
            "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
            "roofline": roofline, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # Rank 0 alone runs the roofline / CPU legs; the others wait for it on the rendezvous store (a host-side
        # wait: no collective is left pending on the device).  The processes then leave without tearing the
        # communicator down: destroying a process group whose collectives live in captured CUDA graphs can hang.
        import datetime

        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("gcnb_bench_done", "1")
        else:
            store.wait(["gcnb_bench_done"], datetime.timedelta(minutes=30))
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Benchmark of the MMSSL hot training step on B200 (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config baby] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): BPR-triples/sec of the hot step = 1x MMSSL.forward (train mode) + BPR +
2x InfoNCE + feat_reg + backward + AdamW on a synthetic bipartite graph of the named shape, B = 1024
triples per GPU per step.  Prints ONE JSON line (rank 0).

  value     : whole-job triples/s, inputs resident in HBM (batch indices staged on the device),
              K steps timed with CUDA events on the launching stream, max over ranks.
  e2e       : the same through the public API `HotStepTrainer.train_step(users, pos, neg) -> loss`,
              each step copying the batch from pinned host memory and reading the loss back.
  roofline  : dominant kernel, algorithmic bytes / CUDA-event duration (measured here, cold L2)
              vs the measured HBM peak in MEASURED_PEAKS.json.
  cpu_baseline / --impl reference : the oracle port of the reference's CPU path
              (oracle/mmssl_oracle.py, stock torch CPU ops, all host threads) on the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH = 1024
METRIC = "bpr_triples_per_sec_hot_step"
UNIT = "triples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--config", default="baby")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "stock-gpu"],
                    help="'stock-gpu': comparator only -- the reference's torch ops (torch.sparse.mm, nn.Linear math, autograd, torch AdamW) on THIS GPU")
    ap.add_argument("--proj", default="tc", choices=["tc", "simt"])
    ap.add_argument("--spmm-impl", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=20)
    ap.add_argument("--cpu-threads", type=int, default=0, help="0 = the count that measured fastest on this host class (tools/cpu_threads.py)")
    ap.add_argument("--seed", type=int, default=2022)
    ap.add_argument("--batch", type=int, default=BATCH,
                    help="triples per GPU per step (reference default 1024, parser.py:54; SURVEY 8d also asks for 16384 at the synthetic configs)")
    ap.add_argument("--dp", default="fused", choices=["fused", "nccl"],
                    help="N>1 optimiser step: 'fused' = one multimem kernel (reduce-scatter + sharded AdamW + all-gather over "
                         "NVSwitch multicast, falls back to nccl when multicast is unavailable); 'nccl' = all-reduce + replicated AdamW")
    ap.add_argument("--extra-configs", default="sports,syn1m",
                    help="N = 1: also time these configs (hot step, stock-torch comparator, isolated kernels); 'none' to skip")
    ap.add_argument("--row-shard", default="sports,syn1m",
                    help="N > 1: also run the row-sharded whole hot step (north_star's scheme) on these configs; 'none' to skip")
    ap.add_argument("--row-exchange", default="multicast", choices=["multicast", "nccl"])
    ap.add_argument("--row-schedule", default="reduce_scatter", choices=["reduce_scatter", "allgather"],
                    help="products with a user-sized operand: partial products + reduce-scatter of the item-sized result, or all-gather of the operand")
    ap.add_argument("--row-graph", type=int, default=1, help="capture the row-sharded step in a CUDA graph (multicast exchange only)")
    ap.add_argument("--graph-comm", action="store_true",
                    help="EXPERIMENTAL (hung in round 1): capture the DP all-reduce + AdamW inside the CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (losses, gradients, updated parameters; rank 0) "
                         "as DIR/<name>.npy in float32, for comparing two builds on the same seeded inputs")
    return ap.parse_args()


# ----------------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_problem(name: str, seed: int, device):
    """Synthetic dataset + parameters + prepared graphs on `device`."""
    from mmssl_b200.engine import LIVE, FeatureStore
    from mmssl_b200.graph import BipartiteGraph
    from mmssl_b200.synthetic import make_dataset
    ds = make_dataset(name, seed=seed)
    g = torch.Generator(device="cpu").manual_seed(seed)
    d = ds.embed_size

    def xavier(r, c):
        b = (6.0 / (r + c)) ** 0.5
        return ((torch.rand(r, c, generator=g) * 2 - 1) * b)

    P = {
        "image_trans.weight": xavier(d, ds.dv), "image_trans.bias": (torch.rand(d, generator=g) * 2 - 1) / ds.dv ** 0.5,
        "text_trans.weight": xavier(d, ds.dt), "text_trans.bias": (torch.rand(d, generator=g) * 2 - 1) / ds.dt ** 0.5,
        "user_id_embedding.weight": xavier(ds.n_users, d), "item_id_embedding.weight": xavier(ds.n_items, d),
        "weight_dict.w_self_attention_cat": xavier(4 * d, d),
        "weight_dict.w_q": xavier(d, d), "weight_dict.w_k": xavier(d, d),
    }
    feats_cpu = (torch.randn(ds.n_items, ds.dv, generator=g), torch.randn(ds.n_items, ds.dt, generator=g))
    if device is None:
        return ds, P, feats_cpu, None, None
    Pd = {k: v.to(device).contiguous() for k, v in P.items()}
    build_problem.last_cpu = (ds, P, feats_cpu)          # the same problem on the host, for the stock-torch comparator
    feats = tuple(FeatureStore(f.to(device), keep_fp32=True) for f in feats_cpu)
    g_ui = BipartiteGraph.from_scipy(ds.ui_norm, device=device)
    g_iu = BipartiteGraph.from_scipy(ds.iu_norm, device=device)
    graphs = (g_ui, g_iu, g_ui, g_iu, g_ui, g_iu)        # modality graphs alias ui/iu (state at step 0, main.py:68-69)
    return ds, Pd, feats, graphs, feats_cpu


class HotStepTrainer:
    """Public API of the fused path: ``train_step(users, pos, neg) -> float loss`` (host in, host out)."""

    def __init__(self, P, feats, graphs, cfg, batch, world=1, sampler=None, graph_comm=False, dp="fused"):
        from mmssl_b200.hotstep import HotStep
        self.world = world
        self.dp_opt = None
        if world > 1 and not graph_comm and dp == "fused":
            # parameters and gradients move into symmetric-memory buckets BEFORE capture, so the graph's kernels
            # read / write them in place and the optimiser is one multimem kernel (parallel.FusedDPOptimizer)
            import torch.distributed as dist
            from mmssl_b200.engine import LIVE
            from mmssl_b200.parallel import FusedDPOptimizer
            try:
                self.dp_opt = FusedDPOptimizer({k: P[k] for k in LIVE}, dist.get_rank(), world, cfg.lr, cfg.beta1, cfg.beta2,
                                               cfg.eps, cfg.weight_decay)
                P = {**P, **self.dp_opt.params}
            except (RuntimeError, ImportError, AttributeError) as e:      # no NVSwitch multicast / symmetric memory here: NCCL path
                if dist.get_rank() == 0:
                    print(f"[bench] fused DP optimiser unavailable ({e}); using the NCCL path", file=sys.stderr)
        self.dp_mode = "fused" if self.dp_opt is not None else "nccl"
        # Default (validated at N = 2, 4, 8): the gradient all-reduce (NCCL) and AdamW are issued eagerly after
        # the graph replay.  graph_comm=True captures them inside the graph; that variant deadlocked on the
        # box in round 1 (NCCL capture) and is kept only as an experiment.
        self.graph_comm = graph_comm or world == 1
        self.dp_in_graph = self.dp_opt is not None and os.environ.get("MMSSL_DP_IN_GRAPH", "1") == "1"
        self.hs = HotStep(P, feats, graphs, cfg, batch=batch, optimizer_step=self.graph_comm, sampler=sampler)
        self.pin_idx = torch.empty(3, batch, dtype=torch.int64).pin_memory()
        self.pin_out = torch.empty(5, dtype=torch.float32).pin_memory()
        if self.dp_opt is not None:
            self.hs.grads.update(self.dp_opt.grads)
            if self.dp_in_graph:      # barriers + the multimem optimiser kernel are part of the captured step
                from mmssl_b200 import ops as _ops
                hs, opt = self.hs, self.dp_opt
                self.hs.grad_sync = lambda: (_ops.step_tick(hs.step_dev), opt.step_captured(hs.step_dev))
        elif world > 1:
            from mmssl_b200.parallel import GradBucket
            self.bucket = GradBucket(self.hs.grads)      # one flat all-reduce bucket for all live parameters
            self.hs.grads.update(self.bucket.views)
            if self.graph_comm:
                self.hs.grad_sync = self.bucket.all_reduce_mean
        self.hs.capture(warmup=2)

    def _finish_step(self):
        if self.dp_opt is not None and self.dp_in_graph:
            return
        if self.dp_opt is not None:
            from mmssl_b200 import ops
            ops.step_tick(self.hs.step_dev)      # the device sampler's counter
            self.dp_opt.step()
        elif self.world > 1 and not self.graph_comm:
            from mmssl_b200 import ops
            from mmssl_b200.engine import LIVE
            self.bucket.all_reduce_mean()
            hs = self.hs
            ops.step_tick(hs.step_dev)
            keys = list(LIVE)
            ops.adamw([hs.P[k] for k in keys], [hs.grads[k] for k in keys], [hs.m[k] for k in keys], [hs.v[k] for k in keys],
                      hs.step_dev, hs.cfg.lr, hs.cfg.beta1, hs.cfg.beta2, hs.cfg.eps, hs.cfg.weight_decay)

    def step_device(self, idx_dev):
        """One step with the batch already on the device."""
        self.hs.idx.copy_(idx_dev, non_blocking=True)
        self.hs.replay()
        self._finish_step()

    def train_step_device_sampled(self) -> float:
        """Batch drawn by the GPU sampler inside the graph: no host input, the loss is the only transfer."""
        self.hs.replay()
        self._finish_step()
        self.pin_out.copy_(self.hs.out5, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(self.pin_out[0])

    def train_step(self, users, pos, neg) -> float:
        self.pin_idx[0].copy_(torch.as_tensor(users)); self.pin_idx[1].copy_(torch.as_tensor(pos)); self.pin_idx[2].copy_(torch.as_tensor(neg))
        self.hs.idx.copy_(self.pin_idx, non_blocking=True)
        self.hs.replay()
        self._finish_step()
        self.pin_out.copy_(self.hs.out5, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(self.pin_out[0])


def l2_flush(buf):
    buf.add_(1.0)


def time_kernel(fn, flush_buf, reps=7):
    """Median CUDA-event duration (ms) of one launch of `fn` with a cold L2."""
    ts = []
    for _ in range(reps):
        l2_flush(flush_buf)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def roofline_objects(ds, P, feats, graphs, hbm_peak, peak_src, dev):
    """Time the two kernel classes that dominate the step, in isolation and with a cold L2."""
    from mmssl_b200 import ops
    d, I, U, nnz = ds.embed_size, ds.n_items, ds.n_users, ds.nnz
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 192 MiB > 126 MB L2
    out = {}
    # --- projection GEMM (image modality, forward): tcgen05 + TMA, HBM-bound on reading F
    fs = feats[0]
    w_hi, w_lo = ops.split_bf16(P["image_trans.weight"])
    floats, sk = ops.gemm_bf16x3_plan(I, d, fs.dim)
    part = torch.empty(floats, dtype=torch.float32, device=dev)
    ms = time_kernel(lambda: ops.gemm_bf16x3(fs.hi, fs.lo, w_hi, w_lo, I, d, fs.dim, sk, part), flush)
    alg = 4 * I * fs.dim + 4 * d * fs.dim + 4 * I * d
    gbs = alg / (ms * 1e-3) / 1e9
    out["projection"] = {"kernel": f"gemm_bf16x3_kernel<{d}> (image_trans forward, tcgen05+TMA)", "bound": "hbm",
                         "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(gbs / hbm_peak, 4),
                         "algorithmic_bytes": alg, "ms": round(ms, 5), "split_k": sk, "peak_source": peak_src,
                         "tflops_bf16_issued": round(3 * 2 * I * fs.dim * d / (ms * 1e-3) / 1e12, 2), "traffic": None}
    # --- SpMM (ui-type propagation, 1 RHS, d=64)
    x = torch.randn(I, d, device=dev)
    y = torch.empty(U, d, device=dev)
    ms = time_kernel(lambda: ops.spmm(graphs[0].fwd, [x], [y]), flush)
    alg = 8 * nnz + 4 * (U + 1) + 4 * d * I + 4 * d * U
    gather = 8 * nnz + 4 * (U + 1) + 4 * d * nnz + 4 * d * U
    gbs = alg / (ms * 1e-3) / 1e9
    out["spmm"] = {"kernel": f"spmm_csr_kernel (A_ui @ X, 1 right-hand side, d={d})", "bound": "hbm", "achieved": round(gbs, 1),
                   "peak": hbm_peak, "unit": "GB/s", "frac": round(gbs / hbm_peak, 4), "algorithmic_bytes": alg,
                   "gather_model_gbs_effective": round(gather / (ms * 1e-3) / 1e9, 1), "ms": round(ms, 5),
                   "peak_source": peak_src, "traffic": None,
                   "note": "compulsory bytes are %.1f MB: at HBM peak that is %.1f us, below launch latency -> latency-bound at this scale"
                           % (alg / 1e6, alg / hbm_peak / 1e3)}
    # `traffic` (dram__bytes of one launch) needs an ncu capture: it is never copied from a file here.  The captures of the same
    # kernels are under profiles/ (see profiles/README.md); in-process it stays null.
    out["library"] = library_kernels(ds, P, feats, graphs, x, y, flush, dev)
    del flush
    return out


def library_kernels(ds, P, feats, graphs, x, y, flush, dev):
    """The stock-torch kernels of the same two operators on this GPU, isolated, cold L2 (SURVEY 2.1: "the Blackwell-capable
    kernel set to beat"): torch.sparse.mm on the reference's COO tensor (Models.py:69-73: coalesce + COO->CSR + cuSPARSE on every
    call), the same on a prepared CSR tensor (cuSPARSE SpMM alone), and nn.Linear's fp32 cuBLAS GEMM (Models.py:173)."""
    import torch.nn.functional as F
    from mmssl_b200 import ops
    out = {}
    coo = ds.ui_norm.tocoo()
    idx = torch.from_numpy(np.vstack([coo.row, coo.col]).astype(np.int64)).to(dev)
    val = torch.from_numpy(coo.data.astype(np.float32)).to(dev)
    a_coo = torch.sparse_coo_tensor(idx, val, coo.shape)             # uncoalesced flag, like the reference's tensors
    a_csr = a_coo.coalesce().to_sparse_csr()
    ours = time_kernel(lambda: ops.spmm(graphs[0].fwd, [x], [y]), flush)
    out["spmm_ui"] = {"ours_ms": round(ours, 5),
                      "torch_sparse_mm_coo_ms": round(time_kernel(lambda: torch.sparse.mm(a_coo, x), flush, reps=5), 5),
                      "cusparse_csr_ms": round(time_kernel(lambda: torch.mm(a_csr, x), flush, reps=5), 5)}
    fs = feats[0]
    if fs.fp32 is not None:
        w, b = P["image_trans.weight"], P["image_trans.bias"]
        I, d = fs.n_items, ds.embed_size
        w_hi, w_lo = ops.split_bf16(w)
        floats, sk = ops.gemm_bf16x3_plan(I, d, fs.dim)
        part = torch.empty(floats, dtype=torch.float32, device=dev)
        yp = torch.empty(I, d, device=dev)

        def ours_proj():
            ops.split_bf16(w)
            ops.gemm_bf16x3(fs.hi, fs.lo, w_hi, w_lo, I, d, fs.dim, sk, part)
            ops.proj_epilogue(part, sk, I, d, b, None, yp)
        tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        out["projection"] = {"ours_ms (split W + tcgen05 GEMM + bias epilogue)": round(time_kernel(ours_proj, flush), 5),
                             "cublas_fp32_linear_ms": round(time_kernel(lambda: F.linear(fs.fp32, w, b), flush, reps=5), 5)}
        torch.backends.cuda.matmul.allow_tf32 = tf32
    return out


CPU_THREADS_DEFAULT = 8      # fastest of {8,16,32,64,128} on the box's 128-thread Xeon 8562Y+: 0.37 s/step vs 40 s/step at 128
                             # threads (profiles/r01_cpu_threads.txt) -- the baseline is reported at its best setting


def cpu_baseline(name, seed, steps, batch, threads=0):
    """The oracle port of the reference's CPU path (stock torch CPU ops) on the host cores.  The thread
    count is the one that measured fastest (more threads make torch's sparse kernels slower here)."""
    from oracle import mmssl_oracle as O
    from mmssl_b200.synthetic import TripleSampler
    ds, P, feats_cpu, _, _ = build_problem(name, seed, None)
    torch.set_num_threads(min(os.cpu_count(), threads if threads > 0 else CPU_THREADS_DEFAULT))
    cfg = O.HotPathConfig(embed_size=ds.embed_size, n_layers=ds.n_layers, batch_size=batch)
    ui, iu = O.to_torch_coo(ds.ui_norm), O.to_torch_coo(ds.iu_norm)
    graphs = (ui, iu, ui, iu, ui, iu)
    cpu = O.CpuHotStep(P, feats_cpu[0], feats_cpu[1], graphs, ds.n_items, cfg)
    smp = TripleSampler(ds.train, seed=seed)
    times = []
    for i in range(steps + 1):
        u, p, n = smp.sample(batch)
        t0 = time.perf_counter()
        cpu.step(u, p, n)
        if i > 0:
            times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"value": round(batch / med, 1), "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{steps} hot steps of config '{name}' (B={batch}) after 1 warm-up, median; min {min(times):.3f}s max {max(times):.3f}s",
            "cpu_model": model, "os_cpu_count": os.cpu_count(), "s_per_step": round(med, 4)}


def stock_gpu_baseline(name, seed, steps, warmup, batch, device, problem=None):
    """SURVEY 8d's second comparator: what the unmodified reference's hot path costs on the same B200 through stock PyTorch
    (cuSPARSE / cuBLAS / ATen element-wise kernels, autograd, torch.optim.AdamW, one float(loss) sync per step like
    main.py:431) -- the restatement in oracle/mmssl_oracle.py run on CUDA tensors.  A comparator, not the product and not the
    target; timed with CUDA events around `steps` steps after `warmup`."""
    from oracle import mmssl_oracle as O
    from mmssl_b200.synthetic import TripleSampler
    ds, P, feats_cpu = problem if problem is not None else build_problem(name, seed, None)[:3]
    cfg = O.HotPathConfig(embed_size=ds.embed_size, n_layers=ds.n_layers, batch_size=batch)
    ui, iu = O.to_torch_coo(ds.ui_norm).to(device), O.to_torch_coo(ds.iu_norm).to(device)
    step = O.CpuHotStep({k: v.to(device) for k, v in P.items()}, feats_cpu[0].to(device), feats_cpu[1].to(device),
                        (ui, iu, ui, iu, ui, iu), ds.n_items, cfg)
    smp = TripleSampler(ds.train, seed=seed)
    batches = [tuple(torch.from_numpy(x).to(device) for x in smp.sample(batch)) for _ in range(8)]
    for i in range(warmup):
        step.step(*batches[i % 8])
    cuda = torch.device(device).type == "cuda"
    if cuda:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    t0 = time.perf_counter()
    for i in range(steps):
        step.step(*batches[i % 8])
    if cuda:
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    else:
        ms = (time.perf_counter() - t0) / steps * 1e3
    return {"value": round(batch / ms * 1e3, 1), "unit": UNIT, "ms_per_step": round(ms, 4), "kind": "stock torch %s on %s" % (torch.__version__, device),
            "sample": f"{steps} hot steps of config '{name}' (B={batch}) after {warmup} warm-up"}


def cpu_full_step_baseline(name, seed, steps, batch, d_state, threads=0):
    """Same role as ``cpu_baseline`` for the whole training iteration (main.py:333-434, oracle/gan_oracle.py:FullStep): used by
    tools/fullstep_bench.py, not by this file's own bench line.  ``d_state``: the Discriminator's initial state_dict (CPU)."""
    from oracle import gan_oracle as GO, mmssl_oracle as O
    from mmssl_b200.synthetic import TripleSampler
    ds, P, feats_cpu, _, _ = build_problem(name, seed, None)
    torch.set_num_threads(min(os.cpu_count(), threads if threads > 0 else CPU_THREADS_DEFAULT))
    d, I = ds.embed_size, ds.n_items
    h1, h2 = int(I / 4), int(I / 8)
    cfg = O.HotPathConfig(embed_size=d, n_layers=ds.n_layers, batch_size=batch)
    R = ds.train.tocsr()
    R.sort_indices()
    cpu = GO.FullStep({k: v.clone() for k, v in P.items()}, {k: v.clone() for k, v in d_state.items()}, feats_cpu[0], feats_cpu[1], R, cfg,
                      GO.GanConfig())
    smp = TripleSampler(ds.train, seed=seed)
    gen = torch.Generator().manual_seed(seed + 3)
    mk = lambda n, w, q: ((torch.rand(n, w, generator=gen) >= q) / (1 - q)).float()
    times = []
    for i in range(steps):
        u, p, n = smp.sample(batch)
        draws = ([mk(I, d, 0.2) for _ in range(4)], [mk(2 * batch, h1, 0.31) for _ in range(4)], [mk(2 * batch, h2, 0.5) for _ in range(4)],
                 torch.rand(batch, I, generator=gen), torch.rand(2 * batch, 1, generator=gen))
        t0 = time.perf_counter()
        cpu.step(u.tolist(), p.tolist(), n.tolist(), *draws)
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": round(batch / med, 1), "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{steps} full iterations (oracle/gan_oracle.py:FullStep) of config '{name}' (B={batch}), median", "s_per_step": round(med, 4)}


def extra_config(name, a, dev, hbm_peak, peak_src):
    """SURVEY 8d / VERDICT r1 #5: the other BASELINE configs on this GPU, lighter than the headline run: device-resident hot
    step (captured graph), the stock-torch hot step on the same GPU, isolated SpMM / projection with their library twins."""
    from mmssl_b200.hotstep import HotStepConfig
    from mmssl_b200.synthetic import CONFIGS, TripleSampler
    U, I, nnz, d, K, dv, dt = CONFIGS[name]
    t0 = time.perf_counter()
    ds, P, feats, graphs, _ = build_problem(name, a.seed, dev)
    cpu_problem = build_problem.last_cpu
    cfg = HotStepConfig(embed_size=d, n_layers=K, batch_size=BATCH, proj_impl=a.proj)
    trainer = HotStepTrainer(P, feats, graphs, cfg, BATCH, world=1)
    smp = TripleSampler(ds.train, seed=a.seed)
    steps, warm = (200, 10) if nnz < 2_000_000 else (30, 5)
    dev_batches = torch.from_numpy(np.stack([np.stack(smp.sample(BATCH)) for _ in range(16)])).to(dev)
    for w in range(warm):
        trainer.step_device(dev_batches[w % 16])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        trainer.step_device(dev_batches[s % 16])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    roofs = roofline_objects(ds, P, feats, graphs, hbm_peak, peak_src, dev)
    out = {"workload": f"{name}: {U}x{I}, {nnz} edges, d={d}, {K}-layer GCN, V{dv}/T{dt}, B={BATCH}", "ms_per_step": round(ms, 4),
           "value": round(BATCH / ms * 1e3, 1), "unit": UNIT, "steps": steps, "roofline_spmm": roofs["spmm"],
           "roofline_projection": roofs["projection"], "library_kernels": roofs["library"]}
    del trainer
    try:
        sg = stock_gpu_baseline(name, a.seed, 20 if nnz < 2_000_000 else 5, 3, BATCH, str(dev), problem=cpu_problem)
        out["stock_gpu"] = {"ms_per_step": sg["ms_per_step"], "value": sg["value"], "kind": sg["kind"], "speedup_ours": round(sg["ms_per_step"] / ms, 2)}
    except Exception as e:                      # the comparator must never take the bench line down (e.g. cuSPARSE out of memory)
        out["stock_gpu"] = {"unavailable": str(e)[:200]}
    out["build_s"] = round(time.perf_counter() - t0, 1)
    return out


def nvlink_counters(index: int):
    """(rx_kib, tx_kib) summed over the NVLink links of GPU `index` from the driver's throughput counters
    (`nvidia-smi nvlink -gt d`), or None where the query is not supported."""
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(index)], capture_output=True, text=True, timeout=20).stdout
    except Exception:
        return None
    rx = tx = 0
    seen = False
    for ln in out.splitlines():
        ln = ln.strip()
        if "Data Rx:" in ln or "Data Tx:" in ln:
            try:
                val = int(ln.split(":")[-1].strip().split()[0])
            except (ValueError, IndexError):
                continue
            seen = True
            if "Rx" in ln:
                rx += val
            else:
                tx += val
    return (rx, tx) if seen else None


def _fixed_masks(I, d, drop, seed, dev):
    g = torch.Generator().manual_seed(seed)
    return tuple(((torch.rand(I, d, generator=g) >= drop) / (1 - drop)).float().to(dev) for _ in range(2))


def dp_parity_vs_1gpu(trainer, P0, feats, graphs, cfg, my_batch, rank, world, dev):
    """VERDICT r1 #1b: the N-GPU data-parallel step against 1-GPU HotSteps ON RANK 0, same fixed global batch (the N replica
    batches) and the same injected dropout masks: mean loss and every live gradient after the cross-GPU reduction.
    The N-GPU side runs the product's own path eagerly (its kernels, then the reduction primitive the optimiser uses:
    multimem.ld_reduce over the symmetric gradient bucket, or the NCCL all-reduce of --dp nccl)."""
    import torch.distributed as dist
    from mmssl_b200 import _lib
    from mmssl_b200._lib import ptr, stream
    from mmssl_b200.engine import LIVE
    from mmssl_b200.hotstep import HotStep
    hs = trainer.hs
    I, d = graphs[0].shape[1], cfg.embed_size
    # restore the initial parameters on every replica so that both sides start from the same point
    for k in LIVE:
        hs.P[k].copy_(P0[k])
    hs.masks = _fixed_masks(I, d, cfg.drop_rate, 1000 + rank, dev)
    hs.idx.copy_(my_batch)
    saved, saved_sync = hs.optimizer_step, hs.grad_sync
    hs.optimizer_step, hs.grad_sync = False, None         # gradients only: the reduction is done explicitly below
    out5 = hs.run().clone()
    hs.optimizer_step, hs.grad_sync = saved, saved_sync
    hs.masks = None
    torch.cuda.synchronize()
    dist.barrier()
    keys = list(LIVE)
    if trainer.dp_opt is not None:          # the switch-reduced sum of the replicas' gradient buckets
        opt = trainer.dp_opt
        red = torch.empty_like(opt.gflat)
        lib = _lib.load(require_device=True)
        opt.hg.barrier()
        import ctypes as C
        _lib.check(lib.mmssl_mc_allreduce_sum(C.c_void_p(opt.g_mc), ptr(red), red.numel(), stream()))
        opt.hg.barrier()
        red.mul_(1.0 / world)
        got = {k: red[(opt.grads[k].data_ptr() - opt.gflat.data_ptr()) // 4:][:opt.grads[k].numel()].view_as(opt.grads[k]) for k in keys}
        how = "multimem.ld_reduce over the symmetric gradient bucket (the fused optimiser's reduction)"
    else:
        flat = trainer.bucket.flat.clone()
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.mul_(1.0 / world)
        got = {k: flat[(trainer.bucket.views[k].data_ptr() - trainer.bucket.flat.data_ptr()) // 4:][:trainer.bucket.views[k].numel()].view_as(trainer.bucket.views[k]) for k in keys}
        how = "NCCL all-reduce of the flat gradient bucket"
    loss = out5[:1].clone()
    dist.all_reduce(loss, op=dist.ReduceOp.SUM)
    all_batches = [torch.empty_like(my_batch) for _ in range(world)]
    dist.all_gather(all_batches, my_batch.contiguous())
    res = None
    if rank == 0:
        ref = HotStep({k: P0[k].clone() for k in P0}, feats, graphs, cfg, batch=my_batch.shape[1], optimizer_step=False)
        acc = {k: torch.zeros_like(P0[k]) for k in keys}
        ref_loss = 0.0
        for r in range(world):
            ref.masks = _fixed_masks(I, d, cfg.drop_rate, 1000 + r, dev)
            ref.idx.copy_(all_batches[r])
            ref_loss += float(ref.run()[0])
            for k in keys:
                acc[k] += ref.grads[k]
        errs = {}
        for k in keys:
            want = acc[k] / world
            errs[k] = float((got[k] - want).abs().max() / want.abs().max().clamp_min(1e-30))
        lerr = abs(float(loss) / world - ref_loss / world) / max(abs(ref_loss / world), 1e-30)
        res = {"loss_rel_err": lerr, "max_grad_rel_err": max(errs.values()), "worst_grad": max(errs, key=errs.get),
               "n_gpu_reduction": how, "reference": f"{world} single-GPU HotStep evaluations on rank 0 (one per replica batch), averaged",
               "tolerance": 1e-4, "ok": bool(lerr < 1e-4 and max(errs.values()) < 1e-4)}
    for k in LIVE:                              # leave the replicas in sync for whatever runs next
        hs.P[k].copy_(P0[k])
    torch.cuda.synchronize()
    dist.barrier()
    return res


def row_shard_report(name, a, rank, world, dev):
    """north_star / SURVEY 8e / VERDICT r1 #2: the WHOLE hot step with embedding tables, features, graphs and optimiser state
    row-sharded over the N GPUs (mmssl_b200/rowshard_step.py), same global batch B as the 1-GPU step: ms/step, speed-up over
    the 1-GPU fused step on the same problem (timed on rank 0 of this run), exchanges and bytes per step, achieved NVLink
    rate, and parity of one step (losses + all gradients, same injected dropout masks) against the 1-GPU step."""
    import torch.distributed as dist
    from mmssl_b200.engine import LIVE, P_EI, P_EU
    from mmssl_b200.hotstep import HotStep, HotStepConfig
    from mmssl_b200.rowshard_step import RowShardedHotStep, shard_problem
    from mmssl_b200.synthetic import CONFIGS, TripleSampler
    U, I, nnz, d, K, dv, dt = CONFIGS[name]
    t0 = time.perf_counter()
    ds, P_cpu, feats_cpu, _, _ = build_problem(name, a.seed, None)            # the same seeded problem on every rank (host)
    cfg = HotStepConfig(embed_size=d, n_layers=K, batch_size=BATCH, proj_impl=a.proj)
    Pl, fl, gl, pu, pi = shard_problem(P_cpu, feats_cpu, ds.ui_norm, ds.iu_norm, rank, world, dev)
    mode = a.row_exchange
    try:
        sh = RowShardedHotStep(Pl, fl, gl, cfg, BATCH, pu, pi, rank, exchange=mode, schedule=a.row_schedule)
    except (RuntimeError, ImportError, AttributeError) as e:
        if rank == 0:
            print(f"[bench] multicast exchange unavailable ({e}); NCCL all-gathers", file=sys.stderr)
        mode = "nccl"
        sh = RowShardedHotStep(Pl, fl, gl, cfg, BATCH, pu, pi, rank, exchange=mode, schedule=a.row_schedule)
    smp = TripleSampler(ds.train, seed=a.seed)
    batches = [tuple(torch.from_numpy(x).to(dev) for x in smp.sample(BATCH)) for _ in range(8)]
    g = torch.Generator().manual_seed(7)
    full_masks = tuple(((torch.rand(I, d, generator=g) >= cfg.drop_rate) / (1 - cfg.drop_rate)).float() for _ in range(2))
    out = {"workload": f"{name}: {U}x{I}, {nnz} edges, d={d}, {K}-layer GCN, V{dv}/T{dt}, global B={BATCH}", "n_gpus": world,
           "exchange": mode, "schedule": sh.schedule}

    # ---- parity of one step (no optimiser) against the 1-GPU fused step on rank 0
    sh.masks = tuple(pi.local(m, rank).to(dev) for m in full_masks)
    sh.optimizer_step = False
    sh.set_indices(*batches[0])
    got5 = sh.run().clone()
    tab = {}
    for k, part in ((P_EU, pu), (P_EI, pi)):
        full = [torch.empty_like(sh.grads[k]) for _ in range(world)]
        dist.all_gather(full, sh.grads[k].contiguous())
        tab[k] = torch.cat(full)[:part.n]
    hs = None
    ms_1gpu = None
    if rank == 0:
        _, Pd, feats, graphs, _ = build_problem(name, a.seed, dev)
        hs = HotStep(Pd, feats, graphs, cfg, batch=BATCH, optimizer_step=False)
        hs.masks = tuple(m.to(dev) for m in full_masks)
        hs.set_indices(*batches[0])
        want5 = hs.run().clone()
        errs = {"losses": float(((got5 - want5).abs() / want5.abs().clamp_min(1e-12)).max())}
        for k in LIVE:
            gk = tab[k] if k in tab else sh.grads[k]
            errs[k] = float((gk - hs.grads[k]).abs().max() / hs.grads[k].abs().max().clamp_min(1e-30))
        worst = max(errs, key=errs.get)
        out["parity_vs_1gpu"] = {"max_rel_err": errs[worst], "worst": worst, "loss_rel_err": errs["losses"], "tolerance": 1e-4,
                                 "ok": bool(errs[worst] < 1e-4)}
        # the 1-GPU step of the same problem, same batch size: the denominator of the speed-up
        hs.masks = None
        hs.optimizer_step = True
        hs.capture(warmup=2)
        n1 = 100 if nnz < 2_000_000 else 20
        for s in range(3):
            hs.set_indices(*batches[s % 8]); hs.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(n1):
            hs.set_indices(*batches[s % 8]); hs.replay()
        e1.record()
        torch.cuda.synchronize()
        ms_1gpu = e0.elapsed_time(e1) / n1
        del hs, Pd, feats, graphs
        torch.cuda.empty_cache()
    dist.barrier()

    # ---- timing (optimiser on, torch-RNG dropout): CUDA graph when every exchange is a kernel + signal-pad barrier
    sh.masks = None
    sh.optimizer_step = True
    captured = False
    if mode == "multicast" and a.row_graph:
        try:
            sh.set_indices(*batches[0])
            sh.capture()
            captured = True
        except RuntimeError as e:
            if rank == 0:
                print(f"[bench] row-sharded step not captured ({e}); eager launches", file=sys.stderr)
    step = sh.replay if captured else sh.run
    steps = 100 if nnz < 2_000_000 else 20
    for s in range(3):
        sh.set_indices(*batches[s % 8]); step()
    torch.cuda.synchronize()
    sh.n_gathers = sh.gathered_bytes = sh.n_reduce_scatters = 0
    # BEFORE the barrier: the query is a subprocess (~80 ms with 8 GPUs).  Between the barrier and the first event it made rank 0
    # enter the loop late while the other ranks' clocks were already running at their first exchange barrier: +75 ms / steps on
    # the max over ranks (round 2: 8 GPUs, Sports 1.31 ms reported vs 0.57 ms measured by tools/rowshard_ab.py, 1M x 200k 11.7 vs ~7.9).
    nv0 = nvlink_counters(dev.index) if rank == 0 else None
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        sh.set_indices(*batches[s % 8]); step()
    e1.record()
    torch.cuda.synchronize()
    nv1 = nvlink_counters(dev.index) if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    if not captured:
        gath, rsc, gbytes = sh.n_gathers // steps, sh.n_reduce_scatters // steps, sh.gathered_bytes / steps
    else:                                       # counted once at capture time: run one eager step to count
        sh.n_gathers = sh.gathered_bytes = sh.n_reduce_scatters = 0
        sh.run()
        torch.cuda.synchronize()
        gath, rsc, gbytes = sh.n_gathers, sh.n_reduce_scatters, float(sh.gathered_bytes)
    out.update({"ms_per_step": round(ms, 4), "value": round(BATCH / ms * 1e3, 1), "unit": UNIT, "steps": steps, "cuda_graph": captured,
                "all_gathers_per_step": int(gath), "reduce_scatters_per_step": int(rsc), "bytes_received_per_rank_per_step": int(gbytes),
                "nvlink_GBps_per_rank_if_serial": round(gbytes / (ms * 1e-3) / 1e9, 1),
                "build_s": round(time.perf_counter() - t0, 1)})
    if rank == 0:
        if nv0 is not None and nv1 is not None:      # the driver's NVLink throughput counters around the timed loop (rank 0's GPU)
            rx, tx = (nv1[0] - nv0[0]) * 1024 / steps, (nv1[1] - nv0[1]) * 1024 / steps
            out["nvlink_counter"] = {"rx_bytes_per_step": int(rx), "tx_bytes_per_step": int(tx), "rx_GBps_over_the_step": round(rx / (ms * 1e-3) / 1e9, 1),
                                     "tx_GBps_over_the_step": round(tx / (ms * 1e-3) / 1e9, 1), "source": "nvidia-smi nvlink -gt d (sum over links, rank 0)"}
        else:
            out["nvlink_counter"] = None
    if rank == 0 and ms_1gpu is not None:
        out["ms_per_step_1gpu"] = round(ms_1gpu, 4)
        out["speedup_vs_1gpu"] = round(ms_1gpu / ms, 3)
    del sh
    torch.cuda.empty_cache()
    dist.barrier()
    return out


DUMP_BYTES = 60 * 2 ** 20


def dump_outputs(out_dir, arrays, seed):
    """Writes every tensor of `arrays` (name -> tensor) as float32 `out_dir/<name>.npy`, DUMP_BYTES of data in all.  The
    smallest are written first and whole; a tensor larger than an even share of the bytes left keeps a seeded random
    sample of its rows, in ascending row order, so that runs with the same arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    g = torch.Generator().manual_seed(seed)
    left, todo = DUMP_BYTES, sorted(arrays.items(), key=lambda kv: (kv[1].numel(), kv[0]))
    for i, (name, t) in enumerate(todo):
        t = t.detach().float().cpu()
        share = left // (len(todo) - i)
        if 4 * t.numel() > share:
            keep = share * t.shape[0] // (4 * t.numel())
            t = t[torch.randperm(t.shape[0], generator=g)[:keep].sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())
        left -= 4 * t.numel()


# ----------------------------------------------------------------------------------------------
def main():
    global BATCH
    a = parse()
    BATCH = a.batch
    torch.manual_seed(a.seed)         # dropout masks: the same arguments draw the same masks
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    from mmssl_b200.synthetic import CONFIGS
    U, I, nnz, d, K, dv, dt = CONFIGS[a.config]
    config = {"workload": f"{a.config}: synthetic bipartite {U}x{I}, {nnz} edges, d={d}, {K}-layer GCN, V{dv}/T{dt} features, "
                          f"B={BATCH} triples per GPU per step, modality graphs alias ui/iu",
              "global_batch": BATCH * max(world, 1), "parallelism": "single GPU" if world == 1 else f"dp{world} (replicated graph, one flat gradient all-reduce per step" + (", captured in the CUDA graph)" if a.graph_comm else ", eager after the graph replay)"),
              "l2_policy": "working set per step (%.0f MB of features) exceeds the 126 MB L2; isolated kernels timed after a 192 MiB L2 flush" % (4 * I * (dv + dt) / 1e6)}

    if a.impl == "reference":
        if rank != 0:
            return
        cb = cpu_baseline(a.config, a.seed, a.steps, BATCH, a.cpu_threads)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
                "warmup": 1, "ms_per_step": round(cb["s_per_step"] * 1e3, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if a.impl == "stock-gpu":
        if rank != 0:
            return
        sg = stock_gpu_baseline(a.config, a.seed, a.steps, max(a.warmup, 3), BATCH, os.environ.get("MMSSL_STOCK_DEVICE", "cuda:0"))
        print(json.dumps({"impl": "stock-torch-gpu", "metric": METRIC, "value": sg["value"], "unit": UNIT, "n_gpus": 1, "steps": a.steps,
                          "warmup": max(a.warmup, 3), "ms_per_step": sg["ms_per_step"], "higher_is_better": True, "dtype": "f32",
                          "data": "synthetic", "config": config, "comparator": sg}))
        return

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from mmssl_b200 import _lib, ops
    from mmssl_b200.hotstep import HotStepConfig
    from mmssl_b200.synthetic import TripleSampler
    _lib.load(require_device=True)
    if a.spmm_impl is not None:
        ops.set_default_spmm_impl(a.spmm_impl)

    ds, P, feats, graphs, _ = build_problem(a.config, a.seed, dev)
    cfg = HotStepConfig(embed_size=d, n_layers=K, batch_size=BATCH, proj_impl=a.proj)
    P0 = {k: v.clone() for k, v in P.items()} if world > 1 else None
    trainer = HotStepTrainer(P, feats, graphs, cfg, BATCH, world=world, graph_comm=a.graph_comm, dp=a.dp)
    if world > 1 and trainer.dp_mode == "fused":
        where = "inside the step's CUDA graph" if trainer.dp_in_graph else "after the graph replay"
        config["parallelism"] = (f"dp{world} (replicated graph; optimiser step = two signal-pad barriers + one multimem kernel {where}: "
                                 f"switch-reduced gradient slice, AdamW on 1/{world} of the parameters, multicast store of the new slice)")
    smp = TripleSampler(ds.train, seed=a.seed + 17 * rank)
    n_batches = a.steps + a.warmup
    host_batches = [np.stack(smp.sample(BATCH)) for _ in range(n_batches)]
    dev_batches = torch.from_numpy(np.stack(host_batches)).to(dev)               # [n, 3, B] resident in HBM

    # launches per step (our kernels only): count one eager step that leaves the optimiser state alone
    c0 = _lib.launch_count
    saved, saved_sync = trainer.hs.optimizer_step, trainer.hs.grad_sync
    trainer.hs.optimizer_step, trainer.hs.grad_sync = False, None
    trainer.hs.run()
    trainer.hs.optimizer_step, trainer.hs.grad_sync = saved, saved_sync
    launches_per_step = (_lib.launch_count - c0) + 2     # + step_tick + adamw

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- (A) device-resident timing
    clocks = ClockSampler(local)      # samples from the warm-up through both timed regions
    if rank == 0:
        clocks.start()
    for w in range(a.warmup):
        trainer.step_device(dev_batches[w])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_seg = 5 if a.steps >= 10 else 1
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(n_seg - 1)]
    seg = a.steps // n_seg
    barrier()
    e0.record()
    for s in range(a.steps):
        trainer.step_device(dev_batches[a.warmup + s])
        if (s + 1) % seg == 0 and (s + 1) // seg <= n_seg - 1:
            marks[(s + 1) // seg - 1].record()              # spread of the timed region (no synchronisation)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    pts = [e0] + marks + [e1]
    seg_steps = [seg] * (n_seg - 1) + [a.steps - seg * (n_seg - 1)]
    seg_ms = [pts[i].elapsed_time(pts[i + 1]) / seg_steps[i] for i in range(n_seg)]
    if a.dump_outputs:                # before (B) steps the parameters on
        if rank == 0:
            from mmssl_b200.engine import LIVE
            hs = trainer.hs
            dump_outputs(a.dump_outputs, {"losses": hs.out5, **{"grad." + k: hs.grads[k] for k in LIVE},
                                          **{"param." + k: hs.P[k] for k in LIVE}}, a.seed)
        barrier()

    # ---------------- (B) end to end through the public API (pinned host -> device, loss read back)
    for w in range(min(3, a.warmup)):
        trainer.train_step(*host_batches[w])
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fmarks = [torch.cuda.Event(enable_timing=True) for _ in range(n_seg - 1)]
    f0.record()
    last_loss = 0.0
    for s in range(a.steps):
        last_loss = trainer.train_step(*host_batches[a.warmup + s])
        if (s + 1) % seg == 0 and (s + 1) // seg <= n_seg - 1:
            fmarks[(s + 1) // seg - 1].record()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    fpts = [f0] + fmarks + [f1]
    seg_ms_e2e = [fpts[i].elapsed_time(fpts[i + 1]) / seg_steps[i] for i in range(n_seg)]
    clk = clocks.stop() if rank == 0 else None

    parity = row_shard = None
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e] + seg_ms + seg_ms_e2e, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])
        seg_ms, seg_ms_e2e = t[2:2 + n_seg].tolist(), t[2 + n_seg:].tolist()
        parity = dp_parity_vs_1gpu(trainer, P0, feats, graphs, cfg, dev_batches[0], rank, world, dev)
        if a.row_shard != "none":
            del trainer
            torch.cuda.empty_cache()
            row_shard = {}
            for name in a.row_shard.split(","):
                if name:
                    try:
                        row_shard[name] = row_shard_report(name, a, rank, world, dev)
                    except Exception as e:          # keep the headline line alive; the failure is reported in place
                        import traceback
                        row_shard[name] = {"failed": repr(e)[:300], "where": traceback.format_exc()[-400:]}

    if rank == 0:
        hbm_peak, peak_src = peaks()
        roofs = roofline_objects(ds, P, feats, graphs, hbm_peak, peak_src, dev)
        # the dominant kernel by time in the step: 4 projection-class GEMM launches vs (16 + 4K) SpMM launches
        n_spmm = 2 * (4 + 2 * K)
        t_proj = roofs["projection"]["ms"] * 2 * (1 + dt / dv)      # fwd + wgrad, image + text (bytes-scaled)
        t_spmm = roofs["spmm"]["ms"] * n_spmm
        dom = "projection" if t_proj >= t_spmm else "spmm"
        roof = {k: roofs[dom][k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
        roof.update({"kernel": roofs[dom]["kernel"], "ms_per_launch": roofs[dom]["ms"], "peak_source": peak_src,
                     "est_share_ms_per_step": {"projection": round(t_proj, 4), "spmm": round(t_spmm, 4)}})
        total_triples = BATCH * world * a.steps
        line = {"metric": METRIC, "value": round(total_triples / (ms_total * 1e-3), 1), "unit": UNIT, "n_gpus": world,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms_total / a.steps, 4), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "clocks": clk, "gpu_launches": launches_per_step * a.steps,
                "ms_per_step_spread": {"segments": n_seg, "min": round(min(seg_ms), 4), "median": round(statistics.median(seg_ms), 4),
                                       "max": round(max(seg_ms), 4), "e2e_min": round(min(seg_ms_e2e), 4),
                                       "e2e_median": round(statistics.median(seg_ms_e2e), 4), "e2e_max": round(max(seg_ms_e2e), 4),
                                       "note": "the timed region cut into equal consecutive segments (events, max over ranks per segment)"},
                "e2e": {"value": round(total_triples / (ms_e2e * 1e-3), 1), "unit": UNIT, "h2d_bytes_per_step": 3 * BATCH * 8,
                        "d2h_bytes_per_step": 5 * 4, "ms_per_step": round(ms_e2e / a.steps, 4), "last_loss": round(last_loss, 6)},
                "roofline": roof, "roofline_spmm": roofs["spmm"], "roofline_projection": roofs["projection"],
                "library_kernels": roofs["library"], "launches_per_step": launches_per_step}
        if parity is not None:
            line["parity_vs_1gpu"] = parity
        if row_shard is not None:
            line["row_shard"] = row_shard
        if world == 1:      # SURVEY 2.1 / 8d: the reference's own ops through stock torch on THIS GPU (comparator, not the product)
            try:
                sg = stock_gpu_baseline(a.config, a.seed, 30, 5, BATCH, str(dev), problem=build_problem.last_cpu)
                line["stock_gpu"] = {"ms_per_step": sg["ms_per_step"], "value": sg["value"], "kind": sg["kind"], "sample": sg["sample"],
                                     "speedup_ours": round(sg["ms_per_step"] / (ms_total / a.steps), 2)}
            except Exception as e:
                line["stock_gpu"] = {"unavailable": str(e)[:200]}
        if world == 1 and BATCH > 1024:
            line["device_sampler_e2e"] = {"unavailable": "one device-sampler launch draws at most 1024 triples (csrc/sampler.cu)"}
        elif world == 1:    # SURVEY 8f next #1: batches drawn on the device (no host sampler, no H2D)
            from mmssl_b200.sampler import DeviceTripleSampler
            P2 = {k: v.clone() for k, v in P.items()}
            tr2 = HotStepTrainer(P2, feats, graphs, cfg, BATCH, world=1, sampler=DeviceTripleSampler(ds.train, device=dev, seed=a.seed))
            for _ in range(3):
                tr2.train_step_device_sampled()
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(a.steps):
                tr2.train_step_device_sampled()
            g1.record()
            torch.cuda.synchronize()
            ms = g0.elapsed_time(g1)
            line["device_sampler_e2e"] = {"value": round(BATCH * a.steps / (ms * 1e-3), 1), "unit": UNIT, "ms_per_step": round(ms / a.steps, 4),
                                          "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 20}
        if world == 1 and a.extra_configs != "none":
            del trainer
            line["configs"] = {}
            for name in a.extra_configs.split(","):
                if name and name != a.config:
                    torch.cuda.empty_cache()
                    try:
                        line["configs"][name] = extra_config(name, a, dev, hbm_peak, peak_src)
                    except Exception as e:
                        line["configs"][name] = {"failed": repr(e)[:300]}
        if not a.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(a.config, a.seed, a.cpu_steps, BATCH, a.cpu_threads)
        print(json.dumps(line))
        if parity is not None and not parity["ok"]:
            print("[bench] N-GPU vs 1-GPU parity FAILED: " + json.dumps(parity), file=sys.stderr)
            sys.exit(3)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

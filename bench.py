#!/usr/bin/env python
"""Benchmark of the HybridVAE hot path (BASELINE.json metric: train users/sec & eval top-K users/sec; % of TC/HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--precision bf16|fp32] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on the host cores

Default workload = BASELINE.json configs[2] (C3): 1M users x 200k items, d = 768, 4,096 users per GPU and step -- the
largest single-GPU configuration and the one the 1/2/4/8-GPU scaling is quoted on.  A "step" is one optimisation step
(forward, multinomial NLL + KL, backward, clip, Adam) over one batch of synthetic users.  Rank 0 prints ONE JSON line;
besides the contract's keys it carries `extra`: the C2 training step, a C4-shape (1M items) evaluation -- item-sharded over
the ranks when N > 1 --, kernel rooflines at the 1M-item shape, the C5 grid sweep (16 configurations spread over the ranks), the
gradient-exchange path and a data-parallel parity number.
See DESIGN.md §6 for how each field is obtained.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for _p in (str(ROOT), str(ROOT / "recommendation-system_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC, UNIT = "train_users_per_sec", "users/s"
DESC = {"c1": "Appliances-shaped synthetic", "c2": "All_Beauty-shaped synthetic", "c3": "1M users x 200k items synthetic"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c1", "c2", "c3"])
    ap.add_argument("--precision", default=os.environ.get("HVAE_B200_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=0, help="users per GPU per step (default: the workload's)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the bounded CPU-baseline sample (b200 arm)")
    ap.add_argument("--ref-seconds", type=float, default=150.0, help="budget of the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (losses, updated weights) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return dict(hbm=float(d["hbm_gbs"]), tc_burst=float(d["bf16_tflops"]), tc_sustained=float(d["bf16_tflops_sustained"]),
                    source="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.samples, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.06)
        self.proc.terminate()
        rows = [s for s in self.samples if t0 is None or t0 - 0.05 <= s[0] <= t1 + 0.05] or self.samples
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for _, line in rows:
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        med = float(np.median(sm)) if sm else None
        return {"sm_mhz": med, "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
def make_workload(name, batch_override=0):
    from hvae_b200.synth import CONFIGS, make_interactions, make_item_embeddings
    c = dict(CONFIGS[name])
    if batch_override:
        c["batch"] = batch_override
    data = make_interactions(c["n_users"], c["n_items"], 0)
    E = make_item_embeddings(c["n_items"], c["emb_dim"], 0)
    return c, data, E


def workload_config(name, c, n_gpus):
    """Identical for both arms (the driver compares them)."""
    return {"workload": f"{name}: {DESC[name]} ({c['n_users']} users x {c['n_items']} items, d={c['emb_dim']}, latent {c['latent_dim']}, "
                        f"hidden {c['hidden_dims']}), HybridVAE training step",
            "users_per_gpu_per_step": c["batch"], "global_batch": c["batch"] * n_gpus,
            "parallelism": f"dp{n_gpus}" if n_gpus > 1 else "single",
            "l2": "working set (W1 + Adam moments + E) exceeds L2 at c3; in addition a 256 MiB write flushes L2 between timed steps (untimed)"}


# ---- the reference's arithmetic on the host cores (oracle port) ------------------------------------------------------
class CpuReference:
    """The reference's train_epoch arithmetic (src/ml/train.py:81-103): DataLoader row densification, dense fp32 forward /
    backward through ATen, clip_grad_norm_(5), Adam -- oracle/hvae_oracle.py, all host threads.  `step(B_s)` runs one
    optimisation step over B_s users of the workload (a bounded sample of the 4,096-user batch when the full one would not fit
    the time budget: at c3 a full step is ~6 TFLOP of dense fp32 GEMM + a 3.3 GB dense batch)."""

    def __init__(self, c, data, E):
        from oracle import hvae_oracle as orc
        self.orc, self.c = orc, c
        torch.set_num_threads(os.cpu_count() or 1)
        torch.manual_seed(0)
        self.m = orc.OracleVAE(c["n_items"], E, c["latent_dim"], c["hidden_dims"], c["dropout"], c["beta"])
        self.opt = orc.make_adam(self.m)
        self.m.train()
        self.csr = data.scipy_csr()
        self.order = np.random.default_rng(0).permutation(c["n_users"])
        self.pos = 0
        self.threads = torch.get_num_threads()

    def step(self, B):
        c, orc = self.c, self.orc
        if self.pos + B > len(self.order):
            self.pos = 0
        rows = self.order[self.pos:self.pos + B]
        self.pos += B
        t0 = time.perf_counter()
        x = torch.stack([torch.FloatTensor(self.csr[int(r)].toarray().flatten()) for r in rows])   # train.py:45-47 + default collate
        self.opt.zero_grad()
        sc, mu, lv = self.m.forward_ref(x)
        loss, _, _ = orc.loss_terms(sc, x, mu, lv, c["beta"])
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.m.parameters(), max_norm=5.0)
        self.opt.step()
        loss.item()
        return time.perf_counter() - t0

    def pick_sample(self, seconds_per_step, B_full):
        """Largest power-of-two-ish sample <= the full batch whose step fits `seconds_per_step` (probe at 128 users; a step's
        cost is affine in the sample size, so the linear extrapolation is conservative)."""
        probe = min(B_full, 128)
        t = self.step(probe)
        t = min(t, self.step(probe))
        B = int(probe * max(1.0, 0.8 * seconds_per_step / t))
        B = min(B_full, max(probe, 1 << (B.bit_length() - 1)))
        return B


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    c, data, E = make_workload(args.workload, args.batch)
    ref = CpuReference(c, data, E)
    W, K = args.warmup, args.steps
    Bs = ref.pick_sample(args.ref_seconds / max(1, W + K), c["batch"])
    for _ in range(W):
        ref.step(Bs)
    secs = sum(ref.step(Bs) for _ in range(K))
    ups = K * Bs / secs
    sample = (f"{K} steps of {Bs} users each (a bounded sample of the {c['batch']}-user batch of the same workload; users/s = sample users / "
              f"step time), oracle/hvae_oracle.py = the reference's train loop incl. row densification, {ref.threads} host threads")
    line = {"impl": "reference", "metric": METRIC, "value": ups, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * secs / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args.workload, c, args.gpus),
            "cpu_baseline": {"value": ups, "unit": UNIT, "cores": ref.threads, "kind": "port", "sample": sample},
            "e2e": {"value": ups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "sample_users_per_step": Bs}
    print(json.dumps(line), flush=True)


def torch_cuda_eager(c, data, E, dev, steps=5):
    """Context only (not the baseline, not the product): the reference's module tree (oracle restatement) moved to the GPU, as the
    reference supports with --device cuda (src/ml/train.py:185-193,360): stock ATen / cuBLAS fp32 kernels on DENSE [B, N] batches
    (built on the device from the CSR; the reference densifies on the host).  One train step = train.py:88-96."""
    from oracle import hvae_oracle as orc
    torch.manual_seed(0)
    m = orc.OracleVAE(c["n_items"], E, c["latent_dim"], c["hidden_dims"], c["dropout"], c["beta"]).to(dev)
    opt = orc.make_adam(m)
    m.train()
    B, N = c["batch"], c["n_items"]
    indptr, indices = torch.from_numpy(data.indptr).to(dev), torch.from_numpy(data.indices.astype(np.int64)).to(dev)

    def dense(rows):
        lens = indptr[rows + 1] - indptr[rows]
        r = torch.repeat_interleave(torch.arange(rows.numel(), device=dev), lens)
        starts = torch.repeat_interleave(indptr[rows], lens)
        off = torch.arange(r.numel(), device=dev) - torch.repeat_interleave(torch.cumsum(lens, 0) - lens, lens)
        x = torch.zeros(rows.numel(), N, device=dev)
        x[r, indices[starts + off]] = 1.0
        return x

    order = torch.from_numpy(np.random.default_rng(0).permutation(c["n_users"])).to(dev)
    ts = []
    for s in range(steps + 2):
        rows = order[s * B:(s + 1) * B]
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        x = dense(rows)
        opt.zero_grad()
        sc, mu, lv = m.forward_ref(x)
        loss, _, _ = orc.loss_terms(sc, x, mu, lv, c["beta"])
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=5.0)
        opt.step()
        loss.item()
        ts.append(time.perf_counter() - t0)
    del m, opt
    gc.collect()
    torch.cuda.empty_cache()
    t = float(np.mean(ts[2:]))
    return {"value": B / t, "unit": UNIT, "ms_per_step": 1e3 * t, "steps": steps, "batch": B,
            "what": "oracle/hvae_oracle.py (the reference's module tree) on device=cuda: stock ATen/cuBLAS fp32 on dense [B, N] batches, "
                    "eager, incl. on-device densification and the loss .item(); context for the CPU baseline, not a baseline itself"}


# ---- helpers of the b200 arm -------------------------------------------------------------------------------------
class Ctx:
    pass


def dist_max(vals, dev, world):
    if world == 1:
        return [float(v) for v in vals]
    import torch.distributed as dist
    t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def barrier(dev, world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize(dev)


def timed_events(fn, n, flush_buf, dev):
    """n calls of fn(i), each bracketed by CUDA events on the current stream, L2 flushed (untimed) before each -> ms list."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for i in range(n):
        if flush_buf is not None:
            flush_buf.fill_(i & 0xFF)
        evs[i][0].record()
        fn(i)
        evs[i][1].record()
    torch.cuda.synchronize(dev)
    return [a.elapsed_time(b) for a, b in evs]


def build_train(name, args, dev, world, rank, batch_override=0):
    """Model + trainer + resident CSR + the walk over global batches of one workload."""
    from hvae_b200.engine import Batch, DeviceCSR
    from hvae_b200.model import HybridVAE
    from hvae_b200.train import VAETrainer
    x = Ctx()
    x.name = name
    x.c, x.data, x.E = make_workload(name, batch_override)
    c = x.c
    x.B, x.U, x.N, x.d = c["batch"], c["n_users"], c["n_items"], c["emb_dim"]
    torch.manual_seed(0)
    x.model = HybridVAE(x.N, x.E, c["latent_dim"], c["hidden_dims"], c["dropout"], c["beta"], precision=args.precision)
    x.trainer = VAETrainer(x.model, dev, lr=1e-3, use_cuda_graph=not args.no_graph)
    x.dp = x.trainer.enable_data_parallel() if world > 1 else None
    x.csr = DeviceCSR.from_arrays(x.data.indptr, x.data.indices, None, x.N, dev)
    x.Bg = x.B * world
    order = np.random.default_rng(0).permutation(x.U).astype(np.int32)
    x.order = np.concatenate([order, order[:x.Bg]])
    x.order_dev = torch.from_numpy(x.order).to(dev)
    x.lens = np.diff(x.data.indptr)
    x.n_batches = max(1, x.U // x.Bg)
    x.cap_local = max(int(x.lens[x.order[i * x.Bg + rank * x.B:i * x.Bg + (rank + 1) * x.B]].sum()) for i in range(x.n_batches))
    x.cap_global = max(int(x.lens[x.order[i * x.Bg:(i + 1) * x.Bg]].sum()) for i in range(x.n_batches))

    def batch_at(s):
        g0 = (s % x.n_batches) * x.Bg
        return Batch(x.csr, x.order_dev[g0 + rank * x.B:g0 + (rank + 1) * x.B], x.B, max(1, x.cap_local), b_global=x.Bg,
                     nnz_cap_global=x.cap_global)
    x.batch_at = batch_at
    x.step = lambda s: x.trainer.train_step(batch_at(s), b_global=x.Bg)
    x.model.train()
    return x


def step_outputs(x, w1_sample=1 << 22):
    """What the most recent training step hands its caller: the three losses and the updated weights under the reference's
    tensor names.  encoder.0.weight ([h0, N], 480 MB at C3) is reduced to a fixed sample of `w1_sample` flat positions of
    its [h0, N] shape, drawn from a seeded generator (`encoder.0.weight.sample`); every other tensor is written whole."""
    out = {"losses": np.asarray(x.trainer.last_losses(), dtype=np.float32)}
    lay, arena = x.model.layout, x.model.arena.data
    for k in lay.reference_keys():
        v = lay.view(arena, k)
        if k == "encoder.0.weight" and v.numel() > w1_sample:
            pos = np.sort(np.random.default_rng(0).integers(0, v.numel(), w1_sample))
            r, c = torch.from_numpy(pos // v.shape[1]).to(v.device), torch.from_numpy(pos % v.shape[1]).to(v.device)
            out[k + ".sample"] = v[r, c].cpu().numpy()
        else:
            out[k] = v.cpu().numpy()
    return out


def measure_train(x, W, K, dev, world, rank, flush_buf, lib, dump_dir=None):
    """W warm-up steps, then K timed steps (per-step CUDA events, L2 flushed in between) and K back-to-back steps.
    dump_dir: rank 0 writes step_outputs() of the last timed step there (before the back-to-back steps)."""
    for s in range(W):
        x.step(s)
    barrier(dev, world)
    l0 = lib.launches
    t0 = time.perf_counter()
    ms = timed_events(lambda i: x.step(W + i), K, flush_buf, dev)
    barrier(dev, world)
    t1 = time.perf_counter()
    launches = lib.launches - l0
    if dump_dir is not None:
        if world > 1:       # per-rank partial sums of the losses -> the global batch's (as train_on_batch returns them)
            import torch.distributed as dist
            dist.all_reduce(x.model.engine.loss_out)
        if rank == 0:
            Path(dump_dir).mkdir(parents=True, exist_ok=True)
            for name, a in step_outputs(x).items():
                np.save(Path(dump_dir) / f"{name}.npy", a)
        barrier(dev, world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(K):
        x.step(W + K + s)
    e1.record()
    barrier(dev, world)
    ms_total, ms_hot = dist_max([sum(ms), e0.elapsed_time(e1)], dev, world)
    return dict(value=K * x.Bg / (ms_total * 1e-3), ms_per_step=ms_total / K, value_hot=K * x.Bg / (ms_hot * 1e-3), ms_hot=ms_hot / K,
                launches=launches, wall=(t0, t1))


def kernel_spans(x, W, K, flush_buf, pk, world, ms_per_step, args):
    """Per-kernel-group durations: CUDA events around each group on its launching stream over un-graphed steps of the same
    workload -> achieved bytes/flops against the measured peaks."""
    eng, trainer, model = x.model.engine, x.trainer, x.model
    graph = trainer.use_cuda_graph
    trainer.use_cuda_graph = False
    eng.prof = {}
    PS = min(K, 30)
    for s in range(PS):
        flush_buf.fill_(1)
        x.step(W + 2 * K + s)
    spans = eng.span_ms()
    eng.prof = None
    trainer.use_cuda_graph = graph
    span_avg = {k: float(np.mean(v)) for k, v in spans.items()}
    lay = model.layout
    B, N, d, h = x.B, x.N, x.d, x.c["hidden_dims"]
    nb = min(4, x.n_batches)
    n_unique_avg = float(np.mean([len(np.unique(np.concatenate([x.data.indices[x.data.indptr[u]:x.data.indptr[u + 1]]
                                                               for u in x.order[i * x.Bg:(i + 1) * x.Bg]]))) for i in range(nb)]))
    ld1 = (h[0] + 3) // 4 * 4
    adam_bytes = 24.0 * lay.n_params + 4.0 * (lay.n_dense + n_unique_avg * ld1)
    flops_fwd = 2.0 * B * N * d
    kernels = {}

    def add(name, ms, bound, amount, extra=None):
        unit = "GB/s" if bound == "hbm" else "TFLOP/s"
        scale = 1e9 if bound == "hbm" else 1e12
        peak = pk["hbm"] if bound == "hbm" else pk["tc_sustained"]
        k = {"ms": ms, "bound": bound, "achieved": amount / (ms * 1e-3) / scale, "peak": peak, "unit": unit,
             ("algorithmic_bytes" if bound == "hbm" else "algorithmic_flops"): amount}
        k["frac"] = k["achieved"] / peak
        k["share_of_step"] = ms / ms_per_step
        if extra:
            k.update(extra)
        kernels[name] = k

    if "adam" in span_avg:      # (two launches: rows of W1^T without a gradient -- beside the backward pass in the captured step -- and the rest)
        add("adam", span_avg["adam"] + span_avg.get("adam_untouched", 0.0), "hbm", adam_bytes)
    if "score_fwd" in span_avg:
        add("score_fwd", span_avg["score_fwd"], "tensor", flops_fwd)
    if "score_bwd" in span_avg:
        add("score_bwd", span_avg["score_bwd"], "tensor", flops_fwd)
    if "score_onepass" in span_avg:     # forward + backward through the scores in one sweep: S = U E^T and O = P E, 2BNd each
        add("score_onepass", span_avg["score_onepass"], "tensor", 2 * flops_fwd,
            {"launches": "one-pass scoring kernel (tcgen05 cta_group::2 for d <= 768) + combine", "executed_flops": 2 * flops_fwd,
             "frac_of_burst_peak": 2 * flops_fwd / (span_avg["score_onepass"] * 1e-3) / 1e12 / pk["tc_burst"]})
    if "gather" in span_avg:
        nnz_avg = float(x.lens[x.order[:x.Bg * nb]].sum()) / nb / world
        add("gather", span_avg["gather"], "hbm", nnz_avg * (ld1 * 4 + 4) + B * (3 * ld1 * 4 + 16))
    dom = max(kernels, key=lambda k: kernels[k]["ms"]) if kernels else None
    roofline = None
    if dom:
        kd = kernels[dom]
        traffic = None
        tf = ROOT / "profiles" / "traffic.json"
        if tf.exists():
            traffic = json.loads(tf.read_text()).get(f"{x.name}:{args.precision}:{dom}")
        roofline = {"kernel": dom, "bound": kd["bound"], "achieved": kd["achieved"], "peak": kd["peak"], "unit": kd["unit"],
                    "frac": kd["frac"], "traffic": traffic, "peak_source": pk["source"] + (" sustained" if kd["bound"] == "tensor" else ""),
                    "ms_per_launch": kd["ms"], "share_of_step": kd["share_of_step"],
                    "how": "CUDA events around the kernel on its launching stream over un-graphed steps of the timed workload; share = "
                           "ms_per_launch / ms_per_step of the captured step"}
    return kernels, span_avg, roofline


def measure_e2e(x, K, dev, world, rank, flush_buf):
    """The public per-batch API with HOST (pinned) inputs: H2D of the batch and D2H of the loss inside every timed step."""
    KE = min(K, 100)
    host = []
    if world == 1:      # the step's input is the batch's CSR slice (indptr, indices, values) in pinned host memory
        for s in range(KE):
            g0 = (s % x.n_batches) * x.Bg
            rows_h = x.order[g0:g0 + x.B].astype(np.int64)
            starts, ln = x.data.indptr[rows_h], x.lens[rows_h]
            crow = np.zeros(x.B + 1, dtype=np.int64)
            np.cumsum(ln, out=crow[1:])
            take = np.repeat(starts - crow[:-1], ln) + np.arange(int(ln.sum()), dtype=np.int64)
            col = x.data.indices[take].astype(np.int32)
            host.append(torch.sparse_csr_tensor(torch.from_numpy(crow).pin_memory(), torch.from_numpy(col).pin_memory(),
                                                torch.ones(col.shape[0], dtype=torch.float32).pin_memory(), size=(x.B, x.N),
                                                check_invariants=False))
        h2d = float(np.mean([t.crow_indices().numel() * 8 + t.col_indices().numel() * 4 + t.values().numel() * 4 for t in host]))
        api = "VAETrainer.train_on_batch(pinned host CSR batch) -> loss floats"
    else:               # data parallel: the interaction CSR is resident on every rank; the step's input is its user ids
        x.trainer.set_interactions(x.csr)
        for s in range(KE):
            g0 = (s % x.n_batches) * x.Bg
            host.append(torch.from_numpy(x.order[g0 + rank * x.B:g0 + (rank + 1) * x.B].copy()).pin_memory())
        h2d = float(x.B * 4)
        api = "VAETrainer.train_on_batch(pinned host user-id batch into the resident CSR) -> loss floats"
    capg = x.cap_global if world > 1 else None
    for s in range(3):
        x.trainer.train_on_batch(host[s], b_global=x.Bg, nnz_cap_global=capg)
    barrier(dev, world)
    t = 0.0
    for s in range(KE):
        flush_buf.fill_(s & 0xFF)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        x.trainer.train_on_batch(host[s], b_global=x.Bg, nnz_cap_global=capg)     # returns python floats -> synchronises
        t += time.perf_counter() - t0
    (t,) = dist_max([t], dev, world)
    return {"value": KE * x.Bg / t, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 12, "steps": KE, "api": api,
            "timing": "wall clock around each call (H2D + captured step + D2H of 3 loss floats), max over ranks"}


def measure_eval(x, dev, world, rank, max_users=262144):
    """Full-ranking top-K + Recall/NDCG/HR (evaluate.py:243-265) at the training workload's shape, users sharded over ranks;
    metric sums are reduced over ranks before the means are formed."""
    from hvae_b200.dist import split_even
    from hvae_b200.evaluate import RecommendationEvaluator
    x.model.eval()
    ev = RecommendationEvaluator(x.model, x.csr, {}, {}, dev, batch_users=4096)
    n_eval = min(x.U, max_users)
    lo, hi = split_even(n_eval, world, rank)
    users = np.arange(lo, hi, dtype=np.int64)
    rel_ptr = np.arange(len(users) + 1, dtype=np.int64)
    rel_idx = x.data.test_items[users].astype(np.int32)
    kv = [5, 10, 20]
    w = min(len(users), 4096)
    ev.evaluate_users(users[:w], rel_ptr[:w + 1], rel_idx[:w], kv)
    barrier(dev, world)
    reps = 2
    t0 = time.perf_counter()
    for _ in range(reps):
        _, idx = ev.topk_users(users, min(max(kv), x.N))
        res, cnt = ev.metrics_from_topk(idx, rel_ptr, rel_idx, kv)    # host ids in, metric sums out (sync)
    barrier(dev, world)
    (t,) = dist_max([(time.perf_counter() - t0) / reps], dev, world)
    sums = torch.tensor([res[k][m] * cnt for k in kv for m in ("recall", "ndcg", "hit_ratio")] + [float(cnt)], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(sums)
    sums = sums.cpu().numpy()
    x.model.train()
    return {"metric": "eval_topk_users_per_sec", "value": n_eval / t, "unit": UNIT, "k_values": kv, "users": n_eval, "items": x.N,
            "sharding": "users" if world > 1 else "none", "ndcg@10": float(sums[4] / max(sums[-1], 1)), "recall@20": float(sums[6] / max(sums[-1], 1)),
            "users_evaluated": int(sums[-1]), "timing": "wall clock incl. H2D of user ids and D2H of metric sums, max over ranks"}


def dp_parity(x, args, dev, world, rank):
    """One optimisation step with INJECTED noise on two fresh copies of the model: data parallel over the ranks vs the same
    global batch on one GPU (every rank recomputes the latter).  -> relative differences of the loss and of the weights."""
    import torch.distributed as dist
    from hvae_b200.engine import Batch
    from hvae_b200.model import HybridVAE
    from hvae_b200.train import VAETrainer
    c = x.c
    sd = x.model.state_dict()
    Bg, B = x.Bg, x.B
    rows_g = x.order_dev[:Bg].contiguous()
    g = torch.Generator(device=dev).manual_seed(1234)
    keep = 1.0 - c["dropout"]
    noise_g = dict(masks=[(torch.rand(Bg, h, device=dev, generator=g) < keep).to(torch.uint8) for h in c["hidden_dims"]],
                   eps=torch.randn(Bg, c["latent_dim"], device=dev, generator=g),
                   pmask=(torch.rand(Bg, x.d, device=dev, generator=g) < keep).to(torch.uint8))
    out = {}
    models = []
    for mode in ("single", "dp"):
        torch.manual_seed(0)
        m = HybridVAE(x.N, np.zeros((x.N, x.d), dtype=np.float32), c["latent_dim"], c["hidden_dims"], c["dropout"], c["beta"], precision=args.precision)
        m.load_state_dict(sd)
        tr = VAETrainer(m, dev, lr=1e-3, use_cuda_graph=False)
        m.train()
        if mode == "single":
            cap = int(x.lens[x.order[:Bg]].sum())
            tr.train_step(Batch(x.csr, rows_g, Bg, max(1, cap)), noise_g)
            loss = np.array(tr.last_losses())
        else:
            tr.enable_data_parallel()
            lo, hi = rank * B, (rank + 1) * B
            nl = dict(masks=[mk[lo:hi].contiguous() for mk in noise_g["masks"]], eps=noise_g["eps"][lo:hi].contiguous(),
                      pmask=noise_g["pmask"][lo:hi].contiguous())
            b = Batch(x.csr, rows_g[lo:hi].contiguous(), B, max(1, int(x.lens[x.order[lo:hi]].sum())), b_global=Bg,
                      nnz_cap_global=int(x.lens[x.order[:Bg]].sum()))
            tr.train_step(b, nl, b_global=Bg)
            part = m.engine.loss_out.clone()
            dist.all_reduce(part)
            loss = part.cpu().numpy()
            out["exchange"] = m.engine.dist.exchange
        out[mode] = loss
        models.append(m)
    a, b = models[0].arena.data, models[1].arena.data
    pdiff = float((a - b).abs().max() / a.abs().max())
    ga, gb = models[0].engine.m, models[1].engine.m          # first Adam moment after one step = (1 - beta1) * clipped gradient
    gdiff = float((ga - gb).abs().max() / ga.abs().max())
    ldiff = float(np.max(np.abs(out["single"] - out["dp"]) / np.abs(out["single"])))
    pdiff, ldiff, gdiff = dist_max([pdiff, ldiff, gdiff], dev, world)
    del models
    gc.collect()
    torch.cuda.empty_cache()
    return {"loss_rel_diff": ldiff, "grad_max_rel_diff": gdiff, "param_max_rel_diff": pdiff,
            "note": "the first Adam step moves every weight by +-lr whatever the size of its gradient, so a last-bit difference of a "
                    "near-zero gradient entry shows up as 2*lr in param_max_rel_diff; grad_max_rel_diff is the meaningful number",
            "global_batch": Bg, "first_step_loss_single_gpu": float(out["single"][0]),
            "first_step_loss_data_parallel": float(out["dp"][0]), "exchange": out.get("exchange"),
            "what": "one step with injected noise: data-parallel over the ranks vs the same global batch on one GPU (max over ranks)"}


# ---- extras ----------------------------------------------------------------------------------------------------------
def extra_c2_train(args, dev, flush_buf, lib, fuse=None):
    """BASELINE.json configs[1] (All_Beauty shape, 512 users per step) on this rank's GPU alone.  fuse: HVAE_FUSE bit mask of the fused
    GEMM epilogues for this run (None = the engine's default), so that the line carries the measured reason why they are off."""
    a2 = argparse.Namespace(**vars(args))
    x = build_train("c2", a2, dev, 1, 0)
    if fuse is not None and x.model.engine.precision != "fp32":
        x.model.engine.fuse = int(fuse)
    r = measure_train(x, 20, 200, dev, 1, 0, flush_buf, lib)
    out = {"workload": workload_config("c2", x.c, 1)["workload"], "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"],
           "value_hot_l2": r["value_hot"], "gpu_launches_per_step": r["launches"] / 200, "n_gpus": 1, "steps": 200, "warmup": 20}
    if fuse is not None:
        out["HVAE_FUSE"] = int(x.model.engine.fuse)
    del x
    gc.collect()
    torch.cuda.empty_cache()
    return out


def extra_c5_sweep(args, dev, world, rank, epochs=3):
    """BASELINE.json configs[4]: 16 (latent_dim, hidden_dims, dropout, beta) configurations at the All_Beauty shape, each trained
    `epochs` epochs (early stopping, patience 3) + validation NDCG@10 under the 99-negative protocol -- the reference's
    run_grid_search loop (src/ml/tune.py:187-322).  Configurations are independent: placed round-robin on the ranks, no
    collective on the data path; the result dicts are gathered at the end (hvae_b200.tune.grid_search_core)."""
    from scipy.sparse import csr_matrix
    from hvae_b200.synth import CONFIGS, make_interactions, make_item_embeddings
    from hvae_b200.tune import grid_search_core
    c = CONFIGS["c2"]
    data = make_interactions(c["n_users"], c["n_items"], 0)
    E = make_item_embeddings(c["n_items"], c["emb_dim"], 0)
    train = data.scipy_csr()
    U = c["n_users"]
    val = csr_matrix((np.ones(U), (np.arange(U), data.test_items)), shape=train.shape)      # 1-hot validation rows (train.py:232,255)
    space = {"latent_dim": [64, 128], "hidden_dims": [[256], [512]], "dropout": [0.3, 0.5], "beta": [0.1, 0.2], "learning_rate": [1e-3]}
    torch.manual_seed(0)
    barrier(dev, world)
    t0 = time.perf_counter()
    out = grid_search_core(train, val, list(range(U)), list(range(U)), (np.arange(U), data.test_items.astype(np.int64)), E, space,
                           epochs_per_config=epochs, patience=3, batch_size=512, use_annealing=True, device=dev, seed=0,
                           precision=args.precision)
    torch.cuda.synchronize(dev)
    (dt,) = dist_max([time.perf_counter() - t0], dev, world)
    ok = [r for r in out["all_results"] if "error" not in r]
    steps = epochs * ((U + 511) // 512) * len(ok)
    gc.collect()
    torch.cuda.empty_cache()
    return {"metric": "grid_sweep_seconds", "value": dt, "unit": "s", "n_gpus": world, "configs": len(out["all_results"]),
            "failed": len(out["all_results"]) - len(ok), "epochs_per_config": epochs, "users": U, "items": c["n_items"],
            "train_users_per_sec_aggregate": steps * 512 / dt, "best_config": str(out["best_config"]), "best_ndcg@10": out["best_metric"],
            "placement": "configurations round-robin over the ranks, one process per GPU, no data-path collective",
            "timing": "wall clock of the whole sweep (16 trainings + 16 validation rankings), max over ranks"}


def extra_c4(args, dev, world, rank, pk, flush_buf):
    """BASELINE.json configs[3] shape: users scored against 1M items (d = 768), top-20 + Recall/NDCG/HR.  N > 1: E sharded by
    item over the ranks (hvae_b200.dist.ShardedEvaluator).  Weights / E are drawn on the device (the CPU initialisation of a
    1M x 600 layer is not the thing measured).  Also times the HBM-bound kernels at this shape."""
    import torch.distributed as dist
    from hvae_b200 import dist as hd
    from hvae_b200._cabi import p
    from hvae_b200.engine import Batch, DeviceCSR, Engine, Layout
    from hvae_b200.evaluate import _metric_tables
    from hvae_b200.synth import make_interactions
    N, d, K, U = 1_000_000, 768, 20, 262_144
    lay = Layout(N, d, 200, [600])
    g = torch.Generator(device=dev).manual_seed(0)           # same weights on every rank
    arena = torch.randn(lay.n_params, device=dev, generator=g) * 0.02
    lay.view(arena, "encoder.1.weight").fill_(1.0)
    E = torch.nn.functional.normalize(torch.randn(N, d, device=dev, generator=g), dim=1)
    eng = Engine(lay, arena, E, 0.5, "bf16")
    data = make_interactions(U, N, 0)
    csr = DeviceCSR.from_arrays(data.indptr, data.indices, None, N, dev)
    users = torch.arange(U, dtype=torch.int32, device=dev)
    rel_ptr = torch.arange(U + 1, dtype=torch.int64, device=dev)
    rel_idx = torch.from_numpy(data.test_items.astype(np.int32)).to(dev)
    kvals = [5, 10, 20]
    disc, idcg = _metric_tables(K)
    t = lambda v, dt: torch.as_tensor(np.asarray(v), dtype=dt, device=dev)
    kv, dd, ii = t(kvals, torch.int32), t(disc, torch.float64), t(idcg, torch.float64)
    out = torch.zeros(len(kvals) * 3 + 1, dtype=torch.float64, device=dev)
    wsd = torch.empty(148 * (len(kvals) * 3 + 1), dtype=torch.float64, device=dev)
    topk_all = torch.empty(U, K, dtype=torch.int32, device=dev)
    mask = torch.empty(U, 4, dtype=torch.int32, device=dev)
    sev = hd.ShardedEvaluator(eng, csr, K, tile=8192)

    def run():
        sev.topk(users, topk_all)
        eng.lib.hit_mask(p(topk_all), U, K, p(rel_ptr), p(rel_idx), p(mask), eng.stream)
        eng.lib.metrics_reduce(p(mask), p(rel_ptr), U, p(kv), len(kvals), p(dd), p(ii), p(wsd), p(out), eng.stream)

    run()
    barrier(dev, world)
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    barrier(dev, world)
    (ms,) = dist_max([e0.elapsed_time(e1) / reps], dev, world)
    # sharding + merge against the un-sharded kernel on the SAME user vectors (the last tile's all-gathered ones): the same
    # arithmetic per item, so the ids must be identical.  (Encoding a different number of users per launch changes the
    # split-K of the TF32 MLP GEMMs, i.e. the last bits of u: not a property of the sharding.)
    from hvae_b200 import tc
    with torch.no_grad():
        T = sev.tile
        v1 = torch.empty(T, K, dtype=torch.float32, device=dev)
        i1 = torch.empty(T, K, dtype=torch.int32, device=dev)
        tc.topk_bf16_from_ub(eng, Batch(csr, sev.rows, T, 1), sev.ub_all, K, True, 0, N, v1, i1)
    same = bool(torch.equal(i1, sev.out_idx))
    o = out.cpu().numpy()
    flops = 2.0 * U * N * d
    res = {"eval_c4": {"metric": "eval_topk_users_per_sec", "value": U / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "users": U, "items": N,
                       "d": d, "K": K, "ms": ms, "sharding": "items" if world > 1 else "none", "items_per_rank": sev.shard.hi - sev.shard.lo,
                       "aggregate_tflops": flops / (ms * 1e-3) / 1e12,
                       "frac_of_sustained_tc_peak_per_gpu": flops / (ms * 1e-3) / 1e12 / world / pk["tc_sustained"],
                       "ids_equal_unsharded": same, "ndcg@10": float(o[4] / max(o[-1], 1)),
                       "timing": "CUDA events, max over ranks: encoder + all-gather of user vectors + fused GEMM/top-K + all-gather of "
                                 "candidates + merge + metrics; one CUDA graph per 8,192-user tile"}}
    if rank == 0:      # kernel rooflines at the 1M-item shape (this GPU alone)
        res["kernels_1m_items"] = kernels_1m(eng, csr, users, dev, pk, flush_buf, data)
    del sev, eng, arena, E
    gc.collect()
    torch.cuda.empty_cache()
    return res


def kernels_1m(eng, csr, users, dev, pk, flush_buf, data):
    """gather (encoder layer 1 of an evaluation tile), fp32 top-K scan, fused tcgen05 LSE and top-K kernels: 1M items."""
    from hvae_b200._cabi import p
    from hvae_b200.engine import Batch
    lib, st, lay = eng.lib, eng.stream, eng.lay
    N, d, h = lay.N, lay.d, lay.hidden[0]
    ld1 = (h + 3) // 4 * 4
    out = {}

    def timeit(fn, reps=5):
        fn(); fn()
        torch.cuda.synchronize(dev)
        return float(np.median(timed_events(lambda i: fn(), reps, flush_buf, dev)))

    # 1. gather-sum + LayerNorm + GELU of 65,536 users (W1^T is [1M, 600] fp32)
    Bq = 65536
    rows = users[:Bq].contiguous()
    pre, act = torch.empty(Bq, ld1, device=dev), torch.empty(Bq, ld1, device=dev)
    mean, rstd = torch.empty(Bq, device=dev), torch.empty(Bq, device=dev)
    ms = timeit(lambda: lib.gather_ln_fwd(p(csr.indptr), p(csr.indices), None, p(rows), Bq, eng.P("encoder.0.weight"), ld1, h,
                                          eng.P("encoder.0.bias"), eng.P("encoder.1.weight"), eng.P("encoder.1.bias"), None, 1.0,
                                          p(pre), p(mean), p(rstd), p(act), st))
    nnz = float(np.diff(data.indptr)[:Bq].sum())
    gbytes = nnz * (ld1 * 4 + 4) + Bq * (2 * ld1 * 4 + 16)
    out["gather_ln_fwd"] = {"ms": ms, "bound": "hbm", "users": Bq, "achieved": gbytes / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                            "frac": gbytes / (ms * 1e-3) / 1e9 / pk["hbm"], "algorithmic_bytes": gbytes}
    del pre, act
    # 2. fp32 seen-mask + top-20 scan of 256 materialised score rows
    R, K = 256, 20
    S = torch.randn(R, N, device=dev)
    nc = int(lib.mask_topk_chunks(R, N))
    cv, ci = torch.empty(R, nc * K, device=dev), torch.empty(R, nc * K, dtype=torch.int32, device=dev)
    ov, oi = torch.empty(R, K, device=dev), torch.empty(R, K, dtype=torch.int32, device=dev)
    r256 = users[:R].contiguous()
    ms = timeit(lambda: lib.mask_topk(p(S), N, R, N, 0, p(csr.indptr), p(csr.indices), p(r256), 1, K, p(cv), p(ci), p(ov), p(oi), st))
    out["mask_topk"] = {"ms": ms, "bound": "hbm", "rows": R, "achieved": R * N * 4.0 / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                        "frac": R * N * 4.0 / (ms * 1e-3) / 1e9 / pk["hbm"], "algorithmic_bytes": R * N * 4.0}
    del S
    # 3. tcgen05 scoring kernels over the 1M items, 4,096 users
    B = 4096
    ld = (d + 7) // 8 * 8
    g = torch.Generator(device=dev).manual_seed(0)
    U = (torch.randn(B, ld, generator=g, device=dev) * 0.3).to(torch.bfloat16)
    Eb = eng.E_bf16
    ns = int(lib.tc_n_splits(B, N))
    ws, lse = torch.empty(2 * B * ns, device=dev), torch.empty(B, device=dev)
    ms = timeit(lambda: lib.tc_score_lse(p(U), ld, B, p(Eb), ld, N, d, p(lse), p(ws), st), 3)
    fl = 2.0 * B * N * d
    out["tc_score_lse"] = {"ms": ms, "bound": "tensor", "achieved": fl / (ms * 1e-3) / 1e12, "peak": pk["tc_sustained"], "unit": "TFLOP/s",
                           "frac": fl / (ms * 1e-3) / 1e12 / pk["tc_sustained"], "algorithmic_flops": fl}
    nst = int(lib.tc_topk_splits(B, N))
    cv, ci = torch.empty(B, nst * K, device=dev), torch.empty(B, nst * K, dtype=torch.int32, device=dev)
    r4k = users[:B].contiguous()
    ms = timeit(lambda: lib.tc_score_topk(p(U), ld, B, p(Eb), ld, N, d, 0, p(csr.indptr), p(csr.indices), p(r4k), K, p(cv), p(ci), st), 3)
    out["tc_score_topk"] = {"ms": ms, "bound": "tensor", "achieved": fl / (ms * 1e-3) / 1e12, "peak": pk["tc_sustained"], "unit": "TFLOP/s",
                            "frac": fl / (ms * 1e-3) / 1e12 / pk["tc_sustained"], "algorithmic_flops": fl, "K": K}
    return out


# ------------------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from hvae_b200 import _cabi
    pk = peaks()
    lib = _cabi.lib()
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    W, K = max(args.warmup, 3), args.steps

    x = build_train(args.workload, args, dev, world, rank, args.batch)
    parity = dp_parity(x, args, dev, world, rank) if world > 1 else None

    clocks = ClockSampler(local) if rank == 0 else None
    r = measure_train(x, W, K, dev, world, rank, flush_buf, lib, args.dump_outputs)
    clk = clocks.stop(*r["wall"]) if clocks else None
    kernels, span_avg, roofline = kernel_spans(x, W, K, flush_buf, pk, world, r["ms_per_step"], args)
    e2e = measure_e2e(x, K, dev, world, rank, flush_buf)
    ev_out = None if args.no_eval else measure_eval(x, dev, world, rank)
    exchange = x.model.engine.dist.exchange if world > 1 else None
    cfg = workload_config(args.workload, x.c, world)
    c_cpu, data_cpu, E_cpu = x.c, x.data, x.E
    x.trainer._graphs.clear()
    del x
    gc.collect()
    torch.cuda.empty_cache()

    extra = {"exchange": exchange, "dp_parity": parity, "precision": args.precision}
    if not args.no_extras:
        extra["c2_train"] = extra_c2_train(args, dev, flush_buf, lib)
        extra.update(extra_c4(args, dev, world, rank, pk, flush_buf))
        extra["c5_sweep"] = extra_c5_sweep(args, dev, world, rank)
        if world == 1:       # the same C2 step with every fused GEMM epilogue on (fewer launches, measured slower: DESIGN.md section 8)
            try:
                extra["c2_train_fused_epilogues"] = extra_c2_train(args, dev, flush_buf, lib, fuse=63)
            except Exception as e:
                extra["c2_train_fused_epilogues"] = {"unavailable": str(e)[:200]}

    if rank != 0:
        return _finish(world, dist, dev)

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            extra["torch_cuda_eager"] = torch_cuda_eager(c_cpu, data_cpu, E_cpu, dev)
        except Exception as e:       # context number only (e.g. out of memory on a smaller GPU)
            extra["torch_cuda_eager"] = {"unavailable": str(e)[:200]}
        ref = CpuReference(c_cpu, data_cpu, E_cpu)
        Bs = ref.pick_sample(args.cpu_seconds / 3.0, c_cpu["batch"])
        ref.step(Bs)
        n, secs = 0, 0.0
        while n < 2 or (secs < args.cpu_seconds and n < 50):
            secs += ref.step(Bs)
            n += 1
        cpu = {"value": n * Bs / secs, "unit": UNIT, "cores": ref.threads, "kind": "port",
               "sample": f"{n} steps of {Bs} users each ({secs:.1f} s; a bounded sample of the {c_cpu['batch']}-user batch of the same workload) "
                         "through oracle/hvae_oracle.py (the reference's train loop incl. per-row densification)"}

    line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic", "config": cfg,
            "e2e": e2e, "gpu_launches": r["launches"], "roofline": roofline, "cpu_baseline": cpu, "clocks": clk,
            "value_hot_l2": r["value_hot"], "ms_per_step_hot_l2": r["ms_hot"], "kernels": kernels, "spans_ms": span_avg, "eval": ev_out,
            "cuda_graph": not args.no_graph, "extra": extra}
    print(json.dumps(line), flush=True)
    _finish(world, dist, dev)


def _finish(world, dist, dev):
    """Multi-rank exit.  The captured graphs that hold NCCL work were dropped above; tear the communicator down, but never wait
    for it longer than a few seconds (a rank stuck in destroy_process_group() would stall the whole job)."""
    if world == 1:
        return
    torch.cuda.synchronize(dev)
    sys.stdout.flush()
    sys.stderr.flush()
    th = threading.Thread(target=dist.destroy_process_group, daemon=True)
    th.start()
    th.join(timeout=15.0)
    if th.is_alive():
        os._exit(0)


if __name__ == "__main__":
    main()

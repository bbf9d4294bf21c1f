"""Cost of Gumbel-top-K sampling in the fused top-K kernels (hvae_tc_score_topk_sampled, hvae_mask_topk_sampled).

    python tools/bench_topk_sampled.py --out DIR [--seconds 1.0] [--train-steps 40]

Per catalogue (N in {200k, 1M}, d = 768) a bf16 HybridVAE is trained for a few steps on synthetic interactions, and the
user vectors of 4,096 of its users are scored: how much sampling costs depends on how far the scores spread against tau,
and random vectors would not spread like a model's.  For K in {20, 100} these launches are timed with CUDA events,
back to back, variants alternating round by round after a warm-up:
  plain        the filtered entry point without allow-sets (seen items masked), i.e. the unsampled launch
  tau_0.25/1/4 the sampled entry point, every row sampled at that temperature
for the tcgen05 kernel (fused scoring, no [B, N] scores) and for the fp32 scan over materialised scores (the GEMM that
materialises them is not timed).  L2 is not flushed: the bf16 item table and the fp32 score rows are larger than the
126 MB L2.  "pass_fraction" is the share of (row, item) columns whose pruning bound s / tau + 16.64 reaches the row's
final K-th key, over 256 rows: the running threshold only rises to that key, so the kernels test at least this share.
Writes DIR/topk_sampled.json with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "recommendation-system_b200"))
from hvae_b200 import _cabi, tc  # noqa: E402
from hvae_b200.engine import Batch, DeviceCSR  # noqa: E402
from hvae_b200.model import HybridVAE  # noqa: E402
from hvae_b200.synth import make_interactions, make_item_embeddings  # noqa: E402
from hvae_b200.train import VAETrainer  # noqa: E402

G_MAX = 16.64
TAUS = (0.25, 1.0, 4.0)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_and_max_sm_clock"] = "not available"
    return info


def trained_user_vectors(N, d, B, steps, dev):
    """fp32 and bf16 user vectors of B users of a bf16 HybridVAE trained for `steps` steps, and their seen-item CSR."""
    n_users = 16 * B
    data = make_interactions(n_users, N, 0)
    torch.manual_seed(0)
    model = HybridVAE(N, make_item_embeddings(N, d, 0), 200, [600], 0.5, 0.2, precision="bf16").to(dev)
    trainer = VAETrainer(model, dev, lr=1e-3, use_cuda_graph=False)
    csr = DeviceCSR.from_arrays(data.indptr, data.indices, None, N, dev)
    lens = np.diff(data.indptr)
    rng = np.random.default_rng(0)
    model.train()
    for _ in range(steps):
        rows = np.sort(rng.choice(n_users, B, replace=False)).astype(np.int32)
        trainer.train_step(Batch(csr, torch.as_tensor(rows, device=dev), B, int(lens[rows].sum())))
    model.eval()
    eng = model.engine
    rows = torch.arange(B, dtype=torch.int32, device=dev)
    with torch.no_grad():
        batch = Batch(csr, rows, B, int(lens[:B].sum()))
        u = eng.user_vectors(batch).clone()
        ub = tc.user_vectors_bf16(eng, u, B).clone()
    return eng, csr, u, ub, [float(x) for x in trainer.last_losses()]


def time_variants(variants, seconds, rounds):
    reps = {}
    for name, fn in variants.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        reps[name] = max(3, int(seconds / rounds / ((time.perf_counter() - t0) / 5)))
    times = {name: [] for name in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps[name]):
                fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / reps[name])
    return times, reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--seconds", type=float, default=1.0, help="timed seconds per variant and shape (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--train-steps", type=int, default=40)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs the GPU"
    dev = torch.device("cuda:0")
    lib = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    B, d = 4096, 768
    info = gpu_info()
    results = []
    for N in (200_000, 1_000_000):
        eng, csr, u, ub, losses = trained_user_vectors(N, d, B, a.train_steps, dev)
        ld8 = ub.shape[1]
        Eb, Ef = eng.E_bf16, eng.E
        S = torch.empty(B, N, device=dev)                       # fp32 scores for the scan (4 GB / 16 GB)
        for r0 in range(0, B, 512):
            eng.gemm(512, N, d, u.data_ptr() + 4 * r0 * u.stride(0), u.stride(0), 1, Ef.data_ptr(), 1, d, S[r0:].data_ptr(), N)
        torch.cuda.synchronize()
        spread = S[:256].std(dim=1)
        seeds = torch.arange(B, dtype=torch.int64, device=dev) * 7919 + 1
        for K in (20, 100):
            ns = int(lib.tc_topk_splits(B, N))
            cv = torch.empty(B, ns * K, device=dev)
            ci = torch.empty(B, ns * K, dtype=torch.int32, device=dev)
            nc = int(lib.mask_topk_chunks(B, N))
            sv = torch.empty(B, nc * K, device=dev)
            si = torch.empty(B, nc * K, dtype=torch.int32, device=dev)
            ov = torch.empty(B, K, device=dev)
            oi = torch.empty(B, K, dtype=torch.int32, device=dev)
            tc_args = (ub.data_ptr(), ld8, B, Eb.data_ptr(), ld8, N, d, 0, csr.indptr.data_ptr(), csr.indices.data_ptr(), None, None, 0,
                       None)
            sc_args = (S.data_ptr(), N, B, N, 0, csr.indptr.data_ptr(), csr.indices.data_ptr(), None, 1, None, 0, None)
            inv = {t: torch.full((B,), 1.0 / t, dtype=torch.float32, device=dev) for t in TAUS}

            def tc_plain():
                lib.tc_score_topk_filtered(*tc_args, K, cv.data_ptr(), ci.data_ptr(), st)

            def tc_sampled(t):
                return lambda: lib.tc_score_topk_sampled(*tc_args, inv[t].data_ptr(), seeds.data_ptr(), K, cv.data_ptr(), ci.data_ptr(), st)

            def sc_plain():
                lib.mask_topk_filtered(*sc_args, K, sv.data_ptr(), si.data_ptr(), ov.data_ptr(), oi.data_ptr(), st)

            def sc_sampled(t):
                return lambda: lib.mask_topk_sampled(*sc_args, inv[t].data_ptr(), seeds.data_ptr(), K, sv.data_ptr(), si.data_ptr(),
                                                     ov.data_ptr(), oi.data_ptr(), st)
            for kernel, plain, sampled in (("tcgen05", tc_plain, tc_sampled), ("fp32_scan", sc_plain, sc_sampled)):
                variants = {"plain": plain, **{f"tau_{t:g}": sampled(t) for t in TAUS}}
                times, reps = time_variants(variants, a.seconds, a.rounds)
                med = {n: float(np.median(v)) for n, v in times.items()}
                row = {"kernel": kernel, "B": B, "N": N, "d": d, "K": K, "ms_median": med,
                       "ms_min": {n: float(np.min(v)) for n, v in times.items()},
                       "ms_max": {n: float(np.max(v)) for n, v in times.items()}, "launches_per_round": reps,
                       "ratio_to_plain": {n: med[n] / med["plain"] for n in med}}
                results.append(row)
                print(json.dumps(row), flush=True)
            # pruning: share of columns whose bound reaches the final K-th key (keys of the scan's last draw at each tau)
            frac = {}
            for t in TAUS:
                sc_sampled(t)()
                kth = ov[:256, K - 1:K]
                frac[f"tau_{t:g}"] = float(((S[:256] / t + G_MAX) >= kth).float().mean())
            row = {"N": N, "K": K, "pass_fraction": frac, "score_std_median": float(spread.median()), "train_losses": losses}
            results.append(row)
            print(json.dumps(row), flush=True)
        del S, eng
        torch.cuda.empty_cache()
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    doc = {"gpu": info, "l2_flushed": False, "rounds": a.rounds, "seconds_per_variant": a.seconds, "train_steps": a.train_steps,
           "timed": "top-K launches only (no merge, no GEMM), CUDA events, variants alternated per round", "results": results}
    (out / "topk_sampled.json").write_text(json.dumps(doc, indent=1))
    print(json.dumps(doc["gpu"]))


if __name__ == "__main__":
    main()

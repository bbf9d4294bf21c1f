"""Cost of item allow-sets and exclusion lists in the fused tcgen05 top-K kernel (hvae_tc_score_topk_filtered).

    python tools/bench_topk_filtered.py --out DIR [--parent-lib path/to/libhvae_b200.so] [--seconds 1.5]

Per shape (B in {256, 4096}, N in {200k, 1M}, d = 768, K in {20, 100}) the variants are timed with CUDA events around
back-to-back launches of the scoring kernel alone (the small merge launch is left out):
  unfiltered      hvae_tc_score_topk (seen items of ~20 per row masked)
  parent          the same entry point of another build of the library (--parent-lib), to show it did not move
  allow_100/10/1  the filtered kernel, four bitmaps with that fraction of the catalogue mixed over the rows
  exclude_50      the unfiltered kernel with 50 extra excluded items per row folded into the mask CSR
The variants alternate round by round; every shape is warmed first.  L2 is not flushed between launches: the bf16 item
table (>= 300 MB) is larger than the 126 MB L2, so every launch streams it from HBM.  Writes DIR/topk_filtered.json with
the GPU's name and power limit read in the same run.
"""
import argparse
import ctypes
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "recommendation-system_b200"))
from hvae_b200 import _cabi  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_and_max_sm_clock"] = "not available"
    return info


def parent_topk(path):
    dll = ctypes.CDLL(str(path))
    fn = dll.hvae_tc_score_topk
    V, I = ctypes.c_void_p, ctypes.c_int
    fn.argtypes = [V, I, I, V, I, I, I, I, V, V, V, I, V, V, V]
    fn.restype = I

    def call(*args):
        if fn(*args):
            raise RuntimeError(f"hvae_tc_score_topk of {path}: {dll.hvae_last_error().decode()}")
    dll.hvae_last_error.restype = ctypes.c_char_p
    return call


def csr(rows, dev):
    indptr = np.zeros(len(rows) + 1, dtype=np.int64)
    indptr[1:] = np.cumsum([len(r) for r in rows])
    return torch.as_tensor(indptr, device=dev), torch.as_tensor(np.concatenate(rows).astype(np.int32), device=dev)


def bitmaps(N, frac, F, rng, dev):
    words = (N + 31) // 32
    bits = rng.random((F, words * 32)) < frac
    bits[:, N:] = False
    return torch.as_tensor(np.packbits(bits, axis=1, bitorder="little").view(np.int32), device=dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--seconds", type=float, default=1.5, help="timed seconds per variant and shape (split over the rounds)")
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs the GPU"
    dev = torch.device("cuda:0")
    lib = _cabi.lib()
    par = parent_topk(a.parent_lib) if a.parent_lib else None
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(0)
    d, F = 768, 4
    info = gpu_info()
    results = []
    Nmax = 1_000_000
    Ef = torch.nn.functional.normalize(torch.randn(Nmax, d, device=dev), dim=1)
    Eb = Ef.to(torch.bfloat16)
    del Ef
    for B in (256, 4096):
        Ub = (torch.randn(B, d, device=dev) * 0.4).to(torch.bfloat16)
        aor = torch.as_tensor((np.arange(B) % F).astype(np.int32), device=dev)
        for N in (200_000, 1_000_000):
            seen = [np.unique(rng.integers(0, N, 20)) for _ in range(B)]
            m_seen = csr(seen, dev)
            m_excl = csr([np.union1d(s, rng.choice(N, 50, replace=False)) for s in seen], dev)
            allow = {f: bitmaps(N, f, F, rng, dev) for f in (1.0, 0.1, 0.01)}
            for K in (20, 100):
                ns = int(lib.tc_topk_splits(B, N))
                cv = torch.empty(B, ns * K, device=dev)
                ci = torch.empty(B, ns * K, dtype=torch.int32, device=dev)
                common = (Ub.data_ptr(), d, B, Eb.data_ptr(), d, N, d, 0)

                def unf(m, fn=lib.tc_score_topk):
                    return lambda: fn(*common, m[0].data_ptr(), m[1].data_ptr(), None, K, cv.data_ptr(), ci.data_ptr(), st)

                def filt(bm):
                    return lambda: lib.tc_score_topk_filtered(*common, m_seen[0].data_ptr(), m_seen[1].data_ptr(), None, bm.data_ptr(),
                                                              bm.stride(0), aor.data_ptr(), K, cv.data_ptr(), ci.data_ptr(), st)
                variants = {"unfiltered": unf(m_seen), "allow_100": filt(allow[1.0]), "allow_10": filt(allow[0.1]),
                            "allow_1": filt(allow[0.01]), "exclude_50": unf(m_excl)}
                if par is not None:
                    variants["parent"] = unf(m_seen, par)
                # warm every variant and size the launch count of a round from one timed launch
                reps = {}
                for name, fn in variants.items():
                    for _ in range(3):
                        fn()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(5):
                        fn()
                    torch.cuda.synchronize()
                    one = (time.perf_counter() - t0) / 5
                    reps[name] = max(3, int(a.seconds / a.rounds / one))
                times = {name: [] for name in variants}
                for _ in range(a.rounds):
                    for name, fn in variants.items():
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(reps[name]):
                            fn()
                        e1.record()
                        e1.synchronize()
                        times[name].append(e0.elapsed_time(e1) / reps[name])
                med = {n: float(np.median(t)) for n, t in times.items()}
                row = {"B": B, "N": N, "d": d, "K": K, "ms_median": med,
                       "ms_min": {n: float(np.min(t)) for n, t in times.items()},
                       "ms_max": {n: float(np.max(t)) for n, t in times.items()},
                       "launches_per_round": reps,
                       "ratio_to_unfiltered": {n: med[n] / med["unfiltered"] for n in med}}
                results.append(row)
                print(json.dumps(row), flush=True)
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    doc = {"gpu": info, "l2_flushed": False, "rounds": a.rounds, "seconds_per_variant": a.seconds,
           "timed": "hvae_tc_score_topk(_filtered) launches only, CUDA events, variants alternated per round", "results": results}
    (out / "topk_filtered.json").write_text(json.dumps(doc, indent=1))
    print(json.dumps(doc["gpu"]))


if __name__ == "__main__":
    main()

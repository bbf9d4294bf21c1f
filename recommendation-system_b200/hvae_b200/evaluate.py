"""Drop-in evaluator: Recall/NDCG/HR@K, RecommendationEvaluator, load_model_from_checkpoint
(reference src/ml/evaluate.py).

The reference scores one user at a time (densify -> five M=1 linears -> D2H of N scores -> NumPy argsort,
evaluate.py:125-147).  Here users are scored in batches on the device: encoder(mu) -> projection -> score
tiles -> seen-item mask -> per-user warp top-K -> hit mask -> metric sums; only K indices per user (or
3*|k_values| sums) leave the GPU.  Ties are ordered (score desc, index desc), i.e. what a stable
argsort()[::-1] gives; the reference's default argsort is unstable, so its order on exact ties is undefined.
"""
from __future__ import annotations

import logging
import threading
from pathlib import Path

import numpy as np
import pandas as pd
import torch
from scipy.sparse import csr_matrix

from . import data as _data
from ._cabi import p
from .engine import Batch, DeviceCSR
from .model import HybridVAE, create_hybrid_vae

logger = logging.getLogger(__name__)
_build_input_matrix = _data.build_input_matrix


# -- metric functions on host arrays, same contract as src/ml/evaluate.py:32-54 --------------------------------
def recall_at_k(recommended: np.ndarray, relevant: np.ndarray, k: int) -> float:
    if len(relevant) == 0:
        return 0.0
    return len(np.intersect1d(recommended[:k], relevant)) / len(relevant)


def ndcg_at_k(recommended: np.ndarray, relevant: np.ndarray, k: int) -> float:
    if len(relevant) == 0:
        return 0.0
    rel = set(np.asarray(relevant).tolist())
    dcg = sum(1.0 / np.log2(i + 2) for i, item in enumerate(recommended[:k]) if item in rel)
    idcg = sum(1.0 / np.log2(i + 2) for i in range(min(len(relevant), k)))
    return dcg / idcg if idcg > 0 else 0.0


def hit_ratio_at_k(recommended: np.ndarray, relevant: np.ndarray, k: int) -> float:
    if len(relevant) == 0:
        return 0.0
    return 1.0 if len(np.intersect1d(recommended[:k], relevant)) > 0 else 0.0


def _aggregate_metrics(all_metrics: dict, k_values) -> dict:
    return {k: {m: float(np.mean(all_metrics[k][m])) if all_metrics[k][m] else 0.0 for m in ("recall", "ndcg", "hit_ratio")}
            for k in k_values}


def _metric_tables(kmax):
    disc = 1.0 / np.log2(np.arange(kmax, dtype=np.float64) + 2.0)
    idcg = np.concatenate([[1.0], np.cumsum(disc)])     # idcg[n] = sum_{i<n} disc[i]; idcg[0] unused (guarded)
    return disc, idcg


class RecommendationEvaluator:
    """src/ml/evaluate.py:106-265, batched on the device."""

    def __init__(self, model: HybridVAE, interaction_matrix: csr_matrix, user_to_idx: dict, item_to_idx: dict,
                 device: torch.device, batch_users: int = 4096):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("hvae_b200.RecommendationEvaluator needs a CUDA device (there is no CPU fallback)")
        self.model = model.to(device)
        self.model.eval()
        self.device = device
        self.interaction_matrix = interaction_matrix
        self.user_to_idx, self.item_to_idx = user_to_idx, item_to_idx
        self.n_items = interaction_matrix.n_items if isinstance(interaction_matrix, DeviceCSR) else interaction_matrix.shape[1]
        self.batch_users = batch_users
        self._csr = interaction_matrix if isinstance(interaction_matrix, DeviceCSR) else DeviceCSR.from_scipy(interaction_matrix, device)
        # (int32 [F, ceil(n_items / 32)] item bitmaps of the named filters, name -> row): replaced as a whole, never written in
        # place, so a top-K call that took the pair keeps a consistent table while another thread registers a filter
        self._filters: tuple = (None, {})
        self._filters_lock = threading.Lock()

    # -- item filters ------------------------------------------------------------------------------------------------
    def add_item_filter(self, name: str, item_indices) -> None:
        """Registers (or replaces) the allow-set `name`: topk_users(..., item_filter=name) then only returns these items."""
        idx = np.asarray(item_indices, dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() >= self.n_items):
            raise ValueError(f"item filter {name!r}: item indices must lie in [0, {self.n_items})")
        words = (self.n_items + 31) // 32
        bits = np.zeros(words * 32, dtype=bool)
        bits[idx] = True
        row = torch.as_tensor(np.packbits(bits, bitorder="little").view(np.int32), device=self.device)   # bit i of word w: item 32w + i
        with self._filters_lock:
            table, rows = self._filters
            if name in rows:
                table = table.clone()
                table[rows[name]] = row
            else:
                rows = {**rows, name: 0 if table is None else table.shape[0]}
                table = row[None] if table is None else torch.cat([table, row[None]])
            self._filters = (table, rows)

    @staticmethod
    def _allow_of_row(item_filter, n, filter_row):
        """-> int32 [n] bitmap rows (-1 = unrestricted) on the host, or None when no user is restricted."""
        names = [item_filter] * n if item_filter is None or isinstance(item_filter, str) else list(item_filter)
        if len(names) != n:
            raise ValueError(f"item_filter: {len(names)} entries for {n} users")
        if all(nm is None for nm in names):
            return None
        for nm in names:
            if nm is not None and (not isinstance(nm, str) or nm not in filter_row):
                raise ValueError(f"unknown item filter {nm!r}")
        return np.array([-1 if nm is None else filter_row[nm] for nm in names], dtype=np.int32)

    def _mask_csr(self, rows, excl, exclude_seen):
        """Sorted union per batch row of the user's seen items (exclude_seen) and the row's exclusion list, built on the device:
        -> (indptr int64 [n+1], indices int32)."""
        n, N, dev = rows.shape[0], self.n_items, self.device
        keys = []
        if exclude_seen:
            start, end = self._csr.indptr[rows.long()], self._csr.indptr[rows.long() + 1]
            cnt = end - start
            row_of = torch.repeat_interleave(torch.arange(n, device=dev), cnt)
            pos = torch.arange(int(cnt.sum()), device=dev) - torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
            keys.append(row_of * N + self._csr.indices[start[row_of] + pos].long())
        lens = [len(e) for e in excl]
        if sum(lens):
            ex = torch.as_tensor(np.concatenate([np.asarray(e, dtype=np.int64).reshape(-1) for e in excl]), device=dev)
            keys.append(torch.repeat_interleave(torch.arange(n, device=dev), torch.as_tensor(lens, device=dev)) * N + ex)
        key = torch.unique(torch.cat(keys)) if keys else torch.empty(0, dtype=torch.int64, device=dev)   # sorted
        indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        indptr[1:] = torch.cumsum(torch.bincount(key // N, minlength=n), 0)
        return indptr, (key % N).to(torch.int32)

    # -- batched primitives ----------------------------------------------------------------------------------------
    def topk_users(self, user_indices, top_k: int, exclude_seen: bool = True, *, item_filter=None, exclude=None):
        """(values [n,K] f32, indices [n,K] int32) device tensors for the given users.

        item_filter: the name of a filter registered with add_item_filter, or one name (or None) per user: that user only gets
        items of the filter.  exclude: one array of item indices per user, left out on top of the seen items.  A user with
        fewer than K admissible items gets (-inf, -1) in the remaining slots."""
        users = torch.as_tensor(np.asarray(user_indices, dtype=np.int32), device=self.device)
        if item_filter is not None or exclude is not None:
            return self._topk_filtered(users, top_k, exclude_seen, item_filter, exclude)
        eng = self.model.engine
        from . import tc
        if eng.precision != "fp32" and exclude_seen and top_k <= tc.MAX_K_REG and users.shape[0] >= 2 * self.batch_users:
            # long user lists: the tile (encoder -> fused GEMM + seen mask + top-K -> merge) is captured once as a CUDA graph and
            # replayed per tile (dist.ShardedEvaluator with a single shard), instead of ~15 eager launches per tile
            key = lambda: (top_k, self.batch_users, eng.arena.data_ptr(), eng.E_bf16.data_ptr(), eng.ws.generation)
            if getattr(self, "_tile_key", None) != key():
                from .dist import ShardedEvaluator
                self._tile_eval, self._tile_key = ShardedEvaluator(eng, self._csr, top_k, tile=self.batch_users, sharded=False), None
            out_v = torch.empty(users.shape[0], top_k, dtype=torch.float32, device=self.device)
            out_i = self._tile_eval.topk(users, None, out_v)
            self._tile_key = key()          # (after the first tile: it may have grown the workspace the captured graph points into)
            return out_v, out_i
        vals, idxs = [], []
        with torch.no_grad():
            for s in range(0, users.shape[0], self.batch_users):
                rows = users[s:s + self.batch_users].contiguous()
                v, i = eng.topk(Batch(self._csr, rows, rows.shape[0], 1), top_k, exclude_seen)
                vals.append(v)
                idxs.append(i)
        if not vals:
            return (torch.empty(0, top_k, device=self.device), torch.empty(0, top_k, dtype=torch.int32, device=self.device))
        return torch.cat(vals), torch.cat(idxs)

    def _topk_filtered(self, users, top_k, exclude_seen, item_filter, exclude):
        n = users.shape[0]
        with self._filters_lock:
            table, filter_row = self._filters
        aor = self._allow_of_row(item_filter, n, filter_row)
        if exclude is not None:
            exclude = list(exclude)
            if len(exclude) != n:
                raise ValueError(f"exclude: {len(exclude)} lists for {n} users")
            for e in exclude:
                e = np.asarray(e).reshape(-1)
                if e.size and (e.min() < 0 or e.max() >= self.n_items):
                    raise ValueError(f"exclude: item indices must lie in [0, {self.n_items})")
        aor_d = None if aor is None else torch.as_tensor(aor, device=self.device)
        eng = self.model.engine
        vals, idxs = [], []
        with torch.no_grad():
            for s in range(0, n, self.batch_users):
                rows = users[s:s + self.batch_users].contiguous()
                mask = None if exclude is None else self._mask_csr(rows, exclude[s:s + rows.shape[0]], exclude_seen)
                allow = None if aor_d is None else (table, aor_d[s:s + rows.shape[0]].contiguous())
                v, i = eng.topk(Batch(self._csr, rows, rows.shape[0], 1), top_k, exclude_seen, mask=mask, allow=allow)
                vals.append(v)
                idxs.append(i)
        if not vals:
            return (torch.empty(0, top_k, device=self.device), torch.empty(0, top_k, dtype=torch.int32, device=self.device))
        return torch.cat(vals), torch.cat(idxs)

    def metrics_from_topk(self, topk_idx: torch.Tensor, rel_ptr: np.ndarray, rel_idx: np.ndarray, k_values):
        """Recall/NDCG/HR sums over rows with >=1 relevant item, reduced on the device (fixed order, float64)."""
        eng = self.model.engine
        n, K = topk_idx.shape
        nk = len(k_values)
        disc, idcg = _metric_tables(K)
        dev = self.device
        t = lambda a, dt: torch.as_tensor(np.asarray(a), dtype=dt, device=dev)
        rp, ri = t(rel_ptr, torch.int64), t(rel_idx, torch.int32)
        mask = torch.empty(max(n, 1), 4, dtype=torch.int32, device=dev)
        out = torch.zeros(nk * 3 + 1, dtype=torch.float64, device=dev)
        wsd = torch.empty(148 * (nk * 3 + 1), dtype=torch.float64, device=dev)
        kv, dd, ii = t(list(k_values), torch.int32), t(disc, torch.float64), t(idcg, torch.float64)   # keep alive until the sync
        eng.lib.hit_mask(p(topk_idx), n, K, p(rp), p(ri), p(mask), eng.stream)
        eng.lib.metrics_reduce(p(mask), p(rp), n, p(kv), nk, p(dd), p(ii), p(wsd), p(out), eng.stream)
        o = out.cpu().numpy()
        cnt = o[-1]
        res = {}
        for q, k in enumerate(k_values):
            res[k] = {m: float(o[q * 3 + j] / cnt) if cnt > 0 else 0.0 for j, m in enumerate(("recall", "ndcg", "hit_ratio"))}
        return res, int(cnt)

    # -- reference API -----------------------------------------------------------------------------------------------
    def _get_user_scores(self, user_idx: int) -> np.ndarray:
        """All-item scores of one user as a host array (src/ml/evaluate.py:125-135)."""
        eng = self.model.engine
        rows = torch.tensor([user_idx], dtype=torch.int32, device=self.device)
        with torch.no_grad():
            u = eng.user_vectors(Batch(self._csr, rows, 1, 1))
            return eng.scores_dense(u, 1)[0].cpu().numpy()

    def get_user_recommendations(self, user_idx: int, top_k: int = 100, exclude_seen: bool = True):
        """(indices int64 [k], scores f32 [k]) -- src/ml/evaluate.py:137-147."""
        k = min(top_k, self.n_items)
        v, i = self.topk_users([user_idx], k, exclude_seen)
        return i[0].cpu().numpy().astype(np.int64), v[0].cpu().numpy()

    def evaluate_user(self, user_id: str, test_items: list, k_values=None) -> dict:
        """src/ml/evaluate.py:217-241."""
        k_values = k_values or [5, 10, 20]
        if user_id not in self.user_to_idx:
            return {}
        test_indices = np.array([self.item_to_idx[i] for i in test_items if i in self.item_to_idx])
        if len(test_indices) == 0:
            return {}
        rec, _ = self.get_user_recommendations(self.user_to_idx[user_id], top_k=max(k_values))
        return {k: {"recall": recall_at_k(rec, test_indices, k), "ndcg": ndcg_at_k(rec, test_indices, k),
                    "hit_ratio": hit_ratio_at_k(rec, test_indices, k)} for k in k_values}

    def evaluate_dataset(self, test_df: pd.DataFrame, k_values=None) -> dict:
        """Full-ranking protocol, src/ml/evaluate.py:243-265."""
        k_values = k_values or [5, 10, 20]
        test_by_user = test_df.groupby("user_id")["asin"].apply(list).to_dict()
        users, rel_ptr, rel_idx = [], [0], []
        for user_id, items in test_by_user.items():
            if user_id not in self.user_to_idx:
                continue
            ti = [self.item_to_idx[i] for i in items if i in self.item_to_idx]
            if not ti:
                continue
            users.append(self.user_to_idx[user_id])
            rel_idx.extend(ti)
            rel_ptr.append(len(rel_idx))
        return self.evaluate_users(np.asarray(users, dtype=np.int64), np.asarray(rel_ptr, dtype=np.int64),
                                   np.asarray(rel_idx, dtype=np.int32), k_values)[0]

    def evaluate_users(self, users, rel_ptr, rel_idx, k_values):
        """Array form of evaluate_dataset: users [n], relevant items CSR (rel_ptr [n+1], rel_idx)."""
        kmax = min(max(k_values), self.n_items)
        _, idx = self.topk_users(users, kmax)
        res, cnt = self.metrics_from_topk(idx, rel_ptr, rel_idx, list(k_values))
        logger.info("Evaluated %d users", cnt)
        return res, idx

    # -- 99-negative protocol (the reference's default CLI protocol, evaluate.py:149-215) ---------------------------
    def evaluate_user_with_negatives(self, user_idx: int, test_item_idx: int, n_negatives: int = 99, k_values=None):
        k_values = k_values or [5, 10, 20]
        seen = self.interaction_matrix[user_idx].indices if not isinstance(self.interaction_matrix, DeviceCSR) else \
            self._csr.indices[self._csr.indptr[user_idx]:self._csr.indptr[user_idx + 1]].cpu().numpy()
        mask = np.ones(self.n_items, dtype=bool)
        mask[list(set(seen))] = False
        mask[test_item_idx] = False
        available = np.where(mask)[0]
        negatives = available if len(available) < n_negatives else np.random.choice(available, n_negatives, replace=False)
        candidates = np.concatenate([[test_item_idx], negatives])
        scores = self._get_user_scores(user_idx)
        ranked = candidates[np.argsort(scores[candidates], kind="stable")[::-1]]
        relevant = np.array([test_item_idx])
        return {k: {"recall": recall_at_k(ranked, relevant, k), "ndcg": ndcg_at_k(ranked, relevant, k),
                    "hit_ratio": hit_ratio_at_k(ranked, relevant, k)} for k in k_values}

    def evaluate_dataset_with_negatives(self, test_df: pd.DataFrame, n_negatives: int = 99, k_values=None, seed=None) -> dict:
        """Batched on the device: per (user, test item) row, 99 unseen negatives are sampled on the host
        (numpy, like the reference; seedable here), the 100 candidate scores come from one gather-dot launch."""
        from . import sampling
        k_values = k_values or [5, 10, 20]
        users, tests = [], []
        for user_id, item_id in zip(test_df["user_id"].values, test_df["asin"].values):
            if user_id in self.user_to_idx and item_id in self.item_to_idx:
                users.append(self.user_to_idx[user_id])
                tests.append(self.item_to_idx[item_id])
        if not users:
            return _aggregate_metrics({k: {"recall": [], "ndcg": [], "hit_ratio": []} for k in k_values}, k_values)
        return sampling.evaluate_with_negatives(self, np.asarray(users), np.asarray(tests), n_negatives, list(k_values), seed)


def load_model_from_checkpoint(checkpoint_path: str, item_embeddings: np.ndarray, device: torch.device,
                               precision: str | None = None) -> HybridVAE:
    """src/ml/evaluate.py:273-291: reads `model_config` + `model_state_dict` of a reference-layout checkpoint."""
    checkpoint = torch.load(checkpoint_path, map_location="cpu", weights_only=False)
    cfg = checkpoint["model_config"]
    model = create_hybrid_vae(n_items=cfg["n_items"], item_embeddings=item_embeddings, latent_dim=cfg["latent_dim"],
                              hidden_dims=cfg.get("hidden_dims"), dropout=cfg.get("dropout", 0.5), beta=cfg.get("beta", 0.2),
                              precision=precision)
    model.load_state_dict(checkpoint["model_state_dict"])
    logger.info("Loaded model from epoch %s", checkpoint.get("epoch"))
    return model.to(device)


def evaluate_recommendation_model(model_path: str, data_dir: str, embeddings_path: str, k_values=None, device=None,
                                  n_negatives=None, precision: str | None = None) -> dict:
    """src/ml/evaluate.py:294-340."""
    k_values = k_values or [5, 10, 20]
    dev = torch.device(device) if device else torch.device("cuda")
    full_matrix, train_df, val_df, mappings = _data.load_training_data(data_dir)
    user_to_idx, item_to_idx = mappings["user_to_idx"], mappings["item_to_idx"]
    input_matrix = _build_input_matrix(train_df, val_df, user_to_idx, item_to_idx, full_matrix.shape)
    test_df = pd.read_csv(Path(data_dir) / "test.csv")
    embeddings, _, _ = _data.load_embeddings(embeddings_path)
    model = load_model_from_checkpoint(model_path, embeddings, dev, precision)
    ev = RecommendationEvaluator(model, input_matrix, user_to_idx, item_to_idx, dev)
    if n_negatives is not None:
        results = ev.evaluate_dataset_with_negatives(test_df, n_negatives, k_values)
    else:
        results = ev.evaluate_dataset(test_df, k_values)
    print(f"\n{'-' * 70}\n{'K':<5} | {'Recall':>12} | {'NDCG':>12} | {'Hit Ratio':>12}\n{'-' * 70}")
    for k in k_values:
        m = results[k]
        print(f"@{k:<4} | {m['recall']:>12.4f} | {m['ndcg']:>12.4f} | {m['hit_ratio']:>12.4f}")
    print("-" * 70)
    return results

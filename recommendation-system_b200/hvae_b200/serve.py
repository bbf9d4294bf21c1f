"""Batched form of the API's scoring call (SURVEY.md §8 a17 / §8f.3; reference: src/api/server.py:115-183).

The reference answers one `/recommend` request at a time: densify the user's row, `get_user_embedding`, `decode`, mask
the seen items with -inf, `argsort`, keep `top_k`, drop -inf entries and items without an id.  `RecommendService` gives
the same answer (same fields, same ordering under (score desc, index desc), same error for an unknown user), but a
whole group of requests becomes ONE encoder + scoring + top-K launch (`RecommendationEvaluator.topk_users`).
`MicroBatcher` collects concurrent requests for a few milliseconds so that independent callers share a launch.
The FastAPI plumbing itself (routes, pydantic models, CORS) is out of scope: a handler calls
`service.recommend(...)` or `await loop.run_in_executor(None, batcher.submit(...).result)`.
"""
from __future__ import annotations

import math
import numbers
import random
import threading
import time
from concurrent.futures import Future
from typing import Callable, Iterable, Sequence

import numpy as np

MAX_TOP_K = 100          # the API's own limit (src/api/server.py: RecommendationRequest.top_k <= 100)
# Sampling temperatures: below 1e-3 the draw is the plain top-K wherever scores differ by more than 0.017, above 1e3 it is
# close to uniform over the admissible items for any trained model; either end is better asked for without a temperature.
MIN_TEMPERATURE, MAX_TEMPERATURE = 1e-3, 1e3
# Boosts: |value| <= 1e6 and |weight| <= 1e3 keep |weight * value| <= 1e9, so a boosted key s + w * value stays finite for any
# finite score (and far from the fp32 range the kernels' bounds work in).
MAX_BOOST_VALUE, MAX_BOOST_WEIGHT = 1e6, 1e3


class UnknownUser(KeyError):
    """The user id is not in the training data (the reference answers HTTP 404, server.py:134-138)."""


def check_temperature(t) -> float:
    """A sampling temperature as float; ValueError unless it is a finite real number in [MIN_TEMPERATURE, MAX_TEMPERATURE]."""
    if isinstance(t, bool) or not isinstance(t, numbers.Real):
        raise ValueError(f"temperature must be a number, got {t!r}")
    t = float(t)
    if not (math.isfinite(t) and MIN_TEMPERATURE <= t <= MAX_TEMPERATURE):
        raise ValueError(f"temperature must lie in [{MIN_TEMPERATURE:g}, {MAX_TEMPERATURE:g}], got {t!r}")
    return t


def check_seed(seed) -> int:
    """A sampling seed as int; ValueError unless it is an integer in [0, 2^64)."""
    if isinstance(seed, bool) or not isinstance(seed, numbers.Integral):
        raise ValueError(f"seed must be an integer, got {seed!r}")
    seed = int(seed)
    if not 0 <= seed < 1 << 64:
        raise ValueError(f"seed must lie in [0, 2^64), got {seed}")
    return seed


def check_boost_weight(w) -> float:
    """A boost weight as float; ValueError unless it is a finite real number with |w| <= MAX_BOOST_WEIGHT."""
    if isinstance(w, bool) or not isinstance(w, numbers.Real):
        raise ValueError(f"boost_weight must be a number, got {w!r}")
    w = float(w)
    if not (math.isfinite(w) and abs(w) <= MAX_BOOST_WEIGHT):
        raise ValueError(f"boost_weight must be finite with |boost_weight| <= {MAX_BOOST_WEIGHT:g}, got {w!r}")
    return w


def check_boost_values(values, n_items: int) -> np.ndarray:
    """Boost values as float32 [n_items]; ValueError unless there is one finite real per item with |value| <= MAX_BOOST_VALUE."""
    try:
        v = np.asarray(values, dtype=np.float64)
    except (TypeError, ValueError) as e:
        raise ValueError(f"boost values must be real numbers: {e}") from None
    if v.shape != (n_items,):
        raise ValueError(f"boost values: expected one value per item ({n_items}), got shape {v.shape}")
    if not (np.isfinite(v).all() and (np.abs(v) <= MAX_BOOST_VALUE).all()):
        raise ValueError(f"boost values must be finite with |value| <= {MAX_BOOST_VALUE:g}")
    return v.astype(np.float32)


def _response(user_id, idx: np.ndarray, val: np.ndarray, top_k: int, idx_to_item: dict, total_items: int) -> dict:
    """RecommendationResponse of the reference (server.py:164-178): -inf scores and unmapped items are dropped."""
    recs = []
    for item_idx, score in zip(idx[:top_k].tolist(), val[:top_k].tolist()):
        if item_idx in idx_to_item and not np.isinf(score):
            recs.append({"item_id": idx_to_item[item_idx], "score": float(score)})
    return {"user_id": user_id, "recommendations": recs, "total_items": total_items}


def _request_parts(req: tuple) -> tuple:
    """(user_id, top_k, exclude_seen, item_filter, exclude_items, temperature, seed, boost, boost_weight) of a 3- to 9-element
    request (boost_weight None: 1.0)."""
    if not 3 <= len(req) <= 9:
        raise ValueError(f"a request has 3 to 9 elements, got {len(req)}")
    parts = tuple(req) + (None,) * (9 - len(req))
    return parts[:8] + (1.0 if parts[8] is None else parts[8],)


class RecommendService:
    """topk_fn(user_indices, K, exclude_seen) -> (values [n, K], indices [n, K]) array-likes; the production binding is
    `RecommendationEvaluator.topk_users` (`from_evaluator`).  A launch whose requests use item filters or exclusions calls
    topk_fn(user_indices, K, exclude_seen, item_filter=[name or None per row], exclude=[item index array per row]);
    add_filter_fn(name, item_indices) registers an allow-set with the backend (RecommendationEvaluator.add_item_filter).
    A launch with sampled requests also passes temperature=[tau or None per row], seed=[seed or None per row], and one with
    boosted requests boost=[name or None per row], boost_weight=[w or None per row]; add_boost_fn(name, values float32
    [n_items]) registers a boost with the backend (RecommendationEvaluator.add_item_boost)."""

    def __init__(self, topk_fn: Callable, user_to_idx: dict, idx_to_item: dict, n_items: int, max_batch: int = 4096,
                 add_filter_fn: Callable | None = None, add_boost_fn: Callable | None = None):
        self.topk_fn, self.user_to_idx, self.idx_to_item = topk_fn, user_to_idx, idx_to_item
        self.n_items, self.max_batch = int(n_items), int(max_batch)
        self.add_filter_fn, self.add_boost_fn = add_filter_fn, add_boost_fn
        self.filters: set = set()
        self.boosts: set = set()
        self._item_to_idx: dict | None = None
        self._seeds = random.Random()         # seeds of sampled requests that bring none (OS entropy)
        self._seeds_lock = threading.Lock()

    @classmethod
    def from_evaluator(cls, evaluator, idx_to_item: dict, max_batch: int = 4096):
        def topk(users, K, exclude_seen, **filters):
            v, i = evaluator.topk_users(users, K, exclude_seen, **filters)
            return v.cpu().numpy(), i.cpu().numpy()
        return cls(topk, evaluator.user_to_idx, idx_to_item, evaluator.n_items, max_batch, evaluator.add_item_filter,
                   evaluator.add_item_boost)

    def _item_index(self) -> dict:
        if self._item_to_idx is None:
            self._item_to_idx = {item: idx for idx, item in self.idx_to_item.items()}
        return self._item_to_idx

    def add_item_filter(self, name: str, item_ids) -> None:
        """Registers (or replaces) the allow-set `name` from API item ids; requests with item_filter=name then only get these
        items.  An id without an item index raises ValueError and registers nothing."""
        if not isinstance(name, str):
            raise ValueError(f"item filter names are strings, got {name!r}")
        to_idx = self._item_index()
        unknown = [i for i in item_ids if i not in to_idx]
        if unknown:
            raise ValueError(f"item filter {name!r}: unknown item ids {unknown[:5]}{' ...' if len(unknown) > 5 else ''}")
        idx = np.array([to_idx[i] for i in item_ids], dtype=np.int64)
        if self.add_filter_fn is not None:
            self.add_filter_fn(name, idx)
        self.filters.add(name)

    def add_item_boost(self, name: str, values: dict) -> None:
        """Registers (or replaces) the boost `name` from {API item id: value}; items not listed get 0.  Requests with
        boost=name and boost_weight=w are then ranked by score + w * value.  Values must be finite with |value| <=
        MAX_BOOST_VALUE; an id without an item index, or a bad value, raises ValueError and registers nothing."""
        if not isinstance(name, str):
            raise ValueError(f"item boost names are strings, got {name!r}")
        to_idx = self._item_index()
        try:
            items = list(values.items())
        except AttributeError:
            raise ValueError("item boost values must be a mapping {item id: value}") from None
        unknown = [i for i, _ in items if i not in to_idx]
        if unknown:
            raise ValueError(f"item boost {name!r}: unknown item ids {unknown[:5]}{' ...' if len(unknown) > 5 else ''}")
        for _, v in items:
            if isinstance(v, bool) or not isinstance(v, numbers.Real):
                raise ValueError(f"item boost {name!r}: values must be numbers, got {v!r}")
        dense = np.zeros(self.n_items, dtype=np.float64)
        for i, v in items:
            dense[to_idx[i]] = v
        dense = check_boost_values(dense, self.n_items)
        if self.add_boost_fn is not None:
            self.add_boost_fn(name, dense)
        self.boosts.add(name)

    def _check(self, user_id, top_k, item_filter=None):
        if user_id not in self.user_to_idx:
            raise UnknownUser(f"User '{user_id}' not found in training data")
        if not 1 <= int(top_k) <= MAX_TOP_K:
            raise ValueError(f"top_k must be in [1, {MAX_TOP_K}], got {top_k}")
        if item_filter is not None and (not isinstance(item_filter, str) or item_filter not in self.filters):
            raise ValueError(f"unknown item filter {item_filter!r}")

    def _excluded(self, exclude_items) -> np.ndarray:
        """Item indices of the API ids in exclude_items (None = nothing); ids without an index are dropped."""
        if exclude_items is None:
            return np.zeros(0, dtype=np.int64)
        if isinstance(exclude_items, (str, bytes)):
            raise ValueError("exclude_items must be a sequence of item ids, not a single string")
        to_idx = self._item_index()
        try:
            return np.array([to_idx[i] for i in exclude_items if i in to_idx], dtype=np.int64)
        except TypeError as e:          # not iterable, or an unhashable id
            raise ValueError(f"exclude_items: {e}") from None

    def _new_seed(self) -> int:
        with self._seeds_lock:
            return self._seeds.getrandbits(53)       # (exact as a JSON number: a client can send it back unchanged)

    def recommend(self, user_id, top_k: int = 10, exclude_seen: bool = True, *, item_filter=None, exclude_items=(),
                  temperature=None, seed=None, boost=None, boost_weight=1.0) -> dict:
        """temperature: None for the top_k best items, else a sampled answer: top_k items drawn without replacement from
        softmax(scores / temperature) (temperature in [MIN_TEMPERATURE, MAX_TEMPERATURE]), in drawn order.  seed: an
        integer in [0, 2^64) (None: the service picks one); the response carries "temperature" and "seed", and the same
        user, seed, temperature, filter, exclusions and model give the same answer.
        boost: the name of a boost registered with add_item_boost; items are then ranked (or, with a temperature, sampled)
        by score + boost_weight * value (boost_weight a finite real with |w| <= MAX_BOOST_WEIGHT).  "score" stays the
        model's score; the response carries "boost" and "boost_weight"."""
        out = self.recommend_many([(user_id, top_k, exclude_seen, item_filter, exclude_items, temperature, seed, boost,
                                    boost_weight)])[0]
        if isinstance(out, Exception):
            raise out
        return out

    def recommend_many(self, requests: Sequence[tuple]) -> list:
        """requests: (user_id, top_k, exclude_seen[, item_filter[, exclude_items[, temperature[, seed[, boost[,
        boost_weight]]]]]]) tuples.  One launch per exclude_seen group (K = the group's largest top_k), whatever filters,
        exclusions, temperatures and boosts its requests carry.  Exclusions are API item ids; ids without an item index are
        ignored (they can never be recommended).  A request with a temperature is sampled, one with a boost re-ranked (see
        recommend).  Returns, in request order, the response dict or the exception that request would have raised."""
        out: list = [None] * len(requests)
        groups: dict[bool, list[int]] = {}
        extra: dict[int, tuple] = {}         # request -> (filter name or None, excluded item indices)
        sampled: dict[int, tuple] = {}       # request -> (temperature, seed)
        boosted: dict[int, tuple] = {}       # request -> (boost name, weight)
        for n, req in enumerate(requests):
            try:
                user_id, top_k, exclude_seen, item_filter, exclude_items, temperature, seed, boost, boost_weight = \
                    _request_parts(req)
                self._check(user_id, top_k, item_filter)
                if boost is not None:
                    if not isinstance(boost, str) or boost not in self.boosts:
                        raise ValueError(f"unknown item boost {boost!r}")
                    boost_weight = check_boost_weight(boost_weight)
                excluded = self._excluded(exclude_items)
                seed = None if seed is None else check_seed(seed)
                if temperature is not None:
                    temperature = check_temperature(temperature)
                    seed = self._new_seed() if seed is None else seed
            except (UnknownUser, ValueError) as e:
                out[n] = e
                continue
            if item_filter is not None or len(excluded):
                extra[n] = (item_filter, excluded)
            if temperature is not None:
                sampled[n] = (temperature, seed)
            if boost is not None:
                boosted[n] = (boost, boost_weight)
            groups.setdefault(bool(exclude_seen), []).append(n)
        for exclude_seen, members in groups.items():
            for s in range(0, len(members), self.max_batch):
                part = members[s:s + self.max_batch]
                K = min(max(int(requests[n][1]) for n in part), self.n_items)
                users = np.array([self.user_to_idx[requests[n][0]] for n in part], dtype=np.int32)
                kw = {}
                if any(n in extra for n in part):
                    none = (None, np.zeros(0, dtype=np.int64))
                    kw.update(item_filter=[extra.get(n, none)[0] for n in part], exclude=[extra.get(n, none)[1] for n in part])
                if any(n in sampled for n in part):
                    kw.update(temperature=[sampled[n][0] if n in sampled else None for n in part],
                              seed=[sampled[n][1] if n in sampled else None for n in part])
                if any(n in boosted for n in part):
                    kw.update(boost=[boosted[n][0] if n in boosted else None for n in part],
                              boost_weight=[boosted[n][1] if n in boosted else None for n in part])
                val, idx = self.topk_fn(users, K, exclude_seen, **kw)
                val, idx = np.asarray(val), np.asarray(idx)
                for r, n in enumerate(part):
                    out[n] = _response(requests[n][0], idx[r], val[r], int(requests[n][1]), self.idx_to_item, self.n_items)
                    if n in sampled:
                        out[n]["temperature"], out[n]["seed"] = sampled[n]
                    if n in boosted:
                        out[n]["boost"], out[n]["boost_weight"] = boosted[n]
        return out


class MicroBatcher:
    """Collects `submit()` calls from any number of threads and serves them with `service.recommend_many` in batches:
    a batch closes after `max_wait_ms` or at `max_batch` requests, whichever comes first."""

    def __init__(self, service: RecommendService, max_batch: int = 256, max_wait_ms: float = 2.0):
        self.service, self.max_batch, self.max_wait = service, int(max_batch), max_wait_ms / 1e3
        self._cv = threading.Condition()
        self._queue: list[tuple[tuple, Future]] = []
        self._closed = False
        self.batches_served = 0
        self._thread = threading.Thread(target=self._run, name="hvae-microbatcher", daemon=True)
        self._thread.start()

    def submit(self, user_id, top_k: int = 10, exclude_seen: bool = True, *, item_filter=None, exclude_items=(), temperature=None,
               seed=None, boost=None, boost_weight=1.0) -> Future:
        fut: Future = Future()
        if exclude_items is not None and not isinstance(exclude_items, (str, bytes)):
            try:
                exclude_items = tuple(exclude_items)      # a copy: the caller may reuse its list
            except TypeError:
                pass                                      # reported for this request by recommend_many
        if boost is not None:
            req = (user_id, top_k, exclude_seen, item_filter, exclude_items, temperature, seed, boost, boost_weight)
        elif temperature is not None or seed is not None:
            req = (user_id, top_k, exclude_seen, item_filter, exclude_items, temperature, seed)
        elif item_filter is None and exclude_items in (None, ()):
            req = (user_id, top_k, exclude_seen)
        else:
            req = (user_id, top_k, exclude_seen, item_filter, exclude_items)
        with self._cv:
            if self._closed:
                raise RuntimeError("MicroBatcher is closed")
            self._queue.append((req, fut))
            self._cv.notify()
        return fut

    def close(self):
        with self._cv:
            self._closed = True
            self._cv.notify()
        self._thread.join()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _take(self) -> list:
        with self._cv:
            while not self._queue and not self._closed:
                self._cv.wait()
            if not self._queue:
                return []
            deadline = time.monotonic() + self.max_wait
            while len(self._queue) < self.max_batch and not self._closed:
                left = deadline - time.monotonic()
                if left <= 0:
                    break
                self._cv.wait(left)
            batch, self._queue = self._queue[:self.max_batch], self._queue[self.max_batch:]
            return batch

    def _run(self):
        while True:
            batch = self._take()
            if not batch:
                return
            try:
                results: Iterable = self.service.recommend_many([req for req, _ in batch])
            except Exception as e:      # a failed launch fails every request of the batch, not the serving thread
                results = [e] * len(batch)
            self.batches_served += 1
            for (_, fut), res in zip(batch, results):
                if isinstance(res, Exception):
                    fut.set_exception(res)
                else:
                    fut.set_result(res)

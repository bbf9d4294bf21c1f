"""CPU: sampled recommendations of the batched serving call (hvae_b200/serve.py) with a fake top-K backend that draws
Gumbel-top-K from a small dense score table -- the 6- and 7-element request forms, seed generation and echo, per-request
validation of temperatures and seeds, plain requests untouched, mixed launches, and MicroBatcher.submit's forwarding."""
import math

import numpy as np
import pytest

from hvae_b200.serve import MAX_TEMPERATURE, MIN_TEMPERATURE, MicroBatcher, RecommendService


def _world(U=8, N=60, seed=0):
    rng = np.random.default_rng(seed)
    scores = rng.permutation(U * N).reshape(U, N).astype(np.float64) / 50.0
    seen = [np.sort(rng.choice(N, size=int(rng.integers(0, 6)), replace=False)) for _ in range(U)]
    user_to_idx = {f"U{u}": u for u in range(U)}
    idx_to_item = {i: f"B{i}" for i in range(N)}
    calls = []

    def topk_fn(users, K, exclude_seen, item_filter=None, exclude=None, **sample):
        calls.append((len(users), K, bool(exclude_seen), sample))
        temps = sample.get("temperature", [None] * len(users))
        seeds = sample.get("seed", [None] * len(users))
        vals, idxs = [], []
        for r, u in enumerate(users):
            s = scores[u].copy()
            if exclude_seen:
                s[seen[u]] = -np.inf
            key = s.copy()
            if temps[r] is not None:          # noise of (seed, item) only, as the kernels draw it
                g = -np.log(-np.log(np.random.default_rng([seeds[r] & 0xFFFFFFFF, seeds[r] >> 32]).random(N)))
                key = s / temps[r] + g
            order = np.lexsort((-np.arange(N), -key))[:K]
            vals.append(s[order]); idxs.append(np.where(np.isinf(s[order]), -1, order))
        return np.array(vals, np.float32), np.array(idxs, np.int32)

    return scores, seen, user_to_idx, idx_to_item, topk_fn, calls


def _service(max_batch=4096):
    scores, seen, u2i, i2it, topk_fn, calls = _world()
    return RecommendService(topk_fn, u2i, i2it, len(i2it), max_batch), calls


def _ids(resp):
    return [r["item_id"] for r in resp["recommendations"]]


def test_tuple_forms_and_seed_echo():
    svc, calls = _service()
    plain = svc.recommend_many([("U1", 5, True)])[0]
    six = svc.recommend_many([("U1", 5, True, None, (), 2.0)])[0]
    seven = svc.recommend_many([("U1", 5, True, None, (), 2.0, 1234)])[0]
    assert "seed" not in plain and "temperature" not in plain
    assert six["temperature"] == 2.0 and isinstance(six["seed"], int) and 0 <= six["seed"] < 2 ** 53
    assert seven["seed"] == 1234 and seven["temperature"] == 2.0
    again = svc.recommend("U1", 5, temperature=2.0, seed=six["seed"])          # the echoed seed reproduces the answer
    assert _ids(again) == _ids(six)
    assert _ids(svc.recommend("U1", 5, temperature=2, seed=1234)) == _ids(seven)
    assert calls[0][3] == {}
    assert calls[1][3] == {"temperature": [2.0], "seed": [six["seed"]]}


def test_generated_seeds_differ():
    svc, _ = _service()
    seeds = {svc.recommend("U2", 3, temperature=1.0)["seed"] for _ in range(20)}
    assert len(seeds) == 20


@pytest.mark.parametrize("temperature", [float("nan"), float("inf"), -1.0, 0.0, MIN_TEMPERATURE / 2, MAX_TEMPERATURE * 2, "1.0",
                                         True, [1.0], complex(1, 0)])
def test_bad_temperature_fails_only_its_request(temperature):
    svc, calls = _service()
    out = svc.recommend_many([("U1", 5, True), ("U2", 5, True, None, (), temperature, 7), ("U3", 5, True, None, (), 1.0, 7)])
    assert isinstance(out[1], ValueError) and "temperature" in str(out[1])
    assert not isinstance(out[0], Exception) and not isinstance(out[2], Exception)
    assert len(calls) == 1 and calls[0][0] == 2 and calls[0][3]["temperature"] == [None, 1.0]
    with pytest.raises(ValueError):
        svc.recommend("U1", 5, temperature=temperature, seed=1)


@pytest.mark.parametrize("seed", [-1, 2 ** 64, 1.5, "3", True, [1]])
def test_bad_seed_fails_only_its_request(seed):
    svc, _ = _service()
    out = svc.recommend_many([("U1", 5, True, None, (), 1.0, seed), ("U3", 5, True, None, (), 1.0, 7)])
    assert isinstance(out[0], ValueError) and "seed" in str(out[0])
    assert out[1]["seed"] == 7
    with pytest.raises(ValueError):
        svc.recommend("U1", 5, temperature=1.0, seed=seed)


def test_range_edges_and_large_seeds_accepted():
    svc, _ = _service()
    for t in (MIN_TEMPERATURE, MAX_TEMPERATURE, np.float32(0.5), np.int64(3)):
        assert svc.recommend("U0", 4, temperature=t, seed=2 ** 64 - 1)["seed"] == 2 ** 64 - 1
    assert svc.recommend("U0", 4, temperature=1.0, seed=np.uint64(2 ** 63))["seed"] == 2 ** 63


def test_plain_requests_unchanged():
    svc, calls = _service()
    reqs = [("U0", 5, True), ("U1", 3, False), ("U2", 7, True, None, ()), ("U3", 2, True, None, None, None, None)]
    out = svc.recommend_many(reqs)
    assert [c[3] for c in calls] == [{}, {}]
    base, calls2 = _service()
    for r, o in zip(reqs, out):
        assert o == base.recommend(*r[:3])
    assert all(c[3] == {} for c in calls2)


def test_mixed_group_one_launch_same_answers():
    svc, calls = _service()
    reqs = [("U0", 5, True), ("U1", 10, True, None, (), 0.5, 11), ("U2", 3, True, None, (), 4.0, 12), ("U3", 4, False, None, (), 1.0, 13),
            ("U4", 6, False)]
    out = svc.recommend_many(reqs)
    assert len(calls) == 2                                        # one launch per exclude_seen group
    by_es = {c[2]: c for c in calls}
    assert by_es[True][1] == 10 and by_es[True][3] == {"temperature": [None, 0.5, 4.0], "seed": [None, 11, 12]}
    assert by_es[False][3] == {"temperature": [1.0, None], "seed": [13, None]}
    alone, _ = _service()
    for r, o in zip(reqs, out):                                  # the same answer alone, with its own K
        one = alone.recommend_many([r])[0]
        assert o == one
    assert [len(o["recommendations"]) for o in out] == [5, 10, 3, 4, 6]


def test_sampled_answers_vary_with_seed_and_keep_scores():
    scores, seen, u2i, i2it, topk_fn, _ = _world()
    svc = RecommendService(topk_fn, u2i, i2it, len(i2it))
    lists = {tuple(_ids(svc.recommend("U5", 5, temperature=MAX_TEMPERATURE, seed=s))) for s in range(10)}
    assert len(lists) > 1
    r = svc.recommend("U5", 8, temperature=1.0, seed=3)
    for rec in r["recommendations"]:                             # scores are the model's scores, not keys
        i = int(rec["item_id"][1:])
        assert math.isclose(rec["score"], np.float32(scores[5, i]), rel_tol=1e-6) and i not in set(seen[5].tolist())


def test_microbatcher_forwards_temperature_and_seed():
    svc, calls = _service()
    with MicroBatcher(svc, max_batch=8, max_wait_ms=50) as mb:
        futs = [mb.submit("U1", 5, temperature=1.0, seed=99), mb.submit("U2", 5), mb.submit("U1", 5, temperature=1.0),
                mb.submit("U3", 5, temperature="hot", seed=1)]
        res = [f.exception() or f.result() for f in futs]
    assert res[0]["seed"] == 99 and "seed" not in res[1] and isinstance(res[2]["seed"], int)
    assert isinstance(res[3], ValueError)
    assert res[0] == svc.recommend("U1", 5, temperature=1.0, seed=99)

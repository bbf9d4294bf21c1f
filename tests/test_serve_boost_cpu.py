"""CPU: boosted recommendations of the batched serving call (hvae_b200/serve.py) with a fake top-K backend that ranks
score + w * value from a small dense score table -- registration from API item ids, the 8- and 9-element request forms,
MicroBatcher.submit's forwarding, per-request validation of boost names and weights, the echoed fields, and which keyword
arguments a launch passes."""
import math

import numpy as np
import pytest

from hvae_b200.serve import MAX_BOOST_VALUE, MAX_BOOST_WEIGHT, MicroBatcher, RecommendService


def _world(U=6, N=40, seed=0):
    rng = np.random.default_rng(seed)
    scores = rng.permutation(U * N).reshape(U, N).astype(np.float64) / 8.0
    seen = [np.sort(rng.choice(N, size=int(rng.integers(0, 5)), replace=False)) for _ in range(U)]
    u2i = {f"U{u}": u for u in range(U)}
    i2it = {i: f"B{i}" for i in range(N)}
    boosts, calls = {}, []

    def add_boost(name, values):
        assert values.dtype == np.float32 and values.shape == (N,)
        boosts[name] = values.astype(np.float64)

    def topk_fn(users, K, exclude_seen, **kw):
        calls.append(kw)
        names = kw.get("boost", [None] * len(users))
        weights = kw.get("boost_weight", [None] * len(users))
        vals, idxs = [], []
        for r, u in enumerate(users):
            s = scores[u].copy()
            if exclude_seen:
                s[seen[u]] = -np.inf
            key = s if names[r] is None else s + weights[r] * boosts[names[r]]
            order = np.lexsort((-np.arange(N), -key))[:K]
            vals.append(s[order]); idxs.append(np.where(np.isinf(s[order]), -1, order))
        return np.array(vals, np.float32), np.array(idxs, np.int32)

    svc = RecommendService(topk_fn, u2i, i2it, N, add_boost_fn=add_boost)
    return svc, scores, seen, boosts, calls


def _ids(resp):
    return [r["item_id"] for r in resp["recommendations"]]


def test_registration_and_boosted_order():
    svc, scores, seen, boosts, calls = _world()
    svc.add_item_boost("promo", {"B3": 100.0, "B7": -2.5})
    assert boosts["promo"][3] == 100.0 and boosts["promo"][7] == -2.5 and np.count_nonzero(boosts["promo"]) == 2
    plain = svc.recommend("U0", 5)
    boosted = svc.recommend("U0", 5, boost="promo", boost_weight=1.0)
    assert "boost" not in plain and "boost_weight" not in plain
    assert boosted["boost"] == "promo" and boosted["boost_weight"] == 1.0
    if 3 not in seen[0]:
        assert _ids(boosted)[0] == "B3"
    s = scores[0].copy(); s[seen[0]] = -np.inf
    for rec in boosted["recommendations"]:              # "score" is the model's score, not the key
        assert rec["score"] == pytest.approx(np.float32(s[int(rec["item_id"][1:])]))
    assert calls[0] == {}                               # a plain launch passes no extra keywords


def test_unknown_ids_register_nothing():
    svc, _, _, boosts, _ = _world()
    with pytest.raises(ValueError, match="unknown item ids"):
        svc.add_item_boost("bad", {"B1": 1.0, "nope": 2.0})
    assert "bad" not in boosts and "bad" not in svc.boosts
    for bad in ({"B1": math.inf}, {"B1": math.nan}, {"B1": 2 * MAX_BOOST_VALUE}, {"B1": "x"}, {"B1": True}, [("B1", 1.0)]):
        with pytest.raises(ValueError):
            svc.add_item_boost("bad", bad)
    with pytest.raises(ValueError):
        svc.add_item_boost(3, {"B1": 1.0})
    assert "bad" not in boosts and not svc.boosts
    svc.add_item_boost("edge", {"B1": MAX_BOOST_VALUE, "B2": -MAX_BOOST_VALUE})
    assert "edge" in svc.boosts


def test_tuple_forms_and_submit():
    svc, _, _, _, calls = _world()
    svc.add_item_boost("promo", {"B5": 50.0})
    eight = svc.recommend_many([("U1", 4, True, None, (), None, None, "promo")])[0]
    nine = svc.recommend_many([("U1", 4, True, None, (), None, None, "promo", 1.0)])[0]
    nine_none = svc.recommend_many([("U1", 4, True, None, (), None, None, "promo", None)])[0]
    assert eight == nine == nine_none and eight["boost_weight"] == 1.0
    assert svc.recommend("U1", 4, boost="promo") == eight
    ten = svc.recommend_many([("U1", 4, True, None, (), None, None, "promo", 1.0, 0)])[0]
    assert isinstance(ten, ValueError) and "3 to 9" in str(ten)
    half = svc.recommend_many([("U1", 4, True, None, (), None, None, "promo", 0.5)])[0]
    assert half["boost_weight"] == 0.5
    with MicroBatcher(svc, max_batch=8, max_wait_ms=1.0) as mb:
        got = mb.submit("U1", 4, boost="promo", boost_weight=0.5).result(timeout=30)
        plain = mb.submit("U1", 4).result(timeout=30)
    assert got == half and "boost" not in plain


def test_validation_fails_only_its_own_request():
    svc, _, _, _, calls = _world()
    svc.add_item_boost("promo", {"B5": 50.0})
    reqs = [("U0", 3, True),
            ("U1", 3, True, None, (), None, None, "missing"),
            ("U2", 3, True, None, (), None, None, 7),
            ("U3", 3, True, None, (), None, None, "promo", math.nan),
            ("U4", 3, True, None, (), None, None, "promo", math.inf),
            ("U5", 3, True, None, (), None, None, "promo", 2 * MAX_BOOST_WEIGHT),
            ("U0", 3, True, None, (), None, None, "promo", "1.0"),
            ("U1", 3, True, None, (), None, None, "promo", True),
            ("U2", 3, True, None, (), None, None, "promo", -MAX_BOOST_WEIGHT)]
    out = svc.recommend_many(reqs)
    assert isinstance(out[0], dict) and isinstance(out[8], dict) and out[8]["boost_weight"] == -MAX_BOOST_WEIGHT
    for r in out[1:8]:
        assert isinstance(r, ValueError)
    with pytest.raises(ValueError, match="unknown item boost"):
        svc.recommend("U0", 3, boost="missing")


def test_mixed_launch_keywords():
    svc, _, _, _, calls = _world()
    svc.add_item_boost("promo", {"B5": 50.0})
    svc.add_item_boost("other", {"B9": -1.0})
    out = svc.recommend_many([("U0", 3, True), ("U1", 5, True, None, (), None, None, "promo", 2.0),
                              ("U2", 2, True, None, (), 1.5, 7, "other"), ("U3", 3, False)])
    assert all(isinstance(r, dict) for r in out)
    by_es = {len(c.get("boost", [])): c for c in calls}
    mixed = by_es[3]
    assert mixed["boost"] == [None, "promo", "other"] and mixed["boost_weight"] == [None, 2.0, 1.0]
    assert mixed["temperature"] == [None, None, 1.5] and mixed["seed"] == [None, None, 7]
    assert by_es[0] == {}                               # the exclude_seen=False launch holds no boosted request
    assert out[2]["boost"] == "other" and out[2]["temperature"] == 1.5 and out[2]["seed"] == 7
    assert "boost" not in out[0] and "boost" not in out[3]


@pytest.mark.parametrize("N", [1, 31, 32, 33, 1000])
def test_item_boost_bounds(N):
    import torch
    from hvae_b200.tc import item_boost_bounds
    t = torch.randn(3, N, generator=torch.Generator().manual_seed(N))
    b = item_boost_bounds(t).numpy()
    tn = t.numpy()
    assert b.shape == (3, 2 * ((N + 31) // 32)) and b.dtype == np.float32
    for j in range((N + 31) // 32):
        blk = tn[:, 32 * j:32 * j + 32]
        assert np.array_equal(b[:, 2 * j], blk.max(1)) and np.array_equal(b[:, 2 * j + 1], blk.min(1))

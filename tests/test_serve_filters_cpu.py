"""CPU: item filters and per-request exclusions of the batched serving call (hvae_b200/serve.py) with a fake top-K backend
on a small dense score table -- one launch per exclude_seen group whatever the filters, validation of filter names and
item ids, the 3-, 4- and 5-element request forms, and MicroBatcher.submit's keyword forwarding."""
import numpy as np
import pytest

from hvae_b200.serve import MicroBatcher, RecommendService, UnknownUser


def _world(U=9, N=40, seed=0):
    rng = np.random.default_rng(seed)
    scores = rng.permutation(U * N).reshape(U, N).astype(np.float32) / 7.0
    seen = [np.sort(rng.choice(N, size=int(rng.integers(0, 6)), replace=False)) for _ in range(U)]
    user_to_idx = {f"U{u}": u for u in range(U)}
    idx_to_item = {i: f"B{i}" for i in range(N) if i != 11}                       # one item without an id
    allow_sets: dict = {}
    calls = []

    def add_filter(name, idx):
        allow_sets[name] = np.asarray(idx)

    def topk_fn(users, K, exclude_seen, item_filter=None, exclude=None):
        calls.append((len(users), K, bool(exclude_seen), item_filter, exclude))
        vals, idxs = [], []
        for r, u in enumerate(users):
            s = scores[u].copy()
            if exclude_seen:
                s[seen[u]] = -np.inf
            if item_filter is not None and item_filter[r] is not None:
                keep = np.zeros(N, dtype=bool)
                keep[allow_sets[item_filter[r]]] = True
                s[~keep] = -np.inf
            if exclude is not None:
                s[exclude[r]] = -np.inf
            order = np.lexsort((-np.arange(N), -s))[:K]
            idx = np.where(np.isinf(s[order]), -1, order)
            vals.append(s[order]); idxs.append(idx)
        return np.array(vals, np.float32), np.array(idxs, np.int32)

    return scores, seen, user_to_idx, idx_to_item, topk_fn, add_filter, calls


def _service(**kw):
    scores, seen, u2i, i2it, topk_fn, add_filter, calls = _world()
    svc = RecommendService(topk_fn, u2i, i2it, scores.shape[1], add_filter_fn=add_filter, **kw)
    return svc, scores, seen, calls


def test_one_launch_per_exclude_seen_group_regardless_of_filters():
    svc, scores, seen, calls = _service()
    svc.add_item_filter("cat", [f"B{i}" for i in range(0, 40, 3) if i != 11])
    svc.add_item_filter("tiny", ["B5", "B7"])
    reqs = [("U0", 5, True), ("U1", 10, True, "cat"), ("U2", 3, True, "tiny", ["B7"]), ("U3", 4, False, None, ["B1", "B2"]),
            ("U4", 6, False, "cat"), ("U5", 2, True, None, ())]
    out = svc.recommend_many(reqs)
    assert len(calls) == 2
    by_group = {c[2]: c for c in calls}
    n, K, _, filt, excl = by_group[True]
    assert (n, K) == (4, 10) and filt == [None, "cat", "tiny", None]
    assert [e.tolist() for e in excl] == [[], [], [7], []]
    n, K, _, filt, excl = by_group[False]
    assert (n, K) == (2, 6) and filt == [None, "cat"] and [e.tolist() for e in excl] == [[1, 2], []]
    assert [r["item_id"] for r in out[2]["recommendations"]] == ["B5"]          # B7 excluded; fewer than top_k answers
    cat = {f"B{i}" for i in range(0, 40, 3)}
    assert all(r["item_id"] in cat for r in out[1]["recommendations"]) and len(out[1]["recommendations"]) == 10
    assert not {"B1", "B2"} & {r["item_id"] for r in out[3]["recommendations"]}


def test_plain_groups_call_topk_fn_without_keywords():
    scores, seen, u2i, i2it, _, _, _ = _world()
    calls = []

    def plain_topk(users, K, exclude_seen):          # the original three-argument protocol
        calls.append(K)
        return np.zeros((len(users), K), np.float32), np.tile(np.arange(K, dtype=np.int32), (len(users), 1))
    svc = RecommendService(plain_topk, u2i, i2it, scores.shape[1])
    out = svc.recommend_many([("U0", 3, True), ("U1", 4, True, None), ("U2", 2, False, None, ())])
    assert calls == [4, 2] and all(isinstance(o, dict) for o in out)


def test_filter_validation():
    svc, scores, seen, calls = _service()
    with pytest.raises(ValueError, match="unknown item ids"):
        svc.add_item_filter("bad", ["B1", "nope"])
    assert "bad" not in svc.filters
    with pytest.raises(ValueError, match="unknown item filter"):
        svc.recommend("U0", 5, item_filter="bad")
    svc.add_item_filter("ok", ["B1", "B2"])
    out = svc.recommend_many([("U0", 5, True, "nope"), ("nobody", 5, True, "ok"), ("U1", 0, True, "ok"), ("U1", 5, False, "ok")])
    assert isinstance(out[0], ValueError) and isinstance(out[1], UnknownUser) and isinstance(out[2], ValueError)
    assert sorted(r["item_id"] for r in out[3]["recommendations"]) == ["B1", "B2"]
    assert len(calls) == 1 and calls[0][0] == 1
    svc.add_item_filter("ok", ["B3"])                       # replaces
    assert [r["item_id"] for r in svc.recommend("U1", 5, False, item_filter="ok")["recommendations"]] == ["B3"]


def test_unknown_excluded_ids_are_ignored():
    svc, scores, seen, calls = _service()
    base = svc.recommend("U6", 8, False)
    top = base["recommendations"][0]["item_id"]
    got = svc.recommend("U6", 8, False, exclude_items=["nope", top, "B11"])
    assert top not in {r["item_id"] for r in got["recommendations"]}
    assert [r["item_id"] for r in got["recommendations"]] == [r["item_id"] for r in svc.recommend(
        "U6", 9, False)["recommendations"] if r["item_id"] != top][:8]
    assert calls[1][4][0].tolist() == [int(top[1:])]


@pytest.mark.parametrize("form", [3, 4, 5])
def test_request_tuple_forms(form):
    svc, scores, seen, calls = _service()
    svc.add_item_filter("cat", [f"B{i}" for i in range(20) if i != 11])
    req = ("U3", 6, True, "cat", ["B0"])[:form]
    got = svc.recommend_many([req])[0]
    kw = {}
    if form > 3:
        kw["item_filter"] = "cat"
    if form > 4:
        kw["exclude_items"] = ["B0"]
    assert got == svc.recommend("U3", 6, True, **kw)
    ids = [r["item_id"] for r in got["recommendations"]]
    if form > 3:
        assert all(int(i[1:]) < 20 for i in ids)
    if form > 4:
        assert "B0" not in ids
    assert (calls[0][3] is None) == (form == 3)


def test_microbatcher_forwards_filter_keywords():
    svc, scores, seen, calls = _service()
    svc.add_item_filter("cat", ["B1", "B2", "B3"])
    seen_reqs = []
    inner = svc.recommend_many

    def spy(reqs):
        seen_reqs.extend(reqs)
        return inner(reqs)
    svc.recommend_many = spy
    with MicroBatcher(svc, max_batch=8, max_wait_ms=50.0) as mb:
        f1 = mb.submit("U0", 5)
        f2 = mb.submit("U1", 5, True, item_filter="cat", exclude_items=["B2"])
        f3 = mb.submit("U2", 5, False, item_filter="missing")
        r1, r2 = f1.result(timeout=10), f2.result(timeout=10)
        with pytest.raises(ValueError):
            f3.result(timeout=10)
    assert ("U0", 5, True) in seen_reqs
    assert ("U1", 5, True, "cat", ("B2",)) in seen_reqs
    assert {r["item_id"] for r in r2["recommendations"]} <= {"B1", "B3"}
    assert r1 == svc.recommend("U0", 5)


def test_malformed_filter_fields_fail_only_their_request():
    svc, scores, seen, calls = _service()
    svc.add_item_filter("cat", ["B1", "B2", "B3"])
    reqs = [("U0", 5, True, None, None), ("U1", 5, True, ["cat"]), ("U2", 5, True, None, 7), ("U3", 5, True, None, [["B1"]]),
            ("U4", 5, True, None, "B1"), ("U5", 5, True, "cat", None)]
    out = svc.recommend_many(reqs)
    assert isinstance(out[0], dict) and out[0] == svc.recommend("U0", 5)
    assert all(isinstance(o, ValueError) for o in out[1:5])
    assert {r["item_id"] for r in out[5]["recommendations"]} <= {"B1", "B2", "B3"}
    with pytest.raises(ValueError):
        svc.add_item_filter(("not", "a", "string"), ["B1"])
    with MicroBatcher(svc, max_batch=8, max_wait_ms=20.0) as mb:
        ok = mb.submit("U6", 5, exclude_items=None)
        bad = mb.submit("U7", 5, exclude_items=7)
        assert isinstance(ok.result(timeout=10), dict)
        with pytest.raises(ValueError):
            bad.result(timeout=10)

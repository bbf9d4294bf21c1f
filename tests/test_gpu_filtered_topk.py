"""GPU: item allow-sets and per-request exclusions in the fused top-K kernels (hvae_tc_score_topk_filtered,
hvae_mask_topk_filtered), the evaluator (topk_users(item_filter=, exclude=)) and the service (recommend(item_filter=,
exclude_items=)).

The main check: a filtered launch with bitmaps A and mask CSR M returns, bit for bit, what the unfiltered kernel returns
with the mask M u (not A): both read the same GEMM tiles, so any difference is a bug in the filter."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from hvae_b200 import _cabi
    return _cabi.lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _r8(n):
    return (n + 7) // 8 * 8


def _operands(lib, B, N, d, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    U = (torch.randn(B, d, generator=g) * 12.0 / d ** 0.5).to(dev)
    E = torch.nn.functional.normalize(torch.randn(N, d, generator=g), dim=1).to(dev)
    out = []
    for x in (U, E):
        ld = _r8(x.shape[1])
        xb = torch.empty(x.shape[0], ld, dtype=torch.bfloat16, device=dev)
        lib.cast_bf16(x.data_ptr(), x.shape[0], x.shape[1], x.shape[1], xb.data_ptr(), ld, _st())
        out += [xb, ld]
    return out


def _pack(allow_bool, dev):
    """bool [F, n_total] -> int32 [F, ceil(n_total/32)] bitmaps (bit i of word w = item 32w + i)."""
    F, n = allow_bool.shape
    bits = np.zeros((F, (n + 31) // 32 * 32), dtype=bool)
    bits[:, :n] = allow_bool
    return torch.as_tensor(np.packbits(bits, axis=1, bitorder="little").view(np.int32), device=dev)


def _filters(n_total, fracs, rng):
    return np.stack([rng.random(n_total) < f for f in fracs])


def _csr(rows_items, dev):
    indptr = np.zeros(len(rows_items) + 1, dtype=np.int64)
    indptr[1:] = np.cumsum([len(r) for r in rows_items])
    idx = np.concatenate([np.asarray(r, dtype=np.int32) for r in rows_items]) if indptr[-1] else np.zeros(0, np.int32)
    return torch.as_tensor(indptr, device=dev), torch.as_tensor(idx, device=dev)


def _seen(B, n_total, rng, per_row=30):
    return [np.unique(rng.integers(0, n_total, rng.integers(0, per_row))).astype(np.int32) for _ in range(B)]


def _tc_topk(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, allow=None, aor=None):
    n_it = hi - lo
    ns = int(lib.tc_topk_splits(B, n_it))
    cv = torch.empty(B, ns * K, device=Ub.device)
    ci = torch.empty(B, ns * K, dtype=torch.int32, device=Ub.device)
    e_ptr = Eb.data_ptr() + 2 * lo * lde
    indptr, indices = mask
    if allow is None:
        lib.tc_score_topk(Ub.data_ptr(), ldu, B, e_ptr, lde, n_it, d, lo, indptr.data_ptr(), indices.data_ptr(), None, K,
                          cv.data_ptr(), ci.data_ptr(), _st())
    else:
        lib.tc_score_topk_filtered(Ub.data_ptr(), ldu, B, e_ptr, lde, n_it, d, lo, indptr.data_ptr(), indices.data_ptr(), None,
                                   allow.data_ptr(), allow.stride(0), aor.data_ptr(), K, cv.data_ptr(), ci.data_ptr(), _st())
    ov = torch.empty(B, K, device=Ub.device)
    oi = torch.empty(B, K, dtype=torch.int32, device=Ub.device)
    lib.topk_merge(cv.data_ptr(), ci.data_ptr(), B, ns * K, K, ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


def _folded(seen, allow_bool, aor):
    """Mask rows M u (not A): the seen items plus every item the row's filter leaves out."""
    out = []
    for b, s in enumerate(seen):
        if aor[b] < 0:
            out.append(s)
        else:
            out.append(np.union1d(s, np.flatnonzero(~allow_bool[aor[b]])).astype(np.int32))
    return out


TC_SHAPES = [(300, 5000, 768, 20), (77, 1000, 24, 1), (130, 4099, 384, 8), (257, 3001, 384, 32), (64, 2050, 768, 33),
             (200, 9000, 384, 100), (129, 12101, 24, 128), (513, 7000, 768, 12), (96, 2600, 384, 16), (96, 2600, 24, 24)]


@pytest.mark.parametrize("B,N,d,K", TC_SHAPES)
def test_tc_filtered_equals_filter_folded_into_mask(dev, lib, B, N, d, K):
    rng = np.random.default_rng(B * 7 + N)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=B)
    allow_bool = _filters(N, (0.5, 0.1, 0.01, 0.003), rng)
    allow = _pack(allow_bool, dev)
    aor_np = rng.integers(-1, 4, B).astype(np.int32)
    aor_np[:5] = [-1, 0, 1, 2, 3][:min(5, B)]
    aor = torch.as_tensor(aor_np, device=dev)
    seen = _seen(B, N, rng)
    mask = _csr(seen, dev)
    folded = _csr(_folded(seen, allow_bool, aor_np), dev)
    lo_shard = N // 3 + 5
    assert lo_shard % 32 != 0
    for lo, hi in [(0, N), (lo_shard, N - 7)]:
        v, i = _tc_topk(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, allow, aor)
        rv, ri = _tc_topk(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, folded)
        assert torch.equal(v, rv) and torch.equal(i, ri), (lo, hi)
        # every finite entry is allowed; the rest are (-inf, -1)
        vn, inn = v.cpu().numpy(), i.cpu().numpy()
        fin = np.isfinite(vn)
        assert np.all(inn[~fin] == -1)
        for b in range(B):
            ids = inn[b][fin[b]]
            assert np.all((ids >= lo) & (ids < hi))
            if aor_np[b] >= 0:
                assert allow_bool[aor_np[b], ids].all()


@pytest.mark.parametrize("B,N,d,K", [(300, 5000, 768, 20), (129, 3001, 384, 100), (77, 1000, 24, 8)])
def test_tc_allow_everything_is_unfiltered(dev, lib, B, N, d, K):
    rng = np.random.default_rng(1)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=2)
    allow = _pack(np.ones((1, N), dtype=bool), dev)
    aor = torch.zeros(B, dtype=torch.int32, device=dev)
    mask = _csr(_seen(B, N, rng), dev)
    for lo, hi in [(0, N), (N // 4 + 3, N)]:
        v, i = _tc_topk(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, allow, aor)
        rv, ri = _tc_topk(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask)
        assert torch.equal(v, rv) and torch.equal(i, ri)


def _check_against_fp64(Ub, Eb, d, v, i, lo, hi, K, admissible_of_row, rows):
    """Sorted by (score desc, id desc), unique, admissible, scores within 1e-5 of fp64, nothing better left out."""
    vn, inn = v.cpu().numpy(), i.cpu().numpy()
    for b in rows:
        adm = admissible_of_row(b)                                     # sorted admissible global ids in [lo, hi)
        s = (Ub[b, :d].double() @ Eb[torch.as_tensor(adm, device=Ub.device).long(), :d].double().t()).cpu().numpy() \
            if len(adm) else np.zeros(0)
        fin = np.isfinite(vn[b])
        n_fin = int(fin.sum())
        assert n_fin == min(K, len(adm)), (b, n_fin, len(adm))
        assert np.all(fin[:n_fin]) and np.all(inn[b][n_fin:] == -1)
        ids, vals = inn[b][:n_fin], vn[b][:n_fin]
        assert len(set(ids.tolist())) == n_fin
        order = np.lexsort((-ids.astype(np.int64), -vals))
        assert np.array_equal(order, np.arange(n_fin))
        pos = np.searchsorted(adm, ids)
        assert np.all(pos < len(adm)) and np.array_equal(adm[np.minimum(pos, len(adm) - 1)], ids)
        np.testing.assert_allclose(vals, s[pos], rtol=0, atol=1e-5)
        rest = np.delete(s, pos)
        if n_fin == K and rest.size:
            assert vals[-1] >= rest.max() - 1e-5


@pytest.mark.parametrize("B,N,d,K", [(300, 5000, 768, 20), (200, 9000, 384, 100), (65, 2049, 24, 32)])
def test_tc_filtered_matches_fp64(dev, lib, B, N, d, K):
    rng = np.random.default_rng(3)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=3)
    allow_bool = _filters(N, (0.3, 0.05, 0.01), rng)
    allow = _pack(allow_bool, dev)
    aor_np = rng.integers(-1, 3, B).astype(np.int32)
    aor = torch.as_tensor(aor_np, device=dev)
    seen = _seen(B, N, rng, 60)
    excl = [np.unique(rng.integers(0, N, 20)).astype(np.int32) for _ in range(B)]
    masked = [np.union1d(s, e).astype(np.int32) for s, e in zip(seen, excl)]
    mask = _csr(masked, dev)
    lo, hi = 37, N - 3
    v, i = _tc_topk(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, allow, aor)

    def adm(b):
        ok = np.ones(N, dtype=bool) if aor_np[b] < 0 else allow_bool[aor_np[b]].copy()
        ok[masked[b]] = False
        ok[:lo] = False
        ok[hi:] = False
        return np.flatnonzero(ok)
    _check_against_fp64(Ub, Eb, d, v, i, lo, hi, K, adm, range(B))


def test_tc_filtered_edges(dev, lib):
    N, d = 3000, 384
    rng = np.random.default_rng(4)
    for B, K in [(1, 20), (40, 100), (40, 8)]:
        Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=B)
        few = np.zeros(N, dtype=bool)
        few[rng.choice(N, 5, replace=False)] = True
        allow_bool = np.stack([few, np.zeros(N, dtype=bool)])          # five items; nothing at all
        allow = _pack(allow_bool, dev)
        seen = _seen(B, N, rng)
        seen[0] = np.union1d(seen[0], np.flatnonzero(few)[:2]).astype(np.int32)       # two of the five already seen
        for f in (0, 1):
            aor = torch.full((B,), f, dtype=torch.int32, device=dev)
            v, i = _tc_topk(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, _csr(seen, dev), allow, aor)
            vn, inn = v.cpu().numpy(), i.cpu().numpy()
            for b in range(B):
                want = np.setdiff1d(np.flatnonzero(allow_bool[f]), seen[b])
                fin = np.isfinite(vn[b])
                assert fin.sum() == len(want) and np.all(fin[:len(want)])
                assert sorted(inn[b][:len(want)].tolist()) == want.tolist()
                assert np.all(inn[b][len(want):] == -1) and np.all(np.isneginf(vn[b][len(want):]))


def test_tc_filtered_fullsize(dev, lib):
    """4,096 users x 1,000,000 items x 768 with 1 % allow-sets (four filters mixed over the rows)."""
    B, N, d, K = 4096, 1_000_000, 768, 20
    rng = np.random.default_rng(5)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=5)
    allow_bool = _filters(N, (0.01, 0.01, 0.01, 0.01), rng)
    allow = _pack(allow_bool, dev)
    aor_np = (np.arange(B) % 4).astype(np.int32)
    aor = torch.as_tensor(aor_np, device=dev)
    seen = _seen(B, N, rng, 200)
    v, i = _tc_topk(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, _csr(seen, dev), allow, aor)

    def adm(b):
        ok = allow_bool[aor_np[b]].copy()
        ok[seen[b]] = False
        return np.flatnonzero(ok)
    _check_against_fp64(Ub, Eb, d, v, i, 0, N, K, adm, list(range(8)) + list(range(B - 8, B)))


# -- fp32 mode: hvae_mask_topk_filtered over materialised scores -------------------------------------------------------
def _mask_topk(lib, S, lo, n_it, K, mask, allow=None, aor=None):
    B = S.shape[0]
    S = S.clone()             # the kernel writes -inf over masked entries
    nc = int(lib.mask_topk_chunks(B, n_it))
    cv = torch.empty(B, nc * K, device=S.device)
    ci = torch.empty(B, nc * K, dtype=torch.int32, device=S.device)
    ov = torch.empty(B, K, device=S.device)
    oi = torch.empty(B, K, dtype=torch.int32, device=S.device)
    args = (S.data_ptr() + 4 * lo, S.stride(0), B, n_it, lo, mask[0].data_ptr(), mask[1].data_ptr(), None, 1)
    if allow is None:
        lib.mask_topk(*args, K, cv.data_ptr(), ci.data_ptr(), ov.data_ptr(), oi.data_ptr(), _st())
    else:
        lib.mask_topk_filtered(*args, allow.data_ptr(), allow.stride(0), aor.data_ptr(), K, cv.data_ptr(), ci.data_ptr(),
                               ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


@pytest.mark.parametrize("B,N,K", [(64, 70000, 20), (300, 5003, 100), (17, 40000, 32), (1, 2000, 8), (128, 1030, 128)])
def test_fp32_filtered_matches_torch(dev, lib, B, N, K):
    rng = np.random.default_rng(N)
    g = torch.Generator().manual_seed(B)
    S = torch.round(torch.randn(B, N, generator=g) * 64) / 64          # coarse values: many exact ties
    S = S.to(dev)
    allow_bool = _filters(N, (0.5, 0.05, 0.002), rng)
    allow = _pack(allow_bool, dev)
    aor_np = rng.integers(-1, 3, B).astype(np.int32)
    aor = torch.as_tensor(aor_np, device=dev)
    seen = _seen(B, N, rng, 80)
    mask = _csr(seen, dev)
    folded = _csr(_folded(seen, allow_bool, aor_np), dev)
    Sn = S.cpu().numpy()
    for lo, hi in [(0, N), (N // 3 + 5, N - 2)]:
        v, i = _mask_topk(lib, S, lo, hi - lo, K, mask, allow, aor)
        vn, inn = v.cpu().numpy(), i.cpu().numpy()
        assert np.all(inn[~np.isfinite(vn)] == -1)
        for b in range(B):
            row = Sn[b].astype(np.float64).copy()
            if aor_np[b] >= 0:
                row[~allow_bool[aor_np[b]]] = -np.inf
            row[seen[b]] = -np.inf
            ids = np.arange(lo, hi)
            r = row[lo:hi]
            order = np.lexsort((-ids, -r))[:K]                       # (score desc, id desc)
            fin = np.isfinite(r[order])
            n_fin = int(fin.sum())
            assert np.array_equal(inn[b][:n_fin], ids[order][:n_fin]), b
            assert np.array_equal(vn[b][:n_fin], r[order][:n_fin].astype(np.float32)), b
            assert not np.isfinite(vn[b][n_fin:]).any()
        # the filter folded into the mask: the same finite entries
        rv, ri = _mask_topk(lib, S, lo, hi - lo, K, folded)
        ri = torch.where(torch.isfinite(rv), ri, torch.full_like(ri, -1))
        assert torch.equal(v, rv) and torch.equal(i, ri)


def test_fp32_allow_everything_is_unfiltered(dev, lib):
    B, N, K = 200, 30000, 20
    rng = np.random.default_rng(9)
    S = torch.randn(B, N, generator=torch.Generator().manual_seed(9)).to(dev)
    mask = _csr(_seen(B, N, rng), dev)
    allow = _pack(np.ones((1, N), dtype=bool), dev)
    aor = torch.zeros(B, dtype=torch.int32, device=dev)
    v, i = _mask_topk(lib, S, 0, N, K, mask, allow, aor)
    rv, ri = _mask_topk(lib, S, 0, N, K, mask)
    assert torch.equal(v, rv) and torch.equal(i, ri)


# -- evaluator and service ---------------------------------------------------------------------------------------------------
def _world(dev, precision, n_users=150, n_items=3000):
    from hvae_b200.evaluate import RecommendationEvaluator
    from hvae_b200.model import HybridVAE
    from hvae_b200.synth import make_interactions, make_item_embeddings
    data = make_interactions(n_users, n_items, 2)
    torch.manual_seed(0)
    m = HybridVAE(n_items, make_item_embeddings(n_items, 64, 2), 64, [96], 0.5, 0.2, precision=precision).to(dev)
    m.eval()
    u2i = {f"u{i}": i for i in range(n_users)}
    i2it = {i: f"i{i}" for i in range(n_items)}
    ev = RecommendationEvaluator(m, data.scipy_csr(), u2i, {v: k for k, v in i2it.items()}, dev, batch_users=64)
    rng = np.random.default_rng(11)
    filters = {"a": rng.choice(n_items, 900, replace=False), "b": rng.choice(n_items, 60, replace=False),
               "c": rng.choice(n_items, 7, replace=False)}
    for k, v in filters.items():
        ev.add_item_filter(k, v)
    return ev, data, filters, i2it, rng


def test_evaluator_fp32_filtered_matches_reference(dev):
    ev, data, filters, _, rng = _world(dev, "fp32")
    n_users, N, K = 150, ev.n_items, 20
    users = np.arange(n_users)
    names = [(None, "a", "b", "c")[u % 4] for u in users]
    excl = [rng.choice(N, rng.integers(0, 40), replace=False) for _ in users]
    for exclude_seen in (True, False):
        v, i = ev.topk_users(users, K, exclude_seen, item_filter=names, exclude=excl)
        vn, inn = v.cpu().numpy(), i.cpu().numpy()
        csr = data.scipy_csr()
        for u in users:
            s = ev._get_user_scores(int(u)).astype(np.float64)
            ok = np.ones(N, dtype=bool)
            if names[u] is not None:
                ok[:] = False
                ok[filters[names[u]]] = True
            if exclude_seen:
                ok[csr[u].indices] = False
            ok[excl[u]] = False
            adm = np.flatnonzero(ok)
            order = adm[np.lexsort((-adm, -s[adm]))][:K]
            fin = np.isfinite(vn[u])
            n_fin = int(fin.sum())
            assert n_fin == len(order) and np.all(inn[u][n_fin:] == -1)
            got = inn[u][:n_fin]
            assert ok[got].all()
            np.testing.assert_allclose(vn[u][:n_fin], s[got], rtol=0, atol=1e-5)
            rest = np.setdiff1d(adm, got)
            if n_fin == K and rest.size:
                assert s[rest].max() <= vn[u][K - 1] + 1e-5
            # identical ids wherever the reference order has no near-tie
            ref_s = s[order]
            for p in range(n_fin):
                gap_prev = ref_s[p - 1] - ref_s[p] if p > 0 else np.inf
                gap_next = ref_s[p] - ref_s[p + 1] if p + 1 < len(ref_s) else np.inf
                if min(gap_prev, gap_next) >= 1e-5 and (p + 1 < n_fin or rest.size == 0 or ref_s[p] - s[rest].max() >= 1e-5):
                    assert got[p] == order[p], (u, p)


def test_evaluator_bf16_filtered_equals_folded_mask(dev):
    from hvae_b200.engine import Batch
    ev, data, filters, _, rng = _world(dev, "bf16")
    n_users, N = 150, ev.n_items
    users = np.arange(n_users)
    names = [(None, "a", "b", "c")[u % 4] for u in users]
    excl = [rng.choice(N, rng.integers(0, 40), replace=False) for _ in users]
    csr = data.scipy_csr()
    for K in (10, 100):
        v, i = ev.topk_users(users, K, True, item_filter=names, exclude=excl)
        rows = []
        for u in users:
            drop = np.union1d(csr[u].indices, excl[u])
            if names[u] is not None:
                drop = np.union1d(drop, np.setdiff1d(np.arange(N), filters[names[u]]))
            rows.append(drop.astype(np.int32))
        outs_v, outs_i = [], []
        for s in range(0, n_users, ev.batch_users):      # the evaluator's tiles: same GEMM shapes
            r = torch.as_tensor(users[s:s + ev.batch_users].astype(np.int32), device=dev)
            mask = _csr(rows[s:s + ev.batch_users], dev)
            with torch.no_grad():
                rv, ri = ev.model.engine.topk(Batch(ev._csr, r, r.shape[0], 1), K, True, mask=mask)
            outs_v.append(rv)
            outs_i.append(ri)
        assert torch.equal(v, torch.cat(outs_v)) and torch.equal(i, torch.cat(outs_i))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_service_mixed_batch(dev, precision):
    from hvae_b200.serve import RecommendService, UnknownUser
    ev, data, filters, i2it, rng = _world(dev, precision)
    svc = RecommendService.from_evaluator(ev, i2it)
    plain_before = [svc.recommend(f"u{u}", 10) for u in range(6)]
    for k, v in filters.items():
        svc.add_item_filter(k, [i2it[int(x)] for x in v])
    reqs = [("u0", 10, True), ("u1", 20, True, "a"), ("u2", 5, True, "c", ["i1", "nope", "i7"]), ("u3", 7, False, None, ["i3"]),
            ("u4", 10, True, "missing"), ("nobody", 5, True, "a"), ("u5", 100, False, "b"), ("u6", 3, True, None, ()),
            ("u7", 30, True, "c")]
    out = svc.recommend_many(reqs)
    for req, got in zip(reqs, out):
        kw = {}
        if len(req) > 3:
            kw["item_filter"] = req[3]
        if len(req) > 4:
            kw["exclude_items"] = req[4]
        try:
            want = svc.recommend(*req[:3], **kw)
        except (UnknownUser, ValueError) as e:
            assert type(got) is type(e) and str(got) == str(e)
            continue
        assert got == want
    assert isinstance(out[4], ValueError) and isinstance(out[5], UnknownUser)
    allowed_c = {i2it[int(x)] for x in filters["c"]}
    assert {r["item_id"] for r in out[2]["recommendations"]} <= allowed_c - {"i1", "i7"}
    assert len(out[8]["recommendations"]) <= 7
    assert all(r["item_id"] != "i3" for r in out[3]["recommendations"])
    # plain requests are untouched by the filters
    assert [svc.recommend(f"u{u}", 10) for u in range(6)] == plain_before

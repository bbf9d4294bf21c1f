"""GPU: boosted recommendations in the fused top-K kernels (hvae_tc_score_topk_boosted, hvae_mask_topk_boosted), the evaluator
(add_item_boost, topk_users(boost=, boost_weight=)) and the service (recommend(boost=, boost_weight=)).

Most cases use exact data: small-integer bf16 operands (every score an exact integer on the tensor cores and in fp32), dyadic
boost values and power-of-two weights, so that every key s + w * beta is exact in fp32 and the reference is a plain float64
(key desc, id desc) top-K without a tolerance.  The pruning cases put each block's only large boost on its lowest-scoring
column, and build a key that ties the K-th key only after rounding; rows without a boost are checked bit for bit against the
sampled kernels, the ids for invariance under batch layout, K, split count and item shards, and boosted + sampled rows for their
uniforms (tests/philox_ref.py) and their first-position frequencies against softmax((s + w beta) / tau)."""
import numpy as np
import pytest
import torch
from scipy.stats import chisquare

import philox_ref

pytestmark = pytest.mark.gpu

SAMPLE_STREAM = 0x53414D50


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


def _ptr(t):
    return None if t is None else t.data_ptr()


def _bf16(lib, x, dev):
    ld = (x.shape[1] + 7) // 8 * 8
    x = x.to(dev, torch.float32).contiguous()
    xb = torch.zeros(x.shape[0], ld, dtype=torch.bfloat16, device=dev)
    lib.cast_bf16(x.data_ptr(), x.shape[0], x.shape[1], x.shape[1], xb.data_ptr(), ld, _st())
    return xb, ld


def _int_operands(lib, B, N, d, dev, seed=0):
    """Integer-valued bf16 operands: every score is an exact integer on the tensor cores and in fp32."""
    g = torch.Generator().manual_seed(seed)
    U = torch.randint(-3, 4, (B, d), generator=g).float()
    E = torch.randint(-3, 4, (N, d), generator=g).float()
    return [*_bf16(lib, U, dev), *_bf16(lib, E, dev), (U.double() @ E.double().T).numpy()]


def _col_operands(lib, s_cols, dev, d=16):
    """bf16 operands whose scores are exactly s_cols[b, i] = sum_j U[b, j] E[i, j] with U rows one-hot: s_cols [B, N] given
    as up to d integer columns of E (E[:, j] for user j)."""
    B, N = s_cols.shape
    U = torch.zeros(B, d); U[torch.arange(B), torch.arange(B) % d] = 1.0
    E = torch.zeros(N, d)
    for b in range(min(B, d)):
        E[:, b] = torch.as_tensor(s_cols[b], dtype=torch.float32)
    return [*_bf16(lib, U, dev), *_bf16(lib, E, dev)]


def _pack(allow_bool, dev):
    F, n = allow_bool.shape
    bits = np.zeros((F, (n + 31) // 32 * 32), dtype=bool)
    bits[:, :n] = allow_bool
    return torch.as_tensor(np.packbits(bits, axis=1, bitorder="little").view(np.int32), device=dev)


def _csr(rows_items, dev):
    indptr = np.zeros(len(rows_items) + 1, dtype=np.int64)
    indptr[1:] = np.cumsum([len(r) for r in rows_items])
    idx = np.concatenate([np.asarray(r, dtype=np.int32) for r in rows_items]) if indptr[-1] else np.zeros(0, np.int32)
    return torch.as_tensor(indptr, device=dev), torch.as_tensor(idx, device=dev)


def _sample_args(inv_tau, seeds, dev):
    it = torch.as_tensor(np.asarray(inv_tau, dtype=np.float32), device=dev)
    sd = torch.as_tensor(np.asarray(seeds, dtype=np.uint64).view(np.int64), device=dev)
    return it, sd


def _boost_args(table, bor, w, dev):
    """(table [V, n] f32, its block bounds, boost_of_row int32 [B], weight f32 [B]) on the device."""
    from hvae_b200.tc import item_boost_bounds
    t = torch.as_tensor(np.asarray(table, dtype=np.float32), device=dev)
    return (t, item_boost_bounds(t), torch.as_tensor(np.asarray(bor, dtype=np.int32), device=dev),
            torch.as_tensor(np.asarray(w, dtype=np.float32), device=dev))


def _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask=None, allow=None, aor=None, sample=None, boost=None, e_ptr=None):
    """One launch over the global items [lo, hi) (E rows from e_ptr, default: row lo of Eb) -> merged (keys, ids).
    boost None: the sampled call (sample given) or the filtered one."""
    n_it = hi - lo
    ns = int(lib.tc_topk_splits(B, n_it))
    cv = torch.empty(B, ns * K, device=Ub.device)
    ci = torch.empty(B, ns * K, dtype=torch.int32, device=Ub.device)
    e_ptr = Eb.data_ptr() + 2 * lo * lde if e_ptr is None else e_ptr
    indptr, indices = mask if mask is not None else (None, None)
    args = (Ub.data_ptr(), ldu, B, e_ptr, lde, n_it, d, lo, _ptr(indptr), _ptr(indices), None, _ptr(allow),
            0 if allow is None else allow.stride(0), _ptr(aor))
    if boost is not None:
        t, bnd, bor, w = boost
        it, sd = sample if sample is not None else (None, None)
        lib.tc_score_topk_boosted(*args, _ptr(it), _ptr(sd), t.data_ptr(), t.stride(0), bnd.data_ptr(), bnd.stride(0),
                                  bor.data_ptr(), w.data_ptr(), K, cv.data_ptr(), ci.data_ptr(), _st())
    elif sample is not None:
        lib.tc_score_topk_sampled(*args, sample[0].data_ptr(), sample[1].data_ptr(), K, cv.data_ptr(), ci.data_ptr(), _st())
    else:
        lib.tc_score_topk_filtered(*args, K, cv.data_ptr(), ci.data_ptr(), _st())
    ov = torch.empty(B, K, device=Ub.device)
    oi = torch.empty(B, K, dtype=torch.int32, device=Ub.device)
    lib.topk_merge(cv.data_ptr(), ci.data_ptr(), B, ns * K, K, ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


def _scan(lib, S, lo, n_it, K, mask=None, allow=None, aor=None, sample=None, boost=None, s_ptr=None):
    """fp32 scan over the global items [lo, lo + n_it) of a copy of S (column 0 = item lo unless s_ptr is given)."""
    B = S.shape[0]
    S = S.clone()
    nc = int(lib.mask_topk_chunks(B, n_it))
    cv = torch.empty(B, nc * K, device=S.device)
    ci = torch.empty(B, nc * K, dtype=torch.int32, device=S.device)
    ov = torch.empty(B, K, device=S.device)
    oi = torch.empty(B, K, dtype=torch.int32, device=S.device)
    indptr, indices = mask if mask is not None else (None, None)
    args = (S.data_ptr() + 4 * (lo if s_ptr is None else s_ptr), S.stride(0), B, n_it, lo, _ptr(indptr), _ptr(indices), None,
            1 if mask is not None else 0, _ptr(allow), 0 if allow is None else allow.stride(0), _ptr(aor))
    if boost is not None:
        t, bnd, bor, w = boost
        it, sd = sample if sample is not None else (None, None)
        lib.mask_topk_boosted(*args, _ptr(it), _ptr(sd), t.data_ptr(), t.stride(0), bnd.data_ptr(), bnd.stride(0), bor.data_ptr(),
                              w.data_ptr(), K, cv.data_ptr(), ci.data_ptr(), ov.data_ptr(), oi.data_ptr(), _st())
    elif sample is not None:
        lib.mask_topk_sampled(*args, sample[0].data_ptr(), sample[1].data_ptr(), K, cv.data_ptr(), ci.data_ptr(), ov.data_ptr(),
                              oi.data_ptr(), _st())
    else:
        lib.mask_topk_filtered(*args, K, cv.data_ptr(), ci.data_ptr(), ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


def _ref_topk(key64, adm, K):
    """(keys, ids) of the float64 (key desc, id desc) top-K over the admissible global ids, padded with (-inf, -1)."""
    order = np.lexsort((-adm, -key64))[:K]
    keys = np.full(K, -np.inf); ids = np.full(K, -1)
    keys[:len(order)], ids[:len(order)] = key64[order], adm[order]
    return keys, ids


def _check_rows(vn, inn, s64, table, bor, w, adm_of, K, lo):
    for b in range(vn.shape[0]):
        adm = adm_of(b)
        key = s64[b, adm - lo] + (w[b] * table[bor[b], adm] if bor[b] >= 0 else 0.0)
        rk, ri = _ref_topk(key, adm, K)
        assert np.array_equal(inn[b], ri), (b, inn[b][:8], ri[:8])
        assert np.array_equal(vn[b], rk.astype(np.float32)), b


def _boost_table(rng, n, V=3):
    """V dyadic boost rows over n global ids; row 2 is zero except for a few very large values (pulls far-away items in)."""
    t = rng.integers(-64, 65, (V, n)).astype(np.float64) / 8
    t[2] = 0.0
    t[2, rng.choice(n, 5, replace=False)] = 4096.0
    return t


WEIGHTS = np.array([0.0, 1.0, -1.0, 0.5, -4.0, 2.0, 0.25, -0.5])


def _rows(B, n_total, rng):
    seen = [np.unique(rng.integers(0, n_total, rng.integers(0, 30))).astype(np.int32) for _ in range(B)]
    allow_bool = np.stack([rng.random(n_total) < 0.5, rng.random(n_total) < 0.05])
    aor = rng.integers(-1, 2, B).astype(np.int32)
    bor = rng.integers(-1, 3, B).astype(np.int32)
    w = rng.choice(WEIGHTS, B).astype(np.float32)

    def adm_of(lo, hi):
        def f(b):
            ok = np.ones(hi - lo, dtype=bool)
            if aor[b] >= 0:
                ok &= allow_bool[aor[b], lo:hi]
            s = seen[b][(seen[b] >= lo) & (seen[b] < hi)] - lo
            ok[s] = False
            return np.flatnonzero(ok) + lo
        return f
    return seen, allow_bool, aor, bor, w, adm_of


# -- exact reference -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,d,K", [(300, 5000, 64, 20), (77, 1000, 24, 1), (130, 4099, 32, 8), (129, 3001, 32, 12),
                                     (64, 2050, 64, 32), (96, 3001, 32, 100), (40, 2600, 24, 128)])
def test_tc_exact_reference(dev, lib, B, N, d, K):
    rng = np.random.default_rng(B + N + K)
    Ub, ldu, Eb, lde, S64 = _int_operands(lib, B, N, d, dev, seed=B)
    seen, allow_bool, aor, bor, w, adm_of = _rows(B, N, rng)
    table = _boost_table(rng, N)
    boost = _boost_args(table, bor, w, dev)
    mask, allow, aor_d = _csr(seen, dev), _pack(allow_bool, dev), torch.as_tensor(aor, device=dev)
    for lo, hi in [(0, N), (N // 3 + 5, N - 7)]:
        v, i = _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, allow, aor_d, boost=boost)
        _check_rows(v.cpu().numpy(), i.cpu().numpy(), S64, table, bor, w, adm_of(lo, hi), K, 0)


@pytest.mark.parametrize("B,N,K", [(64, 70000, 20), (300, 5003, 100), (17, 40000, 32), (1, 2000, 8), (128, 1030, 128),
                                   (33, 9000, 12)])
def test_scan_exact_reference(dev, lib, B, N, K):
    rng = np.random.default_rng(N + K)
    S64 = rng.integers(-40, 41, (B, N)).astype(np.float64) / 4
    S = torch.as_tensor(S64, dtype=torch.float32, device=dev)
    seen, allow_bool, aor, bor, w, adm_of = _rows(B, N, rng)
    table = _boost_table(rng, N)
    boost = _boost_args(table, bor, w, dev)
    mask, allow, aor_d = _csr(seen, dev), _pack(allow_bool, dev), torch.as_tensor(aor, device=dev)
    for lo, n_it in [(0, N), (N // 3 + 5, N - N // 3 - 12)]:
        v, i = _scan(lib, S, lo, n_it, K, mask, allow, aor_d, boost=boost)
        _check_rows(v.cpu().numpy(), i.cpu().numpy(), S64, table, bor, w, adm_of(lo, lo + n_it), K, 0)


@pytest.mark.parametrize("kernel", ["tc", "scan"])
def test_boost_pulls_in_from_far_outside(dev, lib, kernel):
    """A boost on the user's lowest-scoring item of 5,000 brings it to the top from far outside any plain top-128."""
    B, N, d, K = 8, 5000, 32, 10
    Ub, ldu, Eb, lde, S64 = _int_operands(lib, B, N, d, dev, seed=4)
    worst = np.argmin(S64, axis=1)
    table = np.zeros((B, N)); table[np.arange(B), worst] = 4096.0
    boost = _boost_args(table, np.arange(B), np.full(B, 1.0), dev)
    if kernel == "tc":
        _, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, boost=boost)
    else:
        _, i = _scan(lib, torch.as_tensor(S64, dtype=torch.float32, device=dev), 0, N, K, boost=boost)
    inn = i.cpu().numpy()
    for b in range(B):
        assert (S64[b] < S64[b, worst[b]]).sum() == 0 and (S64[b] > S64[b, worst[b]]).sum() > 128
        assert inn[b, 0] == worst[b]
        assert np.array_equal(inn[b, 1:], _ref_topk(S64[b], np.arange(N), K)[1][:K - 1])


# -- adversarial pruning ---------------------------------------------------------------------------------------------------------
OFFSETS = [0, 5, 37, 1000003]


@pytest.mark.parametrize("kernel", ["tc", "scan"])
@pytest.mark.parametrize("lo", OFFSETS)
def test_large_boost_on_lowest_score_of_each_block(dev, lib, kernel, lo):
    """Each aligned 32-block of global ids has one large boost, on its lowest-scoring column (so the block bound is far above
    every other column's key); with negative weights, the large negative value sits on the block's highest score."""
    B, N, d = 16, 6000, 16
    rng = np.random.default_rng(lo + 1)
    s_cols = rng.integers(-200, 201, (B, N)).astype(np.float64)
    Ub, ldu, Eb, lde = _col_operands(lib, s_cols, dev, d)
    g = np.arange(lo, lo + N)
    table = np.zeros((2, lo + N))
    for blk in np.unique(g >> 5):
        cols = np.flatnonzero((g >> 5) == blk)
        table[0, g[cols[np.argmin(s_cols[0, cols])]]] = rng.integers(150, 400)
        table[1, g[cols[np.argmax(s_cols[1, cols])]]] = rng.integers(150, 400)
    table = table.astype(np.float64)
    bor = np.array([0, 1] * (B // 2), dtype=np.int32)
    w = np.array([1.0, -1.0, 0.5, -0.5, 2.0, -2.0, 1.0, -1.0] * (B // 8), dtype=np.float32)
    bor[2::4] = 0; bor[3::4] = 1
    boost = _boost_args(table, bor, w, dev)
    seen = [np.unique(rng.integers(lo, lo + N, 20)).astype(np.int32) for _ in range(B)]
    for K in (1, 20, 100):
        if kernel == "tc":
            v, i = _tc(lib, Ub, ldu, Eb, lde, B, lo, lo + N, d, K, _csr(seen, dev), boost=boost, e_ptr=Eb.data_ptr())
        else:
            v, i = _scan(lib, torch.as_tensor(s_cols, dtype=torch.float32, device=dev), lo, N, K, _csr(seen, dev), boost=boost,
                         s_ptr=0)
        s_glob = np.zeros((B, lo + N)); s_glob[:, lo:] = s_cols
        adm_of = lambda b: g[~np.isin(g, seen[b])]
        _check_rows(v.cpu().numpy(), i.cpu().numpy(), s_glob, table, bor, w, adm_of, K, 0)


@pytest.mark.parametrize("kernel", ["tc", "scan"])
@pytest.mark.parametrize("lo", OFFSETS)
def test_rounded_key_ties_the_threshold(dev, lib, kernel, lo):
    """K = 8.  Items C1..C8 have s = 2^24 + 2 and no boost; item A (a higher id, tested after them) has s = 2^24 - 1 and
    beta = 2.5, so its key 2^24 + 1.5 rounds to 2^24 + 2, ties the list's K-th key and wins on its id.  A is admitted only if
    the list threshold is carried back through that rounding (2^24 + 2 - 2.5 itself rounds to 2^24 > s_A); the other columns
    score far below."""
    N, d, K = 3000, 16, 8
    s_cols = np.full((1, N), -1000.0)
    cs = np.arange(300, 308)
    a = (333 if kernel == "tc" else 2333) + lo % 7    # same CTA (tcgen05) / a later trip of the scan than the C's
    s_cols[0, cs], s_cols[0, a] = 2.0 ** 24 + 2, 2.0 ** 24 - 1
    table = np.zeros((1, lo + N)); table[0, lo + a] = 2.5
    boost = _boost_args(table, [0], [1.0], dev)
    if kernel == "tc":
        U = torch.zeros(1, d); U[0, 0], U[0, 1] = 4096.0, 1.0
        E = torch.zeros(N, d); E[:, 1] = -1000.0
        E[cs, 0], E[cs, 1], E[a, 0], E[a, 1] = 4096.0, 2.0, 4096.0, -1.0      # exact: 2^24 + 2 and 2^24 - 1
        (Ub, ldu), (Eb, lde) = _bf16(lib, U, dev), _bf16(lib, E, dev)
        v, i = _tc(lib, Ub, ldu, Eb, lde, 1, lo, lo + N, d, K, boost=boost, e_ptr=Eb.data_ptr())
    else:
        v, i = _scan(lib, torch.as_tensor(s_cols, dtype=torch.float32, device=dev), lo, N, K, boost=boost, s_ptr=0)
    assert i[0].tolist() == [lo + a] + (lo + cs[::-1][:K - 1]).tolist()
    assert np.all(v[0].cpu().numpy() == 2.0 ** 24 + 2)


# -- rows without a boost: bit for bit the sampled kernels ----------------------------------------------------------------------
@pytest.mark.parametrize("B,N,d,K", [(300, 5000, 768, 20), (77, 1000, 24, 1), (257, 3001, 384, 32), (64, 2050, 768, 33),
                                     (200, 9000, 384, 100), (513, 7000, 768, 12)])
def test_tc_unboosted_rows_equal_sampled(dev, lib, B, N, d, K):
    rng = np.random.default_rng(B * 3 + N)
    g = torch.Generator().manual_seed(B)
    Ub, ldu = _bf16(lib, torch.randn(B, d, generator=g) * 12.0 / d ** 0.5, dev)
    Eb, lde = _bf16(lib, torch.nn.functional.normalize(torch.randn(N, d, generator=g), dim=1), dev)
    seen, allow_bool, aor, bor, w, _ = _rows(B, N, rng)
    inv = rng.choice([0.0, 0.5, 2.0], B).astype(np.float32)
    sample = _sample_args(inv, rng.integers(0, 2 ** 62, B).astype(np.uint64), dev)
    table = rng.standard_normal((3, N))
    boost = _boost_args(table, bor, w, dev)
    plain = torch.as_tensor((bor < 0) | (w == 0), device=dev)
    assert 0 < int(plain.sum()) < B
    mask, allow, aor_d = _csr(seen, dev), _pack(allow_bool, dev), torch.as_tensor(aor, device=dev)
    for lo, hi in [(0, N), (N // 3 + 5, N - 7)]:
        for al, ao in [(allow, aor_d), (None, None)]:
            for smp in (sample, None):
                v, i = _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, al, ao, smp, boost)
                rv, ri = _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, al, ao, smp)
                assert torch.equal(v[plain], rv[plain]) and torch.equal(i[plain], ri[plain])
                assert not torch.equal(i[~plain], ri[~plain])


@pytest.mark.parametrize("B,N,K", [(64, 70000, 20), (300, 5003, 100), (17, 40000, 32), (2, 2000, 8), (128, 1030, 128)])
def test_scan_unboosted_rows_equal_sampled(dev, lib, B, N, K):
    rng = np.random.default_rng(N + 1)
    S = torch.round(torch.randn(B, N, generator=torch.Generator().manual_seed(B)) * 64).to(dev) / 64
    seen, allow_bool, aor, bor, w, _ = _rows(B, N, rng)
    bor[::2] = -1
    inv = rng.choice([0.0, 0.5, 2.0], B).astype(np.float32)
    sample = _sample_args(inv, rng.integers(0, 2 ** 62, B).astype(np.uint64), dev)
    boost = _boost_args(rng.standard_normal((3, N)), bor, w, dev)
    plain = torch.as_tensor((bor < 0) | (w == 0), device=dev)
    mask, allow, aor_d = _csr(seen, dev), _pack(allow_bool, dev), torch.as_tensor(aor, device=dev)
    for al, ao in [(allow, aor_d), (None, None)]:
        for smp in (sample, None):
            v, i = _scan(lib, S, 3, N - 5, K, mask, al, ao, smp, boost)
            rv, ri = _scan(lib, S, 3, N - 5, K, mask, al, ao, smp)
            assert torch.equal(v[plain], rv[plain]) and torch.equal(i[plain], ri[plain])


# -- invariance -------------------------------------------------------------------------------------------------------------------
def _merge(lib, parts, K, dev):
    cv = torch.cat([p[0] for p in parts], 1).contiguous()
    ci = torch.cat([p[1] for p in parts], 1).contiguous()
    B = cv.shape[0]
    ov = torch.empty(B, K, device=dev)
    oi = torch.empty(B, K, dtype=torch.int32, device=dev)
    lib.topk_merge(cv.data_ptr(), ci.data_ptr(), B, cv.shape[1], K, ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


def _sub(args, st):
    return tuple(a if k < 2 else a[st].contiguous() for k, a in enumerate(args))


def test_tc_invariance(dev, lib):
    B, N, d = 300, 20011, 768
    rng = np.random.default_rng(9)
    g = torch.Generator().manual_seed(9)
    Ub, ldu = _bf16(lib, torch.randn(B, d, generator=g) * 12.0 / d ** 0.5, dev)
    Eb, lde = _bf16(lib, torch.nn.functional.normalize(torch.randn(N, d, generator=g), dim=1), dev)
    boost = _boost_args(rng.standard_normal((2, N)), rng.integers(0, 2, B), rng.choice([-0.5, 0.25, 1.0], B), dev)
    v, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, 100, boost=boost)
    for k in (1, 5, 20, 32, 33):
        _, ik = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, k, boost=boost)
        assert torch.equal(ik, i[:, :k]), k
    for sub in (np.arange(B)[::-1].copy(), rng.permutation(B)[:7], np.array([17])):
        st = torch.as_tensor(sub, device=dev)
        _, isub = _tc(lib, Ub[st].contiguous(), ldu, Eb, lde, len(sub), 0, N, d, 100, boost=_sub(boost, st))
        assert torch.equal(isub, i[st])
    assert int(lib.tc_topk_splits(7, N)) != int(lib.tc_topk_splits(B, N))
    cuts = [0, 4999, 5003, 13001, N]                                                    # four ragged shards + merge
    parts = [_tc(lib, Ub, ldu, Eb, lde, B, a, b, d, 100, boost=boost) for a, b in zip(cuts[:-1], cuts[1:])]
    mv, mi = _merge(lib, parts, 100, dev)
    assert torch.equal(mi, i) and torch.equal(mv, v)


def test_scan_invariance(dev, lib):
    B, N = 200, 200003
    rng = np.random.default_rng(10)
    S = torch.randn(B, N, generator=torch.Generator().manual_seed(10)).to(dev) * 2
    boost = _boost_args(rng.standard_normal((2, N)), rng.integers(0, 2, B), rng.choice([-0.5, 0.25, 1.0], B), dev)
    v, i = _scan(lib, S, 0, N, 100, boost=boost)
    for k in (1, 5, 20, 32, 33):
        _, ik = _scan(lib, S, 0, N, k, boost=boost)
        assert torch.equal(ik, i[:, :k]), k
    for sub in (np.arange(B)[::-1].copy(), rng.permutation(B)[:3], np.array([17])):
        st = torch.as_tensor(sub, device=dev)
        _, isub = _scan(lib, S[st].contiguous(), 0, N, 100, boost=_sub(boost, st))
        assert torch.equal(isub, i[st])
    cuts = [0, 16385, 16390, 150001, N]
    parts = [_scan(lib, S, a, b - a, 100, boost=boost) for a, b in zip(cuts[:-1], cuts[1:])]
    mv, mi = _merge(lib, parts, 100, dev)
    assert torch.equal(mi, i) and torch.equal(mv, v)


# -- boosted + sampled --------------------------------------------------------------------------------------------------------------
def _uniform_index(seed, items):
    items = np.asarray(items, dtype=np.uint64)
    wds = philox_ref.philox4x32(items >> np.uint64(2), 0, SAMPLE_STREAM, 0, seed & 0xFFFFFFFF, seed >> 32)
    return (np.choose((items & np.uint64(3)).astype(np.int64), wds) >> 9).astype(np.int64)


@pytest.mark.parametrize("kernel", ["tc", "scan"])
def test_boosted_sampled_uniforms(dev, lib, kernel):
    """Scores c_i and a boost of -c_i / w: every boosted score is exactly 0, so the keys are the bare Gumbel noise and must
    give back each item's reference uniform exactly (with the boost ignored they would be c_i + g)."""
    seeds = [0, 12345, 2 ** 32, 2 ** 64 - 1]
    B, N, K, lo = len(seeds), 128, 128, 37
    rng = np.random.default_rng(21)
    c = rng.integers(-8, 9, N).astype(np.float64) * 2
    w = np.array([1.0, -2.0, 0.5, 4.0], dtype=np.float32)
    table = np.zeros((B, lo + N))
    for b in range(B):
        table[b, lo:] = -c / w[b]
    boost = _boost_args(table, np.arange(B), w, dev)
    sample = _sample_args(np.ones(B), seeds, dev)
    if kernel == "tc":
        Ub, ldu, Eb, lde = _col_operands(lib, np.tile(c, (B, 1)), dev)
        v, i = _tc(lib, Ub, ldu, Eb, lde, B, lo, lo + N, 16, K, sample=sample, boost=boost, e_ptr=Eb.data_ptr())
    else:
        v, i = _scan(lib, torch.as_tensor(np.tile(c, (B, 1)), dtype=torch.float32, device=dev), lo, N, K, sample=sample,
                     boost=boost, s_ptr=0)
    vn, inn = v.cpu().numpy().astype(np.float64), i.cpu().numpy()
    for b, seed in enumerate(seeds):
        assert sorted(inn[b].tolist()) == list(range(lo, lo + N))
        back = np.round(np.exp(-np.exp(-vn[b])) * 2.0 ** 23 - 0.5).astype(np.int64)
        assert np.array_equal(back, _uniform_index(seed, inn[b])), seed


@pytest.mark.parametrize("kernel", ["tc", "scan"])
def test_boosted_sampled_first_position(dev, lib, kernel):
    """First-position frequencies of 102,400 draws against softmax((s + w beta) / tau)."""
    N, B, n_launch, tau = 40, 4096, 25, 1.0
    s = ((np.arange(N) * 7) % 17 - 8) * 0.25
    beta = ((np.arange(N) * 5) % 11 - 5) * 0.5
    wt = -0.5
    first = []
    boost = _boost_args(beta[None], np.zeros(B), np.full(B, wt), dev)
    if kernel == "tc":
        U = torch.zeros(B, 16); U[:, 0] = 1.0
        E = torch.zeros(N, 16); E[:, 0] = torch.as_tensor(s, dtype=torch.float32)
        (Ub, ldu), (Eb, lde) = _bf16(lib, U, dev), _bf16(lib, E, dev)
    else:
        S = torch.as_tensor(np.tile(s, (B, 1)), dtype=torch.float32, device=dev)
    for L in range(n_launch):
        sample = _sample_args(np.full(B, 1 / tau), np.arange(B, dtype=np.uint64) + np.uint64(L * B + 3 * 2 ** 40), dev)
        if kernel == "tc":
            _, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, 16, 1, sample=sample, boost=boost)
        else:
            _, i = _scan(lib, S, 0, N, 1, sample=sample, boost=boost)
        first.append(i[:, 0].cpu().numpy())
    first = np.concatenate(first)
    p = np.exp((s + wt * beta) / tau); p /= p.sum()
    cnt = np.bincount(first, minlength=N)
    assert chisquare(cnt, p * len(first)).pvalue > 1e-4


# -- full size ---------------------------------------------------------------------------------------------------------------------
def test_tc_boosted_fullsize(dev, lib):
    """4,096 users x 1,000,000 items x 768, log-popularity-like boosts at mixed weights, some rows also sampled, seen items."""
    B, N, d, K = 4096, 1_000_000, 768, 20
    rng = np.random.default_rng(14)
    g = torch.Generator().manual_seed(14)
    Ub, ldu = _bf16(lib, torch.randn(B, d, generator=g) * 12.0 / d ** 0.5, dev)
    Eb, lde = _bf16(lib, torch.nn.functional.normalize(torch.randn(N, d, generator=g), dim=1), dev)
    table = np.stack([np.log1p(rng.zipf(1.5, N).clip(max=10 ** 6)), rng.standard_normal(N)])
    bor = rng.integers(-1, 2, B).astype(np.int32)
    w = rng.choice([-1.0, -0.1, 0.5, 0.0], B).astype(np.float32)
    boost = _boost_args(table, bor, w, dev)
    inv = rng.choice([0.0, 0.0, 1.0], B).astype(np.float32)
    sample = _sample_args(inv, rng.integers(0, 2 ** 62, B).astype(np.uint64), dev)
    drop = [np.unique(rng.integers(0, N, 200)).astype(np.int32) for _ in range(B)]
    v, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, _csr(drop, dev), sample=sample, boost=boost)
    inn, vn = i.cpu().numpy(), v.cpu().numpy()
    assert np.all(inn >= 0)
    il = i.long()
    s = torch.einsum("bd,bkd->bk", Ub[:, :d].double(), Eb[il][:, :, :d].double()).cpu().numpy()
    t32 = table.astype(np.float32)
    seeds = sample[1].cpu().numpy().view(np.uint64)
    for b in range(B):
        ids = inn[b]
        assert len(np.unique(ids)) == K and not np.isin(ids, drop[b]).any()
        assert np.all(np.diff(vn[b]) <= 0)
        key = s[b] + (float(w[b]) * t32[bor[b], ids].astype(np.float64) if bor[b] >= 0 else 0.0)    # recomputed from the id
        if inv[b] != 0:
            key = key * float(inv[b]) - np.log(-np.log((_uniform_index(int(seeds[b]), ids) + 0.5) * 2.0 ** -23))
        np.testing.assert_allclose(vn[b], key, rtol=0, atol=1e-4 + 1e-6 * np.abs(key).max())


# -- evaluator and service ------------------------------------------------------------------------------------------------------
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
    return ev, data, i2it


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_evaluator_boosted(dev, precision):
    ev, data, _ = _world(dev, precision)
    users = np.arange(150)
    csr = data.scipy_csr()
    pop = ev.item_popularity()
    assert pop.dtype == np.int64 and pop.sum() == csr.nnz and np.array_equal(pop, np.bincount(csr.indices, minlength=3000))
    logpop = np.round(np.log1p(pop) * 64) / 64                       # dyadic: every key s + w * value is one rounding
    ev.add_item_boost("pop", -logpop)
    rng = np.random.default_rng(5)
    fresh = np.zeros(3000); fresh[rng.choice(3000, 40, replace=False)] = 8.0
    ev.add_item_boost("fresh", fresh)
    names = [None if u % 4 == 0 else ("pop" if u % 2 else "fresh") for u in users]
    wts = [0.5 if u % 3 else -1.0 for u in users]
    v, i = ev.topk_users(users, 20, boost=names, boost_weight=wts)
    pv, pi = ev.topk_users(users, 20, item_filter=[None] * 150)       # the plain answer through the same eager path
    plain = torch.as_tensor([n is None for n in names], device=dev)
    assert torch.equal(v[plain], pv[plain]) and torch.equal(i[plain], pi[plain])
    vn, inn = v.cpu().numpy(), i.cpu().numpy()
    tables = {"pop": -logpop, "fresh": fresh}
    for u in users:
        s = ev._get_user_scores(int(u)).astype(np.float64)
        if names[u] is not None:
            key = (s + wts[u] * tables[names[u]]).astype(np.float32).astype(np.float64)
            adm = np.setdiff1d(np.arange(3000), csr[u].indices)
            rk, ri = _ref_topk(key[adm], adm, 20)
            tol = 1e-5 if precision == "fp32" else 0.05
            for p in range(20):                     # ids equal the reference away from near-ties of the keys
                if (p == 0 or rk[p - 1] - rk[p] > 2 * tol) and (p == 19 or rk[p] - rk[p + 1] > 2 * tol):
                    assert inn[u, p] == ri[p], (u, p)
        # the values are the model's scores of the chosen items, not the keys
        np.testing.assert_allclose(vn[u], s[inn[u]], rtol=1e-5 if precision == "fp32" else 2e-2,
                                   atol=1e-5 if precision == "fp32" else 1e-2)         # (bf16 operands: about 5e-3 here)
    with pytest.raises(ValueError):
        ev.topk_users(users, 10, boost="nope")
    with pytest.raises(ValueError):
        ev.topk_users(users, 10, boost="pop", boost_weight=2e3)
    with pytest.raises(ValueError):
        ev.add_item_boost("bad", np.full(3000, np.inf))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_service_boosted_alone_and_batched(dev, precision):
    from hvae_b200.serve import MicroBatcher, RecommendService
    ev, _, i2it = _world(dev, precision)
    svc = RecommendService.from_evaluator(ev, i2it)
    svc.add_item_boost("promo", {i2it[k]: 4.0 for k in range(0, 3000, 97)})
    reqs = [dict(user_id="u1", top_k=10, boost="promo"), dict(user_id="u2", top_k=50, boost="promo", boost_weight=-0.5),
            dict(user_id="u3", top_k=5, boost="promo", temperature=1.0, seed=7), dict(user_id="u4", top_k=20)]
    alone = [svc.recommend(**r) for r in reqs]
    with MicroBatcher(svc, max_batch=64, max_wait_ms=20) as mb:
        futs = [mb.submit(**r) for r in reqs] + [mb.submit(f"u{k}", 100, boost="promo", boost_weight=0.25) for k in range(10, 40)]
        batched = [f.result() for f in futs]
    assert batched[:4] == alone
    assert alone[0]["boost"] == "promo" and alone[0]["boost_weight"] == 1.0 and "boost" not in alone[3]
    promo = {i2it[k] for k in range(0, 3000, 97)}
    assert sum(r["item_id"] in promo for r in alone[0]["recommendations"]) > 0
    s = ev._get_user_scores(1)
    for r in alone[0]["recommendations"]:          # "score" is the model's score
        want = s[int(r["item_id"][1:])]
        assert abs(r["score"] - want) <= (1e-5 + 1e-5 * abs(want) if precision == "fp32" else 1e-2 + 2e-2 * abs(want))

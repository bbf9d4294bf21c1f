"""GPU: sampled recommendations (Gumbel-top-K) in the fused top-K kernels (hvae_tc_score_topk_sampled,
hvae_mask_topk_sampled), the evaluator (topk_users(temperature=, seed=)) and the service (recommend(temperature=, seed=)).

The noise is checked against the numpy Philox of tests/philox_ref.py: the kernels' keys s / tau + g give back each item's
uniform exactly.  Draws are checked against the float64 Gumbel-top-K of exact scores on those uniforms, rows with
1/tau = 0 bit for bit against the filtered kernels, the ids for invariance under batch layout, K, split count and item
shards, and the frequencies of the first two positions against softmax(s / tau) and its Plackett-Luce conditional."""
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


def _r8(n):
    return (n + 7) // 8 * 8


def _bf16(lib, x, dev):
    ld = _r8(x.shape[1])
    x = x.to(dev, torch.float32).contiguous()
    xb = torch.zeros(x.shape[0], ld, dtype=torch.bfloat16, device=dev)
    lib.cast_bf16(x.data_ptr(), x.shape[0], x.shape[1], x.shape[1], xb.data_ptr(), ld, _st())
    return xb, ld


def _operands(lib, B, N, d, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    U = torch.randn(B, d, generator=g) * 12.0 / d ** 0.5
    E = torch.nn.functional.normalize(torch.randn(N, d, generator=g), dim=1)
    return _bf16(lib, U, dev) + _bf16(lib, E, dev)


def _int_operands(lib, B, N, d, dev, seed=0):
    """Integer-valued bf16 operands: every score is an exact integer on the tensor cores and in fp32."""
    g = torch.Generator().manual_seed(seed)
    U = torch.randint(-3, 4, (B, d), generator=g).float()
    E = torch.randint(-3, 4, (N, d), generator=g).float()
    return [*_bf16(lib, U, dev), *_bf16(lib, E, dev), (U.double() @ E.double().T).numpy()]


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


def _seen(B, n_total, rng, per_row=30):
    return [np.unique(rng.integers(0, n_total, rng.integers(0, per_row))).astype(np.int32) for _ in range(B)]


def _sample_args(inv_tau, seeds, dev):
    it = torch.as_tensor(np.asarray(inv_tau, dtype=np.float32), device=dev)
    sd = torch.as_tensor(np.asarray(seeds, dtype=np.uint64).view(np.int64), device=dev)
    return it, sd


def _ptr(t):
    return None if t is None else t.data_ptr()


def _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask=None, allow=None, aor=None, sample=None, e_ptr=None):
    """One launch over the global items [lo, hi) (E rows from e_ptr, default: row lo of Eb) -> merged (keys, ids)."""
    n_it = hi - lo
    ns = int(lib.tc_topk_splits(B, n_it))
    cv = torch.empty(B, ns * K, device=Ub.device)
    ci = torch.empty(B, ns * K, dtype=torch.int32, device=Ub.device)
    e_ptr = Eb.data_ptr() + 2 * lo * lde if e_ptr is None else e_ptr
    indptr, indices = mask if mask is not None else (None, None)
    args = (Ub.data_ptr(), ldu, B, e_ptr, lde, n_it, d, lo, _ptr(indptr), _ptr(indices), None, _ptr(allow),
            0 if allow is None else allow.stride(0), _ptr(aor))
    if sample is None:
        lib.tc_score_topk_filtered(*args, K, cv.data_ptr(), ci.data_ptr(), _st())
    else:
        lib.tc_score_topk_sampled(*args, sample[0].data_ptr(), sample[1].data_ptr(), K, cv.data_ptr(), ci.data_ptr(), _st())
    ov = torch.empty(B, K, device=Ub.device)
    oi = torch.empty(B, K, dtype=torch.int32, device=Ub.device)
    lib.topk_merge(cv.data_ptr(), ci.data_ptr(), B, ns * K, K, ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


def _scan(lib, S, lo, n_it, K, mask=None, allow=None, aor=None, sample=None, s_ptr=None, lds=None):
    """fp32 scan over the global items [lo, lo + n_it) of a copy of S (column 0 = item lo unless s_ptr is given)."""
    B = S.shape[0]
    S = S.clone()
    nc = int(lib.mask_topk_chunks(B, n_it))
    cv = torch.empty(B, nc * K, device=S.device)
    ci = torch.empty(B, nc * K, dtype=torch.int32, device=S.device)
    ov = torch.empty(B, K, device=S.device)
    oi = torch.empty(B, K, dtype=torch.int32, device=S.device)
    indptr, indices = mask if mask is not None else (None, None)
    args = (S.data_ptr() + 4 * lo if s_ptr is None else S.data_ptr() + 4 * s_ptr, S.stride(0) if lds is None else lds, B, n_it, lo,
            _ptr(indptr), _ptr(indices), None, 1 if mask is not None else 0, _ptr(allow), 0 if allow is None else allow.stride(0),
            _ptr(aor))
    if sample is None:
        lib.mask_topk_filtered(*args, K, cv.data_ptr(), ci.data_ptr(), ov.data_ptr(), oi.data_ptr(), _st())
    else:
        lib.mask_topk_sampled(*args, sample[0].data_ptr(), sample[1].data_ptr(), K, cv.data_ptr(), ci.data_ptr(), ov.data_ptr(),
                              oi.data_ptr(), _st())
    return ov, oi


def _words(seed, items):
    items = np.asarray(items, dtype=np.uint64)
    w = philox_ref.philox4x32(items >> np.uint64(2), 0, SAMPLE_STREAM, 0, seed & 0xFFFFFFFF, seed >> 32)
    k = (items & np.uint64(3)).astype(np.int64)
    return np.choose(k, w)


def _uniform_index(seed, items):
    """r >> 9 of each item: u = (index + 0.5) 2^-23."""
    return (_words(seed, items) >> 9).astype(np.int64)


def _gumbel64(seed, items):
    u = (_uniform_index(seed, items) + 0.5) * 2.0 ** -23
    return -np.log(-np.log(u))


def _key_tol(s_inv):
    """|device key - float64 key| bound: the rounding of fmaf plus the two 1-ulp logf of g (< 2^-21 (1 + |g|))."""
    return 2.0 ** -23 * np.abs(s_inv) + 2.0 ** -21 * 20 + 1e-30


# -- noise: uniforms bit for bit ---------------------------------------------------------------------------------------------
SEEDS = [0, 1, 12345, 2 ** 32 - 1, 2 ** 32, 2 ** 63 + 987654321, 2 ** 64 - 2, 2 ** 64 - 1]
OFFSETS = [0, 5, (1 << 20) + 3, 2 ** 31 - 257, 2 ** 31 - 260]     # (item_offset + 256 stays below 2^31)


def _check_uniforms(keys, ids, seed, items):
    """keys = g of the items (scores 0, 1/tau = 1): each must give back the reference uniform's index exactly."""
    assert sorted(ids.tolist()) == sorted(items.tolist())
    idx = _uniform_index(seed, ids)
    g = keys.astype(np.float64)
    back = np.round(np.exp(-np.exp(-g)) * 2.0 ** 23 - 0.5).astype(np.int64)
    assert np.array_equal(back, idx), (seed, np.flatnonzero(back != idx)[:5])
    g64 = _gumbel64(seed, ids)
    assert np.all(np.abs(g - g64) <= 2.0 ** -21 * np.maximum(1.0, np.abs(g64)))
    assert g.max() < 16.64


def test_tc_uniforms_bit_exact(dev, lib):
    N, d, K = 128, 16, 128
    Ub, ldu = _bf16(lib, torch.zeros(len(SEEDS), d), dev)
    Eb, lde = _bf16(lib, torch.zeros(N, d), dev)
    sample = _sample_args(np.ones(len(SEEDS)), SEEDS, dev)
    for lo in OFFSETS:
        v, i = _tc(lib, Ub, ldu, Eb, lde, len(SEEDS), lo, lo + N, d, K, sample=sample, e_ptr=Eb.data_ptr())
        vn, inn = v.cpu().numpy(), i.cpu().numpy()
        for r, seed in enumerate(SEEDS):
            _check_uniforms(vn[r], inn[r], seed, np.arange(lo, lo + N))


def test_scan_uniforms_bit_exact(dev, lib):
    N, K = 128, 128
    S = torch.zeros(len(SEEDS), N + 8, device=dev)
    sample = _sample_args(np.ones(len(SEEDS)), SEEDS, dev)
    for lo in OFFSETS:
        for col0 in (0, 1, 3):           # 16-byte aligned row start or not: head, body and tail columns
            v, i = _scan(lib, S, lo, N, K, sample=sample, s_ptr=col0)
            vn, inn = v.cpu().numpy(), i.cpu().numpy()
            for r, seed in enumerate(SEEDS):
                _check_uniforms(vn[r], inn[r], seed, np.arange(lo, lo + N))


# -- exactness against float64 Gumbel-top-K ---------------------------------------------------------------------------------
def _check_draw(keys, ids, s64, inv_tau, seed, adm, K, lo=0):
    """The ids equal the float64 Gumbel-top-K of s64 over the admissible global ids, except across near-ties of the keys."""
    if inv_tau == 0:
        key64 = s64[adm - lo]
    else:
        key64 = s64[adm - lo] * np.float64(np.float32(inv_tau)) + _gumbel64(seed, adm)
    order = np.lexsort((-adm, -key64))
    ref, rk = adm[order][:K], key64[order]
    n = len(ref)
    assert np.all(ids[n:] == -1) and np.all(np.isneginf(keys[n:]))
    assert len(set(ids[:n].tolist())) == n and np.isin(ids[:n], adm).all()
    tol = 2 * _key_tol(rk[:min(n + 1, len(rk))]).max() if inv_tau else 0.0
    for p in range(n):
        gap_prev = rk[p - 1] - rk[p] if p > 0 else np.inf
        gap_next = rk[p] - rk[p + 1] if p + 1 < len(rk) else np.inf
        if min(gap_prev, gap_next) > tol:
            assert ids[p] == ref[p], (p, ids[:n], ref)
    np.testing.assert_allclose(keys[:n], rk[:n], rtol=0, atol=tol + 1e-30)


def _rows_setup(B, N, rng, dev):
    allow_bool = np.stack([rng.random(N) < 0.5, rng.random(N) < 0.05])
    aor_np = rng.integers(-1, 2, B).astype(np.int32)
    seen = _seen(B, N, rng)
    inv = rng.choice([0.0, 0.25, 1.0, 4.0, 1 / 0.3], B).astype(np.float32)
    seeds = rng.integers(0, 2 ** 63, B, dtype=np.int64).astype(np.uint64) * np.uint64(2) + np.uint64(1)

    def adm(b, lo, hi):
        ok = np.ones(hi - lo, dtype=bool)
        if aor_np[b] >= 0:
            ok &= allow_bool[aor_np[b], lo:hi]
        s = seen[b][(seen[b] >= lo) & (seen[b] < hi)] - lo
        ok[s] = False
        return np.flatnonzero(ok) + lo
    return allow_bool, aor_np, seen, inv, seeds, adm


@pytest.mark.parametrize("B,N,d,K", [(300, 5000, 64, 20), (77, 1000, 24, 1), (130, 4099, 32, 8), (64, 2050, 64, 33),
                                     (96, 3001, 32, 100), (40, 2600, 24, 128)])
def test_tc_exact_scores_match_float64(dev, lib, B, N, d, K):
    rng = np.random.default_rng(B + N)
    Ub, ldu, Eb, lde, S64 = _int_operands(lib, B, N, d, dev, seed=B)
    allow_bool, aor_np, seen, inv, seeds, adm = _rows_setup(B, N, rng, dev)
    allow, aor = _pack(allow_bool, dev), torch.as_tensor(aor_np, device=dev)
    sample = _sample_args(inv, seeds, dev)
    for lo, hi in [(0, N), (N // 3 + 5, N - 7)]:
        v, i = _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, _csr(seen, dev), allow, aor, sample)
        vn, inn = v.cpu().numpy(), i.cpu().numpy()
        for b in range(B):
            _check_draw(vn[b], inn[b], S64[b, lo:hi], inv[b], int(seeds[b]), adm(b, lo, hi), K, lo)
        # the drawn items' scores, recomputed by hvae_candidate_rank (id -1: -inf, nothing read)
        sc = torch.empty(B, K, device=dev)
        rank = torch.empty(B, dtype=torch.int32, device=dev)
        lib.candidate_rank(Ub.data_ptr(), ldu, Eb.data_ptr(), lde, d, 1, i.data_ptr(), K, B, sc.data_ptr(), rank.data_ptr(), _st())
        scn = sc.cpu().numpy()
        want = np.where(inn >= 0, S64[np.arange(B)[:, None], np.maximum(inn, 0)], -np.inf)
        assert np.array_equal(scn, want.astype(np.float32))


@pytest.mark.parametrize("B,N,K", [(64, 70000, 20), (300, 5003, 100), (17, 40000, 32), (1, 2000, 8), (128, 1030, 128)])
def test_scan_exact_scores_match_float64(dev, lib, B, N, K):
    rng = np.random.default_rng(N)
    S64 = rng.integers(-40, 41, (B, N)).astype(np.float64) / 4
    S = torch.as_tensor(S64, dtype=torch.float32, device=dev)
    allow_bool, aor_np, seen, inv, seeds, adm = _rows_setup(B, N, rng, dev)
    allow, aor = _pack(allow_bool, dev), torch.as_tensor(aor_np, device=dev)
    sample = _sample_args(inv, seeds, dev)
    for lo, n_it in [(0, N), (N // 3 + 5, N - N // 3 - 12)]:
        v, i = _scan(lib, S, lo, n_it, K, _csr(seen, dev), allow, aor, sample)
        vn, inn = v.cpu().numpy(), i.cpu().numpy()
        for b in range(B):
            _check_draw(vn[b], inn[b], S64[b, lo:lo + n_it], inv[b], int(seeds[b]), adm(b, lo, lo + n_it), K, lo)


# -- deterministic rows: bit for bit the filtered kernels ---------------------------------------------------------------------
@pytest.mark.parametrize("B,N,d,K", [(300, 5000, 768, 20), (77, 1000, 24, 1), (130, 4099, 384, 8), (257, 3001, 384, 32),
                                     (64, 2050, 768, 33), (200, 9000, 384, 100), (129, 12101, 24, 128), (513, 7000, 768, 12),
                                     (96, 2600, 384, 16), (96, 2600, 24, 24)])
def test_tc_plain_rows_equal_filtered(dev, lib, B, N, d, K):
    rng = np.random.default_rng(B * 3 + N)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=B)
    allow_bool, aor_np, seen, inv, seeds, _ = _rows_setup(B, N, rng, dev)
    inv[::3] = 0.0
    allow, aor, mask = _pack(allow_bool, dev), torch.as_tensor(aor_np, device=dev), _csr(seen, dev)
    sample = _sample_args(inv, seeds, dev)
    plain = torch.as_tensor(inv == 0, device=dev)
    for lo, hi in [(0, N), (N // 3 + 5, N - 7)]:
        for al, ao in [(allow, aor), (None, None)]:
            v, i = _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, al, ao, sample)
            rv, ri = _tc(lib, Ub, ldu, Eb, lde, B, lo, hi, d, K, mask, al, ao)
            assert torch.equal(v[plain], rv[plain]) and torch.equal(i[plain], ri[plain])
            assert not torch.equal(i[~plain], ri[~plain])


@pytest.mark.parametrize("B,N,K", [(64, 70000, 20), (300, 5003, 100), (17, 40000, 32), (2, 2000, 8), (128, 1030, 128)])
def test_scan_plain_rows_equal_filtered(dev, lib, B, N, K):
    rng = np.random.default_rng(N + 1)
    S = torch.round(torch.randn(B, N, generator=torch.Generator().manual_seed(B)) * 64).to(dev) / 64
    allow_bool, aor_np, seen, inv, seeds, _ = _rows_setup(B, N, rng, dev)
    inv[::2] = 0.0
    allow, aor, mask = _pack(allow_bool, dev), torch.as_tensor(aor_np, device=dev), _csr(seen, dev)
    sample = _sample_args(inv, seeds, dev)
    plain = torch.as_tensor(inv == 0, device=dev)
    for al, ao in [(allow, aor), (None, None)]:
        v, i = _scan(lib, S, 3, N - 5, K, mask, al, ao, sample)
        rv, ri = _scan(lib, S, 3, N - 5, K, mask, al, ao)
        assert torch.equal(v[plain], rv[plain]) and torch.equal(i[plain], ri[plain])


# -- invariance ---------------------------------------------------------------------------------------------------------------
def _merge(lib, parts, K, dev):
    cv = torch.cat([p[0] for p in parts], 1).contiguous()
    ci = torch.cat([p[1] for p in parts], 1).contiguous()
    B = cv.shape[0]
    ov = torch.empty(B, K, device=dev)
    oi = torch.empty(B, K, dtype=torch.int32, device=dev)
    lib.topk_merge(cv.data_ptr(), ci.data_ptr(), B, cv.shape[1], K, ov.data_ptr(), oi.data_ptr(), _st())
    return ov, oi


def test_tc_invariance(dev, lib):
    B, N, d = 300, 20011, 768
    rng = np.random.default_rng(9)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=9)
    inv = rng.choice([0.25, 1.0, 4.0], B).astype(np.float32)
    seeds = rng.integers(0, 2 ** 62, B).astype(np.uint64)
    sample = _sample_args(inv, seeds, dev)
    v, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, 100, sample=sample)
    v2, i2 = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, 100, sample=sample)               # repeated launch
    assert torch.equal(v, v2) and torch.equal(i, i2)
    for k in (1, 5, 20, 32, 33):                                                        # a k-draw is the K-draw's prefix
        _, ik = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, k, sample=sample)
        assert torch.equal(ik, i[:, :k]), k
    for sub in (np.arange(B)[::-1].copy(), rng.permutation(B)[:7], np.array([17])):     # other rows, positions, split counts
        assert int(lib.tc_topk_splits(len(sub), N)) >= 1
        st = torch.as_tensor(sub, device=dev)
        _, isub = _tc(lib, Ub[st].contiguous(), ldu, Eb, lde, len(sub), 0, N, d, 100,
                      sample=(sample[0][st].contiguous(), sample[1][st].contiguous()))
        assert torch.equal(isub, i[st])
    assert int(lib.tc_topk_splits(7, N)) != int(lib.tc_topk_splits(B, N))
    cuts = [0, 4999, 5003, 13001, N]                                                    # four ragged shards + merge
    parts = [_tc(lib, Ub, ldu, Eb, lde, B, a, b, d, 100, sample=sample) for a, b in zip(cuts[:-1], cuts[1:])]
    mv, mi = _merge(lib, parts, 100, dev)
    assert torch.equal(mi, i) and torch.equal(mv, v)


def test_scan_invariance(dev, lib):
    B, N = 200, 200003
    rng = np.random.default_rng(10)
    S = torch.randn(B, N, generator=torch.Generator().manual_seed(10)).to(dev) * 2
    inv = rng.choice([0.25, 1.0, 4.0], B).astype(np.float32)
    seeds = rng.integers(0, 2 ** 62, B).astype(np.uint64)
    sample = _sample_args(inv, seeds, dev)
    v, i = _scan(lib, S, 0, N, 100, sample=sample)
    v2, i2 = _scan(lib, S, 0, N, 100, sample=sample)
    assert torch.equal(v, v2) and torch.equal(i, i2)
    for k in (1, 5, 20, 32, 33):
        _, ik = _scan(lib, S, 0, N, k, sample=sample)
        assert torch.equal(ik, i[:, :k]), k
    for sub in (np.arange(B)[::-1].copy(), rng.permutation(B)[:3], np.array([17])):    # (chunk count follows the row count)
        st = torch.as_tensor(sub, device=dev)
        _, isub = _scan(lib, S[st].contiguous(), 0, N, 100, sample=(sample[0][st].contiguous(), sample[1][st].contiguous()))
        assert torch.equal(isub, i[st])
    assert int(lib.mask_topk_chunks(1, N)) != int(lib.mask_topk_chunks(B, N))
    cuts = [0, 16385, 16390, 150001, N]
    parts = [_scan(lib, S, a, b - a, 100, sample=sample) for a, b in zip(cuts[:-1], cuts[1:])]
    mv, mi = _merge(lib, parts, 100, dev)
    assert torch.equal(mi, i) and torch.equal(mv, v)


def test_tc_and_scan_draw_the_same_items(dev, lib):
    """The same exact scores through both kernels: the same keys, so the same draws."""
    B, N, d, K = 64, 3000, 32, 20
    Ub, ldu, Eb, lde, S64 = _int_operands(lib, B, N, d, dev, seed=3)
    rng = np.random.default_rng(3)
    sample = _sample_args(rng.choice([0.5, 1.0, 2.0], B), rng.integers(0, 2 ** 62, B).astype(np.uint64), dev)
    v, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, sample=sample)
    sv, si = _scan(lib, torch.as_tensor(S64, dtype=torch.float32, device=dev), 0, N, K, sample=sample)
    assert torch.equal(i, si) and torch.equal(v, sv)


# -- distribution --------------------------------------------------------------------------------------------------------------
def _draws(kernel, lib, dev, s, tau, n_launch, B, allow_bool=None, seen=None):
    """First and second drawn ids of n_launch * B rows that all have the scores s, each with its own seed."""
    N = len(s)
    first, second = [], []
    allow = aor = mask = None
    if allow_bool is not None:
        allow, aor = _pack(allow_bool[None], dev), torch.zeros(B, dtype=torch.int32, device=dev)
    if seen is not None:
        mask = _csr([seen] * B, dev)
    if kernel == "tc":
        d = 16
        U = torch.zeros(B, d); U[:, 0] = 1.0
        E = torch.zeros(N, d); E[:, 0] = torch.as_tensor(s, dtype=torch.float32)
        (Ub, ldu), (Eb, lde) = _bf16(lib, U, dev), _bf16(lib, E, dev)
    else:
        S = torch.as_tensor(np.tile(s, (B, 1)), dtype=torch.float32, device=dev)
    for L in range(n_launch):
        sample = _sample_args(np.full(B, 1 / tau), np.arange(B, dtype=np.uint64) + np.uint64(L * B + 7 * 2 ** 40), dev)
        if kernel == "tc":
            _, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, 2, mask, allow, aor, sample)
        else:
            _, i = _scan(lib, S, 0, N, 2, mask, allow, aor, sample)
        i = i.cpu().numpy()
        first.append(i[:, 0]); second.append(i[:, 1])
    return np.concatenate(first), np.concatenate(second)


@pytest.mark.parametrize("kernel", ["tc", "scan"])
@pytest.mark.parametrize("tau,restricted", [(1.0, False), (0.5, False), (2.0, True)])
def test_distribution_first_two_positions(dev, lib, kernel, tau, restricted):
    N = 50
    s = ((np.arange(N) * 7) % 17 - 8) * 0.25                     # exact in bf16
    ok = np.ones(N, dtype=bool)
    allow_bool = seen = None
    if restricted:
        allow_bool = np.zeros(N, dtype=bool); allow_bool[np.arange(0, N, 5)] = True; allow_bool[np.arange(1, N, 3)] = True
        seen = np.array([1, 10, 25], dtype=np.int32)
        ok = allow_bool.copy(); ok[seen] = False
    first, second = _draws(kernel, lib, dev, s, tau, 50, 4096, allow_bool, seen)
    n = len(first)
    assert n >= 200_000
    adm = np.flatnonzero(ok)
    assert np.isin(first, adm).all() and np.isin(second, adm).all() and np.all(first != second)
    w = np.exp(s[adm] / tau)
    p1 = w / w.sum()
    # P(second = j) = sum_{i != j} p_i p_j / (1 - p_i)
    p2 = np.array([sum(p1[a] * p1[b] / (1 - p1[a]) for a in range(len(adm)) if a != b) for b in range(len(adm))])
    for got, p in ((first, p1), (second, p2)):
        cnt = np.array([(got == a).sum() for a in adm])
        assert chisquare(cnt, p * n).pvalue > 1e-4, (kernel, tau, restricted)


# -- edge cases ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["tc", "scan"])
def test_fewer_admissible_than_k(dev, lib, kernel):
    B, N, d, K = 40, 3000, 32, 20
    rng = np.random.default_rng(12)
    Ub, ldu, Eb, lde, S64 = _int_operands(lib, B, N, d, dev, seed=12)
    few = np.zeros(N, dtype=bool); few[rng.choice(N, 6, replace=False)] = True
    allow, aor = _pack(few[None], dev), torch.zeros(B, dtype=torch.int32, device=dev)
    seen = [np.flatnonzero(few)[:1].astype(np.int32)] * B
    sample = _sample_args(np.full(B, 0.7), np.arange(B, dtype=np.uint64), dev)
    if kernel == "tc":
        v, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, _csr(seen, dev), allow, aor, sample)
    else:
        v, i = _scan(lib, torch.as_tensor(S64, dtype=torch.float32, device=dev), 0, N, K, _csr(seen, dev), allow, aor, sample)
    vn, inn = v.cpu().numpy(), i.cpu().numpy()
    want = sorted(np.flatnonzero(few)[1:].tolist())
    for b in range(B):
        assert sorted(inn[b][:5].tolist()) == want and np.all(np.isfinite(vn[b][:5]))
        assert np.all(inn[b][5:] == -1) and np.all(np.isneginf(vn[b][5:]))


@pytest.mark.parametrize("kernel", ["tc", "scan"])
def test_tiny_temperature_is_top_k(dev, lib, kernel):
    """tau = 1e-3 with score gaps >= 1 > 17 tau: the draw is the deterministic top-K."""
    B, N, d, K = 64, 200, 16, 32
    rng = np.random.default_rng(13)
    U = torch.zeros(B, d); U[:, 0] = torch.as_tensor(rng.choice([-2.0, -1.0, 1.0, 2.0], B), dtype=torch.float32)
    E = torch.zeros(N, d); E[:, 0] = torch.as_tensor(rng.permutation(N) - 100.0, dtype=torch.float32)
    (Ub, ldu), (Eb, lde) = _bf16(lib, U, dev), _bf16(lib, E, dev)
    S = (U.double() @ E.double().T).float().to(dev)
    seen = _csr(_seen(B, N, rng, 10), dev)
    sample = _sample_args(np.full(B, np.float32(1 / 1e-3)), rng.integers(0, 2 ** 62, B).astype(np.uint64), dev)
    if kernel == "tc":
        _, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, seen, sample=sample)
        _, ri = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, seen)
    else:
        _, i = _scan(lib, S, 0, N, K, seen, sample=sample)
        _, ri = _scan(lib, S, 0, N, K, seen)
    assert torch.equal(i, ri)


def test_tc_sampled_fullsize(dev, lib):
    """4,096 users x 1,000,000 items x 768, tau in {0.25, 1, 4} mixed with plain rows, seen items, exclusions and allow-sets."""
    B, N, d, K = 4096, 1_000_000, 768, 20
    rng = np.random.default_rng(14)
    Ub, ldu, Eb, lde = _operands(lib, B, N, d, dev, seed=14)
    allow_bool = np.stack([rng.random(N) < 0.3, rng.random(N) < 0.01])
    aor_np = rng.integers(-1, 2, B).astype(np.int32)
    drop = [np.unique(np.concatenate([rng.integers(0, N, 200), rng.integers(0, N, 50)])).astype(np.int32) for _ in range(B)]
    inv = rng.choice([0.0, 0.25, 1.0, 4.0], B).astype(np.float32)
    sample = _sample_args(inv, rng.integers(0, 2 ** 62, B).astype(np.uint64), dev)
    v, i = _tc(lib, Ub, ldu, Eb, lde, B, 0, N, d, K, _csr(drop, dev), _pack(allow_bool, dev), torch.as_tensor(aor_np, device=dev),
               sample)
    sc = torch.empty(B, K, device=dev)
    rank = torch.empty(B, dtype=torch.int32, device=dev)
    lib.candidate_rank(Ub.data_ptr(), ldu, Eb.data_ptr(), lde, d, 1, i.data_ptr(), K, B, sc.data_ptr(), rank.data_ptr(), _st())
    inn = i.cpu().numpy()
    assert np.all(inn >= 0)
    il = i.long()
    ref = torch.einsum("bd,bkd->bk", Ub[:, :d].double(), Eb[il][:, :, :d].double())
    assert torch.allclose(sc.double(), ref, rtol=0, atol=1e-4)
    for b in range(B):
        ids = inn[b]
        assert len(np.unique(ids)) == K and not np.isin(ids, drop[b]).any()
        if aor_np[b] >= 0:
            assert allow_bool[aor_np[b], ids].all()


# -- evaluator and service -----------------------------------------------------------------------------------------------------
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
    ev.add_item_filter("a", np.random.default_rng(11).choice(n_items, 900, replace=False))
    return ev, data, i2it


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_evaluator_sampled(dev, precision):
    ev, data, _ = _world(dev, precision)
    users = np.arange(150)
    csr = data.scipy_csr()
    parts = [ev.topk_users(users[s:s + 64], 20) for s in range(0, 150, 64)]          # (the eager path the sampled call takes)
    plain_v, plain_i = torch.cat([x[0] for x in parts]), torch.cat([x[1] for x in parts])
    v, i = ev.topk_users(users, 20, temperature=[None if u % 5 == 0 else 0.5 for u in users], seed=users * 3 + 1)
    mixed = users % 5 == 0
    assert torch.equal(v[mixed], plain_v[mixed]) and torch.equal(i[mixed], plain_i[mixed])
    assert not torch.equal(i[~mixed], plain_i[~mixed])
    v2, i2 = ev.topk_users(users[::-1].copy(), 10, temperature=0.5, seed=(users * 3 + 1)[::-1].copy())   # other batches, K
    smp = torch.as_tensor(~mixed, device=dev)
    assert torch.equal(i2.flip(0)[smp], i[smp][:, :10])
    vn, inn = v.cpu().numpy(), i.cpu().numpy()
    for u in range(150):
        assert len(set(inn[u].tolist())) == 20 and not np.isin(inn[u], csr[u].indices).any()
        if precision == "fp32":                   # the scores are the model's scores of the drawn items
            np.testing.assert_allclose(vn[u], ev._get_user_scores(u)[inn[u]], rtol=0, atol=1e-5)
    # with an allow-set and exclusions: a 100-draw begins with the 60-draw, and differs from the plain top-100
    allowed = np.zeros(ev.n_items, dtype=bool)
    allowed[np.random.default_rng(11).choice(ev.n_items, 900, replace=False)] = True
    jf = ev.topk_users(users, 100, item_filter="a", exclude=[np.arange(5)] * 150, temperature=2.0, seed=5)[1]
    jf2 = ev.topk_users(users, 60, item_filter="a", exclude=[np.arange(5)] * 150, temperature=2.0, seed=5)[1]
    assert torch.equal(jf[:, :60], jf2)
    jd = ev.topk_users(users, 100, item_filter="a", exclude=[np.arange(5)] * 150)[1]
    assert not torch.equal(jf, jd)
    jfn = jf.cpu().numpy()
    assert allowed[jfn].all() and not np.isin(jfn, np.arange(5)).any()
    with pytest.raises(ValueError):
        ev.topk_users(users, 10, temperature=0.5)          # a temperature needs a seed
    with pytest.raises(ValueError):
        ev.topk_users(users, 10, temperature=1e-4, seed=1)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_service_fixed_seed_alone_and_batched(dev, precision):
    from hvae_b200.serve import MicroBatcher, RecommendService
    ev, _, i2it = _world(dev, precision)
    svc = RecommendService.from_evaluator(ev, i2it)
    svc.add_item_filter("a", [i2it[int(x)] for x in np.random.default_rng(11).choice(3000, 900, replace=False)])
    reqs = [dict(user_id="u1", top_k=10, temperature=0.7, seed=42), dict(user_id="u2", top_k=50, temperature=3.0, seed=2 ** 64 - 1),
            dict(user_id="u3", top_k=5, item_filter="a", exclude_items=["i1", "i2"], temperature=1.0, seed=7),
            dict(user_id="u4", top_k=20)]
    alone = [svc.recommend(**r) for r in reqs]
    with MicroBatcher(svc, max_batch=64, max_wait_ms=20) as mb:
        futs = [mb.submit(**r) for r in reqs] + [mb.submit(f"u{k}", 100, temperature=1.5, seed=k) for k in range(10, 40)]
        batched = [f.result() for f in futs]
    assert batched[:4] == alone
    assert alone[0]["seed"] == 42 and len(alone[1]["recommendations"]) == 50

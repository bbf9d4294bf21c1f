"""Kernel-by-kernel checks of the training step's noise, layer-1 weight gradient, LayerNorm block and optimiser at the
shapes the benchmarked step runs (B up to 9,000, hidden widths up to 2,048), through the C ABI with inputs built here.

Comparisons are bit for bit wherever the arithmetic is exact (Philox masks, dyadic gradient sums, split kernels that
promise the same bits as their fused form).  Everywhere else the tolerance is a first-order rounding-error bound
(u = 2^-24, the fp32 unit roundoff) worked out next to the comparison from the kernel's own operation order."""
import math

import numpy as np
import pytest
import torch

import philox_ref as ph

pytestmark = pytest.mark.gpu

U = 2.0 ** -24          # fp32 unit roundoff
SEED = 0x2545F4914F6CDD1D


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib(dev):
    from hvae_b200 import _cabi
    return _cabi.lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _r4(x):
    return (x + 3) // 4 * 4


def _state(dev):
    from hvae_b200._cabi import STATE_WORDS
    return torch.zeros(STATE_WORDS, dtype=torch.float32, device=dev)


def _set_u32(state, name, v):
    from hvae_b200._cabi import STATE_OFF
    v &= 0xFFFFFFFF
    state.view(torch.int32)[STATE_OFF[name]] = v - (1 << 32) if v >= 1 << 31 else v


def _set_f(state, name, v):
    from hvae_b200._cabi import STATE_OFF
    state[STATE_OFF[name]] = v


def _get(state, name, kind="f"):
    from hvae_b200._cabi import STATE_OFF
    if kind == "f":
        return float(state[STATE_OFF[name]].item())
    return int(state.view(torch.int32)[STATE_OFF[name]].item()) & 0xFFFFFFFF


def _bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# =====================================================================================================================
# 1. Philox noise
def _fill(lib, dev, n_mask, n_eps, keep, seed, offset, sid, state=None):
    mask = torch.full((n_mask + 5,), 7, dtype=torch.uint8, device=dev)
    eps = torch.full((n_eps + 5,), 1234.5, dtype=torch.float32, device=dev)
    lib.fill_noise(_p(mask) if n_mask else None, n_mask, keep, _p(eps) if n_eps else None, n_eps, seed, offset, sid, _p(state), _st())
    torch.cuda.synchronize()
    assert torch.all(mask[n_mask:] == 7) and torch.all(eps[n_eps:] == 1234.5), "wrote past the end"
    return mask[:n_mask].cpu().numpy(), eps[:n_eps].cpu().numpy()


def _eps_bound(ref, rad):
    # logf and sincospif are within 1 ulp (<= 2^-23 relative), sqrtf and the final product are correctly rounded (2^-24):
    # the radius sqrt(-2 logf(u1)) carries half of the log's error plus its own rounding, so |eps - ref| <= 2.5 * 2^-23 |ref|.
    # The float64 reference evaluates cos/sin(2 pi u2) with ~1e-15 absolute error, which matters only at exact zeros.
    return 2.5 * 2.0 ** -23 * np.abs(ref) + 1e-14 * rad


# counter bases within a few counters of 2^32 - 1, reached through `offset` or through the state's noise counter
_BASES = [dict(offset=(1 << 32) - 3, lo=None, hi=None), dict(offset=2, lo=0xFFFFFFFE, hi=0x11),
          dict(offset=(5 << 32) + 123, lo=0x10, hi=0)]


@pytest.mark.parametrize("keep", [0.5, 0.8, 1.0, 0.0])
@pytest.mark.parametrize("base", range(len(_BASES)))
def test_noise_mask_exact(lib, dev, keep, base):
    b = _BASES[base]
    state = None
    ctr = b["offset"]
    if b["lo"] is not None:
        state = _state(dev)
        _set_u32(state, "noise_lo", b["lo"])
        _set_u32(state, "noise_hi", b["hi"])
        ctr += (b["hi"] << 32) | b["lo"]
    for n, sid in ((4 * 1000 + 3, 1), (4 * 517 + 1, 200), (2, 5), (4096 * 600, 1)):
        got, _ = _fill(lib, dev, n, 0, keep, SEED, b["offset"], sid, state)
        want = ph.keep_mask(n, keep, SEED, ctr, sid)
        assert np.array_equal(got, want), (n, sid, int(np.sum(got != want)))


@pytest.mark.parametrize("base", range(len(_BASES)))
def test_noise_eps_box_muller(lib, dev, base):
    b = _BASES[base]
    state = None
    ctr = b["offset"]
    if b["lo"] is not None:
        state = _state(dev)
        _set_u32(state, "noise_lo", b["lo"])
        _set_u32(state, "noise_hi", b["hi"])
        ctr += (b["hi"] << 32) | b["lo"]
    worst = 0.0
    for n, sid in ((2 * 1000 + 1, 100), (4 * 333 + 2, 3), (1, 100), (4096 * 200, 100)):
        _, got = _fill(lib, dev, 0, n, 0.5, SEED, b["offset"], sid, state)
        ref, rad = ph.normals64(n, SEED, ctr, sid)
        err = np.abs(got.astype(np.float64) - ref)
        bound = _eps_bound(ref, rad)
        assert np.all(err <= bound), (n, sid, float(np.max(err / bound)))
        worst = max(worst, float(np.max(err / bound)))
    print(f"eps: largest error / bound = {worst:.3f}")


def test_noise_mask_and_eps_in_one_call(lib, dev):
    """One call with both outputs: the mask on stream id sid, eps on sid + 2^31, both from the same counters."""
    n = 4 * 2500 + 3
    m, e = _fill(lib, dev, n, n, 0.8, SEED, 77, 9)
    assert np.array_equal(m, ph.keep_mask(n, 0.8, SEED, 77, 9))
    ref, rad = ph.normals64(n, SEED, 77, 9)
    assert np.all(np.abs(e - ref) <= _eps_bound(ref, rad))


def test_noise_moments(lib, dev):
    """A large fixed-seed draw: keep fraction and eps mean / variance within 6 sigma of Bernoulli(keep) and N(0, 1)."""
    n, keep = 1 << 24, 0.8
    mask = torch.empty(n, dtype=torch.uint8, device=dev)
    eps = torch.empty(n, dtype=torch.float32, device=dev)
    lib.fill_noise(_p(mask), n, keep, _p(eps), n, 12345, 0, 42, None, _st())
    frac = mask.double().mean().item()
    p_keep = math.ceil(np.float32(keep) * 2 ** 24) / 2 ** 24        # P((r >> 8) * 2^-24 < keep) exactly
    assert abs(frac - p_keep) < 6 * math.sqrt(p_keep * (1 - p_keep) / n), frac
    e = eps.double()
    mean, var = e.mean().item(), e.var().item()
    assert abs(mean) < 6 / math.sqrt(n), mean
    assert abs(var - 1.0) < 6 * math.sqrt(2.0 / n), var
    assert torch.all(torch.isfinite(eps))


def test_step_begin_advances_noise_counter(lib, dev):
    state = _state(dev)

    def begin(advance, stride):
        lib.step_begin(_p(state), 1e-3, 0.9, 0.999, 0.0, 0.2, 0, 64, advance, stride, _st())
        torch.cuda.synchronize()
        return (_get(state, "noise_hi", "u") << 32) | _get(state, "noise_lo", "u")

    _set_u32(state, "noise_lo", 0xFFFFFFF0)
    _set_u32(state, "noise_hi", 5)
    c0 = (5 << 32) | 0xFFFFFFF0
    assert begin(0, 1000) == c0                            # evaluation step: the counter stays
    assert begin(1, 0x20) == c0 + 0x20                     # carry into noise_hi
    assert begin(1, 0xFFFFFFFF) == c0 + 0x20 + 0xFFFFFFFF
    assert begin(1, 7) == c0 + 0x20 + 0xFFFFFFFF + 7
    _set_u32(state, "noise_lo", 0xFFFFFFFF)
    _set_u32(state, "noise_hi", 0xFFFFFFFF)
    assert begin(1, 1) == 0                                # 64-bit wrap


def test_trainer_philox_noise_wiring(dev):
    """Two eager Philox steps of VAETrainer: every mask / eps buffer equals the generator at the trainer's stream ids and
    step counter, and the two steps' counter ranges do not overlap."""
    from hvae_b200.engine import Batch, DeviceCSR
    from hvae_b200.model import HybridVAE
    from hvae_b200.synth import make_interactions, make_item_embeddings
    from hvae_b200.train import VAETrainer
    N, d, L, hid, B = 700, 96, 24, [56, 37], 130
    data = make_interactions(B, N, 5)
    E = make_item_embeddings(N, d, 5)
    torch.manual_seed(0)
    m = HybridVAE(N, E, L, hid, 0.5, 0.2).to(dev)
    tr = VAETrainer(m, dev, use_cuda_graph=False)
    tr._noise_seed = SEED & 0x7FFFFFFFFFFFFFFF
    seed = tr._noise_seed
    eng = m.engine
    csr = DeviceCSR.from_arrays(data.indptr, data.indices, None, N, dev)
    rows = torch.arange(B, dtype=torch.int32, device=dev)
    stride = tr._noise_stride(B)
    draws = [(f"mask{i}", (B, h), 1 + i) for i, h in enumerate(hid)] + [("eps", (B, L), 100), ("pmask", (B, d), 200)]
    assert stride >= max((s[0] * s[1] + 3) // 4 for _, s, _ in draws)
    m.train()
    prev = None
    for step in range(2):
        tr.train_step(Batch(csr, rows, B, int(data.indptr[B])))
        torch.cuda.synchronize()
        ctr = (_get(eng.state, "noise_hi", "u") << 32) | _get(eng.state, "noise_lo", "u")
        assert ctr == (step + 1) * stride
        for name, shape, sid in draws:
            n = shape[0] * shape[1]
            if name == "eps":
                got = eng.ws.get(name, shape).reshape(-1).cpu().numpy()
                ref, rad = ph.normals64(n, seed, ctr, sid)
                assert np.all(np.abs(got - ref) <= _eps_bound(ref, rad)), name
            else:
                got = eng.ws.get(name, shape, torch.uint8).reshape(-1).cpu().numpy()
                assert np.array_equal(got, ph.keep_mask(n, 0.5, seed, ctr, sid)), name
        rng = (ctr, ctr + max((s[0] * s[1] + 3) // 4 for _, s, _ in draws))
        if prev is not None:
            assert rng[0] >= prev[1], (prev, rng)
        prev = rng


# =====================================================================================================================
# 2. Layer-1 weight gradient: batch transpose -> work plan -> w1_grad
def _csr(n_users, n_items, seed, hot=None, empty=(), int_values=True):
    """Zipf CSR (synth.make_interactions) with an optional hot item in every row and some rows emptied."""
    from hvae_b200.synth import make_interactions
    d = make_interactions(n_users, n_items, seed)
    users = np.repeat(np.arange(n_users, dtype=np.int64), np.diff(d.indptr))
    items = d.indices.astype(np.int64)
    if hot is not None:
        users = np.concatenate([users, np.arange(n_users)])
        items = np.concatenate([items, np.full(n_users, hot)])
    keep = ~np.isin(users, np.asarray(empty, dtype=np.int64))
    key = np.unique(users[keep] * n_items + items[keep])
    users, items = key // n_items, (key % n_items).astype(np.int32)
    indptr = np.zeros(n_users + 1, dtype=np.int64)
    np.cumsum(np.bincount(users, minlength=n_users), out=indptr[1:])
    rng = np.random.default_rng(seed + 11)
    vals = (rng.integers(1, 3, items.shape[0]) if int_values else rng.uniform(0.25, 2.0, items.shape[0])).astype(np.float32)
    return indptr, items, vals


def _entries(indptr, indices, values, rows):
    """The batch's entries in batch order (what expand_kernel writes): item, batch row, value."""
    rows = np.asarray(rows, dtype=np.int64)
    rc = np.maximum(rows, 0)
    lens = np.where(rows >= 0, indptr[rc + 1] - indptr[rc], 0)
    boff = np.zeros(rows.shape[0] + 1, dtype=np.int64)
    np.cumsum(lens, out=boff[1:])
    take = np.repeat(indptr[rc] - boff[:-1], lens) + np.arange(int(boff[-1]), dtype=np.int64)
    return indices[take].astype(np.int64), np.repeat(np.arange(rows.shape[0]), lens), values[take]


def _transpose(lib, dev, indptr, indices, values, rows, B, N, cap):
    i32 = torch.int32
    ip = torch.from_numpy(indptr).to(dev)
    ix = torch.from_numpy(indices).to(dev)
    vv = torch.from_numpy(values).to(dev)
    rd = None if rows is None else torch.from_numpy(np.asarray(rows, dtype=np.int32)).to(dev)
    t = {n: torch.full((cap,), -7, dtype=i32, device=dev)
         for n in ("keys", "keys_sorted", "eid", "eid_sorted", "head", "slot", "ent_user", "uniq_item")}
    t["ent_val"] = torch.full((cap,), float("nan"), device=dev)
    t["seg_start"] = torch.full((cap + 1,), -7, dtype=i32, device=dev)
    t["slot_of_item"] = torch.full((N,), -1, dtype=i32, device=dev)
    t["n_unique"] = torch.full((1,), -7, dtype=i32, device=dev)
    t["overflow"] = torch.zeros(1, dtype=i32, device=dev)
    boff = torch.empty(B + 1, dtype=i32, device=dev)
    tb = int(lib.batch_temp_bytes(cap, N))
    temp = torch.empty(tb, dtype=torch.uint8, device=dev)
    lib.batch_offsets(_p(ip), _p(rd), B, _p(boff), _st())
    lib.batch_transpose(_p(ip), _p(ix), _p(vv), _p(rd), B, N, cap, _p(boff), *[_p(t[n]) for n in (
        "keys", "keys_sorted", "eid", "eid_sorted", "head", "slot", "ent_user", "ent_val", "seg_start", "uniq_item",
        "slot_of_item", "n_unique", "overflow")], _p(temp), tb, _st())
    t["chunk_base"] = torch.full((cap + 1,), -7, dtype=i32, device=dev)
    t["part_base"] = torch.full((cap + 1,), -7, dtype=i32, device=dev)
    t["work_slot"] = torch.full((int(lib.w1_max_work(cap)),), -7, dtype=i32, device=dev)
    t["multi_slot"] = torch.full((int(lib.w1_max_partial_rows(cap)),), -7, dtype=i32, device=dev)
    t["n_work"] = torch.full((2,), -7, dtype=i32, device=dev)
    lib.w1_plan(_p(t["seg_start"]), _p(t["n_unique"]), cap, _p(t["chunk_base"]), _p(t["part_base"]), _p(t["work_slot"]),
                _p(t["multi_slot"]), _p(t["n_work"]), _st())
    t["cap"] = cap
    return t


def _transpose_ref(indptr, indices, values, rows, B, N, cap):
    items, users, vals = _entries(indptr, indices, values, np.arange(B) if rows is None else rows)
    nnz = items.shape[0]
    keys = np.full(cap, N, dtype=np.int64)
    keys[:nnz] = items
    order = np.argsort(keys, kind="stable")
    ks = keys[order]
    uniq, start = np.unique(ks[:nnz], return_index=True)
    seg = np.concatenate([start, [nnz]]).astype(np.int64)
    counts = np.diff(seg)
    ch = (counts + 63) // 64
    return dict(nnz=nnz, items=items, users=users, vals=vals, keys_sorted=ks, eid_sorted=order, uniq=uniq, seg=seg,
                counts=counts, chunks=ch, chunk_base=np.concatenate([[0], np.cumsum(ch)]),
                part_base=np.concatenate([[0], np.cumsum(np.where(ch > 1, ch, 0))]))


def _check_transpose(t, r, N):
    c = lambda x: x.cpu().numpy()
    nnz, nu = r["nnz"], r["uniq"].shape[0]
    assert int(t["overflow"].item()) == 0
    assert int(t["n_unique"].item()) == nu
    assert np.array_equal(c(t["keys_sorted"]), r["keys_sorted"])
    assert np.array_equal(c(t["eid_sorted"]), r["eid_sorted"])
    assert np.array_equal(c(t["seg_start"])[:nu + 1], r["seg"])
    assert np.array_equal(c(t["uniq_item"])[:nu], r["uniq"])
    soi = np.full(N, -1)
    soi[r["uniq"]] = np.arange(nu)
    assert np.array_equal(c(t["slot_of_item"]), soi)
    assert np.array_equal(c(t["ent_user"])[:nnz], r["users"])
    assert np.array_equal(c(t["ent_val"])[:nnz], r["vals"])
    assert np.array_equal(c(t["chunk_base"])[:nu + 1], r["chunk_base"])
    assert np.array_equal(c(t["part_base"])[:nu + 1], r["part_base"])
    n_work = c(t["n_work"])
    assert n_work[0] == r["chunks"].sum() and n_work[1] == int((r["chunks"] > 1).sum())
    assert np.array_equal(c(t["work_slot"])[:n_work[0]], np.repeat(np.arange(nu), r["chunks"]))
    assert sorted(c(t["multi_slot"])[:n_work[1]].tolist()) == np.flatnonzero(r["chunks"] > 1).tolist()


# (n_users, n_items, B, rows, cap - nnz, hot item, emptied users)
_TRANSPOSE_CASES = {
    "zipf_b512_hot": dict(U=700, N=5000, B=512, rows="perm", slack=100, hot=17, empty=()),
    "cap_equals_nnz_pow2_items": dict(U=400, N=1024, B=300, rows="perm", slack=0, hot=1023, empty=()),
    "padding_duplicates_empty_rows": dict(U=90, N=2048, B=80, rows="special", slack=17, hot=0, empty=(3, 4, 50)),
    "all_padding": dict(U=10, N=100, B=8, rows="pad", slack=5, hot=None, empty=()),
    "b4096_rows_null_hot": dict(U=4096, N=20000, B=4096, rows=None, slack=333, hot=4321, empty=(9,)),
}


def _rows(kind, U, B, seed):
    rng = np.random.default_rng(seed)
    if kind is None:
        return None
    if kind == "perm":
        return rng.permutation(U)[:B].astype(np.int32)
    if kind == "pad":
        return np.full(B, -1, dtype=np.int32)
    r = rng.permutation(U)[:B].astype(np.int32)
    r[[5, 6, 40, B - 1]] = -1                       # padding slots of a data-parallel global batch
    r[10] = r[11] = r[70] = 33                      # one user three times
    r[20], r[21] = 3, 50                            # users without interactions
    return r


@pytest.mark.parametrize("case", list(_TRANSPOSE_CASES))
def test_batch_transpose_and_plan(lib, dev, case):
    c = _TRANSPOSE_CASES[case]
    indptr, indices, vals = _csr(c["U"], c["N"], 3, hot=c["hot"], empty=c["empty"])
    rows = _rows(c["rows"], c["U"], c["B"], 4)
    nnz = _entries(indptr, indices, vals, np.arange(c["B"]) if rows is None else rows)[0].shape[0]
    cap = max(1, nnz + c["slack"])
    r = _transpose_ref(indptr, indices, vals, rows, c["B"], c["N"], cap)
    t = _transpose(lib, dev, indptr, indices, vals, rows, c["B"], c["N"], cap)
    torch.cuda.synchronize()
    _check_transpose(t, r, c["N"])
    if c["hot"] is not None and c["B"] > 64:
        assert r["chunks"].max() > 1                 # the hot item takes several chunks
    lib.batch_release(_p(t["uniq_item"]), _p(t["n_unique"]), cap, _p(t["slot_of_item"]), _p(t["overflow"]), None, None, _st())
    assert torch.all(t["slot_of_item"] == -1)


def _w1_run(lib, dev, t, dpre, ld, block_rows=0, block_stride=0):
    cap = t["cap"]
    gs = torch.full((cap, ld), float("nan"), device=dev)
    rn2 = torch.full((cap,), float("nan"), device=dev)
    part = torch.full((int(lib.w1_max_partial_rows(cap)), ld), float("nan"), device=dev)
    lib.w1_grad(_p(t["seg_start"]), _p(t["n_unique"]), _p(t["eid_sorted"]), _p(t["ent_user"]), _p(t["ent_val"]), cap,
                _p(t["chunk_base"]), _p(t["part_base"]), _p(t["work_slot"]), _p(t["multi_slot"]), _p(t["n_work"]), _p(dpre), ld,
                block_rows, block_stride, _p(gs), _p(part), _p(rn2), _st())
    nu = int(t["n_unique"].item())
    return gs[:nu], rn2[:nu]


def _blocked(dpre, B, ld):
    """dpre laid out as four blocks of B/4 rows, block_stride > block_rows * ld, NaN in every gap and after the last block."""
    br = B // 4
    bs = br * ld + 12
    buf = torch.full((4 * bs + 8,), float("nan"), device=dpre.device)
    for k in range(4):
        buf[k * bs:k * bs + br * ld] = dpre[k * br:(k + 1) * br].reshape(-1)
    return buf, br, bs


def _w1_ref(r, dpre, ld, dev):
    """float64 X^T dpre over the touched items (index_add_ on the GPU) and sum |x| |dpre| for the bounds."""
    slot = torch.from_numpy(np.searchsorted(r["uniq"], r["items"])).to(dev)
    user = torch.from_numpy(r["users"]).to(dev)
    v = torch.from_numpy(r["vals"].astype(np.float64)).to(dev)[:, None]
    g = dpre.double()[user]
    nu = r["uniq"].shape[0]
    ref = torch.zeros(nu, ld, dtype=torch.float64, device=dev).index_add_(0, slot, v * g)
    mag = torch.zeros(nu, ld, dtype=torch.float64, device=dev).index_add_(0, slot, (v * g).abs())
    return ref, mag


_W1_SHAPES = [(B, h) for B in (1, 512, 4096) for h in (24, 37, 600, 1000, 1500, 2048)] + \
             [(512, h) for h in (200, 300, 500, 700)]       # the remaining NCHUNK arms (2, 3, 4, 6)


def _w1_case(lib, dev, B, h, N, int_values, seed):
    ld = _r4(h)
    n_users = B + 37
    indptr, indices, vals = _csr(n_users, N, seed, hot=N // 3, int_values=int_values)
    rows = np.random.default_rng(seed + 1).permutation(n_users)[:B].astype(np.int32)
    cap = _entries(indptr, indices, vals, rows)[0].shape[0] + 64
    r = _transpose_ref(indptr, indices, vals, rows, B, N, cap)
    t = _transpose(lib, dev, indptr, indices, vals, rows, B, N, cap)
    g = torch.Generator(device=dev).manual_seed(seed)
    if int_values:
        dpre = torch.randint(-2, 3, (B, ld), generator=g, device=dev).float() * 2.0 ** -4
    else:
        dpre = torch.randn(B, ld, generator=g, device=dev)
    dpre[:, h:] = 0
    return t, r, dpre, ld


@pytest.mark.parametrize("B,h", _W1_SHAPES)
def test_w1_grad_exact_blocked_deterministic(lib, dev, B, h):
    """Dyadic data: values in {1, 2}, dpre in {-2..2} * 2^-4.  Every partial sum is a multiple of 2^-4 below 2^24 of
    those units, so fp32 sums it exactly in any order and gs must equal X^T dpre bit for bit."""
    t, r, dpre, ld = _w1_case(lib, dev, B, h, 20000, True, 7 + h)
    gs, rn2 = _w1_run(lib, dev, t, dpre, ld)
    ref, _ = _w1_ref(r, dpre, ld, dev)
    assert torch.equal(gs.double(), ref), float((gs.double() - ref).abs().max())
    # rownorm2 is exact where its own partial sums stay below 2^24 units of 2^-8 (the squares' granularity)
    n2 = (ref * ref).sum(1)
    ok = n2 * 2.0 ** 8 < 2.0 ** 24
    assert ok.any()
    assert torch.equal(rn2.double()[ok], n2[ok])
    assert torch.all((rn2.double()[~ok] - n2[~ok]).abs() <= (ld + 2) * U * n2[~ok])
    if B > 64:
        assert r["chunks"].max() == (B + 63) // 64       # the hot item sits in every row
    # same bits again (fixed summation order), and through the blocked (data-parallel) layout with NaN in the gaps
    gs2, rn22 = _w1_run(lib, dev, t, dpre, ld)
    assert _bits_equal(gs, gs2) and _bits_equal(rn2, rn22)
    if B >= 4:
        buf, br, bs = _blocked(dpre, B, ld)
        gs3, rn23 = _w1_run(lib, dev, t, buf, ld, br, bs)
        assert _bits_equal(gs, gs3) and _bits_equal(rn2, rn23)


def _w1_bound_check(t, r, gs, rn2, dpre, ld, dev):
    ref, mag = _w1_ref(r, dpre, ld, dev)
    n_ent = torch.from_numpy(r["counts"].astype(np.float64)).to(dev)[:, None]
    # a sum of n products, each fused into its running sum (fmaf) and partial rows added in a fixed order:
    # |gs - X^T dpre| <= (n + 2) u sum |x dpre| per element
    bound = (n_ent + 2) * U * mag
    err = (gs.double() - ref).abs()
    assert torch.all(err <= bound), float((err / bound.clamp_min(1e-300)).max())
    g64 = gs.double()
    s2 = (g64 * g64).sum(1)
    err2 = (rn2.double() - s2).abs()
    bound2 = (ld + 2) * U * s2                          # ld rounded squares summed in some order
    assert torch.all(err2 <= bound2)
    return float((err / bound.clamp_min(1e-300)).max()), float((err2 / bound2.clamp_min(1e-300)).max())


@pytest.mark.parametrize("B,h", [(1, 37), (512, 600), (512, 1000), (4096, 37), (4096, 1500), (4096, 2048)])
def test_w1_grad_random_within_bound(lib, dev, B, h):
    t, r, dpre, ld = _w1_case(lib, dev, B, h, 20000, False, 100 + h)
    gs, rn2 = _w1_run(lib, dev, t, dpre, ld)
    e1, e2 = _w1_bound_check(t, r, gs, rn2, dpre, ld, dev)
    print(f"w1_grad B={B} h={h}: gs err/bound {e1:.3g}, rownorm2 err/bound {e2:.3g}")


def test_w1_grad_c3_batch(lib, dev):
    """The benchmarked batch: B = 4,096 over 200,000 items at h = 600, exact (dyadic) and random data."""
    B, h, N = 4096, 600, 200_000
    t, r, dpre, ld = _w1_case(lib, dev, B, h, N, True, 3)
    gs, rn2 = _w1_run(lib, dev, t, dpre, ld)
    ref, _ = _w1_ref(r, dpre, ld, dev)
    assert torch.equal(gs.double(), ref)
    buf, br, bs = _blocked(dpre, B, ld)
    gs3, rn23 = _w1_run(lib, dev, t, buf, ld, br, bs)
    assert _bits_equal(gs, gs3) and _bits_equal(rn2, rn23)
    dr = torch.randn(B, ld, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    dr[:, h:] = 0
    gs, rn2 = _w1_run(lib, dev, t, dr, ld)
    e1, e2 = _w1_bound_check(t, r, gs, rn2, dr, ld, dev)
    print(f"w1_grad C3: gs err/bound {e1:.3g}, rownorm2 err/bound {e2:.3g}")


# =====================================================================================================================
# 3. LayerNorm + GELU + dropout, forward and backward
SQRT1_2 = 1.0 / math.sqrt(2.0)


def _pdf(y):
    return torch.exp(-0.5 * y * y) / math.sqrt(2.0 * math.pi)


def _cdf(y):
    return 0.5 * (1.0 + torch.erf(y * SQRT1_2))


def _ln_inputs(B, h, dev, seed):
    ld = _r4(h)
    g = torch.Generator(device=dev).manual_seed(seed)
    pre = torch.zeros(B, ld, device=dev)
    pre[:, :h] = torch.randn(B, h, generator=g, device=dev) * 1.5 + 0.3
    gamma = 1.0 + 0.3 * torch.randn(h, generator=g, device=dev)
    beta = 0.2 * torch.randn(h, generator=g, device=dev)
    mask = (torch.rand(B, h, generator=g, device=dev) < 0.5).to(torch.uint8)
    dact = torch.zeros(B, ld, device=dev)
    dact[:, :h] = torch.randn(B, h, generator=g, device=dev)
    return ld, pre, gamma, beta, mask, dact


def _ln_fwd_check(pre, gamma, beta, mask, keep_scale, mean, rstd, act, h):
    """mean, rstd and act of the kernel against float64 LayerNorm -> erf-GELU -> dropout of the same pre-activations."""
    p = pre[:, :h].double()
    mu_e = p.mean(1)
    var_e = ((p - mu_e[:, None]) ** 2).mean(1)
    rs_e = 1.0 / torch.sqrt(var_e + 1e-5)
    # mean: h additions -> h u mean|p|, / h -> u |mean|
    d_mu = h * U * p.abs().mean(1) + U * mu_e.abs()
    assert torch.all((mean.double() - mu_e).abs() <= d_mu)
    # var = sum (p - mean32)^2 / h = var_e + (mean32 - mu_e)^2; rounding of d, d^2, h additions, / h -> (h + 4) u var
    d_var = (h + 4) * U * var_e + d_mu ** 2
    # rstd = 1 / sqrtf(var + 1e-5f): half the relative error of var + eps, then add, sqrt and divide (3 u)
    rel_rs = 0.5 * (d_var + U * 1e-5) / (var_e + 1e-5) + 3 * U
    assert torch.all((rstd.double() - rs_e).abs() <= rel_rs * rs_e)
    xh = (p - mu_e[:, None]) * rs_e[:, None]
    gm, bt = gamma.double(), beta.double()
    y = xh * gm + bt
    gl = 0.5 * y * (1.0 + torch.erf(y * SQRT1_2))
    # y error: (p - mean) and * rstd roundings, the mean and rstd errors, the gamma/beta fma
    d_xh = (p - mu_e[:, None]).abs() * (rel_rs * rs_e)[:, None] + rs_e[:, None] * d_mu[:, None] + 2 * U * xh.abs()
    d_y = gm.abs() * d_xh + U * (xh * gm).abs() + U * y.abs()
    # gelu = 0.5 y (1 + erff(y * 0.70710678f)): |gelu'(y)| d_y; erff within 2 ulp (2^-22 |erf|); its argument rounded twice
    # (2 u |a|, times erf'(a) = 2 / sqrt(pi) e^-a^2, i.e. 2 u |y| 2 pdf(y)); the 1 + erf, y * (.) and 0.5 * (.) roundings
    gp = _cdf(y) + y * _pdf(y)
    d_g = gp.abs() * d_y + 0.5 * y.abs() * (2.0 ** -22 * torch.erf(y.abs() * SQRT1_2) + 2 * U * y.abs() * 2 * _pdf(y)
                                            + U * (1.0 + torch.erf(y * SQRT1_2))) + 2 * U * gl.abs()
    ref = gl
    if mask is not None:          # kept entries: * keep_scale (one more rounding); dropped ones are exactly zero
        ref = gl * mask.double() * keep_scale
        d_g = d_g * mask.double() * keep_scale + U * ref.abs()
    err = (act[:, :h].double() - ref).abs()
    assert torch.all(err <= d_g), float((err / d_g.clamp_min(1e-300)).max())
    assert torch.all(act[:, h:] == 0)
    return float((err / d_g.clamp_min(1e-300)).max())


def _ln_bwd_check(pre, mean, rstd, gamma, beta, mask, keep_scale, dact, dpre, dgamma, dbeta, h):
    """dpre, dgamma, dbeta of the kernel against float64 autograd of LayerNorm -> erf-GELU -> dropout; the bound adds up
    the rounding of every operation of ln_act_bwd_kernel and the deviation of the fp32 mean / rstd it was given."""
    B = pre.shape[0]
    p = pre[:, :h].double().requires_grad_(True)
    gm = gamma.double().requires_grad_(True)
    bt = beta.double().requires_grad_(True)
    y_e = torch.nn.functional.layer_norm(p, (h,), gm, bt, eps=1e-5)
    out = torch.nn.functional.gelu(y_e)
    if mask is not None:
        out = out * mask.double() * keep_scale
    da = dact[:, :h].double()
    out.backward(da)
    with torch.no_grad():
        mu_e = p.mean(1, keepdim=True)
        rs_e = 1.0 / torch.sqrt(((p - mu_e) ** 2).mean(1, keepdim=True) + 1e-5)
        mu, rs = mean.double()[:, None], rstd.double()[:, None]
        xh = (p - mu_e) * rs_e
        y = xh * gm + bt
        # xhat = (p - mean) * rstd with fp32 mean / rstd: their deviation from the exact values, plus two roundings
        d_xh = (p - mu_e).abs() * (rs - rs_e).abs() + rs * (mu - mu_e).abs() + 2 * U * xh.abs()
        d_y = gm.abs() * d_xh + U * y.abs()
        # gelu_grad = cdf + y pdf: erff (2 ulp) and 1 + erf; __expf within 2 + 1.173 |x| ulp of exp(x), x = -y^2/2 (itself
        # rounded: relative u y^2/2); the constant and y * pdf roundings; and the curvature |gelu''| = pdf |2 - y^2| times d_y
        pdf, cdf = _pdf(y), _cdf(y)
        gg = cdf + y * pdf
        d_pdf = pdf * (2.0 ** -23 * (2 + 1.173 * 0.5 * y * y) + U * 0.5 * y * y + 3 * U)
        d_gg = 2.0 ** -23 + 2 * U * y.abs() * pdf + 2 * U * cdf + y.abs() * d_pdf + U * (y * pdf).abs() + U * gg.abs() + pdf * (2 - y * y).abs() * d_y
        dg = da * (mask.double() * keep_scale if mask is not None else 1.0)
        dln = dg * gg
        d_dln = dg.abs() * d_gg + 2 * U * dln.abs()
        dx = dln * gm
        d_dx = gm.abs() * d_dln + U * dx.abs()
        # m1 = sum(dx) / h, m2 = sum(dx xhat) / h over h terms (lane sums then the shuffle tree)
        m1 = dx.mean(1, keepdim=True)
        m2 = (dx * xh).mean(1, keepdim=True)
        d_m1 = d_dx.mean(1, keepdim=True) + (h + 1) * U * dx.abs().mean(1, keepdim=True)
        d_m2 = (d_dx * xh.abs() + dx.abs() * d_xh).mean(1, keepdim=True) + (h + 2) * U * (dx * xh).abs().mean(1, keepdim=True)
        inner = dx - m1 - xh * m2
        d_inner = d_dx + d_m1 + m2.abs() * d_xh + xh.abs() * d_m2 + 3 * U * (dx.abs() + m1.abs() + (xh * m2).abs())
        d_dpre = rs * d_inner + inner.abs() * (rs - rs_e).abs() + U * (rs * inner).abs()
        err = (dpre[:, :h].double() - p.grad).abs()
        r1 = float((err / d_dpre.clamp_min(1e-300)).max())
        assert torch.all(err <= d_dpre), r1
        assert torch.all(dpre[:, h:] == 0)
        # d(gamma) = sum_rows dln xhat, d(beta) = sum_rows dln: the per-row errors plus (B + 2) u sum |term| for the
        # fixed-order sums (rows per warp, warps per block, blocks, stages)
        t_g = dln * xh
        d_dg = (d_dln * xh.abs() + dln.abs() * d_xh + U * t_g.abs()).sum(0) + (B + 2) * U * t_g.abs().sum(0)
        d_db = d_dln.sum(0) + (B + 2) * U * dln.abs().sum(0)
        eg, eb = (dgamma.double() - gm.grad).abs(), (dbeta.double() - bt.grad).abs()
        assert torch.all(eg <= d_dg) and torch.all(eb <= d_db), (float((eg / d_dg).max()), float((eb / d_db).max()))
        return r1, float((eg / d_dg.clamp_min(1e-300)).max()), float((eb / d_db.clamp_min(1e-300)).max())


_LN_SHAPES = [(B, h) for B in (8, 592, 593, 4096, 9000) for h in (37, 600, 768, 1000, 2048)]


@pytest.mark.parametrize("B,h", _LN_SHAPES)
def test_ln_act_fwd_bwd(lib, dev, B, h):
    ld, pre, gamma, beta, mask, dact = _ln_inputs(B, h, dev, B * 7 + h)
    keep_scale = 2.0
    worst = {}
    for use_mask in (False, True):
        mk = mask if use_mask else None
        mean = torch.full((B,), float("nan"), device=dev)
        rstd = torch.full((B,), float("nan"), device=dev)
        act = torch.full((B, ld), float("nan"), device=dev)
        lib.ln_act_fwd(_p(pre), B, h, ld, _p(gamma), _p(beta), _p(mk), keep_scale, _p(mean), _p(rstd), _p(act), _st())
        worst[f"fwd mask={use_mask}"] = _ln_fwd_check(pre, gamma, beta, mk, keep_scale, mean, rstd, act, h)
        ws = torch.full((int(lib.ln_bwd_workspace_floats(B, ld)),), float("nan"), device=dev)
        results = []
        for adjacent in (True, False):
            dpre = torch.full((B, ld), float("nan"), device=dev)
            if adjacent:         # d(gamma), d(beta) as adjacent slots of one buffer: one launch over both
                arena = torch.full((2 * ld + 4,), float("nan"), device=dev)
                dgamma, dbeta = arena[:ld], arena[ld:2 * ld]
            else:
                dgamma = torch.full((h,), float("nan"), device=dev)
                dbeta = torch.full((h,), float("nan"), device=dev)
            lib.ln_act_bwd(_p(dact), _p(pre), _p(mean), _p(rstd), _p(gamma), _p(beta), _p(mk), keep_scale, B, h, ld, _p(dpre),
                           _p(dgamma), _p(dbeta), _p(ws), _st())
            if adjacent:
                assert torch.all(dgamma[h:] == 0) and torch.all(dbeta[h:] == 0) and torch.isnan(arena[2 * ld:]).all()
            worst[f"bwd mask={use_mask} adjacent={adjacent}"] = _ln_bwd_check(
                pre, mean, rstd, gamma, beta, mk, keep_scale, dact, dpre, dgamma[:h], dbeta[:h], h)
            results.append((dpre, dgamma[:h].clone(), dbeta[:h].clone()))
        # both reduction tails sum the same partial rows in the same order
        assert all(_bits_equal(a, b) for a, b in zip(results[0], results[1]))
        # dact may alias dpre (what the engine does)
        inplace = dact.clone()
        dg2, db2 = torch.empty(h, device=dev), torch.empty(h, device=dev)
        lib.ln_act_bwd(_p(inplace), _p(pre), _p(mean), _p(rstd), _p(gamma), _p(beta), _p(mk), keep_scale, B, h, ld, _p(inplace),
                       _p(dg2), _p(db2), _p(ws), _st())
        assert _bits_equal(inplace, results[0][0]) and _bits_equal(dg2, results[0][1]) and _bits_equal(db2, results[0][2])
    print(f"ln B={B} h={h}: largest error / bound {worst}")


@pytest.mark.parametrize("B,h", [(8, 37), (593, 600), (593, 2048), (4096, 1000)])
def test_gather_ln_fwd_block_and_warp(lib, dev, monkeypatch, B, h):
    """gather-sum + bias + LN-GELU-dropout: pre against float64 X W1 + b, the LN block against float64 of the kernel's
    own pre; the warp-per-user variant (HVAE_GATHER_WARP) gives the same bits as the CTA-per-user one."""
    ld = _r4(h)
    N = 5000
    indptr, indices, vals = _csr(B + 11, N, 21, hot=7, int_values=False)
    rows = np.random.default_rng(2).permutation(B + 11)[:B].astype(np.int32)
    g = torch.Generator(device=dev).manual_seed(h)
    W1T = torch.zeros(N, ld, device=dev)
    W1T[:, :h] = torch.randn(N, h, generator=g, device=dev) * 0.1
    bias = 0.1 * torch.randn(h, generator=g, device=dev)
    gamma = 1.0 + 0.3 * torch.randn(h, generator=g, device=dev)
    beta = 0.2 * torch.randn(h, generator=g, device=dev)
    mask = (torch.rand(B, h, generator=g, device=dev) < 0.5).to(torch.uint8)
    ip, ix, vv = (torch.from_numpy(a).to(dev) for a in (indptr, indices, vals))
    rd = torch.from_numpy(rows).to(dev)
    outs = {}
    for warp in (False, True):
        if warp:
            monkeypatch.setenv("HVAE_GATHER_WARP", "1")
        else:
            monkeypatch.delenv("HVAE_GATHER_WARP", raising=False)
        o = {k: torch.full(s, float("nan"), device=dev) for k, s in (("pre", (B, ld)), ("mean", (B,)), ("rstd", (B,)), ("act", (B, ld)))}
        lib.gather_ln_fwd(_p(ip), _p(ix), _p(vv), _p(rd), B, _p(W1T), ld, h, _p(bias), _p(gamma), _p(beta), _p(mask), 2.0,
                          _p(o["pre"]), _p(o["mean"]), _p(o["rstd"]), _p(o["act"]), _st())
        outs[warp] = o
    monkeypatch.delenv("HVAE_GATHER_WARP", raising=False)
    for k in ("pre", "mean", "rstd", "act"):
        assert _bits_equal(outs[False][k], outs[True][k]), k
    o = outs[False]
    items, users, v = _entries(indptr, indices, vals, rows)
    ut = torch.from_numpy(users).to(dev)
    terms = torch.from_numpy(v.astype(np.float64)).to(dev)[:, None] * W1T.double()[torch.from_numpy(items).to(dev)]
    ref = torch.zeros(B, ld, dtype=torch.float64, device=dev).index_add_(0, ut, terms)
    mag = torch.zeros(B, ld, dtype=torch.float64, device=dev).index_add_(0, ut, terms.abs())
    n = torch.from_numpy(np.bincount(users, minlength=B).astype(np.float64)).to(dev)[:, None]
    ref[:, :h] += bias.double()
    mag[:, :h] += bias.double().abs()
    err = (o["pre"].double() - ref).abs()
    assert torch.all(err <= (n + 2) * U * mag)        # n fmaf in CSR order, then + bias
    _ln_fwd_check(o["pre"], gamma, beta, mask, 2.0, o["mean"], o["rstd"], o["act"], h)


# =====================================================================================================================
# 4. Optimiser
B1, B2, EPS, LR = np.float32(0.9), np.float32(0.999), np.float32(1e-8), 1e-3


def _adam_setup(dev, seed, n_items=3000, ld1=600, n_dense=100_004, max_rows=700):
    g = torch.Generator(device=dev).manual_seed(seed)
    n_w1 = n_items * ld1
    n = n_w1 + n_dense
    p = torch.randn(n, generator=g, device=dev)
    m = 0.01 * torch.randn(n, generator=g, device=dev)
    v = 1e-4 * (0.5 + torch.rand(n, generator=g, device=dev))
    rng = np.random.default_rng(seed)
    touched = np.sort(rng.choice(n_items, int(0.15 * n_items), replace=False))      # ~15% rows, n_unique < max_rows
    assert touched.shape[0] < max_rows
    uniq = torch.full((max_rows,), -5, dtype=torch.int32, device=dev)
    uniq[:touched.shape[0]] = torch.from_numpy(rng.permutation(touched).astype(np.int32)).to(dev)
    soi = torch.full((n_items,), -1, dtype=torch.int32, device=dev)
    soi[uniq[:touched.shape[0]].long()] = torch.arange(touched.shape[0], dtype=torch.int32, device=dev)
    n_unique = torch.tensor([touched.shape[0]], dtype=torch.int32, device=dev)
    gs = 0.05 * torch.randn(max_rows, ld1, generator=g, device=dev)
    gd = 0.05 * torch.randn(n_dense, generator=g, device=dev)
    return dict(p=p, m=m, v=v, uniq=uniq, soi=soi, n_unique=n_unique, gs=gs, gd=gd, n_w1=n_w1, n=n, ld1=ld1,
                max_rows=max_rows, n_items=n_items)


@pytest.mark.parametrize("wd", [0.0, 1e-2])
@pytest.mark.parametrize("step", [1, 7])
def test_adam_split_equals_fused_and_float64(lib, dev, wd, step):
    a = _adam_setup(dev, 11 + step)
    state = _state(dev)
    for _ in range(step):
        lib.step_begin(_p(state), LR, float(B1), float(B2), 0.0, 0.2, 0, 64, 1, 0, _st())
    _set_f(state, "clip_coef", 0.625)
    wd32 = float(np.float32(wd))
    fused = [a[k].clone() for k in "pmv"]
    lib.adam_step(*[_p(t) for t in fused], a["n"], a["n_w1"], a["ld1"], _p(a["soi"]), _p(a["gs"]), _p(a["gd"]), _p(state),
                  wd32, float(B1), float(B2), float(EPS), _st())
    split = [a[k].clone() for k in "pmv"]
    lib.adam_step_untouched(*[_p(t) for t in split], a["n_w1"], a["ld1"], _p(a["soi"]), _p(state), wd32, float(B1), float(B2),
                            float(EPS), _st())
    lib.adam_step_touched(*[_p(t) for t in split], a["n"], a["n_w1"], a["ld1"], _p(a["uniq"]), _p(a["n_unique"]), a["max_rows"],
                          _p(a["gs"]), _p(a["gd"]), _p(state), wd32, float(B1), float(B2), float(EPS), _st())
    for x, y in zip(fused, split):
        assert _bits_equal(x, y)
    # float64 restatement of torch.optim.Adam (L2 weight decay) after clipping: gradient of W1^T row i is gs[slot[i]] or 0
    gfull = torch.zeros(a["n_items"], a["ld1"], dtype=torch.float64, device=dev)
    nu = int(a["n_unique"].item())
    gfull[a["uniq"][:nu].long()] = a["gs"][:nu].double()
    g = torch.cat([gfull.reshape(-1), a["gd"].double()]) * 0.625
    p0, m0, v0 = (a[k].double() for k in "pmv")
    b1, b2, eps = float(B1), float(B2), float(EPS)
    g = g + wd32 * p0
    m1 = b1 * m0 + (1 - b1) * g
    v1 = b2 * v0 + (1 - b2) * g * g
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    denom = torch.sqrt(v1) / math.sqrt(bc2) + eps
    p1 = p0 - (LR / bc1) * m1 / denom
    # Bounds, with G = |g clip| + wd |p0| >= |g'| (so they hold through cancellation in g' = g clip + wd p0):
    # g': two roundings -> 2 u G.  m = m0 + (1 - b1)(g' - m0): g' - m0, * and + roundings -> <= 5 u (|m0| + (1 - b1) G).
    # v = v0 b2 + ((1 - b2) g') g': g'^2 within 6 u G^2, v0 b2 and the add -> <= 8 u (b2 v0 + (1 - b2) G^2).
    # denom = sqrtf(v) / bc2_sqrt + eps: half of v's relative error, plus sqrt, the fp32 bc2_sqrt, divide, add (4 u).
    # p = p + (-step_size)(m / denom): the fp32 step size, the divide and the product (3 u more), then p's own rounding.
    G = (g - wd32 * p0).abs() + wd32 * p0.abs()
    bnd_m = 5 * U * (m0.abs() + (1 - b1) * G)
    bnd_v = 8 * U * (b2 * v0 + (1 - b2) * G * G)
    rel_den = 0.5 * bnd_v / v1 + 4 * U
    bnd_step = (LR / bc1) * (bnd_m + m1.abs() * (rel_den + 3 * U)) / denom
    bnd_p = (1 + U) * bnd_step + U * p1.abs()             # rounding of p0 - step, |p0 - step| <= |p1| + bnd_step
    worst = []
    for got, ref, bnd in ((fused[1], m1, bnd_m), (fused[2], v1, bnd_v), (fused[0], p1, bnd_p)):
        err = (got.double() - ref).abs()
        assert torch.all(err <= bnd), float((err / bnd).max())
        worst.append(float((err / bnd).max()))
    print(f"adam step={step} wd={wd}: m, v, p err/bound {worst}")


@pytest.mark.parametrize("scale,with_rows", [(1e-4, True), (0.05, True), (0.05, False)])
def test_grad_norm_split_equals_fused_and_float64(lib, dev, scale, with_rows):
    n_dense = 148 * 256 * 3 + 1001                      # > 148 * 256: the grid-stride loop wraps
    g = torch.Generator(device=dev).manual_seed(17)
    gd = scale * torch.randn(n_dense, generator=g, device=dev)
    rn2 = scale * scale * 600 * torch.rand(900, generator=g, device=dev)
    n_unique = torch.tensor([900 if with_rows else 0], dtype=torch.int32, device=dev)
    max_norm = 5.0
    s1, s2 = _state(dev), _state(dev)
    ws1 = torch.full((160,), float("nan"), device=dev)
    ws2 = torch.full((160,), float("nan"), device=dev)
    lib.grad_norm_clip(_p(gd), n_dense, _p(rn2), _p(n_unique), max_norm, _p(s1), _p(ws1), _st())
    lib.grad_sumsq_dense(_p(gd), n_dense, _p(ws2), _st())
    lib.grad_norm_finish(n_dense, _p(rn2), _p(n_unique), max_norm, _p(s2), _p(ws2), _st())
    torch.cuda.synchronize()
    for k in ("norm2", "grad_norm", "clip_coef"):
        assert _get(s1, k) == _get(s2, k), k
    rows = rn2.double().sum().item() if with_rows else 0.0
    ref2 = (gd.double() ** 2).sum().item() + rows
    # each of the 148 * 256 threads sums <= ceil(n / (148 * 256)) squares by fmaf, then 5 shuffle levels, 8 warps, the
    # float64 finish and the final rounding to fp32
    k = -(-n_dense // (148 * 256))
    bound2 = (k + 5 + 8 + 2) * U * (gd.double() ** 2).sum().item() + U * ref2
    assert abs(_get(s1, "norm2") - ref2) <= bound2
    norm = math.sqrt(ref2)
    assert abs(_get(s1, "grad_norm") - norm) <= (0.5 * bound2 / ref2 + U) * norm
    clip = min(1.0, max_norm / (norm + 1e-6))
    if clip == 1.0:
        assert _get(s1, "clip_coef") == 1.0
    else:
        assert abs(_get(s1, "clip_coef") - clip) <= (0.5 * bound2 / ref2 + 4 * U) * clip
    assert (clip < 1.0) == (scale == 0.05)

"""bf16 tensor-core mode of the scoring stage: sequencing of the tcgen05 kernels of csrc/score_tc.cu.

The user vectors u = projection(z) are rounded to bf16, E is held as a bf16 copy; products accumulate in fp32 in
TMEM.  The [B, N] score matrix is never written: the forward kernel's epilogue folds it into per-user
log-sum-exp, the backward kernel recomputes it tile by tile and feeds softmax(S) straight into the second GEMM
(src/ml/model.py:198,281 and their autograd), the evaluation kernel folds it into a per-user top-K
(src/ml/evaluate.py:125-147).
"""
from __future__ import annotations

import torch

from ._cabi import p
from .engine import r4, r8

MAX_K_TC = 128       # K <= 32: register-resident lists in the epilogue; K <= 128: shared-memory lists
MAX_K_REG = 32


def user_vectors_bf16(eng, u, B):
    d = eng.lay.d
    ub = eng.ws.get("u_bf16", (B, r8(d)), torch.bfloat16)
    if getattr(eng, "ub_fresh", None) == (u.data_ptr(), B):       # written by the epilogue of the GEMM that produced u
        eng.ub_fresh = None
        return ub
    eng.lib.cast_bf16(p(u), B, d, r4(d), p(ub), r8(d), eng.stream)
    return ub


def score_loss_bf16(eng, batch, u, want_grad):
    """-> (lse [B], dot [B], xsum [B], O partial sums [splits, B, ld] or None, per-row scale(s) of O).

    Training (want_grad) runs the one-pass kernel: forward and backward through the scores in a single sweep over the
    items (softmax numerators against a score-independent shift, hvae_tc_score_onepass); O is then unnormalised and its
    scale is (xsum, w_part).  HVAE_TWO_PASS=1 selects the forward-LSE + backward pair of launches instead."""
    lay, ws, lib, st = eng.lay, eng.ws, eng.lib, eng.stream
    B, N, d = batch.B, lay.N, lay.d
    ldd, ld8 = r4(d), r8(d)
    csr = batch.csr
    Eb = eng.E_bf16
    onepass = want_grad and not eng.two_pass
    ub = user_vectors_bf16(eng, u, B)
    lse, dot, xsum = ws.get("lse", (B,)), ws.get("dot", (B,)), ws.get("xsum", (B,))
    with eng.side(1):                # independent of the score GEMMs
        lib.sparse_dot_xsum(p(csr.indptr), p(csr.indices), p(csr.values), p(batch.rows), B, p(ub), ld8, p(Eb), ld8, d, 1,
                            p(dot), p(xsum), eng.stream)
    ns = int(lib.tc_n_splits(B, N))
    wsl = ws.get("tc_lse_ws", (2 * B * ns,))
    O = None
    if onepass:
        gs = int(lib.tc_grad_splits(B, N, d))
        O = ws.get("tc_O", (gs, B, ldd))
        n_sub = int(lib.tc_onepass_subparts(d))
        c_part, l_part, w_part = ws.get("tc_c_part", (gs, B)), ws.get("tc_l_part", (gs, n_sub, B)), ws.get("tc_w_part", (gs, B))
        with eng.span("score_onepass"):
            lib.tc_score_onepass(p(ub), ld8, B, p(Eb), ld8, N, d, p(c_part), p(l_part), p(O), ldd, st)
            if not eng.fuse & 32:
                lib.tc_onepass_combine(p(c_part), p(l_part), gs, n_sub, B, p(lse), p(w_part), st)
        if eng.fuse & 32:        # the combination of the splits (-> lse, weights of the O partials) happens inside du_finalize_onepass
            return lse, dot, xsum, O, (xsum, (c_part, l_part, n_sub), lse)
        return lse, dot, xsum, O, (xsum, w_part)
    if want_grad and eng.prof is None:        # two launches: the backward kernel merges the forward partials itself
        gs = int(lib.tc_grad_splits(B, N, d))
        O = ws.get("tc_O", (gs, B, ldd))
        lib.tc_score_lse_grad(p(ub), ld8, B, p(Eb), ld8, N, d, p(lse), p(wsl), p(O), ldd, st)
        return lse, dot, xsum, O, xsum
    with eng.span("score_fwd"):
        lib.tc_score_lse(p(ub), ld8, B, p(Eb), ld8, N, d, p(lse), p(wsl), st)
    if want_grad:
        gs = int(lib.tc_grad_splits(B, N, d))
        O = ws.get("tc_O", (gs, B, ldd))
        with eng.span("score_bwd"):
            lib.tc_score_grad(p(ub), ld8, B, p(Eb), ld8, N, d, p(lse), p(O), ldd, st)
    return lse, dot, xsum, O, xsum


def topk_bf16(eng, batch, u, K, exclude_seen, item_lo, item_hi, out_val, out_idx, mask=None, allow=None) -> bool:
    """Fused score + seen-mask + top-K over items [item_lo, item_hi).  False if K is beyond the fused kernel."""
    if K > MAX_K_TC:
        return False
    return topk_bf16_from_ub(eng, batch, user_vectors_bf16(eng, u, batch.B), K, exclude_seen, item_lo, item_hi, out_val, out_idx,
                             mask, allow)


def topk_bf16_from_ub(eng, batch, ub, K, exclude_seen, item_lo, item_hi, out_val, out_idx, mask=None, allow=None) -> bool:
    """The same with the bf16 user vectors [B, r8(d)] already at hand (item-sharded evaluation all-gathers them).

    mask = (indptr int64 [B+1], indices int32): items to leave out, one sorted row per BATCH row; it replaces the batch's
    seen rows (exclude_seen is then not looked at).  allow = (bitmaps int32 [F, words], allow_of_row int32 [B]): row b only
    returns items whose bit is set in bitmaps[allow_of_row[b]] (-1: unrestricted); slots it cannot fill hold (-inf, -1)."""
    if K > MAX_K_TC:
        return False
    lay, ws, lib, st = eng.lay, eng.ws, eng.lib, eng.stream
    B, d = batch.B, lay.d
    ld8 = r8(d)
    n_it = item_hi - item_lo
    Eb = eng.E_bf16
    ns = int(lib.tc_topk_splits(B, n_it))
    cv = ws.get("tc_cand_v", (B, ns * K))
    ci = ws.get("tc_cand_i", (B, ns * K), torch.int32)
    csr = batch.csr
    with eng.span("score_topk"):
        if mask is None and allow is None:
            lib.tc_score_topk(p(ub), ld8, B, Eb.data_ptr() + 2 * item_lo * ld8, ld8, n_it, d, item_lo,
                              p(csr.indptr) if exclude_seen else None, p(csr.indices), p(batch.rows), K, p(cv), p(ci), st)
        else:
            if mask is not None:
                indptr, indices, rows = mask[0], mask[1], None
            else:
                indptr, indices, rows = (csr.indptr if exclude_seen else None), csr.indices, batch.rows
            bm, aor = allow if allow is not None else (None, None)
            lib.tc_score_topk_filtered(p(ub), ld8, B, Eb.data_ptr() + 2 * item_lo * ld8, ld8, n_it, d, item_lo, p(indptr), p(indices),
                                       p(rows), p(bm), 0 if bm is None else bm.stride(0), p(aor), K, p(cv), p(ci), st)
    lib.topk_merge(p(cv), p(ci), B, ns * K, K, p(out_val), p(out_idx), st)
    return True

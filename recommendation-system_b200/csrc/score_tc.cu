// Tensor-core scoring (bf16 mode): S = U E^T on tcgen05 with TMA-fed shared memory and TMEM accumulators; the
// [B, N] score matrix never leaves the SM.  Replaces decode() + log_softmax of the reference
// (src/ml/model.py:198,281) and the score -> mask -> argsort loop of the evaluator (src/ml/evaluate.py:125-147).
//
//   hvae_tc_score_lse  : per-user log-sum-exp over all items (validation loss / forward of the NLL)
//   hvae_tc_score_topk : per-user top-K over all (or a shard of the) items with seen-item masking
//
// Kernel shape (one CTA = 128 users x a contiguous range of 256-item tiles, 192 threads):
//   warp 0      TMA producer : U k-block [128 x 64] + E k-block [256 x 64] (bf16, 128B swizzle) per pipeline stage
//   warp 1      MMA issuer   : tcgen05.mma 128x256x16, fp32 accumulators in TMEM, two accumulator buffers
//   warps 2..5  epilogue     : tcgen05.ld -> registers; thread <-> user row, so every reduction is thread-local
// Roofline: tensor pipe (2*128*256*d flop per tile); HBM traffic is E once (L2 serves the re-reads across user tiles).
#include <cfloat>
#include <cstdlib>

#include "common.cuh"
#include "hvae_b200.h"
#include "tc_common.cuh"

namespace hvae {
namespace tc {

constexpr int BM = 128, BN = 256, BK = 64, STAGES = 4;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int MAXK_REG = 32;   // top-K list per row in REGISTERS (sorted 64-bit keys): K <= 32
constexpr int MAXK_TC = 128;   // larger K (the API's top_k <= 100): list per row in shared memory, 2-stage operand ring
constexpr int STAGES_SMEM_LIST = 2;
constexpr float kLog2e = 1.4426950408889634f;

enum Mode { MODE_LSE = 0, MODE_TOPK = 1 };

struct StatsParams {
    int B, N, d;          // users in this launch, items in this launch (shard), embedding dim
    int tiles_per_split;  // 256-item tiles per CTA along the item axis
    int n_splits;
    int item_offset;      // global id of item 0 of E (item-sharded evaluation)
    // MODE_LSE
    float* part_m;        // [B, n_splits]
    float* part_l;
    // MODE_TOPK
    int K;
    float* cand_val;      // [B, n_splits * K]
    int32_t* cand_idx;
    const int64_t* indptr;   // seen items (CSR over users), may be null
    const int32_t* indices;
    const int32_t* rows;     // user ids of the batch rows (null = identity)
    // TOPK with FILTER: item allow-sets, bit i of a bitmap row = global item i may be returned
    const uint32_t* allow;        // [F, allow_stride] words
    int64_t allow_stride;
    const int32_t* allow_of_row;  // [B] bitmap row of each batch row, -1 = unrestricted
    // TOPK with SAMPLE: Gumbel-top-K keys s / tau + g (common.cuh: gumbel_of) of rows with row_inv_tau != 0
    const float* row_inv_tau;     // [B] 1 / tau, 0 = the row's plain scores
    const uint64_t* row_seed;     // [B]
};

// One-pass mode (hvae_tc_score_onepass): softmax numerators are taken against a per-row shift c_b that does not depend on the
// scores (0 to begin with) instead of the row's log-sum-exp, so no forward pass has to come first.  fp32 and bf16 share the
// exponent range: as long as the row's numerators sum to something inside [kOnepassUnder, kOnepassOver] neither the largest
// one overflowed nor any relevant one (>= 2^-24 of the largest, N <= 2^26) was flushed, and sum_i exp(S_bi - c_b) /
// sum_i exp(S_bi - c_b) E_i lose nothing.  Otherwise (|scores| beyond ~70: a degenerate model, but it must stay exact) the CTA
// repeats its sweep with c_b -+ kOnepassRetry for the rows concerned; the windows of consecutive shifts overlap widely.
constexpr float kOnepassRetry = 60.0f, kOnepassOver = 1.2676506e30f /* 2^100 */, kOnepassUnder = 8.8817842e-16f /* 2^-50 */;
constexpr int kOnepassMaxSweeps = 64;

struct __align__(8) PipeBarriers {
    uint64_t full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2];
    uint32_t tmem_base;
};

// (score, item id) as ONE 64-bit key whose unsigned order is the evaluator's total order (score desc, index desc):
// the score's bits made monotonic in the high word, the id in the low word; 0 = empty slot (below every real key).
__device__ __forceinline__ uint64_t topk_key(float v, int idx) {
    uint32_t u = __float_as_uint(v + 0.0f);                     // -0.0 -> +0.0: equal scores must tie
    u ^= (u >> 31) ? 0xFFFFFFFFu : 0x80000000u;
    return (uint64_t(u) << 32) | uint32_t(idx);
}
__device__ __forceinline__ float topk_key_value(uint64_t k) {
    uint32_t u = uint32_t(k >> 32);
    u ^= (u >> 31) ? 0x80000000u : 0xFFFFFFFFu;
    return __uint_as_float(u);
}

__device__ __forceinline__ bool better(float v, int i, float tv, int ti) { return v > tv || (v == tv && i > ti); }

// The allow bits of the 256 items g0.. of one tile as eight words (bit j of aw[c] = item g0 + 32c + j), from the row's bitmap
// (null = everything allowed).  g0 need not be a multiple of 32: each word is funnel-shifted out of two neighbours.  Words past
// the one holding item g_end - 1 are not read (the epilogue drops those columns anyway).
__device__ __forceinline__ void tile_allow_words(const uint32_t* arow, int g0, int g_end, uint32_t (&aw)[8]) {
    if (!arow) {
#pragma unroll
        for (int e = 0; e < 8; ++e) aw[e] = 0xFFFFFFFFu;
        return;
    }
    const int w0 = g0 >> 5, sh = g0 & 31, wlast = (g_end - 1) >> 5;
    uint32_t raw[9];
#pragma unroll
    for (int e = 0; e < 8; ++e) raw[e] = w0 + e <= wlast ? __ldg(arow + w0 + e) : 0u;
    raw[8] = sh && w0 + 8 <= wlast ? __ldg(arow + w0 + 8) : 0u;
#pragma unroll
    for (int e = 0; e < 8; ++e) aw[e] = __funnelshift_r(raw[e], raw[e + 1], sh);
}

// STG = operand ring depth; KREG > 0: top-K list of KREG >= K sorted keys per row in registers, KREG == 0: list in shared memory.
// FILTER (TOPK only): a column is a candidate only if the row's allow bitmap has its bit; the words are ANDed into the
// compare mask of each 32-column chunk, so a rejected column never reaches the insertion loop.
// SAMPLE (TOPK, with FILTER; P.allow may then be null): a row with row_inv_tau != 0 ranks the keys fmaf(s, inv_tau, g), g the
// Gumbel noise of (row_seed, global item id).  The compare mask tests the bound fmaf(s, inv_tau, kGumbelMax) instead of s, so
// Philox and the logarithms run only for the columns that pass it, once per group of 4 consecutive items.  The lists and the
// written values hold keys.  A row with row_inv_tau == 0 runs the FILTER kernel's arithmetic on s itself.
template <int MODE, int STG, int KREG, bool FILTER = false, bool SAMPLE = false>
__global__ void __launch_bounds__(192, 1) score_stats_kernel(const __grid_constant__ CUtensorMap tmU,
                                                             const __grid_constant__ CUtensorMap tmE, StatsParams P) {
    constexpr int STAGES = STG;      // (shadows the file-level default)
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    PipeBarriers* bars = reinterpret_cast<PipeBarriers*>(smem + STAGES * STAGE_BYTES);
    float* list_v = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + 256);           // [128][K]   (TOPK, shared-memory list)
    int* list_i = reinterpret_cast<int*>(list_v + BM * (MAXK_TC + 1));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x, split = blockIdx.y;
    const int n_tiles_total = (P.N + BN - 1) / BN;
    const int t0 = split * P.tiles_per_split, t1 = min(n_tiles_total, t0 + P.tiles_per_split);
    const int KB = (P.d + BK - 1) / BK;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmU);
        tma_prefetch_desc(&tmE);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&bars->tmem_full[a], 1); mbar_init(&bars->tmem_empty[a], 4); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<512>(&bars->tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    // "dependents may launch" only now that this CTA holds its TMEM columns: a dependent tensor-core kernel that landed on this
    // SM earlier could take the columns and then park in griddepcontrol.wait on us while we block in tcgen05.alloc
    pdl_launch_dependents();
    pdl_wait();      // everything above (barrier init, TMEM allocation, descriptor prefetch) overlapped the previous kernel

    if (warp == 0) {
        if (lane == 0) {
            int it = 0;
            for (int t = t0; t < t1; ++t)
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&bars->empty[s], ((it / STAGES) & 1) ^ 1);
                    mbar_expect_tx(&bars->full[s], STAGE_BYTES);
                    tma_load_2d(smem + s * STAGE_BYTES, &tmU, kb * BK, m_tile * BM, &bars->full[s]);
                    tma_load_2d(smem + s * STAGE_BYTES + A_BYTES, &tmE, kb * BK, t * BN, &bars->full[s]);
                }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(BM, BN, 0, 0);
            int it = 0;
            for (int t = t0, ti = 0; t < t1; ++t, ++ti) {
                const int acc = ti & 1;
                mbar_wait(&bars->tmem_empty[acc], ((ti >> 1) & 1) ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&bars->full[s], (it / STAGES) & 1);
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(smem + s * STAGE_BYTES), b0 = a0 + A_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        umma_ss(tmem_base + acc * BN, make_desc(a0 + k * 32, 16, 1024), make_desc(b0 + k * 32, 16, 1024), idesc,
                                (kb | k) != 0);
                    }
                    umma_commit(&bars->empty[s]);
                }
                umma_commit(&bars->tmem_full[acc]);
            }
        }
    } else {
        // ---- epilogue: thread <-> user row ------------------------------------------------------------------
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int r_local = q * 32 + lane;
        const int row = m_tile * BM + r_local;
        const bool row_ok = row < P.B;
        float m_run = -INFINITY, l_run = 0.f;
        // top-K state
        float thr_v = -INFINITY;
        int thr_i = -1, thr_pos = 0, cnt = 0;
        float* lv = list_v + r_local * (MAXK_TC + 1);
        int* li = list_i + r_local * (MAXK_TC + 1);
        int64_t seen_p = 0, seen_e = 0;
        int next_seen = INT_MAX;
        // register list (KREG > 0): the best KREG >= K keys seen so far, sorted descending; key[KREG-1] is the admission threshold
        constexpr int KR = KREG > 0 ? KREG : 1;
        uint64_t key[KR];
#pragma unroll
        for (int e = 0; e < KR; ++e) key[e] = 0;
        if (MODE == MODE_TOPK) {
            if (KREG == 0)
                for (int e = 0; e < P.K; ++e) { lv[e] = -INFINITY; li[e] = -1; }
            if (row_ok && P.indptr) {
                const int u = P.rows ? P.rows[row] : row;
                seen_p = P.indptr[u];
                seen_e = P.indptr[u + 1];
                // first seen item at or after this CTA's first item
                const int first = P.item_offset + t0 * BN;
                int64_t lo = seen_p, hi = seen_e;
                while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (P.indices[mid] < first) lo = mid + 1; else hi = mid; }
                seen_p = lo;
                next_seen = seen_p < seen_e ? P.indices[seen_p] : INT_MAX;
            }
        }
        const uint32_t* arow = nullptr;
        if constexpr (FILTER) {
            const int f = row_ok && (!SAMPLE || P.allow) ? P.allow_of_row[row] : -1;
            if (f >= 0) arow = P.allow + (size_t)f * P.allow_stride;
        }
        // SAMPLE: candidate bound fmaf(v, s_a, s_b) (v itself for a deterministic row); the Philox words of item group nz_ctr
        float s_a = 1.f, s_b = 0.f;
        uint64_t seed = 0;
        uint32_t nz[4] = {0u, 0u, 0u, 0u}, nz_ctr = 0xFFFFFFFFu;      // (gi >> 2 < 2^29: never a real group)
        if constexpr (SAMPLE) {
            if (row_ok && P.row_inv_tau[row] != 0.f) { s_a = P.row_inv_tau[row]; s_b = kGumbelMax; seed = P.row_seed[row]; }
        }
        for (int t = t0, ti = 0; t < t1; ++t, ++ti) {
            const int acc = ti & 1;
            uint32_t aw[8];
            if constexpr (FILTER) tile_allow_words(arow, P.item_offset + t * BN, P.item_offset + P.N, aw);   // in flight during the MMA
            mbar_wait(&bars->tmem_full[acc], (ti >> 1) & 1);
            tc_fence_after();
            const int col0 = t * BN;
            const int n_valid = min(BN, P.N - col0);
            // seen items of this row inside the tile (TOPK): local columns, at most 16 tracked exactly
            int mcol[16];
            int nmask = 0;
            if (MODE == MODE_TOPK) {
                const int tile_end = P.item_offset + col0 + BN;
                while (next_seen < tile_end) {
                    if (nmask < 16) mcol[nmask] = next_seen - P.item_offset - col0;
                    ++nmask;
                    ++seen_p;
                    next_seen = seen_p < seen_e ? P.indices[seen_p] : INT_MAX;
                }
            }
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                float v[32];
                tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + acc * BN + c * 32, v);
                tmem_ld_wait();
                if (c * 32 >= n_valid) continue;
                if (MODE == MODE_LSE) {
                    if (c * 32 + 32 > n_valid) {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (c * 32 + j >= n_valid) v[j] = -INFINITY;
                    }
                    float cm = v[0];
#pragma unroll
                    for (int j = 1; j < 32; ++j) cm = fmaxf(cm, v[j]);
                    const float m_new = fmaxf(m_run, cm);
                    const float ms = m_new * kLog2e;
                    float s = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) s += exp2f(fmaf(v[j], kLog2e, -ms));
                    l_run = l_run * exp2f((m_run - m_new) * kLog2e) + s;
                    m_run = m_new;
                } else {
                    // candidate bits first (32 compares), then a compact loop over the few set bits: the insertion
                    // code exists once, not 32 times (instruction-cache footprint), and v[j] is fetched by selects
                    unsigned mbits = 0;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        if constexpr (SAMPLE) mbits |= (fmaf(v[j], s_a, s_b) >= thr_v) ? (1u << j) : 0u;
                        else mbits |= (v[j] >= thr_v) ? (1u << j) : 0u;
                    }
                    const int left = n_valid - c * 32;
                    if (left < 32) mbits &= (1u << left) - 1u;
                    if constexpr (FILTER) {
                        uint32_t a = aw[0];
#pragma unroll
                        for (int e = 1; e < 8; ++e) a = (e == c) ? aw[e] : a;
                        mbits &= a;
                    }
                    if (!row_ok) mbits = 0;
                    while (mbits) {
                        const int j = __ffs(mbits) - 1;
                        mbits &= mbits - 1;
                        float x = v[0];
#pragma unroll
                        for (int t = 1; t < 32; ++t) x = (t == j) ? v[t] : x;
                        const int lc = c * 32 + j, gi = P.item_offset + col0 + lc;
                        if constexpr (SAMPLE) {
                            if (s_b != 0.f) {
                                const uint32_t ctr = (uint32_t)gi >> 2;
                                if (ctr != nz_ctr) { philox(seed, ctr, kSampleStream, nz); nz_ctr = ctr; }
                                x = fmaf(x, s_a, gumbel_of(pick4(nz, gi & 3)));
                            }
                        }
                        uint64_t xk = 0;
                        if (KREG > 0) {
                            xk = topk_key(x, gi);
                            if (xk <= key[KR - 1]) continue;
                        } else if (cnt == P.K && !better(x, gi, thr_v, thr_i)) continue;
                        if (nmask) {
                            bool seen = false;
                            if (nmask <= 16) {
                                for (int e = 0; e < nmask; ++e) seen |= (mcol[e] == lc);
                            } else {  // rare: many seen items in one tile -> exact binary search in the row's CSR slice
                                const int u = P.rows ? P.rows[row] : row;
                                int64_t lo = P.indptr[u], hi = P.indptr[u + 1];
                                while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (P.indices[mid] < gi) lo = mid + 1; else hi = mid; }
                                seen = lo < P.indptr[u + 1] && P.indices[lo] == gi;
                            }
                            if (seen) continue;
                        }
                        if (KREG > 0) {
                            // sorted insertion without memory traffic or dependent loads: entry e takes its upper neighbour if the
                            // new key ranks above that neighbour, the new key if it ranks above entry e only
                            bool above[KR];
#pragma unroll
                            for (int e = 0; e < KR; ++e) above[e] = xk > key[e];
#pragma unroll
                            for (int e = KR - 1; e >= 1; --e) key[e] = above[e - 1] ? key[e - 1] : (above[e] ? xk : key[e]);
                            key[0] = above[0] ? xk : key[0];
                            thr_v = key[KR - 1] ? topk_key_value(key[KR - 1]) : -INFINITY;
                        } else {
                            int pos = thr_pos;
                            if (cnt < P.K) pos = cnt++;
                            lv[pos] = x;
                            li[pos] = gi;
                            if (cnt == P.K) {  // recompute the list's worst element (= threshold)
                                float wv = lv[0]; int wi = li[0], wp = 0;
                                for (int e = 1; e < P.K; ++e) {
                                    const float ev = lv[e]; const int ei = li[e];
                                    if (better(wv, wi, ev, ei)) { wv = ev; wi = ei; wp = e; }
                                }
                                thr_v = wv; thr_i = wi; thr_pos = wp;
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->tmem_empty[acc]);
        }
        if (row_ok) {
            if (MODE == MODE_LSE) {
                P.part_m[(size_t)row * P.n_splits + split] = m_run;
                P.part_l[(size_t)row * P.n_splits + split] = l_run;
            } else {
                float* ov = P.cand_val + ((size_t)row * P.n_splits + split) * P.K;
                int32_t* oi = P.cand_idx + ((size_t)row * P.n_splits + split) * P.K;
                if (KREG > 0) {
#pragma unroll
                    for (int e = 0; e < KR; ++e)
                        if (e < P.K) { ov[e] = key[e] ? topk_key_value(key[e]) : -INFINITY; oi[e] = key[e] ? (int32_t)(uint32_t)key[e] : -1; }
                } else {
                    for (int e = 0; e < P.K; ++e) { ov[e] = lv[e]; oi[e] = li[e]; }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

// lse[b] = log sum_s l_s * exp(m_s - M) + M over the item splits
__global__ void lse_merge_kernel(const float* __restrict__ part_m, const float* __restrict__ part_l, int B, int n_splits,
                                 float* __restrict__ lse) {
    pdl_prologue();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float M = -INFINITY;
    for (int s = 0; s < n_splits; ++s) M = fmaxf(M, part_m[(size_t)b * n_splits + s]);
    float l = 0.f;
    for (int s = 0; s < n_splits; ++s) l += part_l[(size_t)b * n_splits + s] * expf(part_m[(size_t)b * n_splits + s] - M);
    lse[b] = M + logf(l);
}

// fp32 [rows, cols] (leading dim ld_src) -> bf16 [rows, ld_dst] with zero padding of columns cols..ld_dst
__global__ void cast_bf16_kernel(const float* __restrict__ src, int rows, int cols, int ld_src, __nv_bfloat16* __restrict__ dst,
                                 int ld_dst) {
    pdl_prologue();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)rows * ld_dst) return;
    const int r = (int)(i / ld_dst), c = (int)(i - (int64_t)r * ld_dst);
    dst[i] = __float2bfloat16(c < cols ? src[(size_t)r * ld_src + c] : 0.f);
}

// Combination of the one-pass kernel's per-split results of one row (shift c_p, numerator sums l_part[p][sub]), one warp per
// row, lanes over the splits:  M = max_p c_p (all c_p are equal unless a split had to repeat its sweep),
// D = sum_p e^{c_p - M} sum_sub l_part,  lse_b = M + log D,  w_part[p][b] = e^{c_p - M} / D  -- hvae_du_finalize then forms
// O_b = sum_p w_part[p][b] Opart[p][b].
__global__ void __launch_bounds__(256) onepass_combine_kernel(const float* __restrict__ c_part, const float* __restrict__ l_part,
                                                              int n_parts, int n_sub, int B, float* __restrict__ lse,
                                                              float* __restrict__ w_part) {
    pdl_prologue();
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (b >= B) return;
    float M = -INFINITY;
    for (int pp = lane; pp < n_parts; pp += 32) M = fmaxf(M, c_part[(size_t)pp * B + b]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o));
    float D = 0.f;
    for (int pp = lane; pp < n_parts; pp += 32) {
        float l = 0.f;
        for (int sb = 0; sb < n_sub; ++sb) l += l_part[((size_t)pp * n_sub + sb) * B + b];
        D = fmaf(expf(c_part[(size_t)pp * B + b] - M), l, D);
    }
    // fixed-order reduction (xor tree): the same bits on every run
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) D += __shfl_xor_sync(0xffffffffu, D, o);
    const float inv = 1.0f / D;
    for (int pp = lane; pp < n_parts; pp += 32) w_part[(size_t)pp * B + b] = expf(c_part[(size_t)pp * B + b] - M) * inv;
    if (lane == 0) lse[b] = M + logf(D);
}


// ----------------------------------------------------------------------------------------------------------------
// Backward of the multinomial NLL through the scores: O[b,:] = sum_i softmax(S_b)_i * E_i, with S recomputed tile by
// tile (never stored) and the softmax taken against the exact lse of the forward kernel.  Two chained GEMMs per
// 128-item tile:  G1: S = U E_t^T (K = d, accumulators in TMEM)  ->  registers: P = exp(S - lse_b) -> bf16 -> smem
// (128B-swizzled, K-major)  ->  G2: O += P E_t (K = 128 items; B operand = the same E rows read MN-major).
// One CTA = (128 users, <=384 columns of O, a range of item tiles).  No gradient for E (frozen buffer).
// One-pass mode (P.c_part != null): the same sweep also IS the forward pass -- numerators against the fixed shift, their row
// sums to l_part, O left unnormalised; a row outside the safe range makes its CTA (pair) repeat the sweep with another shift.
constexpr int G_BN = 128;                     // items per tile
constexpr int G_STAGES = 4, G_SLOT = 32768;   // ring slot: U [128x64] + E [128x64] for G1, or E [64 x <=256] for G2
constexpr int G_DCHUNK = 384;                 // O columns per CTA (TMEM: 384 O + 128 S = 512)
constexpr int G_PBYTES = 32768;               // P tile [128 users x 128 items] bf16 = two [128x64] swizzle atoms columns

struct GradParams {
    int B, N, d;
    int tiles_per_split, n_splits;
    const float* lse;     // [B], or null: merge the forward kernel's partials below (and publish lse_out)
    const float* part_m;  // [B, lse_splits] per-split running max / sum-exp of score_stats_kernel<LSE>
    const float* part_l;
    int lse_splits;
    float* lse_out;       // [B]
    float* Opart;         // [n_splits][B][ldo]
    int ldo;
    // one-pass mode (c_part != null)
    float* c_part;        // [n_splits][B]  shift the split ended up with
    float* l_part;        // [n_splits][n_sub][B]  row sums of the numerators (n_sub = 2 for the pair kernel: one per CTA)
    int box3d;            // cta_group::2 kernel: the tensor maps are the 3-D (64 columns, rows, 64-column blocks) views
};

// Softmax numerators of one [128 users x 128 items] score tile, thread <-> user row: p = exp2(v * log2e - shift2), packed to
// bf16 and handed to store(item, w0..w3) in 16-byte groups of 8 items.  Returns the row's sum of the (unrounded) numerators
// over the tile's first n_valid items (MASK: the catalogue ends inside this tile; TMA zero-fills the rows beyond it).
template <bool MASK, class Store>
__device__ __forceinline__ float softmax_tile(const float (&v)[4][32], float shift2, int n_valid, Store&& store) {
    float lsum = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8) {         // 8 items -> one 16-byte chunk
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int idx = c * 32 + j8 * 8 + 2 * e;
                float p0 = exp2f(fmaf(v[c][j8 * 8 + 2 * e], kLog2e, -shift2));
                float p1 = exp2f(fmaf(v[c][j8 * 8 + 2 * e + 1], kLog2e, -shift2));
                if (MASK) {
                    if (idx >= n_valid) p0 = 0.f;
                    if (idx + 1 >= n_valid) p1 = 0.f;
                }
                lsum += p0 + p1;
                __nv_bfloat162 h = __floats2bfloat162_rn(p0, p1);
                w[e] = *reinterpret_cast<uint32_t*>(&h);
            }
            store(c * 32 + j8 * 8, w[0], w[1], w[2], w[3]);
        }
    }
    return lsum;
}

struct __align__(8) GradBarriers {
    uint64_t full[G_STAGES], empty[G_STAGES], s_full, s_free, p_full[2], p_free[2], o_full;
    uint32_t tmem_base;
    float rsum[2][BM];        // pair kernel: the row sums of both CTAs' sweeps (each CTA holds both arrays)
};

// Row r of the merged forward partials (two-pass mode without a ready lse).
__device__ __forceinline__ float merged_lse(const float* part_m, const float* part_l, int lse_splits, int row) {
    const float* pm = part_m + (size_t)row * lse_splits;
    const float* pl = part_l + (size_t)row * lse_splits;
    float M = -INFINITY;
    for (int sp = 0; sp < lse_splits; ++sp) M = fmaxf(M, pm[sp]);
    float l = 0.f;
    for (int sp = 0; sp < lse_splits; ++sp) l += pl[sp] * expf(pm[sp] - M);
    return M + logf(l);
}

__global__ void __launch_bounds__(192, 1) score_grad_kernel(const __grid_constant__ CUtensorMap tmU,
                                                            const __grid_constant__ CUtensorMap tmE, GradParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* pbuf = smem + G_STAGES * G_SLOT;                         // 2 x 32 KB
    GradBarriers* bars = reinterpret_cast<GradBarriers*>(pbuf + 2 * G_PBYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x, chunk = blockIdx.y, split = blockIdx.z;
    const int n_tiles_total = (P.N + G_BN - 1) / G_BN;
    const int t0 = split * P.tiles_per_split, t1 = min(n_tiles_total, t0 + P.tiles_per_split);
    const int T = t1 - t0;
    const int KB = (P.d + BK - 1) / BK;
    const int dpad = KB * BK;
    const int dc0 = chunk * G_DCHUNK;                  // first O column of this CTA
    const int DC = min(G_DCHUNK, dpad - dc0);          // multiple of 64
    const int NG = (DC + 255) / 256;                   // column groups of <= 256 per G2 MMA

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmU);
        tma_prefetch_desc(&tmE);
        for (int s = 0; s < G_STAGES; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        mbar_init(&bars->s_full, 1); mbar_init(&bars->s_free, 4); mbar_init(&bars->o_full, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(&bars->p_full[a], 4); mbar_init(&bars->p_free[a], 1); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<512>(&bars->tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    // "dependents may launch" only now that this CTA holds its TMEM columns: a dependent tensor-core kernel that landed on this
    // SM earlier could take the columns and then park in griddepcontrol.wait on us while we block in tcgen05.alloc
    pdl_launch_dependents();
    pdl_wait();      // everything above (barrier init, TMEM allocation, descriptor prefetch) overlapped the previous kernel
    const uint32_t tmem_O = tmem_base, tmem_S = tmem_base + G_DCHUNK;
    const bool onepass = P.c_part != nullptr;

    // epilogue state (warps 2..5): thread <-> user row
    const int q = warp & 3;
    const int r_local = q * 32 + lane;
    const int row = m_tile * BM + r_local;
    const bool row_ok = warp >= 2 && row < P.B;
    const uint32_t lane_base = uint32_t(q * 32) << 16;
    float lse_row = 0.f;      // two-pass: the row's log-sum-exp; one-pass: the shift
    if (row_ok && !onepass) {
        if (P.lse) lse_row = P.lse[row];
        else {                 // merge the forward partials here instead of in a separate launch
            lse_row = merged_lse(P.part_m, P.part_l, P.lse_splits, row);
            if (chunk == 0 && split == 0) P.lse_out[row] = lse_row;
        }
    }
    float lsum = 0.f;
    int it = 0;               // ring position of the producer / the MMA issuer; runs on across sweeps
    // A sweep = all tiles of this CTA.  Barrier phases are derived from g = sweep * T + tile, so that a repeated sweep
    // (one-pass mode, after an overflow) simply continues the sequences.
    for (int sweep = 0;; ++sweep) {
        if (warp == 0) {
            if (lane == 0) {
                auto acquire = [&](uint32_t bytes) {
                    const int s = it % G_STAGES;
                    mbar_wait(&bars->empty[s], ((it / G_STAGES) & 1) ^ 1);
                    mbar_expect_tx(&bars->full[s], bytes);
                    ++it;
                    return s;
                };
                for (int ti = 0; ti <= T; ++ti) {
                    if (ti < T) {          // G1 operands of tile ti
                        const int item0 = (t0 + ti) * G_BN;
                        for (int kb = 0; kb < KB; ++kb) {
                            const int s = acquire(G_SLOT);
                            uint8_t* slot = smem + s * G_SLOT;
                            tma_load_2d(slot, &tmU, kb * BK, m_tile * BM, &bars->full[s]);
                            tma_load_2d(slot + 16384, &tmE, kb * BK, item0, &bars->full[s]);
                            tma_load_2d(slot + 16384 + 8192, &tmE, kb * BK, item0 + 64, &bars->full[s]);
                        }
                    }
                    if (ti >= 1) {         // G2 operands of tile ti-1: E rows as [64 items x (<=256 columns)] blocks
                        const int item0 = (t0 + ti - 1) * G_BN;
                        for (int ih = 0; ih < 2; ++ih)
                            for (int g = 0; g < NG; ++g) {
                                const int nb = min(4, (DC - g * 256) / 64);
                                const int s = acquire(nb * 8192);
                                uint8_t* slot = smem + s * G_SLOT;
                                for (int j = 0; j < nb; ++j)
                                    tma_load_2d(slot + j * 8192, &tmE, dc0 + g * 256 + j * 64, item0 + ih * 64, &bars->full[s]);
                            }
                    }
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {
                constexpr uint32_t idesc1 = make_idesc(BM, G_BN, 0, 0);
                for (int ti = 0; ti <= T; ++ti) {
                    if (ti < T) {          // G1(ti): S = U E_t^T
                        const int g = sweep * T + ti;
                        mbar_wait(&bars->s_free, (g & 1) ^ 1);
                        tc_fence_after();
                        for (int kb = 0; kb < KB; ++kb, ++it) {
                            const int s = it % G_STAGES;
                            mbar_wait(&bars->full[s], (it / G_STAGES) & 1);
                            tc_fence_after();
                            const uint32_t a0 = smem_u32(smem + s * G_SLOT), b0 = a0 + 16384;
#pragma unroll
                            for (int k = 0; k < BK / 16; ++k)
                                umma_ss(tmem_S, make_desc(a0 + k * 32, 16, 1024), make_desc(b0 + k * 32, 16, 1024), idesc1, (kb | k) != 0);
                            umma_commit(&bars->empty[s]);
                        }
                        umma_commit(&bars->s_full);
                    }
                    if (ti >= 1) {         // G2(ti-1): O += P E_t
                        const int tj = ti - 1, g = sweep * T + tj, pb = g & 1;
                        mbar_wait(&bars->p_full[pb], (g >> 1) & 1);
                        tc_fence_after();
                        const uint32_t p0 = smem_u32(pbuf + pb * G_PBYTES);
                        for (int ih = 0; ih < 2; ++ih)
                            for (int gq = 0; gq < NG; ++gq, ++it) {
                                const int ncols = min(256, DC - gq * 256);
                                const uint32_t idesc2 = make_idesc(BM, ncols, 0, 1);
                                const int s = it % G_STAGES;
                                mbar_wait(&bars->full[s], (it / G_STAGES) & 1);
                                tc_fence_after();
                                const uint32_t b0 = smem_u32(smem + s * G_SLOT);
#pragma unroll
                                for (int kk = 0; kk < 4; ++kk)      // K = 16 items per MMA
                                    umma_ss(tmem_O + gq * 256, make_desc(p0 + ih * 16384 + kk * 32, 16, 1024),
                                            make_desc(b0 + kk * 2048, 8192, 1024), idesc2, (tj | ih | kk) != 0);
                                umma_commit(&bars->empty[s]);
                            }
                        umma_commit(&bars->p_free[pb]);
                    }
                }
                umma_commit(&bars->o_full);
            }
        } else {
            const float lse2 = lse_row * kLog2e;
            lsum = 0.f;
            for (int ti = 0; ti < T; ++ti) {
                const int g = sweep * T + ti, pb = g & 1;
                mbar_wait(&bars->s_full, g & 1);
                tc_fence_after();
                float v[4][32];
#pragma unroll
                for (int c = 0; c < 4; ++c) tmem_ld32(tmem_S + lane_base + c * 32, v[c]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->s_free);
                mbar_wait(&bars->p_free[pb], ((g >> 1) & 1) ^ 1);
                uint8_t* prow = pbuf + pb * G_PBYTES + r_local * 128;
                auto store = [&](int item, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {   // item: local index 0..127
                    const int atom = item >> 6, chunk16 = (item & 63) >> 3;
                    uint8_t* dst = prow + atom * 16384 + ((chunk16 ^ (r_local & 7)) << 4);
                    *reinterpret_cast<uint4*>(dst) = make_uint4(w0, w1, w2, w3);
                };
                const int n_valid = P.N - (t0 + ti) * G_BN;
                if (n_valid >= G_BN) lsum += softmax_tile<false>(v, lse2, G_BN, store);
                else lsum += softmax_tile<true>(v, lse2, n_valid, store);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->p_full[pb]);
            }
            mbar_wait(&bars->o_full, sweep & 1);      // every MMA of the sweep has completed
            tc_fence_after();
        }
        __syncwarp();
        if (!onepass) break;
        const bool over = warp >= 2 && lsum > kOnepassOver;          // inf included; NaN is not (it propagates, as in the reference)
        const bool under = warp >= 2 && lsum < kOnepassUnder;
        if (!__syncthreads_or(over || under) || sweep + 1 >= kOnepassMaxSweeps) break;
        lse_row += over ? kOnepassRetry : under ? -kOnepassRetry : 0.f;
    }
    if (warp >= 2) {
        // ---- O (TMEM) -> global partial ---------------------------------------------------------------------
        if (onepass && row_ok && chunk == 0) {
            P.c_part[(size_t)split * P.B + row] = lse_row;
            P.l_part[(size_t)split * P.B + row] = lsum;
        }
        float* orow = P.Opart + ((size_t)split * P.B + row) * P.ldo + dc0;
        for (int c = 0; c < DC / 32; ++c) {
            float v[32];
            tmem_ld32(tmem_O + lane_base + c * 32, v);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (dc0 + c * 32 + j < P.ldo)
                        *reinterpret_cast<float4*>(orow + c * 32 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

// ----------------------------------------------------------------------------------------------------------------
// d > 384: O needs two 384-column chunks (TMEM holds 384 O + 128 S columns), i.e. two CTAs per (user tile, item range).
// Instead of both recomputing S for every item tile, they form a cluster of 2 and split the tiles: CTA r owns the tiles
// with (tile & 1) == r -- it runs G1 and the softmax for them and writes the bf16 P tile into BOTH CTAs' shared memory
// (local st.shared + st.shared::cluster through DSMEM, 32 KB per tile, ~5 B/cycle); both CTAs then run G2 for every tile
// on their own column chunk.  Executed flops drop from 6*B*N*d to the algorithmic 4*B*N*d.
// G2 lags two tiles behind G1 so that a tile's softmax (and the DSMEM copy) hides behind the two G2s in between.
// P buffer b = tile & 1 is always written by CTA b: p_full[b] collects that CTA's four softmax warps (local or remote
// arrives); p_free[b] lives in CTA b and collects the G2 completion of both CTAs (tcgen05.commit to a cluster address).
// Barrier phases count the uses of a buffer across (possibly repeated) sweeps: CTA/buffer b sees nb(b) = #{tile : tile & 1 == b}
// uses per sweep.
__global__ void __launch_bounds__(192, 1) score_grad_pair_kernel(const __grid_constant__ CUtensorMap tmU,
                                                                 const __grid_constant__ CUtensorMap tmE, GradParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* pbuf = smem + G_STAGES * G_SLOT;                         // 2 x 32 KB
    GradBarriers* bars = reinterpret_cast<GradBarriers*>(pbuf + 2 * G_PBYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x, chunk = blockIdx.y, split = blockIdx.z;
    const uint32_t rank = cluster_ctarank(), peer = rank ^ 1u;      // cluster = the two chunk CTAs: rank == chunk
    const int n_tiles_total = (P.N + G_BN - 1) / G_BN;
    const int t0 = split * P.tiles_per_split, t1 = min(n_tiles_total, t0 + P.tiles_per_split);
    const int T = t1 - t0;
    const int KB = (P.d + BK - 1) / BK;
    const int dpad = KB * BK;
    const int dc0 = chunk * G_DCHUNK;
    const int DC = min(G_DCHUNK, dpad - dc0);
    const int NG = (DC + 255) / 256;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmU);
        tma_prefetch_desc(&tmE);
        for (int s = 0; s < G_STAGES; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        mbar_init(&bars->s_full, 1); mbar_init(&bars->s_free, 4); mbar_init(&bars->o_full, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(&bars->p_full[a], 4); mbar_init(&bars->p_free[a], 2); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<512>(&bars->tmem_base);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();            // the peer's barriers are initialised before anybody arrives on them remotely
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    pdl_launch_dependents();       // after the TMEM allocation (see score_stats_kernel)
    pdl_wait();
    const uint32_t tmem_O = tmem_base, tmem_S = tmem_base + G_DCHUNK;
    auto own = [&](int ti) { return (uint32_t)(ti & 1) == rank; };
    auto uses = [&](int b) { return (T + 1 - b) >> 1; };              // tiles of parity b per sweep
    const bool onepass = P.c_part != nullptr;

    const int q = warp & 3;
    const int r_local = q * 32 + lane;
    const int row = m_tile * BM + r_local;
    const bool row_ok = warp >= 2 && row < P.B;
    const uint32_t lane_base = uint32_t(q * 32) << 16;
    float lse_row = 0.f;      // two-pass: the row's log-sum-exp; one-pass: the shift
    if (row_ok && !onepass) {
        if (P.lse) lse_row = P.lse[row];
        else {
            lse_row = merged_lse(P.part_m, P.part_l, P.lse_splits, row);
            if (chunk == 0 && split == 0) P.lse_out[row] = lse_row;
        }
    }
    float lsum = 0.f;
    int it = 0;
    const int pb_mine = (int)rank;                                  // the P buffer this CTA writes
    const uint32_t pfull_local = smem_u32(&bars->p_full[pb_mine]);
    const uint32_t pfull_peer = map_to_cta(pfull_local, peer);
    const uint32_t prow_local = smem_u32(pbuf + pb_mine * G_PBYTES + r_local * 128);
    const uint32_t prow_peer = map_to_cta(prow_local, peer);

    for (int sweep = 0;; ++sweep) {
        if (warp == 0) {
            if (lane == 0) {
                auto acquire = [&](uint32_t bytes) {
                    const int s = it % G_STAGES;
                    mbar_wait(&bars->empty[s], ((it / G_STAGES) & 1) ^ 1);
                    mbar_expect_tx(&bars->full[s], bytes);
                    ++it;
                    return s;
                };
                for (int ti = 0; ti < T + 2; ++ti) {
                    if (ti < T && own(ti)) {          // G1 operands of my tile ti
                        const int item0 = (t0 + ti) * G_BN;
                        for (int kb = 0; kb < KB; ++kb) {
                            const int s = acquire(G_SLOT);
                            uint8_t* slot = smem + s * G_SLOT;
                            tma_load_2d(slot, &tmU, kb * BK, m_tile * BM, &bars->full[s]);
                            tma_load_2d(slot + 16384, &tmE, kb * BK, item0, &bars->full[s]);
                            tma_load_2d(slot + 16384 + 8192, &tmE, kb * BK, item0 + 64, &bars->full[s]);
                        }
                    }
                    if (ti >= 2) {                    // G2 operands of tile ti-2 (every tile, my column chunk)
                        const int item0 = (t0 + ti - 2) * G_BN;
                        for (int ih = 0; ih < 2; ++ih)
                            for (int g = 0; g < NG; ++g) {
                                const int nb = min(4, (DC - g * 256) / 64);
                                const int s = acquire(nb * 8192);
                                uint8_t* slot = smem + s * G_SLOT;
                                for (int j = 0; j < nb; ++j)
                                    tma_load_2d(slot + j * 8192, &tmE, dc0 + g * 256 + j * 64, item0 + ih * 64, &bars->full[s]);
                            }
                    }
                }
            }
        } else if (warp == 1) {
            if (lane == 0) {
                constexpr uint32_t idesc1 = make_idesc(BM, G_BN, 0, 0);
                for (int ti = 0; ti < T + 2; ++ti) {
                    if (ti < T && own(ti)) {          // G1(ti): S = U E_t^T
                        const int k = sweep * uses((int)rank) + (ti >> 1);        // my k-th own tile overall
                        mbar_wait(&bars->s_free, (k & 1) ^ 1);
                        tc_fence_after();
                        for (int kb = 0; kb < KB; ++kb, ++it) {
                            const int s = it % G_STAGES;
                            mbar_wait(&bars->full[s], (it / G_STAGES) & 1);
                            tc_fence_after();
                            const uint32_t a0 = smem_u32(smem + s * G_SLOT), b0 = a0 + 16384;
#pragma unroll
                            for (int kk = 0; kk < BK / 16; ++kk)
                                umma_ss(tmem_S, make_desc(a0 + kk * 32, 16, 1024), make_desc(b0 + kk * 32, 16, 1024), idesc1, (kb | kk) != 0);
                            umma_commit(&bars->empty[s]);
                        }
                        umma_commit(&bars->s_full);
                    }
                    if (ti >= 2) {                    // G2(ti-2): O += P E_t
                        const int tj = ti - 2, pb = tj & 1;
                        const int u = sweep * uses(pb) + (tj >> 1);               // use count of buffer pb
                        mbar_wait_cluster(&bars->p_full[pb], u & 1);              // P may have been written by the peer CTA
                        fence_proxy_async_all();
                        tc_fence_after();
                        const uint32_t p0 = smem_u32(pbuf + pb * G_PBYTES);
                        for (int ih = 0; ih < 2; ++ih)
                            for (int g = 0; g < NG; ++g, ++it) {
                                const int ncols = min(256, DC - g * 256);
                                const uint32_t idesc2 = make_idesc(BM, ncols, 0, 1);
                                const int s = it % G_STAGES;
                                mbar_wait(&bars->full[s], (it / G_STAGES) & 1);
                                tc_fence_after();
                                const uint32_t b0 = smem_u32(smem + s * G_SLOT);
#pragma unroll
                                for (int kk = 0; kk < 4; ++kk)
                                    umma_ss(tmem_O + g * 256, make_desc(p0 + ih * 16384 + kk * 32, 16, 1024),
                                            make_desc(b0 + kk * 2048, 8192, 1024), idesc2, (tj | ih | kk) != 0);
                                umma_commit(&bars->empty[s]);
                            }
                        // buffer pb may be rewritten once BOTH CTAs are done with it: its owner (CTA pb) collects both commits
                        umma_commit_cluster(map_to_cta(smem_u32(&bars->p_free[pb]), (uint32_t)pb));
                    }
                }
                umma_commit(&bars->o_full);
            }
        } else {
            const float lse2 = lse_row * kLog2e;
            lsum = 0.f;
            for (int ti = (int)rank; ti < T; ti += 2) {                 // my tiles only
                const int k = sweep * uses((int)rank) + (ti >> 1);
                mbar_wait(&bars->s_full, k & 1);
                tc_fence_after();
                float v[4][32];
#pragma unroll
                for (int c = 0; c < 4; ++c) tmem_ld32(tmem_S + lane_base + c * 32, v[c]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->s_free);
                mbar_wait_cluster(&bars->p_free[pb_mine], (k & 1) ^ 1);      // both CTAs finished G2 of my previous tile
                auto store = [&](int item, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
                    const uint32_t off = (uint32_t)((item >> 6) * 16384 + ((((item & 63) >> 3) ^ (r_local & 7)) << 4));
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(prow_local + off), "r"(w0), "r"(w1), "r"(w2), "r"(w3) : "memory");
                    st_cluster_v4(prow_peer + off, w0, w1, w2, w3);
                };
                const int n_valid = P.N - (t0 + ti) * G_BN;
                if (n_valid >= G_BN) lsum += softmax_tile<false>(v, lse2, G_BN, store);
                else lsum += softmax_tile<true>(v, lse2, n_valid, store);
                fence_proxy_async_all();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&bars->p_full[pb_mine]);
                    mbar_arrive_cluster(pfull_peer);
                }
            }
            mbar_wait(&bars->o_full, sweep & 1);      // every MMA of this CTA's sweep has completed
            tc_fence_after();
        }
        __syncwarp();
        if (!onepass) break;
        // each CTA saw only its own tiles: the decision is taken on the pair's sum, identically in both CTAs
        if (warp >= 2) {
            bars->rsum[rank][r_local] = lsum;
            const uint32_t remote = map_to_cta(smem_u32(&bars->rsum[rank][r_local]), peer);
            asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(lsum) : "memory");
        }
        cluster_sync_all();
        const float both = warp >= 2 ? bars->rsum[0][r_local] + bars->rsum[1][r_local] : 1.0f;
        const bool over = both > kOnepassOver, under = both < kOnepassUnder;
        if (!__syncthreads_or(over || under) || sweep + 1 >= kOnepassMaxSweeps) break;
        lse_row += over ? kOnepassRetry : under ? -kOnepassRetry : 0.f;
        cluster_sync_all();            // the peer has read this sweep's sums before the next sweep's overwrite them
    }
    if (warp >= 2) {
        // ---- O (TMEM) -> global partial ---------------------------------------------------------------------
        if (onepass && row_ok) {
            if (rank == 0) P.c_part[(size_t)split * P.B + row] = lse_row;
            P.l_part[((size_t)split * 2 + rank) * P.B + row] = lsum;        // each CTA of the pair: its own tiles
        }
        float* orow = P.Opart + ((size_t)split * P.B + row) * P.ldo + dc0;
        for (int c = 0; c < DC / 32; ++c) {
            float v[32];
            tmem_ld32(tmem_O + lane_base + c * 32, v);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (dc0 + c * 32 + j < P.ldo)
                        *reinterpret_cast<float4*>(orow + c * 32 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();            // nobody leaves while the peer may still store into / arrive on this CTA's shared memory
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

constexpr size_t kGradSmem = G_STAGES * G_SLOT + 2 * G_PBYTES + 1536 + 1024;

#include "score_duo.cuh"

// Item splits per (user tile, column chunk): one CTA per SM in a single wave when each CTA would otherwise get only a
// few tiles (the prologue -- barrier init, TMEM alloc, first TMA -- costs about one tile), two waves for long CTAs.
static int pick_wave_splits(int units, int n_tiles) {
    units = max(1, units);
    int splits = max(1, min(n_tiles, kNumSMs / units));
    int tps = (n_tiles + splits - 1) / splits;
    if (tps > 16) {   // long CTAs: pick the wave count (<= 6) that fills the last wave best
        double best = -1.0;
        for (int k = 1; k <= 6; ++k) {
            const int sk = max(1, min(n_tiles, (k * kNumSMs) / units));
            const double util = (double)(units * sk) / (double)(kNumSMs * ((units * sk + kNumSMs - 1) / kNumSMs));
            if (util > best + 0.02) { best = util; splits = sk; }
        }
        tps = (n_tiles + splits - 1) / splits;
    }
    return (n_tiles + tps - 1) / tps;
}
static int pick_grad_splits(int m_tiles, int n_chunks, int n_tiles) { return pick_wave_splits(m_tiles * n_chunks, n_tiles); }

// ---- host: TMA descriptors ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// bf16 row-major [rows, cols] with leading dimension ld (elements); box = [box_rows, 64 cols], 128B swizzle, OOB -> 0
int make_tmap_bf16(CUtensorMap* out, const void* base, int rows, int cols, int ld, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return hvae_fail("cuTensorMapEncodeTiled is not available from the driver");
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld * 2) % 16) return hvae_fail("TMA operand must be 16-byte aligned with ld %% 8 == 0 (ld=%d)", ld);
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return hvae_fail("cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
    return 0;
}

// The same matrix (needs cols % 64 == 0) seen as (64 columns, rows, cols / 64 column blocks): box = [2 blocks][64 rows][64 columns],
// i.e. two consecutive [64 x 64] 128B-swizzled operand boxes per TMA instruction.
int make_tmap_bf16_blocks(CUtensorMap* out, const void* base, int rows, int cols, int ld) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return hvae_fail("cuTensorMapEncodeTiled is not available from the driver");
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld * 2) % 16 || cols % 64) return hvae_fail("blocked TMA view needs cols %% 64 == 0 (cols=%d ld=%d)", cols, ld);
    cuuint64_t dims[3] = {64, (cuuint64_t)rows, (cuuint64_t)(cols / 64)};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2, 128};
    cuuint32_t box[3] = {64, 64, 2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return hvae_fail("cuTensorMapEncodeTiled (blocked view) failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
    return 0;
}

static int pick_splits(int m_tiles, int n_tiles) { return pick_wave_splits(m_tiles, n_tiles); }
// Top-K mode: every item split restarts its per-row candidate list, and a list costs ~K(1 + ln(items/K)) insertions per
// row, so the epilogue work grows with the number of splits: use a single wave of CTAs (at most one CTA per SM).
static int pick_topk_splits(int m_tiles, int n_tiles) {
    const int splits = max(1, min(n_tiles, kNumSMs / max(1, m_tiles)));
    const int tps = (n_tiles + splits - 1) / splits;
    return (n_tiles + tps - 1) / tps;
}

constexpr size_t kStatsSmem = STAGES * STAGE_BYTES + 256 + 1024;                                        // LSE, register-list top-K
constexpr size_t kStatsSmemList = STAGES_SMEM_LIST * STAGE_BYTES + 256 + BM * (MAXK_TC + 1) * 8 + 1024;   // shared-memory-list top-K

// Sets the shared-memory limit of every top-K list bucket of one FILTER / SAMPLE flavour (once per process).
template <bool FILTER, bool SAMPLE>
static int topk_set_attrs() {
    static bool attr_set = false;
    if (!attr_set) {
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES, 8, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES, 12, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES, 16, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES, 20, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES, 24, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES, 32, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_TOPK, STAGES_SMEM_LIST, 0, FILTER, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)kStatsSmemList));
        attr_set = true;
    }
    return 0;
}

// the list capacity is a compile-time size (register arrays): the smallest bucket that holds K.  A list longer than K costs twice: the
// admission threshold is its LAST entry (more insertions) and every insertion walks the whole list -- hence buckets at the evaluation
// protocol's own K values (5, 10, 20: src/ml/evaluate.py k_values)
template <bool FILTER, bool SAMPLE = false>
static int launch_topk(int K, dim3 grid, cudaStream_t st, const CUtensorMap& tmU, const CUtensorMap& tmE, const StatsParams& P) {
    if (int rc = topk_set_attrs<FILTER, SAMPLE>()) return rc;
    static const int force_kreg = getenv("HVAE_TOPK_KREG") ? atoi(getenv("HVAE_TOPK_KREG")) : 0;        // A/B runs: a larger bucket than needed
    if (force_kreg >= K && force_kreg <= MAXK_REG) K = force_kreg;       // (P.K, the number of results written, stays)
    if (K <= 8) launch_pdl(score_stats_kernel<MODE_TOPK, STAGES, 8, FILTER, SAMPLE>, grid, 192, kStatsSmem, st, tmU, tmE, P);
    else if (K <= 12) launch_pdl(score_stats_kernel<MODE_TOPK, STAGES, 12, FILTER, SAMPLE>, grid, 192, kStatsSmem, st, tmU, tmE, P);
    else if (K <= 16) launch_pdl(score_stats_kernel<MODE_TOPK, STAGES, 16, FILTER, SAMPLE>, grid, 192, kStatsSmem, st, tmU, tmE, P);
    else if (K <= 20) launch_pdl(score_stats_kernel<MODE_TOPK, STAGES, 20, FILTER, SAMPLE>, grid, 192, kStatsSmem, st, tmU, tmE, P);
    else if (K <= 24) launch_pdl(score_stats_kernel<MODE_TOPK, STAGES, 24, FILTER, SAMPLE>, grid, 192, kStatsSmem, st, tmU, tmE, P);
    else if (K <= MAXK_REG) launch_pdl(score_stats_kernel<MODE_TOPK, STAGES, 32, FILTER, SAMPLE>, grid, 192, kStatsSmem, st, tmU, tmE, P);
    else launch_pdl(score_stats_kernel<MODE_TOPK, STAGES_SMEM_LIST, 0, FILTER, SAMPLE>, grid, 192, kStatsSmemList, st, tmU, tmE, P);
    HVAE_LAUNCH_CHECK(SAMPLE ? "tc_score_topk_sampled" : FILTER ? "tc_score_topk_filtered" : "tc_score_topk");
    return 0;
}

}  // namespace tc
}  // namespace hvae

using namespace hvae;
using namespace hvae::tc;

extern "C" {

int hvae_cast_bf16(const float* src, int rows, int cols, int ld_src, void* dst, int ld_dst, void* stream) {
    if (rows == 0) return 0;
    const int64_t total = (int64_t)rows * ld_dst;
    launch_pdl(cast_bf16_kernel, (unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream, src, rows, cols, ld_src, (__nv_bfloat16*)dst, ld_dst);
    HVAE_LAUNCH_CHECK("cast_bf16");
    return 0;
}

size_t hvae_tc_n_splits(int B, int N) { return (size_t)pick_splits(ceil_div(B, BM), ceil_div(N, BN)); }
size_t hvae_tc_topk_splits(int B, int N) { return (size_t)pick_topk_splits(ceil_div(B, BM), ceil_div(N, BN)); }

static int launch_stats_lse(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* workspace, int* n_splits,
                            cudaStream_t stream) {
    CUtensorMap tmU, tmE;
    if (int rc = make_tmap_bf16(&tmU, U, B, d, ldu, BM)) return rc;
    if (int rc = make_tmap_bf16(&tmE, E, N, d, lde, BN)) return rc;
    const int m_tiles = ceil_div(B, BM), n_tiles = ceil_div(N, BN);
    StatsParams P{};
    P.B = B; P.N = N; P.d = d;
    P.n_splits = pick_splits(m_tiles, n_tiles);
    P.tiles_per_split = ceil_div(n_tiles, P.n_splits);
    P.part_m = workspace;
    P.part_l = workspace + (size_t)B * P.n_splits;
    static bool attr_set = false;
    if (!attr_set) {
        HVAE_CUDA(cudaFuncSetAttribute(score_stats_kernel<MODE_LSE, STAGES, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStatsSmem));
        attr_set = true;
    }
    launch_pdl(score_stats_kernel<MODE_LSE, STAGES, 0>, dim3(m_tiles, P.n_splits), 192, kStatsSmem, stream, tmU, tmE, P);
    HVAE_LAUNCH_CHECK("tc_score_lse");
    *n_splits = P.n_splits;
    return 0;
}

// Which kernel runs the two chained GEMMs: the CTA-pair kernel (tcgen05 cta_group::2, score_duo.cuh) for d <= 768, the
// DSMEM pair of column-chunk CTAs for 384 < d <= 768 when the former is disabled, the one-CTA-per-chunk kernel otherwise.
// HVAE_SCORE_KERNEL = duo | pair | single overrides (profiling / A-B runs).
enum GradKind { GRAD_SINGLE = 0, GRAD_PAIR = 1, GRAD_DUO = 2 };
static long long* g_duo_trace = nullptr;     // hvae_tc_duo_trace (profiling)
static GradKind grad_kind(int d) {
    static const char* env = getenv("HVAE_SCORE_KERNEL");
    static const bool no_pair = getenv("HVAE_NO_PAIR") != nullptr;
    const bool two_chunks = ceil_div(round_up(d, BK), G_DCHUNK) == 2;
    if (env && env[0] == 's') return GRAD_SINGLE;
    if (env && env[0] == 'p') return two_chunks && !no_pair ? GRAD_PAIR : GRAD_SINGLE;
    if (d <= D_MAXD) return GRAD_DUO;
    return two_chunks && !no_pair ? GRAD_PAIR : GRAD_SINGLE;
}
static int grad_units_per_mtile(int d) { return grad_kind(d) == GRAD_DUO ? 2 : ceil_div(round_up(d, BK), G_DCHUNK); }

static int launch_grad(const void* U, int ldu, int B, const void* E, int lde, int N, int d, const float* lse, const float* part_m,
                       const float* part_l, int lse_splits, float* lse_out, float* Opart, int ldo, cudaStream_t stream,
                       float* c_part = nullptr, float* l_part = nullptr) {
    HVAE_REQUIRE(ldo % 4 == 0 && ldo >= d, "tc_score_grad: bad ldo=%d for d=%d", ldo, d);
    const GradKind kind = grad_kind(d);
    CUtensorMap tmU, tmE;
    static const bool no3d = getenv("HVAE_DUO_NO3D") != nullptr;
    const bool box3d = kind == GRAD_DUO && d % 64 == 0 && !no3d && make_tmap_bf16_blocks(&tmU, U, B, d, ldu) == 0 &&
                       make_tmap_bf16_blocks(&tmE, E, N, d, lde) == 0;
    if (!box3d) {
        if (int rc = make_tmap_bf16(&tmU, U, B, d, ldu, kind == GRAD_DUO ? 64 : BM)) return rc;
        if (int rc = make_tmap_bf16(&tmE, E, N, d, lde, 64)) return rc;
    }
    const int m_tiles = ceil_div(B, BM), n_chunks = ceil_div(round_up(d, BK), G_DCHUNK), n_tiles = ceil_div(N, G_BN);
    GradParams P{};
    P.B = B; P.N = N; P.d = d; P.lse = lse; P.part_m = part_m; P.part_l = part_l; P.lse_splits = lse_splits; P.lse_out = lse_out;
    P.Opart = Opart; P.ldo = ldo;
    P.c_part = c_part; P.l_part = l_part; P.box3d = box3d ? 1 : 0;
    P.n_splits = pick_grad_splits(m_tiles, grad_units_per_mtile(d), n_tiles);
    P.tiles_per_split = ceil_div(n_tiles, P.n_splits);
    static bool attr_set = false;
    if (!attr_set) {
        HVAE_CUDA(cudaFuncSetAttribute(score_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGradSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_grad_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGradSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_grad_duo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDuoSmem));
        HVAE_CUDA(cudaFuncSetAttribute(score_grad_duo_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDuoSmem));
        attr_set = true;
    }
    if (kind != GRAD_SINGLE) {      // clusters of 2 along y: the CTA pair of one (user tile, item range)
        cudaLaunchConfig_t cfg = {};
        // (the CTA pair of a cta_group::2 kernel must lie along x; the DSMEM pair kernel keeps its (user tile, chunk) grid)
        cfg.gridDim = kind == GRAD_DUO ? dim3(2, m_tiles, P.n_splits) : dim3(m_tiles, 2, P.n_splits);
        cfg.blockDim = dim3(192);
        cfg.dynamicSmemBytes = kind == GRAD_DUO ? kDuoSmem : kGradSmem;
        cfg.stream = stream;
        cudaLaunchAttribute attr[2];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kind == GRAD_DUO ? 2 : 1; attr[0].val.clusterDim.y = kind == GRAD_DUO ? 1 : 2; attr[0].val.clusterDim.z = 1;
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = pdl_enabled() ? 2 : 1;
        if (kind == GRAD_DUO && g_duo_trace) HVAE_CUDA(cudaLaunchKernelEx(&cfg, score_grad_duo_kernel<true>, tmU, tmE, P, g_duo_trace));
        else if (kind == GRAD_DUO) HVAE_CUDA(cudaLaunchKernelEx(&cfg, score_grad_duo_kernel<false>, tmU, tmE, P, (long long*)nullptr));
        else HVAE_CUDA(cudaLaunchKernelEx(&cfg, score_grad_pair_kernel, tmU, tmE, P));
        HVAE_LAUNCH_CHECK("tc_score_grad(pair)");
        return 0;
    }
    launch_pdl(score_grad_kernel, dim3(m_tiles, n_chunks, P.n_splits), 192, kGradSmem, stream, tmU, tmE, P);
    HVAE_LAUNCH_CHECK("tc_score_grad");
    return 0;
}

// workspace: 2 * B * n_splits floats
int hvae_tc_score_lse(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* lse, float* workspace, void* stream) {
    if (B == 0) return 0;
    HVAE_REQUIRE(N > 0 && d > 0, "tc_score_lse: empty catalogue");
    int ns = 0;
    if (int rc = launch_stats_lse(U, ldu, B, E, lde, N, d, workspace, &ns, (cudaStream_t)stream)) return rc;
    launch_pdl(lse_merge_kernel, ceil_div(B, 128), 128, 0, (cudaStream_t)stream, workspace, workspace + (size_t)B * ns, B, ns, lse);
    HVAE_LAUNCH_CHECK("tc_score_lse merge");
    return 0;
}

// Forward + backward through the scores in two launches: the backward kernel merges the forward partials itself.
int hvae_tc_score_lse_grad(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* lse, float* workspace,
                           float* Opart, int ldo, void* stream) {
    if (B == 0) return 0;
    HVAE_REQUIRE(N > 0 && d > 0, "tc_score_lse_grad: empty catalogue");
    int ns = 0;
    if (int rc = launch_stats_lse(U, ldu, B, E, lde, N, d, workspace, &ns, (cudaStream_t)stream)) return rc;
    return launch_grad(U, ldu, B, E, lde, N, d, nullptr, workspace, workspace + (size_t)B * ns, ns, lse, Opart, ldo, (cudaStream_t)stream);
}

static int score_topk(const void* U, int ldu, int B, const void* E, int lde, int N, int d, int item_offset, const int64_t* indptr,
                      const int32_t* indices, const int32_t* rows, const uint32_t* allow, int64_t allow_stride,
                      const int32_t* allow_of_row, const float* row_inv_tau, const uint64_t* row_seed, int K, float* cand_val,
                      int32_t* cand_idx, void* stream) {
    if (B == 0) return 0;
    HVAE_REQUIRE(K >= 1 && K <= MAXK_TC, "tc_score_topk: K=%d outside [1,%d]", K, MAXK_TC);
    CUtensorMap tmU, tmE;
    if (int rc = make_tmap_bf16(&tmU, U, B, d, ldu, BM)) return rc;
    if (int rc = make_tmap_bf16(&tmE, E, N, d, lde, BN)) return rc;
    const int m_tiles = ceil_div(B, BM), n_tiles = ceil_div(N, BN);
    StatsParams P{};
    P.B = B; P.N = N; P.d = d; P.K = K; P.item_offset = item_offset;
    P.n_splits = pick_topk_splits(m_tiles, n_tiles);
    P.tiles_per_split = ceil_div(n_tiles, P.n_splits);
    P.cand_val = cand_val; P.cand_idx = cand_idx;
    P.indptr = indptr; P.indices = indices; P.rows = rows;
    P.allow = allow; P.allow_stride = allow_stride; P.allow_of_row = allow_of_row;
    P.row_inv_tau = row_inv_tau; P.row_seed = row_seed;
    const dim3 grid(m_tiles, P.n_splits);
    if (row_inv_tau) return launch_topk<true, true>(K, grid, (cudaStream_t)stream, tmU, tmE, P);
    if (allow) return launch_topk<true>(K, grid, (cudaStream_t)stream, tmU, tmE, P);
    return launch_topk<false>(K, grid, (cudaStream_t)stream, tmU, tmE, P);
}

// Top-K over the N items of E (global ids item_offset..item_offset+N).  cand_val / cand_idx: [B, n_splits*K] scratch;
// the caller reduces them with hvae_topk_merge.  K <= 128 (K <= 32: register-resident lists; above: shared-memory lists).
int hvae_tc_score_topk(const void* U, int ldu, int B, const void* E, int lde, int N, int d, int item_offset, const int64_t* indptr,
                       const int32_t* indices, const int32_t* rows, int K, float* cand_val, int32_t* cand_idx, void* stream) {
    return score_topk(U, ldu, B, E, lde, N, d, item_offset, indptr, indices, rows, nullptr, 0, nullptr, nullptr, nullptr, K, cand_val,
                      cand_idx, stream);
}

// The same restricted to per-row allow-sets: row b may only return items whose bit is set in allow[allow_of_row[b]] (bitmaps over
// global item ids, allow_stride_words >= ceil((item_offset + N) / 32)); allow_of_row[b] == -1: unrestricted.  allow == NULL is
// hvae_tc_score_topk.  A row with fewer than K admissible items pads its list with (-inf, -1).
int hvae_tc_score_topk_filtered(const void* U, int ldu, int B, const void* E, int lde, int N, int d, int item_offset,
                                const int64_t* indptr, const int32_t* indices, const int32_t* rows, const uint32_t* allow,
                                int64_t allow_stride_words, const int32_t* allow_of_row, int K, float* cand_val, int32_t* cand_idx,
                                void* stream) {
    if (allow) {
        HVAE_REQUIRE(allow_of_row, "tc_score_topk_filtered: allow needs allow_of_row");
        HVAE_REQUIRE(item_offset >= 0 && allow_stride_words >= ((int64_t)item_offset + N + 31) / 32,
                     "tc_score_topk_filtered: allow_stride_words=%lld does not cover items up to %lld", (long long)allow_stride_words,
                     (long long)item_offset + N);
    }
    return score_topk(U, ldu, B, E, lde, N, d, item_offset, indptr, indices, rows, allow, allow_stride_words, allow_of_row, nullptr,
                      nullptr, K, cand_val, cand_idx, stream);
}

// Gumbel-top-K sampling on top of hvae_tc_score_topk_filtered (see the header for the noise).  cand_val holds the keys
// s * row_inv_tau + g (s itself where row_inv_tau == 0); merge with hvae_topk_merge, then take the scores of the chosen ids.
int hvae_tc_score_topk_sampled(const void* U, int ldu, int B, const void* E, int lde, int N, int d, int item_offset,
                               const int64_t* indptr, const int32_t* indices, const int32_t* rows, const uint32_t* allow,
                               int64_t allow_stride_words, const int32_t* allow_of_row, const float* row_inv_tau,
                               const uint64_t* row_seed, int K, float* cand_val, int32_t* cand_idx, void* stream) {
    HVAE_REQUIRE(row_inv_tau && row_seed, "tc_score_topk_sampled: row_inv_tau and row_seed are required");
    if (allow) {
        HVAE_REQUIRE(allow_of_row, "tc_score_topk_sampled: allow needs allow_of_row");
        HVAE_REQUIRE(item_offset >= 0 && allow_stride_words >= ((int64_t)item_offset + N + 31) / 32,
                     "tc_score_topk_sampled: allow_stride_words=%lld does not cover items up to %lld", (long long)allow_stride_words,
                     (long long)item_offset + N);
    }
    return score_topk(U, ldu, B, E, lde, N, d, item_offset, indptr, indices, rows, allow, allow_stride_words, allow_of_row,
                      row_inv_tau, row_seed, K, cand_val, cand_idx, stream);
}

// 1 or 2 numerator sums per (split, row): the pair kernel's two CTAs each report the tiles they owned
size_t hvae_tc_onepass_subparts(int d) { return grad_kind(d) != GRAD_SINGLE ? 2 : 1; }

// Forward and backward through the scores in ONE sweep over the items (4 B N d executed flops instead of the 6 B N d of
// hvae_tc_score_lse_grad): the backward kernel takes the softmax numerators against a score-independent shift and also returns
// their row sums.  Opart then holds UNNORMALISED sums; hvae_tc_onepass_combine turns (c_part, l_part) into the log-sum-exp and
// the weights hvae_du_finalize applies to the partials.
int hvae_tc_score_onepass(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* c_part, float* l_part,
                          float* Opart, int ldo, void* stream) {
    if (B == 0) return 0;
    HVAE_REQUIRE(N > 0 && d > 0, "tc_score_onepass: empty catalogue");
    HVAE_REQUIRE(c_part && l_part, "tc_score_onepass: c_part / l_part are required");
    return launch_grad(U, ldu, B, E, lde, N, d, nullptr, nullptr, nullptr, 0, nullptr, Opart, ldo, (cudaStream_t)stream, c_part, l_part);
}

int hvae_tc_onepass_combine(const float* c_part, const float* l_part, int n_parts, int n_sub, int B, float* lse, float* w_part,
                            void* stream) {
    if (B == 0) return 0;
    launch_pdl(onepass_combine_kernel, ceil_div(B, 8), 256, 0, (cudaStream_t)stream, c_part, l_part, n_parts, n_sub, B, lse, w_part);
    HVAE_LAUNCH_CHECK("tc_onepass_combine");
    return 0;
}

// Profiling: while `trace` is non-null the cta_group::2 scoring kernel runs its instrumented build and writes, per CTA and per
// role (0 TMA producer, 1 MMA issuer, 2 first softmax warp), 8 int64 cycle counters: [wait0..wait3, -, -, -, lifetime]
// (producer: wait0 = ring slot free; MMA: S buffer free, G1 operands, P written, G2 operands; softmax: S ready, P buffer free,
// sweep's MMAs done).  trace: [n_splits * m_tiles * 2][3][8] int64 device memory.
int hvae_tc_duo_trace(int64_t* trace_) {
    long long* trace = reinterpret_cast<long long*>(trace_);
    g_duo_trace = trace;
    return 0;
}

// Diagnostic: how many CTA pairs of the cta_group::2 scoring kernel the device can hold at once with `smem_bytes` of dynamic
// shared memory per CTA (0 = the kernel's own size); negative = the query failed (hvae_last_error()).
int hvae_tc_duo_max_clusters(int smem_bytes) {
    const size_t smem = smem_bytes > 0 ? (size_t)smem_bytes : kDuoSmem;
    if (cudaFuncSetAttribute(score_grad_duo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        hvae_fail("tc_duo_max_clusters: %s", cudaGetErrorString(cudaGetLastError()));
        return -1;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2, 1, 74);
    cfg.blockDim = dim3(192);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, score_grad_duo_kernel<false>, &cfg) != cudaSuccess) {
        hvae_fail("tc_duo_max_clusters: %s", cudaGetErrorString(cudaGetLastError()));
        return -2;
    }
    return n;
}

size_t hvae_tc_grad_splits(int B, int N, int d) {
    return (size_t)pick_grad_splits(ceil_div(B, BM), grad_units_per_mtile(d), ceil_div(N, G_BN));
}

// Opart: [hvae_tc_grad_splits(B,N,d)][B][ldo] floats, ldo % 4 == 0, ldo >= d; every partial is fully written for
// columns < min(ldo, round_up(d,64)).  O = sum of the partials (hvae_du_finalize does it).
int hvae_tc_score_grad(const void* U, int ldu, int B, const void* E, int lde, int N, int d, const float* lse, float* Opart, int ldo,
                       void* stream) {
    if (B == 0) return 0;
    return launch_grad(U, ldu, B, E, lde, N, d, lse, nullptr, nullptr, 0, nullptr, Opart, ldo, (cudaStream_t)stream);
}

}  // extern "C"

// Row-wise kernels around the scoring GEMM.
//  * row_lse / row_softmax_scale : log-softmax pieces of the multinomial NLL for the fp32 (materialised) mode
//    (reference src/ml/model.py:281).
//  * sparse_dot_xsum : sum_j x_bj * S_b,idx_j as r sparse dot products u_b . E_idx  (SURVEY.md H4).
//  * du_finalize     : dU_b = scale_b * O_b - (1/Bg) * sum_j x_bj E_idx_j  -- the "-x" half of
//    (softmax*|x| - x) . E (model.py:281 backward) is an embedding-bag gather of E rows.
//  * mask_topk       : seen-item masking + per-user warp-level top-K over a materialised score row
//    (reference src/ml/evaluate.py:143-146), total order (score desc, index desc).
//  * hit_mask / metrics_reduce : Recall/NDCG/HR@K (src/ml/evaluate.py:32-54,90-98).
#include <cuda_bf16.h>

#include "common.cuh"

namespace hvae {

__device__ __forceinline__ void ml_merge(float& m, float& l, float m2, float l2) {
    const float mn = fmaxf(m, m2);
    if (mn == -INFINITY) { m = mn; l = 0.f; return; }
    l = l * expf(m - mn) + l2 * expf(m2 - mn);
    m = mn;
}

__global__ void __launch_bounds__(256) row_lse_kernel(const float* __restrict__ S, int64_t lds, int N, float* __restrict__ lse) {
    pdl_prologue();
    const float* row = S + (size_t)blockIdx.x * lds;
    float m = -INFINITY, l = 0.f;
    for (int i = threadIdx.x; i < N; i += 256) {
        const float v = row[i];
        if (v > m) { l = l * expf(m - v) + 1.0f; m = v; }
        else l += expf(v - m);
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), l2 = __shfl_xor_sync(0xffffffffu, l, o);
        ml_merge(m, l, m2, l2);
    }
    __shared__ float sm[8], sl[8];
    if ((threadIdx.x & 31) == 0) { sm[threadIdx.x >> 5] = m; sl[threadIdx.x >> 5] = l; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) ml_merge(m, l, sm[w], sl[w]);
        lse[blockIdx.x] = m + logf(l);
    }
}

// P = exp(S - lse_b) * xsum_b * inv_bg  in place
__global__ void row_softmax_scale_kernel(float* __restrict__ S, int64_t lds, int rows, int N, const float* __restrict__ lse,
                                         const float* __restrict__ xsum, const float* __restrict__ inv_bg) {
    pdl_prologue();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)rows * N) return;
    const int r = (int)(i / N), c = (int)(i - (int64_t)r * N);
    const size_t off = (size_t)r * lds + c;
    S[off] = expf(S[off] - lse[r]) * (xsum[r] * *inv_bg);
}

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__global__ void __launch_bounds__(256) sparse_dot_xsum_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                              const float* __restrict__ values, const int32_t* __restrict__ rows,
                                                              int B, const T* __restrict__ U, int ldu, const T* __restrict__ E,
                                                              int lde, int d, float* __restrict__ dot, float* __restrict__ xsum) {
    pdl_prologue();
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (b >= B) return;
    const int u = rows ? rows[b] : b;
    float acc = 0.f, xs = 0.f;
    for (int64_t j = indptr[u]; j < indptr[u + 1]; ++j) {
        const float x = values ? values[j] : 1.0f;
        const T* e = E + (size_t)indices[j] * lde;
        float p = 0.f;
        for (int c = lane; c < d; c += 32) p = fmaf(to_f(U[(size_t)b * ldu + c]), to_f(e[c]), p);
        acc += x * p;  // every lane holds a partial; reduced once below
        xs += x;
    }
    acc = warp_sum(acc);
    if (lane == 0) { dot[b] = acc; xsum[b] = xs; }
}

// dU[b,:] = s_b * sum_p O[p][b,:] - inv_bg * sum_j x_bj E[idx_j,:];  s_b = oscale ? oscale[b] * inv_bg : 1
// (O may come as n_parts partial sums over item splits, [n_parts][B][ldo], added in a fixed order.)
// One thread per 4 output columns: the partial sums and the E rows are read as coalesced vectors.
template <typename T>
__device__ __forceinline__ float4 load4(const T* p, int c, int d);
template <>
__device__ __forceinline__ float4 load4<float>(const float* p, int c, int d) {  // fp32 E has lde == d: no padding, scalar loads
    float4 r;
    r.x = c < d ? p[c] : 0.f; r.y = c + 1 < d ? p[c + 1] : 0.f; r.z = c + 2 < d ? p[c + 2] : 0.f; r.w = c + 3 < d ? p[c + 3] : 0.f;
    return r;
}
template <>
__device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p, int c, int d) {  // bf16 E rows are zero-padded to 8
    const uint2 w = *reinterpret_cast<const uint2*>(p + c);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

template <typename T>
__global__ void __launch_bounds__(256) du_finalize_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                          const float* __restrict__ values, const int32_t* __restrict__ rows, int B,
                                                          const float* __restrict__ O, int ldo, int n_parts,
                                                          const float* __restrict__ oscale, const float* __restrict__ w_part,
                                                          const T* __restrict__ E, int lde, int d,
                                                          const float* __restrict__ inv_bg, float* __restrict__ dU, int lddu,
                                                          const float* __restrict__ c_part, const float* __restrict__ l_part, int n_sub,
                                                          float* __restrict__ lse_out) {
    pdl_prologue();
    const int ld4 = lddu >> 2;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * ld4) return;
    const int b = t / ld4, c = (t - b * ld4) * 4;
    const int u = rows ? rows[b] : b;
    const float ib = *inv_bg, s = oscale ? oscale[b] * ib : 1.0f;
    // One-pass scoring (c_part != null): the combination of the per-split results of this row (shift c_p, numerator sums l_p) is done
    // here instead of in a launch of its own -- M = max_p c_p, D = sum_p e^{c_p - M} l_p, weight of split p = e^{c_p - M} / D,
    // lse = M + log D (every thread of a row repeats the few dozen operations; the addresses are warp-uniform)
    float cM = 0.f, cinv = 1.f;
    if (c_part) {
        cM = -INFINITY;
        for (int p0 = 0; p0 < n_parts; p0 += 8) {          // eight loads in flight (a dependent load per iteration costs ~0.2 us each)
            float cc[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) cc[k] = p0 + k < n_parts ? c_part[(size_t)(p0 + k) * B + b] : -INFINITY;
#pragma unroll
            for (int k = 0; k < 8; ++k) cM = fmaxf(cM, cc[k]);
        }
        float D = 0.f;
        for (int p0 = 0; p0 < n_parts; p0 += 8) {
            float cc[8], ll[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const bool ok = p0 + k < n_parts;
                cc[k] = ok ? c_part[(size_t)(p0 + k) * B + b] : -INFINITY;
                ll[k] = 0.f;
                for (int sb = 0; sb < n_sub; ++sb) ll[k] += ok ? l_part[((size_t)(p0 + k) * n_sub + sb) * B + b] : 0.f;
            }
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (p0 + k < n_parts) D = fmaf(expf(cc[k] - cM), ll[k], D);
        }
        cinv = 1.0f / D;
        if (c == 0 && lse_out) lse_out[b] = cM + logf(D);
    }
    const size_t pstride = (size_t)B * ldo;
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* op = O + (size_t)b * ldo + c;
    // partial sums in a fixed order, four loads in flight (a training step at the C2 shape has 37 item splits)
    for (int p0 = 0; p0 < n_parts; p0 += 4) {
        float4 v[4]; float w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const bool ok = p0 + q < n_parts;
            v[q] = ok ? *reinterpret_cast<const float4*>(op + (size_t)(p0 + q) * pstride) : make_float4(0.f, 0.f, 0.f, 0.f);
            w[q] = !ok ? 1.0f : c_part ? expf(c_part[(size_t)(p0 + q) * B + b] - cM) * cinv : w_part ? w_part[(size_t)(p0 + q) * B + b] : 1.0f;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (p0 + q < n_parts) { o.x = fmaf(w[q], v[q].x, o.x); o.y = fmaf(w[q], v[q].y, o.y); o.z = fmaf(w[q], v[q].z, o.z); o.w = fmaf(w[q], v[q].w, o.w); }
        }
    }
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t js = indptr[u], je = indptr[u + 1];
    for (int64_t j = js; j < je; j += 4) {       // four E rows in flight, entries accumulated in CSR order
        const int n = (int)min((int64_t)4, je - j);
        int id[4]; float x[4]; float4 e[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { id[q] = q < n ? indices[j + q] : 0; x[q] = (values && q < n) ? values[j + q] : 1.0f; }
#pragma unroll
        for (int q = 0; q < 4; ++q) e[q] = q < n ? load4<T>(E + (size_t)id[q] * lde, c, d) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (q < n) { a.x = fmaf(x[q], e[q].x, a.x); a.y = fmaf(x[q], e[q].y, a.y); a.z = fmaf(x[q], e[q].z, a.z); a.w = fmaf(x[q], e[q].w, a.w); }
        }
    }
    float4 g;
    g.x = c < d ? s * o.x - ib * a.x : 0.f;
    g.y = c + 1 < d ? s * o.y - ib * a.y : 0.f;
    g.z = c + 2 < d ? s * o.z - ib * a.z : 0.f;
    g.w = c + 3 < d ? s * o.w - ib * a.w : 0.f;
    *reinterpret_cast<float4*>(dU + (size_t)b * lddu + c) = g;
}

// bf16 fast path of sparse_dot_xsum: U row chunks live in registers, E rows are read as 16-byte vectors.
__global__ void __launch_bounds__(256) sparse_dot_xsum_bf16_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                                   const float* __restrict__ values, const int32_t* __restrict__ rows,
                                                                   int B, const __nv_bfloat16* __restrict__ U, int ldu,
                                                                   const __nv_bfloat16* __restrict__ E, int lde, int nchunks,
                                                                   float* __restrict__ dot, float* __restrict__ xsum) {
    pdl_prologue();
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (b >= B) return;
    const int u = rows ? rows[b] : b;
    float ur[4][8];
#pragma unroll
    for (int pss = 0; pss < 4; ++pss) {
        const int ch = lane + 32 * pss;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (ch < nchunks) w = *reinterpret_cast<const uint4*>(U + (size_t)b * ldu + ch * 8);
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ww[e]));
            ur[pss][2 * e] = f.x; ur[pss][2 * e + 1] = f.y;
        }
    }
    float acc = 0.f, xs = 0.f;
    const int64_t js = indptr[u], je = indptr[u + 1];
    for (int64_t j = js; j < je; j += 4) {       // four E rows in flight per trip; same accumulation order as one by one
        const int n = (int)min((int64_t)4, je - j);
        int id[4]; float x[4]; uint4 w[4][4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { id[q] = q < n ? indices[j + q] : 0; x[q] = (values && q < n) ? values[j + q] : 1.0f; }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const __nv_bfloat16* e = E + (size_t)id[q] * lde;
#pragma unroll
            for (int pss = 0; pss < 4; ++pss) {
                const int ch = lane + 32 * pss;
                w[q][pss] = (q < n && ch < nchunks) ? __ldg(reinterpret_cast<const uint4*>(e + ch * 8)) : make_uint4(0, 0, 0, 0);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (q >= n) continue;
            float p = 0.f;
#pragma unroll
            for (int pss = 0; pss < 4; ++pss) {
                if (lane + 32 * pss < nchunks) {
                    const uint32_t ww[4] = {w[q][pss].x, w[q][pss].y, w[q][pss].z, w[q][pss].w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ww[k]));
                        p = fmaf(ur[pss][2 * k], f.x, p);
                        p = fmaf(ur[pss][2 * k + 1], f.y, p);
                    }
                }
            }
            acc = fmaf(x[q], p, acc);
            xs += x[q];
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) { dot[b] = acc; xsum[b] = xs; }
}

// Negative-sampling protocol (reference src/ml/evaluate.py:149-185): per row, the scores of C candidate items
// (candidate 0 = the held-out test item) as C sparse dot products u_b . E_c, and the 0-based rank of candidate 0
// under a stable descending sort (ties: later candidates first, as argsort(kind="stable")[::-1] orders them).
template <typename T>
__global__ void __launch_bounds__(256) candidate_rank_kernel(const T* __restrict__ U, int ldu, const T* __restrict__ E, int lde, int d,
                                                             const int32_t* __restrict__ cand, int C, int B, float* __restrict__ scores,
                                                             int32_t* __restrict__ rank) {
    pdl_prologue();
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (b >= B) return;
    float s0 = 0.f;
    int r = 0;
    for (int c = 0; c < C; ++c) {
        const T* e = E + (size_t)cand[(size_t)b * C + c] * lde;
        float p = 0.f;
        for (int k = lane; k < d; k += 32) p = fmaf(to_f(U[(size_t)b * ldu + k]), to_f(e[k]), p);
        p = warp_sum(p);
        if (c == 0) s0 = p;
        else r += (p >= s0) ? 1 : 0;
        if (scores && lane == 0) scores[(size_t)b * C + c] = p;
    }
    if (lane == 0) rank[b] = r;
}

// ---------------------------------------------------------------------------------------------------
// top-K
__device__ __forceinline__ bool better(float v, int i, float tv, int ti) { return v > tv || (v == tv && i > ti); }

// One warp per score row.  The list (sv, si) lives in shared memory sorted best-first.
__device__ __noinline__ void topk_insert(float* sv, int* si, int K, float cv, int ci, int lane) {
    int cnt = 0;
    for (int e = lane; e < K; e += 32) cnt += better(sv[e], si[e], cv, ci) ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    const int pos = cnt;
    if (pos >= K) return;
    float tv[4]; int ti[4];  // K <= 128
    int n = 0;
    for (int e = lane; e < K - 1; e += 32, ++n) { tv[n] = sv[e]; ti[n] = si[e]; }
    __syncwarp();
    n = 0;
    for (int e = lane; e < K - 1; e += 32, ++n)
        if (e >= pos) { sv[e + 1] = tv[n]; si[e + 1] = ti[n]; }
    if (lane == 0) { sv[pos] = cv; si[pos] = ci; }
    __syncwarp();
}

// Warp-level running top-K under the total order (score desc, index desc).  K <= 32: the list lives in registers, one
// entry per lane, sorted best-first -- an insertion is a ballot, a popcount and two shuffles.  K <= 128: sorted list in
// shared memory (topk_insert).  offer() is warp-uniform: every lane offers one (value, id); id < 0 = nothing to offer.
// (thr_v, thr_i) is the admission threshold: only elements better than it are looked at.  It never decreases; besides the
// list's own K-th entry it can be raised from outside (raise()) by any pair known to have K elements at or above it.
struct WarpTopK {
    float lv; int li;            // register list (K <= 32): lane l holds the l-th best
    float* sv; int* si;          // shared-memory list (K > 32)
    float thr_v; int thr_i;
    int K, lane;
    bool in_regs, improved;
    __device__ __forceinline__ void init(int K_, int lane_, float* sv_, int* si_) {
        K = K_; lane = lane_; sv = sv_; si = si_; in_regs = K_ <= 32; improved = false;
        lv = -INFINITY; li = -1; thr_v = -INFINITY; thr_i = -1;
        if (!in_regs) { for (int e = lane; e < K; e += 32) { sv[e] = -INFINITY; si[e] = -1; } __syncwarp(); }
    }
    __device__ __forceinline__ void raise(float v, int i) {
        if (better(v, i, thr_v, thr_i)) { thr_v = v; thr_i = i; }
    }
    __device__ __forceinline__ void insert(float cv, int ci) {      // warp-uniform (cv, ci)
        float kv; int ki;
        if (in_regs) {
            const int pos = __popc(__ballot_sync(0xffffffffu, better(lv, li, cv, ci)));    // entries ahead of the candidate
            if (pos >= K) return;
            const float uv = __shfl_up_sync(0xffffffffu, lv, 1);
            const int ui = __shfl_up_sync(0xffffffffu, li, 1);
            if (lane == pos) { lv = cv; li = ci; }
            else if (lane > pos) { lv = uv; li = ui; }
            if (lane >= K) { lv = -INFINITY; li = -1; }
            kv = __shfl_sync(0xffffffffu, lv, K - 1);
            ki = __shfl_sync(0xffffffffu, li, K - 1);
        } else {
            topk_insert(sv, si, K, cv, ci, lane);
            kv = sv[K - 1];
            ki = si[K - 1];
        }
        if (better(kv, ki, thr_v, thr_i)) { thr_v = kv; thr_i = ki; improved = true; }
    }
    __device__ __forceinline__ void offer(float v, int gi) {
        unsigned bal = __ballot_sync(0xffffffffu, gi >= 0 && better(v, gi, thr_v, thr_i));
        while (bal) {
            const int src = __ffs(bal) - 1;
            bal &= bal - 1;
            const float cv = __shfl_sync(0xffffffffu, v, src);
            const int ci = __shfl_sync(0xffffffffu, gi, src);
            if (better(cv, ci, thr_v, thr_i)) insert(cv, ci);
        }
    }
    __device__ __forceinline__ void store(float* ov, int32_t* oi) {
        if (in_regs) { if (lane < K) { ov[lane] = lv; oi[lane] = li; } }
        else { __syncwarp(); for (int e = lane; e < K; e += 32) { ov[e] = sv[e]; oi[e] = si[e]; } }
    }
};

constexpr int kTopkWarps = 4;
constexpr int kMaxK = 128;
constexpr int kTopkSeg = 8;          // 512-byte row segments per trip of the scan (and as many again in flight)

// One warp per (score row, column chunk): seen-item masking + top-K of the chunk under the total order
// (score desc, index desc); the per-chunk lists of a row are then reduced by topk_merge_kernel.
// What the scan costs is set by how often a trip (4 KB = 1024 scores) holds a candidate, i.e. a score at or above the
// list's current K-th best: after n scores that happens with probability ~min(1, 1024 K / n), so the threshold only does
// its job once a warp has seen a few hundred K scores.  Hence LONG chunks (>= 64k scores when the launch has enough rows,
// see topk_chunks) on FEW warps per SM, and memory latency is covered by depth instead of occupancy: 16-byte loads, eight
// segments in registers and the next eight in flight per warp (~100 registers).  Fast path per trip: the lane's maximum of
// its 32 scores against the threshold and one vote.  Candidates are taken straight from the registers: a ballot per
// segment finds the lanes, four shuffles bring the lane's scores to the whole warp, insertion is warp-uniform.
// The first trip doubles as a probe: the K-th largest of the 32 per-lane maxima has K scores at or above it, so it is a
// valid threshold before the first insertion (about rank 40 of the trip's 1024 scores: most of the warm-up is skipped).
// FILTER: row r may only return items whose bit is set in allow[allow_of_row[r]] (-1: unrestricted).  The allow bits of a
// trip's scores are fetched with the scores and applied when the trip is consumed (a disallowed score becomes -inf), so the
// scan keeps its single read of S and its loads in flight; entries left at -inf are written with id -1.
template <bool FILTER>
__global__ void __launch_bounds__(kTopkWarps * 32) mask_topk_kernel(float* __restrict__ S, int64_t lds, int n_rows, int N,
                                                                    int item_offset, const int64_t* __restrict__ indptr,
                                                                    const int32_t* __restrict__ indices,
                                                                    const int32_t* __restrict__ rows, int exclude_seen, int K,
                                                                    int n_chunks, int chunk_len, float* __restrict__ out_val,
                                                                    int32_t* __restrict__ out_idx, const uint32_t* __restrict__ allow,
                                                                    int64_t allow_stride, const int32_t* __restrict__ allow_of_row) {
    pdl_prologue();
    __shared__ float sv_all[kTopkWarps][kMaxK];
    __shared__ int si_all[kTopkWarps][kMaxK];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t unit = (int64_t)blockIdx.x * kTopkWarps + warp;
    if (unit >= (int64_t)n_rows * n_chunks) return;
    const int r = (int)(unit / n_chunks), ch = (int)(unit - (int64_t)r * n_chunks);
    const int c0 = ch * chunk_len, c1 = min(N, c0 + chunk_len);
    float* row = S + (size_t)r * lds;
    if (exclude_seen) {
        const int u = rows ? rows[r] : r;
        for (int64_t j = indptr[u] + lane; j < indptr[u + 1]; j += 32) {
            const int c = indices[j] - item_offset;
            if (c >= c0 && c < c1) row[c] = -INFINITY;
        }
    }
    __syncwarp();
    WarpTopK top;
    top.init(K, lane, sv_all[warp], si_all[warp]);
    // [c0, cs): up to 3 scores before the first 16-byte boundary of the row (row strides need not be multiples of 4);
    // [cs, c1v): the vector body; [c1v, c1): up to 3 tail scores
    const int head = min(c1 - c0, (int)((4 - ((reinterpret_cast<uintptr_t>(row + c0) >> 2) & 3)) & 3));
    const int cs = c0 + head;
    const int c1v = cs + ((c1 - cs) / 4) * 4;
    const float4 ninf = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    auto fetch = [&](int base) { const int c = base + lane * 4; return (base < c1v && c < c1v) ? *reinterpret_cast<const float4*>(row + c) : ninf; };
    const uint32_t* arow = nullptr;
    if constexpr (FILTER) {
        const int f = allow_of_row[r];
        if (f >= 0) arow = allow + (size_t)f * allow_stride;
    }
    auto allowed = [&](int c) { const int g = item_offset + c; return !arow || ((__ldg(arow + (g >> 5)) >> (g & 31)) & 1u); };
    // allow bits of the 4 scores of each segment of a trip, packed 4 per segment (all set when unrestricted)
    auto fetch_allow = [&](int base) {
        uint32_t m = 0xFFFFFFFFu;
        if (arow) {
            m = 0;
#pragma unroll
            for (int q = 0; q < kTopkSeg; ++q) {
                const int c = base + q * 128 + lane * 4, g = item_offset + c;
                if (base < c1v && c < c1v) {     // g + 3 < item_offset + N: the second word exists whenever it is needed
                    const uint32_t lo = __ldg(arow + (g >> 5)), hi = (g & 31) > 28 ? __ldg(arow + (g >> 5) + 1) : 0u;
                    m |= (__funnelshift_r(lo, hi, g & 31) & 0xFu) << (4 * q);
                }
            }
        }
        return m;
    };
    float4 cur[kTopkSeg], nxt[kTopkSeg];
    uint32_t cur_allow = 0, nxt_allow = 0;
#pragma unroll
    for (int q = 0; q < kTopkSeg; ++q) cur[q] = fetch(cs + q * 128);
    if constexpr (FILTER) cur_allow = fetch_allow(cs);
    {
        const bool h = lane < head && (!FILTER || allowed(c0 + lane));
        top.offer(h ? row[c0 + lane] : -INFINITY, h ? item_offset + c0 + lane : -1);
    }
    bool probe = K <= 32 && c1v - cs >= kTopkSeg * 128;
    for (int base = cs; base < c1v; base += kTopkSeg * 128) {
#pragma unroll
        for (int q = 0; q < kTopkSeg; ++q) nxt[q] = fetch(base + kTopkSeg * 128 + q * 128);
        if constexpr (FILTER) {
            nxt_allow = fetch_allow(base + kTopkSeg * 128);
#pragma unroll
            for (int q = 0; q < kTopkSeg; ++q) {
                if (!((cur_allow >> (4 * q)) & 1u)) cur[q].x = -INFINITY;
                if (!((cur_allow >> (4 * q + 1)) & 1u)) cur[q].y = -INFINITY;
                if (!((cur_allow >> (4 * q + 2)) & 1u)) cur[q].z = -INFINITY;
                if (!((cur_allow >> (4 * q + 3)) & 1u)) cur[q].w = -INFINITY;
            }
        }
        float mq[kTopkSeg];
#pragma unroll
        for (int q = 0; q < kTopkSeg; ++q) mq[q] = fmaxf(fmaxf(cur[q].x, cur[q].y), fmaxf(cur[q].z, cur[q].w));
        float m = mq[0];
#pragma unroll
        for (int q = 1; q < kTopkSeg; ++q) m = fmaxf(m, mq[q]);
        if (probe) {        // first trip (all 1024 scores in range): seed the threshold from the lane maxima
            probe = false;
            int mi = -1;    // id of this lane's maximum (largest id among equals: the better pair)
#pragma unroll
            for (int q = 0; q < kTopkSeg; ++q) {
                const int g = item_offset + base + q * 128 + lane * 4;
                if (cur[q].x == m) mi = g;
                if (cur[q].y == m) mi = g + 1;
                if (cur[q].z == m) mi = g + 2;
                if (cur[q].w == m) mi = g + 3;
            }
            int rank = 0;   // lanes holding a better pair (ids are distinct: a strict order)
#pragma unroll
            for (int o = 0; o < 32; ++o) rank += better(__shfl_sync(0xffffffffu, m, o), __shfl_sync(0xffffffffu, mi, o), m, mi) ? 1 : 0;
            const int src = __ffs(__ballot_sync(0xffffffffu, rank == K - 1)) - 1;
            if (src >= 0) top.raise(__shfl_sync(0xffffffffu, m, src), __shfl_sync(0xffffffffu, mi, src) - 1);   // "- 1": that pair itself is admitted
        }
        if (__any_sync(0xffffffffu, m >= top.thr_v)) {
#pragma unroll
            for (int q = 0; q < kTopkSeg; ++q) {
                const int c = base + q * 128 + lane * 4;
                unsigned bal = __ballot_sync(0xffffffffu, c < c1v && mq[q] >= top.thr_v);
                while (bal) {
                    const int src = __ffs(bal) - 1;
                    bal &= bal - 1;
                    const int g = item_offset + base + q * 128 + src * 4;
                    const float x = __shfl_sync(0xffffffffu, cur[q].x, src), y = __shfl_sync(0xffffffffu, cur[q].y, src);
                    const float z = __shfl_sync(0xffffffffu, cur[q].z, src), w = __shfl_sync(0xffffffffu, cur[q].w, src);
                    if (better(x, g, top.thr_v, top.thr_i)) top.insert(x, g);
                    if (better(y, g + 1, top.thr_v, top.thr_i)) top.insert(y, g + 1);
                    if (better(z, g + 2, top.thr_v, top.thr_i)) top.insert(z, g + 2);
                    if (better(w, g + 3, top.thr_v, top.thr_i)) top.insert(w, g + 3);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < kTopkSeg; ++q) cur[q] = nxt[q];
        if constexpr (FILTER) cur_allow = nxt_allow;
    }
    {   // <= 3 tail columns
        const int c = c1v + lane;
        const bool t = c < c1 && (!FILTER || allowed(c));
        top.offer(t ? row[c] : -INFINITY, t ? item_offset + c : -1);
    }
    float* ov = out_val + ((size_t)r * n_chunks + ch) * K;
    int32_t* oi = out_idx + ((size_t)r * n_chunks + ch) * K;
    top.store(ov, oi);
    if constexpr (FILTER) {      // (each lane rereads the slots it wrote)
        for (int e = lane; e < K; e += 32)
            if (ov[e] == -INFINITY) oi[e] = -1;
    }
}

// Merge G candidate lists per row (item-sharded evaluation, SURVEY.md §8e) -> top K.  Candidate j of row r sits at
// g * group_stride + r * group_len + (j - g * group_len), g = j / group_len: one [n_rows, GK] array (n_groups = 1, group_len = GK)
// or the blocks of an all-gather ([rank][n_rows][K]: group_len = K, group_stride = the per-rank block), read in place.
__global__ void __launch_bounds__(kTopkWarps * 32) topk_merge_kernel(const float* __restrict__ cval, const int32_t* __restrict__ cidx,
                                                                     int n_rows, int n_groups, int group_len, int64_t group_stride,
                                                                     int K, float* __restrict__ out_val,
                                                                     int32_t* __restrict__ out_idx) {
    pdl_prologue();
    __shared__ float sv_all[kTopkWarps][kMaxK];
    __shared__ int si_all[kTopkWarps][kMaxK];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * kTopkWarps + warp;
    if (r >= n_rows) return;
    WarpTopK top;
    top.init(K, lane, sv_all[warp], si_all[warp]);
    const int GK = n_groups * group_len;
    const float* cv = cval + (size_t)r * group_len;
    const int32_t* ci = cidx + (size_t)r * group_len;
    for (int base = 0; base < GK; base += 128) {       // four candidates per lane in flight
        float v[4]; int id[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = base + q * 32 + lane;
            const int g = j / group_len;
            const int64_t off = (int64_t)g * group_stride + (j - g * group_len);
            v[q] = j < GK ? cv[off] : -INFINITY;
            id[q] = j < GK ? ci[off] : -1;
        }
        const float tv = top.thr_v;
        if (!__any_sync(0xffffffffu, v[0] >= tv || v[1] >= tv || v[2] >= tv || v[3] >= tv)) continue;
#pragma unroll
        for (int q = 0; q < 4; ++q) top.offer(v[q], id[q]);
    }
    top.store(out_val + (size_t)r * K, out_idx + (size_t)r * K);
}

// hit mask: bit p of mask[r] (4 x u32 per row) is set iff topk[r][p] is one of the row's relevant items.
__global__ void hit_mask_kernel(const int32_t* __restrict__ topk, int n_rows, int K, const int64_t* __restrict__ rel_ptr,
                                const int32_t* __restrict__ rel_idx, uint32_t* __restrict__ mask) {
    pdl_prologue();
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= n_rows) return;
    const int64_t s = rel_ptr[r], e = rel_ptr[r + 1];
    for (int w = 0; w < 4; ++w) {
        const int p = w * 32 + lane;
        bool hit = false;
        if (p < K) {
            const int it = topk[(size_t)r * K + p];
            for (int64_t j = s; j < e; ++j) hit |= (rel_idx[j] == it);
        }
        const unsigned b = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) mask[(size_t)r * 4 + w] = b;
    }
}

// Per-row Recall/NDCG/HR for up to 8 cut-offs, summed in double in a fixed order.
// disc[p] = 1/log2(p+2), idcg[n] = sum_{i<n} disc[i] (host-computed in float64 with numpy, as the reference does).
// sums: [gridDim.x][nk*3 + 1] doubles (last = evaluated-row count); reduce with a second launch (n_rows = -gridDim).
__global__ void __launch_bounds__(256) metrics_partial_kernel(const uint32_t* __restrict__ mask, const int64_t* __restrict__ rel_ptr,
                                                              int n_rows, const int32_t* __restrict__ kvals, int nk,
                                                              const double* __restrict__ disc, const double* __restrict__ idcg,
                                                              double* __restrict__ sums) {
    pdl_prologue();
    __shared__ double red[8][25];
    double acc[25];
    for (int i = 0; i < 25; ++i) acc[i] = 0.0;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += gridDim.x * blockDim.x) {
        const int nrel = (int)(rel_ptr[r + 1] - rel_ptr[r]);
        if (nrel == 0) continue;
        acc[nk * 3] += 1.0;
        uint32_t m[4] = {mask[(size_t)r * 4], mask[(size_t)r * 4 + 1], mask[(size_t)r * 4 + 2], mask[(size_t)r * 4 + 3]};
        for (int q = 0; q < nk; ++q) {
            const int k = kvals[q];
            int hits = 0;
            double dcg = 0.0;
            for (int p = 0; p < k; ++p)
                if ((m[p >> 5] >> (p & 31)) & 1u) { ++hits; dcg += disc[p]; }
            acc[q * 3 + 0] += (double)hits / (double)nrel;
            acc[q * 3 + 1] += dcg / idcg[min(nrel, k)];
            acc[q * 3 + 2] += hits > 0 ? 1.0 : 0.0;
        }
    }
    const int nv = nk * 3 + 1, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = 0; i < nv; ++i) {
        double v = acc[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < nv) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        sums[(size_t)blockIdx.x * nv + threadIdx.x] = v;
    }
}

__global__ void metrics_final_kernel(const double* __restrict__ partial, int nblocks, int nv, double* __restrict__ out) {
    pdl_prologue();
    const int i = threadIdx.x;
    if (i >= nv) return;
    double v = 0.0;
    for (int b = 0; b < nblocks; ++b) v += partial[(size_t)b * nv + i];
    out[i] = v;
}

}  // namespace hvae

using namespace hvae;

extern "C" {

int hvae_row_lse(const float* S, int64_t lds, int rows, int N, float* lse, void* stream) {
    if (rows == 0) return 0;
    launch_pdl(row_lse_kernel, rows, 256, 0, (cudaStream_t)stream, S, lds, N, lse);
    HVAE_LAUNCH_CHECK("row_lse");
    return 0;
}

int hvae_row_softmax_scale(float* S, int64_t lds, int rows, int N, const float* lse, const float* xsum, const float* inv_bg,
                           void* stream) {
    if (rows == 0) return 0;
    const int64_t total = (int64_t)rows * N;
    launch_pdl(row_softmax_scale_kernel, (unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream, S, lds, rows, N, lse, xsum, inv_bg);
    HVAE_LAUNCH_CHECK("row_softmax_scale");
    return 0;
}

int hvae_sparse_dot_xsum(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                         const void* U, int ldu, const void* E, int lde, int d, int is_bf16, float* dot, float* xsum, void* stream) {
    if (B == 0) return 0;
    if (is_bf16 && ldu % 8 == 0 && lde % 8 == 0 && d <= 1024)
        launch_pdl(sparse_dot_xsum_bf16_kernel, ceil_div(B, 8), 256, 0, (cudaStream_t)stream, 
            indptr, indices, values, rows, B, (const __nv_bfloat16*)U, ldu, (const __nv_bfloat16*)E, lde, ceil_div(d, 8), dot, xsum);
    else if (is_bf16)
        launch_pdl(sparse_dot_xsum_kernel<__nv_bfloat16>, ceil_div(B, 8), 256, 0, (cudaStream_t)stream, 
            indptr, indices, values, rows, B, (const __nv_bfloat16*)U, ldu, (const __nv_bfloat16*)E, lde, d, dot, xsum);
    else
        launch_pdl(sparse_dot_xsum_kernel<float>, ceil_div(B, 8), 256, 0, (cudaStream_t)stream, indptr, indices, values, rows, B, (const float*)U,
                                                                                       ldu, (const float*)E, lde, d, dot, xsum);
    HVAE_LAUNCH_CHECK("sparse_dot_xsum");
    return 0;
}

static int du_finalize_launch(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B, const float* O,
                              int ldo, int n_parts, const float* oscale, const float* w_part, const void* E, int lde, int d, int is_bf16,
                              const float* inv_bg, float* dU, int lddu, const float* c_part, const float* l_part, int n_sub, float* lse,
                              void* stream) {
    if (B == 0) return 0;
    HVAE_REQUIRE(lddu % 4 == 0 && ldo % 4 == 0 && (!is_bf16 || lde % 8 == 0), "du_finalize: leading dimensions must be multiples of 4 (bf16 E: 8)");
    const int nb = ceil_div(B * (lddu / 4), 256);
    if (is_bf16)
        launch_pdl(du_finalize_kernel<__nv_bfloat16>, nb, 256, 0, (cudaStream_t)stream, indptr, indices, values, rows, B, O, ldo, n_parts, oscale,
                   w_part, (const __nv_bfloat16*)E, lde, d, inv_bg, dU, lddu, c_part, l_part, n_sub, lse);
    else
        launch_pdl(du_finalize_kernel<float>, nb, 256, 0, (cudaStream_t)stream, indptr, indices, values, rows, B, O, ldo, n_parts, oscale,
                   w_part, (const float*)E, lde, d, inv_bg, dU, lddu, c_part, l_part, n_sub, lse);
    HVAE_LAUNCH_CHECK("du_finalize");
    return 0;
}

int hvae_du_finalize(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B, const float* O,
                     int ldo, int n_parts, const float* oscale, const float* w_part, const void* E, int lde, int d, int is_bf16,
                     const float* inv_bg, float* dU, int lddu, void* stream) {
    return du_finalize_launch(indptr, indices, values, rows, B, O, ldo, n_parts, oscale, w_part, E, lde, d, is_bf16, inv_bg, dU, lddu, nullptr,
                              nullptr, 0, nullptr, stream);
}

// The same after the one-pass scoring kernel, with hvae_tc_onepass_combine folded in: the weights of the O partial sums come
// straight from the kernel's per-split shifts c_part [n_parts, B] and numerator sums l_part [n_parts, n_sub, B]; lse [B] is written too.
int hvae_du_finalize_onepass(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B, const float* O,
                             int ldo, int n_parts, const float* oscale, const float* c_part, const float* l_part, int n_sub, float* lse,
                             const void* E, int lde, int d, int is_bf16, const float* inv_bg, float* dU, int lddu, void* stream) {
    HVAE_REQUIRE(c_part && l_part && n_sub >= 1, "du_finalize_onepass: the one-pass kernel's partial results are required");
    return du_finalize_launch(indptr, indices, values, rows, B, O, ldo, n_parts, oscale, nullptr, E, lde, d, is_bf16, inv_bg, dU, lddu, c_part,
                              l_part, n_sub, lse, stream);
}

int hvae_candidate_rank(const void* U, int ldu, const void* E, int lde, int d, int is_bf16, const int32_t* cand, int C, int B,
                        float* scores, int32_t* rank, void* stream) {
    if (B == 0) return 0;
    HVAE_REQUIRE(C >= 1, "candidate_rank: need at least the test item");
    if (is_bf16)
        launch_pdl(candidate_rank_kernel<__nv_bfloat16>, ceil_div(B, 8), 256, 0, (cudaStream_t)stream, (const __nv_bfloat16*)U, ldu, (const __nv_bfloat16*)E,
                                                                                               lde, d, cand, C, B, scores, rank);
    else
        launch_pdl(candidate_rank_kernel<float>, ceil_div(B, 8), 256, 0, (cudaStream_t)stream, (const float*)U, ldu, (const float*)E, lde, d, cand, C, B,
                                                                                       scores, rank);
    HVAE_LAUNCH_CHECK("candidate_rank");
    return 0;
}

// Column chunks per row.  Long chunks keep the scan on its fast path (see mask_topk_kernel), so a row is only cut when the
// launch would otherwise have fewer warps than ~12 per SM, and never below 16k scores per chunk; multiples of 1024.
static void topk_chunks(int n_rows, int N, int* n_chunks, int* chunk_len) {
    const int want_warps = 12 * kNumSMs;      // measured best at 256 x 1M (6: 63 %, 10: 71 %, 12: 72 %, 16: 51 % of HBM peak)
    int nc = max(1, ceil_div(want_warps, max(1, n_rows)));
    nc = max(1, min(nc, N / 16384));
    const int len = round_up(ceil_div(N, nc), 1024);
    *chunk_len = len;
    *n_chunks = max(1, ceil_div(N, len));
}

size_t hvae_mask_topk_chunks(int n_rows, int N) {
    int nc, len;
    topk_chunks(n_rows, N, &nc, &len);
    return (size_t)nc;
}

static int mask_topk(float* S, int64_t lds, int n_rows, int N, int item_offset, const int64_t* indptr, const int32_t* indices,
                     const int32_t* rows, int exclude_seen, const uint32_t* allow, int64_t allow_stride, const int32_t* allow_of_row,
                     int K, float* cand_val, int32_t* cand_idx, float* out_val, int32_t* out_idx, void* stream) {
    HVAE_REQUIRE(K >= 1 && K <= kMaxK, "mask_topk: K=%d outside [1,%d]", K, kMaxK);
    if (n_rows == 0) return 0;
    int nc, len;
    topk_chunks(n_rows, N, &nc, &len);
    HVAE_REQUIRE(nc == 1 || (cand_val && cand_idx), "mask_topk: %d column chunks need candidate scratch", nc);
    const int64_t units = (int64_t)n_rows * nc;
    float* cv = nc == 1 ? out_val : cand_val;
    int32_t* ci = nc == 1 ? out_idx : cand_idx;
    const unsigned blocks = (unsigned)((units + kTopkWarps - 1) / kTopkWarps);
    if (allow)
        launch_pdl(mask_topk_kernel<true>, blocks, kTopkWarps * 32, 0, (cudaStream_t)stream, S, lds, n_rows, N, item_offset, indptr, indices,
                   rows, exclude_seen, K, nc, len, cv, ci, allow, allow_stride, allow_of_row);
    else
        launch_pdl(mask_topk_kernel<false>, blocks, kTopkWarps * 32, 0, (cudaStream_t)stream, S, lds, n_rows, N, item_offset, indptr, indices,
                   rows, exclude_seen, K, nc, len, cv, ci, (const uint32_t*)nullptr, (int64_t)0, (const int32_t*)nullptr);
    HVAE_LAUNCH_CHECK(allow ? "mask_topk_filtered" : "mask_topk");
    if (nc > 1) {
        launch_pdl(topk_merge_kernel, ceil_div(n_rows, kTopkWarps), kTopkWarps * 32, 0, (cudaStream_t)stream, (const float*)cv,
                   (const int32_t*)ci, n_rows, 1, nc * K, (int64_t)0, K, out_val, out_idx);
        HVAE_LAUNCH_CHECK("mask_topk merge");
    }
    return 0;
}

// scratch cand_val / cand_idx: [n_rows, hvae_mask_topk_chunks(n_rows, N) * K] (may be NULL when that is 1)
int hvae_mask_topk(float* S, int64_t lds, int n_rows, int N, int item_offset, const int64_t* indptr, const int32_t* indices,
                   const int32_t* rows, int exclude_seen, int K, float* cand_val, int32_t* cand_idx, float* out_val, int32_t* out_idx,
                   void* stream) {
    return mask_topk(S, lds, n_rows, N, item_offset, indptr, indices, rows, exclude_seen, nullptr, 0, nullptr, K, cand_val, cand_idx,
                     out_val, out_idx, stream);
}

// The same restricted to per-row allow-sets (bitmaps over global item ids, see hvae_tc_score_topk_filtered); allow == NULL is
// hvae_mask_topk.  Slots a row cannot fill hold (-inf, -1).
int hvae_mask_topk_filtered(float* S, int64_t lds, int n_rows, int N, int item_offset, const int64_t* indptr, const int32_t* indices,
                            const int32_t* rows, int exclude_seen, const uint32_t* allow, int64_t allow_stride_words,
                            const int32_t* allow_of_row, int K, float* cand_val, int32_t* cand_idx, float* out_val, int32_t* out_idx,
                            void* stream) {
    if (allow) {
        HVAE_REQUIRE(allow_of_row, "mask_topk_filtered: allow needs allow_of_row");
        HVAE_REQUIRE(item_offset >= 0 && allow_stride_words >= ((int64_t)item_offset + N + 31) / 32,
                     "mask_topk_filtered: allow_stride_words=%lld does not cover items up to %lld", (long long)allow_stride_words,
                     (long long)item_offset + N);
    }
    return mask_topk(S, lds, n_rows, N, item_offset, indptr, indices, rows, exclude_seen, allow, allow_stride_words, allow_of_row, K,
                     cand_val, cand_idx, out_val, out_idx, stream);
}

int hvae_topk_merge(const float* cval, const int32_t* cidx, int n_rows, int GK, int K, float* out_val, int32_t* out_idx, void* stream) {
    HVAE_REQUIRE(K >= 1 && K <= kMaxK, "topk_merge: K=%d outside [1,%d]", K, kMaxK);
    if (n_rows == 0) return 0;
    launch_pdl(topk_merge_kernel, ceil_div(n_rows, kTopkWarps), kTopkWarps * 32, 0, (cudaStream_t)stream, cval, cidx, n_rows, 1, GK, (int64_t)0, K,
               out_val, out_idx);
    HVAE_LAUNCH_CHECK("topk_merge");
    return 0;
}

// The same merge over the blocks of an all-gather read in place: rank g's K candidates of row r at cval/cidx[g * group_stride + r * K].
int hvae_topk_merge_groups(const float* cval, const int32_t* cidx, int n_rows, int n_groups, int64_t group_stride, int K, float* out_val,
                           int32_t* out_idx, void* stream) {
    HVAE_REQUIRE(K >= 1 && K <= kMaxK && n_groups >= 1, "topk_merge_groups: K=%d outside [1,%d] or no groups", K, kMaxK);
    if (n_rows == 0) return 0;
    launch_pdl(topk_merge_kernel, ceil_div(n_rows, kTopkWarps), kTopkWarps * 32, 0, (cudaStream_t)stream, cval, cidx, n_rows, n_groups, K,
               group_stride, K, out_val, out_idx);
    HVAE_LAUNCH_CHECK("topk_merge_groups");
    return 0;
}

int hvae_hit_mask(const int32_t* topk, int n_rows, int K, const int64_t* rel_ptr, const int32_t* rel_idx, uint32_t* mask, void* stream) {
    HVAE_REQUIRE(K >= 1 && K <= kMaxK, "hit_mask: K=%d outside [1,%d]", K, kMaxK);
    if (n_rows == 0) return 0;
    launch_pdl(hit_mask_kernel, ceil_div(n_rows, 8), 256, 0, (cudaStream_t)stream, topk, n_rows, K, rel_ptr, rel_idx, mask);
    HVAE_LAUNCH_CHECK("hit_mask");
    return 0;
}

// out: nk*3+1 doubles = per cut-off {recall, ndcg, hit} sums, then the evaluated-row count.  workspace >= 148*(nk*3+1) doubles.
int hvae_metrics_reduce(const uint32_t* mask, const int64_t* rel_ptr, int n_rows, const int32_t* kvals, int nk, const double* disc,
                        const double* idcg, double* workspace, double* out, void* stream) {
    HVAE_REQUIRE(nk >= 1 && nk <= 8, "metrics_reduce: nk=%d outside [1,8]", nk);
    const int blocks = max(1, min(kNumSMs, ceil_div(n_rows, 256)));
    launch_pdl(metrics_partial_kernel, blocks, 256, 0, (cudaStream_t)stream, mask, rel_ptr, n_rows, kvals, nk, disc, idcg, workspace);
    launch_pdl(metrics_final_kernel, 1, 32, 0, (cudaStream_t)stream, workspace, blocks, nk * 3 + 1, out);
    HVAE_LAUNCH_CHECK("metrics_reduce");
    return 0;
}

}  // extern "C"

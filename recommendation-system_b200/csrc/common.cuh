// Shared device helpers for the hvae_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// Records a message retrievable through hvae_last_error() and returns a non-zero status.
int hvae_fail(const char* fmt, ...);

#define HVAE_LAUNCH_CHECK(what)                                                       \
    do {                                                                              \
        cudaError_t _e = cudaGetLastError();                                          \
        if (_e != cudaSuccess) return hvae_fail("%s: %s", what, cudaGetErrorString(_e)); \
    } while (0)

#define HVAE_REQUIRE(cond, ...)                    \
    do {                                           \
        if (!(cond)) return hvae_fail(__VA_ARGS__); \
    } while (0)

#define HVAE_CUDA(call)                                                                   \
    do {                                                                                  \
        cudaError_t _e = (call);                                                          \
        if (_e != cudaSuccess) return hvae_fail("%s: %s", #call, cudaGetErrorString(_e)); \
    } while (0)

namespace hvae {

constexpr int kNumSMs = 148;

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------
// Every kernel of the library is launched with the programmatic-stream-serialization attribute and starts with
// pdl_prologue(): "my dependents may start launching" + "wait until the kernel(s) before me have completed and flushed".
// Inside a captured step this overlaps the launch latency / prologue of kernel N+1 with the execution of kernel N (the
// tensor-core kernels do their barrier init, TMEM allocation and descriptor prefetch before the wait).  Without the
// attribute both instructions are no-ops.  HVAE_NO_PDL=1 disables the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() { pdl_launch_dependents(); pdl_wait(); }

bool pdl_enabled();   // capi.cu

template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// exact-erf GELU and its derivative (nn.GELU() default, reference src/ml/model.py:92,116)
__device__ __forceinline__ float gelu(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_grad(float x) {
    const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
    const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
    return cdf + x * pdf;
}

// ---- counter-based random numbers (Philox4x32-10): counter {ctr_lo, ctr_hi, stream_id, 0}, key {seed_lo, seed_hi} ----
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    c[1] = (uint32_t)p1; c[3] = (uint32_t)p0; c[0] = n0; c[2] = n2;
}
__device__ __forceinline__ void philox(uint64_t seed, uint64_t ctr, uint32_t stream_id, uint32_t (&out)[4]) {
    uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), stream_id, 0u};
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) { philox_round(c, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

// ---- Gumbel-top-K sampling of the top-K kernels (include/hvae_b200.h, hvae_tc_score_topk_sampled) ----
// Item gi of a row with seed s draws word gi & 3 of philox(s, gi >> 2, kSampleStream): the noise depends on (seed, global
// item id) only, never on the batch row, the item split, the shard or K.
constexpr uint32_t kSampleStream = 0x53414D50u;   // "SAMP"
// Above every Gumbel value gumbel_of() can return: the largest uniform, 1 - 2^-24, gives -log(-log(u)) = 16.63553 exactly, and
// the two 1-ulp logf evaluations move that by less than 1e-5.  The top-K kernels admit a column only if
// fmaf(s, inv_tau, kGumbelMax) >= threshold, which every key fmaf(s, inv_tau, g) at or above the threshold passes.
constexpr float kGumbelMax = 16.64f;
// u = ((r >> 9) + 0.5) 2^-23 is exact in fp32 and lies in [2^-24, 1 - 2^-24], so both logarithms are finite.
__device__ __forceinline__ float gumbel_of(uint32_t r) {
    const float u = ((float)(r >> 9) + 0.5f) * 1.1920928955078125e-7f;
    return -logf(-logf(u));
}
__device__ __forceinline__ uint32_t pick4(const uint32_t (&w)[4], int k) {
    return k == 0 ? w[0] : k == 1 ? w[1] : k == 2 ? w[2] : w[3];
}

// ---- Boosted top-K (include/hvae_b200.h, hvae_tc_score_topk_boosted): score thresholds for exact pruning ----
// A boosted row ranks k = fmaf(w, beta_i, s) (and, sampled, fmaf(k, inv_tau, g)).  The kernels compare each score s with one
// threshold per group of columns, the list threshold thr carried back through the key's roundings.  With round() the fp32
// rounding to nearest, which is monotone, and pred(T) the float below T: round(x) >= T implies x > pred(T) (an x <= pred(T)
// rounds to at most pred(T)).  The derivations start from key >= thr, so a key that ties the threshold (and may win on its id)
// passes; the result of sample_threshold is a bound on k, fed to boost_threshold as T for a row that is both.
// sample_threshold: key = round(k*a + g) >= thr, g <= kGumbelMax, a = inv_tau > 0
//     => k*a > pred(thr) - kGumbelMax >= D = fsub_rd(pred(thr), kGumbelMax)  =>  k > D/a >= fdiv_rd(D, a).
// boost_threshold: k = round(s + w*beta_i) >= T, w*beta_i <= bplus (bplus rounded up from w * the block max, or w * the
// block min when w < 0)  =>  s + bplus > pred(T)  =>  s > pred(T) - bplus >= fsub_rd(pred(T), bplus).
// thr = -inf gives -inf in both (every column passes).  A column below the result can never enter the list; the list itself
// is then updated with the exactly computed key, so the result only decides how much arithmetic runs.
__device__ __forceinline__ float sample_threshold(float thr, float inv_tau) {
    return __fdiv_rd(__fsub_rd(nextafterf(thr, -INFINITY), kGumbelMax), inv_tau);
}
__device__ __forceinline__ float boost_threshold(float T, float bplus) { return __fsub_rd(nextafterf(T, -INFINITY), bplus); }
// bplus of the columns in blocks with extremes e0, e1 (block maxima when w >= 0, minima when w < 0; e0 == e1 for one block)
__device__ __forceinline__ float boost_bplus(float w, float e0, float e1) {
    return __fmul_ru(w, w >= 0.f ? fmaxf(e0, e1) : fminf(e0, e1));
}
// The boost arguments of hvae_tc_score_topk_boosted / hvae_mask_topk_boosted.
struct BoostArgs {
    const float* boost; int64_t boost_stride;
    const float* bound; int64_t bound_stride;
    const int32_t* boost_of_row; const float* row_weight;
};
// 0, or hvae_fail's status when the tables do not cover the global ids item_offset .. item_offset + N - 1
inline int check_boost_args(const char* what, const BoostArgs& b, int item_offset, int N) {
    const int64_t end = (int64_t)item_offset + N;
    HVAE_REQUIRE(b.bound && b.boost_of_row && b.row_weight, "%s: boost needs boost_bound, boost_of_row and row_boost_weight", what);
    HVAE_REQUIRE(item_offset >= 0 && b.boost_stride >= end && b.bound_stride >= 2 * ((end + 31) / 32),
                 "%s: boost_stride=%lld / bound_stride=%lld do not cover items up to %lld", what, (long long)b.boost_stride,
                 (long long)b.bound_stride, (long long)end);
    return 0;
}

__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ __forceinline__ int round_up(int a, int b) { return (a + b - 1) / b * b; }

}  // namespace hvae

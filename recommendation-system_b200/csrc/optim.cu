// Optimiser-side kernels: per-step scalars, global grad-norm clip and the fused Adam step.
// Replaces optimizer.zero_grad / clip_grad_norm_(5.0) / torch.optim.Adam.step of the reference
// (src/ml/train.py:63,88-92) and AnnealedVAE's beta schedule (src/ml/model.py:312-323).
// HBM-bound: Adam touches p, m, v once each (24 B/param + the sparse layer-1 gradient rows).
#include "common.cuh"
#include "hvae_b200.h"

namespace hvae {

// All step-dependent scalars live on the device so that a captured CUDA graph can be replayed unchanged.
__global__ void step_begin_kernel(hvae_step_state* st, double lr, double b1, double b2, double beta_min, double beta_max,
                                  int anneal_steps, int b_global, int advance_adam, uint32_t noise_stride) {
    pdl_prologue();
    if (advance_adam) {
        const int step = ++st->adam_step;
        const double bc1 = 1.0 - pow(b1, (double)step);
        const double bc2 = 1.0 - pow(b2, (double)step);
        st->step_size = (float)(lr / bc1);
        st->bc2_sqrt = (float)sqrt(bc2);
    }
    double beta = beta_max;
    if (anneal_steps > 0) {  // src/ml/model.py:312-319, then step_annealing() (:321-323)
        const int cur = st->anneal_step;
        if (cur < anneal_steps) beta = beta_min + ((double)cur / (double)anneal_steps) * (beta_max - beta_min);
        if (advance_adam) st->anneal_step = cur + 1;
    }
    if (advance_adam) {
        const uint64_t ctr = ((uint64_t)st->noise_hi << 32 | st->noise_lo) + noise_stride;
        st->noise_lo = (uint32_t)ctr;
        st->noise_hi = (uint32_t)(ctr >> 32);
    }
    st->beta_kl = (float)beta;
    st->inv_bg = 1.0f / (float)b_global;
    st->kl_coef = (float)beta / (float)b_global;
}

__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ partial) {
    pdl_prologue();
    float s = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s = fmaf(g[i], g[i], s);
    __shared__ float red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        partial[blockIdx.x] = t;
    }
}

// norm2 = sum(partial) + sum(rownorm2[0..n_unique)) (+ extra2, e.g. a value already all-reduced); clip coefficient as
// torch.nn.utils.clip_grad_norm_: max_norm / (norm + 1e-6), clamped to 1.
__global__ void __launch_bounds__(1024) gradnorm_final_kernel(const float* __restrict__ partial, int npartial,
                                                               const float* __restrict__ rownorm2, const int32_t* __restrict__ n_unique,
                                                               float max_norm, hvae_step_state* st) {
    pdl_prologue();
    __shared__ double red[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < npartial; i += blockDim.x) s += (double)partial[i];
    if (rownorm2) {
        const int n = *n_unique;
        for (int i = threadIdx.x; i < n; i += blockDim.x) s += (double)rownorm2[i];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += red[w];
        const float norm = (float)sqrt(t);
        st->norm2 = (float)t;
        st->grad_norm = norm;
        st->clip_coef = fminf(1.0f, max_norm / (norm + 1e-6f));
    }
}

__device__ __forceinline__ void adam_one(float& p, float& m, float& v, float g, float clip, float wd, float b1, float b2, float eps,
                                         float step_size, float bc2_sqrt) {
    g *= clip;
    if (wd != 0.f) g = fmaf(wd, p, g);
    m = m + (1.0f - b1) * (g - m);              // exp_avg.lerp_(grad, 1 - beta1)
    v = v * b2 + (1.0f - b2) * g * g;           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    const float denom = sqrtf(v) / bc2_sqrt + eps;
    p = p + (-step_size) * (m / denom);         // param.addcdiv_(exp_avg, denom, value=-step_size)
}

// One thread per float4.  [0, n_w1_4): layer-1 weight W1^T whose gradient exists only for the rows listed in
// slot_of_item (row -> compact gradient row, -1 = zero gradient); [n_w1_4, n4): dense gradient gd.
// untouched_only: just the W1^T rows WITHOUT a gradient in this step (slot < 0).  Their update (g = 0: moments decay, the parameter moves
// along the old momentum) needs nothing from this step's backward pass -- not even the clip coefficient -- so a step can run it beside
// the backward kernels; adam_touched_kernel then finishes the rows with a gradient and the dense tensors.  Same arithmetic per element.
__global__ void __launch_bounds__(256) adam_kernel(float4* __restrict__ p, float4* __restrict__ m, float4* __restrict__ v, int64_t n4,
                                                   int64_t n_w1_4, int ld4, const int32_t* __restrict__ slot_of_item,
                                                   const float4* __restrict__ gs, const float4* __restrict__ gd,
                                                   const hvae_step_state* __restrict__ st, float wd, float b1, float b2, float eps,
                                                   int untouched_only) {
    pdl_prologue();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float4 g;
    if (i < n_w1_4) {
        const int64_t row = i / ld4;
        const int slot = slot_of_item[row];
        if (untouched_only && slot >= 0) return;
        g = slot >= 0 ? gs[(int64_t)slot * ld4 + (i - row * ld4)] : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
        g = gd[i - n_w1_4];
    }
    const float clip = st->clip_coef, ss = st->step_size, bs = st->bc2_sqrt;
    float4 pp = p[i], mm = m[i], vv = v[i];
    adam_one(pp.x, mm.x, vv.x, g.x, clip, wd, b1, b2, eps, ss, bs);
    adam_one(pp.y, mm.y, vv.y, g.y, clip, wd, b1, b2, eps, ss, bs);
    adam_one(pp.z, mm.z, vv.z, g.z, clip, wd, b1, b2, eps, ss, bs);
    adam_one(pp.w, mm.w, vv.w, g.w, clip, wd, b1, b2, eps, ss, bs);
    p[i] = pp; m[i] = mm; v[i] = vv;
}

// The rows of W1^T that DO have a gradient (compact row k of gs belongs to item uniq[k], k < *n_unique) and, behind them, the dense
// tensors.  Grid: max_rows * ld4 + (n4 - n_w1_4) threads.
__global__ void __launch_bounds__(256) adam_touched_kernel(float4* __restrict__ p, float4* __restrict__ m, float4* __restrict__ v, int64_t n4,
                                                           int64_t n_w1_4, int ld4, const int32_t* __restrict__ uniq,
                                                           const int32_t* __restrict__ n_unique, int max_rows,
                                                           const float4* __restrict__ gs, const float4* __restrict__ gd,
                                                           const hvae_step_state* __restrict__ st, float wd, float b1, float b2, float eps) {
    pdl_prologue();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n_row4 = (int64_t)max_rows * ld4;
    int64_t i;
    float4 g;
    if (idx < n_row4) {
        const int k = (int)(idx / ld4);
        if (k >= *n_unique) return;
        i = (int64_t)uniq[k] * ld4 + (idx - (int64_t)k * ld4);
        g = gs[idx];
    } else {
        const int64_t j = idx - n_row4;
        if (j >= n4 - n_w1_4) return;
        i = n_w1_4 + j;
        g = gd[j];
    }
    const float clip = st->clip_coef, ss = st->step_size, bs = st->bc2_sqrt;
    float4 pp = p[i], mm = m[i], vv = v[i];
    adam_one(pp.x, mm.x, vv.x, g.x, clip, wd, b1, b2, eps, ss, bs);
    adam_one(pp.y, mm.y, vv.y, g.y, clip, wd, b1, b2, eps, ss, bs);
    adam_one(pp.z, mm.z, vv.z, g.z, clip, wd, b1, b2, eps, ss, bs);
    adam_one(pp.w, mm.w, vv.w, g.w, clip, wd, b1, b2, eps, ss, bs);
    p[i] = pp; m[i] = mm; v[i] = vv;
}

// ---- counter-based noise (philox, common.cuh) for the throughput mode; parity mode passes torch's own tensors ----
__global__ void noise_mask_kernel(uint8_t* __restrict__ mask, int64_t n, float keep, uint64_t seed, uint64_t offset, uint32_t sid,
                                  const hvae_step_state* __restrict__ st) {
    pdl_prologue();
    const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i4 * 4 >= n) return;
    if (st) offset += ((uint64_t)st->noise_hi << 32 | st->noise_lo);
    uint32_t r[4];
    philox(seed, offset + (uint64_t)i4, sid, r);
    for (int k = 0; k < 4; ++k) {
        const int64_t i = i4 * 4 + k;
        if (i < n) mask[i] = ((r[k] >> 8) * (1.0f / 16777216.0f)) < keep ? 1 : 0;
    }
}

__global__ void noise_normal_kernel(float* __restrict__ eps, int64_t n, uint64_t seed, uint64_t offset, uint32_t sid,
                                    const hvae_step_state* __restrict__ st) {
    pdl_prologue();
    const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i4 * 4 >= n) return;
    if (st) offset += ((uint64_t)st->noise_hi << 32 | st->noise_lo);
    uint32_t r[4];
    philox(seed, offset + (uint64_t)i4, sid, r);
    for (int k = 0; k < 4; k += 2) {
        const float u1 = ((r[k] >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0,1]
        const float u2 = (r[k + 1] >> 8) * (1.0f / 16777216.0f);
        const float rad = sqrtf(-2.0f * logf(u1));
        float s, c;
        sincospif(2.0f * u2, &s, &c);
        const int64_t i = i4 * 4 + k;
        if (i < n) eps[i] = rad * c;
        if (i + 1 < n) eps[i + 1] = rad * s;
    }
}

// One-shot all-gather over NVLink / NVSwitch: every rank stores its block straight into the other ranks' receive
// buffers -- through the NVSwitch multicast address when there is one (one store, the switch replicates it: multimem.st),
// else through the peers' unicast mappings.  Ordering across ranks comes from the symmetric-memory barrier the caller
// issues before (receive buffers free) and after (stores visible) this kernel.
__global__ void __launch_bounds__(256) nvl_push_kernel(const float4* __restrict__ src, int64_t n4, float* mc_dst,
                                                       const uint64_t* __restrict__ peer_ptrs, int world, int64_t dst_off) {
    pdl_prologue();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const float4 v = src[i];
    if (mc_dst) {
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_dst + dst_off + 4 * i), "f"(v.x), "f"(v.y),
                     "f"(v.z), "f"(v.w)
                     : "memory");
    } else {
        for (int r = 0; r < world; ++r) {
            float4* d = reinterpret_cast<float4*>(reinterpret_cast<float*>(peer_ptrs[r]) + dst_off) + i;
            asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(d), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
        }
    }
}

}  // namespace hvae

using namespace hvae;

extern "C" {

int hvae_step_begin(hvae_step_state* state, double lr, double beta1, double beta2, double kl_beta_min, double kl_beta_max,
                    int anneal_steps, int b_global, int advance, uint32_t noise_stride, void* stream) {
    HVAE_REQUIRE(b_global > 0, "step_begin: global batch must be positive");
    launch_pdl(step_begin_kernel, 1, 1, 0, (cudaStream_t)stream, state, lr, beta1, beta2, kl_beta_min, kl_beta_max, anneal_steps, b_global, advance,
                                                         noise_stride);
    HVAE_LAUNCH_CHECK("step_begin");
    return 0;
}

// workspace >= 148 floats
int hvae_grad_norm_clip(const float* gdense, int64_t n_dense, const float* rownorm2, const int32_t* n_unique, float max_norm,
                        hvae_step_state* state, float* workspace, void* stream) {
    const int blocks = (int)max((int64_t)1, min((int64_t)kNumSMs, (n_dense + 255) / 256));
    launch_pdl(sumsq_partial_kernel, blocks, 256, 0, (cudaStream_t)stream, gdense, n_dense, workspace);
    launch_pdl(gradnorm_final_kernel, 1, 1024, 0, (cudaStream_t)stream, workspace, blocks, rownorm2, n_unique, max_norm, state);
    HVAE_LAUNCH_CHECK("grad_norm_clip");
    return 0;
}

// The two halves of hvae_grad_norm_clip as separate calls: the dense part only needs the dense gradients, so a captured step runs it
// beside the layer-1 weight-gradient kernels instead of after them.  workspace >= 149 floats (partials, then their count).
int hvae_grad_sumsq_dense(const float* gdense, int64_t n_dense, float* workspace, void* stream) {
    const int blocks = (int)max((int64_t)1, min((int64_t)kNumSMs, (n_dense + 255) / 256));
    launch_pdl(sumsq_partial_kernel, blocks, 256, 0, (cudaStream_t)stream, gdense, n_dense, workspace);
    HVAE_LAUNCH_CHECK("grad_sumsq_dense");
    return 0;
}

int hvae_grad_norm_finish(int64_t n_dense, const float* rownorm2, const int32_t* n_unique, float max_norm, hvae_step_state* state,
                          const float* workspace, void* stream) {
    const int blocks = (int)max((int64_t)1, min((int64_t)kNumSMs, (n_dense + 255) / 256));
    launch_pdl(gradnorm_final_kernel, 1, 1024, 0, (cudaStream_t)stream, workspace, blocks, rownorm2, n_unique, max_norm, state);
    HVAE_LAUNCH_CHECK("grad_norm_finish");
    return 0;
}

int hvae_adam_step(float* params, float* exp_avg, float* exp_avg_sq, int64_t n_params, int64_t n_w1, int ld1,
                   const int32_t* slot_of_item, const float* gsparse, const float* gdense, const hvae_step_state* state,
                   float weight_decay, float beta1, float beta2, float eps, void* stream) {
    HVAE_REQUIRE(n_params % 4 == 0 && n_w1 % 4 == 0 && ld1 % 4 == 0, "adam_step: sizes must be multiples of 4");
    if (n_params == 0) return 0;
    const int64_t n4 = n_params / 4;
    launch_pdl(adam_kernel, (unsigned)((n4 + 255) / 256), 256, 0, (cudaStream_t)stream,
        (float4*)params, (float4*)exp_avg, (float4*)exp_avg_sq, n4, n_w1 / 4, ld1 / 4, slot_of_item, (const float4*)gsparse,
        (const float4*)gdense, state, weight_decay, beta1, beta2, eps, 0);
    HVAE_LAUNCH_CHECK("adam_step");
    return 0;
}

// hvae_adam_step in two calls with the same result: first the W1^T rows without a gradient in this step (needs slot_of_item of the
// step's batch and the step scalars only: may run beside the backward pass), then the rows with one (uniq / n_unique of
// hvae_batch_transpose; at most max_rows of them) and the dense tensors.
int hvae_adam_step_untouched(float* params, float* exp_avg, float* exp_avg_sq, int64_t n_w1, int ld1, const int32_t* slot_of_item,
                             const hvae_step_state* state, float weight_decay, float beta1, float beta2, float eps, void* stream) {
    HVAE_REQUIRE(n_w1 % 4 == 0 && ld1 % 4 == 0, "adam_step_untouched: sizes must be multiples of 4");
    if (n_w1 == 0) return 0;
    const int64_t n4 = n_w1 / 4;
    launch_pdl(adam_kernel, (unsigned)((n4 + 255) / 256), 256, 0, (cudaStream_t)stream, (float4*)params, (float4*)exp_avg, (float4*)exp_avg_sq, n4,
               n4, ld1 / 4, slot_of_item, (const float4*)nullptr, (const float4*)nullptr, state, weight_decay, beta1, beta2, eps, 1);
    HVAE_LAUNCH_CHECK("adam_step_untouched");
    return 0;
}

int hvae_adam_step_touched(float* params, float* exp_avg, float* exp_avg_sq, int64_t n_params, int64_t n_w1, int ld1,
                           const int32_t* uniq_item, const int32_t* n_unique, int max_rows, const float* gsparse, const float* gdense,
                           const hvae_step_state* state, float weight_decay, float beta1, float beta2, float eps, void* stream) {
    HVAE_REQUIRE(n_params % 4 == 0 && n_w1 % 4 == 0 && ld1 % 4 == 0, "adam_step_touched: sizes must be multiples of 4");
    const int64_t n4 = n_params / 4, total = (int64_t)max_rows * (ld1 / 4) + (n4 - n_w1 / 4);
    if (total == 0) return 0;
    launch_pdl(adam_touched_kernel, (unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream, (float4*)params, (float4*)exp_avg,
               (float4*)exp_avg_sq, n4, n_w1 / 4, ld1 / 4, uniq_item, n_unique, max_rows, (const float4*)gsparse, (const float4*)gdense, state,
               weight_decay, beta1, beta2, eps);
    HVAE_LAUNCH_CHECK("adam_step_touched");
    return 0;
}

int hvae_fill_noise(uint8_t* mask, int64_t n_mask, float keep_prob, float* eps, int64_t n_eps, uint64_t seed, uint64_t offset,
                    uint32_t stream_id, const hvae_step_state* state, void* stream) {
    if (mask && n_mask > 0)
        launch_pdl(noise_mask_kernel, (unsigned)((n_mask / 4 + 256) / 256), 256, 0, (cudaStream_t)stream, mask, n_mask, keep_prob, seed, offset, stream_id,
                                                                                                  state);
    if (eps && n_eps > 0)
        launch_pdl(noise_normal_kernel, (unsigned)((n_eps / 4 + 256) / 256), 256, 0, (cudaStream_t)stream, eps, n_eps, seed, offset,
                                                                                                    stream_id + 0x80000000u, state);
    HVAE_LAUNCH_CHECK("fill_noise");
    return 0;
}

// src: n floats (multiple of 4, 16-byte aligned) of this rank; destination = offset dst_off (floats) inside every rank's
// symmetric receive buffer: mc_dst = its multicast address (or NULL), peer_ptrs = device array of the `world` unicast addresses.
int hvae_nvl_push(const float* src, int64_t n, float* mc_dst, const uint64_t* peer_ptrs, int world, int64_t dst_off, void* stream) {
    HVAE_REQUIRE(n % 4 == 0 && dst_off % 4 == 0, "nvl_push: sizes and offsets must be multiples of 4 floats");
    if (n == 0) return 0;
    launch_pdl(nvl_push_kernel, (unsigned)((n / 4 + 255) / 256), 256, 0, (cudaStream_t)stream, (const float4*)src, n / 4, mc_dst, peer_ptrs,
               world, dst_off);
    HVAE_LAUNCH_CHECK("nvl_push");
    return 0;
}

}  // extern "C"

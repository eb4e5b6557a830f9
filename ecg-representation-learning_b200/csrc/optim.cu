// Fused global-norm gradient clipping + AdamW over FLAT fp32 buffers (all 140 parameter tensors of the model
// live in one contiguous allocation, so "multi-tensor" is a single launch).
// Replaces nn.utils.clip_grad_norm_(params, 1.0, error_if_nonfinite=True) (~300 launches) and
// torch.optim.AdamW.step (~1.1 k launches) of /root/reference/ecg_transformer/models/train.py:281-282.
// HBM-bound: 28 B/param algorithmic (p, m, v read+write, g read) + 2 B/param for the bf16 weight shadow
// (+ 8 B/param for the fused weight EMA: read + write).
#include "common.cuh"

namespace ecgvit {

namespace {

enum { H_LR = 0, H_BETA1, H_BETA2, H_EPS, H_WD, H_BC1, H_BC2, H_MAXNORM, H_GSCALE,
       H_ONE_MINUS_B1, H_ONE_MINUS_B2, H_DECAY, H_STEP_SIZE, H_BC2_SQRT, H_SKIP, H_EMA_RATE };
enum { S_SUMSQ = 0, S_NONFINITE, S_NORM, S_SKIPPED };

// Stage 1: one partial sum of squares per CTA (fixed grid-stride order inside the CTA).
// Stage 2: a single CTA adds the partials in index order.  No atomics: the total norm must be BIT-IDENTICAL on every
// data-parallel replica (it scales the update through the clip coefficient), and run-to-run reproducible.
constexpr int SUMSQ_MAX_BLOCKS = 2048;
constexpr int S_PARTIALS = 4;  // stats[4 .. 4 + SUMSQ_MAX_BLOCKS) is scratch for the per-CTA partials

// four consecutive gradients as fp32 (the flat gradient buffer is fp32, or bf16 after a data-parallel bf16 all-reduce)
__device__ __forceinline__ float4 load_grad4(const float *g, int64_t i) { return __ldg(reinterpret_cast<const float4 *>(g) + i); }
__device__ __forceinline__ float4 load_grad4(const bf16 *g, int64_t i) {
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(g) + i);
    float4 v;
    unpack_bf16x2(u.x, v.x, v.y);
    unpack_bf16x2(u.y, v.z, v.w);
    return v;
}

// group id of the 64-element blocks that neither count in the norm nor get updated (frozen / in no group)
constexpr uint8_t ADAMW_UNGROUPED = 255;

// kGrouped: gmap holds one group id per 64-element block of g (n is then a multiple of 64); blocks with id
// ADAMW_UNGROUPED contribute nothing.  The partials and their order are those of the plain kernel.
template <typename TG, bool kGrouped = false>
__global__ void __launch_bounds__(256) grad_sumsq_kernel(const TG *__restrict__ g, int64_t n,
                                                          const float *__restrict__ hyper, float *__restrict__ stats,
                                                          const uint8_t *__restrict__ gmap = nullptr) {
    __shared__ float red[8];
    const float gs = hyper[H_GSCALE];
    const int64_t n4 = n / 4;
    float s = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        if (kGrouped && __ldg(gmap + (i >> 4)) == ADAMW_UNGROUPED) continue;   // 16 float4 = one 64-element block
        const float4 v = load_grad4(g, i);
        const float a = v.x * gs, b = v.y * gs, c = v.z * gs, d = v.w * gs;
        s = fmaf(a, a, s); s = fmaf(b, b, s); s = fmaf(c, c, s); s = fmaf(d, d, s);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = n4 * 4; i < n; ++i) { const float a = to_f32(g[i]) * gs; s = fmaf(a, a, s); }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
        t = warp_sum(t);
        if (threadIdx.x == 0) stats[S_PARTIALS + blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(256) grad_sumsq_finalize_kernel(float *__restrict__ stats, int nblocks) {
    __shared__ float red[8];
    float s = 0.f;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) s += stats[S_PARTIALS + i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
        t = warp_sum(t);
        if (threadIdx.x == 0) {
            stats[S_SUMSQ] = t;
            stats[S_NONFINITE] = isfinite(t) ? 0.0f : 1.0f;
            stats[S_NORM] = sqrtf(t);   // the total norm is known here already (AdamW may run much later when deferred)
        }
    }
}

__device__ __forceinline__ float clip_coef_from(const float *hyper, const float *stats, float &total_norm) {
    total_norm = sqrtf(stats[S_SUMSQ]);
    const float max_norm = hyper[H_MAXNORM];
    if (max_norm <= 0.f) return 1.0f;
    return fminf(max_norm / (total_norm + 1e-6f), 1.0f);
}

// kGrouped: per-parameter-group learning rate / weight decay.  gmap holds one group id per 64-element block of the
// flat buffers (every tensor starts on a 64-element boundary); gtable[2 * id] = 1 - lr_g * wd_g and
// gtable[2 * id + 1] = lr_g / (1 - beta1^t) replace hyper's decay / step size; id ADAMW_UNGROUPED leaves p, m, v and
// the shadow untouched.  Everything else (clip, skip, the non-finite counter, the update itself) is shared.
// kEma: after the update, ema += hyper[H_EMA_RATE] * (p_new - ema) from the registers holding p_new (the rate 1 - d_t
// is derived by the host in double precision).  Whatever leaves p untouched (skip, non-finite norm, id 255) leaves the
// EMA untouched too.

template <bool kShadow, typename TG, bool kGrouped = false, bool kEma = false>
__global__ void __launch_bounds__(256) adamw_kernel(float *__restrict__ p, float *__restrict__ m,
                                                     float *__restrict__ v, const TG *__restrict__ g,
                                                     bf16 *__restrict__ shadow, int64_t n,
                                                     const float *__restrict__ hyper, float *__restrict__ stats,
                                                     bool count_skips, const uint8_t *__restrict__ gmap = nullptr,
                                                     const float *__restrict__ gtable = nullptr,
                                                     float *__restrict__ ema = nullptr) {
    if (hyper[H_SKIP] != 0.f) return;   // a deferred-update slot with nothing pending (first step, or just flushed)
    float total_norm;
    const float clip = clip_coef_from(hyper, stats, total_norm);
    if (count_skips && blockIdx.x == 0 && threadIdx.x == 0) stats[S_NORM] = total_norm;
    // error_if_nonfinite: leave parameters and state untouched and COUNT the skipped update (sticky until the host clears
    // it: a poll every k steps cannot miss one); the host raises when it polls
    if (!isfinite(total_norm)) {
        if (count_skips && blockIdx.x == 0 && threadIdx.x == 0) stats[S_SKIPPED] += 1.0f;
        return;
    }
    // the derived scalars are computed by the host in double precision exactly like torch.optim.AdamW does
    // (1 - beta in fp32 differs from fp32(1 - beta) by 1.3e-5 relative for beta2 = 0.999)
    const float beta2 = hyper[H_BETA2], eps = hyper[H_EPS];
    const float one_m_b1 = hyper[H_ONE_MINUS_B1], one_m_b2 = hyper[H_ONE_MINUS_B2];
    float decay = hyper[H_DECAY], step_size = hyper[H_STEP_SIZE];
    const float bc2_sqrt = hyper[H_BC2_SQRT];
    const float ema_rate = kEma ? hyper[H_EMA_RATE] : 0.f;
    const float gmul = hyper[H_GSCALE] * clip;
    const int64_t n4 = n / 4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        if (kGrouped) {
            const uint8_t id = __ldg(gmap + (i >> 4));   // 16 float4 = one 64-element block
            if (id == ADAMW_UNGROUPED) continue;
            decay = __ldg(gtable + 2 * id);
            step_size = __ldg(gtable + 2 * id + 1);
        }
        const float4 g4 = load_grad4(g, i);
        float4 p4 = reinterpret_cast<float4 *>(p)[i], m4 = reinterpret_cast<float4 *>(m)[i],
               v4 = reinterpret_cast<float4 *>(v)[i];
        float pp[4] = {p4.x, p4.y, p4.z, p4.w}, mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
        const float gg[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float gr = gg[k] * gmul;
            pp[k] *= decay;
            mm[k] = fmaf(gr - mm[k], one_m_b1, mm[k]);            // exp_avg.lerp_(g, 1 - beta1)
            vv[k] = fmaf(one_m_b2 * gr, gr, vv[k] * beta2);        // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)
            const float denom = sqrtf(vv[k]) / bc2_sqrt + eps;     // (exp_avg_sq.sqrt() / sqrt(bc2)).add_(eps)
            pp[k] -= step_size * (mm[k] / denom);                  // addcdiv_(exp_avg, denom, -lr / bc1)
        }
        reinterpret_cast<float4 *>(p)[i] = make_float4(pp[0], pp[1], pp[2], pp[3]);
        reinterpret_cast<float4 *>(m)[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
        reinterpret_cast<float4 *>(v)[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
        if (kShadow) {
            uint2 u;
            u.x = pack_bf16x2(pp[0], pp[1]);
            u.y = pack_bf16x2(pp[2], pp[3]);
            reinterpret_cast<uint2 *>(shadow)[i] = u;
        }
        if (kEma) {
            float4 e4 = reinterpret_cast<float4 *>(ema)[i];
            e4.x = fmaf(ema_rate, pp[0] - e4.x, e4.x);
            e4.y = fmaf(ema_rate, pp[1] - e4.y, e4.y);
            e4.z = fmaf(ema_rate, pp[2] - e4.z, e4.z);
            e4.w = fmaf(ema_rate, pp[3] - e4.w, e4.w);
            reinterpret_cast<float4 *>(ema)[i] = e4;
        }
    }
}

template <bool kShadow, typename TG, bool kGrouped>
void launch_adamw_ema(int grid, cudaStream_t s, float *p, float *m, float *v, const void *g, void *shadow, int64_t n,
                      const float *hyper, float *stats, bool count, const uint8_t *gmap, const float *gtable,
                      float *ema) {
    adamw_kernel<kShadow, TG, kGrouped, true><<<grid, 256, 0, s>>>(p, m, v, (const TG *)g, (bf16 *)shadow, n, hyper,
                                                                    stats, count, gmap, gtable, ema);
}

template <bool kShadow, typename TG>
void launch_adamw_ema(bool grouped, int grid, cudaStream_t s, float *p, float *m, float *v, const void *g, void *shadow,
                      int64_t n, const float *hyper, float *stats, bool count, const uint8_t *gmap, const float *gtable,
                      float *ema) {
    if (grouped) launch_adamw_ema<kShadow, TG, true>(grid, s, p, m, v, g, shadow, n, hyper, stats, count, gmap, gtable, ema);
    else launch_adamw_ema<kShadow, TG, false>(grid, s, p, m, v, g, shadow, n, hyper, stats, count, nullptr, nullptr, ema);
}

__global__ void __launch_bounds__(256) grad_scale_kernel(float *__restrict__ g, int64_t n,
                                                          const float *__restrict__ hyper, float *__restrict__ stats) {
    float total_norm;
    const float mul = clip_coef_from(hyper, stats, total_norm) * hyper[H_GSCALE];
    if (blockIdx.x == 0 && threadIdx.x == 0) stats[S_NORM] = total_norm;
    if (!isfinite(total_norm) || mul == 1.0f) return;
    const int64_t n4 = n / 4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = reinterpret_cast<float4 *>(g)[i];
        v.x *= mul; v.y *= mul; v.z *= mul; v.w *= mul;
        reinterpret_cast<float4 *>(g)[i] = v;
    }
}

inline int flat_grid(int64_t n) {
    int64_t blocks = (n / 4 + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

}  // namespace
}  // namespace ecgvit

using namespace ecgvit;

extern "C" {

int ecgvit_grad_sumsq(const void *g, int grad_dtype, int64_t n, const float *hyper, float *stats, void *stream) {
    ECGVIT_REQUIRE(g && hyper && stats && n > 0, "grad_sumsq: bad arguments");
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "grad_sumsq: g must be 16-byte aligned");
    ECGVIT_REQUIRE(grad_dtype == ECGVIT_F32 || grad_dtype == ECGVIT_BF16, "grad_sumsq: unknown gradient dtype %d", grad_dtype);
    int grid = flat_grid(n);
    if (grid > SUMSQ_MAX_BLOCKS) grid = SUMSQ_MAX_BLOCKS;
    if (grad_dtype == ECGVIT_F32)
        grad_sumsq_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((const float *)g, n, hyper, stats);
    else
        grad_sumsq_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>((const bf16 *)g, n, hyper, stats);
    int rc = check_launch("grad_sumsq");
    if (rc) return rc;
    grad_sumsq_finalize_kernel<<<1, 256, 0, as_stream(stream)>>>(stats, grid);
    return check_launch("grad_sumsq_finalize");
}

int ecgvit_grad_sumsq_grouped(const void *g, int grad_dtype, int64_t n, const uint8_t *group_map, const float *hyper,
                              float *stats, void *stream) {
    ECGVIT_REQUIRE(g && group_map && hyper && stats && n > 0, "grad_sumsq_grouped: bad arguments");
    ECGVIT_REQUIRE(n % 64 == 0, "grad_sumsq_grouped: length %lld must be a multiple of 64 (one group id per 64 elements)",
                   (long long)n);
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "grad_sumsq_grouped: g must be 16-byte aligned");
    ECGVIT_REQUIRE(grad_dtype == ECGVIT_F32 || grad_dtype == ECGVIT_BF16, "grad_sumsq_grouped: unknown gradient dtype %d",
                   grad_dtype);
    int grid = flat_grid(n);
    if (grid > SUMSQ_MAX_BLOCKS) grid = SUMSQ_MAX_BLOCKS;
    if (grad_dtype == ECGVIT_F32)
        grad_sumsq_kernel<float, true><<<grid, 256, 0, as_stream(stream)>>>((const float *)g, n, hyper, stats, group_map);
    else
        grad_sumsq_kernel<bf16, true><<<grid, 256, 0, as_stream(stream)>>>((const bf16 *)g, n, hyper, stats, group_map);
    int rc = check_launch("grad_sumsq_grouped");
    if (rc) return rc;
    grad_sumsq_finalize_kernel<<<1, 256, 0, as_stream(stream)>>>(stats, grid);
    return check_launch("grad_sumsq_finalize");
}

int ecgvit_grad_sumsq_partial(const void *g, int grad_dtype, int64_t n, const float *hyper, float *stats,
                              int first_block, int n_blocks, void *stream) {
    ECGVIT_REQUIRE(g && hyper && stats && n > 0, "grad_sumsq_partial: bad arguments");
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "grad_sumsq_partial: g must be 16-byte aligned");
    ECGVIT_REQUIRE(grad_dtype == ECGVIT_F32 || grad_dtype == ECGVIT_BF16, "grad_sumsq_partial: unknown gradient dtype %d", grad_dtype);
    ECGVIT_REQUIRE(first_block >= 0 && n_blocks >= 1 && first_block + n_blocks <= SUMSQ_MAX_BLOCKS,
                   "grad_sumsq_partial: partial slots [%d, %d) outside [0, %d)", first_block, first_block + n_blocks,
                   SUMSQ_MAX_BLOCKS);
    // the kernel parks the partial of CTA i at stats[4 + i]: offsetting the pointer selects this slice's slots
    if (grad_dtype == ECGVIT_F32)
        grad_sumsq_kernel<float><<<n_blocks, 256, 0, as_stream(stream)>>>((const float *)g, n, hyper, stats + first_block);
    else
        grad_sumsq_kernel<bf16><<<n_blocks, 256, 0, as_stream(stream)>>>((const bf16 *)g, n, hyper, stats + first_block);
    return check_launch("grad_sumsq_partial");
}

int ecgvit_grad_sumsq_finalize(float *stats, int n_blocks, void *stream) {
    ECGVIT_REQUIRE(stats && n_blocks >= 1 && n_blocks <= SUMSQ_MAX_BLOCKS, "grad_sumsq_finalize: bad arguments");
    grad_sumsq_finalize_kernel<<<1, 256, 0, as_stream(stream)>>>(stats, n_blocks);
    return check_launch("grad_sumsq_finalize");
}

int ecgvit_adamw_step(float *p, float *m, float *v, const void *g, int grad_dtype, void *shadow_bf16, int64_t n,
                      const float *hyper, float *stats, int flags, void *stream) {
    ECGVIT_REQUIRE(p && m && v && g && hyper && stats && n > 0, "adamw_step: bad arguments");
    ECGVIT_REQUIRE(n % 4 == 0, "adamw_step: flat length %lld must be a multiple of 4 (pad the flat buffer)", (long long)n);
    ECGVIT_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v) |
                     reinterpret_cast<uintptr_t>(g)) & 15) == 0,
                   "adamw_step: buffers must be 16-byte aligned");
    ECGVIT_REQUIRE(grad_dtype == ECGVIT_F32 || grad_dtype == ECGVIT_BF16, "adamw_step: unknown gradient dtype %d", grad_dtype);
    cudaStream_t s = as_stream(stream);
    // ECGVIT_ADAMW_SLICE: this call updates one slice of a larger buffer next to other work (the deferred optimizer runs
    // layer by layer beside the next forward pass): short-lived CTAs (one pass each) that never hold an SM for long, and
    // only the call flagged ECGVIT_ADAMW_FIRST_SLICE records the norm / counts a skipped update
    const bool slice = (flags & ECGVIT_ADAMW_SLICE) != 0;
    const bool count = !slice || (flags & ECGVIT_ADAMW_FIRST_SLICE) != 0;
    const int grid = slice ? (int)((n / 4 + 255) / 256) : flat_grid(n);
    bf16 *sh = (bf16 *)shadow_bf16;
    if (grad_dtype == ECGVIT_F32) {
        if (sh) adamw_kernel<true, float><<<grid, 256, 0, s>>>(p, m, v, (const float *)g, sh, n, hyper, stats, count);
        else adamw_kernel<false, float><<<grid, 256, 0, s>>>(p, m, v, (const float *)g, nullptr, n, hyper, stats, count);
    } else {
        if (sh) adamw_kernel<true, bf16><<<grid, 256, 0, s>>>(p, m, v, (const bf16 *)g, sh, n, hyper, stats, count);
        else adamw_kernel<false, bf16><<<grid, 256, 0, s>>>(p, m, v, (const bf16 *)g, nullptr, n, hyper, stats, count);
    }
    return check_launch("adamw_step");
}

int ecgvit_adamw_step_grouped(float *p, float *m, float *v, const void *g, int grad_dtype, void *shadow_bf16, int64_t n,
                              const uint8_t *group_map, const float *group_table, const float *hyper, float *stats,
                              int flags, void *stream) {
    ECGVIT_REQUIRE(p && m && v && g && group_map && group_table && hyper && stats && n > 0,
                   "adamw_step_grouped: bad arguments");
    ECGVIT_REQUIRE(n % 64 == 0, "adamw_step_grouped: length %lld must be a multiple of 64 (one group id per 64 elements)",
                   (long long)n);
    ECGVIT_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v) |
                     reinterpret_cast<uintptr_t>(g)) & 15) == 0,
                   "adamw_step_grouped: buffers must be 16-byte aligned");
    ECGVIT_REQUIRE(grad_dtype == ECGVIT_F32 || grad_dtype == ECGVIT_BF16, "adamw_step_grouped: unknown gradient dtype %d",
                   grad_dtype);
    cudaStream_t s = as_stream(stream);
    const bool slice = (flags & ECGVIT_ADAMW_SLICE) != 0;
    const bool count = !slice || (flags & ECGVIT_ADAMW_FIRST_SLICE) != 0;
    const int grid = slice ? (int)((n / 4 + 255) / 256) : flat_grid(n);
    bf16 *sh = (bf16 *)shadow_bf16;
    const uint8_t *gm = group_map;
    const float *gt = group_table;
    if (grad_dtype == ECGVIT_F32) {
        if (sh) adamw_kernel<true, float, true><<<grid, 256, 0, s>>>(p, m, v, (const float *)g, sh, n, hyper, stats, count, gm, gt);
        else adamw_kernel<false, float, true><<<grid, 256, 0, s>>>(p, m, v, (const float *)g, nullptr, n, hyper, stats, count, gm, gt);
    } else {
        if (sh) adamw_kernel<true, bf16, true><<<grid, 256, 0, s>>>(p, m, v, (const bf16 *)g, sh, n, hyper, stats, count, gm, gt);
        else adamw_kernel<false, bf16, true><<<grid, 256, 0, s>>>(p, m, v, (const bf16 *)g, nullptr, n, hyper, stats, count, gm, gt);
    }
    return check_launch("adamw_step_grouped");
}

int ecgvit_adamw_step_ema(float *p, float *m, float *v, const void *g, int grad_dtype, void *shadow_bf16, float *ema,
                          int64_t n, const uint8_t *group_map, const float *group_table, const float *hyper,
                          float *stats, int flags, void *stream) {
    const bool grouped = group_map != nullptr;
    ECGVIT_REQUIRE(p && m && v && g && ema && hyper && stats && n > 0, "adamw_step_ema: bad arguments");
    ECGVIT_REQUIRE(!grouped || group_table, "adamw_step_ema: a group map needs a group table");
    ECGVIT_REQUIRE(n % (grouped ? 64 : 4) == 0, "adamw_step_ema: length %lld must be a multiple of %d%s", (long long)n,
                   grouped ? 64 : 4, grouped ? " (one group id per 64 elements)" : " (pad the flat buffer)");
    ECGVIT_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v) |
                     reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(ema)) & 15) == 0,
                   "adamw_step_ema: buffers must be 16-byte aligned");
    ECGVIT_REQUIRE(grad_dtype == ECGVIT_F32 || grad_dtype == ECGVIT_BF16, "adamw_step_ema: unknown gradient dtype %d",
                   grad_dtype);
    cudaStream_t s = as_stream(stream);
    const bool slice = (flags & ECGVIT_ADAMW_SLICE) != 0;
    const bool count = !slice || (flags & ECGVIT_ADAMW_FIRST_SLICE) != 0;
    const int grid = slice ? (int)((n / 4 + 255) / 256) : flat_grid(n);
    void *sh = shadow_bf16;
    const uint8_t *gm = group_map;
    const float *gt = group_table;
    if (grad_dtype == ECGVIT_F32) {
        if (sh) launch_adamw_ema<true, float>(grouped, grid, s, p, m, v, g, sh, n, hyper, stats, count, gm, gt, ema);
        else launch_adamw_ema<false, float>(grouped, grid, s, p, m, v, g, nullptr, n, hyper, stats, count, gm, gt, ema);
    } else {
        if (sh) launch_adamw_ema<true, bf16>(grouped, grid, s, p, m, v, g, sh, n, hyper, stats, count, gm, gt, ema);
        else launch_adamw_ema<false, bf16>(grouped, grid, s, p, m, v, g, nullptr, n, hyper, stats, count, gm, gt, ema);
    }
    return check_launch("adamw_step_ema");
}

int ecgvit_grad_scale_by_clip(float *g, int64_t n, const float *hyper, float *stats, void *stream) {
    ECGVIT_REQUIRE(g && hyper && stats && n > 0 && n % 4 == 0, "grad_scale_by_clip: bad arguments");
    grad_scale_kernel<<<flat_grid(n), 256, 0, as_stream(stream)>>>(g, n, hyper, stats);
    return check_launch("grad_scale_by_clip");
}

}  // extern "C"

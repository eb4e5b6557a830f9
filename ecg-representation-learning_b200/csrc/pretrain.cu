// Masked-patch pre-training (SimMIM-style): the mask draw, the MAE index build and row gather, the loss fold of the reconstruction GEMM's row partials
// (ECGVIT_EPI_BIAS_SUB_ROWSQ), the gradient of that loss w.r.t. the prediction, and the fp32 reconstruction output.
// The encoder, the masked token assembly and the patch-row LayerNorm live in elementwise.cu; the GEMMs in gemm_*.cu.
#include "common.cuh"

namespace ecgvit {

namespace {

constexpr int kMaskThreads = 256;
// keys in dynamic shared memory; with the kernel's static warp totals the block stays under the 48 KB a launch gets
// without an opt-in attribute
constexpr int kMaxMaskPatches = 12000;

// one CTA per record: every patch's rank among the record's keys (ties by index) decides; exactly k are masked.
// seed == nullptr: the mask is the caller's, only counted.
__global__ void __launch_bounds__(kMaskThreads) mpm_mask_kernel(const uint32_t *__restrict__ seed_ptr, int n, int k,
                                                                 uint32_t site, uint8_t *__restrict__ mask,
                                                                 int *__restrict__ counts) {
    extern __shared__ uint32_t keys[];
    const int b = blockIdx.x;
    uint8_t *m = mask + (int64_t)b * n;
    int mine = 0;
    if (seed_ptr != nullptr) {
        const uint32_t seed = __ldg(seed_ptr);
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            keys[i] = dropout_hash(seed, site, static_cast<uint32_t>((int64_t)b * n + i));
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const uint32_t ki = keys[i];
            int rank = 0;
            for (int j = 0; j < n; ++j) {
                const uint32_t kj = keys[j];   // the same address for the whole warp: a broadcast
                rank += (kj < ki) || (kj == ki && j < i);
            }
            const bool masked = rank < k;
            m[i] = masked ? 1 : 0;
            mine += masked;
        }
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) mine += m[i] != 0;
    }
    // integer sums: exact in any order
    mine = __reduce_add_sync(0xffffffffu, mine);
    __shared__ int warp_tot[kMaskThreads / 32];
    if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kMaskThreads / 32; ++w) t += warp_tot[w];
        counts[b] = t;
    }
}

constexpr int kLossThreads = 1024;

// one CTA: thread t folds rows t, t + 1024, ... (groups in order), then a fixed tree over the threads
__global__ void __launch_bounds__(kLossThreads) mpm_loss_kernel(const float *__restrict__ rowsq, int n_groups,
                                                                 const uint8_t *__restrict__ mask,
                                                                 const int *__restrict__ counts, int B, int64_t rows,
                                                                 int K, float *__restrict__ loss,
                                                                 float *__restrict__ count) {
    __shared__ float red[kLossThreads];
    __shared__ int cnt[kLossThreads];
    pdl_launch_dependents();
    pdl_wait();
    float s = 0.f;
    for (int64_t r = threadIdx.x; r < rows; r += kLossThreads) {
        if (mask[r] != 0) {
            float t = 0.f;
            for (int g = 0; g < n_groups; ++g) t += rowsq[(int64_t)g * rows + r];
            s += t;
        }
    }
    int c = 0;
    for (int b = threadIdx.x; b < B; b += kLossThreads) c += counts[b];
    red[threadIdx.x] = s;
    cnt[threadIdx.x] = c;
    __syncthreads();
    for (int h = kLossThreads / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) {
            red[threadIdx.x] += red[threadIdx.x + h];
            cnt[threadIdx.x] += cnt[threadIdx.x + h];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float total = static_cast<float>(cnt[0]);
        count[0] = total;
        loss[0] = red[0] / (total * static_cast<float>(K));
    }
}

// dpred = r * mask_row * 2 * gs / (count * K), 8 elements per thread
template <typename T>
__global__ void mpm_dpred_kernel(const T *__restrict__ r, const uint8_t *__restrict__ mask,
                                 const float *__restrict__ count, int64_t rows, int ld, int K, float grad_scale,
                                 const float *__restrict__ grad_scale_dev, T *__restrict__ dpred) {
    pdl_launch_dependents();
    pdl_wait();
    float gs = grad_scale;
    if (grad_scale_dev != nullptr) gs *= __ldg(grad_scale_dev);
    const float scale = 2.0f * gs / (__ldg(count) * static_cast<float>(K));
    const int vec = ld / 8;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * vec; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i / vec;
        const int64_t off = row * ld + (i % vec) * 8;
        float v[8];
        load8(r + off, v);
        const float f = mask[row] != 0 ? scale : 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] *= f;
        store8(dpred + off, v);
    }
}

template <typename T>
__global__ void mpm_reconstruction_kernel(const T *__restrict__ r, const T *__restrict__ target, float *__restrict__ out,
                                          int64_t rows, int ld, int K) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * K; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = (i / K) * ld + (i % K);
        out[i] = to_f32(r[off]) + to_f32(target[off]);
    }
}

// MAE index build, one CTA per record: a block prefix sum over the visible flags.  Thread t owns the contiguous chunk
// [t * chunk, (t + 1) * chunk) of the record's patches; a warp scan of the chunk counts, then a scan of the warp totals.
constexpr int kIndexThreads = 256;
__global__ void __launch_bounds__(kIndexThreads) mae_index_kernel(const uint8_t *__restrict__ mask, int n, int n_vis,
                                                                   int *__restrict__ vis_idx, int *__restrict__ slot) {
    __shared__ int warp_tot[kIndexThreads / 32];
    pdl_launch_dependents();
    pdl_wait();
    const int b = blockIdx.x;
    const uint8_t *m = mask + (int64_t)b * n;
    const int chunk = (n + kIndexThreads - 1) / kIndexThreads;
    const int lo = min(threadIdx.x * chunk, n), hi = min(lo + chunk, n);
    int cnt = 0;
    for (int i = lo; i < hi; ++i) cnt += m[i] == 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int run = incl - cnt;
    for (int w = 0; w < warp; ++w) run += warp_tot[w];
    int *sl = slot + (int64_t)b * n;
    int *vi = vis_idx + (int64_t)b * n_vis;
    for (int i = lo; i < hi; ++i) {
        if (m[i] == 0) {
            sl[i] = run;
            if (run < n_vis) vi[run] = i;   // a mask with more visible patches than n_vis cannot write past the row
            ++run;
        } else {
            sl[i] = -1;
        }
    }
}

// dst row b*n_dst + j = src row b*n_src + idx[b*n_dst + j]; rows of vec 16-byte words
__global__ void row_gather_kernel(const uint4 *__restrict__ src, uint4 *__restrict__ dst, const int *__restrict__ idx,
                                  int n_src, int n_dst, int64_t rows, int vec) {
    pdl_launch_dependents();
    pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * vec; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / vec;
        const int v = (int)(i - r * vec);
        const int64_t s = (r / n_dst) * n_src + idx[r];
        dst[i] = src[s * vec + v];
    }
}

inline int grid_cap(int64_t items, int threads) {
    int64_t g = (items + threads - 1) / threads;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (g > cap) g = cap;
    return g < 1 ? 1 : (int)g;
}

}  // namespace
}  // namespace ecgvit

using namespace ecgvit;

extern "C" {

int ecgvit_mpm_mask(const uint32_t *seed, int B, int n_patch, int k, int site, uint8_t *mask, int *counts,
                    void *stream) {
    ECGVIT_REQUIRE(mask && counts && B > 0 && n_patch > 0, "mpm_mask: bad arguments");
    ECGVIT_REQUIRE(n_patch <= kMaxMaskPatches, "mpm_mask: n_patch=%d exceeds %d", n_patch, kMaxMaskPatches);
    ECGVIT_REQUIRE(seed == nullptr || (k >= 0 && k <= n_patch), "mpm_mask: k=%d outside [0, n_patch=%d]", k, n_patch);
    const size_t smem = seed != nullptr ? (size_t)n_patch * sizeof(uint32_t) : 0;
    mpm_mask_kernel<<<B, kMaskThreads, smem, as_stream(stream)>>>(seed, n_patch, k, static_cast<uint32_t>(site), mask,
                                                                  counts);
    return check_launch("mpm_mask");
}

int ecgvit_mae_index(const uint8_t *mask, int B, int n_patch, int n_vis, int *vis_idx, int *slot, void *stream) {
    ECGVIT_REQUIRE(mask && vis_idx && slot && B > 0 && n_patch > 0 && n_vis > 0 && n_vis <= n_patch,
                   "mae_index: bad arguments");
    ECGVIT_REQUIRE(n_patch <= kMaxMaskPatches, "mae_index: n_patch=%d exceeds %d", n_patch, kMaxMaskPatches);
    launch_pdl(mae_index_kernel, dim3(B), dim3(kIndexThreads), 0, as_stream(stream), mask, n_patch, n_vis, vis_idx, slot);
    return check_launch("mae_index");
}

int ecgvit_row_gather(const void *src, void *dst, const int *idx, int B, int n_src, int n_dst, int ld, int dtype,
                      void *stream) {
    ECGVIT_REQUIRE(src && dst && idx && B > 0 && n_src > 0 && n_dst > 0 && ld > 0, "row_gather: bad arguments");
    int esz;
    if (dtype == ECGVIT_BF16) esz = 2;
    else if (dtype == ECGVIT_F32) esz = 4;
    else return fail(-1, "row_gather: unknown dtype %d", dtype);
    ECGVIT_REQUIRE(((int64_t)ld * esz) % 16 == 0, "row_gather: rows of %d elements are not 16-byte multiples", ld);
    const int vec = (int)((int64_t)ld * esz / 16);
    const int64_t rows = (int64_t)B * n_dst;
    launch_pdl(row_gather_kernel, dim3(grid_cap(rows * vec, 256)), dim3(256), 0, as_stream(stream), (const uint4 *)src,
               (uint4 *)dst, idx, n_src, n_dst, rows, vec);
    return check_launch("row_gather");
}

int ecgvit_mpm_loss(const float *rowsq, int n_groups, const uint8_t *mask, const int *counts, int B, int n_patch,
                    int K, float *loss, float *count, void *stream) {
    ECGVIT_REQUIRE(rowsq && mask && counts && loss && count && n_groups > 0 && B > 0 && n_patch > 0 && K > 0,
                   "mpm_loss: bad arguments");
    launch_pdl(mpm_loss_kernel, dim3(1), dim3(kLossThreads), 0, as_stream(stream), rowsq, n_groups, mask, counts, B,
               (int64_t)B * n_patch, K, loss, count);
    return check_launch("mpm_loss");
}

int ecgvit_mpm_dpred(const void *r, const uint8_t *mask, const float *count, int rows, int ld, int K,
                     float grad_scale, const float *grad_scale_dev, void *dpred, int dtype, void *stream) {
    ECGVIT_REQUIRE(r && mask && count && dpred && rows > 0 && K > 0 && ld >= K, "mpm_dpred: bad arguments");
    ECGVIT_REQUIRE(ld % 8 == 0, "mpm_dpred: ld=%d must be a multiple of 8", ld);
    const int grid = grid_cap((int64_t)rows * (ld / 8), 256);
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        launch_pdl(mpm_dpred_kernel<bf16>, dim3(grid), dim3(256), 0, st, (const bf16 *)r, mask, count, (int64_t)rows, ld,
                   K, grad_scale, grad_scale_dev, (bf16 *)dpred);
    else if (dtype == ECGVIT_F32)
        launch_pdl(mpm_dpred_kernel<float>, dim3(grid), dim3(256), 0, st, (const float *)r, mask, count, (int64_t)rows,
                   ld, K, grad_scale, grad_scale_dev, (float *)dpred);
    else return fail(-1, "mpm_dpred: unknown dtype %d", dtype);
    return check_launch("mpm_dpred");
}

int ecgvit_mpm_reconstruction(const void *r, const void *target, float *out, int rows, int ld, int K, int dtype,
                              void *stream) {
    ECGVIT_REQUIRE(r && target && out && rows > 0 && K > 0 && ld >= K, "mpm_reconstruction: bad arguments");
    const int grid = grid_cap((int64_t)rows * K, 256);
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        mpm_reconstruction_kernel<bf16><<<grid, 256, 0, st>>>((const bf16 *)r, (const bf16 *)target, out, rows, ld, K);
    else if (dtype == ECGVIT_F32)
        mpm_reconstruction_kernel<float><<<grid, 256, 0, st>>>((const float *)r, (const float *)target, out, rows, ld, K);
    else return fail(-1, "mpm_reconstruction: unknown dtype %d", dtype);
    return check_launch("mpm_reconstruction");
}

}  // extern "C"

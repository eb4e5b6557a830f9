// Attention front door: picks the kernel for (dtype, N, dh).
#include "common.cuh"

namespace ecgvit {
int attention_fwd_simt(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale, int dtype,
                       DropoutParams drop, cudaStream_t stream);
int attention_bwd_simt(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, int B, int N,
                       int H, int dh, float scale, int dtype, DropoutParams drop, cudaStream_t stream);
int attention_fwd_mma(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale,
                      DropoutParams drop, cudaStream_t stream);
int attention_bwd_mma(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, int B, int N,
                      int H, int dh, float scale, DropoutParams drop, cudaStream_t stream);
bool attention_mma_supported(int N, int dh);
// attention_flash.cu: tiled kernels for N > 64 (bf16)
int attention_fwd_flash(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale,
                        DropoutParams drop, cudaStream_t stream);
int attention_bwd_flash(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, float *dscratch,
                        int B, int N, int H, int dh, float scale, DropoutParams drop, cudaStream_t stream);
bool attention_flash_supported(int N, int dh);
// attention_tc.cu: tcgen05 / TMEM / TMA kernels (bf16, head dim 64, any N)
int attention_fwd_tc(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale, DropoutParams drop,
                     cudaStream_t stream);
int attention_bwd_tc(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, float *scratch, int B,
                     int N, int H, int dh, float scale, DropoutParams drop, cudaStream_t stream);
int64_t attention_bwd_tc_scratch_floats(int B, int N, int H);
bool attention_tc_supported(int N, int dh);

// the dropout counter of the attention probabilities is a 32-bit element index ((b*H + h) * Np + i) * Np + j
static bool dropout_index_fits(int B, int N, int H) {
    const int64_t Np = (N + 63) / 64 * 64;
    return (int64_t)B * H * Np * Np <= ((int64_t)1 << 32);
}
}  // namespace ecgvit

namespace ecgvit {
namespace {

// Slow path for vit_pytorch's Recorder (hooks Attention.attend; reference use ecg_vit.py:176-193): the softmax
// probabilities themselves, which the training kernels never materialise.  One warp per (b, h, query row): a lane owns
// keys lane, lane + 32, ...; raw scores are parked in the output row, then exponentiated and normalised in place.
template <typename T>
__global__ void __launch_bounds__(128) attention_probs_kernel(const T *__restrict__ qkv, float *__restrict__ probs,
                                                               int B, int N, int H, int dh, float scale,
                                                               int64_t batch_stride) {
    extern __shared__ float s_q[];  // [4 warps][dh]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * 4 + wib;  // (b * H + h) * N + i
    if (row >= (int64_t)B * H * N) return;
    const int i = (int)(row % N);
    const int h = (int)((row / N) % H);
    const int64_t b = row / ((int64_t)N * H);
    const int inner = H * dh;
    const int64_t ld = 3 * (int64_t)inner;
    float *q = s_q + wib * dh;
    const T *qrow = qkv + (b * N + i) * ld + h * dh;
    for (int c = lane; c < dh; c += 32) q[c] = to_f32(qrow[c]);
    __syncwarp();
    float *out = probs + b * batch_stride + ((int64_t)h * N + i) * N;
    float mx = -INFINITY;
    for (int j = lane; j < N; j += 32) {
        const T *krow = qkv + (b * N + j) * ld + inner + h * dh;
        float acc = 0.f;
        for (int c = 0; c < dh; c += 8) {
            float kv[8];
            load8(krow + c, kv);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc = fmaf(q[c + k], kv[k], acc);
        }
        acc *= scale;
        out[j] = acc;
        mx = fmaxf(mx, acc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < N; j += 32) {
        const float e = expf(out[j] - mx);
        out[j] = e;
        sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    for (int j = lane; j < N; j += 32) out[j] *= inv;
}

}  // namespace
}  // namespace ecgvit

using namespace ecgvit;

extern "C" {

int ecgvit_attention_probs(const void *qkv, float *probs, int B, int N, int H, int dh, float scale,
                           int64_t batch_stride, int dtype, void *stream) {
    ECGVIT_REQUIRE(qkv && probs && B > 0 && N > 0 && H > 0, "attention_probs: bad arguments");
    ECGVIT_REQUIRE(dh % 8 == 0, "attention_probs: head dim %d must be a multiple of 8", dh);
    ECGVIT_REQUIRE(batch_stride >= (int64_t)H * N * N, "attention_probs: batch stride %lld < H*N*N",
                   (long long)batch_stride);
    const int64_t rows = (int64_t)B * H * N;
    const unsigned grid = (unsigned)((rows + 3) / 4);
    const size_t smem = 4 * (size_t)dh * sizeof(float);
    if (dtype == ECGVIT_BF16)
        attention_probs_kernel<bf16><<<grid, 128, smem, as_stream(stream)>>>((const bf16 *)qkv, probs, B, N, H, dh, scale, batch_stride);
    else if (dtype == ECGVIT_F32)
        attention_probs_kernel<float><<<grid, 128, smem, as_stream(stream)>>>((const float *)qkv, probs, B, N, H, dh, scale, batch_stride);
    else return fail(-1, "attention_probs: unknown dtype %d", dtype);
    return check_launch("attention_probs");
}

int ecgvit_attention_fwd(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale,
                         float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(qkv && o && lse && B > 0 && N > 0 && H > 0, "attention_fwd: bad arguments");
    ECGVIT_REQUIRE(dh % 8 == 0, "attention_fwd: head dim %d must be a multiple of 8", dh);
    ECGVIT_REQUIRE(dtype == ECGVIT_F32 || dtype == ECGVIT_BF16, "attention_fwd: unknown dtype %d", dtype);
    ECGVIT_REQUIRE(drop.threshold == 0 || dropout_index_fits(B, N, H),
                   "attention_fwd: B*H*Np*Np = %d*%d*Np^2 overflows the 32-bit dropout counter (N=%d)", B, H, N);
    if (dtype == ECGVIT_BF16 && attention_tc_supported(N, dh))
        return attention_fwd_tc(qkv, o, lse, B, N, H, dh, scale, drop, as_stream(stream));
    if (dtype == ECGVIT_BF16 && attention_mma_supported(N, dh))
        return attention_fwd_mma(qkv, o, lse, B, N, H, dh, scale, drop, as_stream(stream));
    if (dtype == ECGVIT_BF16 && attention_flash_supported(N, dh))
        return attention_fwd_flash(qkv, o, lse, B, N, H, dh, scale, drop, as_stream(stream));
    return attention_fwd_simt(qkv, o, lse, B, N, H, dh, scale, dtype, drop, as_stream(stream));
}

int64_t ecgvit_attention_bwd_scratch_floats(int B, int N, int H, int dh, int dtype) {
    if (dtype == ECGVIT_BF16 && attention_tc_supported(N, dh)) return attention_bwd_tc_scratch_floats(B, N, H);
    return (dtype == ECGVIT_BF16 && attention_flash_supported(N, dh)) ? (int64_t)B * H * N : 0;
}

int ecgvit_attention_bwd(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, float *scratch,
                         int B, int N, int H, int dh, float scale, float dropout_p, int dropout_stream,
                         const uint32_t *dropout_seed, int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(qkv && o && d_o && lse && dqkv && B > 0 && N > 0 && H > 0, "attention_bwd: bad arguments");
    ECGVIT_REQUIRE(dh % 8 == 0, "attention_bwd: head dim %d must be a multiple of 8", dh);
    ECGVIT_REQUIRE(dtype == ECGVIT_F32 || dtype == ECGVIT_BF16, "attention_bwd: unknown dtype %d", dtype);
    ECGVIT_REQUIRE(drop.threshold == 0 || dropout_index_fits(B, N, H),
                   "attention_bwd: B*H*Np*Np = %d*%d*Np^2 overflows the 32-bit dropout counter (N=%d)", B, H, N);
    if (dtype == ECGVIT_BF16 && attention_tc_supported(N, dh))
        return attention_bwd_tc(qkv, o, d_o, lse, dqkv, scratch, B, N, H, dh, scale, drop, as_stream(stream));
    if (dtype == ECGVIT_BF16 && attention_mma_supported(N, dh))
        return attention_bwd_mma(qkv, o, d_o, lse, dqkv, B, N, H, dh, scale, drop, as_stream(stream));
    if (dtype == ECGVIT_BF16 && attention_flash_supported(N, dh)) {
        ECGVIT_REQUIRE(scratch != nullptr && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0,
                       "attention_bwd: N=%d needs the (16-byte aligned) scratch of ecgvit_attention_bwd_scratch_floats", N);
        return attention_bwd_flash(qkv, o, d_o, lse, dqkv, scratch, B, N, H, dh, scale, drop, as_stream(stream));
    }
    return attention_bwd_simt(qkv, o, d_o, lse, dqkv, B, N, H, dh, scale, dtype, drop, as_stream(stream));
}

}  // extern "C"

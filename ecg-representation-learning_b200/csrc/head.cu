// CLS pool + mlp_head (LayerNorm + Linear(d -> n_class)) + BCE-with-logits loss, forward and backward.
// Replaces x[:, 0] -> mlp_head (vit_pytorch ViT.forward) and nn.BCEWithLogitsLoss
// (/root/reference/ecg_transformer/models/ecg_vit.py:118,148).  B x n_class is tiny (256 x 71): FFMA + shuffles.
#include "common.cuh"

#include <algorithm>

namespace ecgvit {

namespace {

constexpr int HEAD_MAXV = 4;  // d <= 1024

constexpr int HEAD_SPB = 8;   // samples per CTA (one warp each)

// One CTA = HEAD_SPB samples, one warp each: the warp LayerNorms its sample's CLS row and parks it in shared memory; then
// the warps split the classes, and every weight row a warp fetches is used for all HEAD_SPB samples (one CTA per sample
// made 256 CTAs pull the same 218 KB of W through L2 at the same time: 56 MB of L2 traffic, 23 us for 28 MFLOP).
// All loads are branch-free (clamped address + select): an `if (c < d) { load; use }` per vector becomes its own basic
// block and ptxas then waits for every 32-byte piece in turn (the round-1 kernel: 54 serial L2 round trips per warp).
template <typename T>
__global__ void __launch_bounds__(32 * HEAD_SPB) head_fwd_kernel(const T *__restrict__ tok, const float *__restrict__ gamma,
                                                                  const float *__restrict__ beta,
                                                                  const float *__restrict__ w,
                                                                  const float *__restrict__ bias, float *__restrict__ xn,
                                                                  float *__restrict__ mean_out,
                                                                  float *__restrict__ rstd_out,
                                                                  float *__restrict__ logits, int B, int N, int d,
                                                                  int n_class, float eps) {
    extern __shared__ float xs[];   // [HEAD_SPB][d] normalised CLS rows (zeros for samples beyond B)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * HEAD_SPB + warp;
    int cc[HEAD_MAXV];
    bool ok[HEAD_MAXV];
#pragma unroll
    for (int i = 0; i < HEAD_MAXV; ++i) {
        const int c = (i * 32 + lane) * 8;
        ok[i] = c < d;
        cc[i] = ok[i] ? c : 0;
    }
    auto load_w = [&](int cls, float (*dst)[8]) {
        const float *wr = w + (int64_t)min(cls, n_class - 1) * d;
#pragma unroll
        for (int i = 0; i < HEAD_MAXV; ++i) load8(wr + cc[i], dst[i]);
    };
    float wv[HEAD_MAXV][8], wn[HEAD_MAXV][8];
    // gridDim.y CTAs share a group of samples and split the classes (each normalises the rows for itself: latency, not
    // throughput); CTA y = 0 writes xn / mean / rstd
    const int cls_first = warp + HEAD_SPB * blockIdx.y, cls_step = HEAD_SPB * gridDim.y;
    const bool writer = blockIdx.y == 0;
    load_w(cls_first, wv);   // the first weight row travels while the row is normalised
    {
        const T *xr = tok + (int64_t)min(b, B - 1) * N * d;
        float v[HEAD_MAXV][8], g[HEAD_MAXV][8], bt[HEAD_MAXV][8];
#pragma unroll
        for (int i = 0; i < HEAD_MAXV; ++i) {
            load8(xr + cc[i], v[i]);
            load8(gamma + cc[i], g[i]);
            load8(beta + cc[i], bt[i]);
        }
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < HEAD_MAXV; ++i)
#pragma unroll
            for (int k = 0; k < 8; ++k) s += ok[i] ? v[i][k] : 0.f;
        const float mean = warp_sum(s) / (float)d;
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < HEAD_MAXV; ++i)
#pragma unroll
            for (int k = 0; k < 8; ++k) { const float t = ok[i] ? v[i][k] - mean : 0.f; sq += t * t; }
        const float rstd = rsqrtf(warp_sum(sq) / (float)d + eps);
#pragma unroll
        for (int i = 0; i < HEAD_MAXV; ++i) {
#pragma unroll
            for (int k = 0; k < 8; ++k) v[i][k] = b < B ? fmaf((v[i][k] - mean) * rstd, g[i][k], bt[i][k]) : 0.f;
            if (ok[i]) {
                if (b < B && writer) store8(xn + (int64_t)b * d + cc[i], v[i]);
                store8(xs + warp * d + cc[i], v[i]);
            }
        }
        if (lane == 0 && b < B && writer) { mean_out[b] = mean; rstd_out[b] = rstd; }
    }
    __syncthreads();
    const int n_here = min(HEAD_SPB, B - blockIdx.x * HEAD_SPB);
    for (int cls = cls_first; cls < n_class; cls += cls_step) {
        load_w(cls + cls_step, wn);   // next row in flight (clamped past the end)
        const float bs = bias[cls];
        // the dot products of all HEAD_SPB samples with this row, then their shuffle trees interleaved.  Per sample the
        // order is the one of a lone warp: per-lane FMAs over the vectors, then the butterfly.
        float acc[HEAD_SPB];
#pragma unroll
        for (int sidx = 0; sidx < HEAD_SPB; ++sidx) {
            acc[sidx] = 0.f;
#pragma unroll
            for (int i = 0; i < HEAD_MAXV; ++i) {
                float xv[8];
                load8(xs + sidx * d + cc[i], xv);
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[sidx] = fmaf(xv[k], ok[i] ? wv[i][k] : 0.f, acc[sidx]);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1)
#pragma unroll
            for (int sidx = 0; sidx < HEAD_SPB; ++sidx) acc[sidx] += __shfl_xor_sync(0xffffffffu, acc[sidx], off);
        if (lane < n_here) {
            float mine = acc[0];
#pragma unroll
            for (int sidx = 1; sidx < HEAD_SPB; ++sidx) mine = lane == sidx ? acc[sidx] : mine;
            logits[(int64_t)(blockIdx.x * HEAD_SPB + lane) * n_class + cls] = mine + bs;
        }
#pragma unroll
        for (int i = 0; i < HEAD_MAXV; ++i)
#pragma unroll
            for (int k = 0; k < 8; ++k) wv[i][k] = wn[i][k];
    }
}

__device__ __forceinline__ float bce_with_logits(float z, float y) {
    // max(z,0) - z*y + log1p(exp(-|z|))   (ATen's stable form)
    return fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
}

// `weight[labels.long()]` of ecg_vit.py:144-147: the element weight is looked up by the integer value of the label
__device__ __forceinline__ float label_weight(const float *__restrict__ table, int n_weight, float y) {
    if (table == nullptr) return 1.f;
    const int i = min(max(static_cast<int>(y), 0), n_weight - 1);
    return __ldg(table + i);
}

// single CTA, deterministic tree reduction
__global__ void __launch_bounds__(1024) bce_loss_kernel(const float *__restrict__ logits,
                                                         const float *__restrict__ labels, float *__restrict__ loss,
                                                         int n, int reduction, const float *__restrict__ loss_weight,
                                                         int n_weight) {
    __shared__ float red[32];
    float s = 0.f;
    // four independent (logit, label) loads in flight per thread: a single CTA walking 18 k elements one dependent load
    // pair at a time was pure latency (10 us)
    for (int i0 = threadIdx.x; i0 < n; i0 += 4 * blockDim.x) {
        float z[4], y[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = i0 + j * blockDim.x;
            z[j] = i < n ? logits[i] : 0.f;
            y[j] = i < n ? labels[i] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = i0 + j * blockDim.x;
            if (i < n) {
                const float l = label_weight(loss_weight, n_weight, y[j]) * bce_with_logits(z[j], y[j]);
                if (reduction == ECGVIT_REDUCTION_NONE) loss[i] = l;
                s += l;
            }
        }
    }
    if (reduction == ECGVIT_REDUCTION_NONE) return;
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
        t = warp_sum(t);
        if (threadIdx.x == 0) loss[0] = (reduction == ECGVIT_REDUCTION_MEAN) ? t / (float)n : t;
    }
}

// backward A: per sample, dlogits -> dxn = dlogits W -> LayerNorm' -> CLS row of dtok.
// One CTA = HEAD_SPB samples (one warp each); the weight rows go through shared memory, so W is read once per CTA instead
// of once per sample.
__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(dst))),
                 "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <typename T, typename TX = T>
__global__ void __launch_bounds__(32 * HEAD_SPB) head_bwd_rows_kernel(
    const TX *__restrict__ tok, const float *__restrict__ gamma, const float *__restrict__ w,
    const float *__restrict__ labels, const float *__restrict__ mean_in, const float *__restrict__ rstd_in,
    const float *__restrict__ logits, T *__restrict__ dtok, float *__restrict__ dxn_out, float *__restrict__ dlog_out,
    int B, int N, int d, int n_class, float coef_host, const float *__restrict__ coef_dev,
    const float *__restrict__ loss_weight, int n_weight, int ch_classes) {
    extern __shared__ float wsm[];   // [ch_classes][d]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * HEAD_SPB + warp;
    const bool live = b < B;
    // upstream gradient of the loss: a host scalar and / or a DEVICE scalar (autograd's grad_output: no host sync)
    const float coef = coef_dev != nullptr ? coef_host * __ldg(coef_dev) : coef_host;
    // dlogits of the sample: lane l holds classes l, l + 32, l + 64 (n_class <= 96 per pass; more classes loop)
    float dxn[HEAD_MAXV][8];
#pragma unroll
    for (int i = 0; i < HEAD_MAXV; ++i)
#pragma unroll
        for (int k = 0; k < 8; ++k) dxn[i][k] = 0.f;
    int cc[HEAD_MAXV];
#pragma unroll
    for (int i = 0; i < HEAD_MAXV; ++i) {
        const int c = (i * 32 + lane) * 8;
        cc[i] = c < d ? c : 0;
    }
    // the sample's CLS row, gamma and row statistics are only needed after the class loop: fetched now (branch-free)
    const int bb = min(b, B - 1);
    float xv[HEAD_MAXV][8], gm[HEAD_MAXV][8];
#pragma unroll
    for (int i = 0; i < HEAD_MAXV; ++i) {
        load8(tok + (int64_t)bb * N * d + cc[i], xv[i]);
        load8(gamma + cc[i], gm[i]);
    }
    const float mean = mean_in[bb], rstd = rstd_in[bb];
    // W goes through shared memory in chunks of `ch_classes` rows (all 71 rows of the base model at once: 213 KB), copied
    // with cp.async by the whole CTA so that every 16-byte piece is in flight at the same time
    float dl_lane = 0.f;
    for (int c0 = 0; c0 < n_class; c0 += ch_classes) {
        const int n_here = min(ch_classes, n_class - c0);
        if (c0 > 0) __syncthreads();   // everyone is done with the previous chunk
        {
            const float4 *src = reinterpret_cast<const float4 *>(w + (int64_t)c0 * d);
            float4 *dst = reinterpret_cast<float4 *>(wsm);
            for (int idx = threadIdx.x; idx < n_here * d / 4; idx += blockDim.x) cp_async16(dst + idx, src + idx);
            cp_async_wait_all();
        }
        __syncthreads();
        for (int j = 0; j < n_here; ++j) {
            const int cls = c0 + j;
            if ((cls & 31) == 0) {   // a new group of 32 classes: every lane computes one dlogit
                const int mine = cls + lane;
                dl_lane = 0.f;
                if (live && mine < n_class) {
                    const float z = logits[(int64_t)b * n_class + mine], y = labels[(int64_t)b * n_class + mine];
                    dl_lane = coef * label_weight(loss_weight, n_weight, y) * (1.0f / (1.0f + expf(-z)) - y);
                    dlog_out[(int64_t)b * n_class + mine] = dl_lane;
                }
            }
            const float dl = __shfl_sync(0xffffffffu, dl_lane, cls & 31);
#pragma unroll
            for (int i = 0; i < HEAD_MAXV; ++i) {   // lanes beyond d accumulate vector 0 again: never read
                float wv[8];
                load8(wsm + j * d + cc[i], wv);
#pragma unroll
                for (int k = 0; k < 8; ++k) dxn[i][k] = fmaf(dl, wv[k], dxn[i][k]);
            }
        }
    }
    if (!live) return;
    float g[HEAD_MAXV][8], xh[HEAD_MAXV][8];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < HEAD_MAXV; ++i) {
        const bool ok = (i * 32 + lane) * 8 < d;
        if (ok) store8(dxn_out + (int64_t)b * d + cc[i], dxn[i]);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            xh[i][k] = (xv[i][k] - mean) * rstd;
            g[i][k] = ok ? dxn[i][k] * gm[i][k] : 0.f;
            s1 += g[i][k];
            s2 = fmaf(g[i][k], xh[i][k], s2);
        }
    }
    s1 = warp_sum(s1) / (float)d;
    s2 = warp_sum(s2) / (float)d;
    T *dr = dtok + (int64_t)b * N * d;
#pragma unroll
    for (int i = 0; i < HEAD_MAXV; ++i) {
        if ((i * 32 + lane) * 8 < d) {
            float o[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] = rstd * (g[i][k] - s1 - xh[i][k] * s2);
            store8(dr + cc[i], o);
        }
    }
}

// backward B: per column k: dgamma, dbeta of the head LayerNorm and the column sum of the CLS-row gradients.
// block = 32 columns x 8 sample groups, smem tree at the end
template <typename T, typename TX = T>
__global__ void __launch_bounds__(256) head_bwd_cols_kernel(const TX *__restrict__ tok, const T *__restrict__ dtok,
                                                             const float *__restrict__ dxn,
                                                             const float *__restrict__ mean_in,
                                                             const float *__restrict__ rstd_in,
                                                             float *__restrict__ dgamma, float *__restrict__ dbeta,
                                                             float *__restrict__ dcolsum, int B, int N, int d) {
    __shared__ float red[3][8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + tx;
    float sg = 0.f, sb = 0.f, sc = 0.f;
    if (k < d) {
        // four samples in flight per thread (their CLS rows are N * d elements apart: every load is its own HBM round trip)
        for (int b0 = ty; b0 < B; b0 += 32) {
            float xv[4], mv[4], rv[4], dv[4], gv[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int b = min(b0 + 8 * j, B - 1);
                xv[j] = to_f32(tok[(int64_t)b * N * d + k]);
                mv[j] = mean_in[b];
                rv[j] = rstd_in[b];
                dv[j] = dxn[(int64_t)b * d + k];
                gv[j] = to_f32(dtok[(int64_t)b * N * d + k]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (b0 + 8 * j < B) {
                    sg = fmaf(dv[j], (xv[j] - mv[j]) * rv[j], sg);
                    sb += dv[j];
                    sc += gv[j];
                }
            }
        }
    }
    red[0][ty][tx] = sg; red[1][ty][tx] = sb; red[2][ty][tx] = sc;
    __syncthreads();
    if (ty == 0 && k < d) {
        float a = 0.f, bsum = 0.f, c = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) { a += red[0][y][tx]; bsum += red[1][y][tx]; c += red[2][y][tx]; }
        dgamma[k] += a;
        dbeta[k] += bsum;
        if (dcolsum != nullptr) dcolsum[k] += c;
    }
}

// backward C: dW[c,k] += sum_b dlogits[b,c] xn[b,k];  db[c] += sum_b dlogits[b,c]
// grid (d/32, n_class), block = 32 columns x 8 sample groups
__global__ void __launch_bounds__(256) head_bwd_weight_kernel(const float *__restrict__ dlog,
                                                               const float *__restrict__ xn, float *__restrict__ dw,
                                                               float *__restrict__ db, int B, int d, int n_class) {
    __shared__ float red[2][8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int cls = blockIdx.y;
    const int k = blockIdx.x * 32 + tx;
    float s = 0.f, sb = 0.f;
    if (k < d) {
        for (int b = ty; b < B; b += 8) {
            const float dl = dlog[(int64_t)b * n_class + cls];
            s = fmaf(dl, xn[(int64_t)b * d + k], s);
            sb += dl;
        }
    }
    red[0][ty][tx] = s; red[1][ty][tx] = sb;
    __syncthreads();
    if (ty == 0 && k < d) {
        float a = 0.f, bsum = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) { a += red[0][y][tx]; bsum += red[1][y][tx]; }
        dw[(int64_t)cls * d + k] += a;
        if (k == 0) db[cls] += bsum;
    }
}

// Mean pool (vit_pytorch pool='mean'): out[b, k] = sum_t tok[b, t, k] / N over all N tokens, CLS included.
// One CTA = one record x 256 columns; thread (tx, ty) sums 8 columns over the rows t = ty, ty + 8, ... in order, and the
// 8 row groups are folded in order: a fixed summation order, no atomics, so the result is bit-identical run to run.
constexpr int MEAN_ROWG = 8;
template <typename T>
__global__ void __launch_bounds__(32 * MEAN_ROWG) token_mean_kernel(const T *__restrict__ tok, float *__restrict__ out,
                                                                     int N, int d) {
    __shared__ float red[MEAN_ROWG][256 + 8];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int b = blockIdx.y;
    const int c = blockIdx.x * 256 + tx * 8;
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c < d) {
        const T *xr = tok + (int64_t)b * N * d + c;
        for (int t = ty; t < N; t += MEAN_ROWG) {
            float v[8];
            load8(xr + (int64_t)t * d, v);
#pragma unroll
            for (int k = 0; k < 8; ++k) s[k] += v[k];
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[ty][tx * 8 + k] = s[k];
    __syncthreads();
    if (ty == 0 && c < d) {
        float o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float a = red[0][tx * 8 + k];
#pragma unroll
            for (int y = 1; y < MEAN_ROWG; ++y) a += red[y][tx * 8 + k];
            o[k] = a / (float)N;
        }
        store8(out + (int64_t)b * d + c, o);
    }
}

// its backward: dtok[b, t, :] = dpool[b, :] / N for every token t
template <typename T>
__global__ void __launch_bounds__(256) token_mean_bwd_kernel(const float *__restrict__ dpool, T *__restrict__ dtok,
                                                              int B, int N, int d) {
    const int dv = d / 8;
    const int64_t total = (int64_t)B * N * dv;
    const float inv = 1.0f / (float)N;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % dv) * 8;
        const int64_t row = i / dv;
        const int b = (int)(row / N);
        float v[8];
        load8(dpool + (int64_t)b * d + c, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] *= inv;
        store8(dtok + row * d + c, v);
    }
}

}  // namespace
}  // namespace ecgvit

using namespace ecgvit;

extern "C" {

int ecgvit_head_fwd(const void *tok, const float *gamma, const float *beta, const float *w, const float *b,
                    const float *labels, const float *loss_weight, int n_weight, float *xn, float *mean, float *rstd,
                    float *logits, float *loss, int B, int N, int d, int n_class, int reduction, float eps, int dtype,
                    void *stream) {
    ECGVIT_REQUIRE(tok && gamma && beta && w && b && xn && mean && rstd && logits, "head_fwd: null argument");
    ECGVIT_REQUIRE(B > 0 && N > 0 && n_class > 0, "head_fwd: bad sizes");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * HEAD_MAXV, "head_fwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * HEAD_MAXV);
    ECGVIT_REQUIRE(labels == nullptr || loss != nullptr, "head_fwd: labels given but loss is null");
    ECGVIT_REQUIRE(loss_weight == nullptr || n_weight >= 1, "head_fwd: loss_weight table needs n_weight >= 1");
    const dim3 grid((B + HEAD_SPB - 1) / HEAD_SPB, 3);           // 3 class groups per sample group
    const size_t smem = (size_t)HEAD_SPB * d * sizeof(float);   // <= 32 KB
    if (dtype == ECGVIT_BF16)
        head_fwd_kernel<bf16><<<grid, 32 * HEAD_SPB, smem, as_stream(stream)>>>((const bf16 *)tok, gamma, beta, w, b, xn, mean, rstd, logits, B, N, d, n_class, eps);
    else if (dtype == ECGVIT_F32 || dtype == ECGVIT_BF16_RES32)   // fp32 tokens (parity mode / fp32 residual stream)
        head_fwd_kernel<float><<<grid, 32 * HEAD_SPB, smem, as_stream(stream)>>>((const float *)tok, gamma, beta, w, b, xn, mean, rstd, logits, B, N, d, n_class, eps);
    else return fail(-1, "head_fwd: unknown dtype %d", dtype);
    int rc = check_launch("head_fwd");
    if (rc) return rc;
    if (labels != nullptr) {
        bce_loss_kernel<<<1, 1024, 0, as_stream(stream)>>>(logits, labels, loss, B * n_class, reduction, loss_weight,
                                                              n_weight);
        rc = check_launch("bce_loss");
    }
    return rc;
}

int ecgvit_head_bwd(const void *tok, const float *gamma, const float *w, const float *labels, const float *loss_weight,
                    int n_weight, const float *xn, const float *mean, const float *rstd, const float *logits, void *dtok,
                    float *dw, float *db,
                    float *dgamma, float *dbeta, float *dcolsum, float *scratch, int B, int N, int d, int n_class,
                    int reduction, float grad_scale, const float *grad_scale_dev, int dtype, void *stream) {
    ECGVIT_REQUIRE(tok && gamma && w && labels && xn && mean && rstd && logits && dtok && dw && db && dgamma &&
                       dbeta && scratch,
                   "head_bwd: null argument");
    ECGVIT_REQUIRE(reduction == ECGVIT_REDUCTION_MEAN || reduction == ECGVIT_REDUCTION_SUM,
                   "head_bwd: reduction must be mean or sum");
    ECGVIT_REQUIRE(loss_weight == nullptr || n_weight >= 1, "head_bwd: loss_weight table needs n_weight >= 1");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * HEAD_MAXV, "head_bwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * HEAD_MAXV);
    cudaStream_t s = as_stream(stream);
    const size_t esz = dtype == ECGVIT_F32 ? 4 : 2;   // dtok is bf16 in both bf16 modes
    cudaError_t e = cudaMemsetAsync(dtok, 0, (size_t)B * N * d * esz, s);
    if (e != cudaSuccess) return fail((int)e, "head_bwd: memset: %s", cudaGetErrorString(e));
    const float coef = grad_scale * (reduction == ECGVIT_REDUCTION_MEAN ? 1.0f / ((float)B * (float)n_class) : 1.0f);
    float *dxn = scratch, *dlog = scratch + (size_t)B * d;
    const int grid = (B + HEAD_SPB - 1) / HEAD_SPB;
    // as many weight rows per shared-memory chunk as fit in 216 KB (all of them up to d = 768 x 71 classes)
    const int ch_classes = std::min(n_class, (216 * 1024) / (d * (int)sizeof(float)));
    const size_t smem_rows = (size_t)ch_classes * d * sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        const int max_smem = 216 * 1024;
        cudaFuncSetAttribute(head_bwd_rows_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        cudaFuncSetAttribute(head_bwd_rows_kernel<bf16, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        cudaFuncSetAttribute(head_bwd_rows_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        attr_set = true;
    }
    if (dtype == ECGVIT_BF16) {
        head_bwd_rows_kernel<bf16><<<grid, 32 * HEAD_SPB, smem_rows, s>>>((const bf16 *)tok, gamma, w, labels, mean, rstd, logits, (bf16 *)dtok, dxn, dlog, B, N, d, n_class, coef, grad_scale_dev, loss_weight, n_weight, ch_classes);
        head_bwd_cols_kernel<bf16><<<(d + 31) / 32, 256, 0, s>>>((const bf16 *)tok, (const bf16 *)dtok, dxn, mean, rstd, dgamma, dbeta, dcolsum, B, N, d);
    } else if (dtype == ECGVIT_BF16_RES32) {
        head_bwd_rows_kernel<bf16, float><<<grid, 32 * HEAD_SPB, smem_rows, s>>>((const float *)tok, gamma, w, labels, mean, rstd, logits, (bf16 *)dtok, dxn, dlog, B, N, d, n_class, coef, grad_scale_dev, loss_weight, n_weight, ch_classes);
        head_bwd_cols_kernel<bf16, float><<<(d + 31) / 32, 256, 0, s>>>((const float *)tok, (const bf16 *)dtok, dxn, mean, rstd, dgamma, dbeta, dcolsum, B, N, d);
    } else if (dtype == ECGVIT_F32) {
        head_bwd_rows_kernel<float><<<grid, 32 * HEAD_SPB, smem_rows, s>>>((const float *)tok, gamma, w, labels, mean, rstd, logits, (float *)dtok, dxn, dlog, B, N, d, n_class, coef, grad_scale_dev, loss_weight, n_weight, ch_classes);
        head_bwd_cols_kernel<float><<<(d + 31) / 32, 256, 0, s>>>((const float *)tok, (const float *)dtok, dxn, mean, rstd, dgamma, dbeta, dcolsum, B, N, d);
    } else return fail(-1, "head_bwd: unknown dtype %d", dtype);
    dim3 gw((d + 31) / 32, n_class);
    head_bwd_weight_kernel<<<gw, 256, 0, s>>>(dlog, xn, dw, db, B, d, n_class);
    return check_launch("head_bwd");
}

int ecgvit_token_mean(const void *tok, float *out, int B, int N, int d, int dtype, void *stream) {
    ECGVIT_REQUIRE(tok && out && B > 0 && N > 0 && d > 0, "token_mean: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "token_mean: d=%d must be a multiple of 8", d);
    const dim3 grid((d + 255) / 256, B);
    if (dtype == ECGVIT_BF16)
        token_mean_kernel<bf16><<<grid, 32 * MEAN_ROWG, 0, as_stream(stream)>>>((const bf16 *)tok, out, N, d);
    else if (dtype == ECGVIT_F32 || dtype == ECGVIT_BF16_RES32)   // fp32 tokens (parity mode / fp32 residual stream)
        token_mean_kernel<float><<<grid, 32 * MEAN_ROWG, 0, as_stream(stream)>>>((const float *)tok, out, N, d);
    else return fail(-1, "token_mean: unknown dtype %d", dtype);
    return check_launch("token_mean");
}

int ecgvit_token_mean_bwd(const float *dpool, void *dtok, int B, int N, int d, int dtype, void *stream) {
    ECGVIT_REQUIRE(dpool && dtok && B > 0 && N > 0 && d > 0, "token_mean_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "token_mean_bwd: d=%d must be a multiple of 8", d);
    const int64_t vecs = (int64_t)B * N * (d / 8);
    const int grid = (int)std::min<int64_t>((vecs + 255) / 256, (int64_t)sm_count() * 8);
    if (dtype == ECGVIT_BF16 || dtype == ECGVIT_BF16_RES32)   // the token-shaped gradient is bf16 in both bf16 modes
        token_mean_bwd_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>(dpool, (bf16 *)dtok, B, N, d);
    else if (dtype == ECGVIT_F32)
        token_mean_bwd_kernel<float><<<grid, 256, 0, as_stream(stream)>>>(dpool, (float *)dtok, B, N, d);
    else return fail(-1, "token_mean_bwd: unknown dtype %d", dtype);
    return check_launch("token_mean_bwd");
}

}  // extern "C"

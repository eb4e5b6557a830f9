// HBM-bound kernels of the ECG-ViT step: patch gather, CLS/pos assemble, LayerNorm fwd/bwd, column sums, casts.
// All use 128-bit accesses and warp-shuffle reductions; statistics are fp32.
#include "common.cuh"

#include <stdlib.h>

namespace ecgvit {

namespace {

// ---------------------------------------------------------------------------------------------------
// patchify: a[(b*n+w), t*C+c] = x[b, c, w*P+t]     (einops 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)', h=p1=1)
// with the reference's input pipeline optionally fused in front of it (preprocess/transform.py, applied per record by
// EcgDataset.__getitem__ in this order): Normalize (x - mean[c]) / std[c]  ->  TimeEndPad (zeros from L_valid on)  ->
// TimeOut (zeros on [start, start + len) of every lead of sample b).  IEEE subtract / divide, so fp32 results are
// bit-identical to numpy's; the transformed signal itself is never written to memory.
//
// One CTA per (sample, group of WG consecutive windows): every lead contributes WG * P contiguous samples (coalesced
// reads, four leads in flight per thread), the group is transposed through shared memory into output order, and because
// the WG output rows are adjacent in `a` they leave as one contiguous run of 16-byte stores.  (One CTA per window with
// an integer division per element and 2-byte stores took 24 us for 46 MB.)
template <typename T>
__global__ void __launch_bounds__(256) patchify_kernel(const float *__restrict__ x, const float *__restrict__ mean,
                                                        const float *__restrict__ stdev, const int *__restrict__ spans,
                                                        T *__restrict__ a, int C, int64_t x_ld, int L_valid, int n_patch,
                                                        int P, int WG, float inv_P) {
    extern __shared__ float tile[];  // [WG][P*C] in output order
    const int groups = (n_patch + WG - 1) / WG;
    const int b = blockIdx.x / groups;
    const int w0 = (blockIdx.x - b * groups) * WG;
    const int nw = min(WG, n_patch - w0);
    const int PC = P * C;
    const int span = nw * P;  // time steps of this group
    const float *xb = x + (int64_t)b * C * x_ld;
    int cut0 = 0, cut1 = 0;  // zeroed span of this sample
    if (spans != nullptr) {
        cut0 = spans[2 * b];
        cut1 = cut0 + spans[2 * b + 1];
    }
    for (int tt = threadIdx.x; tt < span; tt += blockDim.x) {
        const int pos = w0 * P + tt;
        const int wl = __float2int_rd(((float)tt + 0.5f) * inv_P);  // tt / P (exact: tt + 0.5 is never within 0.5 / P of a multiple)
        const int t = tt - wl * P;
        const bool live = pos < L_valid && !(pos >= cut0 && pos < cut1);
        float *dst = tile + wl * PC + t * C;
        for (int c0 = 0; c0 < C; c0 += 4) {
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {   // branch-free: all four loads are issued before the first use
                const int c = min(c0 + j, C - 1);
                v[j] = xb[(int64_t)c * x_ld + (live ? pos : 0)];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + j;
                if (c < C) {
                    float r = 0.f;
                    if (live) r = mean != nullptr ? __fdiv_rn(__fsub_rn(v[j], mean[c]), stdev[c]) : v[j];
                    dst[c] = r;
                }
            }
        }
    }
    __syncthreads();
    const int total = nw * PC;
    T *out = a + ((int64_t)b * n_patch + w0) * PC;
    if ((PC & 7) == 0) {   // every group starts 16-byte aligned
        for (int i = threadIdx.x * 8; i < total; i += blockDim.x * 8) {
            float v[8];
            load8(tile + i, v);
            store8(out + i, v);
        }
    } else {
        for (int i = threadIdx.x; i < total; i += blockDim.x) out[i] = from_f32<T>(tile[i]);
    }
}

// per-lead tokens (BASELINE.json configs[3]: vit_pytorch ViT(image_size=(C, L), patch_size=(1, P), channels=1) fed
// [B, 1, C, L]): token (c, w) of record b holds the P samples x[b, c, w*P : (w+1)*P]; rows are padded with zeros to Kp
// features (a multiple of 8) so the embedding GEMM's operand rows stay 16-byte aligned.  Same optional transforms as
// patchify_transform_kernel.  One thread per output element.
template <typename T>
__global__ void patchify_leads_kernel(const float *__restrict__ x, const float *__restrict__ mean,
                                      const float *__restrict__ stdev, const int *__restrict__ spans,
                                      T *__restrict__ a, int64_t total, int C, int64_t x_ld, int L_valid, int n_w, int P,
                                      int Kp) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int t = (int)(i % Kp);
        const int64_t tok = i / Kp;  // (b * C + c) * n_w + w
        const int w = (int)(tok % n_w);
        const int64_t bc = tok / n_w;
        const int c = (int)(bc % C);
        const int64_t b = bc / C;
        const int pos = w * P + t;
        float v = 0.f;
        if (t < P && pos < L_valid) {
            bool cut = false;
            if (spans != nullptr) {
                const int s0 = spans[2 * b];
                cut = pos >= s0 && pos < s0 + spans[2 * b + 1];
            }
            if (!cut) {
                v = x[bc * x_ld + pos];
                if (mean != nullptr) v = __fdiv_rn(__fsub_rn(v, mean[c]), stdev[c]);
            }
        }
        a[i] = from_f32<T>(v);
    }
}

// dst[r, 0:cols_padded] = src[r, 0:cols] followed by zeros
template <typename T>
__global__ void pad_cols_kernel(const T *__restrict__ src, T *__restrict__ dst, int64_t rows, int cols, int cols_padded) {
    const int64_t total = rows * cols_padded;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cols_padded);
        const int64_t r = i / cols_padded;
        dst[i] = c < cols ? src[r * cols + c] : from_f32<T>(0.f);
    }
}
// dst[r, c] += src[r, c] for c < cols (src rows are cols_padded long)
__global__ void unpad_add_kernel(const float *__restrict__ src, float *__restrict__ dst, int64_t rows, int cols,
                                 int cols_padded) {
    const int64_t total = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cols);
        const int64_t r = i / cols;
        dst[i] += src[r * cols_padded + c];
    }
}

// ---------------------------------------------------------------------------------------------------
// tok[b,0,:] = cls + pos[0];  tok[b,1+w,:] = e[b*n+w,:] + pos[1+w,:]
// kMasked: rows with mask[b*n+w] != 0 take mask_token instead of e (masked-patch pre-training)
// kVisible: n_patch is the number of VISIBLE patches of every record (MAE encoder); row 1+j of record b takes
// e[b*n_patch+j] and pos[1 + vis_idx[b*n_patch+j]]
template <typename T, typename TO, bool kMasked = false, bool kVisible = false>
__global__ void embed_assemble_kernel(const T *__restrict__ e, const float *__restrict__ cls,
                                      const float *__restrict__ pos, TO *__restrict__ tok, int B, int n_patch, int d,
                                      DropoutParams drop, const float *__restrict__ mask_token = nullptr,
                                      const uint8_t *__restrict__ mask = nullptr,
                                      const int *__restrict__ vis_idx = nullptr) {
    if constexpr (kVisible) {
        pdl_launch_dependents();
        pdl_wait();
    }
    const bool dropping = drop.threshold != 0;
    const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
    const int N = n_patch + 1;
    const int vec_per_row = d / 8;
    const int64_t total = (int64_t)B * N * vec_per_row;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % vec_per_row) * 8;
        const int64_t r = i / vec_per_row;
        const int j = (int)(r % N);
        const int64_t b = r / N;
        float v[8], p[8];
        if constexpr (kVisible) load8(pos + (int64_t)(j == 0 ? 0 : 1 + vis_idx[b * n_patch + (j - 1)]) * d + c, p);
        else load8(pos + (int64_t)j * d + c, p);
        if (j == 0) load8(cls + c, v);
        else if (kMasked && mask[b * n_patch + (j - 1)] != 0) load8(mask_token + c, v);
        else load8(e + (b * n_patch + (j - 1)) * d + c, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] += p[k];
        if (dropping) dropout_apply<8>(drop, seed, static_cast<uint32_t>(r * d + c), v);
        store8(tok + r * d + c, v);
    }
}

// backward: grid (token position j, 256-column slab), block = 32 lanes x 8 columns each x 8 batch groups; the masked
// gradient rows are copied to `de` on the way (16-byte accesses, one dropout hash per pair) and the batch sums are folded
// through shared memory.  (One 2-byte element per thread with a hash per element was instruction bound: 22 us for 40 MB.)
// kMasked: masked rows (mask[b*n+w] != 0) send their gradient to dmask_token instead of de / dbias (de rows are zeroed)
// kVisible (MAE encoder, n_vis visible patches per record, dtok [B*(n_vis+1), d], de [B*n_vis, d]): blockIdx.x is the
// patch POSITION p (0 = CLS); record b contributes its token row 1 + slot[b*n_patch+p-1] when that patch is visible.
// Instead of the atomic bias add, the position's sum goes to pos_sums[p-1] for a fixed-order fold (no float atomics).
template <typename T, bool kMasked = false, bool kVisible = false>
__global__ void __launch_bounds__(256) embed_assemble_bwd_kernel(const T *__restrict__ dtok, T *__restrict__ de,
                                                                  float *__restrict__ dcls, float *__restrict__ dpos,
                                                                  float *__restrict__ dbias, int B, int n_patch, int d,
                                                                  DropoutParams drop,
                                                                  const uint8_t *__restrict__ mask = nullptr,
                                                                  float *__restrict__ dmask_token = nullptr,
                                                                  const int *__restrict__ slot = nullptr, int n_vis = 0,
                                                                  float *__restrict__ pos_sums = nullptr) {
    __shared__ float red[kMasked ? 16 : 8][256 + 8];
    if constexpr (kVisible) {
        pdl_launch_dependents();
        pdl_wait();
    }
    const int N = kVisible ? n_vis + 1 : n_patch + 1;
    const int n_e = kVisible ? n_vis : n_patch;   // rows of de per record
    const int p_blk = blockIdx.x;
    const int j = kVisible ? 0 : p_blk;   // token row (per record under kVisible, see row_of)
    // token row of record b at this block's position, -1 when the patch is masked
    auto row_of = [&](int b) -> int {
        if constexpr (kVisible) return p_blk == 0 ? 0 : (slot[(int64_t)b * n_patch + (p_blk - 1)] >= 0 ?
                                                         1 + slot[(int64_t)b * n_patch + (p_blk - 1)] : -1);
        else return j;
    };
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int col = (blockIdx.y * 32 + tx) * 8;
    const bool dropping = drop.threshold != 0;
    const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
    float s[8], sm[8];   // sums of the visible rows (all rows without kMasked) / of the masked rows
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = sm[k] = 0.f;
    if (col < d) {
        // two samples in flight per thread (rows N * d elements apart)
        for (int b0 = ty; b0 < B; b0 += 16) {
            float gv[2][8];
            int jq[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int bq = min(b0 + 8 * q, B - 1);
                jq[q] = row_of(bq);
                if (!kVisible || jq[q] >= 0) load8(dtok + ((int64_t)bq * N + jq[q]) * d + col, gv[q]);
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int b = b0 + 8 * q;
                if (b < B && (!kVisible || jq[q] >= 0)) {
                    const int j = jq[q];
                    const int64_t idx = ((int64_t)b * N + j) * d + col;
                    if (dropping) dropout_apply<8>(drop, seed, static_cast<uint32_t>(idx), gv[q]);
                    if (kMasked && j > 0 && mask[(int64_t)b * n_patch + (j - 1)] != 0) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            sm[k] += to_f32(from_f32<T>(gv[q][k]));
                            gv[q][k] = 0.f;
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            gv[q][k] = to_f32(from_f32<T>(gv[q][k]));   // the sums are those of the rounded rows
                            s[k] += gv[q][k];
                        }
                    }
                    if (j > 0) store8(de + ((int64_t)b * n_e + (j - 1)) * d + col, gv[q]);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[ty][tx * 8 + k] = s[k];
    if (kMasked) {
#pragma unroll
        for (int k = 0; k < 8; ++k) red[8 + ty][tx * 8 + k] = sm[k];
    }
    __syncthreads();
    const int c = blockIdx.y * 256 + threadIdx.x;   // one column per thread for the fold
    if (c < d) {
        float t = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) t += red[y][threadIdx.x];
        if (kMasked) {
            float tm = 0.f;
#pragma unroll
            for (int y = 0; y < 8; ++y) tm += red[8 + y][threadIdx.x];
            dpos[(int64_t)j * d + c] += t + tm;
            if (j == 0) dcls[c] += t;
            else {
                atomicAdd(dbias + c, t);
                atomicAdd(dmask_token + c, tm);
            }
        } else if constexpr (kVisible) {
            dpos[(int64_t)p_blk * d + c] += t;
            if (p_blk == 0) dcls[c] += t;
            else pos_sums[(int64_t)(p_blk - 1) * d + c] = t;
        } else {
            dpos[(int64_t)j * d + c] += t;
            if (j == 0) dcls[c] += t;
            else atomicAdd(dbias + c, t);
        }
    }
}

// Column sums of an fp32 [rows, d] scratch in a fixed order, in two launches (bit-identical from launch to launch; the
// deterministic second half of the visible-assemble and unshuffle backward):
//   chunk pass: CTA (column slab x, chunk g) sums rows [g * kFoldChunk, (g + 1) * kFoldChunk) over 32 row groups and
//               a fixed fold, and writes the sum over the chunk's FIRST row (only this CTA reads that chunk);
//   final pass: one CTA per column slab folds the chunk sums (rows 0, kFoldChunk, 2 kFoldChunk, ...) into out.
// fold_rows_kernel is both: rows are r * row_stride, and out == nullptr selects the chunk pass.
constexpr int kFoldGroups = 32;
constexpr int kFoldChunk = 128;
__global__ void __launch_bounds__(32 * kFoldGroups) fold_rows_kernel(float *__restrict__ S, int rows, int row_stride,
                                                                     int d, float *__restrict__ out) {
    __shared__ float red[kFoldGroups][33];
    pdl_launch_dependents();
    pdl_wait();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    const int r0 = out == nullptr ? blockIdx.y * kFoldChunk : 0;
    const int r1 = out == nullptr ? min(r0 + kFoldChunk, rows) : rows;
    float s = 0.f;
    if (c < d)
        for (int r = r0 + ty; r < r1; r += kFoldGroups) s += S[(int64_t)r * row_stride * d + c];
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < d) {
        float t = 0.f;
#pragma unroll
        for (int y = 0; y < kFoldGroups; ++y) t += red[y][tx];
        if (out == nullptr) S[(int64_t)r0 * d + c] = t;
        else out[c] += t;
    }
}

// MAE decoder input: u[b, 0] = t[b, 0] + pos[0]; u[b, 1+p] = (slot[b, p] >= 0 ? t[b, 1 + slot[b, p]] : mask_token)
// + pos[1+p], with t [B*(n_vis+1), d] and u [B*(n_patch+1), d]
template <typename T, typename TO>
__global__ void mae_unshuffle_kernel(const T *__restrict__ t, const float *__restrict__ mask_token,
                                     const float *__restrict__ pos, const int *__restrict__ slot, TO *__restrict__ u,
                                     int B, int n_patch, int n_vis, int d) {
    pdl_launch_dependents();
    pdl_wait();
    const int N = n_patch + 1, Nv = n_vis + 1;
    const int vec_per_row = d / 8;
    const int64_t total = (int64_t)B * N * vec_per_row;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % vec_per_row) * 8;
        const int64_t r = i / vec_per_row;
        const int p = (int)(r % N);
        const int64_t b = r / N;
        float v[8], q[8];
        load8(pos + (int64_t)p * d + c, q);
        const int s = p == 0 ? -1 : slot[b * n_patch + (p - 1)];
        if (p == 0) load8(t + b * Nv * d + c, v);
        else if (s >= 0) load8(t + (b * Nv + 1 + s) * d + c, v);
        else load8(mask_token + c, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] += q[k];
        store8(u + r * d + c, v);
    }
}

// its backward: grid (position p, 256-column slab), block = 32 lanes x 8 columns x 8 record groups.  dt rows are
// copied from du (every row of t feeds exactly one row of u); dpos[p] += sum_b du[b, p]; the masked rows' sum of
// position p goes to mask_sums[p-1] for the fixed-order fold into the mask-token gradient.
template <typename T>
__global__ void __launch_bounds__(256) mae_unshuffle_bwd_kernel(const T *__restrict__ du, const int *__restrict__ slot,
                                                                 T *__restrict__ dt, float *__restrict__ dpos,
                                                                 float *__restrict__ mask_sums, int B, int n_patch,
                                                                 int n_vis, int d) {
    __shared__ float red[16][256 + 8];
    pdl_launch_dependents();
    pdl_wait();
    const int N = n_patch + 1, Nv = n_vis + 1;
    const int p = blockIdx.x;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int col = (blockIdx.y * 32 + tx) * 8;
    float s[8], sm[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = sm[k] = 0.f;
    if (col < d) {
        for (int b = ty; b < B; b += 8) {
            float g[8];
            load8(du + ((int64_t)b * N + p) * d + col, g);
            const int sl = p == 0 ? 0 : slot[(int64_t)b * n_patch + (p - 1)];
#pragma unroll
            for (int k = 0; k < 8; ++k) s[k] += g[k];
            if (p == 0) store8(dt + (int64_t)b * Nv * d + col, g);
            else if (sl >= 0) store8(dt + ((int64_t)b * Nv + 1 + sl) * d + col, g);
            else {
#pragma unroll
                for (int k = 0; k < 8; ++k) sm[k] += g[k];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        red[ty][tx * 8 + k] = s[k];
        red[8 + ty][tx * 8 + k] = sm[k];
    }
    __syncthreads();
    const int c = blockIdx.y * 256 + threadIdx.x;
    if (c < d) {
        float a = 0.f, am = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) {
            a += red[y][threadIdx.x];
            am += red[8 + y][threadIdx.x];
        }
        dpos[(int64_t)p * d + c] += a;
        if (p > 0) mask_sums[(int64_t)(p - 1) * d + c] = am;
    }
}

// zeros the CLS rows (b * N, b = 0..B-1) of a token-shaped [B*N, d] matrix
template <typename T>
__global__ void zero_cls_rows_kernel(T *__restrict__ tok, int B, int N, int d) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)B * d; i += (int64_t)gridDim.x * blockDim.x)
        tok[(i / d) * N * d + (i % d)] = from_f32<T>(0.f);
}

constexpr int LN_MAXV = 4;  // 4 x 8 elements per lane


// LayerNorm backward (+ residual-gradient add, + column sums of the result for the bias gradient upstream).
// One warp per row, NV 8-element vectors per lane (d <= 256 * NV).  The three inputs of a row (dy, x, dres) are fetched
// together and kept PACKED in registers (their fp32 expansions are recomputed in the second pass), gamma is read from
// shared memory, so that with the 3 x 8 x NV per-lane column accumulators the kernel still fits 2 CTAs (16 warps) per
// SM: this kernel lives on memory-level parallelism.
template <typename T> struct Packed8;
template <> struct Packed8<bf16> { uint4 v; };
template <> struct Packed8<float> { float4 a, b; };
__device__ __forceinline__ void ld_packed(Packed8<bf16> &p, const bf16 *src) { p.v = *reinterpret_cast<const uint4 *>(src); }
__device__ __forceinline__ void ld_packed(Packed8<float> &p, const float *src) {
    p.a = *reinterpret_cast<const float4 *>(src);
    p.b = *reinterpret_cast<const float4 *>(src + 4);
}
__device__ __forceinline__ void unpack(const Packed8<bf16> &p, float v[8]) {
    unpack_bf16x2(p.v.x, v[0], v[1]); unpack_bf16x2(p.v.y, v[2], v[3]);
    unpack_bf16x2(p.v.z, v[4], v[5]); unpack_bf16x2(p.v.w, v[6], v[7]);
}
__device__ __forceinline__ void unpack(const Packed8<float> &p, float v[8]) {
    v[0] = p.a.x; v[1] = p.a.y; v[2] = p.a.z; v[3] = p.a.w; v[4] = p.b.x; v[5] = p.b.y; v[6] = p.b.z; v[7] = p.b.w;
}

// 8 packed elements -> four fp32x2 pairs
__device__ __forceinline__ void unpack_pairs(const Packed8<bf16> &p, uint64_t v[4]) {
    const uint32_t w[4] = {p.v.x, p.v.y, p.v.z, p.v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = pack2(__uint_as_float(w[k] << 16), __uint_as_float(w[k] & 0xffff0000u));
}
__device__ __forceinline__ void unpack_pairs(const Packed8<float> &p, uint64_t v[4]) {
    v[0] = pack2(p.a.x, p.a.y); v[1] = pack2(p.a.z, p.a.w); v[2] = pack2(p.b.x, p.b.y); v[3] = pack2(p.b.z, p.b.w);
}
__device__ __forceinline__ void store_pairs(bf16 *dst, const uint64_t v[4]) {
    uint4 u;
    float a, b;
    unpack2(v[0], a, b); u.x = pack_bf16x2(a, b);
    unpack2(v[1], a, b); u.y = pack_bf16x2(a, b);
    unpack2(v[2], a, b); u.z = pack_bf16x2(a, b);
    unpack2(v[3], a, b); u.w = pack_bf16x2(a, b);
    *reinterpret_cast<uint4 *>(dst) = u;
}
__device__ __forceinline__ void store_pairs(float *dst, const uint64_t v[4]) {
    float a, b, c, d;
    unpack2(v[0], a, b); unpack2(v[1], c, d);
    *reinterpret_cast<float4 *>(dst) = make_float4(a, b, c, d);
    unpack2(v[2], a, b); unpack2(v[3], c, d);
    *reinterpret_cast<float4 *>(dst + 4) = make_float4(a, b, c, d);
}
__device__ __forceinline__ float pair_sum(uint64_t v) {
    float a, b;
    unpack2(v, a, b);
    return a + b;
}

// LayerNorm forward: one warp per row, NV 8-element vectors per lane (d <= 256 * NV), packed fp32x2 math, two-pass
// statistics (mean, then centred sum of squares) like ATen.  Persistent: MINB CTAs per SM, every warp walks its rows with
// gamma / beta held in registers for the whole kernel and the NEXT row's loads in flight while the current row is reduced
// (the kernel is latency bound: a row is load -> two shuffle reductions -> store, and the first version re-read gamma /
// beta from L1 for every row and had nothing in flight during the reductions: 19.5 us for 40 MB in the round-1 profile).
// kPatch: output row i reads input row i + i / n_patch + 1 (the patch rows of a [B*(n_patch+1), d] token matrix)
template <typename T, int NV, int R, int MINB, typename TX = T, bool kPatch = false>
__global__ void __launch_bounds__(256, MINB) layernorm_fwd_kernel(const TX *__restrict__ x, const float *__restrict__ gamma,
                                                             const float *__restrict__ beta, T *__restrict__ y,
                                                             float *__restrict__ mean_out, float *__restrict__ rstd_out,
                                                             int M, int d, float eps, int n_patch) {
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t total_warps = (int64_t)gridDim.x * warps_per_block;
    const float inv_d = 1.0f / (float)d;
    // parameters: not produced by the previous kernel, so they are fetched before the dependency wait
    uint64_t g2[NV][4], b2[NV][4];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int c = (i * 32 + lane) * 8;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            g2[i][k] = c < d ? __ldg(reinterpret_cast<const uint64_t *>(gamma + c) + k) : 0ull;
            b2[i][k] = c < d ? __ldg(reinterpret_cast<const uint64_t *>(beta + c) + k) : 0ull;
        }
    }
    pdl_wait();
    int64_t row = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    Packed8<TX> cur[NV], nxt[NV];
    if (row < M) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) ld_packed(cur[i], x + (kPatch ? row + row / n_patch + 1 : row) * d + c);
        }
    }
    for (; row < M; row += total_warps) {
        const int64_t row_n = row + total_warps;
        if (row_n < M) {
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int c = (i * 32 + lane) * 8;
                if (c < d) ld_packed(nxt[i], x + (kPatch ? row_n + row_n / n_patch + 1 : row_n) * d + c);
            }
        }
        uint64_t v[NV][4];
        uint64_t s2 = 0ull;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) {
                unpack_pairs(cur[i], v[i]);
#pragma unroll
                for (int k = 0; k < 4; ++k) s2 = add2(s2, v[i][k]);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) v[i][k] = 0ull;
            }
        }
        const float mean = warp_sum(pair_sum(s2)) * inv_d;
        const uint64_t nmean2 = splat2(-mean);
        uint64_t sq2 = 0ull;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    v[i][k] = add2(v[i][k], nmean2);  // centred
                    sq2 = fma2(v[i][k], v[i][k], sq2);
                }
            }
        }
        const float rstd = rsqrtf(warp_sum(pair_sum(sq2)) * inv_d + eps);
        const uint64_t rstd2 = splat2(rstd);
        T *yr = y + row * d;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) {
                uint64_t o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) o[k] = fma2(mul2(v[i][k], rstd2), g2[i][k], b2[i][k]);
                store_pairs(yr + c, o);
            }
        }
        if (lane == 0) {
            if (mean_out) mean_out[row] = mean;
            if (rstd_out) rstd_out[row] = rstd;
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) cur[i] = nxt[i];
    }
}

// All per-element math runs on packed fp32x2 (FFMA2 / FADD2 / FMUL2): ~11 issue slots per element instead of ~25.
//   dx = dy * (rstd * gamma) + x * B + C,  B = -rstd^2 * s2,  C = rstd * (mean * rstd * s2 - s1)
//   with s1 = mean_c(dy * gamma), s2 = mean_c(dy * gamma * xhat)
// kDrop: dx feeds a Linear through a dropout (to_out[1] / net[4] of the block below): additionally write
// dxm = mask * dx / (1 - p) (that Linear's dgrad / wgrad operand) and make the column sums those of dxm (its bias grad).
// kPatch: dy / mean / rstd are compact patch rows; x is read from, and dx written to, token row i + i / n_patch + 1
// kPath (with kDrop): drop path on the branch as well: dxm = s[row / rows_per_record] * mask * dx, where the element mask
// is all ones when drop.threshold == 0
template <typename T, int NV, bool kDrop, typename TX = T, bool kPatch = false, bool kPath = false>
__global__ void __launch_bounds__(256, 1) layernorm_bwd_kernel(const T *__restrict__ dy, const TX *__restrict__ x,
                                                                const float *__restrict__ gamma,
                                                                const float *__restrict__ mean_in,
                                                                const float *__restrict__ rstd_in, const T *dres, T *dx,
                                                                float *__restrict__ dgamma, float *__restrict__ dbeta,
                                                                float *__restrict__ dcolsum, float *__restrict__ partial,
                                                                int M, int d, T *__restrict__ dxm,
                                                                DropParamsFor<kPath> drop, int n_patch) {
    extern __shared__ float red[];  // [warps][3][d] column partials, then [NV * 256] permuted gamma
    pdl_launch_dependents();
    pdl_wait();
    float *sgamma = red + (blockDim.x >> 5) * 3 * d;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int warps_per_block = blockDim.x >> 5;
    const float inv_d = 1.0f / (float)d;

    uint64_t acc_g[NV][4], acc_b[NV][4], acc_c[NV][4];
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) { acc_g[i][k] = 0ull; acc_b[i][k] = 0ull; acc_c[i][k] = 0ull; }
    // gamma is staged PERMUTED: pair k (0..3) of vector i of lane l sits at ((i * 4 + k) * 32 + l) * 2, so the LDS.64 a
    // warp issues for one (i, k) reads 256 consecutive bytes (the natural layout strides lanes by 32 bytes: 2-way
    // bank conflicts on every read, 24 reads per row)
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        const int i = c >> 8, l = (c >> 3) & 31, k = (c >> 1) & 3;
        sgamma[((i * 4 + k) * 32 + l) * 2 + (c & 1)] = gamma[c];
    }
    __syncthreads();
    const uint64_t *sg2 = reinterpret_cast<const uint64_t *>(sgamma) + lane;  // + (i * 4 + k) * 32

    // one CTA (8 warps) per SM with the whole register file: the NEXT row's three inputs are in flight while the current
    // row is processed (the kernel used to sit at 16 warps / SM x one row each and stalled on every row's loads:
    // 29 us for 100 MB in the round-2 profile)
    const int64_t stride = (int64_t)gridDim.x * warps_per_block;
    int64_t row = (int64_t)blockIdx.x * warps_per_block + warp;
    Packed8<T> pdy[NV], pres[NV], ndy[NV], nres[NV];
    Packed8<TX> px[NV], nx[NV];
    auto fetch = [&](int64_t r_, Packed8<T> *a, Packed8<TX> *b, Packed8<T> *c_) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) {
                ld_packed(a[i], dy + r_ * d + c);
                ld_packed(b[i], x + (kPatch ? r_ + r_ / n_patch + 1 : r_) * d + c);
                if (dres != nullptr) ld_packed(c_[i], dres + r_ * d + c);
            }
        }
    };
    // the row statistics come from L2 / HBM as well: fetched one row ahead like the row itself
    float mean_n = 0.f, rstd_n = 0.f;
    if (row < M) {
        fetch(row, pdy, px, pres);
        mean_n = __ldg(mean_in + row);
        rstd_n = __ldg(rstd_in + row);
    }
    for (; row < M; row += stride) {
        const float mean = mean_n, rstd = rstd_n;
        if (row + stride < M) {
            fetch(row + stride, ndy, nx, nres);
            mean_n = __ldg(mean_in + row + stride);
            rstd_n = __ldg(rstd_in + row + stride);
        }
        const uint64_t rstd2 = splat2(rstd), nmr2 = splat2(-mean * rstd);
        uint64_t s1_2 = 0ull, s2_2 = 0ull;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) {
                uint64_t dy2[4], x2[4];
                unpack_pairs(pdy[i], dy2);
                unpack_pairs(px[i], x2);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint64_t xh = fma2(x2[k], rstd2, nmr2);
                    const uint64_t g = mul2(dy2[k], sg2[(i * 4 + k) * 32]);
                    s1_2 = add2(s1_2, g);
                    s2_2 = fma2(g, xh, s2_2);
                    acc_g[i][k] = fma2(dy2[k], xh, acc_g[i][k]);
                    acc_b[i][k] = add2(acc_b[i][k], dy2[k]);
                }
            }
        }
        const float s1 = warp_sum(pair_sum(s1_2)) * inv_d;
        const float s2 = warp_sum(pair_sum(s2_2)) * inv_d;
        const uint64_t B2 = splat2(-rstd * rstd * s2), C2 = splat2(rstd * (mean * rstd * s2 - s1));
        uint64_t rs2 = 0ull;
        if constexpr (kPath) rs2 = splat2(path_factor(drop.path, row));
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int c = (i * 32 + lane) * 8;
            if (c < d) {
                uint64_t dy2[4], x2[4], o2[4];
                unpack_pairs(pdy[i], dy2);
                unpack_pairs(px[i], x2);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    o2[k] = fma2(dy2[k], mul2(sg2[(i * 4 + k) * 32], rstd2), fma2(x2[k], B2, C2));
                if (dres != nullptr) {
                    uint64_t r2[4];
                    unpack_pairs(pres[i], r2);
#pragma unroll
                    for (int k = 0; k < 4; ++k) o2[k] = add2(o2[k], r2[k]);
                }
                store_pairs(dx + (kPatch ? row + row / n_patch + 1 : row) * d + c, o2);
                if constexpr (kPath) {
                    const uint32_t seed = __ldg(drop.path.drop.seed);
                    const uint32_t e0 = static_cast<uint32_t>(row * d + c);
                    if (drop.threshold != 0) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            float m0, m1;
                            dropout_pair(drop, seed, e0 + 2 * k, m0, m1);
                            o2[k] = mul2(o2[k], pack2(m0, m1));
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) o2[k] = mul2(o2[k], rs2);
                    store_pairs(dxm + row * d + c, o2);
                } else if (kDrop) {
                    const uint32_t seed = __ldg(drop.seed);
                    const uint32_t e0 = static_cast<uint32_t>(row * d + c);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float m0, m1;
                        dropout_pair(drop, seed, e0 + 2 * k, m0, m1);
                        o2[k] = mul2(o2[k], pack2(m0, m1));
                    }
                    store_pairs(dxm + row * d + c, o2);
                }
                if (dcolsum != nullptr) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) acc_c[i][k] = add2(acc_c[i][k], o2[k]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            pdy[i] = ndy[i];
            px[i] = nx[i];
            pres[i] = nres[i];
        }
    }
    // block reduce: every warp parks its per-lane column sums in its own smem slab (plain stores), then the CTA adds
    // the slabs and writes ONE partial row per CTA; a tiny second kernel folds the partial rows into the gradients.
    // (fp32 atomics are avoided on purpose: shared-memory float atomics are CAS loops, and 296 CTAs x 3 x d global
    // atomics on 3 x d addresses serialise in L2.)
    float *slab = red + warp * 3 * d;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int c = (i * 32 + lane) * 8;
        if (c < d) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                *reinterpret_cast<uint64_t *>(slab + c + 2 * k) = acc_g[i][k];
                *reinterpret_cast<uint64_t *>(slab + d + c + 2 * k) = acc_b[i][k];
                *reinterpret_cast<uint64_t *>(slab + 2 * d + c + 2 * k) = acc_c[i][k];
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * d; i += blockDim.x) {
        float t = 0.f;
        for (int w = 0; w < warps_per_block; ++w) t += red[w * 3 * d + i];
        partial[(int64_t)blockIdx.x * 3 * d + i] = t;
    }
}

// folds the per-CTA partial rows: dgamma += sum_b partial[b][0], dbeta += ...[1], dcolsum += ...[2].
// block = 32 columns x 8 row groups (coalesced 128-byte reads, 8 independent chains per column), smem tree at the end
__global__ void __launch_bounds__(256) layernorm_bwd_finalize_kernel(const float *__restrict__ partial, int nblocks,
                                                                      float *__restrict__ dgamma,
                                                                      float *__restrict__ dbeta,
                                                                      float *__restrict__ dcolsum, int d) {
    __shared__ float red[8][33];
    pdl_launch_dependents();
    pdl_wait();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + tx;
    float t = 0.f;
    if (i < 3 * d)
        for (int b = ty; b < nblocks; b += 8) t += partial[(int64_t)b * 3 * d + i];
    red[ty][tx] = t;
    __syncthreads();
    if (ty == 0 && i < 3 * d) {
        float s = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) s += red[y][tx];
        if (i < d) dgamma[i] += s;
        else if (i < 2 * d) dbeta[i - d] += s;
        else if (dcolsum != nullptr) dcolsum[i - 2 * d] += s;
    }
}

constexpr int LN_BWD_MAX_BLOCKS = 2 * 160;  // scratch rows; the kernel runs one CTA per SM

// ---------------------------------------------------------------------------------------------------
// dym = mask * dy / (1 - p);  dcolsum[n] += sum_m dym[m, n].  Same block shape as colsum_kernel.
// kPath: dym = s[row / rows_per_record] * mask * dy, the element mask all ones when drop.threshold == 0
template <typename T, bool kPath = false>
__global__ void __launch_bounds__(256) dropout_bwd_copy_kernel(const T *__restrict__ dy, T *__restrict__ dym,
                                                                float *__restrict__ dcolsum, int M, int N, int64_t ld,
                                                                int rows_per_block, DropParamsFor<kPath> drop) {
    __shared__ float red[8][32 * 8 + 1];
    pdl_launch_dependents();
    pdl_wait();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + tx) * 8;
    const int r0 = blockIdx.y * rows_per_block;
    const int r1 = min(r0 + rows_per_block, M);
    uint32_t seed;
    if constexpr (kPath) seed = __ldg(drop.path.drop.seed);
    else seed = __ldg(drop.seed);
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    if (c < N) {
        for (int r = r0 + ty; r < r1; r += 8) {
            float v[8];
            load8(dy + (int64_t)r * ld + c, v);
            if constexpr (kPath) {
                if (drop.threshold != 0) dropout_apply<8>(drop, seed, static_cast<uint32_t>((int64_t)r * ld + c), v);
                const float rs = path_factor(drop.path, r);
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] *= rs;
            } else {
                dropout_apply<8>(drop, seed, static_cast<uint32_t>((int64_t)r * ld + c), v);
            }
            store8(dym + (int64_t)r * ld + c, v);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] += to_f32(from_f32<T>(v[k]));
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[ty][tx * 8 + k] = acc[k];
    __syncthreads();
    if (dcolsum != nullptr) {
        float s = 0.f;
#pragma unroll
        for (int y = 0; y < 8; ++y) s += red[y][threadIdx.x];
        const int col = blockIdx.x * 256 + threadIdx.x;
        if (col < N) atomicAdd(dcolsum + col, s);
    }
}

// ---------------------------------------------------------------------------------------------------
// out[n] += sum_m x[m, n]; block = 32 column-vectors (8 wide) x 8 row lanes; grid.y splits the rows
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T *__restrict__ x, float *__restrict__ out, int M, int N,
                                                      int64_t ld, int rows_per_block) {
    __shared__ float red[8][32 * 8 + 1];
    pdl_launch_dependents();
    pdl_wait();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + tx) * 8;
    const int r0 = blockIdx.y * rows_per_block;
    const int r1 = min(r0 + rows_per_block, M);
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    if (c < N) {
        for (int r = r0 + ty; r < r1; r += 8) {
            float v[8];
            load8(x + (int64_t)r * ld + c, v);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] += v[k];
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[ty][tx * 8 + k] = acc[k];
    __syncthreads();
    const int col_local = threadIdx.x;  // 256 columns per block
    float s = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) s += red[y][col_local];
    const int col = blockIdx.x * 256 + col_local;
    if (col < N) atomicAdd(out + col, s);
}

__global__ void cast_f32_bf16_kernel(const float *__restrict__ src, bf16 *__restrict__ dst, int64_t n) {
    const int64_t n8 = n / 8;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        float v[8];
        load8(src + i * 8, v);
        store8(dst + i * 8, v);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = n8 * 8; i < n; ++i) dst[i] = __float2bfloat16_rn(src[i]);
}

inline int grid_for(int64_t work_items, int threads, int max_blocks_per_sm = 8) {
    int64_t g = (work_items + threads - 1) / threads;
    const int64_t cap = (int64_t)sm_count() * max_blocks_per_sm;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace
}  // namespace ecgvit

using namespace ecgvit;

// windows per CTA of the patch gather: up to 8, as many as fit 48 KB of staging
static int patchify_group(int n_patch, int P, int C) {
    int wg = (int)((48 * 1024) / ((size_t)P * C * sizeof(float)));
    if (wg > 8) wg = 8;
    if (wg > n_patch) wg = n_patch;
    return wg < 1 ? 1 : wg;
}

// fixed-order column sums of scratch [rows, d] into out (two launches, see fold_rows_kernel); scratch is overwritten
static void fold_rows(float *scratch, int rows, int d, float *out, cudaStream_t st) {
    const int chunks = (rows + kFoldChunk - 1) / kFoldChunk;
    launch_pdl(fold_rows_kernel, dim3((d + 31) / 32, chunks), dim3(32 * kFoldGroups), 0, st, scratch, rows, 1, d,
               (float *)nullptr);
    launch_pdl(fold_rows_kernel, dim3((d + 31) / 32, 1), dim3(32 * kFoldGroups), 0, st, scratch, chunks, kFoldChunk, d,
               out);
}

extern "C" {

int ecgvit_patchify(const float *x, void *a, int B, int C, int64_t x_ld, int n_patch, int P, int dtype,
                    void *stream) {
    ECGVIT_REQUIRE(x && a && B > 0 && C > 0 && n_patch > 0 && P > 0, "patchify: bad arguments");
    ECGVIT_REQUIRE(x_ld >= (int64_t)n_patch * P, "patchify: x_ld=%lld shorter than n_patch*P=%d", (long long)x_ld,
                   n_patch * P);
    ECGVIT_REQUIRE((size_t)P * C * sizeof(float) <= 48 * 1024, "patchify: patch of %d x %d elements exceeds 48 KB staging", P, C);
    const int WG = patchify_group(n_patch, P, C);
    const size_t smem = (size_t)WG * P * C * sizeof(float);
    const int grid = B * ((n_patch + WG - 1) / WG);
    const int L_all = n_patch * P;
    if (dtype == ECGVIT_BF16)
        patchify_kernel<bf16><<<grid, 256, smem, as_stream(stream)>>>(x, nullptr, nullptr, nullptr, (bf16 *)a, C, x_ld, L_all, n_patch, P, WG, 1.0f / (float)P);
    else if (dtype == ECGVIT_F32)
        patchify_kernel<float><<<grid, 256, smem, as_stream(stream)>>>(x, nullptr, nullptr, nullptr, (float *)a, C, x_ld, L_all, n_patch, P, WG, 1.0f / (float)P);
    else return fail(-1, "patchify: unknown dtype %d", dtype);
    return check_launch("patchify");
}

int ecgvit_patchify_transform(const float *x, const float *mean, const float *stdev, const int *spans, void *a, int B,
                              int C, int64_t x_ld, int L_valid, int n_patch, int P, int dtype, void *stream) {
    ECGVIT_REQUIRE(x && a && B > 0 && C > 0 && n_patch > 0 && P > 0, "patchify_transform: bad arguments");
    ECGVIT_REQUIRE((mean == nullptr) == (stdev == nullptr), "patchify_transform: mean and std come together");
    ECGVIT_REQUIRE(L_valid > 0 && L_valid <= x_ld, "patchify_transform: L_valid=%d outside (0, x_ld=%lld]", L_valid,
                   (long long)x_ld);
    ECGVIT_REQUIRE((int64_t)n_patch * P >= L_valid, "patchify_transform: n_patch*P=%d drops samples of L_valid=%d",
                   n_patch * P, L_valid);
    ECGVIT_REQUIRE((size_t)P * C * sizeof(float) <= 48 * 1024, "patchify_transform: patch of %d x %d elements exceeds 48 KB staging", P, C);
    const int WG = patchify_group(n_patch, P, C);
    const size_t smem = (size_t)WG * P * C * sizeof(float);
    const int grid = B * ((n_patch + WG - 1) / WG);
    if (dtype == ECGVIT_BF16)
        patchify_kernel<bf16><<<grid, 256, smem, as_stream(stream)>>>(x, mean, stdev, spans, (bf16 *)a, C, x_ld, L_valid, n_patch, P, WG, 1.0f / (float)P);
    else if (dtype == ECGVIT_F32)
        patchify_kernel<float><<<grid, 256, smem, as_stream(stream)>>>(x, mean, stdev, spans, (float *)a, C, x_ld, L_valid, n_patch, P, WG, 1.0f / (float)P);
    else return fail(-1, "patchify_transform: unknown dtype %d", dtype);
    return check_launch("patchify_transform");
}

int ecgvit_patchify_leads(const float *x, const float *mean, const float *stdev, const int *spans, void *a, int B, int C,
                          int64_t x_ld, int L_valid, int n_w, int P, int Kp, int dtype, void *stream) {
    ECGVIT_REQUIRE(x && a && B > 0 && C > 0 && n_w > 0 && P > 0, "patchify_leads: bad arguments");
    ECGVIT_REQUIRE((mean == nullptr) == (stdev == nullptr), "patchify_leads: mean and std come together");
    ECGVIT_REQUIRE(Kp >= P && Kp % 8 == 0, "patchify_leads: padded row length %d must be a multiple of 8 >= P=%d", Kp, P);
    ECGVIT_REQUIRE(L_valid > 0 && L_valid <= x_ld && (int64_t)n_w * P >= L_valid,
                   "patchify_leads: L_valid=%d must fit x_ld=%lld and n_w*P=%d", L_valid, (long long)x_ld, n_w * P);
    const int64_t total = (int64_t)B * C * n_w * Kp;
    const int grid = grid_for(total, 256);
    if (dtype == ECGVIT_BF16)
        patchify_leads_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>(x, mean, stdev, spans, (bf16 *)a, total, C, x_ld, L_valid, n_w, P, Kp);
    else if (dtype == ECGVIT_F32)
        patchify_leads_kernel<float><<<grid, 256, 0, as_stream(stream)>>>(x, mean, stdev, spans, (float *)a, total, C, x_ld, L_valid, n_w, P, Kp);
    else return fail(-1, "patchify_leads: unknown dtype %d", dtype);
    return check_launch("patchify_leads");
}

int ecgvit_pad_cols(const void *src, void *dst, int64_t rows, int cols, int cols_padded, int dtype, void *stream) {
    ECGVIT_REQUIRE(src && dst && rows > 0 && cols > 0 && cols_padded >= cols, "pad_cols: bad arguments");
    const int grid = grid_for(rows * cols_padded, 256);
    if (dtype == ECGVIT_BF16)
        pad_cols_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>((const bf16 *)src, (bf16 *)dst, rows, cols, cols_padded);
    else if (dtype == ECGVIT_F32)
        pad_cols_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((const float *)src, (float *)dst, rows, cols, cols_padded);
    else return fail(-1, "pad_cols: unknown dtype %d", dtype);
    return check_launch("pad_cols");
}

int ecgvit_unpad_add_f32(const float *src, float *dst, int64_t rows, int cols, int cols_padded, void *stream) {
    ECGVIT_REQUIRE(src && dst && rows > 0 && cols > 0 && cols_padded >= cols, "unpad_add: bad arguments");
    unpad_add_kernel<<<grid_for(rows * cols, 256), 256, 0, as_stream(stream)>>>(src, dst, rows, cols, cols_padded);
    return check_launch("unpad_add");
}

int ecgvit_embed_assemble(const void *e, const float *cls, const float *pos, void *tok, int B, int n_patch, int d,
                          float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(e && cls && pos && tok && B > 0 && n_patch > 0, "embed_assemble: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "embed_assemble: d=%d must be a multiple of 8", d);
    const int64_t total = (int64_t)B * (n_patch + 1) * (d / 8);
    const int grid = grid_for(total, 256);
    if (dtype == ECGVIT_BF16)
        embed_assemble_kernel<bf16, bf16><<<grid, 256, 0, as_stream(stream)>>>((const bf16 *)e, cls, pos, (bf16 *)tok, B, n_patch, d, drop);
    else if (dtype == ECGVIT_BF16_RES32)
        embed_assemble_kernel<bf16, float><<<grid, 256, 0, as_stream(stream)>>>((const bf16 *)e, cls, pos, (float *)tok, B, n_patch, d, drop);
    else if (dtype == ECGVIT_F32)
        embed_assemble_kernel<float, float><<<grid, 256, 0, as_stream(stream)>>>((const float *)e, cls, pos, (float *)tok, B, n_patch, d, drop);
    else return fail(-1, "embed_assemble: unknown dtype %d", dtype);
    return check_launch("embed_assemble");
}

int ecgvit_embed_assemble_bwd(const void *dtok, void *de, float *dcls, float *dpos, float *dbias, int B,
                              int n_patch, int d, float dropout_p, int dropout_stream, const uint32_t *dropout_seed,
                              int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(dtok && de && dcls && dpos && dbias && B > 0 && n_patch > 0 && d > 0, "embed_assemble_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "embed_assemble_bwd: d=%d must be a multiple of 8", d);
    dim3 grid(n_patch + 1, (d + 255) / 256);
    if (dtype == ECGVIT_BF16)
        embed_assemble_bwd_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>((const bf16 *)dtok, (bf16 *)de, dcls, dpos, dbias, B, n_patch, d, drop);
    else if (dtype == ECGVIT_F32)
        embed_assemble_bwd_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((const float *)dtok, (float *)de, dcls, dpos, dbias, B, n_patch, d, drop);
    else return fail(-1, "embed_assemble_bwd: unknown dtype %d", dtype);
    return check_launch("embed_assemble_bwd");
}

int ecgvit_embed_assemble_masked(const void *e, const float *cls, const float *pos, const float *mask_token,
                                 const uint8_t *mask, void *tok, int B, int n_patch, int d, float dropout_p,
                                 int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(e && cls && pos && mask_token && mask && tok && B > 0 && n_patch > 0,
                   "embed_assemble_masked: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "embed_assemble_masked: d=%d must be a multiple of 8", d);
    const int64_t total = (int64_t)B * (n_patch + 1) * (d / 8);
    const int grid = grid_for(total, 256);
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        embed_assemble_kernel<bf16, bf16, true><<<grid, 256, 0, st>>>((const bf16 *)e, cls, pos, (bf16 *)tok, B, n_patch, d, drop, mask_token, mask);
    else if (dtype == ECGVIT_BF16_RES32)
        embed_assemble_kernel<bf16, float, true><<<grid, 256, 0, st>>>((const bf16 *)e, cls, pos, (float *)tok, B, n_patch, d, drop, mask_token, mask);
    else if (dtype == ECGVIT_F32)
        embed_assemble_kernel<float, float, true><<<grid, 256, 0, st>>>((const float *)e, cls, pos, (float *)tok, B, n_patch, d, drop, mask_token, mask);
    else return fail(-1, "embed_assemble_masked: unknown dtype %d", dtype);
    return check_launch("embed_assemble_masked");
}

int ecgvit_embed_assemble_masked_bwd(const void *dtok, const uint8_t *mask, void *de, float *dcls, float *dpos,
                                     float *dbias, float *dmask_token, int B, int n_patch, int d, float dropout_p,
                                     int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(dtok && mask && de && dcls && dpos && dbias && dmask_token && B > 0 && n_patch > 0 && d > 0,
                   "embed_assemble_masked_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "embed_assemble_masked_bwd: d=%d must be a multiple of 8", d);
    dim3 grid(n_patch + 1, (d + 255) / 256);
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        embed_assemble_bwd_kernel<bf16, true><<<grid, 256, 0, st>>>((const bf16 *)dtok, (bf16 *)de, dcls, dpos, dbias, B, n_patch, d, drop, mask, dmask_token);
    else if (dtype == ECGVIT_F32)
        embed_assemble_bwd_kernel<float, true><<<grid, 256, 0, st>>>((const float *)dtok, (float *)de, dcls, dpos, dbias, B, n_patch, d, drop, mask, dmask_token);
    else return fail(-1, "embed_assemble_masked_bwd: unknown dtype %d", dtype);
    return check_launch("embed_assemble_masked_bwd");
}

int ecgvit_embed_assemble_visible(const void *e, const float *cls, const float *pos, const int *vis_idx, void *tok,
                                  int B, int n_vis, int d, float dropout_p, int dropout_stream,
                                  const uint32_t *dropout_seed, int dtype, void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(e && cls && pos && vis_idx && tok && B > 0 && n_vis > 0, "embed_assemble_visible: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "embed_assemble_visible: d=%d must be a multiple of 8", d);
    const int64_t total = (int64_t)B * (n_vis + 1) * (d / 8);
    const dim3 grid(grid_for(total, 256));
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        launch_pdl(embed_assemble_kernel<bf16, bf16, false, true>, grid, dim3(256), 0, st, (const bf16 *)e, cls, pos,
                   (bf16 *)tok, B, n_vis, d, drop, (const float *)nullptr, (const uint8_t *)nullptr, vis_idx);
    else if (dtype == ECGVIT_BF16_RES32)
        launch_pdl(embed_assemble_kernel<bf16, float, false, true>, grid, dim3(256), 0, st, (const bf16 *)e, cls, pos,
                   (float *)tok, B, n_vis, d, drop, (const float *)nullptr, (const uint8_t *)nullptr, vis_idx);
    else if (dtype == ECGVIT_F32)
        launch_pdl(embed_assemble_kernel<float, float, false, true>, grid, dim3(256), 0, st, (const float *)e, cls, pos,
                   (float *)tok, B, n_vis, d, drop, (const float *)nullptr, (const uint8_t *)nullptr, vis_idx);
    else return fail(-1, "embed_assemble_visible: unknown dtype %d", dtype);
    return check_launch("embed_assemble_visible");
}

int ecgvit_embed_assemble_visible_bwd(const void *dtok, const int *slot, void *de, float *dcls, float *dpos,
                                      float *dbias, float *scratch, int B, int n_patch, int n_vis, int d,
                                      float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype,
                                      void *stream) {
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(dtok && slot && de && dcls && dpos && dbias && scratch && B > 0 && n_vis > 0 && n_vis <= n_patch &&
                   d > 0, "embed_assemble_visible_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "embed_assemble_visible_bwd: d=%d must be a multiple of 8", d);
    const dim3 grid(n_patch + 1, (d + 255) / 256);
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        launch_pdl(embed_assemble_bwd_kernel<bf16, false, true>, grid, dim3(256), 0, st, (const bf16 *)dtok, (bf16 *)de,
                   dcls, dpos, dbias, B, n_patch, d, drop, (const uint8_t *)nullptr, (float *)nullptr, slot, n_vis,
                   scratch);
    else if (dtype == ECGVIT_F32)
        launch_pdl(embed_assemble_bwd_kernel<float, false, true>, grid, dim3(256), 0, st, (const float *)dtok,
                   (float *)de, dcls, dpos, dbias, B, n_patch, d, drop, (const uint8_t *)nullptr, (float *)nullptr, slot,
                   n_vis, scratch);
    else return fail(-1, "embed_assemble_visible_bwd: unknown dtype %d", dtype);
    int rc = check_launch("embed_assemble_visible_bwd");
    if (rc) return rc;
    fold_rows(scratch, n_patch, d, dbias, st);
    return check_launch("embed_assemble_visible_bwd");
}

int ecgvit_mae_unshuffle(const void *t, const float *mask_token, const float *pos, const int *slot, void *u, int B,
                         int n_patch, int n_vis, int d, int dtype, void *stream) {
    ECGVIT_REQUIRE(t && mask_token && pos && slot && u && B > 0 && n_vis > 0 && n_vis <= n_patch,
                   "mae_unshuffle: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "mae_unshuffle: d=%d must be a multiple of 8", d);
    const dim3 grid(grid_for((int64_t)B * (n_patch + 1) * (d / 8), 256));
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        launch_pdl(mae_unshuffle_kernel<bf16, bf16>, grid, dim3(256), 0, st, (const bf16 *)t, mask_token, pos, slot,
                   (bf16 *)u, B, n_patch, n_vis, d);
    else if (dtype == ECGVIT_BF16_RES32)
        launch_pdl(mae_unshuffle_kernel<bf16, float>, grid, dim3(256), 0, st, (const bf16 *)t, mask_token, pos, slot,
                   (float *)u, B, n_patch, n_vis, d);
    else if (dtype == ECGVIT_F32)
        launch_pdl(mae_unshuffle_kernel<float, float>, grid, dim3(256), 0, st, (const float *)t, mask_token, pos, slot,
                   (float *)u, B, n_patch, n_vis, d);
    else return fail(-1, "mae_unshuffle: unknown dtype %d", dtype);
    return check_launch("mae_unshuffle");
}

int ecgvit_mae_unshuffle_bwd(const void *du, const int *slot, void *dt, float *dpos, float *dmask_token,
                             float *scratch, int B, int n_patch, int n_vis, int d, int dtype, void *stream) {
    ECGVIT_REQUIRE(du && slot && dt && dpos && dmask_token && scratch && B > 0 && n_vis > 0 && n_vis <= n_patch,
                   "mae_unshuffle_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0, "mae_unshuffle_bwd: d=%d must be a multiple of 8", d);
    const dim3 grid(n_patch + 1, (d + 255) / 256);
    cudaStream_t st = as_stream(stream);
    if (dtype == ECGVIT_BF16)
        launch_pdl(mae_unshuffle_bwd_kernel<bf16>, grid, dim3(256), 0, st, (const bf16 *)du, slot, (bf16 *)dt, dpos,
                   scratch, B, n_patch, n_vis, d);
    else if (dtype == ECGVIT_F32)
        launch_pdl(mae_unshuffle_bwd_kernel<float>, grid, dim3(256), 0, st, (const float *)du, slot, (float *)dt, dpos,
                   scratch, B, n_patch, n_vis, d);
    else return fail(-1, "mae_unshuffle_bwd: unknown dtype %d", dtype);
    int rc = check_launch("mae_unshuffle_bwd");
    if (rc) return rc;
    fold_rows(scratch, n_patch, d, dmask_token, st);
    return check_launch("mae_unshuffle_bwd");
}

int ecgvit_layernorm_patch_fwd(const void *tok, const float *gamma, const float *beta, void *y, float *mean,
                               float *rstd, int B, int n_patch, int d, float eps, int dtype, void *stream) {
    ECGVIT_REQUIRE(tok && gamma && beta && y && B > 0 && n_patch > 0, "layernorm_patch_fwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * LN_MAXV, "layernorm_patch_fwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * LN_MAXV);
    const int M = B * n_patch;
    const int nv = (d + 255) / 256;
    cudaStream_t st = as_stream(stream);
    int grid = grid_for((int64_t)M * 32, 256);
    if (grid > sm_count() * 2) grid = sm_count() * 2;
#define ECGVIT_LNP_FWD(TT, NVV, TXX)                                                                                    \
    launch_pdl(layernorm_fwd_kernel<TT, NVV, 1, 2, TXX, true>, dim3(grid), dim3(256), 0, st, (const TXX *)tok, gamma, \
               beta, (TT *)y, mean, rstd, M, d, eps, n_patch)
#define ECGVIT_LNP_FWD_NV(TT, TXX)                   \
    switch (nv) {                                    \
        case 1: ECGVIT_LNP_FWD(TT, 1, TXX); break;   \
        case 2: ECGVIT_LNP_FWD(TT, 2, TXX); break;   \
        case 3: ECGVIT_LNP_FWD(TT, 3, TXX); break;   \
        default: ECGVIT_LNP_FWD(TT, 4, TXX); break;  \
    }
    if (dtype == ECGVIT_BF16) { ECGVIT_LNP_FWD_NV(bf16, bf16) }
    else if (dtype == ECGVIT_BF16_RES32) { ECGVIT_LNP_FWD_NV(bf16, float) }
    else if (dtype == ECGVIT_F32) { ECGVIT_LNP_FWD_NV(float, float) }
    else return fail(-1, "layernorm_patch_fwd: unknown dtype %d", dtype);
#undef ECGVIT_LNP_FWD_NV
#undef ECGVIT_LNP_FWD
    return check_launch("layernorm_patch_fwd");
}

int ecgvit_layernorm_fwd(const void *x, const float *gamma, const float *beta, void *y, float *mean, float *rstd,
                         int M, int d, float eps, int dtype, void *stream) {
    ECGVIT_REQUIRE(x && gamma && beta && y && M > 0, "layernorm_fwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * LN_MAXV, "layernorm_fwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * LN_MAXV);
    const int nv = (d + 255) / 256;
    cudaStream_t st = as_stream(stream);
    // persistent: 2 CTAs (16 warps) per SM (gamma / beta / two rows live in registers: ~100 of them), each warp walks its
    // rows with the next row's loads in flight
    int grid = grid_for((int64_t)M * 32, 256);
    if (grid > sm_count() * 2) grid = sm_count() * 2;
#define ECGVIT_LN_FWD(TT, NVV)                                                                                          \
    launch_pdl(layernorm_fwd_kernel<TT, NVV, 1, 2>, dim3(grid), dim3(256), 0, st, (const TT *)x, gamma, beta, (TT *)y,   \
               mean, rstd, M, d, eps, 1)
    if (dtype == ECGVIT_BF16) {
        switch (nv) {
            case 1: ECGVIT_LN_FWD(bf16, 1); break;
            case 2: ECGVIT_LN_FWD(bf16, 2); break;
            case 3: ECGVIT_LN_FWD(bf16, 3); break;
            default: ECGVIT_LN_FWD(bf16, 4); break;
        }
    } else if (dtype == ECGVIT_BF16_RES32) {   // fp32 residual stream in, bf16 operand out
#define ECGVIT_LN_FWD_R(NVV)                                                                                            \
    launch_pdl(layernorm_fwd_kernel<bf16, NVV, 1, 2, float>, dim3(grid), dim3(256), 0, st, (const float *)x, gamma, beta, \
               (bf16 *)y, mean, rstd, M, d, eps, 1)
        switch (nv) {
            case 1: ECGVIT_LN_FWD_R(1); break;
            case 2: ECGVIT_LN_FWD_R(2); break;
            case 3: ECGVIT_LN_FWD_R(3); break;
            default: ECGVIT_LN_FWD_R(4); break;
        }
#undef ECGVIT_LN_FWD_R
    } else if (dtype == ECGVIT_F32) {
        switch (nv) {
            case 1: ECGVIT_LN_FWD(float, 1); break;
            case 2: ECGVIT_LN_FWD(float, 2); break;
            case 3: ECGVIT_LN_FWD(float, 3); break;
            default: ECGVIT_LN_FWD(float, 4); break;
        }
    } else return fail(-1, "layernorm_fwd: unknown dtype %d", dtype);
#undef ECGVIT_LN_FWD
    return check_launch("layernorm_fwd");
}

int64_t ecgvit_layernorm_bwd_scratch_floats(int d) { return (int64_t)LN_BWD_MAX_BLOCKS * 3 * d; }

static int ln_bwd_blocks(int M) {
    int grid = grid_for((int64_t)M * 32, 256, 1);
    return grid > LN_BWD_MAX_BLOCKS ? LN_BWD_MAX_BLOCKS : grid;
}

int ecgvit_layernorm_bwd_finalize(const float *scratch, float *dgamma, float *dbeta, float *dcolsum, int M, int d,
                                  void *stream) {
    ECGVIT_REQUIRE(scratch && dgamma && dbeta && M > 0 && d > 0, "layernorm_bwd_finalize: bad arguments");
    launch_pdl(layernorm_bwd_finalize_kernel, dim3((3 * d + 31) / 32), dim3(256), 0, as_stream(stream), scratch,
               ln_bwd_blocks(M), dgamma, dbeta, dcolsum, d);
    return check_launch("layernorm_bwd_finalize");
}

}  // extern "C"

// dxm (when `dropping`) = mask * dx, or with kPath s[row / rows_per_record] * mask * dx
template <bool kPath>
static int layernorm_bwd_launch(const void *dy, const void *x, const float *gamma, const float *mean, const float *rstd,
                                const void *dres, void *dx, float *dgamma, float *dbeta, float *dcolsum, float *scratch,
                                void *dxm, const DropParamsFor<kPath> &drop, bool dropping, int M, int d,
                                int defer_finalize, int dtype, void *stream) {
    const int grid = ln_bwd_blocks(M);
    const int nv = (d + 255) / 256;
    const size_t smem = (8 * 3 * (size_t)d + (size_t)nv * 256) * sizeof(float);  // warp slabs + permuted gamma
    cudaStream_t st = as_stream(stream);
#define ECGVIT_LN_BWD2(TT, NVV, DROP, TXX)                                                                             \
    do {                                                                                                               \
        static bool attr_set = false;                                                                                  \
        if (!attr_set) {                                                                                               \
            cudaFuncSetAttribute(layernorm_bwd_kernel<TT, NVV, DROP, TXX, false, kPath>,                               \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 25 * 1024 * 4);                          \
            attr_set = true;                                                                                           \
        }                                                                                                              \
        launch_pdl(layernorm_bwd_kernel<TT, NVV, DROP, TXX, false, kPath>, dim3(grid), dim3(256), smem, st,            \
                   (const TT *)dy, (const TXX *)x, gamma, mean, rstd, (const TT *)dres, (TT *)dx, dgamma, dbeta,       \
                   dcolsum, scratch, M, d, (TT *)dxm, drop, 1);                                                        \
    } while (0)
    // (the drop-path kernels always write dxm)
#define ECGVIT_LN_BWD(TT, NVV) do { if constexpr (kPath) ECGVIT_LN_BWD2(TT, NVV, true, TT); else if (dropping) ECGVIT_LN_BWD2(TT, NVV, true, TT); else ECGVIT_LN_BWD2(TT, NVV, false, TT); } while (0)
#define ECGVIT_LN_BWD_R(NVV) do { if constexpr (kPath) ECGVIT_LN_BWD2(bf16, NVV, true, float); else if (dropping) ECGVIT_LN_BWD2(bf16, NVV, true, float); else ECGVIT_LN_BWD2(bf16, NVV, false, float); } while (0)
    if (dtype == ECGVIT_BF16) {
        switch (nv) {
            case 1: ECGVIT_LN_BWD(bf16, 1); break;
            case 2: ECGVIT_LN_BWD(bf16, 2); break;
            case 3: ECGVIT_LN_BWD(bf16, 3); break;
            default: ECGVIT_LN_BWD(bf16, 4); break;
        }
    } else if (dtype == ECGVIT_BF16_RES32) {   // x (the residual stream) is fp32, gradients stay bf16
        switch (nv) {
            case 1: ECGVIT_LN_BWD_R(1); break;
            case 2: ECGVIT_LN_BWD_R(2); break;
            case 3: ECGVIT_LN_BWD_R(3); break;
            default: ECGVIT_LN_BWD_R(4); break;
        }
    } else if (dtype == ECGVIT_F32) {
        switch (nv) {
            case 1: ECGVIT_LN_BWD(float, 1); break;
            case 2: ECGVIT_LN_BWD(float, 2); break;
            case 3: ECGVIT_LN_BWD(float, 3); break;
            default: ECGVIT_LN_BWD(float, 4); break;
        }
    } else return fail(-1, "layernorm_bwd: unknown dtype %d", dtype);
#undef ECGVIT_LN_BWD
#undef ECGVIT_LN_BWD_R
#undef ECGVIT_LN_BWD2
    int rc = check_launch("layernorm_bwd");
    if (rc || defer_finalize) return rc;
    return ecgvit_layernorm_bwd_finalize(scratch, dgamma, dbeta, dcolsum, M, d, stream);
}

extern "C" {

int ecgvit_layernorm_bwd(const void *dy, const void *x, const float *gamma, const float *mean, const float *rstd,
                         const void *dres, void *dx, float *dgamma, float *dbeta, float *dcolsum, float *scratch,
                         void *dxm, float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int M, int d,
                         int defer_finalize, int dtype, void *stream) {
    ECGVIT_REQUIRE(dy && x && gamma && mean && rstd && dx && dgamma && dbeta && scratch && M > 0,
                   "layernorm_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * LN_MAXV, "layernorm_bwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * LN_MAXV);
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    const bool dropping = drop.threshold != 0 && dxm != nullptr;
    return layernorm_bwd_launch<false>(dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta, dcolsum, scratch, dxm, drop,
                                       dropping, M, d, defer_finalize, dtype, stream);
}

int ecgvit_layernorm_bwd_drop_path(const void *dy, const void *x, const float *gamma, const float *mean,
                                   const float *rstd, const void *dres, void *dx, float *dgamma, float *dbeta,
                                   float *dcolsum, float *scratch, void *dxm, float dropout_p, int dropout_stream,
                                   const uint32_t *dropout_seed, int M, int d, int defer_finalize, int dtype,
                                   float path_p, int path_stream, int rows_per_record, void *stream) {
    PathParams pp;
    if (int rc = make_path("layernorm_bwd_drop_path", path_p, path_stream, rows_per_record, dropout_seed, pp)) return rc;
    if (pp.drop.threshold == 0)
        return ecgvit_layernorm_bwd(dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta, dcolsum, scratch, dxm, dropout_p,
                                    dropout_stream, dropout_seed, M, d, defer_finalize, dtype, stream);
    ECGVIT_REQUIRE(dy && x && gamma && mean && rstd && dx && dgamma && dbeta && scratch && dxm && M > 0,
                   "layernorm_bwd_drop_path: bad arguments (drop path writes dxm)");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * LN_MAXV, "layernorm_bwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * LN_MAXV);
    DropoutPathParams drop;
    static_cast<DropoutParams &>(drop) = make_dropout(dropout_p, dropout_stream, dropout_seed);
    drop.path = pp;
    return layernorm_bwd_launch<true>(dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta, dcolsum, scratch, dxm, drop,
                                      true, M, d, defer_finalize, dtype, stream);
}

int ecgvit_layernorm_patch_bwd(const void *dy, const void *tok, const float *gamma, const float *mean,
                               const float *rstd, void *dtok, float *dgamma, float *dbeta, float *dcolsum,
                               float *scratch, int B, int n_patch, int d, int dtype, void *stream) {
    ECGVIT_REQUIRE(dy && tok && gamma && mean && rstd && dtok && dgamma && dbeta && scratch && B > 0 && n_patch > 0,
                   "layernorm_patch_bwd: bad arguments");
    ECGVIT_REQUIRE(d % 8 == 0 && d <= 8 * 32 * LN_MAXV, "layernorm_patch_bwd: d=%d must be a multiple of 8 and <= %d", d,
                   8 * 32 * LN_MAXV);
    const int M = B * n_patch;
    const int grid = ln_bwd_blocks(M);
    const int nv = (d + 255) / 256;
    const size_t smem = (8 * 3 * (size_t)d + (size_t)nv * 256) * sizeof(float);
    cudaStream_t st = as_stream(stream);
    const DropoutParams nodrop = make_dropout(0.f, 0, nullptr);
    const bool bf = dtype == ECGVIT_BF16 || dtype == ECGVIT_BF16_RES32;
    if (!bf && dtype != ECGVIT_F32) return fail(-1, "layernorm_patch_bwd: unknown dtype %d", dtype);
    const int zgrid = grid_for((int64_t)B * d, 256);
    if (bf) zero_cls_rows_kernel<bf16><<<zgrid, 256, 0, st>>>((bf16 *)dtok, B, n_patch + 1, d);
    else zero_cls_rows_kernel<float><<<zgrid, 256, 0, st>>>((float *)dtok, B, n_patch + 1, d);
#define ECGVIT_LNP_BWD(TT, NVV, TXX)                                                                                   \
    do {                                                                                                               \
        static bool attr_set = false;                                                                                  \
        if (!attr_set) {                                                                                               \
            cudaFuncSetAttribute(layernorm_bwd_kernel<TT, NVV, false, TXX, true>,                                      \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 25 * 1024 * 4);                          \
            attr_set = true;                                                                                           \
        }                                                                                                              \
        launch_pdl(layernorm_bwd_kernel<TT, NVV, false, TXX, true>, dim3(grid), dim3(256), smem, st, (const TT *)dy,  \
                   (const TXX *)tok, gamma, mean, rstd, (const TT *)nullptr, (TT *)dtok, dgamma, dbeta, dcolsum,       \
                   scratch, M, d, (TT *)nullptr, nodrop, n_patch);                                                     \
    } while (0)
#define ECGVIT_LNP_BWD_NV(TT, TXX)                   \
    switch (nv) {                                    \
        case 1: ECGVIT_LNP_BWD(TT, 1, TXX); break;   \
        case 2: ECGVIT_LNP_BWD(TT, 2, TXX); break;   \
        case 3: ECGVIT_LNP_BWD(TT, 3, TXX); break;   \
        default: ECGVIT_LNP_BWD(TT, 4, TXX); break;  \
    }
    if (dtype == ECGVIT_BF16) { ECGVIT_LNP_BWD_NV(bf16, bf16) }
    else if (dtype == ECGVIT_BF16_RES32) { ECGVIT_LNP_BWD_NV(bf16, float) }
    else { ECGVIT_LNP_BWD_NV(float, float) }
#undef ECGVIT_LNP_BWD_NV
#undef ECGVIT_LNP_BWD
    const int rc = check_launch("layernorm_patch_bwd");
    if (rc) return rc;
    return ecgvit_layernorm_bwd_finalize(scratch, dgamma, dbeta, dcolsum, M, d, stream);
}

int ecgvit_colsum(const void *x, float *out, int M, int N, int64_t ld, int dtype, void *stream) {
    ECGVIT_REQUIRE(x && out && M > 0 && N > 0, "colsum: bad arguments");
    ECGVIT_REQUIRE(N % 8 == 0 && ld % 8 == 0, "colsum: N=%d and ld=%lld must be multiples of 8", N, (long long)ld);
    const int col_blocks = (N + 255) / 256;
    int row_blocks = (sm_count() * 4 + col_blocks - 1) / col_blocks;
    if (row_blocks > (M + 63) / 64) row_blocks = (M + 63) / 64;
    if (row_blocks < 1) row_blocks = 1;
    const int rows_per_block = (M + row_blocks - 1) / row_blocks;
    dim3 grid(col_blocks, (M + rows_per_block - 1) / rows_per_block);
    if (dtype == ECGVIT_BF16)
        launch_pdl(colsum_kernel<bf16>, grid, dim3(256), 0, as_stream(stream), (const bf16 *)x, out, M, N, ld, rows_per_block);
    else if (dtype == ECGVIT_F32)
        colsum_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((const float *)x, out, M, N, ld, rows_per_block);
    else return fail(-1, "colsum: unknown dtype %d", dtype);
    return check_launch("colsum");
}

}  // extern "C"

template <bool kPath>
static int dropout_bwd_copy_launch(const void *dy, void *dym, float *dcolsum, int M, int N, int64_t ld,
                                   const DropParamsFor<kPath> &drop, int dtype, void *stream) {
    const int col_blocks = (N + 255) / 256;
    int row_blocks = (sm_count() * 4 + col_blocks - 1) / col_blocks;
    if (row_blocks > (M + 63) / 64) row_blocks = (M + 63) / 64;
    if (row_blocks < 1) row_blocks = 1;
    const int rows_per_block = (M + row_blocks - 1) / row_blocks;
    dim3 grid(col_blocks, (M + rows_per_block - 1) / rows_per_block);
    if (dtype == ECGVIT_BF16)
        launch_pdl(dropout_bwd_copy_kernel<bf16, kPath>, grid, dim3(256), 0, as_stream(stream), (const bf16 *)dy, (bf16 *)dym, dcolsum, M, N, ld, rows_per_block, drop);
    else if (dtype == ECGVIT_F32)
        dropout_bwd_copy_kernel<float, kPath><<<grid, 256, 0, as_stream(stream)>>>((const float *)dy, (float *)dym, dcolsum, M, N, ld, rows_per_block, drop);
    else return fail(-1, "dropout_bwd_copy: unknown dtype %d", dtype);
    return check_launch("dropout_bwd_copy");
}

extern "C" {

int ecgvit_dropout_bwd_copy(const void *dy, void *dym, float *dcolsum, int M, int N, int64_t ld, float dropout_p,
                            int dropout_stream, const uint32_t *dropout_seed, int dtype, void *stream) {
    ECGVIT_REQUIRE(dy && dym && M > 0 && N > 0, "dropout_bwd_copy: bad arguments");
    ECGVIT_REQUIRE(N % 8 == 0 && ld % 8 == 0, "dropout_bwd_copy: N=%d and ld=%lld must be multiples of 8", N, (long long)ld);
    const DropoutParams drop = make_dropout(dropout_p, dropout_stream, dropout_seed);
    ECGVIT_REQUIRE(drop.threshold != 0, "dropout_bwd_copy: needs p > 0 and a seed");
    return dropout_bwd_copy_launch<false>(dy, dym, dcolsum, M, N, ld, drop, dtype, stream);
}

int ecgvit_dropout_bwd_copy_drop_path(const void *dy, void *dym, float *dcolsum, int M, int N, int64_t ld,
                                      float dropout_p, int dropout_stream, const uint32_t *dropout_seed, int dtype,
                                      float path_p, int path_stream, int rows_per_record, void *stream) {
    PathParams pp;
    if (int rc = make_path("dropout_bwd_copy_drop_path", path_p, path_stream, rows_per_record, dropout_seed, pp))
        return rc;
    if (pp.drop.threshold == 0)
        return ecgvit_dropout_bwd_copy(dy, dym, dcolsum, M, N, ld, dropout_p, dropout_stream, dropout_seed, dtype, stream);
    ECGVIT_REQUIRE(dy && dym && M > 0 && N > 0, "dropout_bwd_copy_drop_path: bad arguments");
    ECGVIT_REQUIRE(N % 8 == 0 && ld % 8 == 0, "dropout_bwd_copy: N=%d and ld=%lld must be multiples of 8", N, (long long)ld);
    DropoutPathParams drop;
    static_cast<DropoutParams &>(drop) = make_dropout(dropout_p, dropout_stream, dropout_seed);
    drop.path = pp;
    return dropout_bwd_copy_launch<true>(dy, dym, dcolsum, M, N, ld, drop, dtype, stream);
}

int ecgvit_cast_f32_to_bf16(const float *src, void *dst, int64_t n, void *stream) {
    ECGVIT_REQUIRE(src && dst && n >= 0, "cast: bad arguments");
    if (n == 0) return 0;
    const int grid = grid_for(n / 8 + 1, 256);
    cast_f32_bf16_kernel<<<grid, 256, 0, as_stream(stream)>>>(src, (bf16 *)dst, n);
    return check_launch("cast_f32_to_bf16");
}

}  // extern "C"

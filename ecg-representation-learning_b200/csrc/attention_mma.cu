// Tensor-core softmax attention for short sequences (N <= 64 tokens) with head dim 16 or 32, bf16 operands, fp32
// softmax statistics (head dim 64 runs on the tcgen05 kernels of attention_tc.cu).  One CTA (4 warps) per
// (batch, head); each warp owns 16 query rows, with warp-level mma.sync m16n8k16 (HMMA).
//
// The whole (b,h) problem lives in shared memory / registers, so the forward never materialises the [B,H,N,N]
// probability tensor that vit_pytorch's Attention.forward writes, and the backward recomputes P from the saved
// log-sum-exp.  q | k | v are read in place from the packed projection (no chunk / rearrange copies).
#include "common.cuh"

namespace ecgvit {

namespace {

#include "attention_mma.cuh"

template <int DH, int NT>
__global__ void __launch_bounds__(128) attention_fwd_mma_kernel(const bf16 *__restrict__ qkv, bf16 *__restrict__ o,
                                                                 float *__restrict__ lse, int N, int H, float scale,
                                                                 DropoutParams drop) {
    __shared__ __align__(16) bf16 sQ[NMAX][DH + 8];
    __shared__ __align__(16) bf16 sK[NMAX][DH + 8];
    __shared__ __align__(16) bf16 sV[NMAX][DH + 8];
    pdl_launch_dependents();
    pdl_wait();
    const int h = blockIdx.x % H, b = blockIdx.x / H;
    const int inner = H * DH;
    const int ld = 3 * inner;
    const bf16 *base = qkv + (int64_t)b * N * ld + h * DH;
    load_tile<DH>(sQ, base, ld, N);
    load_tile<DH>(sK, base + inner, ld, N);
    load_tile<DH>(sV, base + 2 * inner, ld, N);
    cp_async_wait_all();
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = warp * 16;
    if (m0 >= N) return;
    const int g = lane >> 2, t = lane & 3;

    float s[2 * NT][4];
    rows_times_transposed<DH, NT>(s, sQ, sK, m0, lane);
    const float sl2 = scale * LOG2E;
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 2 * NT; ++j) {
        if (8 * j + 8 > N) {  // warp-uniform: only the last one or two 8-key groups reach past the sequence
            const int c = 8 * j + 2 * t;
            if (c >= N) { s[j][0] = -INFINITY; s[j][2] = -INFINITY; }
            if (c + 1 >= N) { s[j][1] = -INFINITY; s[j][3] = -INFINITY; }
        }
        mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
        mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
    }
    mx0 = quad_max(mx0);
    mx1 = quad_max(mx1);
    const float nm0 = -mx0 * sl2, nm1 = -mx1 * sl2;  // exp2(s * sl2 - max * sl2): one FFMA per element
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int j = 0; j < 2 * NT; ++j) {
        s[j][0] = ex2_approx(fmaf(s[j][0], sl2, nm0)); s[j][1] = ex2_approx(fmaf(s[j][1], sl2, nm0));
        s[j][2] = ex2_approx(fmaf(s[j][2], sl2, nm1)); s[j][3] = ex2_approx(fmaf(s[j][3], sl2, nm1));
        sum0 += s[j][0] + s[j][1];
        sum1 += s[j][2] + s[j][3];
    }
    sum0 = quad_sum(sum0);
    sum1 = quad_sum(sum1);
    if (drop.threshold != 0) {
        // attention-probability dropout: mask the (still unnormalised) probabilities that feed P V; the row sums
        // keep normalising with the undropped values.  element index = ((b*H + h) * 64 + query) * 64 + key
        const uint32_t seed = __ldg(drop.seed);
        const uint32_t base0 = (static_cast<uint32_t>(blockIdx.x) * NMAX + (m0 + g)) * NMAX + 2 * t;
#pragma unroll
        for (int j = 0; j < 2 * NT; ++j) {
            float a0, a1;
            dropout_pair(drop, seed, base0 + 8 * j, a0, a1);
            s[j][0] *= a0; s[j][1] *= a1;
            dropout_pair(drop, seed, base0 + 8 * NMAX + 8 * j, a0, a1);
            s[j][2] *= a0; s[j][3] *= a1;
        }
    }
    uint32_t pa[NT][4];
#pragma unroll
    for (int kk = 0; kk < NT; ++kk) {
        pa[kk][0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
        pa[kk][1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
        pa[kk][2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[kk][3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
    }
    float acc[DH / 8][4];
#pragma unroll
    for (int j = 0; j < DH / 8; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
    frag_times_rows<DH, NT>(acc, pa, sV, lane);
    const int r0 = m0 + g, r1 = r0 + 8;
    bf16 *ob = o + (int64_t)b * N * inner + h * DH;
    store_rows<DH>(ob, inner, acc, r0, r1, N, t, 1.0f / sum0, 1.0f / sum1);
    if (t == 0) {
        float *l = lse + ((int64_t)b * H + h) * N;
        if (r0 < N) l[r0] = mx0 * scale + logf(sum0);
        if (r1 < N) l[r1] = mx1 * scale + logf(sum1);
    }
}

template <int DH, int NT>
__global__ void __launch_bounds__(128) attention_bwd_mma_kernel(const bf16 *__restrict__ qkv, const bf16 *__restrict__ o,
                                                                 const bf16 *__restrict__ d_o,
                                                                 const float *__restrict__ lse, bf16 *__restrict__ dqkv,
                                                                 int N, int H, float scale, DropoutParams drop) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    typedef bf16(*TileD)[DH + 8];
    typedef bf16(*TileN)[NMAX + 8];
    TileD sQ = reinterpret_cast<TileD>(smem_raw);
    TileD sK = sQ + NMAX, sV = sK + NMAX, sdO = sV + NMAX;
    TileN sP = reinterpret_cast<TileN>(sdO + NMAX);
    TileN sdS = sP + NMAX;

    float *sD = reinterpret_cast<float *>(sdS + NMAX);  // [NMAX] rowsum(dO * O)
    pdl_launch_dependents();
    pdl_wait();

    const int h = blockIdx.x % H, b = blockIdx.x / H;
    const int inner = H * DH;
    const int ld = 3 * inner;
    const bf16 *base = qkv + (int64_t)b * N * ld + h * DH;
    const bf16 *ob = o + (int64_t)b * N * inner + h * DH;
    const bf16 *dob = d_o + (int64_t)b * N * inner + h * DH;
    load_tile<DH>(sQ, base, ld, N);
    load_tile<DH>(sK, base + inner, ld, N);
    load_tile<DH>(sV, base + 2 * inner, ld, N);
    load_tile<DH>(sdO, dob, inner, N);
    // the O tile never goes to shared memory: its chunks stay in registers until dO has landed, then
    // D[r] = sum_d dO[r,d] * O[r,d] is reduced over the DH/8 consecutive threads that hold row r
    constexpr int VPR = DH / 8;
    constexpr int CHUNKS = (NMAX * VPR) / 128;
    uint4 oreg[CHUNKS];
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k) {
        const int i = threadIdx.x + k * 128;
        const int r = i / VPR, c = (i % VPR) * 8;
        oreg[k] = make_uint4(0u, 0u, 0u, 0u);
        if (r < N) oreg[k] = *reinterpret_cast<const uint4 *>(ob + r * inner + c);
    }
    cp_async_wait_all();
    __syncthreads();
#pragma unroll
    for (int k = 0; k < CHUNKS; ++k) {
        const int i = threadIdx.x + k * 128;
        const int r = i / VPR, c = (i % VPR) * 8;
        float ov[8], dv[8];
        const uint4 d4 = *reinterpret_cast<const uint4 *>(&sdO[r][c]);
        unpack_bf16x2(oreg[k].x, ov[0], ov[1]); unpack_bf16x2(oreg[k].y, ov[2], ov[3]);
        unpack_bf16x2(oreg[k].z, ov[4], ov[5]); unpack_bf16x2(oreg[k].w, ov[6], ov[7]);
        unpack_bf16x2(d4.x, dv[0], dv[1]); unpack_bf16x2(d4.y, dv[2], dv[3]);
        unpack_bf16x2(d4.z, dv[4], dv[5]); unpack_bf16x2(d4.w, dv[6], dv[7]);
        float part = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) part = fmaf(ov[e], dv[e], part);
#pragma unroll
        for (int off = VPR / 2; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
        if ((i % VPR) == 0) sD[r] = part;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = warp * 16;
    const int g = lane >> 2, t = lane & 3;
    bf16 *dq = dqkv + (int64_t)b * N * ld + h * DH;
    const bool active = m0 < N;  // this warp owns query rows (and, later, key rows) m0 .. m0+15

    if (active) {
        const int r0 = m0 + g, r1 = r0 + 8;
        const float D0 = sD[r0], D1 = sD[r1];
        const float *l = lse + ((int64_t)b * H + h) * N;
        const float nl0 = r0 < N ? -l[r0] * LOG2E : 0.f, nl1 = r1 < N ? -l[r1] * LOG2E : 0.f;

        float s[2 * NT][4], dp[2 * NT][4];
        rows_times_transposed<DH, NT>(s, sQ, sK, m0, lane);    // S = Q K^T
        rows_times_transposed<DH, NT>(dp, sdO, sV, m0, lane);  // dP = dO V^T
        const float sl2 = scale * LOG2E;
        const bool dropping = drop.threshold != 0;
        const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
        const uint32_t base0 = (static_cast<uint32_t>(blockIdx.x) * NMAX + r0) * NMAX + 2 * t;
        uint32_t dsa[NT][4];
#pragma unroll
        for (int j = 0; j < 2 * NT; ++j) {
            const int c = 8 * j + 2 * t;
            float p[4], ds[4], mk[4] = {1.f, 1.f, 1.f, 1.f};
            if (dropping) {
                dropout_pair(drop, seed, base0 + 8 * j, mk[0], mk[1]);
                dropout_pair(drop, seed, base0 + 8 * NMAX + 8 * j, mk[2], mk[3]);
            }
            // No validity tests: padded Q / K / V / dO rows are zero in shared memory, so whatever P and dS hold for
            // padded queries or keys multiplies zero rows in dQ = dS K, dK = dS^T Q, dV = P^T dO, or lands in rows that
            // are never stored.
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float pu = ex2_approx(fmaf(s[j][i], sl2, i < 2 ? nl0 : nl1));  // softmax probability
                ds[i] = pu * (dp[j][i] * mk[i] - (i < 2 ? D0 : D1)) * scale;        // dS uses the undropped P
                p[i] = pu * mk[i];                                                  // dV uses the dropped P
            }
            const uint32_t p01 = pack_bf16x2(p[0], p[1]), p23 = pack_bf16x2(p[2], p[3]);
            const uint32_t d01 = pack_bf16x2(ds[0], ds[1]), d23 = pack_bf16x2(ds[2], ds[3]);
            *reinterpret_cast<uint32_t *>(&sP[r0][c]) = p01;
            *reinterpret_cast<uint32_t *>(&sP[r1][c]) = p23;
            *reinterpret_cast<uint32_t *>(&sdS[r0][c]) = d01;
            *reinterpret_cast<uint32_t *>(&sdS[r1][c]) = d23;
            dsa[j >> 1][(j & 1) * 2] = d01;
            dsa[j >> 1][(j & 1) * 2 + 1] = d23;
        }
        // dQ = dS K
        float acc[DH / 8][4];
#pragma unroll
        for (int j = 0; j < DH / 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
        frag_times_rows<DH, NT>(acc, dsa, sK, lane);
        store_rows<DH>(dq, ld, acc, r0, r1, N, t, 1.f, 1.f);
    }
    __syncthreads();
    if (active) {
        const int r0 = m0 + g, r1 = r0 + 8;  // now key rows
        float acc[DH / 8][4];
#pragma unroll
        for (int j = 0; j < DH / 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
        transposed_times_rows<DH, NT>(acc, sdS, sQ, m0, lane);  // dK = dS^T Q
        store_rows<DH>(dq + inner, ld, acc, r0, r1, N, t, 1.f, 1.f);
#pragma unroll
        for (int j = 0; j < DH / 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
        transposed_times_rows<DH, NT>(acc, sP, sdO, m0, lane);  // dV = P^T dO
        store_rows<DH>(dq + 2 * inner, ld, acc, r0, r1, N, t, 1.f, 1.f);
    }
}

template <int DH> constexpr size_t bwd_smem_bytes() {
    return sizeof(bf16) * (4 * NMAX * (DH + 8) + 2 * NMAX * (NMAX + 8)) + sizeof(float) * NMAX;
}

template <int DH, int NT>
int launch_bwd(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, int B, int N, int H,
               float scale, DropoutParams drop, cudaStream_t stream) {
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(attention_bwd_mma_kernel<DH, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)bwd_smem_bytes<DH>());
        if (e != cudaSuccess) return fail((int)e, "attention_bwd_mma: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    launch_pdl(attention_bwd_mma_kernel<DH, NT>, dim3(B * H), dim3(128), bwd_smem_bytes<DH>(), stream,
               (const bf16 *)qkv, (const bf16 *)o, (const bf16 *)d_o, lse, (bf16 *)dqkv, N, H, scale, drop);
    return check_launch("attention_bwd_mma");
}

template <int DH, int NT>
int launch_fwd(const void *qkv, void *o, float *lse, int B, int N, int H, float scale, DropoutParams drop,
               cudaStream_t stream) {
    launch_pdl(attention_fwd_mma_kernel<DH, NT>, dim3(B * H), dim3(128), 0, stream, (const bf16 *)qkv, (bf16 *)o, lse, N,
               H, scale, drop);
    return check_launch("attention_fwd_mma");
}

}  // namespace

bool attention_mma_supported(int N, int dh) { return N <= NMAX && (dh == 16 || dh == 32); }

// the number of 16-key tiles is a template parameter so the inner loops carry no runtime predicates
#define ECGVIT_ATTN_DISPATCH(FN, ...)                                                     \
    do {                                                                                  \
        const int nt = (N + 15) / 16;                                                     \
        switch (dh * 8 + nt) {                                                            \
            case 16 * 8 + 1: return FN<16, 1>(__VA_ARGS__);                               \
            case 16 * 8 + 2: return FN<16, 2>(__VA_ARGS__);                               \
            case 16 * 8 + 3: return FN<16, 3>(__VA_ARGS__);                               \
            case 16 * 8 + 4: return FN<16, 4>(__VA_ARGS__);                               \
            case 32 * 8 + 1: return FN<32, 1>(__VA_ARGS__);                               \
            case 32 * 8 + 2: return FN<32, 2>(__VA_ARGS__);                               \
            case 32 * 8 + 3: return FN<32, 3>(__VA_ARGS__);                               \
            case 32 * 8 + 4: return FN<32, 4>(__VA_ARGS__);                               \
            default: return fail(-1, "attention_mma: unsupported head dim %d / length %d", dh, N); \
        }                                                                                 \
    } while (0)

int attention_fwd_mma(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale,
                      DropoutParams drop, cudaStream_t stream) {
    ECGVIT_ATTN_DISPATCH(launch_fwd, qkv, o, lse, B, N, H, scale, drop, stream);
}

int attention_bwd_mma(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, int B, int N,
                      int H, int dh, float scale, DropoutParams drop, cudaStream_t stream) {
    ECGVIT_ATTN_DISPATCH(launch_bwd, qkv, o, d_o, lse, dqkv, B, N, H, scale, drop, stream);
}

}  // namespace ecgvit

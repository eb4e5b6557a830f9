// Tiled ("flash") softmax attention for sequences longer than one 64-token tile with head dim 32 (head dim 64 runs on
// the tcgen05 kernels of attention_tc.cu).  bf16 operands, fp32 statistics, mma.sync m16n8k16; 64 queries x 64 keys
// per inner step, K / V (or Q / dO) tiles double-buffered with cp.async.
//
// Nothing of size N x N is ever written: forward keeps a running (max, sum) per query row and saves the log-sum-exp;
// backward recomputes the probabilities from it in two kernels that need no atomics:
//   flash_bwd_dq_kernel   one CTA per 64-query tile, walks the key tiles:   dQ  = sum_k dS K
//   flash_bwd_dkv_kernel  one CTA per 64-key tile,   walks the query tiles: dK  = sum_q dS^T Q,  dV = sum_q P^T dO
// The second one computes the TRANSPOSED products (S^T = K Q^T, dP^T = V dO^T) so that P^T / dS^T come out of the tensor
// cores already in A-fragment layout; no probability tile goes through shared memory.
//
// Attention-probability dropout uses the same counter as the short kernels: element index
// ((b*H + h) * Np + query) * Np + key with Np = N rounded up to 64 (must stay below 2^32).
#include "common.cuh"

namespace ecgvit {

namespace {

#include "attention_mma.cuh"

constexpr int TILE = NMAX;  // 64 rows per tile

// rows [row0, row0 + 64) of an [N x DH] head matrix (row stride ld) -> smem tile, zero-filling rows >= N
template <int DH>
__device__ __forceinline__ void load_rows(bf16 (*dst)[DH + 8], const bf16 *src, int64_t ld, int row0, int N) {
    // 128 threads: thread t owns 16-byte chunk (t % VPR) of tile rows t / VPR + k * (128 / VPR); constant pointer steps
    constexpr int VPR = DH / 8;
    constexpr int ROWS_PER_STEP = 128 / VPR;
    const int c = (threadIdx.x % VPR) * 8;
    int r = threadIdx.x / VPR;
    const bf16 *p = src + (int64_t)(row0 + r) * ld + c;
    bf16 *q = &dst[r][c];
    const int64_t pstep = (int64_t)ROWS_PER_STEP * ld;
    if (row0 + TILE <= N) {  // interior tile (block-uniform): no bounds tests
#pragma unroll
        for (int k = 0; k < TILE / ROWS_PER_STEP; ++k) {
            cp_async16(q, p);
            p += pstep;
            q += ROWS_PER_STEP * (DH + 8);
        }
    } else {
#pragma unroll
        for (int k = 0; k < TILE / ROWS_PER_STEP; ++k) {
            if (row0 + r < N) cp_async16(q, p);
            else *reinterpret_cast<uint4 *>(q) = make_uint4(0u, 0u, 0u, 0u);
            r += ROWS_PER_STEP;
            p += pstep;
            q += ROWS_PER_STEP * (DH + 8);
        }
    }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <int DH> struct FlashSmem {
    typedef bf16 (*Tile)[DH + 8];
    static constexpr size_t TILE_BYTES = sizeof(bf16) * TILE * (DH + 8);
};

// ---------------------------------------------------------------------------------------------------------------
template <int DH>
__global__ void __launch_bounds__(128) flash_fwd_kernel(const bf16 *__restrict__ qkv, bf16 *__restrict__ o,
                                                         float *__restrict__ lse, int N, int H, float scale,
                                                         DropoutParams drop) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    typedef typename FlashSmem<DH>::Tile Tile;
    Tile sQ = reinterpret_cast<Tile>(smem_raw);
    Tile sK0 = sQ + TILE, sV0 = sQ + 3 * TILE;  // two buffers each: [buf * TILE]
    // grid: one flat x over (b*H + h, query tile), query tile fastest (B * H may exceed the 65535 of grid.y)
    const int bh = (int)(blockIdx.x / ((N + TILE - 1) / TILE)), h = bh % H, b = bh / H;
    const int q0 = (int)(blockIdx.x - bh * ((N + TILE - 1) / TILE)) * TILE;
    const int inner = H * DH;
    const int64_t ld = 3 * (int64_t)inner;
    const bf16 *base = qkv + (int64_t)b * N * ld + h * DH;
    const int n_kt = (N + TILE - 1) / TILE;
    const int Np = n_kt * TILE;
    load_rows<DH>(sQ, base, ld, q0, N);
    load_rows<DH>(sK0, base + inner, ld, 0, N);
    load_rows<DH>(sV0, base + 2 * inner, ld, 0, N);
    cp_async_commit();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = warp * 16;
    const int g = lane >> 2, t = lane & 3;
    const int r0 = q0 + m0 + g, r1 = r0 + 8;  // global query rows of this thread
    const float sl2 = scale * LOG2E;
    const bool dropping = drop.threshold != 0;
    const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
    float mx0 = -INFINITY, mx1 = -INFINITY, sum0 = 0.f, sum1 = 0.f;
    float acc[DH / 8][4];
#pragma unroll
    for (int j = 0; j < DH / 8; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;

    for (int kt = 0; kt < n_kt; ++kt) {
        const int buf = kt & 1;
        Tile sKb = sK0 + buf * TILE, sVb = sV0 + buf * TILE;
        cp_async_wait0();
        __syncthreads();  // tile kt has landed, and every warp is done with the buffer tile kt + 1 goes into
        if (kt + 1 < n_kt) {
            load_rows<DH>(sK0 + (buf ^ 1) * TILE, base + inner, ld, (kt + 1) * TILE, N);
            load_rows<DH>(sV0 + (buf ^ 1) * TILE, base + 2 * inner, ld, (kt + 1) * TILE, N);
        }
        cp_async_commit();
        float s[8][4];
        rows_times_transposed<DH, 4>(s, sQ, sKb, m0, lane);
        const int k0 = kt * TILE;
        float tmx0 = mx0, tmx1 = mx1;
        if (k0 + TILE > N) {  // only the last key tile has columns past the sequence (block-uniform)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = k0 + 8 * j + 2 * t;
                if (c >= N) { s[j][0] = -INFINITY; s[j][2] = -INFINITY; }
                if (c + 1 >= N) { s[j][1] = -INFINITY; s[j][3] = -INFINITY; }
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            tmx0 = fmaxf(tmx0, fmaxf(s[j][0], s[j][1]));
            tmx1 = fmaxf(tmx1, fmaxf(s[j][2], s[j][3]));
        }
        tmx0 = quad_max(tmx0);
        tmx1 = quad_max(tmx1);
        // every key tile holds at least one valid key (k0 < N), so the running maxima are finite from tile 0 on
        const float alpha0 = ex2_approx((mx0 - tmx0) * sl2), alpha1 = ex2_approx((mx1 - tmx1) * sl2);
        mx0 = tmx0;
        mx1 = tmx1;
        const float nm0 = -mx0 * sl2, nm1 = -mx1 * sl2;  // exp2(s * sl2 - max * sl2): one FFMA per element
        float ts0 = 0.f, ts1 = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            s[j][0] = ex2_approx(fmaf(s[j][0], sl2, nm0)); s[j][1] = ex2_approx(fmaf(s[j][1], sl2, nm0));
            s[j][2] = ex2_approx(fmaf(s[j][2], sl2, nm1)); s[j][3] = ex2_approx(fmaf(s[j][3], sl2, nm1));
            ts0 += s[j][0] + s[j][1];
            ts1 += s[j][2] + s[j][3];
        }
        sum0 = sum0 * alpha0 + quad_sum(ts0);
        sum1 = sum1 * alpha1 + quad_sum(ts1);
#pragma unroll
        for (int j = 0; j < DH / 8; ++j) {
            acc[j][0] *= alpha0; acc[j][1] *= alpha0;
            acc[j][2] *= alpha1; acc[j][3] *= alpha1;
        }
        if (dropping) {
            const uint32_t e0 = (static_cast<uint32_t>(bh) * Np + r0) * Np + k0 + 2 * t;
            const uint32_t e1 = e0 + 8u * Np;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float a0, a1;
                dropout_pair(drop, seed, e0 + 8 * j, a0, a1);
                s[j][0] *= a0; s[j][1] *= a1;
                dropout_pair(drop, seed, e1 + 8 * j, a0, a1);
                s[j][2] *= a0; s[j][3] *= a1;
            }
        }
        uint32_t pa[4][4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            pa[kk][0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
            pa[kk][1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
            pa[kk][2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
            pa[kk][3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        }
        frag_times_rows<DH, 4>(acc, pa, sVb, lane);
    }
    bf16 *ob = o + (int64_t)b * N * inner + h * DH;
    store_rows<DH>(ob, inner, acc, r0, r1, N, t, 1.0f / sum0, 1.0f / sum1);
    if (t == 0) {
        float *l = lse + (int64_t)bh * N;
        if (r0 < N) l[r0] = mx0 * scale + logf(sum0);
        if (r1 < N) l[r1] = mx1 * scale + logf(sum1);
    }
}

// D[b, h, i] = sum_d dO[i, d] * O[i, d]; one warp per (row, head)
template <int DH>
__global__ void __launch_bounds__(256) flash_bwd_dot_kernel(const bf16 *__restrict__ o, const bf16 *__restrict__ d_o,
                                                             float *__restrict__ D, int B, int N, int H) {
    const int lane = threadIdx.x & 31;
    const int64_t wid = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);  // (b * N + i) * H + h
    if (wid >= (int64_t)B * N * H) return;
    const int h = (int)(wid % H);
    const int64_t row = wid / H;  // b * N + i
    const bf16 *po = o + row * (int64_t)(H * DH) + h * DH, *pd = d_o + row * (int64_t)(H * DH) + h * DH;
    float part = 0.f;
    for (int c = lane * 2; c < DH; c += 64) {
        float a0, a1, b0, b1;
        unpack_bf16x2(*reinterpret_cast<const uint32_t *>(po + c), a0, a1);
        unpack_bf16x2(*reinterpret_cast<const uint32_t *>(pd + c), b0, b1);
        part = fmaf(a0, b0, fmaf(a1, b1, part));
    }
    part = warp_sum(part);
    if (lane == 0) {
        const int64_t b = row / N, i = row % N;
        D[(b * H + h) * N + i] = part;
    }
}

// ---------------------------------------------------------------------------------------------------------------
template <int DH>
__global__ void __launch_bounds__(128) flash_bwd_dq_kernel(const bf16 *__restrict__ qkv, const bf16 *__restrict__ d_o,
                                                            const float *__restrict__ lse, const float *__restrict__ D,
                                                            bf16 *__restrict__ dqkv, int N, int H, float scale,
                                                            DropoutParams drop) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    typedef typename FlashSmem<DH>::Tile Tile;
    Tile sQ = reinterpret_cast<Tile>(smem_raw);
    Tile sdO = sQ + TILE;
    Tile sK0 = sQ + 2 * TILE, sV0 = sQ + 4 * TILE;  // two buffers each: [buf * TILE]
    const int bh = (int)(blockIdx.x / ((N + TILE - 1) / TILE)), h = bh % H, b = bh / H;  // grid as in flash_fwd_kernel
    const int q0 = (int)(blockIdx.x - bh * ((N + TILE - 1) / TILE)) * TILE;
    const int inner = H * DH;
    const int64_t ld = 3 * (int64_t)inner;
    const bf16 *base = qkv + (int64_t)b * N * ld + h * DH;
    const bf16 *dob = d_o + (int64_t)b * N * inner + h * DH;
    const int n_kt = (N + TILE - 1) / TILE;
    const int Np = n_kt * TILE;
    load_rows<DH>(sQ, base, ld, q0, N);
    load_rows<DH>(sdO, dob, inner, q0, N);
    load_rows<DH>(sK0, base + inner, ld, 0, N);
    load_rows<DH>(sV0, base + 2 * inner, ld, 0, N);
    cp_async_commit();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = warp * 16;
    const int g = lane >> 2, t = lane & 3;
    const int r0 = q0 + m0 + g, r1 = r0 + 8;
    const float sl2 = scale * LOG2E;
    const bool dropping = drop.threshold != 0;
    const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
    const float *lrow = lse + (int64_t)bh * N, *drow = D + (int64_t)bh * N;
    const float l0 = r0 < N ? lrow[r0] * LOG2E : 0.f, l1 = r1 < N ? lrow[r1] * LOG2E : 0.f;
    const float D0 = r0 < N ? drow[r0] : 0.f, D1 = r1 < N ? drow[r1] : 0.f;
    float acc[DH / 8][4];
#pragma unroll
    for (int j = 0; j < DH / 8; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;

    for (int kt = 0; kt < n_kt; ++kt) {
        const int buf = kt & 1;
        Tile sKb = sK0 + buf * TILE, sVb = sV0 + buf * TILE;
        cp_async_wait0();
        __syncthreads();
        if (kt + 1 < n_kt) {
            load_rows<DH>(sK0 + (buf ^ 1) * TILE, base + inner, ld, (kt + 1) * TILE, N);
            load_rows<DH>(sV0 + (buf ^ 1) * TILE, base + 2 * inner, ld, (kt + 1) * TILE, N);
        }
        cp_async_commit();
        float s[8][4], dp[8][4];
        rows_times_transposed<DH, 4>(s, sQ, sKb, m0, lane);    // S  = Q K^T
        rows_times_transposed<DH, 4>(dp, sdO, sVb, m0, lane);  // dP = dO V^T
        const int k0 = kt * TILE;
        const uint32_t e0 = (static_cast<uint32_t>(bh) * Np + r0) * Np + k0 + 2 * t;
        const uint32_t e1 = e0 + 8u * Np;
        uint32_t dsa[4][4];
        // No validity tests: padded Q / K / V / dO rows are zero in shared memory, so what P and dS hold for padded
        // queries or keys only ever multiplies zero rows or lands in rows that are never stored.
        const float nl0 = -l0, nl1 = -l1;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = k0 + 8 * j + 2 * t;
            float mk[4] = {1.f, 1.f, 1.f, 1.f}, ds[4];
            if (dropping) {
                dropout_pair(drop, seed, e0 + 8 * j, mk[0], mk[1]);
                dropout_pair(drop, seed, e1 + 8 * j, mk[2], mk[3]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float pu = ex2_approx(fmaf(s[j][i], sl2, i < 2 ? nl0 : nl1));
                ds[i] = pu * (dp[j][i] * mk[i] - (i < 2 ? D0 : D1)) * scale;
            }
            dsa[j >> 1][(j & 1) * 2] = pack_bf16x2(ds[0], ds[1]);
            dsa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(ds[2], ds[3]);
        }
        frag_times_rows<DH, 4>(acc, dsa, sKb, lane);  // dQ += dS K
    }
    bf16 *dq = dqkv + (int64_t)b * N * ld + h * DH;
    store_rows<DH>(dq, (int)ld, acc, r0 - 0, r1 - 0, N, t, 1.f, 1.f);
}

// ---------------------------------------------------------------------------------------------------------------
template <int DH>
__global__ void __launch_bounds__(128) flash_bwd_dkv_kernel(const bf16 *__restrict__ qkv, const bf16 *__restrict__ d_o,
                                                             const float *__restrict__ lse, const float *__restrict__ D,
                                                             bf16 *__restrict__ dqkv, int N, int H, float scale,
                                                             DropoutParams drop) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    typedef typename FlashSmem<DH>::Tile Tile;
    Tile sK = reinterpret_cast<Tile>(smem_raw);
    Tile sV = sK + TILE;
    Tile sQ0 = sK + 2 * TILE, sdO0 = sK + 4 * TILE;  // two buffers each: [buf * TILE]
    float *sL = reinterpret_cast<float *>(sK + 6 * TILE);  // [2][TILE] lse * log2(e) of the query tile
    float *sD = sL + 2 * TILE;                             // [2][TILE]
    const int bh = (int)(blockIdx.x / ((N + TILE - 1) / TILE)), h = bh % H, b = bh / H;  // grid as in flash_fwd_kernel
    const int k0 = (int)(blockIdx.x - bh * ((N + TILE - 1) / TILE)) * TILE;
    const int inner = H * DH;
    const int64_t ld = 3 * (int64_t)inner;
    const bf16 *base = qkv + (int64_t)b * N * ld + h * DH;
    const bf16 *dob = d_o + (int64_t)b * N * inner + h * DH;
    const float *lrow = lse + (int64_t)bh * N, *drow = D + (int64_t)bh * N;
    const int n_qt = (N + TILE - 1) / TILE;
    const int Np = n_qt * TILE;
    auto load_q_side = [&](int qt, int buf) {
        load_rows<DH>(sQ0 + buf * TILE, base, ld, qt * TILE, N);
        load_rows<DH>(sdO0 + buf * TILE, dob, inner, qt * TILE, N);
        if (threadIdx.x < TILE) {
            const int r = qt * TILE + threadIdx.x;
            sL[buf * TILE + threadIdx.x] = r < N ? lrow[r] * LOG2E : 0.f;
            sD[buf * TILE + threadIdx.x] = r < N ? drow[r] : 0.f;
        }
    };
    load_rows<DH>(sK, base + inner, ld, k0, N);
    load_rows<DH>(sV, base + 2 * inner, ld, k0, N);
    load_q_side(0, 0);
    cp_async_commit();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = warp * 16;  // key rows of this warp inside the tile
    const int g = lane >> 2, t = lane & 3;
    const int r0 = k0 + m0 + g, r1 = r0 + 8;  // global key rows of this thread
    const float sl2 = scale * LOG2E;
    const bool dropping = drop.threshold != 0;
    const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
    float dk[DH / 8][4], dv[DH / 8][4];
#pragma unroll
    for (int j = 0; j < DH / 8; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) { dk[j][i] = 0.f; dv[j][i] = 0.f; }

    for (int qt = 0; qt < n_qt; ++qt) {
        const int buf = qt & 1;
        Tile sQb = sQ0 + buf * TILE, sdOb = sdO0 + buf * TILE;
        cp_async_wait0();
        __syncthreads();
        if (qt + 1 < n_qt) load_q_side(qt + 1, buf ^ 1);
        cp_async_commit();
        float st[8][4], dpt[8][4];
        rows_times_transposed<DH, 4>(st, sK, sQb, m0, lane);    // S^T  = K Q^T   (rows = keys, columns = queries)
        rows_times_transposed<DH, 4>(dpt, sV, sdOb, m0, lane);  // dP^T = V dO^T
        const int q0 = qt * TILE;
        const float *L = sL + buf * TILE, *Dq = sD + buf * TILE;
        uint32_t pa[4][4], dsa[4][4];
        // no validity tests (see flash_bwd_dq_kernel): padded rows are zero in shared memory
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = 8 * j + 2 * t;  // query column inside the tile
            float p[4], ds[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int qi = q0 + c + (i & 1);       // global query
                const int kj = (i < 2) ? r0 : r1;      // global key
                const float pu = ex2_approx(fmaf(st[j][i], sl2, -L[c + (i & 1)]));
                float mk = 1.f;
                if (dropping) mk = dropout_one(drop, seed, (static_cast<uint32_t>(bh) * Np + qi) * Np + kj);
                ds[i] = pu * (dpt[j][i] * mk - Dq[c + (i & 1)]) * scale;
                p[i] = pu * mk;
            }
            pa[j >> 1][(j & 1) * 2] = pack_bf16x2(p[0], p[1]);
            pa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(p[2], p[3]);
            dsa[j >> 1][(j & 1) * 2] = pack_bf16x2(ds[0], ds[1]);
            dsa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(ds[2], ds[3]);
        }
        frag_times_rows<DH, 4>(dv, pa, sdOb, lane);  // dV += P^T dO
        frag_times_rows<DH, 4>(dk, dsa, sQb, lane);  // dK += dS^T Q
    }
    bf16 *dq = dqkv + (int64_t)b * N * ld + h * DH;
    store_rows<DH>(dq + inner, (int)ld, dk, r0, r1, N, t, 1.f, 1.f);
    store_rows<DH>(dq + 2 * inner, (int)ld, dv, r0, r1, N, t, 1.f, 1.f);
}

template <typename K> int set_smem(K kernel, size_t bytes, const char *what) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(e));
    return 0;
}

template <int DH>
int flash_fwd(const void *qkv, void *o, float *lse, int B, int N, int H, float scale, DropoutParams drop,
              cudaStream_t stream) {
    const size_t smem = 5 * FlashSmem<DH>::TILE_BYTES;
    static bool attr_set = false;
    if (!attr_set) {
        int rc = set_smem(flash_fwd_kernel<DH>, smem, "attention_flash_fwd");
        if (rc) return rc;
        attr_set = true;
    }
    const unsigned grid = (unsigned)((N + TILE - 1) / TILE) * (unsigned)(B * H);
    flash_fwd_kernel<DH><<<grid, 128, smem, stream>>>((const bf16 *)qkv, (bf16 *)o, lse, N, H, scale, drop);
    return check_launch("attention_flash_fwd");
}

template <int DH>
int flash_bwd(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, float *dscratch, int B,
              int N, int H, float scale, DropoutParams drop, cudaStream_t stream) {
    const size_t smem_dq = 6 * FlashSmem<DH>::TILE_BYTES;
    const size_t smem_dkv = 6 * FlashSmem<DH>::TILE_BYTES + 4 * TILE * sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        int rc = set_smem(flash_bwd_dq_kernel<DH>, smem_dq, "attention_flash_bwd_dq");
        if (rc) return rc;
        rc = set_smem(flash_bwd_dkv_kernel<DH>, smem_dkv, "attention_flash_bwd_dkv");
        if (rc) return rc;
        attr_set = true;
    }
    const int64_t rows = (int64_t)B * N * H;
    flash_bwd_dot_kernel<DH><<<(unsigned)((rows + 7) / 8), 256, 0, stream>>>((const bf16 *)o, (const bf16 *)d_o, dscratch,
                                                                               B, N, H);
    int rc = check_launch("attention_flash_bwd_dot");
    if (rc) return rc;
    const unsigned grid = (unsigned)((N + TILE - 1) / TILE) * (unsigned)(B * H);   // flat, as in flash_fwd
    flash_bwd_dq_kernel<DH><<<grid, 128, smem_dq, stream>>>((const bf16 *)qkv, (const bf16 *)d_o, lse, dscratch,
                                                             (bf16 *)dqkv, N, H, scale, drop);
    rc = check_launch("attention_flash_bwd_dq");
    if (rc) return rc;
    flash_bwd_dkv_kernel<DH><<<grid, 128, smem_dkv, stream>>>((const bf16 *)qkv, (const bf16 *)d_o, lse, dscratch,
                                                               (bf16 *)dqkv, N, H, scale, drop);
    return check_launch("attention_flash_bwd_dkv");
}

}  // namespace

bool attention_flash_supported(int N, int dh) { return N > NMAX && dh == 32; }

int attention_fwd_flash(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale,
                        DropoutParams drop, cudaStream_t stream) {
    ECGVIT_REQUIRE(dh == 32, "attention_fwd_flash: head dim %d (only 32)", dh);
    return flash_fwd<32>(qkv, o, lse, B, N, H, scale, drop, stream);
}

int attention_bwd_flash(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, float *dscratch,
                        int B, int N, int H, int dh, float scale, DropoutParams drop, cudaStream_t stream) {
    ECGVIT_REQUIRE(dh == 32, "attention_bwd_flash: head dim %d (only 32)", dh);
    return flash_bwd<32>(qkv, o, d_o, lse, dqkv, dscratch, B, N, H, scale, drop, stream);
}

}  // namespace ecgvit

// fp32 FFMA GEMM (parity mode):  C[m,n] = sum_k A(m,k) * B(n,k) with the same fused epilogues as the tcgen05
// kernel.  fp32 logits / loss must match the reference's CPU fp32 model to 1e-5 relative (BASELINE.json
// north_star), which no tensor-core input format reaches, so the fp32 mode contracts on the FFMA pipe.
// It is the precision mode of the product for small configurations (cfg1), not a fallback for bf16.
#include "common.cuh"

namespace ecgvit {

namespace {

constexpr int TM = 64, TN = 64, TK = 16;

template <int MODE>
__global__ void __launch_bounds__(256) gemm_ffma_kernel(const float *__restrict__ A, int64_t sAm, int64_t sAk,
                                                         const float *__restrict__ B, int64_t sBn, int64_t sBk,
                                                         int M, int N, int K, EpiParams ep) {
    __shared__ float As[TK][TM + 4];
    __shared__ float Bs[TK][TN + 4];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, 4 x 4 outputs each
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
    const bool a_k_contig = (sAk == 1), b_k_contig = (sBk == 1);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < K; k0 += TK) {
#pragma unroll
        for (int i = tid; i < TM * TK; i += 256) {
            int m, k;
            if (a_k_contig) { m = i / TK; k = i % TK; } else { k = i / TM; m = i % TM; }
            const int gm = m0 + m, gk = k0 + k;
            As[k][m] = (gm < M && gk < K) ? A[gm * sAm + gk * sAk] : 0.f;
        }
#pragma unroll
        for (int i = tid; i < TN * TK; i += 256) {
            int n, k;
            if (b_k_contig) { n = i / TK; k = i % TK; } else { k = i / TN; n = i % TN; }
            const int gn = n0 + n, gk = k0 + k;
            Bs[k][n] = (gn < N && gk < K) ? B[gn * sBn + gk * sBk] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < TK; ++k) {
            const float4 a = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    const int col = n0 + tx * 4;
    if (MODE == ECGVIT_EPI_BIAS_SUB_ROWSQ) {
        // row partial of r^2 over this 64-column tile: the 16 threads of a row (tx, one half-warp) fold in a fixed order
        float *rowsq = reinterpret_cast<float *>(ep.out2);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int row = m0 + ty * 4 + i;
            float s = 0.f;
            if (col < N && row < M) {
                epilogue_store<MODE, float, 4, true>(ep, row, col, acc[i]);
#pragma unroll
                for (int j = 0; j < 4; ++j) s = fmaf(acc[i][j], acc[i][j], s);
            }
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (tx == 0 && row < M) rowsq[(int64_t)blockIdx.x * M + row] = s;
        }
        return;
    }
    if (col < N) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int row = m0 + ty * 4 + i;
            if (row < M) epilogue_store<MODE, float, 4, true>(ep, row, col, acc[i]);
        }
    }
}

}  // namespace

int gemm_f32_ffma(const ecgvit_gemm_args *g, cudaStream_t stream) {
    ECGVIT_REQUIRE(g->M > 0 && g->N > 0 && g->K > 0, "gemm: empty problem M=%d N=%d K=%d", g->M, g->N, g->K);
    ECGVIT_REQUIRE(g->N % 4 == 0 && g->ldo % 4 == 0, "gemm(f32): N=%d and ldo=%lld must be multiples of 4", g->N,
                   (long long)g->ldo);
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(g->out) & 15) == 0, "gemm(f32): out must be 16-byte aligned");
    ECGVIT_REQUIRE(g->epilogue != ECGVIT_EPI_BIAS_SUB_ROWSQ || (g->aux != nullptr && g->out2 != nullptr),
                   "gemm(f32): the row-square epilogue needs aux (target) and out2 (row partials)");
    const float *A = reinterpret_cast<const float *>(g->A), *B = reinterpret_cast<const float *>(g->B);
    const int64_t sAm = g->a_kmajor ? g->lda : 1, sAk = g->a_kmajor ? 1 : g->lda;
    const int64_t sBn = g->b_kmajor ? g->ldb : 1, sBk = g->b_kmajor ? 1 : g->ldb;
    EpiParams ep{g->out, g->out2, g->aux, g->bias, g->ldo, make_dropout(g->dropout_p, g->dropout_stream, g->dropout_seed)};
    dim3 grid((g->N + TN - 1) / TN, (g->M + TM - 1) / TM);
    switch (g->epilogue) {
#define ECGVIT_CASE(MODE) \
    case MODE: gemm_ffma_kernel<MODE><<<grid, 256, 0, stream>>>(A, sAm, sAk, B, sBn, sBk, g->M, g->N, g->K, ep); break;
        ECGVIT_CASE(ECGVIT_EPI_STORE)
        ECGVIT_CASE(ECGVIT_EPI_BIAS_RES)
        ECGVIT_CASE(ECGVIT_EPI_BIAS_GELU)
        ECGVIT_CASE(ECGVIT_EPI_DGELU)
        ECGVIT_CASE(ECGVIT_EPI_ATOMIC_F32)
        ECGVIT_CASE(ECGVIT_EPI_BIAS_SUB_ROWSQ)
#undef ECGVIT_CASE
        default: return fail(-1, "gemm(f32): unknown epilogue %d", g->epilogue);
    }
    return check_launch("gemm_ffma");
}

}  // namespace ecgvit

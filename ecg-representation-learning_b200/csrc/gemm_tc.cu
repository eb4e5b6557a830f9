// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[m,n] = sum_k A(m,k) * B(n,k), bf16 operands, fp32 accumulate.
//
// Persistent, warp-specialised, one CTA PAIR (cluster of 2, tcgen05 cta_group::2) per 256 x BN tile: see gemm_tc_pair.cuh.
// Both operands may be K-major (row-major [rows, K]) or MN-major (row-major [K, rows]); the latter is what the
// autograd dgrad (B = W[N,K] read as [K-out, n]) and wgrad (A = dY^T, B = X^T) contractions need, so no
// transposed copies of activations or weights are ever materialised.
//
// Replaces: nn.Linear forward/backward library GEMMs inside vit_pytorch (reference call site
// /root/reference/ecg_transformer/models/ecg_vit.py:141 and autograd at models/train.py:280).
#include "common.cuh"
#include "ptx.cuh"

#include <cudaTypedefs.h>
#include <stdlib.h>

namespace ecgvit {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle row
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BM * BK * 2;

#include "gemm_tc_pair.cuh"

// ---- host side ------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (fn == nullptr) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

// 2-D bf16 tensor map over a row-major [outer, inner] matrix with leading dimension ld (elements)
int make_tmap(CUtensorMap *tm, const void *base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_inner,
              uint32_t box_outer, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B, bool fp32 = false) {
    PFN_cuTensorMapEncodeTiled_v12000 enc = get_encode_fn();
    if (enc == nullptr) return fail(-2, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {ld * (fp32 ? 4 : 2)};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                     const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(-3, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

// CTA pairs the persistent GEMM grid may use: all of them (SMs / 2) unless ecgvit_set_gemm_sm_budget() or the environment
// variable ECGVIT_GEMM_CLUSTERS lowered it (data-parallel runs leave a few SMs to NCCL's collective kernels: a persistent
// grid that cannot place its last CTAs runs a second, nearly empty wave)
int g_gemm_clusters = -1;
int gemm_clusters() {
    if (g_gemm_clusters < 0) {
        const char *e = getenv("ECGVIT_GEMM_CLUSTERS");
        const int all = sm_count() / 2;
        int v = e != nullptr ? atoi(e) : all;
        g_gemm_clusters = (v >= 1 && v <= all) ? v : all;
    }
    return g_gemm_clusters;
}

// Counters of the in-kernel unit scheduler: one (next unit, clusters done) pair per launch, taken round-robin from a static
// array.  A kernel leaves its pair at zero when its last cluster runs dry, so a slot can be re-used by any later launch
// (a replayed CUDA graph re-uses the slots baked into its nodes); 4096 slots keep concurrent launches apart.
constexpr int kSchedSlots = 4096;
__device__ int g_sched_ctr[2 * kSchedSlots];
int *next_sched_slot() {
    static int *base = nullptr;
    static unsigned next = 0;
    if (base == nullptr) {
        void *p = nullptr;
        if (cudaGetSymbolAddress(&p, g_sched_ctr) != cudaSuccess) return nullptr;
        base = static_cast<int *>(p);
    }
    return base + 2 * (__atomic_fetch_add(&next, 1u, __ATOMIC_RELAXED) % kSchedSlots);
}

template <int BN, bool A_MN, bool B_MN, int MODE, bool kPath = false>
int launch_pair(const ecgvit_gemm_args *g, int split_k, cudaStream_t stream, const PathParams *path = nullptr) {
    constexpr bool kWide = MODE == ECGVIT_EPI_BIAS_RES_F32;   // fp32 residual stream: 128-byte staging rows
    using Cfg = PairCfgFor<BN, B_MN, MODE>;
    CUtensorMap ta, tb;
    int rc;
    if (!A_MN) rc = make_tmap(&ta, g->A, g->K, g->M, g->lda, BK, BM);
    else rc = make_tmap(&ta, g->A, g->M, g->K, g->lda, 64, BK);
    if (rc) return rc;
    if (!B_MN) rc = make_tmap(&tb, g->B, g->K, g->N, g->ldb, BK, Cfg::B_HALF);
    else rc = make_tmap(&tb, g->B, g->N, g->K, g->ldb, 64, BK);
    if (rc) return rc;
    // outputs leave (and the residual / pre-activation operand arrives) through TMA on 32-row x 32-column tiles
    // with 64-byte swizzle; TMA clips at M x N
    CUtensorMap to = ta, to2 = ta, tx = ta;
    if (kWide) {
        if ((rc = make_tmap(&to, g->out, g->N, g->M, g->ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B, true))) return rc;
        if ((rc = make_tmap(&tx, g->aux, g->N, g->M, g->ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B, true))) return rc;
    } else if (MODE == ECGVIT_EPI_ATOMIC_F32) {
        // fp32 partial sums are added into the gradient buffer by TMA reduce (cp.reduce.async.bulk.tensor .add)
        if ((rc = make_tmap(&to, g->out, g->N, g->M, g->ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B, true))) return rc;
    } else {
        if ((rc = make_tmap(&to, g->out, g->N, g->M, g->ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
        if (MODE == ECGVIT_EPI_BIAS_GELU &&
            (rc = make_tmap(&to2, g->out2, g->N, g->M, g->ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
        if ((MODE == ECGVIT_EPI_BIAS_RES || MODE == ECGVIT_EPI_DGELU || MODE == ECGVIT_EPI_BIAS_SUB_ROWSQ) &&
            (rc = make_tmap(&tx, g->aux, g->N, g->M, g->ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B))) return rc;
    }
    auto kern = gemm_tc2_kernel<BN, A_MN, B_MN, MODE, kPath>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
        if (e != cudaSuccess) return fail((int)e, "cudaFuncSetAttribute(gemm_tc2): %s", cudaGetErrorString(e));
        attr_set = true;
    }
    const int tiles_m = (g->M + 2 * BM - 1) / (2 * BM), tiles_n = (g->N + BN - 1) / BN;
    const int units = tiles_m * tiles_n * split_k;
    const int clusters = gemm_clusters();
    const int grid = 2 * (units < clusters ? units : clusters);
    EpiParamsFor<kPath> ep;
    static_cast<EpiParams &>(ep) =
        EpiParams{g->out, g->out2, g->aux, g->bias, g->ldo, make_dropout(g->dropout_p, g->dropout_stream, g->dropout_seed)};
    if constexpr (kPath) ep.path = *path;
    static const int dynamic = [] { const char *e = getenv("ECGVIT_GEMM_DYNAMIC"); return e == nullptr || atoi(e) != 0; }();
    int *sched = next_sched_slot();
    if (sched == nullptr) return fail(-4, "gemm_tc2: cannot resolve the scheduler counters");
    cudaError_t le = launch_pdl(kern, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, stream, ta, tb, to, to2, tx, g->M,
                                g->N, g->K, split_k, ep, sched, dynamic);
    if (le != cudaSuccess) return fail((int)le, "gemm_tc2 launch: %s", cudaGetErrorString(le));
    return check_launch("gemm_tc2");
}

template <int BN> int dispatch_pair(const ecgvit_gemm_args *g, int split_k, cudaStream_t s, const PathParams *path) {
    const bool a_mn = !g->a_kmajor, b_mn = !g->b_kmajor;
    const int mode = g->epilogue;
    if (path != nullptr) {   // drop path: the K-major residual epilogues only (the entry point checked the epilogue)
        if (a_mn || b_mn) return fail(-1, "gemm(bf16): drop path needs K-major operands");
        if (mode == ECGVIT_EPI_BIAS_RES) return launch_pair<BN, false, false, ECGVIT_EPI_BIAS_RES, true>(g, split_k, s, path);
        if (BN < 256 && mode == ECGVIT_EPI_BIAS_RES_F32) {
            constexpr int BNW = BN < 256 ? BN : 192;
            return launch_pair<BNW, false, false, ECGVIT_EPI_BIAS_RES_F32, true>(g, split_k, s, path);
        }
        return fail(-1, "gemm(bf16): drop path needs a residual epilogue (got %d)", mode);
    }
#define ECGVIT_CASE(AM, BMN, MODE) \
    if (a_mn == AM && b_mn == BMN && mode == MODE) return launch_pair<BN, AM, BMN, MODE>(g, split_k, s);
    ECGVIT_CASE(false, false, ECGVIT_EPI_STORE)
    ECGVIT_CASE(false, false, ECGVIT_EPI_BIAS_RES)
    ECGVIT_CASE(false, false, ECGVIT_EPI_BIAS_GELU)
    ECGVIT_CASE(false, false, ECGVIT_EPI_BIAS_SUB_ROWSQ)
    ECGVIT_CASE(false, true, ECGVIT_EPI_STORE)
    ECGVIT_CASE(false, true, ECGVIT_EPI_DGELU)
    ECGVIT_CASE(true, true, ECGVIT_EPI_ATOMIC_F32)
    ECGVIT_CASE(true, true, ECGVIT_EPI_STORE)
    ECGVIT_CASE(true, false, ECGVIT_EPI_STORE)
    if (BN < 256) {   // the fp32 staging tiles of this epilogue leave too few pipeline stages at BN = 256
        constexpr int BNW = BN < 256 ? BN : 192;
        if (!a_mn && !b_mn && mode == ECGVIT_EPI_BIAS_RES_F32)
            return launch_pair<BNW, false, false, ECGVIT_EPI_BIAS_RES_F32>(g, split_k, s);
    }
#undef ECGVIT_CASE
    return fail(-1, "gemm(bf16): unsupported combination a_kmajor=%d b_kmajor=%d epilogue=%d", g->a_kmajor,
                g->b_kmajor, mode);
}

inline double b_kmajor_eff(int b_kmajor) { return b_kmajor ? 0.88 : 0.82; }  // MN-major B over-fetches at 192

}  // namespace

int gemm_bf16_tc(const ecgvit_gemm_args *g, cudaStream_t stream, const PathParams *path) {
    ECGVIT_REQUIRE(g->M > 0 && g->N > 0 && g->K > 0, "gemm: empty problem M=%d N=%d K=%d", g->M, g->N, g->K);
    ECGVIT_REQUIRE(g->N % 8 == 0, "gemm(bf16): N=%d must be a multiple of 8", g->N);
    ECGVIT_REQUIRE(g->lda % 8 == 0 && g->ldb % 8 == 0, "gemm(bf16): lda=%lld ldb=%lld must be multiples of 8",
                   (long long)g->lda, (long long)g->ldb);
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(g->A) & 15) == 0 && (reinterpret_cast<uintptr_t>(g->B) & 15) == 0,
                   "gemm(bf16): operand pointers must be 16-byte aligned");
    ECGVIT_REQUIRE(g->ldo % 8 == 0 && (reinterpret_cast<uintptr_t>(g->out) & 15) == 0,
                   "gemm(bf16): output must be 16-byte aligned with ldo %% 8 == 0");
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(g->bias) & 15) == 0, "gemm(bf16): bias must be 16-byte aligned");
    ECGVIT_REQUIRE(g->epilogue != ECGVIT_EPI_BIAS_RES_F32 || (g->aux != nullptr && g->a_kmajor && g->b_kmajor),
                   "gemm(bf16): the fp32-residual epilogue needs aux and K-major operands");
    ECGVIT_REQUIRE(g->epilogue != ECGVIT_EPI_BIAS_SUB_ROWSQ || (g->aux != nullptr && g->out2 != nullptr),
                   "gemm(bf16): the row-square epilogue needs aux (target) and out2 (row partials)");
    const int sms = sm_count();
    const int kb_total = (g->K + BK - 1) / BK;
    int split_k = g->split_k > 1 ? g->split_k : 1;
    ECGVIT_REQUIRE(split_k == 1 || g->epilogue == ECGVIT_EPI_ATOMIC_F32, "gemm: split_k needs the atomic epilogue");
    if (g->epilogue == ECGVIT_EPI_ATOMIC_F32 && g->split_k <= 0) {
        // auto: smallest split (>= 8 k blocks each) whose work units fill >= 90 % of their last wave
        const int pair = 2;  // work units are 256-row tiles run by CTA pairs
        const int workers = gemm_clusters();
        const long tiles = (long)((g->M + pair * BM - 1) / (pair * BM)) * ((g->N + 255) / 256);
        int best = 1;
        double best_eff = 0.0;
        for (int s = 1; s <= 32 && s * 8 <= kb_total; ++s) {
            const long units = tiles * s;
            const double eff = (double)units / (double)(((units + workers - 1) / workers) * workers);
            if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
            if (eff >= 0.9) { best = s; break; }
        }
        split_k = best;
    }
    if (split_k > kb_total) split_k = kb_total;
    // every split must own at least one k block
    while (split_k > 1 && ((kb_total + split_k - 1) / split_k) * (split_k - 1) >= kb_total) --split_k;

    // Tile width.  Narrow tiles stage more bytes per flop (a 128-wide single-CTA tile needs the full 128 B/clk of
    // shared-memory bandwidth for operand reads alone), so they are only chosen when the wide tile would waste a
    // large part of its last wave.
    // Shared memory moves 128 B/clk per SM and every staged byte is written once (TMA) and read once (MMA), so a
    // 256 x BN pair tile can sustain at most min(1, 128 / (2 * bytes per k block / MMA clocks per k block)) of the
    // tensor peak: 1.00 at BN = 256, 0.88 at 192, 0.67 at 128.  Pick the width with the best (tile efficiency x
    // last-wave occupancy).
    const int clusters = gemm_clusters();
    const long tiles_m2 = (g->M + 2 * BM - 1) / (2 * BM);
    auto score = [&](int bn, double eff) {
        const long units = tiles_m2 * ((g->N + bn - 1) / bn) * split_k;
        const long waves = (units + clusters - 1) / clusters;
        // time ~ waves * bn / eff  (per-tile MMA time is proportional to bn)
        return (double)waves * bn / eff;
    };
    const bool wide_ok = g->epilogue != ECGVIT_EPI_BIAS_RES_F32;   // see dispatch_pair
    static const int forced_bn = [] { const char *e = getenv("ECGVIT_GEMM_BN"); return e != nullptr ? atoi(e) : 0; }();
    if (forced_bn == 128) return dispatch_pair<128>(g, split_k, stream, path);   // experiments only
    if (forced_bn == 192) return dispatch_pair<192>(g, split_k, stream, path);
    if (forced_bn == 256 && wide_ok) return dispatch_pair<256>(g, split_k, stream, path);
    const double s256 = wide_ok ? score(256, 1.0) : 1e30, s192 = score(192, b_kmajor_eff(g->b_kmajor)), s128 = score(128, 0.67);
    if (g->N <= 128 || (s128 < s256 && s128 < s192)) return dispatch_pair<128>(g, split_k, stream, path);
    if (s192 < s256) return dispatch_pair<192>(g, split_k, stream, path);
    return dispatch_pair<256>(g, split_k, stream, path);
}

}  // namespace ecgvit

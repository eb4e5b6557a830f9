// C-ABI plumbing: error string, device query, GEMM front door.
#include "common.cuh"

#include <stdlib.h>

namespace ecgvit {

char *last_error_buffer() {
    static thread_local char buf[512] = {0};
    return buf;
}

int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

bool pdl_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("ECGVIT_PDL");
        v = (e != nullptr && e[0] == '0') ? 0 : 1;
    }
    return v == 1;
}

// path: drop-path factor of the residual epilogues, or nullptr
int gemm_bf16_tc(const ecgvit_gemm_args *g, cudaStream_t stream, const PathParams *path = nullptr);   // gemm_tc.cu
int gemm_f32_ffma(const ecgvit_gemm_args *g, cudaStream_t stream, const PathParams *path = nullptr);  // gemm_simt.cu

}  // namespace ecgvit

extern "C" {

int ecgvit_abi_version(void) { return ECGVIT_ABI_VERSION; }

const char *ecgvit_last_error(void) { return ecgvit::last_error_buffer(); }

int ecgvit_device_ok(void) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
    return major == 10 ? 1 : 0;
}

int ecgvit_gemm(const ecgvit_gemm_args *g, void *stream) {
    if (g == nullptr) return ecgvit::fail(-1, "gemm: null argument block");
    if (g->A == nullptr || g->B == nullptr || g->out == nullptr) return ecgvit::fail(-1, "gemm: null operand");
    if (g->epilogue == ECGVIT_EPI_BIAS_GELU && g->out2 == nullptr) return ecgvit::fail(-1, "gemm: BIAS_GELU needs out2");
    if ((g->epilogue == ECGVIT_EPI_BIAS_RES || g->epilogue == ECGVIT_EPI_DGELU) && g->aux == nullptr)
        return ecgvit::fail(-1, "gemm: epilogue %d needs aux", g->epilogue);
    if (g->epilogue == ECGVIT_EPI_BIAS_RES_F32 && g->dtype != ECGVIT_BF16)
        return ecgvit::fail(-1, "gemm: the fp32-residual epilogue belongs to bf16 mode (fp32 mode uses BIAS_RES)");
    if (g->dtype == ECGVIT_BF16) return ecgvit::gemm_bf16_tc(g, ecgvit::as_stream(stream));
    if (g->dtype == ECGVIT_F32) return ecgvit::gemm_f32_ffma(g, ecgvit::as_stream(stream));
    return ecgvit::fail(-1, "gemm: unknown dtype %d", g->dtype);
}

int ecgvit_gemm_drop_path(const ecgvit_gemm_args *g, float path_p, int path_stream, int rows_per_record, void *stream) {
    if (g == nullptr) return ecgvit::fail(-1, "gemm_drop_path: null argument block");
    ecgvit::PathParams pp;
    if (int rc = ecgvit::make_path("gemm_drop_path", path_p, path_stream, rows_per_record, g->dropout_seed, pp)) return rc;
    if (path_p > 0.f && g->epilogue != ECGVIT_EPI_BIAS_RES && g->epilogue != ECGVIT_EPI_BIAS_RES_F32)
        return ecgvit::fail(-1, "gemm_drop_path: drop path needs epilogue BIAS_RES or BIAS_RES_F32, got %d", g->epilogue);
    if (pp.drop.threshold == 0) return ecgvit_gemm(g, stream);
    if (g->A == nullptr || g->B == nullptr || g->out == nullptr || g->aux == nullptr)
        return ecgvit::fail(-1, "gemm_drop_path: null operand");
    if (g->epilogue == ECGVIT_EPI_BIAS_RES_F32 && g->dtype != ECGVIT_BF16)
        return ecgvit::fail(-1, "gemm: the fp32-residual epilogue belongs to bf16 mode (fp32 mode uses BIAS_RES)");
    if (g->dtype == ECGVIT_BF16) return ecgvit::gemm_bf16_tc(g, ecgvit::as_stream(stream), &pp);
    if (g->dtype == ECGVIT_F32) {
        if (g->epilogue != ECGVIT_EPI_BIAS_RES) return ecgvit::fail(-1, "gemm_drop_path(f32): epilogue must be BIAS_RES");
        return ecgvit::gemm_f32_ffma(g, ecgvit::as_stream(stream), &pp);
    }
    return ecgvit::fail(-1, "gemm: unknown dtype %d", g->dtype);
}

}  // extern "C"

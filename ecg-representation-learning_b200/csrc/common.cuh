// Shared helpers for the ecgvit_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <type_traits>

#include "../../include/ecgvit_b200.h"

namespace ecgvit {

// ---- error plumbing -------------------------------------------------------------------------------
char *last_error_buffer();  // thread-local, 512 bytes (api.cu)

inline int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(last_error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

inline int check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
    return 0;
}

#define ECGVIT_REQUIRE(cond, ...) \
    do { if (!(cond)) return ::ecgvit::fail(-1, __VA_ARGS__); } while (0)

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

int sm_count();  // cached multiprocessor count of the current device (api.cu)

// ---- programmatic dependent launch --------------------------------------------------------------------
// The per-layer kernels are launched with programmaticStreamSerialization: kernel N+1 may be scheduled while kernel
// N drains its last wave, runs its prologue (barrier init, TMEM alloc, tensormap prefetch, smem setup) and then
// blocks in pdl_wait() until kernel N has completed and flushed.  Every such kernel calls pdl_launch_dependents()
// first thing (the dependent launch fires once ALL CTAs of the grid have done so, i.e. when the last wave is
// resident) and pdl_wait() before its first access to global memory.  ECGVIT_PDL=0 disables the attribute.
bool pdl_enabled();  // api.cu
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- element type helpers -------------------------------------------------------------------------
typedef __nv_bfloat16 bf16;

template <typename T> struct Vec8;  // 8 consecutive elements
template <> struct Vec8<float> { float4 a, b; };
template <> struct Vec8<bf16> { uint4 v; };

__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(bf16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float x) { return __float2bfloat16_rn(x); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&h);
}
__device__ __forceinline__ void unpack_bf16x2(uint32_t u, float &lo, float &hi) {
    lo = __uint_as_float(u << 16);
    hi = __uint_as_float(u & 0xffff0000u);
}

// load / store 8 consecutive elements (16-byte aligned for bf16, 32-byte for float) as fp32
__device__ __forceinline__ void load8(const float *p, float v[8]) {
    float4 a = *reinterpret_cast<const float4 *>(p), b = *reinterpret_cast<const float4 *>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const bf16 *p, float v[8]) {
    uint4 u = *reinterpret_cast<const uint4 *>(p);
    unpack_bf16x2(u.x, v[0], v[1]); unpack_bf16x2(u.y, v[2], v[3]);
    unpack_bf16x2(u.z, v[4], v[5]); unpack_bf16x2(u.w, v[6], v[7]);
}
__device__ __forceinline__ void store8(float *p, const float v[8]) {
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(bf16 *p, const float v[8]) {
    uint4 u;
    u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
    u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4 *>(p) = u;
}
// 4-wide variants
__device__ __forceinline__ void load4(const float *p, float v[4]) {
    float4 a = *reinterpret_cast<const float4 *>(p);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
__device__ __forceinline__ void load4(const bf16 *p, float v[4]) {
    uint2 u = *reinterpret_cast<const uint2 *>(p);
    unpack_bf16x2(u.x, v[0], v[1]); unpack_bf16x2(u.y, v[2], v[3]);
}
__device__ __forceinline__ void store4(float *p, const float v[4]) {
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void store4(bf16 *p, const float v[4]) {
    uint2 u;
    u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
    *reinterpret_cast<uint2 *>(p) = u;
}

// ---- reductions -----------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- GELU (exact, erf) ----------------------------------------------------------------------------
// kExact: libdevice erff (parity mode, fp32).  Otherwise Abramowitz-Stegun 7.1.26 (|err| < 1.5e-7,
// far below bf16 resolution): one MUFU.RCP + one MUFU.EX2 + a degree-5 Horner.
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
template <bool kExact> __device__ __forceinline__ void gelu_parts(float u, float &cdf, float &pdf) {
    const float x = u * 0.70710678118654752f;  // u / sqrt(2)
    if (kExact) {
        cdf = 0.5f * (1.0f + erff(x));
        pdf = 0.39894228040143268f * expf(-0.5f * u * u);
    } else {
        // ~17 issue slots per element, 2 of them MUFU (rcp.approx, ex2.approx: both ~1 ulp, far inside the 1.5e-7 of
        // the formula itself): the epilogue has to keep up with a 128 x 256 x 768 mainloop
        const float ax = fabsf(x);
        const float t = rcp_approx(fmaf(0.3275911f, ax, 1.0f));
        const float e = ex2_approx((ax * -1.4426950408889634f) * ax);  // exp(-x^2) = exp(-u^2 / 2)
        float poly = fmaf(1.061405429f, t, -1.453152027f);
        poly = fmaf(poly, t, 1.421413741f);
        poly = fmaf(poly, t, -0.284496736f);
        poly = fmaf(poly, t, 0.254829592f);
        const float half_erf = fmaf(-0.5f * poly * t, e, 0.5f);  // 0.5 * erf(|x|)
        cdf = 0.5f + copysignf(half_erf, x);
        pdf = 0.39894228040143268f * e;
    }
}
// ---- packed fp32x2 math (FFMA2 / FMUL2 / FADD2 on sm_100): two lanes of a Horner step per issue slot -----------
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t splat2(float c) { return pack2(c, c); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// Shared part of the fast erf-GELU for a PAIR of pre-activations (Abramowitz-Stegun 7.1.26 in u directly):
//   half_erf = 0.5 * erf(|u| / sqrt2) = 0.5 - (-0.5 * poly(t) * t) ... with t = 1 / (1 + p |u| / sqrt2), e = exp(-u^2/2)
// ~8.5 issue slots per element (4 of the 17 per pair are MUFU).
__device__ __forceinline__ void gelu_pair_parts(uint64_t u, uint64_t au, uint64_t &half_erf, uint64_t &e) {
    const uint64_t q = fma2(au, splat2(0.3275911f * 0.70710678118654752f), splat2(1.0f));
    float q0, q1;
    unpack2(q, q0, q1);
    const uint64_t t = pack2(rcp_approx(q0), rcp_approx(q1));
    const uint64_t arg = mul2(mul2(u, u), splat2(-0.5f * 1.4426950408889634f));
    float a0, a1;
    unpack2(arg, a0, a1);
    e = pack2(ex2_approx(a0), ex2_approx(a1));
    // coefficients pre-multiplied by -0.5
    uint64_t poly = fma2(t, splat2(-0.5f * 1.061405429f), splat2(0.5f * 1.453152027f));
    poly = fma2(poly, t, splat2(-0.5f * 1.421413741f));
    poly = fma2(poly, t, splat2(0.5f * 0.284496736f));
    poly = fma2(poly, t, splat2(-0.5f * 0.254829592f));
    half_erf = fma2(mul2(poly, t), e, splat2(0.5f));
}
// h = gelu(u) for two values:  u * Phi(u) = 0.5 u + |u| * half_erf
__device__ __forceinline__ void gelu_fwd_pair(float u0, float u1, float &h0, float &h1) {
    const uint64_t u = pack2(u0, u1), au = pack2(fabsf(u0), fabsf(u1));
    uint64_t herf, e;
    gelu_pair_parts(u, au, herf, e);
    unpack2(fma2(au, herf, mul2(u, splat2(0.5f))), h0, h1);
}
// g = gelu'(u) for two values:  Phi(u) + u * phi(u)
__device__ __forceinline__ void gelu_grad_pair(float u0, float u1, float &g0, float &g1) {
    const uint64_t u = pack2(u0, u1), au = pack2(fabsf(u0), fabsf(u1));
    uint64_t herf, e;
    gelu_pair_parts(u, au, herf, e);
    float h0, h1;
    unpack2(herf, h0, h1);
    const uint64_t cdf = add2(pack2(copysignf(h0, u0), copysignf(h1, u1)), splat2(0.5f));
    unpack2(fma2(mul2(u, e), splat2(0.39894228040143268f), cdf), g0, g1);
}

template <bool kExact> __device__ __forceinline__ float gelu_fwd(float u) {
    float cdf, pdf;
    gelu_parts<kExact>(u, cdf, pdf);
    return u * cdf;
}
template <bool kExact> __device__ __forceinline__ float gelu_grad(float u) {
    float cdf, pdf;
    gelu_parts<kExact>(u, cdf, pdf);
    return fmaf(u, pdf, cdf);
}

// ---- dropout ----------------------------------------------------------------------------------------
// Counter-based: the keep decision of element `idx` of dropout site `stream` is a pure function of
// (seed, stream, idx), so backward regenerates the mask instead of reading one from HBM.  One 32-bit hash
// decides an aligned PAIR of elements with 16 bits each: drop if bits < threshold = round(p * 65536).
// nn.Dropout semantics: y = x * keep / (1 - p).  (torch's Philox stream cannot be reproduced bit-for-bit by any other
// implementation; tests inject this mask into the oracle instead.)
struct DropoutParams {
    const uint32_t *seed;  // device scalar, refreshed by the host every step; nullptr / threshold 0 = no dropout
    uint32_t stream;       // which dropout site
    uint32_t threshold;    // round(p * 65536)
    float scale;           // 1 / (1 - threshold / 65536)
};
// two rounds of multiply-and-fold (32 x 32 -> 64 bit product, xor of its halves): 5 issue slots per pair of elements
// (IMAD.WIDE + LOP3 per round), against 9 for a xorshift-multiply hash -- the GELU epilogues are instruction bound
__device__ __forceinline__ uint32_t dropout_hash(uint32_t seed, uint32_t stream, uint32_t pair) {
    const uint32_t key = seed ^ (stream * 0x85EBCA77u + 0xC2B2AE3Du);
    uint64_t m = static_cast<uint64_t>(pair ^ key) * 0x9E3779B1u;
    uint32_t h = static_cast<uint32_t>(m) ^ static_cast<uint32_t>(m >> 32);
    m = static_cast<uint64_t>(h) * 0x7FEB352Du;
    return static_cast<uint32_t>(m) ^ static_cast<uint32_t>(m >> 32);
}
// multipliers (0 or scale) for elements idx (even) and idx + 1.  The 16-bit fields are compared in place
// (high half against threshold << 16, low half after one shift) instead of being extracted first.
__device__ __forceinline__ void dropout_pair(const DropoutParams &d, uint32_t seed, uint32_t idx_even, float &m0,
                                             float &m1) {
    const uint32_t h = dropout_hash(seed, d.stream, idx_even >> 1);
    const uint32_t t = d.threshold << 16;
    m0 = (h << 16) >= t ? d.scale : 0.f;
    m1 = h >= t ? d.scale : 0.f;
}
// multiplier of a single element (any parity)
__device__ __forceinline__ float dropout_one(const DropoutParams &d, uint32_t seed, uint32_t idx) {
    const uint32_t h = dropout_hash(seed, d.stream, idx >> 1);
    const uint32_t bits = (idx & 1u) ? (h >> 16) : (h & 0xffffu);
    return bits >= d.threshold ? d.scale : 0.f;
}
// scale NV (even) consecutive values starting at even element index idx0
template <int NV>
__device__ __forceinline__ void dropout_apply(const DropoutParams &d, uint32_t seed, uint32_t idx0, float v[NV]) {
#pragma unroll
    for (int i = 0; i < NV; i += 2) {
        float m0, m1;
        dropout_pair(d, seed, idx0 + i, m0, m1);
        v[i] *= m0;
        v[i + 1] *= m1;
    }
}

inline DropoutParams make_dropout(float p, int stream, const uint32_t *seed) {
    DropoutParams d{nullptr, 0u, 0u, 1.0f};
    if (seed != nullptr && p > 0.f) {
        uint32_t thr = static_cast<uint32_t>(p * 65536.0f + 0.5f);
        if (thr > 65535u) thr = 65535u;
        if (thr > 0u) d = DropoutParams{seed, static_cast<uint32_t>(stream), thr, 1.0f / (1.0f - thr / 65536.0f)};
    }
    return d;
}

// ---- drop path (stochastic depth) -------------------------------------------------------------------
// One keep decision per RECORD for a residual branch: record b = row / rows_per_record of a [B * N, d] token matrix
// draws dropout_one(drop, seed, b) (0 or 1 / (1 - r)) from the counter hash above, so forward, backward and an
// activation-checkpointing recompute all see the same factor without a stored mask.  Kernels instantiated with a
// PathParams always have drop.threshold > 0 (the entry points run the plain kernels otherwise).
struct PathParams {
    DropoutParams drop;
    int rows_per_record;
};
__device__ __forceinline__ float path_factor(const PathParams &pp, int64_t row) {
    return dropout_one(pp.drop, __ldg(pp.drop.seed), static_cast<uint32_t>(row / pp.rows_per_record));
}
// element dropout and drop path of one branch together (the drop-path variants of the backward masked copies)
struct DropoutPathParams : DropoutParams {
    PathParams path;
};
template <bool kPath> using DropParamsFor = typename std::conditional<kPath, DropoutPathParams, DropoutParams>::type;
// host: checks the drop-path arguments of a *_drop_path entry point.  The rate is quantised like dropout's
// (round(p * 65536)); pp.drop.threshold == 0 means the call is the plain entry point's.  The seed is the dropout seed.
inline int make_path(const char *what, float p, int stream, int rows_per_record, const uint32_t *seed, PathParams &pp) {
    if (!(p >= 0.f && p < 1.f)) return fail(-1, "%s: drop-path rate %g outside [0, 1)", what, (double)p);
    if (rows_per_record <= 0) return fail(-1, "%s: rows_per_record=%d must be positive", what, rows_per_record);
    if (p > 0.f && seed == nullptr) return fail(-1, "%s: drop path needs a dropout seed", what);
    pp = PathParams{make_dropout(p, stream, seed), rows_per_record};
    return 0;
}

// ---- GEMM epilogue parameters shared by the tcgen05 and FFMA kernels -----------------------------
struct EpiParams {
    void *out;
    void *out2;
    const void *aux;
    const float *bias;
    int64_t ldo;
    DropoutParams drop;  // BIAS_RES: on (acc + bias); BIAS_GELU: on gelu(out); DGELU: on acc
};
// BIAS_RES / BIAS_RES_F32 with drop path: out = s[row / rows_per_record] * drop(acc + bias) + aux
struct EpiPathParams : EpiParams {
    PathParams path;
};

// Applies epilogue MODE to NV (4 or 8) consecutive accumulator columns of one row and stores them.
// `col` is a multiple of NV and the caller guarantees row/col are in bounds.
// EP = EpiPathParams (BIAS_RES only) scales the dropped branch by the row's drop-path factor before the residual add.
template <int MODE, typename T, int NV, bool kExactGelu, typename EP>
__device__ __forceinline__ void epilogue_store(const EP &p, int64_t row, int col, float acc[NV]) {
    const int64_t off = row * p.ldo + col;
    if (MODE == ECGVIT_EPI_ATOMIC_F32) {
        float *o = reinterpret_cast<float *>(p.out) + off;
#pragma unroll
        for (int i = 0; i < NV; i += 4)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + i), "f"(acc[i]),
                         "f"(acc[i + 1]), "f"(acc[i + 2]), "f"(acc[i + 3])
                         : "memory");
        return;
    }
    if (MODE != ECGVIT_EPI_DGELU && p.bias != nullptr) {
#pragma unroll
        for (int i = 0; i < NV; i += 4) {
            const float4 b = __ldg(reinterpret_cast<const float4 *>(p.bias + col + i));
            acc[i] += b.x; acc[i + 1] += b.y; acc[i + 2] += b.z; acc[i + 3] += b.w;
        }
    }
    T *o = reinterpret_cast<T *>(p.out) + off;
    const bool drop = p.drop.threshold != 0;
    const uint32_t seed = drop ? __ldg(p.drop.seed) : 0u;
    if (drop && (MODE == ECGVIT_EPI_BIAS_RES || MODE == ECGVIT_EPI_DGELU))
        dropout_apply<NV>(p.drop, seed, static_cast<uint32_t>(off), acc);
    if constexpr (std::is_same<EP, EpiPathParams>::value) {
        static_assert(MODE == ECGVIT_EPI_BIAS_RES, "drop path belongs to the residual epilogue");
        const float s = path_factor(p.path, row);
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] *= s;
    }
    if (MODE == ECGVIT_EPI_BIAS_RES) {
        float r[NV];
        if (NV == 8) load8(reinterpret_cast<const T *>(p.aux) + off, r);
        else load4(reinterpret_cast<const T *>(p.aux) + off, r);
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] += r[i];
    } else if (MODE == ECGVIT_EPI_BIAS_SUB_ROWSQ) {   // acc keeps the fp32 residual for the caller's row sum
        float t[NV];
        if (NV == 8) load8(reinterpret_cast<const T *>(p.aux) + off, t);
        else load4(reinterpret_cast<const T *>(p.aux) + off, t);
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] -= t[i];
    } else if (MODE == ECGVIT_EPI_DGELU) {
        float u[NV];
        if (NV == 8) load8(reinterpret_cast<const T *>(p.aux) + off, u);
        else load4(reinterpret_cast<const T *>(p.aux) + off, u);
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] *= gelu_grad<kExactGelu>(u[i]);
    } else if (MODE == ECGVIT_EPI_BIAS_GELU) {
        float h[NV];
        // the saved pre-activation is what backward differentiates, so round it first (bf16 mode)
#pragma unroll
        for (int i = 0; i < NV; ++i) h[i] = gelu_fwd<kExactGelu>(to_f32(from_f32<T>(acc[i])));
        if (drop) dropout_apply<NV>(p.drop, seed, static_cast<uint32_t>(off), h);
        T *o2 = reinterpret_cast<T *>(p.out2) + off;
        if (NV == 8) store8(o2, h); else store4(o2, h);
    }
    if (NV == 8) store8(o, acc); else store4(o, acc);
}

}  // namespace ecgvit

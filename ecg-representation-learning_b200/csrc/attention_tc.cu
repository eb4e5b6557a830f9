// Softmax attention on the 5th-generation tensor cores (tcgen05 / TMEM / TMA) for head dim 64, bf16.
//
// Replaces chunk(3) + rearrange + q k^T * scale + Softmax + Dropout + attn v + rearrange back of vit_pytorch's
// Attention.forward (reached from /root/reference/ecg_transformer/models/ecg_vit.py:102-116,141) and its autograd
// backward (models/train.py:280).  Operates in place on the packed projection qkv [B*N, 3*H*64] (q | k | v, head-major)
// through 3-D TMA boxes of the [B][N][3*H*64] view, so sequences are zero-padded by the TMA unit, never in memory.
//
// Two geometries share every kernel:
//   packed (N <= 64; BASELINE.json configs[1]: N = 51): one 128-row tile holds TWO (batch, head) problems (64 padded
//     rows each); S = Q K^T is a 128 x 128 product whose diagonal 64 x 64 blocks are the two problems, P is kept
//     block-diagonal (zeros elsewhere) so one 128 x 64 x 128 product gives both outputs.  One key block per tile: these
//     kernels live on the TMA ring that keeps loads of the next tiles in flight (the shape is HBM-bound).
//   long (N > 64; configs[3]: N = 2401 per-lead tokens): a tile is 128 queries of one (batch, head), key blocks of 128 are
//     streamed with a running (max, sum); nothing of size N x N is ever written.
//
// Forward (attn_tc_fwd_kernel), one persistent CTA per SM, 12 warps:
//   warp 0   TMA producer: Q tiles (2-deep ring per tile slot) and K/V blocks (4-deep ring)
//   warp 1   MMA issuer : S_t = Q_t K^T (SS, 128x128x64) and O_t += P_t V (TS: P from TMEM, V MN-major from smem)
//   warp 2   TMEM allocator (512 columns: S0 S1 | O0 O1 | P0 P1)
//   warps 4-7 / 8-11  softmax warpgroup of tile 0 / tile 1 (thread = query row): S -> registers, running max / sum,
//            exp2, dropout, P (bf16, packed two per column) -> TMEM, lazy rescale of O, final O / l -> smem -> TMA store
// The two tiles of a CTA ping-pong: the tensor core runs tile 1's products while tile 0's warpgroup is in its softmax.
// In the long geometry both tiles are consecutive query tiles of the same head and share every K/V block.
#include "common.cuh"
#include "ptx.cuh"

#include <cudaTypedefs.h>

namespace ecgvit {

namespace {

constexpr int DH = 64;               // head dim served by these kernels
constexpr int TM = 128;              // query rows per tile = TMEM lanes
constexpr int TN = 128;              // keys per block
constexpr int TILE_BYTES = TM * DH * 2;  // 16 KB: one [128 x 64] bf16 tile, 128-byte rows, SWIZZLE_128B
constexpr float LOG2E_F = 1.4426950408889634f;

// ---- forward shared-memory map (offsets from a 1024-byte aligned base) -----------------------------------------------
constexpr int F_Q_OFF = 0;                               // [tile 2][slot 2] Q tiles
constexpr int F_KV_OFF = F_Q_OFF + 4 * TILE_BYTES;       // [stage 4] K tile | V tile
constexpr int F_KV_STAGES = 4;
constexpr int F_OST_OFF = F_KV_OFF + F_KV_STAGES * 2 * TILE_BYTES;  // [tile 2] output staging
constexpr int F_BAR_OFF = F_OST_OFF + 2 * TILE_BYTES;
constexpr int F_SMEM_BYTES = F_BAR_OFF + 256 + 1024;     // + barrier block + alignment slack
// TMEM columns
constexpr uint32_t F_TM_S = 0, F_TM_O = 256, F_TM_P = 384;  // S_t at S + 128 t, O_t at O + 64 t, P_t at P + 64 t

struct FwdBars {
    uint64_t q_full[2][2], q_empty[2][2];
    uint64_t kv_full[F_KV_STAGES], kv_empty[F_KV_STAGES];
    uint64_t s_full[2], s_free[2], p_full[2], pv_done[2], out_full[2], out_free[2];
    uint32_t tmem_ptr;
};
static_assert(sizeof(FwdBars) <= 256, "barrier block");

// work decomposition shared by all roles (everything here is CTA-uniform)
template <bool kPacked> struct FwdItem {
    bool valid[2];
    int prob[2][2];  // packed: the two (b*H + h) problems of tile t; long: prob[t][0] = b*H + h
    int q0[2];       // long: first query row of tile t
};
// kk = how many items this CTA has already taken.  Packed tiles are dealt out one by one (tile = bid + (2 kk + t) * nblk),
// so the last round leaves at most one tile per CTA idle; long items (a pair of query tiles) are dealt bid + kk * nblk.
// valid[0] == false means the CTA has run out of work.
template <bool kPacked>
__device__ __forceinline__ void fwd_decode(int kk, int B, int N, int H, FwdItem<kPacked> &it) {
    const int bid = blockIdx.x, nblk = gridDim.x;
    if (kPacked) {
        const int n_prob = B * H, n_pt = (n_prob + 1) >> 1;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const int pt = bid + (2 * kk + t) * nblk;
            it.valid[t] = pt < n_pt;
            it.prob[t][0] = 2 * pt;
            it.prob[t][1] = 2 * pt + 1;  // may equal n_prob: its loads are fully out of bounds (zeros), its stores clipped
            it.q0[t] = 0;
        }
    } else {
        const int nqt = (N + TM - 1) / TM, pairs = (nqt + 1) >> 1;
        const int item = bid + kk * nblk;
        const int bh = item / pairs, qp = item - bh * pairs;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            // an odd number of query tiles: the last pair runs its tile twice (identical stores) rather than leaving
            // slot 1 dry in the middle of the CTA's sequence
            it.valid[t] = item < B * H * pairs;
            it.prob[t][0] = it.prob[t][1] = bh;
            it.q0[t] = min(2 * qp + t, nqt - 1) * TM;
        }
    }
}

__device__ __forceinline__ float pair_sum2(uint64_t v) {
    float a, b;
    unpack2(v, a, b);
    return a + b;
}

// ---- softmax building blocks (thread = one row; 32-column chunks of S) --------------------------------------------
// running maximum over one chunk, four independent chains; kMasked: columns >= lim do not exist
template <bool kMasked> __device__ __forceinline__ void chunk_max(const uint32_t s[32], int lim, float mx[4]) {
#pragma unroll
    for (int i = 0; i < 32; i += 4)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float v = __uint_as_float(s[i + k]);
            if (kMasked && i + k >= lim) v = -INFINITY;
            mx[k] = fmaxf(mx[k], v);
        }
}
// p = exp2(s * sl2 + nm) (0 for masked columns), added to two packed partial sums, dropped, packed to bf16 pairs
template <bool kMasked>
__device__ __forceinline__ void chunk_exp(const uint32_t s[32], int lim, float sl2, float nm, uint64_t sum2[2],
                                          const DropoutParams &drop, uint32_t seed, uint32_t e0, uint32_t pk[16]) {
    float p[32];
    const uint64_t sl2_2 = splat2(sl2), nm_2 = splat2(nm);
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
        float x0, x1;
        unpack2(fma2(pack2(__uint_as_float(s[i]), __uint_as_float(s[i + 1])), sl2_2, nm_2), x0, x1);
        p[i] = ex2_approx(x0);
        p[i + 1] = ex2_approx(x1);
        if (kMasked) {
            if (i >= lim) p[i] = 0.f;
            if (i + 1 >= lim) p[i + 1] = 0.f;
        }
        sum2[(i >> 1) & 1] = add2(sum2[(i >> 1) & 1], pack2(p[i], p[i + 1]));
    }
    if (drop.threshold != 0) {
        // keep / drop only: the 1 / (1 - p) factor of the kept probabilities is applied once, to the finished row of O
        const uint32_t thr = drop.threshold << 16;
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            const uint32_t h = dropout_hash(seed, drop.stream, (e0 + i) >> 1);
            p[i] = (h << 16) >= thr ? p[i] : 0.f;
            p[i + 1] = h >= thr ? p[i + 1] : 0.f;
        }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) pk[i] = pack_bf16x2(p[2 * i], p[2 * i + 1]);
}

// byte offset of 16-byte chunk j (0..7) of row r inside a [rows x 128 B] SWIZZLE_128B tile (1024-byte aligned base)
__device__ __forceinline__ uint32_t sw128_offset(int r, int j) {
    return static_cast<uint32_t>(r) * 128u + (static_cast<uint32_t>(j ^ (r & 7)) << 4);
}

template <bool kPacked>
__global__ void __launch_bounds__(384, 1)
attn_tc_fwd_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_o,
                   float *__restrict__ lse, int B, int N, int H, float scale, DropoutParams drop) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    FwdBars *bars = reinterpret_cast<FwdBars *>(smem + F_BAR_OFF);

    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int inner = H * DH;
    const int nkb = kPacked ? 1 : (N + TN - 1) / TN;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_qkv);
        ptx::prefetch_tensormap(&tm_o);
    }
    if (warp == 1 && lane == 0) {
        for (int t = 0; t < 2; ++t) {
            for (int s = 0; s < 2; ++s) {
                ptx::mbar_init(&bars->q_full[t][s], 1);
                ptx::mbar_init(&bars->q_empty[t][s], 1);
            }
            ptx::mbar_init(&bars->s_full[t], 1);
            ptx::mbar_init(&bars->s_free[t], 4);   // one arrival per warp of the tile's softmax warpgroup
            ptx::mbar_init(&bars->p_full[t], 4);
            ptx::mbar_init(&bars->pv_done[t], 1);
            ptx::mbar_init(&bars->out_full[t], 4);
            ptx::mbar_init(&bars->out_free[t], 1);
        }
        for (int s = 0; s < F_KV_STAGES; ++s) {
            ptx::mbar_init(&bars->kv_full[s], 1);
            ptx::mbar_init(&bars->kv_empty[s], 1);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc(&bars->tmem_ptr, 512);
    ptx::tcgen05_fence_before();
    __syncthreads();
    ptx::tcgen05_fence_after();
    const uint32_t tmem_base = bars->tmem_ptr;
    pdl_wait();

    // registers: the eight softmax warps hold a whole row of scores each; the four service warps need few
    if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 0) {
        // ================================ TMA producer ==================================================
        int qcnt[2] = {0, 0}, kvcnt = 0;
        for (int kk = 0;; ++kk) {
            FwdItem<kPacked> it;
            fwd_decode<kPacked>(kk, B, N, H, it);
            if (!it.valid[0]) break;
            auto load_q = [&](int t) {
                const int slot = qcnt[t] & 1;
                ptx::mbar_wait(&bars->q_empty[t][slot], ((qcnt[t] >> 1) & 1) ^ 1);
                if (ptx::elect_one()) {
                    uint8_t *dst = smem + F_Q_OFF + (t * 2 + slot) * TILE_BYTES;
                    ptx::mbar_arrive_expect_tx(&bars->q_full[t][slot], TILE_BYTES);
                    if (kPacked) {
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
                            const int p = it.prob[t][i];
                            ptx::tma_load_3d(dst + i * (TILE_BYTES / 2), &tm_qkv, &bars->q_full[t][slot], (p % H) * DH, 0,
                                             p / H);
                        }
                    } else {
                        const int p = it.prob[t][0];
                        ptx::tma_load_3d(dst, &tm_qkv, &bars->q_full[t][slot], (p % H) * DH, it.q0[t], p / H);
                    }
                }
                __syncwarp();
                ++qcnt[t];
            };
            // K block (rows k0.. of problem(s) `prob`) and the matching V block into the next ring stage
            auto load_kv = [&](const int prob[2], int k0) {
                const int st = kvcnt % F_KV_STAGES;
                ptx::mbar_wait(&bars->kv_empty[st], ((kvcnt / F_KV_STAGES) & 1) ^ 1);
                if (ptx::elect_one()) {
                    uint8_t *dst = smem + F_KV_OFF + st * 2 * TILE_BYTES;
                    ptx::mbar_arrive_expect_tx(&bars->kv_full[st], 2 * TILE_BYTES);
                    if (kPacked) {
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
                            const int p = prob[i], c = (p % H) * DH, b = p / H;
                            ptx::tma_load_3d(dst + i * (TILE_BYTES / 2), &tm_qkv, &bars->kv_full[st], inner + c, 0, b);
                            ptx::tma_load_3d(dst + TILE_BYTES + i * (TILE_BYTES / 2), &tm_qkv, &bars->kv_full[st],
                                             2 * inner + c, 0, b);
                        }
                    } else {
                        const int p = prob[0], c = (p % H) * DH, b = p / H;
                        ptx::tma_load_3d(dst, &tm_qkv, &bars->kv_full[st], inner + c, k0, b);
                        ptx::tma_load_3d(dst + TILE_BYTES, &tm_qkv, &bars->kv_full[st], 2 * inner + c, k0, b);
                    }
                }
                __syncwarp();
                ++kvcnt;
            };
            if (kPacked) {
#pragma unroll
                for (int t = 0; t < 2; ++t)
                    if (it.valid[t]) {
                        load_q(t);
                        load_kv(it.prob[t], 0);
                    }
            } else {
#pragma unroll
                for (int t = 0; t < 2; ++t)
                    if (it.valid[t]) load_q(t);
                for (int j = 0; j < nkb; ++j) load_kv(it.prob[0], j * TN);
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ====================================================
        // Per tile the products form a chain of steps (item, key block).  At every step the issuer first launches the
        // NEXT step's S = Q K^T (it only needs the S buffer back, which the softmax warpgroup hands over as soon as it has
        // S in registers) and then, once P has been written, this step's O += P V: the tensor core works on the next
        // scores while the warpgroup is still exponentiating the current ones.
        constexpr uint32_t idesc_qk = ptx::make_idesc_bf16(TM, TN, 0, 0);
        constexpr uint32_t idesc_pv = ptx::make_idesc_bf16(TM, DH, 0, 1);
        const uint32_t smem_base = ptx::smem_u32(smem);
        int qcnt[2] = {0, 0}, kvcnt = 0;      // Q tiles / K-V stages consumed so far
        uint32_t pph[2] = {0, 0}, fph[2] = {0, 0};
        int slot_cur[2] = {0, 0}, st_cur[2] = {0, 0}, st_next[2] = {0, 0};
        // S_t = Q_t K^T with K from ring stage `st`
        auto issue_qk = [&](int t, int slot, int st, bool last_of_item) {
            ptx::tcgen05_fence_after();
            if (ptx::elect_one()) {
                const uint64_t da = ptx::make_smem_desc(smem_base + F_Q_OFF + (t * 2 + slot) * TILE_BYTES, 16, 1024);
                const uint64_t db = ptx::make_smem_desc(smem_base + F_KV_OFF + st * 2 * TILE_BYTES, 16, 1024);
#pragma unroll
                for (int k = 0; k < DH / 16; ++k)
                    ptx::umma_bf16(tmem_base + F_TM_S + t * TN, da + 2 * k, db + 2 * k, idesc_qk, k > 0 ? 1u : 0u);
                ptx::umma_commit(&bars->s_full[t]);
                if (last_of_item) ptx::umma_commit(&bars->q_empty[t][slot]);  // Q_t is not read again
            }
            __syncwarp();
        };
        // O_t (+)= P_t V with V from ring stage `st` (MN-major: one key per 128-byte row, 16 keys = 2048 B per UMMA_K)
        auto issue_pv = [&](int t, int st, bool acc, bool release_kv) {
            ptx::tcgen05_fence_after();
            if (ptx::elect_one()) {
                const uint64_t db = ptx::make_smem_desc(smem_base + F_KV_OFF + st * 2 * TILE_BYTES + TILE_BYTES, 8192, 1024);
#pragma unroll
                for (int k = 0; k < TN / 16; ++k)
                    ptx::umma_bf16_ts(tmem_base + F_TM_O + t * DH, tmem_base + F_TM_P + t * (TN / 2) + 8 * k,
                                      db + 128 * k, idesc_pv, (acc || k > 0) ? 1u : 0u);
                ptx::umma_commit(&bars->pv_done[t]);
                if (release_kv) ptx::umma_commit(&bars->kv_empty[st]);
            }
            __syncwarp();
        };
        // next K/V ring stage (waits for its bytes)
        auto take_kv = [&]() {
            const int st = kvcnt % F_KV_STAGES;
            ptx::mbar_wait(&bars->kv_full[st], (kvcnt / F_KV_STAGES) & 1);
            ++kvcnt;
            return st;
        };
        // first product of an item for tile t (long: `st_shared` is the stage of key block 0, shared by both tiles)
        auto first_qk = [&](int t, int st_shared) {
            const int slot = qcnt[t] & 1;
            ptx::mbar_wait(&bars->q_full[t][slot], (qcnt[t] >> 1) & 1);
            ++qcnt[t];
            const int st = kPacked ? take_kv() : st_shared;
            issue_qk(t, slot, st, nkb == 1);
            slot_cur[t] = slot;
            return st;
        };
        FwdItem<kPacked> it;
        fwd_decode<kPacked>(0, B, N, H, it);
        if (it.valid[0]) {
            const int st0 = kPacked ? 0 : take_kv();
#pragma unroll
            for (int t = 0; t < 2; ++t)
                if (it.valid[t]) st_cur[t] = first_qk(t, st0);
        }
        for (int kk = 0; it.valid[0]; ++kk) {
            FwdItem<kPacked> nxt;
            fwd_decode<kPacked>(kk + 1, B, N, H, nxt);
            for (int j = 0; j < nkb; ++j) {
                int st_shared = 0;
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    if (!it.valid[t]) continue;
                    // ---- the successor step's scores
                    const bool more_blocks = j + 1 < nkb;
                    if (more_blocks || nxt.valid[t]) {
                        ptx::mbar_wait(&bars->s_free[t], fph[t]);   // S_t is in the warpgroup's registers
                        fph[t] ^= 1;
                        if (more_blocks) {
                            if (t == 0) st_shared = take_kv();      // tile 0 exists whenever tile 1 does
                            issue_qk(t, slot_cur[t], st_shared, j + 2 == nkb);
                            st_next[t] = st_shared;
                        } else {
                            if (!kPacked && t == 0) st_shared = take_kv();
                            st_next[t] = first_qk(t, st_shared);
                        }
                    }
                    // ---- this step's output product
                    ptx::mbar_wait(&bars->p_full[t], pph[t]);
                    pph[t] ^= 1;
                    issue_pv(t, st_cur[t], j > 0, kPacked || !it.valid[1] || t == 1);
                    st_cur[t] = st_next[t];
                }
            }
            it = nxt;
        }
    } else if (warp == 3) {
        // ================================ result warp: TMA stores of the finished O tiles ==============
        uint32_t oph[2] = {0, 0};
        for (int kk = 0;; ++kk) {
            FwdItem<kPacked> it;
            fwd_decode<kPacked>(kk, B, N, H, it);
            if (!it.valid[0]) break;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                if (!it.valid[t]) continue;
                ptx::mbar_wait(&bars->out_full[t], oph[t]);
                oph[t] ^= 1;
                if (ptx::elect_one()) {
                    const uint8_t *ost = smem + F_OST_OFF + t * TILE_BYTES;
                    if (kPacked) {
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
                            const int p = it.prob[t][i];
                            ptx::tma_store_3d(&tm_o, ost + i * (TILE_BYTES / 2), (p % H) * DH, 0, p / H);
                        }
                    } else {
                        const int p = it.prob[t][0];
                        ptx::tma_store_3d(&tm_o, ost, (p % H) * DH, it.q0[t], p / H);
                    }
                    ptx::tma_store_commit();
                    ptx::tma_store_wait_read<0>();
                    ptx::mbar_arrive(&bars->out_free[t]);
                }
                __syncwarp();
            }
        }
        if (ptx::elect_one()) ptx::tma_store_wait_all<0>();
        __syncwarp();
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
        // ================================ softmax warpgroups (tile = (warp - 4) / 4) ==================
        const int t = (warp - 4) >> 2;
        const int q = warp & 3;                 // TMEM lane quadrant of this warp
        const int r = q * 32 + lane;            // row of the tile owned by this thread
        const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
        const uint32_t tS = lane_addr + F_TM_S + t * TN, tO = lane_addr + F_TM_O + t * DH,
                       tP = lane_addr + F_TM_P + t * (TN / 2);
        const float sl2 = scale * LOG2E_F;
        const uint32_t seed = drop.threshold != 0 ? __ldg(drop.seed) : 0u;
        const int Np = (N + 63) / 64 * 64;      // row pitch of the dropout counter (shared with the other kernels)
        // packed: this thread's problem is half `hf` of the tile; it reads S columns [64 hf, 64 hf + 64)
        const int hf = kPacked ? (r >> 6) : 0;
        const int col0 = kPacked ? 64 * hf : 0;
        constexpr int NCH = kPacked ? 2 : 4;    // 32-column chunks of S read per key block
        uint8_t *ost = smem + F_OST_OFF + t * TILE_BYTES;
        if (kPacked) {
            // the off-diagonal half of P never changes: zero it once (TMEM is not cleared by allocation)
            uint32_t z[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] = 0u;
            ptx::tmem_st_32x16(tP + (hf ? 0 : 32), z);
            ptx::tmem_st_32x16(tP + (hf ? 0 : 32) + 16, z);
            ptx::tmem_st_wait();
        }
        uint32_t sph = 0, dph = 0, oph = 0;
        for (int kk = 0;; ++kk) {
            FwdItem<kPacked> it;
            fwd_decode<kPacked>(kk, B, N, H, it);
            if (!it.valid[t]) break;   // once a tile slot runs dry it stays dry (and slot 0 outlives slot 1)
            const int prob = it.prob[t][hf];
            const int qrow = kPacked ? (r & 63) : it.q0[t] + r;    // query index inside the problem
            float m = -INFINITY, l = 0.f;
            for (int j = 0; j < nkb; ++j) {
                const int nvalid = kPacked ? N : min(TN, N - j * TN);  // valid keys of this block (>= 1)
                const bool partial = nvalid < NCH * 32;                // CTA-uniform
                ptx::mbar_wait(&bars->s_full[t], sph);
                sph ^= 1;
                ptx::tcgen05_fence_after();
                // ---- the whole row of scores into registers, then hand S_t back to the tensor core
                uint32_t s[NCH][32];
#pragma unroll
                for (int c = 0; c < NCH; ++c) ptx::tmem_ld_32x32(tS + col0 + 32 * c, s[c]);
#pragma unroll
                for (int c = 0; c < NCH; ++c) ptx::tmem_ld_wait_bind32(s[c]);
                ptx::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&bars->s_free[t]);
                // ---- running max
                float mx4[4] = {m, m, m, m};
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    if (partial) chunk_max<true>(s[c], nvalid - 32 * c, mx4);
                    else chunk_max<false>(s[c], 32, mx4);
                }
                const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
                const float alpha = ex2_approx((m - mx) * sl2);   // 0 on the first block (m = -inf)
                m = mx;
                const float nm = -m * sl2;
                // ---- p = exp2(s * sl2 - m * sl2), row sum, dropout, bf16 pack (in registers)
                uint64_t sum2[2] = {0ull, 0ull};
                const uint32_t e_row = (static_cast<uint32_t>(prob) * Np + static_cast<uint32_t>(qrow)) * Np +
                                       static_cast<uint32_t>(j * TN);
                uint32_t pk[NCH][16];
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    if (partial) chunk_exp<true>(s[c], nvalid - 32 * c, sl2, nm, sum2, drop, seed, e_row + 32 * c, pk[c]);
                    else chunk_exp<false>(s[c], 32, sl2, nm, sum2, drop, seed, e_row + 32 * c, pk[c]);
                }
                l = l * alpha + (pair_sum2(sum2[0]) + pair_sum2(sum2[1]));
                if (j > 0) {
                    // P_t and O_t are free once the previous block's P V product has retired
                    ptx::mbar_wait(&bars->pv_done[t], dph);
                    dph ^= 1;
                    ptx::tcgen05_fence_after();
                    if (__any_sync(0xffffffffu, alpha != 1.0f)) {   // lazy: the running max rarely moves after a few blocks
#pragma unroll 1
                        for (int c = 0; c < DH / 32; ++c) {
                            uint32_t o[32];
                            ptx::tmem_ld_32x32(tO + 32 * c, o);
                            ptx::tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                            ptx::tmem_st_32x32(tO + 32 * c, o);
                        }
                    }
                }
#pragma unroll
                for (int c = 0; c < NCH; ++c) ptx::tmem_st_32x16(tP + (col0 >> 1) + 16 * c, pk[c]);
                ptx::tmem_st_wait();
                ptx::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&bars->p_full[t]);
            }
            // ---- epilogue: O / l -> bf16 -> swizzled staging tile -> TMA store; log-sum-exp of the scaled scores
            ptx::mbar_wait(&bars->pv_done[t], dph);
            dph ^= 1;
            ptx::tcgen05_fence_after();
            ptx::mbar_wait(&bars->out_free[t], oph ^ 1);   // warp 3's previous store of this tile has read `ost`
            oph ^= 1;
            const float inv_l = drop.scale / l;   // drop.scale = 1 / (1 - p) of the attention dropout (1 when off)
#pragma unroll 1
            for (int c = 0; c < DH / 32; ++c) {
                uint32_t o[32];
                ptx::tmem_ld_32x32(tO + 32 * c, o);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    uint4 v;
                    v.x = pack_bf16x2(__uint_as_float(o[8 * jj + 0]) * inv_l, __uint_as_float(o[8 * jj + 1]) * inv_l);
                    v.y = pack_bf16x2(__uint_as_float(o[8 * jj + 2]) * inv_l, __uint_as_float(o[8 * jj + 3]) * inv_l);
                    v.z = pack_bf16x2(__uint_as_float(o[8 * jj + 4]) * inv_l, __uint_as_float(o[8 * jj + 5]) * inv_l);
                    v.w = pack_bf16x2(__uint_as_float(o[8 * jj + 6]) * inv_l, __uint_as_float(o[8 * jj + 7]) * inv_l);
                    *reinterpret_cast<uint4 *>(ost + sw128_offset(r, 4 * c + jj)) = v;
                }
            }
            ptx::tcgen05_fence_before();   // O_t has been read: the next item's first P V may overwrite it
            if (qrow < N && prob < B * H) lse[static_cast<int64_t>(prob) * N + qrow] = m * scale + __logf(l);
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&bars->out_full[t]);   // warp 3 issues the TMA store
        }
    }

    ptx::tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tcgen05_fence_after();
        ptx::tmem_dealloc(tmem_base, 512);
    }
}

// ---- host side ----------------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
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

// bf16 [B][N][cols] view (row pitch `ld` elements, batch pitch N * ld) with a {64 features, box_rows tokens, 1} box
int make_tmap3(CUtensorMap *tm, const void *base, int cols, int N, int B, int64_t ld, int box_rows, bool fp32 = false) {
    PFN_cuTensorMapEncodeTiled_v12000 enc = encode_fn();
    if (enc == nullptr) return fail(-2, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)N, (cuuint64_t)B};
    const cuuint64_t esz = fp32 ? 4 : 2;   // either way a box row is 128 bytes (64 bf16 / 32 fp32)
    cuuint64_t strides[2] = {(cuuint64_t)ld * esz, (cuuint64_t)N * (cuuint64_t)ld * esz};
    cuuint32_t box[3] = {fp32 ? 32u : 64u, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(tm, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(-3, "cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)r);
    return 0;
}

template <bool kPacked>
int launch_fwd(const void *qkv, void *o, float *lse, int B, int N, int H, float scale, DropoutParams drop,
               cudaStream_t stream) {
    const int inner = H * DH;
    CUtensorMap tq, to;
    int rc;
    if ((rc = make_tmap3(&tq, qkv, 3 * inner, N, B, 3 * (int64_t)inner, kPacked ? 64 : TM))) return rc;
    if ((rc = make_tmap3(&to, o, inner, N, B, inner, kPacked ? 64 : TM))) return rc;
    auto kern = attn_tc_fwd_kernel<kPacked>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, F_SMEM_BYTES);
        if (e != cudaSuccess) return fail((int)e, "cudaFuncSetAttribute(attn_tc_fwd): %s", cudaGetErrorString(e));
        attr_set = true;
    }
    int items;  // packed: tiles (two problems each); long: pairs of query tiles
    if (kPacked) items = (B * H + 1) >> 1;
    else items = B * H * ((((N + TM - 1) / TM) + 1) >> 1);
    const int grid = items < sm_count() ? items : sm_count();
    cudaError_t le = launch_pdl(kern, dim3(grid), dim3(384), F_SMEM_BYTES, stream, tq, to, lse, B, N, H, scale, drop);
    if (le != cudaSuccess) return fail((int)le, "attn_tc_fwd launch: %s", cudaGetErrorString(le));
    return check_launch("attn_tc_fwd");
}


// =====================================================================================================================
// Backward.  One kernel serves both geometries:
//   packed: an item is one 128-row tile (two problems), one step per item;
//   long:   an item is one 128-key block of one (batch, head) whose K / V stay in shared memory while the query blocks
//           stream past (one step each); dK / dV accumulate in TMEM over the steps, dQ of every step is added to an fp32
//           accumulator in HBM by TMA reduce-add (converted to bf16 afterwards).
// Per step, with S / dP / dV / dK / dQ in TMEM (448 columns):
//   MMA   S = Q K^T, dP = dO V^T                                   (SS, 128 x 128 x 64 each)
//   warps P = exp2(S sl2 - lse), Pd = P mask, dS = P (dP mask - D) scale  -> bf16 tiles Pd_s, dS_s in shared memory,
//         laid out [query][key] in 128-byte rows: K-major A operand for dS K and MN-major A operand for Pd^T dO, dS^T Q
//   MMA   dV += Pd^T dO, dK += dS^T Q, dQ = dS K                   (SS, 128 x 64 x 128 each)
//   warps drain dQ (and dK, dV after the item's last step) from TMEM into a shared-memory staging area; warp 3 sends the
//         staged tiles to HBM with TMA stores / TMA reduce-adds
// The issuer launches the NEXT step's S / dP as soon as the warps hold the current ones in registers, so the tensor
// core is never waiting for the exponentials of the step it just finished.
// D = rowsum(dO * O): packed rows are whole in one tile, so D = sum_j Pd_ij dP_ij is formed in the kernel (the two
// threads of a row swap partial sums through shared memory); long rows take it from a small pre-pass over O and dO.
// shared-memory map.  Pd_s / dS_s are two [128 query x 64 key] chunks each; in the packed geometry only the diagonal
// quarters are ever non-zero, so the chunks overlap on one shared 8 KB block of zeros (chunk stride 8 KB instead of 16):
//   [rows 0..63 of chunk 0 | zeros = rows 64..127 of chunk 0 = rows 0..63 of chunk 1 | rows 64..127 of chunk 1]
// OUT is the staging area the results leave through (TMA store / reduce-add issued by warp 3):
//   packed: dQ | dK | dV tiles (bf16);  long: dQ as two fp32 [128 x 32] sub-tiles, reused for dK | dV at the item's end
template <bool kPacked> struct BwdMap {
    static constexpr int QD_STAGES = 2;
    static constexpr int CHUNK = kPacked ? TILE_BYTES / 2 : TILE_BYTES;   // byte distance between the two key chunks
    static constexpr int PD_BYTES = CHUNK + TILE_BYTES;
    static constexpr int KV_OFF = 0;                                      // [slot 2] K tile | V tile
    static constexpr int QD_OFF = KV_OFF + 2 * 2 * TILE_BYTES;            // [stage] Q tile | dO tile
    static constexpr int PD_OFF = QD_OFF + QD_STAGES * 2 * TILE_BYTES;
    static constexpr int DS_OFF = PD_OFF + PD_BYTES;
    static constexpr int OUT_OFF = DS_OFF + PD_BYTES;
    static constexpr int OUT_BYTES = kPacked ? 3 * TILE_BYTES : 2 * TILE_BYTES;
    static constexpr int DX_OFF = OUT_OFF + OUT_BYTES;                    // float [parity 2][half 2][128] (packed only)
    static constexpr int BAR_OFF = DX_OFF + (kPacked ? 2048 : 0);
    static constexpr int SMEM_BYTES = BAR_OFF + 256;                      // the dynamic array is declared 1024-aligned
    static_assert(SMEM_BYTES <= 232448, "backward shared memory");
};
constexpr int G_QD_MAX_STAGES = 2;
constexpr uint32_t G_TM_S = 0, G_TM_DP = 128, G_TM_DV = 256, G_TM_DK = 320, G_TM_DQ = 384;

struct BwdBars {
    uint64_t kv_full[2], kv_empty[2];
    uint64_t qd_full[G_QD_MAX_STAGES], qd_empty[G_QD_MAX_STAGES];
    uint64_t sdp_full, sdp_free, pds_full, mma2_done, out_full, out_free;
    uint32_t tmem_ptr;
};
static_assert(sizeof(BwdBars) <= 256, "barrier block");

template <bool kPacked> struct BwdItem {
    bool valid;
    int prob[2];  // packed: the two problems of the tile; long: prob[0] = b*H + h
    int k0;       // long: first key of the block
};
template <bool kPacked>
__device__ __forceinline__ void bwd_decode(int kk, int B, int N, int H, BwdItem<kPacked> &it) {
    const int idx = blockIdx.x + kk * gridDim.x;
    if (kPacked) {
        it.valid = idx < ((B * H + 1) >> 1);
        it.prob[0] = 2 * idx;
        it.prob[1] = 2 * idx + 1;
        it.k0 = 0;
    } else {
        const int nkb = (N + TN - 1) / TN;
        it.valid = idx < B * H * nkb;
        it.prob[0] = it.prob[1] = idx / nkb;
        it.k0 = (idx - it.prob[0] * nkb) * TN;
    }
}

template <bool kPacked>
__global__ void __launch_bounds__(384, 1)
attn_tc_bwd_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_do,
                   const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ CUtensorMap tm_acc,
                   const float *__restrict__ lse, const float *__restrict__ Drow, int B, int N, int H, float scale,
                   DropoutParams drop) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((ptx::smem_u32(smem) & 1023u) != 0) asm volatile("trap;");   // SWIZZLE_128B tiles need the declared alignment
    using Map = BwdMap<kPacked>;
    constexpr int G_KV_OFF = Map::KV_OFF, G_QD_OFF = Map::QD_OFF, G_PD_OFF = Map::PD_OFF, G_DS_OFF = Map::DS_OFF,
                  G_DX_OFF = Map::DX_OFF, G_QD_STAGES = Map::QD_STAGES, G_OUT_OFF = Map::OUT_OFF, G_CHUNK = Map::CHUNK;
    BwdBars *bars = reinterpret_cast<BwdBars *>(smem + Map::BAR_OFF);

    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int inner = H * DH;
    const int nsteps = kPacked ? 1 : (N + TM - 1) / TM;   // query blocks per item

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_qkv);
        ptx::prefetch_tensormap(&tm_do);
        ptx::prefetch_tensormap(&tm_out);
        if (!kPacked) ptx::prefetch_tensormap(&tm_acc);
    }
    if (warp == 1 && lane == 0) {
        ptx::mbar_init(&bars->out_full, 8);
        ptx::mbar_init(&bars->out_free, 1);
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(&bars->kv_full[s], 1);
            ptx::mbar_init(&bars->kv_empty[s], 1);
        }
        for (int s = 0; s < G_QD_STAGES; ++s) {
            ptx::mbar_init(&bars->qd_full[s], 1);
            ptx::mbar_init(&bars->qd_empty[s], 1);
        }
        ptx::mbar_init(&bars->sdp_full, 1);
        ptx::mbar_init(&bars->sdp_free, 8);   // one arrival per compute warp
        ptx::mbar_init(&bars->pds_full, 8);
        ptx::mbar_init(&bars->mma2_done, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc(&bars->tmem_ptr, 512);
    if (kPacked && warp >= 4) {
        // the shared block of zeros of Pd_s and of dS_s (never written afterwards)
        const int tid = threadIdx.x - 128;
        for (int i = tid; i < 2 * 512; i += 256) {
            uint8_t *base = smem + ((i >> 9) ? G_DS_OFF : G_PD_OFF) + G_CHUNK;
            *reinterpret_cast<uint4 *>(base + (i & 511) * 16) = make_uint4(0u, 0u, 0u, 0u);
        }
        ptx::fence_proxy_async_smem();
    }
    ptx::tcgen05_fence_before();
    __syncthreads();
    ptx::tcgen05_fence_after();
    const uint32_t tmem_base = bars->tmem_ptr;
    pdl_wait();

    if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 0) {
        // ================================ TMA producer ==================================================
        int kvc = 0, qdc = 0;
        for (int kk = 0;; ++kk) {
            BwdItem<kPacked> it;
            bwd_decode<kPacked>(kk, B, N, H, it);
            if (!it.valid) break;
            {
                const int slot = kvc & 1;
                ptx::mbar_wait(&bars->kv_empty[slot], ((kvc >> 1) & 1) ^ 1);
                if (ptx::elect_one()) {
                    uint8_t *dst = smem + G_KV_OFF + slot * 2 * TILE_BYTES;
                    ptx::mbar_arrive_expect_tx(&bars->kv_full[slot], 2 * TILE_BYTES);
                    if (kPacked) {
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
                            const int p = it.prob[i], c = (p % H) * DH, b = p / H;
                            ptx::tma_load_3d(dst + i * (TILE_BYTES / 2), &tm_qkv, &bars->kv_full[slot], inner + c, 0, b);
                            ptx::tma_load_3d(dst + TILE_BYTES + i * (TILE_BYTES / 2), &tm_qkv, &bars->kv_full[slot],
                                             2 * inner + c, 0, b);
                        }
                    } else {
                        const int p = it.prob[0], c = (p % H) * DH, b = p / H;
                        ptx::tma_load_3d(dst, &tm_qkv, &bars->kv_full[slot], inner + c, it.k0, b);
                        ptx::tma_load_3d(dst + TILE_BYTES, &tm_qkv, &bars->kv_full[slot], 2 * inner + c, it.k0, b);
                    }
                }
                __syncwarp();
                ++kvc;
            }
            for (int i = 0; i < nsteps; ++i) {
                const int st = qdc % G_QD_STAGES;
                ptx::mbar_wait(&bars->qd_empty[st], ((qdc / G_QD_STAGES) & 1) ^ 1);
                if (ptx::elect_one()) {
                    uint8_t *dst = smem + G_QD_OFF + st * 2 * TILE_BYTES;
                    ptx::mbar_arrive_expect_tx(&bars->qd_full[st], 2 * TILE_BYTES);
                    if (kPacked) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const int p = it.prob[j], c = (p % H) * DH, b = p / H;
                            ptx::tma_load_3d(dst + j * (TILE_BYTES / 2), &tm_qkv, &bars->qd_full[st], c, 0, b);
                            ptx::tma_load_3d(dst + TILE_BYTES + j * (TILE_BYTES / 2), &tm_do, &bars->qd_full[st], c, 0, b);
                        }
                    } else {
                        const int p = it.prob[0], c = (p % H) * DH, b = p / H;
                        ptx::tma_load_3d(dst, &tm_qkv, &bars->qd_full[st], c, i * TM, b);
                        ptx::tma_load_3d(dst + TILE_BYTES, &tm_do, &bars->qd_full[st], c, i * TM, b);
                    }
                }
                __syncwarp();
                ++qdc;
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ====================================================
        constexpr uint32_t idesc_s = ptx::make_idesc_bf16(TM, TN, 0, 0);    // S, dP: both operands K-major
        constexpr uint32_t idesc_kv = ptx::make_idesc_bf16(TN, DH, 1, 1);   // dV, dK: A = Pd_s / dS_s transposed, B = dO / Q
        constexpr uint32_t idesc_q = ptx::make_idesc_bf16(TM, DH, 0, 1);    // dQ: A = dS_s, B = K (MN-major)
        const uint32_t sb = ptx::smem_u32(smem);
        int kvc = 0, qdc = 0;
        uint32_t fph = 0, pph = 0;
        auto mma1 = [&](int kvslot, int st) {
            ptx::tcgen05_fence_after();
            if (ptx::elect_one()) {
                const uint32_t kv = sb + G_KV_OFF + kvslot * 2 * TILE_BYTES, qd = sb + G_QD_OFF + st * 2 * TILE_BYTES;
                const uint64_t dq_ = ptx::make_smem_desc(qd, 16, 1024), dk_ = ptx::make_smem_desc(kv, 16, 1024);
                const uint64_t ddo = ptx::make_smem_desc(qd + TILE_BYTES, 16, 1024),
                               dv_ = ptx::make_smem_desc(kv + TILE_BYTES, 16, 1024);
#pragma unroll
                for (int k = 0; k < DH / 16; ++k)
                    ptx::umma_bf16(tmem_base + G_TM_S, dq_ + 2 * k, dk_ + 2 * k, idesc_s, k > 0 ? 1u : 0u);
#pragma unroll
                for (int k = 0; k < DH / 16; ++k)
                    ptx::umma_bf16(tmem_base + G_TM_DP, ddo + 2 * k, dv_ + 2 * k, idesc_s, k > 0 ? 1u : 0u);
                ptx::umma_commit(&bars->sdp_full);
            }
            __syncwarp();
        };
        auto mma2 = [&](int kvslot, int st, bool acc, bool last_of_item) {
            ptx::tcgen05_fence_after();
            if (ptx::elect_one()) {
                const uint32_t kv = sb + G_KV_OFF + kvslot * 2 * TILE_BYTES, qd = sb + G_QD_OFF + st * 2 * TILE_BYTES;
                // MN-major operands: 16 contraction rows (queries / keys) = 2048 B per UMMA_K; A spans two 64-wide chunks
                const uint64_t a_pd = ptx::make_smem_desc(sb + G_PD_OFF, G_CHUNK, 1024);
                const uint64_t a_ds = ptx::make_smem_desc(sb + G_DS_OFF, G_CHUNK, 1024);
                const uint64_t b_do = ptx::make_smem_desc(qd + TILE_BYTES, 8192, 1024);
                const uint64_t b_q = ptx::make_smem_desc(qd, 8192, 1024);
                const uint64_t b_k = ptx::make_smem_desc(kv, 8192, 1024);
                const uint64_t a_dsk = ptx::make_smem_desc(sb + G_DS_OFF, 16, 1024);   // dS_s as a K-major operand
#pragma unroll
                for (int k = 0; k < TM / 16; ++k)
                    ptx::umma_bf16(tmem_base + G_TM_DV, a_pd + 128 * k, b_do + 128 * k, idesc_kv, (acc || k > 0) ? 1u : 0u);
#pragma unroll
                for (int k = 0; k < TM / 16; ++k)
                    ptx::umma_bf16(tmem_base + G_TM_DK, a_ds + 128 * k, b_q + 128 * k, idesc_kv, (acc || k > 0) ? 1u : 0u);
#pragma unroll
                for (int k = 0; k < TN / 16; ++k)   // keys: chunk k / 4, 32 B per UMMA_K inside the chunk
                    ptx::umma_bf16(tmem_base + G_TM_DQ, a_dsk + (k >> 2) * (G_CHUNK >> 4) + 2 * (k & 3), b_k + 128 * k,
                                   idesc_q, k > 0 ? 1u : 0u);
                ptx::umma_commit(&bars->mma2_done);
                ptx::umma_commit(&bars->qd_empty[st]);
                if (last_of_item) ptx::umma_commit(&bars->kv_empty[kvslot]);
            }
            __syncwarp();
        };
        auto wait_kv = [&]() {
            const int slot = kvc & 1;
            ptx::mbar_wait(&bars->kv_full[slot], (kvc >> 1) & 1);
            ++kvc;
            return slot;
        };
        auto wait_qd = [&]() {
            const int st = qdc % G_QD_STAGES;
            ptx::mbar_wait(&bars->qd_full[st], (qdc / G_QD_STAGES) & 1);
            ++qdc;
            return st;
        };
        BwdItem<kPacked> it;
        bwd_decode<kPacked>(0, B, N, H, it);
        int kv_cur = 0, st_cur = 0;
        if (it.valid) {
            kv_cur = wait_kv();
            st_cur = wait_qd();
            mma1(kv_cur, st_cur);
        }
        for (int kk = 0; it.valid; ++kk) {
            BwdItem<kPacked> nxt;
            bwd_decode<kPacked>(kk + 1, B, N, H, nxt);
            for (int i = 0; i < nsteps; ++i) {
                const bool last = i + 1 == nsteps;
                int kv_next = kv_cur, st_next = 0;
                if (!last || nxt.valid) {
                    ptx::mbar_wait(&bars->sdp_free, fph);   // S and dP are in the compute warps' registers
                    fph ^= 1;
                    // (issuing this step's second group of products first whenever the next operands are still in flight
                    // was measured slower: 43.1 vs 41.1 us at cfg2 -- the next S / dP then arrive late for the warps)
                    if (last) kv_next = wait_kv();
                    st_next = wait_qd();
                    mma1(kv_next, st_next);
                }
                ptx::mbar_wait(&bars->pds_full, pph);       // Pd_s / dS_s written, previous outputs drained
                pph ^= 1;
                mma2(kv_cur, st_cur, i > 0, last);
                kv_cur = kv_next;
                st_cur = st_next;
            }
            it = nxt;
        }
    } else if (warp == 3) {
        // ================================ result warp: TMA stores / reduce-adds out of the staging area ==
        uint32_t oph = 0;
        uint8_t *out = smem + G_OUT_OFF;
        for (int kk = 0;; ++kk) {
            BwdItem<kPacked> it;
            bwd_decode<kPacked>(kk, B, N, H, it);
            if (!it.valid) break;
            for (int i = 0; i < nsteps; ++i) {
                ptx::mbar_wait(&bars->out_full, oph);
                oph ^= 1;
                if (ptx::elect_one()) {
                    if (kPacked) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const int p = it.prob[j], c = (p % H) * DH, b = p / H;
#pragma unroll
                            for (int w = 0; w < 3; ++w)   // dQ, dK, dV
                                ptx::tma_store_3d(&tm_out, out + w * TILE_BYTES + j * (TILE_BYTES / 2), w * inner + c, 0, b);
                        }
                    } else {
                        const int p = it.prob[0], c = (p % H) * DH, b = p / H;
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh)
                            ptx::tma_reduce_add_3d(&tm_acc, out + hh * TILE_BYTES, c + 32 * hh, i * TM, b);
                    }
                    ptx::tma_store_commit();
                    ptx::tma_store_wait_read<0>();
                    ptx::mbar_arrive(&bars->out_free);
                }
                __syncwarp();
                if (!kPacked && i + 1 == nsteps) {
                    ptx::mbar_wait(&bars->out_full, oph);
                    oph ^= 1;
                    if (ptx::elect_one()) {
                        const int p = it.prob[0], c = (p % H) * DH, b = p / H;
                        ptx::tma_store_3d(&tm_out, out, inner + c, it.k0, b);
                        ptx::tma_store_3d(&tm_out, out + TILE_BYTES, 2 * inner + c, it.k0, b);
                        ptx::tma_store_commit();
                        ptx::tma_store_wait_read<0>();
                        ptx::mbar_arrive(&bars->out_free);
                    }
                    __syncwarp();
                }
            }
        }
        if (ptx::elect_one()) ptx::tma_store_wait_all<0>();
        __syncwarp();
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
        // ================================ compute warps (8): thread = (row, column half) ================
        const int g = (warp - 4) >> 2;          // column half handled by this warpgroup
        const int q = warp & 3;                 // TMEM lane quadrant
        const int r = q * 32 + lane;            // row of the tile
        const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
        constexpr int NCH = kPacked ? 1 : 2;    // 32-column chunks per thread
        const int hf = kPacked ? (r >> 6) : 0;  // packed: problem of this row
        const int cbase = kPacked ? 64 * hf + 32 * g : 64 * g;   // first S / dP column of this thread
        const int kcol = kPacked ? 32 * g : 64 * g;              // the same, counted inside the problem's key block
        const float sl2 = scale * LOG2E_F;
        const bool dropping = drop.threshold != 0;
        const uint32_t seed = dropping ? __ldg(drop.seed) : 0u;
        const uint32_t thr = drop.threshold << 16;
        const float sd = drop.scale;
        const int Np = (N + 63) / 64 * 64;
        float *dx = reinterpret_cast<float *>(smem + G_DX_OFF);
        // destination of this thread's Pd / dS values: chunk cbase / 64, 16-byte pieces (cbase % 64) / 8 ... of row r
        uint8_t *pd_row = smem + G_PD_OFF + (cbase >> 6) * G_CHUNK, *ds_row = smem + G_DS_OFF + (cbase >> 6) * G_CHUNK;
        const int piece0 = (cbase & 63) >> 3;

        uint32_t sph = 0, dph = 0;
        int step = 0;
        // what the previous step left in TMEM for this thread to drain
        bool have_prev = false, prev_last = false;
        uint32_t oph = 0;
        uint8_t *out = smem + G_OUT_OFF;
        // 32 accumulator columns of this thread's row -> bf16 -> pieces 4 g .. 4 g + 3 of row r of a staged [128 x 64] tile
        auto stage_bf16 = [&](uint32_t tmem_col, uint8_t *tile, float mul) {
            uint32_t v[32];
            ptx::tmem_ld_32x32(lane_addr + tmem_col + 32 * g, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint4 u;
                u.x = pack_bf16x2(__uint_as_float(v[8 * j + 0]) * mul, __uint_as_float(v[8 * j + 1]) * mul);
                u.y = pack_bf16x2(__uint_as_float(v[8 * j + 2]) * mul, __uint_as_float(v[8 * j + 3]) * mul);
                u.z = pack_bf16x2(__uint_as_float(v[8 * j + 4]) * mul, __uint_as_float(v[8 * j + 5]) * mul);
                u.w = pack_bf16x2(__uint_as_float(v[8 * j + 6]) * mul, __uint_as_float(v[8 * j + 7]) * mul);
                *reinterpret_cast<uint4 *>(tile + sw128_offset(r, 4 * g + j)) = u;
            }
        };
        auto publish = [&]() {
            ptx::tcgen05_fence_before();
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&bars->out_full);
        };
        auto wait_out_free = [&]() {
            ptx::mbar_wait(&bars->out_free, oph ^ 1);   // the result warp's previous operations have read the staging area
            oph ^= 1;
        };
        // the previous step's results leave TMEM through the staging area (warp 3 issues the TMA operations)
        auto drain = [&]() {
            ptx::mbar_wait(&bars->mma2_done, dph);
            dph ^= 1;
            ptx::tcgen05_fence_after();
            wait_out_free();
            if (kPacked) {
                stage_bf16(G_TM_DQ, out, scale);
                stage_bf16(G_TM_DK, out + TILE_BYTES, scale);
                stage_bf16(G_TM_DV, out + 2 * TILE_BYTES, 1.0f);
                publish();
            } else {
                {   // dQ of the step, fp32: sub-tile g holds columns 32 g .. 32 g + 31 (128-byte rows)
                    uint32_t v[32];
                    ptx::tmem_ld_32x32(lane_addr + G_TM_DQ + 32 * g, v);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<uint4 *>(out + g * TILE_BYTES + sw128_offset(r, j)) =
                            make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                }
                publish();
                if (prev_last) {
                    wait_out_free();
                    stage_bf16(G_TM_DK, out, scale);
                    stage_bf16(G_TM_DV, out + TILE_BYTES, 1.0f);
                    publish();
                }
            }
        };

        // row statistics of step (kk, i): log-sum-exp (+inf for rows that do not exist: P = 0) and, long geometry, D.
        // They come from HBM / L2 and are fetched ONE STEP AHEAD (the packed kernel stalled ~1.5 k cycles per tile on them)
        auto row_stats = [&](int kk_, int i_, float &lse_o, float &D_o) {
            BwdItem<kPacked> it_;
            bwd_decode<kPacked>(kk_, B, N, H, it_);
            lse_o = INFINITY;
            D_o = 0.f;
            if (!it_.valid) return;
            const int prob_ = it_.prob[hf];
            const int qrow_ = kPacked ? (r & 63) : i_ * TM + r;
            if (qrow_ < N && prob_ < B * H) {
                lse_o = __ldg(lse + static_cast<int64_t>(prob_) * N + qrow_);
                if (!kPacked) D_o = __ldg(Drow + static_cast<int64_t>(prob_) * N + qrow_);
            }
        };
        float lse_next, D_next;
        row_stats(0, 0, lse_next, D_next);
        for (int kk = 0;; ++kk) {
            BwdItem<kPacked> it;
            bwd_decode<kPacked>(kk, B, N, H, it);
            if (!it.valid) break;
            const int prob = it.prob[hf];
            for (int i = 0; i < nsteps; ++i, ++step) {
                const int qrow = kPacked ? (r & 63) : i * TM + r;       // query index inside the problem
                const float lse_r = lse_next;
                float D = D_next;
                if (i + 1 < nsteps) row_stats(kk, i + 1, lse_next, D_next);
                else row_stats(kk + 1, 0, lse_next, D_next);
                ptx::mbar_wait(&bars->sdp_full, sph);
                sph ^= 1;
                ptx::tcgen05_fence_after();
                uint32_t s[NCH][32], dp[NCH][32];
#pragma unroll
                for (int c = 0; c < NCH; ++c) ptx::tmem_ld_32x32(lane_addr + G_TM_S + cbase + 32 * c, s[c]);
#pragma unroll
                for (int c = 0; c < NCH; ++c) ptx::tmem_ld_32x32(lane_addr + G_TM_DP + cbase + 32 * c, dp[c]);
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    ptx::tmem_ld_wait_bind32(s[c]);
                    ptx::tmem_ld_wait_bind32(dp[c]);
                }
                ptx::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&bars->sdp_free);
                // ---- P = exp2(S sl2 - lse log2e), t = dP * mask, Pd = P * mask, dS' = P (t - D)   (packed fp32x2 math;
                //      the softmax scale of dS is applied when dQ / dK leave TMEM)
                const float nl2 = -lse_r * LOG2E_F;   // -inf for rows that do not exist: P = 0
                const uint32_t e_row = (static_cast<uint32_t>(prob) * Np + static_cast<uint32_t>(qrow)) * Np +
                                       static_cast<uint32_t>(it.k0 + kcol);
                const uint64_t sl2_2 = splat2(sl2), nl2_2 = splat2(nl2);
                uint32_t pdk[NCH][16], dsk[NCH][16];
                if (!kPacked) {
                    // D is known (pre-pass): one sweep
                    const uint64_t nD2 = splat2(-D);
#pragma unroll
                    for (int c = 0; c < NCH; ++c)
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            float x0, x1;
                            unpack2(fma2(pack2(__uint_as_float(s[c][j]), __uint_as_float(s[c][j + 1])), sl2_2, nl2_2), x0, x1);
                            float p0 = ex2_approx(x0), p1 = ex2_approx(x1);
                            float t0 = __uint_as_float(dp[c][j]), t1 = __uint_as_float(dp[c][j + 1]);
                            float d0 = p0, d1 = p1;
                            if (dropping) {
                                const uint32_t h = dropout_hash(seed, drop.stream, (e_row + 32 * c + j) >> 1);
                                const bool k0 = (h << 16) >= thr, k1 = h >= thr;
                                t0 = k0 ? t0 * sd : 0.f;
                                t1 = k1 ? t1 * sd : 0.f;
                                d0 = k0 ? p0 * sd : 0.f;
                                d1 = k1 ? p1 * sd : 0.f;
                            }
                            float g0, g1;
                            unpack2(mul2(pack2(p0, p1), add2(pack2(t0, t1), nD2)), g0, g1);
                            pdk[c][j >> 1] = pack_bf16x2(d0, d1);
                            dsk[c][j >> 1] = pack_bf16x2(g0, g1);
                        }
                } else {
                    // D = sum over the row's 64 keys of Pd * dP: first sweep keeps P and t in place and packs Pd, then the
                    // two threads of a row swap partial sums through shared memory, then dS'
                    uint64_t part2 = 0ull;
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        float x0, x1;
                        unpack2(fma2(pack2(__uint_as_float(s[0][j]), __uint_as_float(s[0][j + 1])), sl2_2, nl2_2), x0, x1);
                        const float p0 = ex2_approx(x0), p1 = ex2_approx(x1);
                        float t0 = __uint_as_float(dp[0][j]), t1 = __uint_as_float(dp[0][j + 1]);
                        float d0 = p0, d1 = p1;
                        if (dropping) {
                            const uint32_t h = dropout_hash(seed, drop.stream, (e_row + j) >> 1);
                            const bool k0 = (h << 16) >= thr, k1 = h >= thr;
                            t0 = k0 ? t0 * sd : 0.f;
                            t1 = k1 ? t1 * sd : 0.f;
                            d0 = k0 ? p0 * sd : 0.f;
                            d1 = k1 ? p1 * sd : 0.f;
                        }
                        part2 = fma2(pack2(p0, p1), pack2(t0, t1), part2);
                        pdk[0][j >> 1] = pack_bf16x2(d0, d1);
                        s[0][j] = __float_as_uint(p0);
                        s[0][j + 1] = __float_as_uint(p1);
                        dp[0][j] = __float_as_uint(t0);
                        dp[0][j + 1] = __float_as_uint(t1);
                    }
                    const float part = pair_sum2(part2);
                    float *slot = dx + (step & 1) * 256;
                    slot[g * 128 + r] = part;
                    ptx::named_bar_sync(3, 256);
                    const uint64_t nD2 = splat2(-(part + slot[(g ^ 1) * 128 + r]));
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        float g0, g1;
                        unpack2(mul2(pack2(__uint_as_float(s[0][j]), __uint_as_float(s[0][j + 1])),
                                     add2(pack2(__uint_as_float(dp[0][j]), __uint_as_float(dp[0][j + 1])), nD2)), g0, g1);
                        dsk[0][j >> 1] = pack_bf16x2(g0, g1);
                    }
                }
                // ---- the previous step's outputs leave TMEM before the tensor core may overwrite them
                if (have_prev) drain();
                // ---- Pd_s / dS_s rows (swizzled 16-byte pieces), then hand over to the tensor core
#pragma unroll
                for (int c = 0; c < NCH; ++c)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t off = sw128_offset(r, piece0 + 4 * c + j);
                        *reinterpret_cast<uint4 *>(pd_row + off) =
                            make_uint4(pdk[c][4 * j], pdk[c][4 * j + 1], pdk[c][4 * j + 2], pdk[c][4 * j + 3]);
                        *reinterpret_cast<uint4 *>(ds_row + off) =
                            make_uint4(dsk[c][4 * j], dsk[c][4 * j + 1], dsk[c][4 * j + 2], dsk[c][4 * j + 3]);
                    }
                ptx::fence_proxy_async_smem();
                ptx::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&bars->pds_full);
                have_prev = true;
                prev_last = i + 1 == nsteps;
            }
        }
        if (have_prev) drain();
    }

    ptx::tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tcgen05_fence_after();
        ptx::tmem_dealloc(tmem_base, 512);
    }
}

// D[b, h, i] = sum_d dO[i, d] * O[i, d] for the long geometry; one warp per (token row, head)
__global__ void __launch_bounds__(256) attn_tc_dot_kernel(const bf16 *__restrict__ o, const bf16 *__restrict__ d_o,
                                                           float *__restrict__ D, int B, int N, int H) {
    pdl_launch_dependents();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t wid = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);   // (b * N + i) * H + h
    if (wid >= static_cast<int64_t>(B) * N * H) return;
    const int h = static_cast<int>(wid % H);
    const int64_t row = wid / H;
    const int64_t off = row * (static_cast<int64_t>(H) * DH) + h * DH + 2 * lane;
    float a0, a1, b0, b1;
    unpack_bf16x2(*reinterpret_cast<const uint32_t *>(o + off), a0, a1);
    unpack_bf16x2(*reinterpret_cast<const uint32_t *>(d_o + off), b0, b1);
    const float part = warp_sum(fmaf(a0, b0, a1 * b1));
    if (lane == 0) D[((row / N) * H + h) * N + row % N] = part;
}

// dqkv[:, 0 : inner] = bf16(scale * dq_acc)   (long geometry: dS K was accumulated in fp32 across the key blocks)
__global__ void __launch_bounds__(256) attn_tc_dq_convert_kernel(const float *__restrict__ acc, bf16 *__restrict__ dqkv,
                                                                  int64_t rows, int inner, float mul) {
    pdl_launch_dependents();
    pdl_wait();
    const int64_t n8 = rows * (inner / 8);
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t row = i / (inner / 8);
        const int c = static_cast<int>(i - row * (inner / 8)) * 8;
        float v[8];
        load8(acc + row * inner + c, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] *= mul;
        store8(dqkv + row * 3 * static_cast<int64_t>(inner) + c, v);
    }
}

template <bool kPacked>
int launch_bwd(const void *qkv, const void *d_o, const float *lse, const float *Drow, void *dqkv, float *dq_acc, int B,
               int N, int H, float scale, DropoutParams drop, cudaStream_t stream) {
    const int inner = H * DH;
    CUtensorMap tq, td, tout, tacc;
    int rc;
    if ((rc = make_tmap3(&tq, qkv, 3 * inner, N, B, 3 * (int64_t)inner, kPacked ? 64 : TM))) return rc;
    if ((rc = make_tmap3(&td, d_o, inner, N, B, inner, kPacked ? 64 : TM))) return rc;
    if ((rc = make_tmap3(&tout, dqkv, 3 * inner, N, B, 3 * (int64_t)inner, kPacked ? 64 : TM))) return rc;
    tacc = tout;
    if (!kPacked && (rc = make_tmap3(&tacc, dq_acc, inner, N, B, inner, TM, /*fp32=*/true))) return rc;
    auto kern = attn_tc_bwd_kernel<kPacked>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdMap<kPacked>::SMEM_BYTES);
        if (e != cudaSuccess) return fail((int)e, "cudaFuncSetAttribute(attn_tc_bwd): %s", cudaGetErrorString(e));
        attr_set = true;
    }
    const int items = kPacked ? (B * H + 1) >> 1 : B * H * ((N + TN - 1) / TN);
    const int grid = items < sm_count() ? items : sm_count();
    cudaError_t le = launch_pdl(kern, dim3(grid), dim3(384), BwdMap<kPacked>::SMEM_BYTES, stream, tq, td, tout, tacc, lse,
                                Drow, B, N, H, scale, drop);
    if (le != cudaSuccess) return fail((int)le, "attn_tc_bwd launch: %s", cudaGetErrorString(le));
    return check_launch("attn_tc_bwd");
}

}  // namespace

bool attention_tc_supported(int N, int dh) { return dh == DH && N >= 1; }

int attention_fwd_tc(const void *qkv, void *o, float *lse, int B, int N, int H, int dh, float scale, DropoutParams drop,
                     cudaStream_t stream) {
    ECGVIT_REQUIRE(dh == DH, "attention_fwd_tc: head dim %d (only 64)", dh);
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(o) & 15) == 0,
                   "attention_fwd_tc: qkv / o must be 16-byte aligned");
    if (N <= 64) return launch_fwd<true>(qkv, o, lse, B, N, H, scale, drop, stream);
    return launch_fwd<false>(qkv, o, lse, B, N, H, scale, drop, stream);
}

// fp32 scratch of the long geometry: D [B, H, N] followed by the dQ accumulator [B * N, H * 64]
int64_t attention_bwd_tc_scratch_floats(int B, int N, int H) {
    if (N <= 64) return 0;
    const int64_t d_floats = (static_cast<int64_t>(B) * H * N + 63) / 64 * 64;   // keeps the accumulator 256-byte aligned
    return d_floats + static_cast<int64_t>(B) * N * H * DH;
}

int attention_bwd_tc(const void *qkv, const void *o, const void *d_o, const float *lse, void *dqkv, float *scratch, int B,
                     int N, int H, int dh, float scale, DropoutParams drop, cudaStream_t stream) {
    ECGVIT_REQUIRE(dh == DH, "attention_bwd_tc: head dim %d (only 64)", dh);
    ECGVIT_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_o) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(dqkv) & 15) == 0,
                   "attention_bwd_tc: qkv / d_o / dqkv must be 16-byte aligned");
    if (N <= 64) return launch_bwd<true>(qkv, d_o, lse, nullptr, dqkv, nullptr, B, N, H, scale, drop, stream);
    ECGVIT_REQUIRE(scratch != nullptr && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0,
                   "attention_bwd_tc: N=%d needs the (16-byte aligned) scratch of ecgvit_attention_bwd_scratch_floats", N);
    float *Drow = scratch, *dq_acc = scratch + (static_cast<int64_t>(B) * H * N + 63) / 64 * 64;
    const int64_t rows = static_cast<int64_t>(B) * N, inner = static_cast<int64_t>(H) * DH;
    cudaError_t e = cudaMemsetAsync(dq_acc, 0, sizeof(float) * rows * inner, stream);
    if (e != cudaSuccess) return fail((int)e, "attention_bwd_tc memset: %s", cudaGetErrorString(e));
    const int64_t n_warps = rows * H;
    e = launch_pdl(attn_tc_dot_kernel, dim3((unsigned)((n_warps + 7) / 8)), dim3(256), 0, stream,
                   reinterpret_cast<const bf16 *>(o), reinterpret_cast<const bf16 *>(d_o), Drow, B, N, H);
    if (e != cudaSuccess) return fail((int)e, "attn_tc_dot launch: %s", cudaGetErrorString(e));
    int rc = launch_bwd<false>(qkv, d_o, lse, Drow, dqkv, dq_acc, B, N, H, scale, drop, stream);
    if (rc) return rc;
    e = launch_pdl(attn_tc_dq_convert_kernel, dim3(sm_count() * 4), dim3(256), 0, stream,
                   static_cast<const float *>(dq_acc), reinterpret_cast<bf16 *>(dqkv), rows, (int)inner, scale);
    if (e != cudaSuccess) return fail((int)e, "attn_tc_dq_convert launch: %s", cudaGetErrorString(e));
    return check_launch("attn_tc_dq_convert");
}

}  // namespace ecgvit

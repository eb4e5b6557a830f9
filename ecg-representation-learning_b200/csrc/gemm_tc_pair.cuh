// CTA-pair GEMM kernel (tcgen05 cta_group::2).  Included by gemm_tc.cu inside namespace ecgvit::{anonymous} after the
// tile constants (BM, BK, UMMA_K, kNumThreads, kNumEpilogueWarps, A_STAGE_BYTES) are defined.
//
// A cluster of two CTAs (two SMs of one TPC) owns a 256 x BN output tile.  Each CTA stages only ITS 128 rows of A and
// ITS BN/2 rows of B per k block (32 KB instead of 48 KB at BN = 256); the leader CTA issues one 256 x BN x 16 MMA per
// UMMA_K that reads both halves, and each CTA's TMEM receives its own 128 rows of the accumulator.  This halves the
// B traffic through L2 and through each SM's shared memory (every staged byte is written once by TMA and read once by
// the tensor core, so staging bandwidth is what a single-CTA tile runs out of first).
//
// Synchronisation (all mbarriers live at the same smem offset in both CTAs):
//   full[s]        on the LEADER : leader's arrive.expect_tx(2 x stage bytes); both CTAs' TMA loads complete_tx on it
//   empty[s]       on BOTH       : leader's tcgen05.commit multicast -> each CTA's producer may refill stage s
//   tmem_full[a]   on BOTH       : leader's tcgen05.commit multicast -> each CTA's epilogue drains its 128 rows
//   tmem_empty[a]  on the LEADER : 8 epilogue warps x 2 CTAs arrive (remote arrive from the peer)
//
// Work distribution: the first 256 x BN unit of a cluster is static (unit = cluster index); every further unit comes from
// a global counter.  Warp 3 of the leader fetches the next unit index with one atomicAdd and hands it to every warp of
// both CTAs through a two-slot shared-memory ring:
//   sched_full[s]  on BOTH       : the leader's scheduler stores the index into its own slot and arrives; the peer's slot
//                                  receives it by st.async, which completes 4 expected bytes on the peer's barrier
//   sched_empty[s] on the LEADER : every consumer warp of both CTAs arrives after reading the slot
// A cluster that becomes resident late (its SMs were still held by a kernel of the other stream, or by NCCL) therefore
// takes fewer units instead of making the whole grid wait for its statically assigned share.
#pragma once

template <int BN, bool B_MN, bool WIDE = false, int TILES = 2> struct PairCfg {
    static constexpr int B_HALF = BN / 2;                                      // B rows (N values) per CTA
    // MN-major B is staged in 64-wide chunks; at BN = 192 the second chunk is only half used (over-fetch)
    static constexpr int B_LOAD_ROWS = B_MN ? ((B_HALF + 63) / 64) * 64 : B_HALF;
    static constexpr int B_STAGE_BYTES = B_LOAD_ROWS * BK * 2;
    static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;          // per CTA
    // epilogue: one warp per (TMEM lane quadrant, 64-column group) -> BN / 16 warps, 2 units of 32 columns each.
    // More, narrower epilogue warps (16 at BN = 256) keep the 4 issue slots of the SM busy: the GELU / dropout
    // epilogues are instruction bound and two warps per scheduler cannot hide their own latencies.
    static constexpr int EPI_WARPS = BN / 16;
    static constexpr int THREADS = 128 + 32 * EPI_WARPS;
    static constexpr int UNITS_PER_WARP = 2;                                   // 32-column units per epilogue warp
    // staging: every epilogue warp owns two 32-row x 32-column tiles: 64-byte rows of bf16 (SWIZZLE_64B), or 128-byte
    // rows of fp32 (SWIZZLE_128B) for the fp32 residual stream and the split-K reduction (WIDE; the latter with one
    // tile per warp, which leaves the weight-gradient contraction its five pipeline stages at BN = 256)
    static constexpr int EPI_TILE_BYTES = WIDE ? 32 * 128 : 32 * 64;
    static constexpr int EPI_TILES_PER_WARP = TILES;
    static constexpr int EPI_BYTES = EPI_WARPS * EPI_TILES_PER_WARP * EPI_TILE_BYTES;
    static constexpr int SCHED_SLOTS = 2;                                      // unit indices in flight per cluster
    static constexpr int NUM_BARRIERS = 2 * 8 + 4 + EPI_WARPS * EPI_TILES_PER_WARP + 2 * SCHED_SLOTS;
    static constexpr int PIPE_BUDGET = 232448 - 1024 - 1024 - EPI_BYTES;
    static constexpr int STAGES = (PIPE_BUDGET / STAGE_BYTES) > 8 ? 8 : (PIPE_BUDGET / STAGE_BYTES);
    static constexpr int TMEM_COLS = (2 * BN <= 256) ? 256 : 512;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 1024 + 1024;
    static_assert(NUM_BARRIERS * 8 + 16 + 4 * SCHED_SLOTS <= 1024, "barrier block");
    static_assert(BN % 64 == 0, "tile width");
};
// the configuration of one (tile width, B layout, epilogue) instantiation
template <int BN, bool B_MN, int MODE>
using PairCfgFor = PairCfg<BN, B_MN, MODE == ECGVIT_EPI_BIAS_RES_F32 || MODE == ECGVIT_EPI_ATOMIC_F32,
                           MODE == ECGVIT_EPI_ATOMIC_F32 ? 1 : 2>;

// byte offset of 16-byte chunk j (0..3) of row `lane` inside a 32 x 64-byte SWIZZLE_64B tile
__device__ __forceinline__ uint32_t sw64_offset(int lane, int j) {
    return static_cast<uint32_t>(lane) * 64u + (static_cast<uint32_t>(j ^ ((lane >> 1) & 3)) << 4);
}

// Epilogue math for 32 consecutive accumulator columns of one row (thread = row).  Results are written as bf16 into
// the warp's swizzled staging tile(s); for BIAS_RES / DGELU the tile already holds the aux operand (residual /
// pre-activation), fetched by TMA while the mainloop was still running, and is updated in place.
// The caller then issues one TMA store per tile (TMA clips rows >= M and columns >= N, so there are no guards here).
// BIAS_SUB_ROWSQ: the tile holds the target; out = acc + bias - target, and `sq` accumulates the fp32 squares.
// kPath (BIAS_RES): the dropped branch is scaled by the row's drop-path factor `rs` before the residual add.
template <int MODE, bool kPath = false>
__device__ __forceinline__ void epilogue_half16(const EpiParams &ep, int64_t row, int col_base, int jbase,
                                                const uint32_t r[16], uint8_t *tile0, uint8_t *tile1, int lane,
                                                int n_cols, float &sq, float rs = 1.f) {
    const bool drop = ep.drop.threshold != 0;  // kernel-uniform
    const uint32_t seed = drop ? __ldg(ep.drop.seed) : 0u;
#pragma unroll
    for (int jj = 0; jj < 2; ++jj) {
        const int j = jbase + jj;  // 16-byte chunk of the 32-column tile
        const int col = col_base + 8 * j;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[8 * jj + i]);
        if (MODE != ECGVIT_EPI_DGELU && ep.bias != nullptr && col < n_cols) {
            // every lane reads the same 32 bytes (one L1 wavefront per load, the 3 K floats of a bias stay L1 resident):
            // two broadcast loads instead of eight shuffles per 8 columns
            const float4 b0 = __ldg(reinterpret_cast<const float4 *>(ep.bias + col));
            const float4 b1 = __ldg(reinterpret_cast<const float4 *>(ep.bias + col + 4));
            v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
            v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
        }
        const uint32_t soff = sw64_offset(lane, j);
        const uint32_t eidx = static_cast<uint32_t>(row * ep.ldo + col);  // element index of v[0] (even)
        if (drop && (MODE == ECGVIT_EPI_BIAS_RES || MODE == ECGVIT_EPI_DGELU)) dropout_apply<8>(ep.drop, seed, eidx, v);
        if (kPath) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] *= rs;
        }
        if (MODE == ECGVIT_EPI_BIAS_RES || MODE == ECGVIT_EPI_DGELU || MODE == ECGVIT_EPI_BIAS_SUB_ROWSQ) {
            const uint4 a4 = *reinterpret_cast<const uint4 *>(tile0 + soff);
            float a[8];
            unpack_bf16x2(a4.x, a[0], a[1]); unpack_bf16x2(a4.y, a[2], a[3]);
            unpack_bf16x2(a4.z, a[4], a[5]); unpack_bf16x2(a4.w, a[6], a[7]);
            if (MODE == ECGVIT_EPI_BIAS_RES) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += a[i];
            } else if (MODE == ECGVIT_EPI_BIAS_SUB_ROWSQ) {
                // columns >= N hold zeros on both sides (zero-filled B rows and target columns, no bias): they add 0
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    v[i] -= a[i];
                    sq = fmaf(v[i], v[i], sq);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; i += 2) {
                    float g0, g1;
                    gelu_grad_pair(a[i], a[i + 1], g0, g1);
                    v[i] *= g0;
                    v[i + 1] *= g1;
                }
            }
        }
        uint4 packed;
        packed.x = pack_bf16x2(v[0], v[1]); packed.y = pack_bf16x2(v[2], v[3]);
        packed.z = pack_bf16x2(v[4], v[5]); packed.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4 *>(tile0 + soff) = packed;
        if (MODE == ECGVIT_EPI_BIAS_GELU) {
            // gelu of the fp32 pre-activation (its bf16 rounding, which backward differentiates, moves h by less than
            // h's own bf16 rounding)
            float h[8];
#pragma unroll
            for (int i = 0; i < 8; i += 2) gelu_fwd_pair(v[i], v[i + 1], h[i], h[i + 1]);
            if (drop) dropout_apply<8>(ep.drop, seed, eidx, h);
            uint4 ph;
            ph.x = pack_bf16x2(h[0], h[1]); ph.y = pack_bf16x2(h[2], h[3]);
            ph.z = pack_bf16x2(h[4], h[5]); ph.w = pack_bf16x2(h[6], h[7]);
            *reinterpret_cast<uint4 *>(tile1 + soff) = ph;
        }
    }
}

// fp32 residual stream (ECGVIT_EPI_BIAS_RES_F32): out = drop(acc + bias) + aux with aux / out fp32.  The warp's staging
// tile is 32 rows x 128 bytes (SWIZZLE_128B) and already holds the residual; 16 columns = four 16-byte pieces per call.
// kPath: out = rs * drop(acc + bias) + aux with the row's drop-path factor rs.
template <bool kPath = false>
__device__ __forceinline__ void epilogue_half16_f32(const EpiParams &ep, int64_t row, int col_base, int half,
                                                    const uint32_t r[16], uint8_t *tile, int lane, int n_cols,
                                                    float rs = 1.f) {
    const bool drop = ep.drop.threshold != 0;  // kernel-uniform
    const uint32_t seed = drop ? __ldg(ep.drop.seed) : 0u;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        const int jc = 4 * half + jj;  // 16-byte piece (4 floats) of the 32-column row
        const int col = col_base + 4 * jc;
        float v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[4 * jj + i]);
        if (ep.bias != nullptr && col < n_cols) {
            const float4 b = __ldg(reinterpret_cast<const float4 *>(ep.bias + col));
            v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
        }
        if (drop) dropout_apply<4>(ep.drop, seed, static_cast<uint32_t>(row * ep.ldo + col), v);
        if (kPath) {
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] *= rs;
        }
        float4 *p = reinterpret_cast<float4 *>(tile + static_cast<uint32_t>(lane) * 128u +
                                               (static_cast<uint32_t>(jc ^ (lane & 7)) << 4));
        float4 a = *p;
        a.x += v[0]; a.y += v[1]; a.z += v[2]; a.w += v[3];
        *p = a;
    }
}

// kPath: the drop-path variant of the residual epilogues (BIAS_RES / BIAS_RES_F32), whose `ep` is an EpiPathParams
template <bool kPath> using EpiParamsFor = typename std::conditional<kPath, EpiPathParams, EpiParams>::type;

template <int BN, bool A_MN, bool B_MN, int MODE, bool kPath = false>
__global__ void __cluster_dims__(2, 1, 1)
__launch_bounds__(PairCfgFor<BN, B_MN, MODE>::THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_out2,
                const __grid_constant__ CUtensorMap tmap_aux, int M, int N, int K, int split_k, EpiParamsFor<kPath> ep,
                int *__restrict__ sched_ctr) {
    constexpr bool kWide = MODE == ECGVIT_EPI_BIAS_RES_F32;   // (the split-K epilogue has its own fp32 path below)
    using Cfg = PairCfgFor<BN, B_MN, MODE>;
    constexpr bool kRowSq = MODE == ECGVIT_EPI_BIAS_SUB_ROWSQ;
    constexpr bool kHasAux = (MODE == ECGVIT_EPI_BIAS_RES || MODE == ECGVIT_EPI_DGELU || kWide || kRowSq);
    constexpr int STAGES = Cfg::STAGES;
    constexpr int BM2 = 2 * BM;  // rows of the pair tile
    static_assert(!kPath || MODE == ECGVIT_EPI_BIAS_RES || kWide, "drop path belongs to the residual epilogues");

    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *epi_smem = smem + STAGES * Cfg::STAGE_BYTES;  // 1024-byte aligned (stage sizes are multiples of 8 KB)
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(epi_smem + Cfg::EPI_BYTES);
    uint64_t *empty_bar = full_bar + STAGES;
    uint64_t *tmem_full_bar = empty_bar + STAGES;
    uint64_t *tmem_empty_bar = tmem_full_bar + 2;
    uint64_t *aux_bar = tmem_empty_bar + 2;  // [epilogue warp][unit]
    uint64_t *sched_full = aux_bar + Cfg::EPI_WARPS * Cfg::EPI_TILES_PER_WARP;
    uint64_t *sched_empty = sched_full + Cfg::SCHED_SLOTS;
    uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(sched_empty + Cfg::SCHED_SLOTS);
    volatile int *sched_unit = reinterpret_cast<volatile int *>(tmem_ptr_smem + 2);   // [SCHED_SLOTS]
    constexpr int kNoUnit = 0x7fffffff;

    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1;
    const int num_clusters = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tmap_a);
        ptx::prefetch_tensormap(&tmap_b);
        ptx::prefetch_tensormap(&tmap_out);
        if (MODE == ECGVIT_EPI_BIAS_GELU) ptx::prefetch_tensormap(&tmap_out2);
        if (kHasAux) ptx::prefetch_tensormap(&tmap_aux);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            ptx::mbar_init(&tmem_full_bar[a], 1);
            ptx::mbar_init(&tmem_empty_bar[a], 2 * Cfg::EPI_WARPS);
        }
        for (int i = 0; i < Cfg::EPI_WARPS * Cfg::EPI_TILES_PER_WARP; ++i) ptx::mbar_init(&aux_bar[i], 1);
        for (int i = 0; i < Cfg::SCHED_SLOTS; ++i) {
            ptx::mbar_init(&sched_full[i], 1);
            // consumers: TMA producer and epilogue warps of both CTAs, the leader's MMA issuer
            ptx::mbar_init(&sched_empty[i], 2 * Cfg::EPI_WARPS + 3);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc_2sm(tmem_ptr_smem, Cfg::TMEM_COLS);
    ptx::tcgen05_fence_before();
    ptx::cluster_sync_all();
    ptx::tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    pdl_wait();  // everything above overlapped the previous kernel's tail; from here on global memory is touched

    const int tiles_m = (M + BM2 - 1) / BM2;
    const int tiles_n = (N + BN - 1) / BN;
    const int kb_total = (K + BK - 1) / BK;
    const int kb_per_split = (kb_total + split_k - 1) / split_k;
    const int num_units = tiles_m * tiles_n * split_k;
    // called by a whole consumer warp when it is done with its unit number `n_done - 1`: the index of its next unit
    auto next_unit = [&](int n_done) -> int {
        const int slot = (n_done - 1) % Cfg::SCHED_SLOTS;
        ptx::mbar_wait(&sched_full[slot], ((n_done - 1) / Cfg::SCHED_SLOTS) & 1);
        const int u = sched_unit[slot];
        __syncwarp();
        // the arrive is made to depend on the value read (never -1), so it cannot be issued while the load of the slot is
        // still in flight: the scheduler overwrites the slot once every consumer has arrived
        if (lane == 0 && u != -1) ptx::mbar_arrive_cluster(&sched_empty[slot], 0);
        return u;
    };

    if (warp == 0) {
        // ================================ TMA producer (both CTAs) ================================
        // the whole warp walks the loop (warp-uniform control flow and addresses); one elected lane issues
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        for (int u = cluster_id; u != kNoUnit; u = next_unit(++it)) {
            const int tile_n = u % tiles_n;
            const int tile_m = (u / tiles_n) % tiles_m;
            const int split = u / (tiles_n * tiles_m);
            const int kb0 = split * kb_per_split;
            const int kb1 = min(kb0 + kb_per_split, kb_total);
            const int row0 = tile_m * BM2 + rank * BM;          // this CTA's rows of A
            const int col0 = tile_n * BN + rank * Cfg::B_HALF;  // this CTA's rows of B
            for (int kb = kb0; kb < kb1; ++kb) {
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                if (ptx::elect_one()) {
                    uint8_t *sa = smem + stage * Cfg::STAGE_BYTES;
                    uint8_t *sb = sa + A_STAGE_BYTES;
                    if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
                    if (!A_MN) {
                        ptx::tma_load_2d_2sm(sa, &tmap_a, &full_bar[stage], kb * BK, row0);
                    } else {
#pragma unroll
                        for (int j = 0; j < BM / 64; ++j)
                            ptx::tma_load_2d_2sm(sa + j * 8192, &tmap_a, &full_bar[stage], row0 + j * 64, kb * BK);
                    }
                    if (!B_MN) {
                        ptx::tma_load_2d_2sm(sb, &tmap_b, &full_bar[stage], kb * BK, col0);
                    } else {
#pragma unroll
                        for (int j = 0; j < Cfg::B_LOAD_ROWS / 64; ++j)
                            ptx::tma_load_2d_2sm(sb + j * 8192, &tmap_b, &full_bar[stage], col0 + j * 64, kb * BK);
                    }
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer (leader CTA only) ============================
        if (leader) {
            constexpr uint32_t idesc = ptx::make_idesc_bf16(BM2, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
            // descriptors of stage 0 / k = 0; every other (stage, k) only moves the 14-bit start-address field
            const uint32_t smem_base = ptx::smem_u32(smem);
            const uint64_t da0 = A_MN ? ptx::make_smem_desc(smem_base, 8192, 1024) : ptx::make_smem_desc(smem_base, 16, 1024);
            const uint64_t db0 = B_MN ? ptx::make_smem_desc(smem_base + A_STAGE_BYTES, 8192, 1024)
                                      : ptx::make_smem_desc(smem_base + A_STAGE_BYTES, 16, 1024);
            constexpr uint32_t A_KSTEP = (A_MN ? 2048 : 32) >> 4, B_KSTEP = (B_MN ? 2048 : 32) >> 4;
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int u = cluster_id; u != kNoUnit; u = next_unit(++it)) {
                const int split = u / (tiles_n * tiles_m);
                const int kb0 = split * kb_per_split;
                const int kb1 = min(kb0 + kb_per_split, kb_total);
                const int acc = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
                ptx::tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = kb0; kb < kb1; ++kb) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tcgen05_fence_after();
                    if (ptx::elect_one()) {
                        const uint32_t stage_off = static_cast<uint32_t>(stage * Cfg::STAGE_BYTES) >> 4;
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k)
                            ptx::umma_bf16_2sm(tmem_d, da0 + (stage_off + k * A_KSTEP), db0 + (stage_off + k * B_KSTEP),
                                               idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                        ptx::umma_commit_2sm(&empty_bar[stage], 0b11);  // frees the stage in both CTAs
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (ptx::elect_one())
                    ptx::umma_commit_2sm(&tmem_full_bar[acc], 0b11);  // both CTAs' epilogues may drain their half
                __syncwarp();
            }
        }
    } else if (warp == 3) {
        // ================================ unit scheduler (leader CTA, one thread) =================
        if (leader && lane == 0) {
            for (int k = 0;; ++k) {
                const int slot = k % Cfg::SCHED_SLOTS;
                ptx::mbar_wait(&sched_empty[slot], ((k / Cfg::SCHED_SLOTS) & 1) ^ 1);
                int u = num_clusters + atomicAdd(&sched_ctr[0], 1);
                if (u >= num_units) u = kNoUnit;
                sched_unit[slot] = u;
                ptx::mbar_arrive(&sched_full[slot]);
                ptx::mbar_arrive_expect_tx_cluster(&sched_full[slot], 1, 4);
                ptx::st_async_cluster_u32(const_cast<int *>(&sched_unit[slot]), &sched_full[slot], 1,
                                          static_cast<uint32_t>(u));
                if (u == kNoUnit) break;
            }
            // the last cluster to run dry re-arms the counters for the next launch that uses this slot
            __threadfence();
            if (atomicAdd(&sched_ctr[1], 1) == num_clusters - 1) {
                sched_ctr[0] = 0;
                sched_ctr[1] = 0;
                __threadfence();
            }
        }
    } else if (warp >= 4) {
        // ================================ epilogue (both CTAs, own 128 rows) ======================
        const int q = warp & 3;              // TMEM lane quadrant this warp may access
        const int group = (warp - 4) >> 2;   // 64-column group of the tile
        constexpr int UNITS = Cfg::UNITS_PER_WARP;
        uint8_t *tiles = epi_smem + (warp - 4) * Cfg::EPI_TILES_PER_WARP * Cfg::EPI_TILE_BYTES;
        uint64_t *my_aux_bar = aux_bar + (warp - 4) * Cfg::EPI_TILES_PER_WARP;
        // phase of each aux barrier: it only advances on tiles where the unit lies inside the matrix (a partial last
        // column tile skips the load), so it is tracked per barrier, not derived from the tile count
        uint32_t aux_phase = 0;
        int it = 0;
        for (int u = cluster_id; u != kNoUnit; u = next_unit(++it)) {
            const int tile_n = u % tiles_n;
            const int tile_m = (u / tiles_n) % tiles_m;
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            const int row_base = tile_m * BM2 + rank * BM + q * 32;
            const int col_warp = tile_n * BN + group * 64;  // first column of this warp's two units
            if (MODE != ECGVIT_EPI_ATOMIC_F32) {
                // staging tiles are reused every tile: the previous tile's TMA stores must have read them
                if (lane == 0) {
                    ptx::tma_store_wait_read<0>();
                    if (kHasAux) {
                        // fetch the residual / pre-activation tiles now, while the mainloop of this tile is running
#pragma unroll
                        for (int i = 0; i < UNITS; ++i) {
                            if (col_warp + 32 * i < N) {
                                ptx::mbar_arrive_expect_tx(&my_aux_bar[i], Cfg::EPI_TILE_BYTES);
                                ptx::tma_load_2d(tiles + i * Cfg::EPI_TILE_BYTES, &tmap_aux, &my_aux_bar[i],
                                                 col_warp + 32 * i, row_base);
                            }
                        }
                    }
                }
                __syncwarp();
            }
            ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
            ptx::tcgen05_fence_after();
            const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + group * 64;
            const int64_t row = static_cast<int64_t>(row_base) + lane;
            if (MODE == ECGVIT_EPI_ATOMIC_F32) {
                // split-K partial sums: fp32 tile -> swizzled staging -> one TMA reduce-add per 32 x 32 unit (the L2
                // adds whole lines; per-thread red.v4 made this epilogue as long as a 25-k-block mainloop)
                const int n_units = (col_warp >= N) ? 0 : ((col_warp + 32 < N) ? UNITS : 1);
                uint32_t ra[16], rb[16];
                if (n_units > 0) ptx::tmem_ld_32x16(taddr0, ra);
#pragma unroll 1
                for (int i = 0; i < n_units; ++i) {
                    ptx::tmem_ld_wait_bind(ra);
                    ptx::tmem_ld_32x16(taddr0 + 32 * i + 16, rb);
                    if (lane == 0) ptx::tma_store_wait_read<0>();   // the previous unit's reduce has read the tile
                    __syncwarp();
                    uint8_t *trow = tiles + static_cast<uint32_t>(lane) * 128u;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4 *>(trow + (static_cast<uint32_t>(j ^ (lane & 7)) << 4)) =
                            make_uint4(ra[4 * j], ra[4 * j + 1], ra[4 * j + 2], ra[4 * j + 3]);
                    ptx::tmem_ld_wait_bind(rb);
                    if (i + 1 < n_units) ptx::tmem_ld_32x16(taddr0 + 32 * (i + 1), ra);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4 *>(trow + (static_cast<uint32_t>((4 + j) ^ (lane & 7)) << 4)) =
                            make_uint4(rb[4 * j], rb[4 * j + 1], rb[4 * j + 2], rb[4 * j + 3]);
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_reduce_add_2d(&tmap_out, tiles, col_warp + 32 * i, row_base);
                        ptx::tma_store_commit();
                    }
                }
            } else {
                // units entirely outside the matrix are skipped (warp-uniform)
                const int n_units = (col_warp >= N) ? 0 : ((UNITS > 1 && col_warp + 32 < N) ? UNITS : 1);
                // TMEM loads are software-pipelined over the 16-column halves: the load of half s + 1 is in flight
                // while half s is being computed (two register buffers)
                uint32_t ra[16], rb[16];
                float sq = 0.f;   // BIAS_SUB_ROWSQ: this row's squares over the warp's 64 columns
                float rs = 1.f;   // kPath: this row's drop-path factor (one hash per row and tile)
                if constexpr (kPath) rs = path_factor(ep.path, row);
                if (n_units > 0) ptx::tmem_ld_32x16(taddr0, ra);
#pragma unroll 1
                for (int i = 0; i < n_units; ++i) {
                    const int col_base = col_warp + 32 * i;
                    uint8_t *t0, *t1 = nullptr;
                    if (MODE == ECGVIT_EPI_BIAS_GELU) {
                        // one (u, h) tile pair per warp: unit 1 reuses it once unit 0's stores have read it
                        t0 = tiles;
                        t1 = tiles + Cfg::EPI_TILE_BYTES;
                    } else {
                        t0 = tiles + i * Cfg::EPI_TILE_BYTES;
                        if (kHasAux) {
                            ptx::mbar_wait(&my_aux_bar[i], (aux_phase >> i) & 1u);
                            aux_phase ^= 1u << i;
                        }
                    }
                    ptx::tmem_ld_wait_bind(ra);
                    ptx::tmem_ld_32x16(taddr0 + 32 * i + 16, rb);
                    if (MODE == ECGVIT_EPI_BIAS_GELU && i > 0) {
                        if (lane == 0) ptx::tma_store_wait_read<0>();
                        __syncwarp();
                    }
                    if (kWide) epilogue_half16_f32<kPath>(ep, row, col_base, 0, ra, t0, lane, N, rs);
                    else epilogue_half16<MODE, kPath>(ep, row, col_base, 0, ra, t0, t1, lane, N, sq, rs);
                    ptx::tmem_ld_wait_bind(rb);
                    if (i + 1 < n_units) ptx::tmem_ld_32x16(taddr0 + 32 * (i + 1), ra);
                    if (kWide) epilogue_half16_f32<kPath>(ep, row, col_base, 1, rb, t0, lane, N, rs);
                    else epilogue_half16<MODE, kPath>(ep, row, col_base, 2, rb, t0, t1, lane, N, sq, rs);
                    ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_store_2d(&tmap_out, t0, col_base, row_base);
                        if (MODE == ECGVIT_EPI_BIAS_GELU) ptx::tma_store_2d(&tmap_out2, t1, col_base, row_base);
                        ptx::tma_store_commit();
                    }
                }
                // one fp32 partial per (64-column group, row): tiles are multiples of 64 columns wide, so the group index
                // is global and every (group, row) has exactly one writer
                if (kRowSq && n_units > 0 && row < M)
                    reinterpret_cast<float *>(ep.out2)[static_cast<int64_t>(col_warp >> 6) * M + row] = sq;
            }
            ptx::tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);  // the leader's barrier
        }
        if (lane == 0) ptx::tma_store_wait_all<0>();
    }

    ptx::tcgen05_fence_before();
    ptx::cluster_sync_all();  // nobody exits (or frees TMEM) while the peer can still touch this CTA's smem / barriers
    if (warp == 2) {
        ptx::tcgen05_fence_after();
        ptx::tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
    }
}

// gram.cu — Gram matrix of the Laplace deviation matrix on the 5th-gen tensor cores (sm_100a).
//
// Reference: the only dense contraction in lucagiorgetti/Laplace-DQN-Snake-game is on the deviation matrix D
// (P x K Float64, compute_D.jl:53,67-81): plot_traj.jl:10-16 takes svd(D) and uses S.^2/(K-1), which is the
// spectrum of the K x K Gram  G = D' * D  (rows of A = D' are the weight snapshots).  This file computes G.
//
//   G = A A^T,  A = D^T  (K x P, row k = snapshot k, contraction over the P = 181,395 weights)
//
// Precision: tcgen05 has no FP64 kind.  A is split a = hi + lo (+ eps), hi = bf16(a), lo = bf16(a - hi)
// (|eps| <= 2^-18 |a|), and
//      a b ~= hi_a hi_b + hi_a lo_b + lo_a hi_b            (the dropped lo_a lo_b is <= 2^-18 |a b|)
// All three products of a k-step go into ONE TMEM accumulator (FP32), so a tile comes out finished.  Because G is
// symmetric only the tiles that meet the upper triangle are computed (3 products each = 1.5 per output tile on
// average; round 1 computed Y = hi hi^T + hi (2 lo)^T on every tile and G = (Y + Y^T)/2: 2 per tile); the reduction
// pass mirrors them into the lower triangle, so G is exactly symmetric.  terms = 1 issues only hi hi^T (plain bf16).
//
// Kernel: persistent, warp-specialised (canonical sm_100 shape):
//   warp 0   TMA producer   cp.async.bulk.tensor.2d (SWIZZLE_128B / 64B boxes) -> smem ring, mbarrier expect_tx
//   warp 1   MMA issuer     one thread issues tcgen05.mma.cta_group::1.kind::f16, M=128 N=256 K=16, D in TMEM;
//                           tcgen05.commit releases smem stages and publishes the accumulator
//   warps 2-9 accumulate    every CHUNK_K contraction elements (<= 48 MMA steps): tcgen05.ld 32x32b.x32 -> += FP32 registers
//                           (bounds the tensor core's truncating accumulation chain); at the end of the work
//                           item the registers go to the partial tile in the workspace
// Two TMEM accumulator stages (2 x 256 columns): the tensor core fills one while the other is drained.
// Work item = (128 x 256 output tile, split of the contraction); partial tiles are reduced (deterministically)
// by k_gram_finish, which also mirrors the upper triangle of a symmetric problem.
#include <cuda_bf16.h>
#include <string.h>

#include "common.h"
#include "sm100.h"

namespace snk {
namespace gram {

constexpr int BM = 128;           // UMMA M (rows of the A-side operand per tile)
constexpr int BN = 256;           // UMMA N (rows of the B-side operand per tile)
constexpr int UMMA_K = 16;        // bf16
constexpr int NUM_THREADS = 320;  // warp 0 TMA, warp 1 MMA (+TMEM alloc), warps 2..9 accumulate/epilogue
constexpr int NUM_EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;    // 2 accumulator stages x BN fp32 columns
// The tensor core adds into its FP32 accumulator with truncation: a long chain of positive products (the
// diagonal of a Gram) drifts low by ~5e-8 per MMA step.  So the TMEM accumulator only ever holds CHUNK_K
// contraction elements (32 MMA steps for plain bf16, 16 k-slices x 3 products = 48 for the split); the 8 accumulate
// warps drain it (tcgen05.ld) and add it, round-to-nearest, into FP32 registers while the tensor core fills the other
// TMEM stage.
template <int TERMS> constexpr int chunk_k() { return TERMS > 1 ? 256 : 512; }

template <int BK, int TERMS>
struct Cfg {
    static constexpr int ROW_BYTES = BK * 2;                                   // 64 (SW64) or 128 (SW128)
    static constexpr int A_BYTES = BM * ROW_BYTES;
    static constexpr int B_BYTES = BN * ROW_BYTES;
    static constexpr int PLANES = TERMS > 1 ? 2 : 1;                            // stage = [A hi | A lo | B hi | B lo]
    static constexpr int STAGE_BYTES = (A_BYTES + B_BYTES) * PLANES;
    static constexpr int STAGES = (200 * 1024) / STAGE_BYTES > 8 ? 8 : (200 * 1024) / STAGE_BYTES;
    static constexpr int CH = chunk_k<TERMS>() / BK;                            // k-blocks per TMEM accumulation chunk
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
    static constexpr uint64_t LAYOUT = (BK == 64) ? LAYOUT_SW128 : LAYOUT_SW64;
    static constexpr uint32_t SBO_BYTES = 8 * ROW_BYTES;                       // 8-row swizzle atom pitch
};

// Tile order: column panels PANEL tiles wide, swept down the rows.  The CTAs (or CTA pairs) that run concurrently then
// cover a roughly square block of the output, so per k-step they pull ~2*sqrt(n) distinct operand tiles through L2
// instead of n + 1 (one A row-block against every B tile).
constexpr int PANEL = 8;
__device__ __forceinline__ void tile_coords(int tile, int tiles_m, int tiles_n, int &tm, int &tn) {
    const int per_panel = PANEL * tiles_m;
    const int panel = tile / per_panel, within = tile - panel * per_panel;
    const int width = min(PANEL, tiles_n - panel * PANEL);
    tm = within / width;
    tn = panel * PANEL + within - tm * width;
}

// Symmetric problems (A side == B side) only need the tiles that meet the upper triangle j >= i: row tm (bm rows high)
// starts at column tile (tm*bm)/BN.  Same column panels, restricted to those tiles; the decode walks panels and rows
// (a few hundred iterations at most, once per work item of millions of cycles).  Shared by device and host.
__host__ __device__ inline int sym_tile_coords(int tile, int tiles_m, int tiles_n, int bm, int &tm, int &tn) {
    int seen = 0;
    for (int p0 = 0; p0 < tiles_n; p0 += PANEL) {
        const int p1 = (p0 + PANEL < tiles_n) ? p0 + PANEL : tiles_n;
        for (int r = 0; r < tiles_m; r++) {
            const int first = (r * bm) / BN, f = first > p0 ? first : p0;
            if (f >= p1) break;                       // rows further down start right of this panel
            const int cnt = p1 - f;
            if (tile >= 0 && tile < seen + cnt) { tm = r; tn = f + (tile - seen); return seen; }
            seen += cnt;
        }
    }
    return seen;                                      // tile < 0: the number of tiles
}

struct GramArgs {
    float *partials;        // [splits][Mt][Nt] fp32, Mt = tiles_m*BM, Nt = tiles_n*BN
    int tiles_m, tiles_n, splits;
    int n_tiles;            // tiles_m*tiles_n, or the upper-triangle count when sym
    int sym;
    int kblocks;            // ceil(P / BK)
    int kb_per_split;
    long long ld_part;      // Nt
    long long split_stride; // Mt*Nt
};

__device__ __forceinline__ void work_coords(const GramArgs &g, int tile, int bm, int &tm, int &tn) {
    if (g.sym) sym_tile_coords(tile, g.tiles_m, g.tiles_n, bm, tm, tn);
    else tile_coords(tile, g.tiles_m, g.tiles_n, tm, tn);
}

template <int BK, int TERMS>
__global__ void __launch_bounds__(NUM_THREADS, 1)
k_gram(const __grid_constant__ CUtensorMap map_a_hi,   // A side hi, box BM rows x BK
       const __grid_constant__ CUtensorMap map_a_lo,   // A side lo
       const __grid_constant__ CUtensorMap map_b_hi,   // B side hi, box BN rows x BK
       const __grid_constant__ CUtensorMap map_b_lo,   // B side lo
       const GramArgs g) {
    using C = Cfg<BK, TERMS>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // swizzle atoms need 1024-B alignment
    uint64_t *bars = (uint64_t *)(smem + C::STAGES * C::STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + C::STAGES, *acc_full = bars + 2 * C::STAGES, *acc_empty = acc_full + 2;
    uint32_t *tmem_slot = (uint32_t *)(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles = g.n_tiles;
    const int n_work = n_tiles * g.splits;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a_hi);
        tma_prefetch_desc(&map_b_hi);
        if (TERMS > 1) { tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_lo); }
        for (int s = 0; s < C::STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], NUM_EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
                const int split = w / n_tiles, tile = w % n_tiles;      // split-major: concurrent CTAs share a k-range
                int tm, tn;
                work_coords(g, tile, BM, tm, tn);
                const int kb0 = split * g.kb_per_split;
                const int kb1 = min(kb0 + g.kb_per_split, g.kblocks);
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t *st = smem + stage * C::STAGE_BYTES;
                    mbar_expect_tx(&full[stage], C::STAGE_BYTES);
                    tma_load_2d(&map_a_hi, &full[stage], st, kb * BK, tm * BM);
                    tma_load_2d(&map_b_hi, &full[stage], st + C::PLANES * C::A_BYTES, kb * BK, tn * BN);
                    if (TERMS > 1) {
                        tma_load_2d(&map_a_lo, &full[stage], st + C::A_BYTES, kb * BK, tm * BM);
                        tma_load_2d(&map_b_lo, &full[stage], st + 2 * C::A_BYTES + C::B_BYTES, kb * BK, tn * BN);
                    }
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (one thread) =================
        if (lane == 0) {
            constexpr int CH = C::CH;                                 // k-blocks per TMEM accumulation chunk
            constexpr uint32_t IDESC = idesc_bf16(BM, BN);
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
                const int split = w / n_tiles;
                const int kb0 = split * g.kb_per_split;
                const int kb1 = min(kb0 + g.kb_per_split, g.kblocks);
                for (int kb = kb0; kb < kb1; kb++) {
                    const int in_chunk = (kb - kb0) % CH;
                    if (in_chunk == 0) {
                        mbar_wait(&acc_empty[acc], acc_phase ^ 1);    // accumulate warps have drained this stage
                        tc_fence_after();
                    }
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    mbar_wait(&full[stage], phase);                   // TMA bytes have landed
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + stage * C::STAGE_BYTES);
                    const uint64_t ah_desc = desc_sw<C::SBO_BYTES, C::LAYOUT>(a_addr);
                    const uint64_t al_desc = desc_sw<C::SBO_BYTES, C::LAYOUT>(a_addr + C::A_BYTES);
                    const uint64_t bh_desc = desc_sw<C::SBO_BYTES, C::LAYOUT>(a_addr + C::PLANES * C::A_BYTES);
                    const uint64_t bl_desc = desc_sw<C::SBO_BYTES, C::LAYOUT>(a_addr + 2 * C::A_BYTES + C::B_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adv = (uint64_t)((k * UMMA_K * 2) >> 4);   // +32 B along K inside the swizzled row
                        umma_bf16(d_tmem, ah_desc + adv, bh_desc + adv, IDESC, (in_chunk > 0 || k > 0) ? 1u : 0u);
                        if (TERMS > 1) {
                            umma_bf16(d_tmem, ah_desc + adv, bl_desc + adv, IDESC, 1u);
                            umma_bf16(d_tmem, al_desc + adv, bh_desc + adv, IDESC, 1u);
                        }
                    }
                    umma_commit(&empty[stage]);                       // frees the smem stage when the MMAs retire
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    if (in_chunk == CH - 1 || kb == kb1 - 1) {
                        umma_commit(&acc_full[acc]);                  // chunk complete -> accumulate warps
                        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                    }
                }
            }
        }
    } else {
        // ================= accumulate warps: TMEM chunk -> += registers; then -> partial tile =================
        constexpr int CH = C::CH;
        const int q = warp & 3;                                       // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;                             // which 128 columns of the 256-wide tile
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int split = w / n_tiles, tile = w % n_tiles;
            int tm, tn;
            work_coords(g, tile, BM, tm, tn);
            const int kb0 = split * g.kb_per_split;
            const int kb1 = min(kb0 + g.kb_per_split, g.kblocks);
            const int n_chunks = (kb1 - kb0 + CH - 1) / CH;
            float r[128];
#pragma unroll
            for (int j = 0; j < 128; j++) r[j] = 0.f;
            for (int ch = 0; ch < n_chunks; ch++) {
                mbar_wait(&acc_full[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + half * 128);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    uint32_t v[32];
                    tmem_ld_32x32(taddr + (uint32_t)(c * 32), v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j++) r[c * 32 + j] += __uint_as_float(v[j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            const int row = tm * BM + q * 32 + lane;
            float4 *d4 = reinterpret_cast<float4 *>(g.partials + (long long)split * g.split_stride +
                                                    (long long)row * g.ld_part + (long long)tn * BN + half * 128);
#pragma unroll
            for (int j = 0; j < 32; j++) d4[j] = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// =================================================================================================================
// CTA-pair variant (cta_group::2): two CTAs of a cluster share one 256 x 256 output tile.  Each CTA stages its own
// 128 rows of the A-side operand and only HALF (128 rows) of each B-side operand; the pair's tensor cores read the
// other half across the pair.  Per CTA and k-step this cuts the shared-memory operand fetch — what the single-CTA
// kernel is bound by — from A + B to A + B/2, and the smem footprint per stage from 80 KB to 48 KB (4 stages).
//   CTA rank r: A rows tm*256 + r*128, B rows tn*256 + r*128, accumulator rows r*128.. of the tile in its own TMEM.
//   Only the leader (rank 0) issues tcgen05.mma.cta_group::2; both CTAs run a TMA producer whose transactions
//   complete on the LEADER's full barrier; tcgen05.commit multicasts the stage release / accumulator-ready
//   arrivals to both CTAs; the peer's accumulate warps release the accumulator on the leader's barrier (mapa).
// =================================================================================================================
constexpr int BM2 = 256;

template <int BK, int TERMS>
struct Cfg2 {
    static constexpr int ROW_BYTES = BK * 2;
    static constexpr int A_BYTES = BM * ROW_BYTES;            // 128 rows per CTA
    static constexpr int B_BYTES = (BN / 2) * ROW_BYTES;      // half of the 256 B rows per CTA
    static constexpr int PLANES = TERMS > 1 ? 2 : 1;
    static constexpr int STAGE_BYTES = (A_BYTES + B_BYTES) * PLANES;
    static constexpr int STAGES = (200 * 1024) / STAGE_BYTES > 8 ? 8 : (200 * 1024) / STAGE_BYTES;
    static constexpr int CH = chunk_k<TERMS>() / BK;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
};

template <int BK, int TERMS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
k_gram2(const __grid_constant__ CUtensorMap map_a_hi,   // hi of the A side, box 128 rows x BK
        const __grid_constant__ CUtensorMap map_a_lo,   // lo of the A side
        const __grid_constant__ CUtensorMap map_b_hi,   // hi of the B side, box 128 rows x BK
        const __grid_constant__ CUtensorMap map_b_lo,   // lo of the B side
        const GramArgs g) {
    using C = Cfg2<BK, TERMS>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = (uint64_t *)(smem + C::STAGES * C::STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + C::STAGES, *acc_full = bars + 2 * C::STAGES, *acc_empty = acc_full + 2;
    uint32_t *tmem_slot = (uint32_t *)(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_tiles = g.n_tiles;
    const int n_work = n_tiles * g.splits;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a_hi);
        tma_prefetch_desc(&map_b_hi);
        if (TERMS > 1) { tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_lo); }
        for (int s = 0; s < C::STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], 2 * NUM_EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc2(tmem_slot, TMEM_COLS);
    tc_fence_before();
    cluster_sync_all();                                   // barriers of BOTH CTAs are initialised before any remote arrive / TMA
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer (both CTAs: own A rows, own half of the B rows) =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int w = cluster_id; w < n_work; w += n_clusters) {
                const int split = w / n_tiles, tile = w % n_tiles;
                int tm, tn;
                work_coords(g, tile, BM2, tm, tn);
                const int kb0 = split * g.kb_per_split;
                const int kb1 = min(kb0 + g.kb_per_split, g.kblocks);
                const int row_a = tm * BM2 + (int)rank * BM, row_b = tn * BN + (int)rank * (BN / 2);
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t *st = smem + stage * C::STAGE_BYTES;
                    if (rank == 0) mbar_expect_tx(&full[stage], 2 * C::STAGE_BYTES);      // both CTAs' bytes land here
                    tma_load_2d_pair(&map_a_hi, &full[stage], st, kb * BK, row_a);
                    tma_load_2d_pair(&map_b_hi, &full[stage], st + C::PLANES * C::A_BYTES, kb * BK, row_b);
                    if (TERMS > 1) {
                        tma_load_2d_pair(&map_a_lo, &full[stage], st + C::A_BYTES, kb * BK, row_a);
                        tma_load_2d_pair(&map_b_lo, &full[stage], st + 2 * C::A_BYTES + C::B_BYTES, kb * BK, row_b);
                    }
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: one thread of the leader CTA =================
        if (lane == 0 && rank == 0) {
            constexpr int CH = C::CH;
            constexpr uint32_t IDESC = idesc_bf16(BM2, BN);
            using D = Cfg<BK, TERMS>;                                 // a CTA's operand rows have the single-CTA kernel's layout
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int w = cluster_id; w < n_work; w += n_clusters) {
                const int split = w / n_tiles;
                const int kb0 = split * g.kb_per_split;
                const int kb1 = min(kb0 + g.kb_per_split, g.kblocks);
                for (int kb = kb0; kb < kb1; kb++) {
                    const int in_chunk = (kb - kb0) % CH;
                    if (in_chunk == 0) {
                        mbar_wait(&acc_empty[acc], acc_phase ^ 1);    // both CTAs' accumulate warps have drained this stage
                        tc_fence_after();
                    }
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + stage * C::STAGE_BYTES);
                    const uint64_t ah_desc = desc_sw<D::SBO_BYTES, D::LAYOUT>(a_addr);
                    const uint64_t al_desc = desc_sw<D::SBO_BYTES, D::LAYOUT>(a_addr + C::A_BYTES);
                    const uint64_t bh_desc = desc_sw<D::SBO_BYTES, D::LAYOUT>(a_addr + C::PLANES * C::A_BYTES);
                    const uint64_t bl_desc = desc_sw<D::SBO_BYTES, D::LAYOUT>(a_addr + 2 * C::A_BYTES + C::B_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adv = (uint64_t)((k * UMMA_K * 2) >> 4);
                        umma2_bf16(d_tmem, ah_desc + adv, bh_desc + adv, IDESC, (in_chunk > 0 || k > 0) ? 1u : 0u);
                        if (TERMS > 1) {
                            umma2_bf16(d_tmem, ah_desc + adv, bl_desc + adv, IDESC, 1u);
                            umma2_bf16(d_tmem, al_desc + adv, bh_desc + adv, IDESC, 1u);
                        }
                    }
                    umma2_commit_mc(&empty[stage]);                   // frees the stage in both CTAs
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    if (in_chunk == CH - 1 || kb == kb1 - 1) {
                        umma2_commit_mc(&acc_full[acc]);              // chunk complete -> accumulate warps of both CTAs
                        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                    }
                }
            }
        }
    } else {
        // ================= accumulate warps (both CTAs): own 128 rows of the 256 x 256 tile =================
        constexpr int CH = C::CH;
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int w = cluster_id; w < n_work; w += n_clusters) {
            const int split = w / n_tiles, tile = w % n_tiles;
            int tm, tn;
            work_coords(g, tile, BM2, tm, tn);
            const int kb0 = split * g.kb_per_split;
            const int kb1 = min(kb0 + g.kb_per_split, g.kblocks);
            const int n_chunks = (kb1 - kb0 + CH - 1) / CH;
            float r[128];
#pragma unroll
            for (int j = 0; j < 128; j++) r[j] = 0.f;
            for (int ch = 0; ch < n_chunks; ch++) {
                mbar_wait(&acc_full[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + half * 128);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    uint32_t v[32];
                    tmem_ld_32x32(taddr + (uint32_t)(c * 32), v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j++) r[c * 32 + j] += __uint_as_float(v[j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_on_rank(&acc_empty[acc], 0);   // the leader's barrier counts both CTAs' warps
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            const int row = tm * BM2 + (int)rank * BM + q * 32 + lane;
            float4 *d4 = reinterpret_cast<float4 *>(g.partials + (long long)split * g.split_stride +
                                                    (long long)row * g.ld_part + (long long)tn * BN + half * 128);
#pragma unroll
            for (int j = 0; j < 32; j++) d4[j] = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
        }
    }

    tc_fence_before();
    cluster_sync_all();                                   // neither CTA may exit while the pair still touches its smem / TMEM
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc2(tmem_base, TMEM_COLS);
    }
}

// D (P x K column-major, i.e. row k of A contiguous) -> hi[k][p], lo[k][p] bf16 with row pitch Ppad.
// One thread packs 8 consecutive elements: eight coalesced scalar loads (rows of odd length start unaligned), one
// 16-byte store per plane.  HBM-bound: reads the source once, writes 4 bytes per element.
template <typename T>
__global__ void k_gram_pack(const T *__restrict__ A, long long P, long long K, long long Ppad,
                            __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo) {
    const long long k = blockIdx.y;
    const T *row = A + k * P;
    for (long long p8 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; p8 < Ppad; p8 += (long long)gridDim.x * blockDim.x * 8) {
        T a[8];
#pragma unroll
        for (int j = 0; j < 8; j++) a[j] = (p8 + j < P) ? row[p8 + j] : (T)0;
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            __nv_bfloat16 hh[2], ll[2];
#pragma unroll
            for (int e = 0; e < 2; e++) {
                // For fp32 input the remainder a - hi is exact in fp32, so the fp32 path gives the same bits as the fp64
                // one without the emulated double->bf16 conversions.
                if constexpr (sizeof(T) == 4) {
                    const float v = (float)a[2 * j + e];
                    hh[e] = __float2bfloat16_rn(v);
                    ll[e] = __float2bfloat16_rn(v - __bfloat162float(hh[e]));
                } else {
                    const double v = (double)a[2 * j + e];
                    hh[e] = __double2bfloat16(v);
                    ll[e] = __double2bfloat16(v - (double)__bfloat162float(hh[e]));
                }
            }
            h[j] = (uint32_t)__bfloat16_as_ushort(hh[0]) | ((uint32_t)__bfloat16_as_ushort(hh[1]) << 16);
            l[j] = (uint32_t)__bfloat16_as_ushort(ll[0]) | ((uint32_t)__bfloat16_as_ushort(ll[1]) << 16);
        }
        *reinterpret_cast<uint4 *>(hi + k * Ppad + p8) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4 *>(lo + k * Ppad + p8) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// ---- host side -------------------------------------------------------------------------------------
struct Plan {
    long long rows_a, rows_b, P, Ppad, Mt, Nt;
    int tiles_m, tiles_n, n_tiles, sym, splits, kblocks, kb_per_split, bk, pair;
    size_t scratch_bytes;
};

static int g_cta_group = 2;      // 2 = CTA-pair kernel (k_gram2), 1 = single-CTA kernel (k_gram)

static long long pitch_of(long long P) { return (P + 63) / 64 * 64; }

static void make_plan(long long rows_a, long long rows_b, long long P, int bk, int splits_req, Plan *pl, int terms, int sym) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    pl->rows_a = rows_a; pl->rows_b = rows_b; pl->P = P; pl->bk = bk;
    pl->pair = g_cta_group == 2 ? 1 : 0;
    // measured: with plain bf16 (one MMA per k-step) a problem too small to give every CTA pair its own tile
    // runs faster on single-CTA tiles (K=1000: 0.28 vs 0.30 ms); the hi/lo split always prefers the pair
    if (pl->pair && terms == 1 && ((rows_a + BM2 - 1) / BM2) * ((rows_b + BN - 1) / BN) < sms / 2) pl->pair = 0;
    const int bm = pl->pair ? BM2 : BM;
    const int units = pl->pair ? sms / 2 : sms;                 // schedulable units: CTA pairs or CTAs
    pl->Ppad = pitch_of(P);
    pl->tiles_m = (int)((rows_a + bm - 1) / bm);
    pl->tiles_n = (int)((rows_b + BN - 1) / BN);
    pl->Mt = (long long)pl->tiles_m * bm;
    pl->Nt = (long long)pl->tiles_n * BN;
    pl->kblocks = (int)((P + bk - 1) / bk);
    int tm_ = 0, tn_ = 0;
    pl->sym = sym;
    pl->n_tiles = sym ? sym_tile_coords(-1, pl->tiles_m, pl->tiles_n, bm, tm_, tn_) : pl->tiles_m * pl->tiles_n;
    int tiles = pl->n_tiles;
    // split-K fills the machine when there are fewer tiles than CTAs (or pairs): one round of work items, or two when that
    // wastes noticeably fewer slots (measured at K=1000, 10 upper-triangle tiles on 74 pairs: 7 splits 0.441 ms, 14 splits 0.452)
    int splits = splits_req;
    if (splits <= 0) {
        splits = 1;
        if (tiles < units) {
            const int s1 = units / tiles, s2 = (2 * units) / tiles;
            const double e1 = (double)tiles * s1 / units, e2 = (double)tiles * s2 / (2.0 * units);
            splits = e2 > e1 + 0.03 ? s2 : s1;
        }
        // (with more tiles than units, cutting each tile's contraction to shorten the partly empty last round was measured at
        // the 5b block size — 325 tiles on 74 pairs — and changed nothing: those launches run power-limited, time follows the
        // MMA count, idle SMs hand their power to the busy ones)
    }
    if (splits > pl->kblocks) splits = pl->kblocks;
    if (splits > 64) splits = 64;
    pl->kb_per_split = (pl->kblocks + splits - 1) / splits;
    pl->splits = (pl->kblocks + pl->kb_per_split - 1) / pl->kb_per_split;          // no empty split
    pl->scratch_bytes = (size_t)pl->splits * pl->Mt * pl->Nt * 4;
}

template <int BK, int TERMS>
static int launch(const Plan &pl, const void *a_hi, const void *a_lo, const void *b_hi, const void *b_lo, float *scratch,
                  cudaStream_t st) {
    using C = Cfg<BK, TERMS>;
    if (TERMS == 1) { a_lo = a_hi; b_lo = b_hi; }               // the lo maps are never dereferenced then
    const int box_b = pl.pair ? BN / 2 : BN;                     // the pair stages half a B tile per CTA
    auto make_map = [&](CUtensorMap *m, const void *base, long long rows, int box_rows) {      // swizzle matches C::LAYOUT
        return make_map_2d_16bit(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rows, pl.P, pl.Ppad, box_rows, BK,
                                 BK == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
    };
    CUtensorMap mah, mal, mbh, mbl;
    int rc;
    if ((rc = make_map(&mah, a_hi, pl.rows_a, BM)) != SNK_OK) return rc;
    if ((rc = make_map(&mal, a_lo, pl.rows_a, BM)) != SNK_OK) return rc;
    if ((rc = make_map(&mbh, b_hi, pl.rows_b, box_b)) != SNK_OK) return rc;
    if ((rc = make_map(&mbl, b_lo, pl.rows_b, box_b)) != SNK_OK) return rc;
    GramArgs g;
    g.partials = scratch;
    g.tiles_m = pl.tiles_m; g.tiles_n = pl.tiles_n; g.n_tiles = pl.n_tiles; g.sym = pl.sym; g.splits = pl.splits;
    g.kblocks = pl.kblocks; g.kb_per_split = pl.kb_per_split; g.ld_part = pl.Nt; g.split_stride = pl.Mt * pl.Nt;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int n_work = pl.n_tiles * pl.splits;
    if (pl.pair) {
        using C2 = Cfg2<BK, TERMS>;
        int pairs = sms / 2;
        int grid2 = 2 * (n_work < pairs ? n_work : pairs);
        SNK_CUDA(cudaFuncSetAttribute(k_gram2<BK, TERMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, C2::SMEM_BYTES));
        k_gram2<BK, TERMS><<<grid2, NUM_THREADS, C2::SMEM_BYTES, st>>>(mah, mal, mbh, mbl, g);
        SNK_CUDA(cudaGetLastError());
        return SNK_OK;
    }
    int grid = n_work < sms ? n_work : sms;
    SNK_CUDA(cudaFuncSetAttribute(k_gram<BK, TERMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    k_gram<BK, TERMS><<<grid, NUM_THREADS, C::SMEM_BYTES, st>>>(mah, mal, mbh, mbl, g);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

static int run_block(const Plan &pl, int terms, const void *a_hi, const void *a_lo, const void *b_hi, const void *b_lo,
                     float *scratch, cudaStream_t st) {
    if (pl.bk == 64)
        return terms == 1 ? launch<64, 1>(pl, a_hi, a_lo, b_hi, b_lo, scratch, st) : launch<64, 3>(pl, a_hi, a_lo, b_hi, b_lo, scratch, st);
    return terms == 1 ? launch<32, 1>(pl, a_hi, a_lo, b_hi, b_lo, scratch, st) : launch<32, 3>(pl, a_hi, a_lo, b_hi, b_lo, scratch, st);
}

// out[i][j] = sum_s part[s][i][j], the partials summed in split order (deterministic).  sym: only the tiles meeting the upper
// triangle hold data; out[i][j] for j >= i comes from the partials and out[j][i] is the same value — G is exactly symmetric.
__global__ void k_gram_finish(const float *__restrict__ part, int splits, long long split_stride, long long ld_part, int rows_a,
                              int rows_b, float *__restrict__ out, long long ld_out, int sym) {
    __shared__ float tile[32][33];
    const int bi = blockIdx.y * 32, bj = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;          // 32 x 8
    if (sym && bj < bi) return;
    for (int r = ty; r < 32; r += 8) {
        const int i = bi + r, j = bj + tx;
        float acc = 0.f;
        if (i < rows_a && j < rows_b) {
            for (int s = 0; s < splits; s++) acc += part[s * split_stride + (long long)i * ld_part + j];
            if (!sym || j >= i) out[(long long)i * ld_out + j] = acc;
        }
        tile[r][tx] = acc;
    }
    if (!sym) return;
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {                     // the mirror image, written row-wise: out[bj + r][bi + tx]
        const int i = bi + tx, j = bj + r;
        if (i < rows_a && j < rows_b && j > i) out[(long long)j * ld_out + i] = tile[tx][r];
    }
}

// out[i][j] = src[j][i]  (out rows_a x rows_b, src rows_b x rows_a).  src may live in a PEER's memory (row-sharded Gram:
// the blocks this rank did not compute are the transposes of blocks its peers did) — plain coalesced loads over NVLink.
__global__ void k_transpose_block(const float *__restrict__ src, long long ld_src, int rows_a, int rows_b, float *__restrict__ out,
                                  long long ld_out) {
    __shared__ float tile[32][33];
    const int bi = blockIdx.y * 32, bj = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;
    for (int r = ty; r < 32; r += 8) {
        const int j = bj + r, i = bi + tx;
        tile[r][tx] = (j < rows_b && i < rows_a) ? src[(long long)j * ld_src + i] : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int i = bi + r, j = bj + tx;
        if (i < rows_a && j < rows_b) out[(long long)i * ld_out + j] = tile[tx][r];
    }
}

}  // namespace gram
}  // namespace snk

using namespace snk;
using namespace snk::gram;

extern "C" {

int snk_gram_config(int cta_group) {
    SNK_REQUIRE(cta_group == 1 || cta_group == 2, "cta_group must be 1 (single-CTA tiles) or 2 (CTA-pair tiles)");
    g_cta_group = cta_group;
    return SNK_OK;
}

int snk_gram_planes_layout(int64_t rows, int64_t P, size_t *plane_bytes, int64_t *pitch_elems) {
    SNK_REQUIRE(rows > 0 && P > 0, "bad argument");
    if (pitch_elems) *pitch_elems = pitch_of(P);
    if (plane_bytes) *plane_bytes = ((size_t)rows * pitch_of(P) * 2 + 1023) & ~(size_t)1023;
    return SNK_OK;
}

int snk_gram_pack_planes(const void *A, int a_dtype, int64_t P, int64_t rows, void *hi, void *lo, void *cuda_stream) {
    DeviceGuard guard__(device_of(hi));
    SNK_REQUIRE(A != nullptr && hi != nullptr && lo != nullptr && rows > 0 && P > 0, "bad argument");
    SNK_REQUIRE(a_dtype == SNK_DTYPE_F64 || a_dtype == SNK_DTYPE_F32, "a_dtype must be SNK_DTYPE_F64 or SNK_DTYPE_F32");
    const long long Ppad = pitch_of(P);
    dim3 grid((unsigned)((Ppad / 8 + 255) / 256 < 96 ? (Ppad / 8 + 255) / 256 : 96), (unsigned)rows);
    if (a_dtype == SNK_DTYPE_F64)
        k_gram_pack<double><<<grid, 256, 0, (cudaStream_t)cuda_stream>>>((const double *)A, P, rows, Ppad, (__nv_bfloat16 *)hi,
                                                                         (__nv_bfloat16 *)lo);
    else
        k_gram_pack<float><<<grid, 256, 0, (cudaStream_t)cuda_stream>>>((const float *)A, P, rows, Ppad, (__nv_bfloat16 *)hi,
                                                                        (__nv_bfloat16 *)lo);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_gram_block_scratch_bytes(int64_t rows_a, int64_t rows_b, int64_t P, int splits, size_t *bytes) {
    SNK_REQUIRE(bytes != nullptr && rows_a > 0 && rows_b > 0 && P > 0 && splits >= 0, "bad argument");
    size_t best = 0;
    const int saved = g_cta_group;
    for (int cg = 1; cg <= 2; cg++)
        for (int bk = 32; bk <= 64; bk += 32) {
            for (int terms = 1; terms <= 3; terms += 2)
                for (int sym = 0; sym <= (rows_a == rows_b ? 1 : 0); sym++) {
                    Plan p;
                    g_cta_group = cg;
                    make_plan(rows_a, rows_b, P, bk, splits, &p, terms, sym);
                    if (p.scratch_bytes > best) best = p.scratch_bytes;
                }
        }
    g_cta_group = saved;
    *bytes = best;
    return SNK_OK;
}

int snk_gram_block(const void *a_hi, const void *a_lo, int64_t rows_a, const void *b_hi, const void *b_lo, int64_t rows_b, int64_t P,
                   int terms, int symmetric, int block_k, int splits, void *scratch, float *Y, int64_t ldY, void *cuda_stream) {
    DeviceGuard guard__(device_of(scratch));
    SNK_REQUIRE(a_hi && b_hi && scratch && Y && rows_a > 0 && rows_b > 0 && P > 0, "bad argument");
    SNK_REQUIRE(terms == 1 || (terms == 3 && a_lo != nullptr && b_lo != nullptr), "terms must be 1 (bf16) or 3 (hi/lo split, needs both lo planes)");
    SNK_REQUIRE(!symmetric || (a_hi == b_hi && rows_a == rows_b), "symmetric needs the same planes on both sides");
    if (block_k == 0) block_k = 64;
    SNK_REQUIRE(block_k == 32 || block_k == 64, "block_k must be 32 or 64");
    SNK_REQUIRE(ldY >= rows_b, "ldY too small");
    Plan pl;
    make_plan(rows_a, rows_b, P, block_k, splits, &pl, terms, symmetric ? 1 : 0);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int rc = run_block(pl, terms, a_hi, a_lo, b_hi, b_lo, (float *)scratch, st);
    if (rc != SNK_OK) return rc;
    dim3 rb(32, 8), rg((unsigned)((rows_b + 31) / 32), (unsigned)((rows_a + 31) / 32));
    k_gram_finish<<<rg, rb, 0, st>>>((const float *)scratch, pl.splits, pl.Mt * pl.Nt, pl.Nt, (int)rows_a, (int)rows_b, Y, ldY,
                                     pl.sym);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_gram_block_flops(int64_t rows_a, int64_t rows_b, int64_t P, int terms, int symmetric, double *executed) {
    SNK_REQUIRE(executed != nullptr && rows_a > 0 && rows_b > 0 && P > 0 && (terms == 1 || terms == 3), "bad argument");
    SNK_REQUIRE(!symmetric || rows_a == rows_b, "symmetric needs a square block");
    Plan pl;
    make_plan(rows_a, rows_b, P, 64, 1, &pl, terms, symmetric ? 1 : 0);
    // what the tensor pipe executes: every computed tile, padded, times the products per k-step
    *executed = 2.0 * (pl.pair ? BM2 : BM) * BN * (double)pl.Ppad * pl.n_tiles * (terms == 3 ? 3 : 1);
    return SNK_OK;
}

int snk_gram_transpose_block(const float *YT, int64_t ldYT, int64_t rows_a, int64_t rows_b, float *G, int64_t ldG, void *cuda_stream) {
    DeviceGuard guard__(device_of(G));
    SNK_REQUIRE(YT && G && rows_a > 0 && rows_b > 0 && ldYT >= rows_a && ldG >= rows_b, "bad argument");
    dim3 rb(32, 8), rg((unsigned)((rows_b + 31) / 32), (unsigned)((rows_a + 31) / 32));
    k_transpose_block<<<rg, rb, 0, (cudaStream_t)cuda_stream>>>(YT, ldYT, (int)rows_a, (int)rows_b, G, ldG);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

// ---- single-GPU convenience: workspace = [hi | lo | scratch] ---------------------------------------
int snk_gram_workspace_bytes(int64_t K, int64_t P, int splits, size_t *bytes) {
    SNK_REQUIRE(bytes != nullptr && K > 0 && P > 0 && splits >= 0, "bad argument");
    size_t plane = 0, scratch = 0;
    snk_gram_planes_layout(K, P, &plane, nullptr);
    snk_gram_block_scratch_bytes(K, K, P, splits, &scratch);
    *bytes = 2 * plane + scratch;
    return SNK_OK;
}

int snk_gram_pack(const void *A, int a_dtype, int64_t P, int64_t K, void *workspace, void *cuda_stream) {
    SNK_REQUIRE(workspace != nullptr && K > 0 && P > 0, "bad argument");
    size_t plane = 0;
    snk_gram_planes_layout(K, P, &plane, nullptr);
    return snk_gram_pack_planes(A, a_dtype, P, K, workspace, (uint8_t *)workspace + plane, cuda_stream);
}

int snk_gram(const void *workspace, int64_t P, int64_t K, int terms, int block_k, int splits, float *G, void *cuda_stream) {
    DeviceGuard guard__(device_of(workspace));
    SNK_REQUIRE(workspace != nullptr && G != nullptr && K > 0 && P > 0, "bad argument");
    SNK_REQUIRE(terms == 1 || terms == 3, "terms must be 1 (bf16) or 3 (bf16 hi/lo split)");
    if (block_k == 0) block_k = 64;
    SNK_REQUIRE(block_k == 32 || block_k == 64, "block_k must be 32 or 64");
    size_t plane = 0;
    snk_gram_planes_layout(K, P, &plane, nullptr);
    const uint8_t *ws = (const uint8_t *)workspace;
    float *scratch = (float *)(ws + 2 * plane);
    Plan pl;
    make_plan(K, K, P, block_k, splits, &pl, terms, 1);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int rc = run_block(pl, terms, ws, ws + plane, ws, ws + plane, scratch, st);
    if (rc != SNK_OK) return rc;
    // G = sum of the split partials of the upper-triangle tiles, mirrored into the lower triangle
    dim3 rb(32, 8), rg((unsigned)((K + 31) / 32), (unsigned)((K + 31) / 32));
    k_gram_finish<<<rg, rb, 0, st>>>(scratch, pl.splits, pl.Mt * pl.Nt, pl.Nt, (int)K, (int)K, G, K, 1);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

// ---- peer-memory plumbing for the row-sharded Gram (one process per GPU) ---------------------------
int snk_ipc_alloc(void **p, size_t bytes) {
    SNK_REQUIRE(p != nullptr && bytes > 0, "bad argument");
    SNK_CUDA(cudaMalloc(p, bytes));
    return SNK_OK;
}
int snk_ipc_free(void *p) {
    if (p) SNK_CUDA(cudaFree(p));
    return SNK_OK;
}
int snk_ipc_export(void *p, uint8_t *handle64) {
    SNK_REQUIRE(p != nullptr && handle64 != nullptr, "bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    SNK_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(handle64, &h, 64);
    return SNK_OK;
}
int snk_ipc_import(const uint8_t *handle64, void **p) {
    SNK_REQUIRE(p != nullptr && handle64 != nullptr, "bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    SNK_CUDA(cudaIpcOpenMemHandle(p, h, cudaIpcMemLazyEnablePeerAccess));
    return SNK_OK;
}
int snk_ipc_close(void *p) {
    if (p) SNK_CUDA(cudaIpcCloseMemHandle(p));
    return SNK_OK;
}
int snk_copy_async(void *dst, const void *src, size_t bytes, void *cuda_stream) {
    SNK_REQUIRE(dst != nullptr && src != nullptr, "bad argument");
    SNK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)cuda_stream));
    return SNK_OK;
}

}  // extern "C"

// sm100.h — the sm_100a synchronisation, asynchronous-copy and tensor-core (tcgen05) primitives of the library's kernels,
// and the host-side tensor-map builder their TMA loads use.  Header-only; every PTX string is written here once.
#pragma once
#include <cuda.h>

#include "common.h"

namespace snk {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrives on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_on_rank(uint64_t *bar, uint32_t rank) {
    asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
                 ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred P1;\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\tselp.b32 %0, 1, 0, P1;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must fault (trap) after ~2 s, never hang the GPU.
constexpr long long MBAR_TIMEOUT_CYCLES = 4000000000ll;
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > MBAR_TIMEOUT_CYCLES) {
            printf("snk: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}
// the same for a wait that is known to be long (an epilogue warp waiting for a whole MMA phase): back off between polls so
// that a dozen polling warps do not compete with the tensor core's operand fetch for the shared-memory pipeline
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(128);
        if (clock64() - t0 > MBAR_TIMEOUT_CYCLES) {
            printf("snk: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
        }
    }
}

// ---- fences and barriers -----------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// named barrier `id` over `n` threads (a multiple of 32)
__device__ __forceinline__ void nbar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nbar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.b32 %0, 1, 0, P1;\n\t}" : "=r"(p));
    return p != 0;
}

// ---- asynchronous copies -----------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(const CUtensorMap *map, uint64_t *bar, void *dst, int c_inner, int c_row) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_row) : "memory");
}
// CTA-pair form: the transaction bytes are credited to the LEADER CTA's barrier (peer bit of the shared::cluster address cleared)
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap *map, uint64_t *leader_bar, void *dst, int c_inner, int c_row) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(leader_bar) & 0xFEFFFFFFu), "r"(c_inner), "r"(c_row) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}
__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"((uint64_t)src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- tcgen05: tensor memory and MMA --------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t *dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T ; both operands K-major
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// CTA-pair MMA, issued by the leader CTA
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the mbarrier once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// the same for CTA-pair MMAs: arrives on this barrier in BOTH CTAs of the pair
__device__ __forceinline__ void umma2_commit_mc(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint4 &lo, const uint4 &hi) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- descriptors (cute::UMMA::SmemDescriptor / InstrDescriptor bit layouts) -----------------------------------------
// no-swizzle K-major operand descriptor: core matrix = 8 rows x 16 B; LBO = byte distance between the two 8-element
// K chunks of one K=16 MMA, SBO = byte distance between 8-row groups (layout_type 0)
__device__ __forceinline__ uint64_t desc_nosw(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// swizzled K-major operand descriptor:
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (1: unused for swizzled K-major)
//   [32,46) stride byte offset >> 4 (SBO_BYTES: pitch between 8-row swizzle atoms) | [46,48) version = 1 | [61,64) layout
// SBO and the layout are template arguments: as runtime arguments they changed the code ptxas made for the kernels.
constexpr uint64_t LAYOUT_SW128 = 2, LAYOUT_SW64 = 4;
template <uint32_t SBO_BYTES, uint64_t LAYOUT>
__device__ __forceinline__ uint64_t desc_sw(uint32_t addr) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(SBO_BYTES >> 4) << 32) | (1ull << 46) | (LAYOUT << 61);
}
// instruction descriptors: FP32 accumulator, both operands K-major, M x N; bf16 x bf16 or fp16 x fp16
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) {      // a_format = b_format = 0 (F16)
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- host: TMA tensor maps -----------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled is reached through the runtime's driver entry point, so the library does not link -lcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline int tensor_map_encoder(EncodeTiledFn *out) {
    static EncodeTiledFn cached = nullptr;
    if (cached == nullptr) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        SNK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || p == nullptr)
            return fail(SNK_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
        cached = (EncodeTiledFn)p;
    }
    *out = cached;
    return SNK_OK;
}

// 2-D map over a row-major matrix of 16-bit elements (`dtype` BFLOAT16 or FLOAT16), rows `pitch_elems` apart; one TMA
// load fetches a box of box_rows x box_cols elements
inline int make_map_2d_16bit(CUtensorMap *m, CUtensorMapDataType dtype, const void *base, long long rows, long long cols,
                             long long pitch_elems, int box_rows, int box_cols, CUtensorMapSwizzle swizzle) {
    EncodeTiledFn enc = nullptr;
    int rc = tensor_map_encoder(&enc);
    if (rc != SNK_OK) return rc;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};          // innermost first
    cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, dtype, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SNK_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return SNK_OK;
}

}  // namespace snk

// gemm_tc.cuh -- tcgen05 / TMEM / TMA / mbarrier PTX wrappers, the split-operand plane formats and the tensor-map helpers shared by
// the tensor-core kernels of libmorl_b200.so (gemm_planes.cu, qhead_envelope.cu).  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace morl {

// ---- PTX wrappers -------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t g_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void g_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(g_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void g_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(g_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void g_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(g_smem_u32(bar)) : "memory");
}
// Bounded spin: a protocol bug becomes a trap (launch error) instead of a hung GPU.
__device__ __forceinline__ void g_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    for (uint32_t it = 0; it < (1u << 26); ++it) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.b32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(g_smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(g_smem_u32(dst)),
        "l"(map), "r"(g_smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// ---- CTA-pair (cta_group::2) flavours: the pair's TMA loads signal the LEADER's (cluster rank 0) mbarrier, the leader's MMA
// commit is multicast to the same barrier offset in both CTAs, the peer's epilogue releases the accumulator remotely ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank0(uint32_t smem_addr) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(smem_addr));
    return r;
}
__device__ __forceinline__ void tma_load_3d_pair(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            g_smem_u32(dst)),
        "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// same, with an L2 eviction-priority hint (createpolicy): activations are read once (evict_first), weight planes by every tile (evict_last)
__device__ __forceinline__ void tma_load_3d_pair_hint(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, int c2, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(
            g_smem_u32(dst)),
        "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
        : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(g_smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(g_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr));
}
// one column of a warp's 32 TMEM lanes (waits for the load)
__device__ __forceinline__ uint32_t tc_ld1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n\ttcgen05.wait::ld.sync.aligned;" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- operand formats ------------------------------------------------------------------------------------------------------
template <int FMT>
struct PlaneFmt;

template <>
struct PlaneFmt<MORL_FMT_BF16X3> {
    static constexpr int P = 3, NPROD = 6;
    static constexpr int BK = 32;                                  // 16-bit elements per K-major stage row (64-byte swizzle)
    static constexpr uint32_t kIdescAB = (1u << 7) | (1u << 10);   // instruction descriptor: a_format = b_format = BF16
    static constexpr uint32_t kOnes2 = 0x3F803F80u;                // two packed 1.0
    static constexpr int kStages1 = 2, kStages2 = 3, kStagesMn = 3;
    // small terms first: A2B0, A0B2, A1B1, A1B0, A0B1, A0B0
    __device__ static constexpr int pa(int t) { return t == 0 ? 2 : (t == 2 || t == 3) ? 1 : 0; }
    __device__ static constexpr int pb(int t) { return t == 1 ? 2 : (t == 2 || t == 4) ? 1 : 0; }
    // (a, b) -> P words, word p = plane p of a (low half) and b (high half)
    __device__ __forceinline__ static void split2(float a, float b, uint32_t (&w)[3], float&) {
        const __nv_bfloat16 a0 = __float2bfloat16_rn(a), b0 = __float2bfloat16_rn(b);
        const float ra = a - __bfloat162float(a0), rb = b - __bfloat162float(b0);
        const __nv_bfloat16 a1 = __float2bfloat16_rn(ra), b1 = __float2bfloat16_rn(rb);
        const float sa = ra - __bfloat162float(a1), sb = rb - __bfloat162float(b1);
        const __nv_bfloat16 a2 = __float2bfloat16_rn(sa), b2 = __float2bfloat16_rn(sb);
        w[0] = (uint32_t)__bfloat16_as_ushort(a0) | ((uint32_t)__bfloat16_as_ushort(b0) << 16);
        w[1] = (uint32_t)__bfloat16_as_ushort(a1) | ((uint32_t)__bfloat16_as_ushort(b1) << 16);
        w[2] = (uint32_t)__bfloat16_as_ushort(a2) | ((uint32_t)__bfloat16_as_ushort(b2) << 16);
    }
    __device__ __forceinline__ static void split1(float a, uint16_t (&h)[3], float&) {
        const __nv_bfloat16 a0 = __float2bfloat16_rn(a);
        const float ra = a - __bfloat162float(a0);
        const __nv_bfloat16 a1 = __float2bfloat16_rn(ra);
        const __nv_bfloat16 a2 = __float2bfloat16_rn(ra - __bfloat162float(a1));
        h[0] = __bfloat16_as_ushort(a0); h[1] = __bfloat16_as_ushort(a1); h[2] = __bfloat16_as_ushort(a2);
    }
    __device__ __forceinline__ static void add8(float (&acc)[8], const uint4 v) {  // += eight packed elements of one plane
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            acc[2 * q] += __uint_as_float(w[q] << 16);
            acc[2 * q + 1] += __uint_as_float(w[q] & 0xFFFF0000u);
        }
    }
};

template <>
struct PlaneFmt<MORL_FMT_F16X2> {
    static constexpr int P = 2, NPROD = 3;
    static constexpr int BK = 64;                                  // 128-byte swizzle rows
    static constexpr uint32_t kIdescAB = 0u;                       // a_format = b_format = F16
    static constexpr uint32_t kOnes2 = 0x3C003C00u;
    static constexpr int kStages1 = 2, kStages2 = 3, kStagesMn = 4;
    // small terms first: A1B0, A0B1, A0B0
    __device__ static constexpr int pa(int t) { return t == 0 ? 1 : 0; }
    __device__ static constexpr int pb(int t) { return t == 1 ? 1 : 0; }
    // `amax` tracks max |a| of the (already scaled) values, for the fp16-range check
    __device__ __forceinline__ static void split2(float a, float b, uint32_t (&w)[2], float& amax) {
        amax = fmaxf(amax, fmaxf(fabsf(a), fabsf(b)));
        const __half2 h0 = __floats2half2_rn(a, b);
        const float2 f0 = __half22float2(h0);
        const __half2 h1 = __floats2half2_rn(a - f0.x, b - f0.y);
        w[0] = *reinterpret_cast<const uint32_t*>(&h0);
        w[1] = *reinterpret_cast<const uint32_t*>(&h1);
    }
    __device__ __forceinline__ static void split1(float a, uint16_t (&h)[2], float& amax) {
        amax = fmaxf(amax, fabsf(a));
        const __half h0 = __float2half_rn(a);
        const __half h1 = __float2half_rn(a - __half2float(h0));
        h[0] = __half_as_ushort(h0); h[1] = __half_as_ushort(h1);
    }
    __device__ __forceinline__ static void add8(float (&acc)[8], const uint4 v) {
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
            acc[2 * q] += f.x;
            acc[2 * q + 1] += f.y;
        }
    }
};

__device__ __forceinline__ float ld_scale(const float* p) { return p ? __ldg(p) : 1.0f; }

// Shared-memory matrix descriptor, K-major canonical layout (cute::UMMA::SmemDescriptor, version 1) with ROWB-byte rows = the swizzle
// span (64 B -> SWIZZLE_64B, 128 B -> SWIZZLE_128B); 8-row groups are contiguous: SBO = 8 * ROWB; LBO unused (1).  A K step of 16
// elements inside the swizzle span is a +32 B advance of the start address.
template <int ROWB>
__device__ __forceinline__ uint64_t make_desc_k(uint32_t smem_addr) {
    static_assert(ROWB == 64 || ROWB == 128, "swizzle span");
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);        // start address, 16-byte units
    d |= (uint64_t)1 << 16;                            // leading byte offset (ignored for swizzled K-major), 16-byte units
    d |= (uint64_t)((8 * ROWB) >> 4) << 32;            // stride byte offset: 8 rows x ROWB
    d |= (uint64_t)1 << 46;                            // descriptor version (Blackwell)
    d |= (uint64_t)(ROWB == 64 ? 4 : 2) << 61;         // layout type: SWIZZLE_64B = 4, SWIZZLE_128B = 2
    return d;
}

// ---- host side: tensor maps through the driver entry point (no link-time dependency on libcuda) ----------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            (void)cudaGetLastError();
    }
    return fn;
}

static inline int fmt_planes(int fmt) { return fmt == MORL_FMT_F16X2 ? 2 : 3; }
static inline CUtensorMapDataType fmt_tm_type(int fmt) { return fmt == MORL_FMT_F16X2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16; }

// [P][rows][K] plane tensor, box = P x box_rows x box_k elements, swizzle span = box_k * 2 bytes (64 or 128)
static inline int make_plane_map(CUtensorMap* map, int fmt, const void* base, int rows, int K, long long plane_stride_elems, int box_rows, int box_k) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return -1;
    const cuuint32_t P = (cuuint32_t)fmt_planes(fmt);
    const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, P};
    const cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)plane_stride_elems * 2};
    const cuuint32_t box[3] = {(cuuint32_t)box_k, (cuuint32_t)box_rows, P};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(map, fmt_tm_type(fmt), 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           box_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)r;
}

}  // namespace morl

// gemm_planes.cu -- FP32-accurate dense layers on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
// Replaces the cuBLAS SIMT sgemm calls behind the reference's nn.Linear layers (common/networks.py:10-48, called from
// multi_policy/envelope/envelope.py:59-77, 300, 420, 429) on the 65,536-row effective batch.  The 1e-5 parity bar rules out
// plain TF32/BF16/FP16, so every fp32 operand is carried as a small number of 16-bit PLANES whose sum reproduces it, and a product
// A.B^T is the sum of the significant plane-by-plane tensor-core MMAs, accumulated in fp32 in tensor memory.  Two operand formats:
//
//   MORL_FMT_F16X2  (default of the update path)   s x = h0 + h1: two fp16 planes (11 + 11 significand bits) of the operand scaled
//       by a power of two s (device-resident, per tensor) -- exact to 2^-22 relative; THREE MMAs  A1B0 + A0B1 + A0B0  per product
//       (the dropped A1B1 term is O(2^-22)), 4 bytes per element.  Each fp16 x fp16 product is exact in fp32.  fp16 has 5 exponent
//       bits: |s x| must stay below 65,504 (an overflow becomes Inf/NaN downstream AND raises a device flag, morl_plane_overflow_count),
//       elements below 2^-14 / s lose relative (not absolute) accuracy -- the scales are chosen so that this floor sits >= 2^-26 below
//       the typical magnitude (DESIGN.md section 4.6).
//   MORL_FMT_BF16X3 (wide-range format)            x = x0 + x1 + x2: three bf16 planes (8 + 8 + 8 bits, fp32 exponent range, no scale),
//       exact to 2^-24; SIX MMAs  A2B0 + A0B2 + A1B1 + A1B0 + A0B1 + A0B0, 6 bytes per element.
// Either way the result differs from an fp32 GEMM only at the level of its own accumulation-order noise (tests/test_gemm_gpu.py).
//
// K-major kernel anatomy (persistent, one CTA per SM -- or one CTA PAIR per TPC with tcgen05 cta_group::2 --, 320 threads):
//   warp 0   : TMA producer   -- cp.async.bulk.tensor.3d of a [P planes x 128 rows x BK] A box and a [P x BN x BK] B box per stage
//              (f16x2: BK = 64, 128-byte swizzle, 3 x 64 KB stages; bf16x3: BK = 32, 64-byte swizzle, 3 x 48 KB stages), mbarrier ring;
//   warp 1   : MMA issuer     -- one elected thread issues NPROD x BK/16 tcgen05.mma.kind::f16 (M=128/256, N=BN, K=16) per stage and
//              commits the stage back to the producer; accumulators live in TMEM (2 x BN columns, double buffered);
//   warps 2-9: epilogue       -- tcgen05.ld (32 lanes x 32 columns per warp-instruction), x 2^-(sA+sB), + bias, ReLU / ReLU-mask, then
//              an fp32 row-major store and/or a re-split into planes (the operand format of the next layer) through a TMA store, so
//              intermediate activations never exist in fp32 in HBM.
// Operands: A [P][M][K] (K-major), B [P][N_pad][K] (K-major), K % BK == 0, N_pad % 32 == 0, N_pad <= 256.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "gemm_tc.cuh"

namespace morl {

constexpr int kGemmBM = 128;
constexpr int kGemmThreads = 320;  // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two warps per TMEM lane quadrant)

__device__ unsigned int g_plane_overflow;  // number of kernel launches (approx.) that saw an f16x2 element out of fp16 range


// |scaled value| beyond the largest finite fp16: the planes hold Inf / NaN from here on (they propagate to the loss) and the flag says why
__device__ __forceinline__ void note_overflow(float amax) {
    if (amax > 65504.f) atomicAdd(&g_plane_overflow, 1u);
}

#define MORL_DISPATCH_FMT(F_, ...)                                                         \
    switch (F_) {                                                                          \
        case MORL_FMT_BF16X3: { constexpr int kFmt = MORL_FMT_BF16X3; __VA_ARGS__; } break; \
        case MORL_FMT_F16X2: { constexpr int kFmt = MORL_FMT_F16X2; __VA_ARGS__; } break;   \
        default: break;                                                                    \
    }


struct GemmArgs {
    int M, N, N_pad, K;          // N_pad = B rows covered by the tensor map box (multiple of 16, <= 256)
    const float* bias;           // [N] or nullptr
    float* c_f32;                // [M, ldc] or nullptr
    int ldc;
    void* c_planes;              // [P][M][ldp] or nullptr (re-split output: operand of the next layer)
    int ldp;                     // columns of a plane row (>= N, multiple of 32; columns [N, ldp) are written as zero)
    long long plane_stride;      // elements between planes
    const uint16_t* mask;        // plane 0 of the forward activation [M][ld_mask] for the ReLU-backward mask, or nullptr
    int ld_mask;
    const uint32_t* bits_in;     // ReLU-backward mask as BITS [M][8] words (see morl_b200.h "ReLU bit masks"), or nullptr
    uint32_t* bits_out;          // forward: bit = (output > 0) per column, same layout, or nullptr
    int n_stages;                // depth of the TMA ring: as many (A box + B box) stages as fit (3 at N_pad = 256, more for narrow outputs)
    uint32_t b_stage;            // bytes of one B stage slot (the B box rounded up to 1 KB)
    int relu;
    const float* a_scale;        // device scalars (powers of two) the A / B planes were scaled by; nullptr = 1
    const float* b_scale;
    const float* c_scale;        // scale applied to the output before it is re-split into c_planes; nullptr = 1
    int l2_hint;                 // L2 eviction hints on the operand loads (MORL_GEMM_L2HINT=1, default off): A evict_first, B evict_last
    int skip_b;                  // TIMING EXPERIMENT ONLY (MORL_GEMM_SKIPB=1, wrong results): B boxes are loaded for the first tile of a CTA only
    int pdl;                     // launched with programmatic stream serialisation: overlap this grid's prologue with the predecessor's tail
    int reverse;                 // walk the row tiles from the last to the first (see morl_gemm_planes_f32: L2 reuse between chained layers)
    unsigned long long* stats;   // diagnostics (MORL_GEMM_STATS=1), else nullptr: [0] MMA wait-on-TMA cycles, [1] MMA wait-on-epilogue,
                                 // [2] MMA loop total, [3] producer wait-on-free-stage, [4] epilogue wait-on-accumulator, [5] epilogue busy
};

__device__ unsigned long long g_gemm_stats[8];

// shared-memory plan of the K-major kernel (host and device agree through these)
template <int NCTA, int FMT>
struct KPlan {
    using F = PlaneFmt<FMT>;
    static constexpr int kStages = NCTA == 2 ? F::kStages2 : F::kStages1;  // ring depth at N_pad = 256
    static constexpr int kMaxStages = 8;                                          // barrier slots (narrow outputs run a deeper ring)
    static constexpr uint32_t kRowB = F::BK * 2;                                  // bytes per staged row = swizzle span
    static constexpr uint32_t kAStage = F::P * kGemmBM * kRowB;                   // A box bytes
    static constexpr uint32_t kBStage = F::P * (256 / NCTA) * kRowB;              // B box bytes at N_pad = 256
    static constexpr uint32_t kStageC = F::P * 2048;                              // per-epilogue-warp TMA-store tile: P x 32 rows x 64 B
    static constexpr uint32_t kOffB = kStages * kAStage;
    static constexpr uint32_t kOffC = kOffB + kStages * kBStage;                  // 1024-aligned (all stage sizes are multiples of 1 KB)
    static constexpr uint32_t kOffBar = kOffC + 8 * kStageC;
    static constexpr uint32_t kOffBias = kOffBar + 256;
    static constexpr uint32_t kBytes = kOffBias + 1024 + 1024;                    // + alignment slack of the dynamic segment
};

// NCTA = 1: one CTA per 128-row tile.  NCTA = 2: a CTA pair (cluster of 2 on one TPC) per 256-row tile, tcgen05 cta_group::2 --
// each CTA stages its own 128 A rows and HALF of the B (weight) rows, the pair's tensor cores read both halves, so the L2 -> smem
// traffic of the weight planes is halved.
// SPLIT = 1 ("split accumulators"): the tensor cores accumulate in fp32 with TRUNCATION (round toward zero) at every MMA, a bias of
// about -0.5 ulp of the running sum per instruction; with all NPROD x K/16 products in one accumulator that is ~2e-6 (f16x2) to ~4e-6
// (bf16x3) of systematic shrinkage per layer at K = 256 (measured: scripts/gemm_error_probe.py).  In split mode the LEADING products
// A0B0 go to accumulator 0 and the correction products (2^-11 / 2^-8 of the magnitude) to accumulator 1, so only K/16 truncations happen
// at full magnitude; the epilogue adds the two with one correctly rounded fp32 add.  Cost: the two TMEM buffers no longer double-buffer
// the accumulator, so the epilogue of a tile does not overlap the MMAs of the next one (the TMA ring still runs ahead).
template <int NCTA, int FMT, int SPLIT>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_planes_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmBh,
                   const __grid_constant__ CUtensorMap tmC, const GemmArgs g) {
    using F = PlaneFmt<FMT>;
    using L = KPlan<NCTA, FMT>;
    constexpr int P = F::P;
    constexpr int BK = F::BK;
    constexpr int kMaxStages = L::kMaxStages;
    constexpr uint32_t ROWB = L::kRowB;
    const int kStages = g.n_stages;  // runtime: narrow B boxes leave room for a deeper ring (host: plan_stages)
    extern __shared__ uint8_t gsmem_raw[];
    // 1 KB alignment by pointer arithmetic ON the shared array (not through an integer cast), so that the compiler keeps every derived
    // pointer in the shared address space: through the cast the bias / staging accesses were generic LD.E / ST.E (long-scoreboard stalls)
    uint8_t* gsmem = gsmem_raw + ((1024u - (g_smem_u32(gsmem_raw) & 1023u)) & 1023u);
    const int BN = g.N_pad;
    constexpr uint32_t a_stage_bytes = L::kAStage;
    const uint32_t b_stage_stride = g.b_stage;
    uint8_t* smA = gsmem;
    uint8_t* smB = gsmem + (uint32_t)kStages * a_stage_bytes;  // (n_stages * (A + B) <= kOffC, checked on the host)
    uint8_t* stage_c = gsmem + L::kOffC;  // per-epilogue-warp staging tiles for the TMA store of the re-split activations
    uint64_t* full = reinterpret_cast<uint64_t*>(gsmem + L::kOffBar);
    uint64_t* empty = full + kMaxStages;
    uint64_t* tfull = empty + kMaxStages;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* bias_s = reinterpret_cast<float*>(gsmem + L::kOffBias);  // [256]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = NCTA == 2 ? cluster_ctarank() : 0u;
    const int unit = blockIdx.x / NCTA, n_units = gridDim.x / NCTA;  // a unit = one CTA (NCTA = 1) or one CTA pair
    const int n_tiles = (g.M + kGemmBM * NCTA - 1) / (kGemmBM * NCTA);
    const int n_kblk = g.K / BK;
    // Work units.  A static round-robin over `n_units` workers leaves a tail of L = n_tiles % n_units tiles that costs a whole
    // extra round (65,536 rows: 256 pair tiles on 74 pairs = 3.46 -> 4 rounds).  When 2L <= n_units the tail tiles are split into
    // two half-width (N/2) units each, so the tail costs half a round.  All three roles enumerate the same sequence.
    const int full_units = (n_tiles / n_units) * n_units;
    const int tail = n_tiles - full_units;
    const bool split_tail = NCTA == 2 && tail > 0 && 2 * tail <= n_units && (BN % 64) == 0;
    const int n_work = split_tail ? full_units + 2 * tail : n_tiles;
    auto unit_of = [&](int u, int& tile, int& n_begin, int& n_cnt) {
        if (!split_tail || u < full_units) {
            tile = u; n_begin = 0; n_cnt = BN;
        } else {
            const int r = u - full_units;
            tile = full_units + (r >> 1); n_cnt = BN >> 1; n_begin = (r & 1) * n_cnt;
        }
        if (g.reverse) tile = n_tiles - 1 - tile;
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            g_mbar_init(&full[s], 1);
            g_mbar_init(&empty[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            g_mbar_init(&tfull[s], 1);
            g_mbar_init(&tempty[s], 8 * NCTA);  // one arrival per epilogue warp (of both CTAs of a pair, on the leader's barrier)
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: 512 columns (two BN-column accumulators); in a pair both CTAs' warp 1 execute the paired allocation
        if (NCTA == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(g_smem_u32(tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(g_smem_u32(tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    if (g.pdl) {
        // programmatic dependent launch: this grid may have become resident (barrier init, TMEM allocation above) while the previous kernel
        // of the stream was still draining its last tiles; let OUR successor do the same, then wait until the predecessor's results are
        // visible -- nothing above this line reads global memory, everything below may
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    for (int t = threadIdx.x; t < 256; t += blockDim.x) bias_s[t] = (g.bias && t < g.N) ? g.bias[t] : 0.f;
    tc_fence_before();
    __syncthreads();
    if (NCTA == 2) cluster_sync_all();  // the peer's barriers are initialised before any remote arrive / complete_tx
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
            uint32_t stage = 0, phase = 0;
            long long w_empty = 0;
            const uint64_t pol_a = l2_policy_evict_first(), pol_b = l2_policy_evict_last();
            for (int u = unit; u < n_work; u += n_units) {
                int tile, n_begin, n_cnt;
                unit_of(u, tile, n_begin, n_cnt);
                const int row0 = (tile * NCTA + (int)cta_rank) * kGemmBM;
                const int b_rows = n_cnt / NCTA;  // B rows this CTA stages for the unit
                for (int kb = 0; kb < n_kblk; ++kb) {
                    const long long c0 = g.stats ? clock64() : 0;
                    g_mbar_wait(&empty[stage], phase ^ 1u);
                    if (g.stats) w_empty += clock64() - c0;
                    if (NCTA == 2) {
                        const bool load_b = !(g.skip_b && u != unit);
                        // one expect_tx (leader) covers the four boxes of the pair; every box completes on the leader's barrier
                        if (cta_rank == 0) g_mbar_expect_tx(&full[stage], 2u * (a_stage_bytes + (load_b ? (uint32_t)P * (uint32_t)b_rows * ROWB : 0u)));
                        const uint32_t lbar = mapa_rank0(g_smem_u32(&full[stage]));
                        if (!load_b) {
                            tma_load_3d_pair(smA + stage * a_stage_bytes, &tmA, lbar, kb * BK, row0, 0);
                        } else if (g.l2_hint) {
                            tma_load_3d_pair_hint(smA + stage * a_stage_bytes, &tmA, lbar, kb * BK, row0, 0, pol_a);
                            tma_load_3d_pair_hint(smB + stage * b_stage_stride, n_cnt == BN ? &tmB : &tmBh, lbar, kb * BK,
                                                  n_begin + (int)cta_rank * b_rows, 0, pol_b);
                        } else {
                            tma_load_3d_pair(smA + stage * a_stage_bytes, &tmA, lbar, kb * BK, row0, 0);
                            tma_load_3d_pair(smB + stage * b_stage_stride, n_cnt == BN ? &tmB : &tmBh, lbar, kb * BK,
                                             n_begin + (int)cta_rank * b_rows, 0);
                        }
                    } else {
                        g_mbar_expect_tx(&full[stage], a_stage_bytes + (uint32_t)P * (uint32_t)BN * ROWB);
                        tma_load_3d(smA + stage * a_stage_bytes, &tmA, &full[stage], kb * BK, row0, 0);
                        tma_load_3d(smB + stage * b_stage_stride, &tmB, &full[stage], kb * BK, 0, 0);
                    }
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
            if (g.stats) atomicAdd(&g.stats[3], (unsigned long long)w_empty);
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0 && cta_rank == 0) {  // in a pair only the leader issues; its MMAs drive both CTAs' tensor cores
            // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A/B format of the plane type, K-major both, N, M=128 (256 per pair)
            constexpr uint32_t a_plane = kGemmBM * ROWB;
            uint32_t stage = 0, phase = 0, it = 0;
            long long w_full = 0, w_tempty = 0;
            const long long t_begin = g.stats ? clock64() : 0;
            for (int u = unit; u < n_work; u += n_units, ++it) {
                int tile, n_begin, n_cnt;
                unit_of(u, tile, n_begin, n_cnt);
                const uint32_t idesc = (1u << 4) | F::kIdescAB | ((uint32_t)(n_cnt >> 3) << 17) | ((uint32_t)((kGemmBM * NCTA) >> 4) << 24);
                const uint32_t b_plane = (uint32_t)(n_cnt / NCTA) * ROWB;
                const uint32_t as = SPLIT ? 0u : (it & 1u);
                long long c0 = g.stats ? clock64() : 0;
                g_mbar_wait(&tempty[as], SPLIT ? ((it & 1u) ^ 1u) : (((it >> 1) & 1u) ^ 1u));
                if (g.stats) w_tempty += clock64() - c0;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + as * 256u;
                for (int kb = 0; kb < n_kblk; ++kb) {
                    c0 = g.stats ? clock64() : 0;
                    g_mbar_wait(&full[stage], phase);
                    if (g.stats) w_full += clock64() - c0;
                    tc_fence_after();
                    const uint32_t a0 = g_smem_u32(smA + stage * a_stage_bytes);
                    const uint32_t b0 = g_smem_u32(smB + stage * b_stage_stride);
#pragma unroll
                    for (int ks = 0; ks < BK / 16; ++ks) {
#pragma unroll
                        for (int t = 0; t < F::NPROD; ++t) {
                            const uint64_t ad = make_desc_k<ROWB>(a0 + F::pa(t) * a_plane + ks * 32);
                            const uint64_t bd = make_desc_k<ROWB>(b0 + F::pb(t) * b_plane + ks * 32);
                            // split mode: the last product of the list is the leading one (A0B0) -> accumulator 0, the rest -> accumulator 1
                            const bool lead = t == F::NPROD - 1;
                            const uint32_t d = SPLIT ? (lead ? d_tmem : d_tmem + 256u) : d_tmem;
                            const uint32_t acc = SPLIT ? ((lead ? (kb | ks) : (kb | ks | t)) != 0 ? 1u : 0u) : ((kb | ks | t) != 0 ? 1u : 0u);
                            if (NCTA == 2)
                                tc_mma_bf16_pair(d, ad, bd, idesc, acc);
                            else
                                tc_mma_bf16(d, ad, bd, idesc, acc);
                        }
                    }
                    // frees the smem stage (in both CTAs of a pair) when the MMAs above have read it
                    if (NCTA == 2) tc_commit_pair(&empty[stage]); else tc_commit(&empty[stage]);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
                if (NCTA == 2) tc_commit_pair(&tfull[as]); else tc_commit(&tfull[as]);  // accumulator complete
            }
            if (g.stats) {
                atomicAdd(&g.stats[0], (unsigned long long)w_full);
                atomicAdd(&g.stats[1], (unsigned long long)w_tempty);
                atomicAdd(&g.stats[2], (unsigned long long)(clock64() - t_begin));
            }
        }
    } else {
        // ================= epilogue warps (2..9) =================
        // warp w may only touch TMEM lanes [32*(w%4), +32); the two warps of a quadrant take alternating 32-column chunks
        const int quad = warp & 3;
        const int half = (warp - 2) >> 2;
        uint8_t* my_stage = stage_c + (warp - 2) * L::kStageC;
        // x = acc / (sA sB) + bias; when only planes are written (the hidden layers) the output scale is FOLDED into the two constants:
        // fold * x = acc * (fold / (sA sB)) + fold * bias (exact, powers of two), and max / mask commute with a positive factor
        const float c_mul = ld_scale(g.c_scale);
        const bool folded = g.c_f32 == nullptr;
        const float fold = folded ? c_mul : 1.0f;
        const float k_acc = fold / (ld_scale(g.a_scale) * ld_scale(g.b_scale));
        if (warp == 2 && folded)  // (bias_s was filled before the CTA barrier; one warp rescales it)
            for (int t = lane; t < 256; t += 32) bias_s[t] *= fold;
        asm volatile("bar.sync 1, 256;" ::: "memory");  // the 8 epilogue warps only
        float amax = 0.f;
        uint4 tile_bits = make_uint4(0u, 0u, 0u, 0u);
        uint4 out_bits = make_uint4(0u, 0u, 0u, 0u);
        auto process = [&](const uint32_t (&v)[32], int n0, int row, bool row_ok) {
            // ReLU bit masks: word (c & 1) * 4 + (c >> 1) of the row holds columns [32 c, 32 c + 32); a thread owns the chunks of one parity
            // (its `half`), so its words of a tile are the four consecutive ones prefetched into tile_bits before the accumulator wait
            // (both uses are warp-uniform branches: the no-grad forward passes, 8 of the 16 GEMMs of an update, pay nothing for them -- the
            // epilogue has ~30 % of slack against the MMAs of the next tile and an unconditional version used it up)
            float x[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                float f = __fmaf_rn(__uint_as_float(v[j]), k_acc, bias_s[n0 + j]);
                if (g.relu) f = (f < 0.f) ? 0.f : f;  // (NaN stays NaN, like torch.relu: an overflow upstream must reach the loss)
                x[j] = f;
            }
            if (g.bits_in) {
                const int i4 = n0 >> 6;
                const uint32_t keep = i4 == 0 ? tile_bits.x : (i4 == 1 ? tile_bits.y : (i4 == 2 ? tile_bits.z : tile_bits.w));
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (!((keep >> j) & 1u)) x[j] = 0.f;
            }
            if (g.bits_out) {
                // collected per unit and written ONCE after the column loop (one 16-byte store per thread and tile instead of four scattered
                // 4-byte stores: the forward GEMMs of the training pass ran 37 us against 30 us for the same layer without the mask)
                uint32_t positive = 0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (x[j] > 0.f) positive |= 1u << j;
                const int i4 = n0 >> 6;
                if (i4 == 0) out_bits.x = positive; else if (i4 == 1) out_bits.y = positive; else if (i4 == 2) out_bits.z = positive; else out_bits.w = positive;
            }
            if (g.mask && row_ok) {
                const uint4* mrow = reinterpret_cast<const uint4*>(g.mask + (size_t)row * g.ld_mask + n0);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint4 mm = __ldg(mrow + q);
                    const uint32_t w4[4] = {mm.x, mm.y, mm.z, mm.w};
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const uint32_t bits = (e & 1) ? (w4[e >> 1] >> 16) : (w4[e >> 1] & 0xFFFFu);
                        // (bf16 or fp16) > 0  <=>  sign bit clear and magnitude non-zero (NaN never occurs in a ReLU output)
                        if ((bits & 0x8000u) || (bits & 0x7FFFu) == 0u) x[8 * q + e] = 0.f;
                    }
                }
            }
            if (row_ok && g.c_f32) {
                float* crow = g.c_f32 + (size_t)row * g.ldc + n0;
                if (n0 + 32 <= g.N && (g.ldc % 4 == 0)) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(crow + j) = make_float4(x[j], x[j + 1], x[j + 2], x[j + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (n0 + j < g.N) crow[j] = x[j];
                }
            }
            if (g.c_planes && n0 < g.ldp) {
                if (n0 + 32 > g.N) {  // ragged last chunk: columns [N, ldp) are written as zero
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (n0 + j >= g.N) x[j] = 0.f;
                }
                // re-split (c_scale x) into P planes, two columns per word
                uint32_t pw[P][16];
                if (folded) {
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        uint32_t w[P];
                        F::split2(x[j], x[j + 1], w, amax);
#pragma unroll
                        for (int p = 0; p < P; ++p) pw[p][j / 2] = w[p];
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        uint32_t w[P];
                        F::split2(x[j] * c_mul, x[j + 1] * c_mul, w, amax);
#pragma unroll
                        for (int p = 0; p < P; ++p) pw[p][j / 2] = w[p];
                    }
                }
                // stage the warp's [32 rows x 32 cols] x P planes in shared memory (TMA SWIZZLE_64B pattern: 16-byte chunk index
                // XOR ((row >> 1) & 3), bank-conflict free), then ONE bulk tensor store writes it out coalesced and asynchronously
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // previous store has read the staging tile
                __syncwarp();
                uint8_t* st = my_stage + lane * 64;
                const int sw = (lane >> 1) & 3;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int off = ((q ^ sw) << 4);
#pragma unroll
                    for (int p = 0; p < P; ++p)
                        *reinterpret_cast<uint4*>(st + p * 2048 + off) = make_uint4(pw[p][4 * q], pw[p][4 * q + 1], pw[p][4 * q + 2], pw[p][4 * q + 3]);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(&tmC), "r"(g_smem_u32(my_stage)),
                                 "r"(n0), "r"(row - lane), "r"(0)
                                 : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
        };
        uint32_t it = 0;
        long long w_tfull = 0, busy = 0;
        for (int u = unit; u < n_work; u += n_units, ++it) {
            int tile, n_begin, n_cnt;
            unit_of(u, tile, n_begin, n_cnt);
            const uint32_t as = SPLIT ? 0u : (it & 1u);
            if (g.bits_in) {  // independent of the MMAs: in flight while this warp waits for the accumulator
                const int prow = (tile * NCTA + (int)cta_rank) * kGemmBM + quad * 32 + lane;
                tile_bits = prow < g.M ? __ldg(reinterpret_cast<const uint4*>(g.bits_in + (size_t)prow * 8 + half * 4)) : make_uint4(0u, 0u, 0u, 0u);
            }
            const long long c0 = g.stats ? clock64() : 0;
            g_mbar_wait(&tfull[as], SPLIT ? (it & 1u) : ((it >> 1) & 1u));
            const long long c1 = g.stats ? clock64() : 0;
            w_tfull += c1 - c0;
            tc_fence_after();
            const int row = (tile * NCTA + (int)cta_rank) * kGemmBM + quad * 32 + lane;
            const bool row_ok = row < g.M;
            const uint32_t t_row = tmem_base + as * 256u + ((uint32_t)(quad * 32) << 16);
            uint32_t va[32], vb[32];
            int n0 = 32 * half;  // accumulator column of the unit; the output column is n_begin + n0
            if constexpr (SPLIT) {
                // leading + correction accumulators: two TMEM loads per chunk, one correctly rounded add
                while (n0 < n_cnt) {
                    tc_ld32(t_row + (uint32_t)n0, va);
                    tc_ld32(t_row + 256u + (uint32_t)n0, vb);
                    tc_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) va[j] = __float_as_uint(__fadd_rn(__uint_as_float(va[j]), __uint_as_float(vb[j])));
                    process(va, n_begin + n0, row, row_ok);
                    n0 += 64;
                }
            } else {
                // software pipeline over this warp's chunks n0 = 32*half, 32*half + 64, ...: the TMEM load of the next chunk is in
                // flight while the current one is converted and stored
                if (n0 < n_cnt) {
                    tc_ld32(t_row + (uint32_t)n0, va);
                    tc_ld_wait();
                }
                while (n0 < n_cnt) {
                    const int n1 = n0 + 64;
                    if (n1 < n_cnt) tc_ld32(t_row + (uint32_t)n1, vb);
                    process(va, n_begin + n0, row, row_ok);
                    tc_ld_wait();
                    if (n1 >= n_cnt) break;
                    const int n2 = n1 + 64;
                    if (n2 < n_cnt) tc_ld32(t_row + (uint32_t)n2, va);
                    process(vb, n_begin + n1, row, row_ok);
                    tc_ld_wait();
                    n0 = n2;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (NCTA == 2) mbar_arrive_remote(mapa_rank0(g_smem_u32(&tempty[as]))); else g_mbar_arrive(&tempty[as]);
            }
            if (g.bits_out && row_ok) {
                // this thread's chunks of the unit: output columns n_begin + 32 half + 64 k < n_begin + n_cnt, i.e. words (n_begin >> 6) ...
                uint32_t* dst = g.bits_out + (size_t)row * 8 + half * 4;
                const int w0 = n_begin >> 6, w1 = (n_begin + n_cnt - 32 * half + 63) >> 6;  // [w0, w1) of the four words this thread owns
                if (w0 == 0 && w1 == 4) {
                    *reinterpret_cast<uint4*>(dst) = out_bits;
                } else {
                    const uint32_t wv[4] = {out_bits.x, out_bits.y, out_bits.z, out_bits.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (q >= w0 && q < w1) dst[q] = wv[q];
                }
            }
            if (g.stats) busy += clock64() - c1;
        }
        if (g.stats && warp == 2 && lane == 0) {
            atomicAdd(&g.stats[4], (unsigned long long)w_tfull);
            atomicAdd(&g.stats[5], (unsigned long long)busy);
        }
        if (FMT == MORL_FMT_F16X2) note_overflow(amax);
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // all bulk stores of this warp have completed
    }

    tc_fence_before();
    __syncthreads();
    if (NCTA == 2) cluster_sync_all();  // no CTA of a pair exits (or frees TMEM) while its peer can still signal it
    if (warp == 1) {
        tc_fence_after();
        if (NCTA == 2)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// =================================================================================================================
// CHAIN kernel: several dense hidden layers of one or two networks in ONE persistent launch (CTA pairs, f16x2 / bf16x3 planes, N = 256 wide
// layers).  A layer's output rows depend only on the same rows of its input, so a CTA pair can take one of its 256-row tiles through ALL
// layers: the tile it stores for layer l is the tile it loads for layer l+1 a few units later -- by then still in the 126 MB L2, so only the
// first layer's input is read from HBM (the per-layer launches re-read every intermediate activation from HBM: 6 x 134 MB for the two
// no-grad passes of an Envelope update against 6 x 67 MB + 2 x 67 MB here), and the launch prologue / drain is paid once instead of per
// layer.  Work of a pair: its tiles in groups of `lanes / n_chains`; per group, for every layer, one unit per LANE (lane = (chain, tile
// of the group)): four lanes keep the dependency distance at four units (unit (l, lane) needs the stores of unit (l-1, lane)), so the
// producer never waits for the epilogue that has just finished.  Same roles, barriers and arithmetic as gemm_planes_kernel<2, FMT, 0>
// (bit-identical outputs: tests/test_gemm_gpu.py); additional barrier stored[lane]: the epilogue warps of a CTA arrive once their bulk
// stores of the unit have COMPLETED, the producer of the same CTA waits for it before loading the next layer of that lane.
// =================================================================================================================
constexpr int kChainMaxJobs = 8;   // chains x layers
constexpr int kChainLanes = 4;

struct alignas(64) ChainMaps {
    CUtensorMap A[kChainMaxJobs];  // load map of the INPUT of job (chain c, layer l): [P][M][K], box P x 128 x BK
    CUtensorMap B[kChainMaxJobs];  // weight planes of the job: [P][256][K], box P x 128 x BK (each CTA of the pair stages half of the rows)
    CUtensorMap C[kChainMaxJobs];  // store map of the OUTPUT of the job: [P][M][256], box P x 32 x 32 (64-byte swizzle)
};

struct ChainArgs {
    int M, K;                      // rows, reduction length (= width of the layers: square 256-wide layers, K % BK == 0)
    int k_first;                   // reduction length of layer 0 of every chain (its INPUT may be narrower: the dX product of the output layer), K % BK == 0
    int n_chains, n_layers;
    const float* bias[kChainMaxJobs];
    const float* b_scale[kChainMaxJobs];
    uint32_t* bits_out[kChainMaxJobs];  // ReLU bit masks of the job's output, or nullptr
    const uint32_t* bits_in[kChainMaxJobs];  // ReLU-backward masks applied to the job's output (dX chains), or nullptr
    const float* a_scale;          // activation scale (input AND output of every layer), device scalar or nullptr
    int relu;                      // max(x, 0) on every job's output (forward chains)
    int n_stages;
    int pdl;
};

template <int FMT>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_chain_kernel(const __grid_constant__ ChainMaps maps, const ChainArgs g) {
    using F = PlaneFmt<FMT>;
    using L = KPlan<2, FMT>;
    constexpr int P = F::P;
    constexpr int BK = F::BK;
    constexpr int BN = 256;
    constexpr int kMaxStages = L::kMaxStages;
    constexpr uint32_t ROWB = L::kRowB;
    const int kStages = g.n_stages;
    extern __shared__ uint8_t gsmem_raw[];
    uint8_t* gsmem = gsmem_raw + ((1024u - (g_smem_u32(gsmem_raw) & 1023u)) & 1023u);
    constexpr uint32_t a_stage_bytes = L::kAStage;
    constexpr uint32_t b_stage_bytes = L::kBStage;
    uint8_t* smA = gsmem;
    uint8_t* smB = gsmem + (uint32_t)kStages * a_stage_bytes;
    uint8_t* stage_c = gsmem + L::kOffC;
    uint64_t* full = reinterpret_cast<uint64_t*>(gsmem + L::kOffBar);
    uint64_t* empty = full + kMaxStages;
    uint64_t* tfull = empty + kMaxStages;
    uint64_t* tempty = tfull + 2;
    uint64_t* stored = tempty + 2;  // [kChainLanes]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stored + kChainLanes);
    float* bias_s = reinterpret_cast<float*>(gsmem + L::kOffBias);  // [256], refilled per unit by the epilogue warps

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const int unit = blockIdx.x / 2, n_units = gridDim.x / 2;
    const int n_tiles = (g.M + 2 * kGemmBM - 1) / (2 * kGemmBM);
    const int n_kblk_full = g.K / BK, n_kblk_first = g.k_first / BK;
    const int tiles_per_group = kChainLanes / g.n_chains;  // lanes of a group: (tile of the group) x (chain)
    // Tile t of chain c goes to pair (t + offset_c) mod n_units with a DIFFERENT rotation per chain: 256 tiles on 74 pairs leave 34 pairs with
    // four tiles and 40 with three; with both chains on the same pairs the launch lasted 4/3.46 of the balanced time (the 3-tile pairs idled
    // for a quarter of it), rotated by half the pairs every pair gets 4 + 3 or 3 + 3.
    const int cu0 = unit, cu1 = (unit + n_units / 2) % n_units;
    const int mt0 = cu0 < n_tiles ? (n_tiles - cu0 + n_units - 1) / n_units : 0;
    const int mt1 = g.n_chains > 1 ? (cu1 < n_tiles ? (n_tiles - cu1 + n_units - 1) / n_units : 0) : 0;
    const int n_groups = ((mt0 > mt1 ? mt0 : mt1) + tiles_per_group - 1) / tiles_per_group;
    // unit (group gi, layer l, lane ln) -> (job, tile) or tile = -1 (no such tile for this pair)
    auto unit_of = [&](int gi, int l, int ln, int& job, int& tile) {
        const int c = ln % g.n_chains, ti = gi * tiles_per_group + ln / g.n_chains;
        job = c * g.n_layers + l;
        tile = ti < (c ? mt1 : mt0) ? (c ? cu1 : cu0) + ti * n_units : -1;
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            g_mbar_init(&full[s], 1);
            g_mbar_init(&empty[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            g_mbar_init(&tfull[s], 1);
            g_mbar_init(&tempty[s], 16);  // one arrival per epilogue warp of both CTAs, on the leader's barrier
        }
        for (int s = 0; s < kChainLanes; ++s) g_mbar_init(&stored[s], 8);  // the 8 epilogue warps of THIS CTA
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(g_smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    if (g.pdl) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            uint32_t done_on_lane[kChainLanes] = {0u, 0u, 0u, 0u};  // units already issued on each lane = completions of stored[lane] to expect
            for (int gi = 0; gi < n_groups; ++gi)
                for (int l = 0; l < g.n_layers; ++l)
                    for (int ln = 0; ln < kChainLanes; ++ln) {
                        int job, tile;
                        unit_of(gi, l, ln, job, tile);
                        if (tile < 0) continue;
                        if (l > 0) {
                            // the input tile of this unit is the output tile of the lane's previous unit: wait until THIS CTA's stores of
                            // it have completed (completion number done_on_lane[ln] of stored[ln])
                            g_mbar_wait(&stored[ln], (done_on_lane[ln] - 1u) & 1u);
                            asm volatile("fence.proxy.async.global;" ::: "memory");
                        }
                        ++done_on_lane[ln];
                        const int row0 = (tile * 2 + (int)cta_rank) * kGemmBM;
                        const int n_kblk = l == 0 ? n_kblk_first : n_kblk_full;
                        for (int kb = 0; kb < n_kblk; ++kb) {
                            g_mbar_wait(&empty[stage], phase ^ 1u);
                            if (cta_rank == 0) g_mbar_expect_tx(&full[stage], 2u * (a_stage_bytes + b_stage_bytes));
                            const uint32_t lbar = mapa_rank0(g_smem_u32(&full[stage]));
                            tma_load_3d_pair(smA + stage * a_stage_bytes, &maps.A[job], lbar, kb * BK, row0, 0);
                            tma_load_3d_pair(smB + stage * b_stage_bytes, &maps.B[job], lbar, kb * BK, (int)cta_rank * (BN / 2), 0);
                            if (++stage == (uint32_t)kStages) {
                                stage = 0;
                                phase ^= 1u;
                            }
                        }
                    }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (leader CTA only) =================
        if (lane == 0 && cta_rank == 0) {
            constexpr uint32_t idesc = (1u << 4) | F::kIdescAB | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((kGemmBM * 2) >> 4) << 24);
            constexpr uint32_t a_plane = kGemmBM * ROWB;
            constexpr uint32_t b_plane = (uint32_t)(BN / 2) * ROWB;
            uint32_t stage = 0, phase = 0, it = 0;
            for (int gi = 0; gi < n_groups; ++gi)
                for (int l = 0; l < g.n_layers; ++l)
                    for (int ln = 0; ln < kChainLanes; ++ln) {
                        int job, tile;
                        unit_of(gi, l, ln, job, tile);
                        if (tile < 0) continue;
                        const uint32_t as = it & 1u;
                        g_mbar_wait(&tempty[as], ((it >> 1) & 1u) ^ 1u);
                        tc_fence_after();
                        const uint32_t d_tmem = tmem_base + as * 256u;
                        const int n_kblk = l == 0 ? n_kblk_first : n_kblk_full;
                        for (int kb = 0; kb < n_kblk; ++kb) {
                            g_mbar_wait(&full[stage], phase);
                            tc_fence_after();
                            const uint32_t a0 = g_smem_u32(smA + stage * a_stage_bytes);
                            const uint32_t b0 = g_smem_u32(smB + stage * b_stage_bytes);
#pragma unroll
                            for (int ks = 0; ks < BK / 16; ++ks) {
#pragma unroll
                                for (int t = 0; t < F::NPROD; ++t) {
                                    const uint64_t ad = make_desc_k<ROWB>(a0 + F::pa(t) * a_plane + ks * 32);
                                    const uint64_t bd = make_desc_k<ROWB>(b0 + F::pb(t) * b_plane + ks * 32);
                                    tc_mma_bf16_pair(d_tmem, ad, bd, idesc, (kb | ks | t) != 0 ? 1u : 0u);
                                }
                            }
                            tc_commit_pair(&empty[stage]);
                            if (++stage == (uint32_t)kStages) {
                                stage = 0;
                                phase ^= 1u;
                            }
                        }
                        tc_commit_pair(&tfull[as]);
                        ++it;
                    }
        }
    } else {
        // ================= epilogue warps (2..9) =================
        const int quad = warp & 3;
        const int half = (warp - 2) >> 2;
        const int et = threadIdx.x - 64;  // 0..255 among the epilogue threads
        uint8_t* my_stage = stage_c + (warp - 2) * L::kStageC;
        const float s_act = ld_scale(g.a_scale);
        float amax = 0.f;
        uint32_t it = 0;
        for (int gi = 0; gi < n_groups; ++gi)
            for (int l = 0; l < g.n_layers; ++l)
                for (int ln = 0; ln < kChainLanes; ++ln) {
                    int job, tile;
                    unit_of(gi, l, ln, job, tile);
                    if (tile < 0) continue;
                    const uint32_t as = it & 1u;
                    // this unit's bias (times the folded output scale) into shared memory: every epilogue warp has left the previous unit
                    asm volatile("bar.sync 1, 256;" ::: "memory");
                    bias_s[et] = (g.bias[job] ? __ldg(g.bias[job] + et) : 0.f) * s_act;
                    asm volatile("bar.sync 1, 256;" ::: "memory");
                    // x * s_act = acc * (s_act / (s_act * sB)) + s_act * bias  (powers of two: exact), as gemm_planes_kernel's folded epilogue
                    const float k_acc = s_act / (s_act * ld_scale(g.b_scale[job]));
                    uint32_t* bits_out = g.bits_out[job];
                    const uint32_t* bits_in = g.bits_in[job];
                    uint4 out_bits = make_uint4(0u, 0u, 0u, 0u);
                    const int row = (tile * 2 + (int)cta_rank) * kGemmBM + quad * 32 + lane;
                    const bool row_ok = row < g.M;
                    uint4 in_bits = make_uint4(0u, 0u, 0u, 0u);  // (independent of the MMAs: in flight while this warp waits for the accumulator)
                    if (bits_in && row_ok) in_bits = __ldg(reinterpret_cast<const uint4*>(bits_in + (size_t)row * 8 + half * 4));
                    g_mbar_wait(&tfull[as], (it >> 1) & 1u);
                    tc_fence_after();
                    const uint32_t t_row = tmem_base + as * 256u + ((uint32_t)(quad * 32) << 16);
                    uint32_t va[32], vb[32];
                    auto process = [&](const uint32_t (&v)[32], int n0) {
                        float x[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            float f = __fmaf_rn(__uint_as_float(v[j]), k_acc, bias_s[n0 + j]);
                            if (g.relu) f = (f < 0.f) ? 0.f : f;  // (NaN stays NaN)
                            x[j] = f;
                        }
                        if (bits_in) {
                            const int i4 = n0 >> 6;
                            const uint32_t keep = i4 == 0 ? in_bits.x : (i4 == 1 ? in_bits.y : (i4 == 2 ? in_bits.z : in_bits.w));
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (!((keep >> j) & 1u)) x[j] = 0.f;
                        }
                        if (bits_out) {
                            uint32_t positive = 0;
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (x[j] > 0.f) positive |= 1u << j;
                            const int i4 = n0 >> 6;
                            if (i4 == 0) out_bits.x = positive; else if (i4 == 1) out_bits.y = positive; else if (i4 == 2) out_bits.z = positive; else out_bits.w = positive;
                        }
                        uint32_t pw[P][16];
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            uint32_t w[P];
                            F::split2(x[j], x[j + 1], w, amax);
#pragma unroll
                            for (int p = 0; p < P; ++p) pw[p][j / 2] = w[p];
                        }
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        __syncwarp();
                        uint8_t* st = my_stage + lane * 64;
                        const int sw = (lane >> 1) & 3;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int off = ((q ^ sw) << 4);
#pragma unroll
                            for (int p = 0; p < P; ++p)
                                *reinterpret_cast<uint4*>(st + p * 2048 + off) = make_uint4(pw[p][4 * q], pw[p][4 * q + 1], pw[p][4 * q + 2], pw[p][4 * q + 3]);
                        }
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(&maps.C[job]),
                                         "r"(g_smem_u32(my_stage)), "r"(n0), "r"(row - lane), "r"(0)
                                         : "memory");
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                    };
                    int n0 = 32 * half;
                    tc_ld32(t_row + (uint32_t)n0, va);
                    tc_ld_wait();
                    while (n0 < BN) {
                        const int n1 = n0 + 64;
                        if (n1 < BN) tc_ld32(t_row + (uint32_t)n1, vb);
                        process(va, n0);
                        tc_ld_wait();
                        if (n1 >= BN) break;
                        const int n2 = n1 + 64;
                        if (n2 < BN) tc_ld32(t_row + (uint32_t)n2, va);
                        process(vb, n1);
                        tc_ld_wait();
                        n0 = n2;
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_remote(mapa_rank0(g_smem_u32(&tempty[as])));
                    if (bits_out && row_ok) *reinterpret_cast<uint4*>(bits_out + (size_t)row * 8 + half * 4) = out_bits;
                    // the lane's next layer loads what this unit stored: signal once the bulk stores of this warp have completed
                    if (lane == 0) {
                        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
                        g_mbar_arrive(&stored[ln]);
                    }
                    ++it;
                }
        if (FMT == MORL_FMT_F16X2) note_overflow(amax);
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// =================================================================================================================
// MN-major split-K variant: weight gradients  dW[n, k] = sum_m G[m, n] * H[m, k]  (reduction over the 65,536 batch rows).
// Both operands are the row-major plane tensors the forward/backward GEMMs already produced, read "MN-major" (the MMA's M / N
// index is the contiguous one), 128-byte swizzle:  A = G^T (M_mma = n, 128 per unit), B = H^T (N_mma = k <= 256), K_mma = m.
// A unit of work is (128-row block of n, split s of the m range); its fp32 partial tile is summed over the splits by a separate
// reduction launch (deterministic, no atomics), which also removes the operand scales.
// =================================================================================================================
constexpr int kMnKT = 32;  // batch rows (K_mma direction) per pipeline stage

// canonical MN-major layout, SWIZZLE_128B: 64 contiguous MN elements (128 B) x 8 K-rows per 1 KB atom;
// SBO = 1024 B (next 8 K-rows), LBO = distance between 64-element MN chunks.
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;  // SWIZZLE_128B
    return d;
}

// shared memory of the MN-major kernel: the TMA ring (A: 2 chunks, B: up to 4 chunks per stage), barriers, the 4 KB tile of ones, slack
template <int FMT>
constexpr size_t mn_smem_bytes() {
    return (size_t)PlaneFmt<FMT>::kStagesMn * (6u * PlaneFmt<FMT>::P * kMnKT * 128u) + 256 + 1024 + 64 + 1024 + 4096;
}

// -----------------------------------------------------------------------------------------------------------------
// Several weight-gradient products  dW_j = G_j^T H_j (+ db_j = colsum(G_j))  in ONE persistent launch (the backward pass of an update:
// the output layer and every hidden layer), or one product alone (morl_gemm_planes_mn_f32).  A unit is (job, column tile, split); a job's
// split boundaries, MMA shape and MMA issue order do not depend on the other jobs of the launch, so every partial is the same whether the
// product runs alone or with others; units are dealt round-robin to the CTAs.  What a launch of several jobs gains is continuity: the TMA
// ring streams the next unit's operands while the current unit's MMAs and epilogue run, and the prologue (barriers, TMEM allocation, tile
// of ones) is paid once instead of once per layer.
// The accumulator (256 + 16 columns) cannot be double-buffered in 512 TMEM columns: the 8 epilogue warps copy it to registers (two warps per
// lane quadrant, half of the columns each), release it, and store the partials while the MMAs of the next unit already run.
// Only the real rows (n < g_cols) of a tile are stored: partials are [S][g_cols][NB].
// -----------------------------------------------------------------------------------------------------------------
constexpr int kMnMaxJobs = MORL_MN_MAX_JOBS;

struct MnJobArgs {
    int n_tiles, NB, rows_per_split, S;  // column tiles of 128, N_mma (h_cols rounded up to 64), batch rows per split, splits
    int g_cols, h_cols, ld_out;
    int unit0;                           // first unit of the job in the launch's unit sequence
    int red_block0, red_main_blocks;     // reduction launch: first block of the job; blocks of the matrix part (column-sum blocks follow)
    float* partial;                      // [S][g_cols][NB]
    float* colsum_partial;               // [S][g_cols] or nullptr
    float* out;                          // [g_cols][ld_out]
    float* colsum_out;                   // [g_cols] or nullptr
    const float* g_scale;
    const float* h_scale;
};

struct alignas(64) MnMulti {
    CUtensorMap tmA[kMnMaxJobs], tmB[kMnMaxJobs];  // G_j (A = G^T) and H_j (B = H^T), make_plane_map_mn
    MnJobArgs job[kMnMaxJobs];
    int n_jobs, n_units, M;
};

template <int FMT>
__global__ void __launch_bounds__(kGemmThreads, 1) gemm_planes_mn_multi_kernel(const __grid_constant__ MnMulti mj) {
    using F = PlaneFmt<FMT>;
    constexpr int P = F::P;
    constexpr int kStages = F::kStagesMn;
    extern __shared__ uint8_t gsmem_raw[];
    uint8_t* gsmem = gsmem_raw + ((1024u - (g_smem_u32(gsmem_raw) & 1023u)) & 1023u);
    constexpr uint32_t chunk_bytes = (uint32_t)P * kMnKT * 128u;
    constexpr uint32_t a_stage = 2u * chunk_bytes;
    constexpr uint32_t b_stage = 4u * chunk_bytes;
    uint8_t* smA = gsmem;
    uint8_t* smB = gsmem + kStages * a_stage;
    uint64_t* full = reinterpret_cast<uint64_t*>(smB + kStages * b_stage);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;  // accumulator complete (MMA commit)
    uint64_t* tempty = tfull + 1;       // accumulator copied to registers (8 epilogue warps)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
    uint8_t* ones_b = reinterpret_cast<uint8_t*>(tmem_slot + 4);
    uint32_t* ones = reinterpret_cast<uint32_t*>(ones_b + ((1024u - (g_smem_u32(ones_b) & 1023u)) & 1023u));
    for (int t = threadIdx.x; t < 1024; t += blockDim.x) ones[t] = F::kOnes2;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto job_of = [&](int u) {
        int j = 0;
        while (j + 1 < mj.n_jobs && u >= mj.job[j + 1].unit0) ++j;
        return j;
    };
    // unit u -> job j, column tile nt, split and its row range
    auto unit_of = [&](int u, int& j, int& nt, int& split, int& m_begin, int& n_kblk) {
        j = job_of(u);
        const MnJobArgs& jb = mj.job[j];
        const int l = u - jb.unit0;
        nt = l % jb.n_tiles;
        split = l / jb.n_tiles;
        m_begin = split * jb.rows_per_split;
        const int m_end = min(mj.M, m_begin + jb.rows_per_split);
        n_kblk = (m_end - m_begin + kMnKT - 1) / kMnKT;  // >= 1: the host sizes S so that no split is empty
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            g_mbar_init(&full[s], 1);
            g_mbar_init(&empty[s], 1);
        }
        g_mbar_init(tfull, 1);
        g_mbar_init(tempty, 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(g_smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_enter();  // (nothing above touches global memory)

    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;  // one ring across all units of the CTA
            for (int u = blockIdx.x; u < mj.n_units; u += gridDim.x) {
                int j, nt, split, m_begin, n_kblk;
                unit_of(u, j, nt, split, m_begin, n_kblk);
                const CUtensorMap* tmA = &mj.tmA[j];
                const CUtensorMap* tmB = &mj.tmB[j];
                const int nb_chunks = mj.job[j].NB / 64;
                for (int kb = 0; kb < n_kblk; ++kb) {
                    g_mbar_wait(&empty[stage], phase ^ 1u);
                    g_mbar_expect_tx(&full[stage], (2u + (uint32_t)nb_chunks) * chunk_bytes);
                    const int m0 = m_begin + kb * kMnKT;
                    for (int c = 0; c < 2; ++c) tma_load_3d(smA + stage * a_stage + c * chunk_bytes, tmA, &full[stage], nt * 128 + c * 64, m0, 0);
                    for (int c = 0; c < nb_chunks; ++c) tma_load_3d(smB + stage * b_stage + c * chunk_bytes, tmB, &full[stage], c * 64, m0, 0);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc_ones = (1u << 4) | F::kIdescAB | (1u << 15) | (1u << 16) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            const uint64_t ones_desc = make_desc_mn_sw128(g_smem_u32(ones), chunk_bytes);
            constexpr uint32_t plane = kMnKT * 128u;
            uint32_t stage = 0, phase = 0, it = 0;
            for (int u = blockIdx.x; u < mj.n_units; u += gridDim.x, ++it) {
                int j, nt, split, m_begin, n_kblk;
                unit_of(u, j, nt, split, m_begin, n_kblk);
                const bool colsum = mj.job[j].colsum_partial != nullptr;
                const uint32_t idesc = (1u << 4) | F::kIdescAB | (1u << 15) | (1u << 16) | ((uint32_t)(mj.job[j].NB >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
                g_mbar_wait(tempty, (it & 1u) ^ 1u);  // the previous unit's accumulator has been copied out
                tc_fence_after();
                for (int kb = 0; kb < n_kblk; ++kb) {
                    g_mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a0 = g_smem_u32(smA + stage * a_stage);
                    const uint32_t b0 = g_smem_u32(smB + stage * b_stage);
#pragma unroll
                    for (int ks = 0; ks < kMnKT / 16; ++ks) {
#pragma unroll
                        for (int t = 0; t < F::NPROD; ++t) {
                            const uint64_t ad = make_desc_mn_sw128(a0 + F::pa(t) * plane + ks * 2048u, chunk_bytes);
                            const uint64_t bd = make_desc_mn_sw128(b0 + F::pb(t) * plane + ks * 2048u, chunk_bytes);
                            tc_mma_bf16(tmem_base, ad, bd, idesc, (kb | ks | t) != 0 ? 1u : 0u);
                        }
                        if (colsum) {
#pragma unroll
                            for (int pl = P - 1; pl >= 0; --pl)
                                tc_mma_bf16(tmem_base + 256u, make_desc_mn_sw128(a0 + pl * plane + ks * 2048u, chunk_bytes), ones_desc, idesc_ones,
                                            (kb | ks | (P - 1 - pl)) != 0 ? 1u : 0u);
                        }
                    }
                    tc_commit(&empty[stage]);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
                tc_commit(tfull);
            }
        }
    } else {
        const int quad = warp & 3;
        const int half = (warp - 2) >> 2;
        const uint32_t t_row = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t it = 0;
        for (int u = blockIdx.x; u < mj.n_units; u += gridDim.x, ++it) {
            // (only the job is live across the accumulator copy: 128 registers of it leave little room)
            const int j = job_of(u);
            const int ncol = mj.job[j].NB >> 1;  // this warp's accumulator columns: [half * ncol, half * ncol + ncol), a multiple of 32
            const bool colsum = half == 0 && mj.job[j].colsum_partial != nullptr;
            g_mbar_wait(tfull, it & 1u);
            tc_fence_after();
            uint32_t cs = 0;
            if (colsum) cs = tc_ld1(t_row + 256u);
            uint32_t v[4][32];
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c * 32 < ncol) tc_ld32(t_row + (uint32_t)(half * ncol + c * 32), v[c]);
            tc_ld_wait();
            // the values must be in registers before the accumulator is released: tie them to this point
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
                for (int e = 0; e < 32; ++e) asm volatile("" : "+r"(v[c][e]));
            tc_fence_before();
            __syncwarp();
            if (lane == 0) g_mbar_arrive(tempty);
            const MnJobArgs& jb = mj.job[j];
            const int l = u - jb.unit0, nt = l % jb.n_tiles, split = l / jb.n_tiles;
            const int row = nt * 128 + quad * 32 + lane;  // output row (n)
            if (row < jb.g_cols) {
                float* prow = jb.partial + ((size_t)split * jb.g_cols + row) * jb.NB + half * ncol;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c * 32 < ncol) {
#pragma unroll
                        for (int e = 0; e < 32; e += 4)
                            *reinterpret_cast<float4*>(prow + c * 32 + e) = make_float4(__uint_as_float(v[c][e]), __uint_as_float(v[c][e + 1]),
                                                                                         __uint_as_float(v[c][e + 2]), __uint_as_float(v[c][e + 3]));
                    }
                if (colsum) jb.colsum_partial[(size_t)split * jb.g_cols + row] = __uint_as_float(cs);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// out[r][c] (or out[c][r] if transpose) = mul * sum_s partial[s][r][c] for r < rows, c < cols, mul = 1 / (scale_a * scale_b).
// blockDim = (32, 8): 32 consecutive output elements per block, the S partials are strided over threadIdx.y (fixed order:
// deterministic), then combined through shared memory.
// Blocks beyond the matrix (blockIdx.x >= main_blocks) reduce the fused column-sum partials vec_partial[s][prow] into vec_out[rows]
// (mul = 1 / scale_a).
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partial, int S, int prow, int pcol, int rows, int cols,
                                                              int transpose, float* __restrict__ out, int ld_out, int main_blocks,
                                                              const float* __restrict__ vec_partial, float* __restrict__ vec_out,
                                                              const float* __restrict__ scale_a, const float* __restrict__ scale_b) {
    pdl_enter();
    __shared__ float red[8][33];
    float mul = 1.0f / (ld_scale(scale_a) * ld_scale(scale_b));
    if ((int)blockIdx.x >= main_blocks) {  // uniform per block
        partial = vec_partial;
        out = vec_out;
        pcol = 1; cols = 1; transpose = 0; ld_out = 1;
        mul = 1.0f / ld_scale(scale_a);
    }
    const int e = ((int)blockIdx.x >= main_blocks ? (int)blockIdx.x - main_blocks : (int)blockIdx.x) * 32 + threadIdx.x;
    const int total = rows * cols;
    float acc = 0.f;
    int r = 0, c = 0;
    if (e < total) {
        r = e / cols;
        c = e - r * cols;
        const float* p = partial + (size_t)r * pcol + c;
        const size_t stride = (size_t)prow * pcol;
        float a0 = 0.f, a1 = 0.f;
        int s = threadIdx.y;
        for (; s + 8 < S; s += 16) {
            a0 += p[(size_t)s * stride];
            a1 += p[(size_t)(s + 8) * stride];
        }
        if (s < S) a0 += p[(size_t)s * stride];
        acc = a0 + a1;
    }
    red[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && e < total) {
        float t = red[0][threadIdx.x];
#pragma unroll
        for (int y = 1; y < 8; ++y) t += red[y][threadIdx.x];
        t *= mul;
        if (transpose)
            out[(size_t)c * ld_out + r] = t;
        else
            out[(size_t)r * ld_out + c] = t;
    }
}

// Same reduction, four consecutive columns per thread (128-bit loads of the partial tiles): out[r][c..c+3] = mul * sum_s partial[s][r][c..c+3]
// for the non-transposed case with cols % 4 == 0 -- the weight-gradient tiles [256 x 256] x 74 splits of every update go through here.
// blockDim = (32, 8): 128 consecutive output elements per block, the S partials strided over threadIdx.y in the SAME fixed order as
// reduce_partials_kernel (bit-identical results).  Blocks beyond the matrix reduce the fused column-sum partials (scalar path).
// (the body of one block of reduce_partials_vec4_multi_kernel, `block` = its index among the blocks of its job)
__device__ __forceinline__ void reduce_partials_vec4_block(int block, const float* __restrict__ partial, int S, int prow, int pcol, int rows, int cols,
                                                           float* __restrict__ out, int ld_out, int main_blocks, const float* __restrict__ vec_partial,
                                                           float* __restrict__ vec_out, const float* __restrict__ scale_a, const float* __restrict__ scale_b) {
    __shared__ float4 red[8][33];
    if (block >= main_blocks) {  // column-sum tail: one element per thread, as the scalar kernel
        const float mul = 1.0f / ld_scale(scale_a);
        const int e = (block - main_blocks) * 32 + threadIdx.x;
        float acc = 0.f;
        if (e < rows) {
            const float* p = vec_partial + e;
            float a0 = 0.f, a1 = 0.f;
            int s = threadIdx.y;
            for (; s + 8 < S; s += 16) {
                a0 += p[(size_t)s * prow];
                a1 += p[(size_t)(s + 8) * prow];
            }
            if (s < S) a0 += p[(size_t)s * prow];
            acc = a0 + a1;
        }
        red[threadIdx.y][threadIdx.x].x = acc;
        __syncthreads();
        if (threadIdx.y == 0 && e < rows) {
            float t = red[0][threadIdx.x].x;
#pragma unroll
            for (int y = 1; y < 8; ++y) t += red[y][threadIdx.x].x;
            vec_out[e] = t * mul;
        }
        return;
    }
    const float mul = 1.0f / (ld_scale(scale_a) * ld_scale(scale_b));
    const int e4 = (block * 32 + threadIdx.x) * 4;  // first of this thread's four output elements (row-major over rows x cols)
    const int total = rows * cols;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int r = 0, c = 0;
    if (e4 < total) {
        r = e4 / cols;
        c = e4 - r * cols;
        const float* p = partial + (size_t)r * pcol + c;
        const size_t stride = (size_t)prow * pcol;
        // this thread's partials (s = y, y + 8, ...; at most kRedMax of them) are loaded first -- independent 128-bit loads in flight
        // together -- and then added in the same alternating a0 / a1 order as the scalar kernel (bit-identical sums)
        constexpr int kRedMax = 12;
        float4 a0 = acc, a1 = acc;
        if (S <= 8 * kRedMax) {
            float4 v[kRedMax];
#pragma unroll
            for (int k = 0; k < kRedMax; ++k) {
                const int sk = threadIdx.y + 8 * k;
                v[k] = sk < S ? __ldcg(reinterpret_cast<const float4*>(p + (size_t)sk * stride)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int k = 0; k < kRedMax; ++k) {
                if ((int)threadIdx.y + 8 * k < S) {
                    if (k & 1) { a1.x += v[k].x; a1.y += v[k].y; a1.z += v[k].z; a1.w += v[k].w; }
                    else       { a0.x += v[k].x; a0.y += v[k].y; a0.z += v[k].z; a0.w += v[k].w; }
                }
            }
        } else {
            int s = threadIdx.y;
            for (; s + 8 < S; s += 16) {
                const float4 u = *reinterpret_cast<const float4*>(p + (size_t)s * stride);
                const float4 v = *reinterpret_cast<const float4*>(p + (size_t)(s + 8) * stride);
                a0.x += u.x; a0.y += u.y; a0.z += u.z; a0.w += u.w;
                a1.x += v.x; a1.y += v.y; a1.z += v.z; a1.w += v.w;
            }
            if (s < S) {
                const float4 u = *reinterpret_cast<const float4*>(p + (size_t)s * stride);
                a0.x += u.x; a0.y += u.y; a0.z += u.z; a0.w += u.w;
            }
        }
        acc = make_float4(a0.x + a1.x, a0.y + a1.y, a0.z + a1.z, a0.w + a1.w);
    }
    red[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0 && e4 < total) {
        float4 t = red[0][threadIdx.x];
#pragma unroll
        for (int y = 1; y < 8; ++y) {
            const float4 q = red[y][threadIdx.x];
            t.x += q.x; t.y += q.y; t.z += q.z; t.w += q.w;
        }
        *reinterpret_cast<float4*>(out + (size_t)r * ld_out + c) = make_float4(t.x * mul, t.y * mul, t.z * mul, t.w * mul);
    }
}

// the reductions of every job of a gemm_planes_mn_multi_kernel launch in one grid: job j owns blocks [red_block0, next job's red_block0)
__global__ void __launch_bounds__(256) reduce_partials_vec4_multi_kernel(const __grid_constant__ MnMulti mj) {
    pdl_enter();
    int j = 0;
    while (j + 1 < mj.n_jobs && (int)blockIdx.x >= mj.job[j + 1].red_block0) ++j;
    const MnJobArgs& jb = mj.job[j];
    reduce_partials_vec4_block((int)blockIdx.x - jb.red_block0, jb.partial, jb.S, jb.g_cols, jb.NB, jb.g_cols, jb.h_cols, jb.out, jb.ld_out, jb.red_main_blocks,
                               jb.colsum_partial, jb.colsum_out, jb.g_scale, jb.h_scale);
}

// column sums of a plane tensor: part[chunk][n] = sum over the chunk's rows and the P planes of G[p][m][n] (still scaled).
// blockDim = (32, 8): a thread owns 8 consecutive columns (one 16-byte load per plane per row) and every 8th row.
template <int FMT>
__global__ void __launch_bounds__(256) colsum_planes_kernel(const uint16_t* __restrict__ planes, long long plane_stride, int M, int ld, int N,
                                                            int rows_per_chunk, float* __restrict__ part) {
    using F = PlaneFmt<FMT>;
    __shared__ float red[8][32][9];
    const int n0 = (blockIdx.y * 32 + threadIdx.x) * 8;
    const int m0 = blockIdx.x * rows_per_chunk, m1 = min(M, m0 + rows_per_chunk);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    if (n0 < ld) {
        for (int m = m0 + threadIdx.y; m < m1; m += 8) {
            const size_t o = (size_t)m * ld + n0;
#pragma unroll
            for (int p = 0; p < F::P; ++p) F::add8(acc, __ldg(reinterpret_cast<const uint4*>(planes + p * plane_stride + o)));
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[threadIdx.y][threadIdx.x][j] = acc[j];
    __syncthreads();
    if (threadIdx.y == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float t = 0.f;
#pragma unroll
            for (int y = 0; y < 8; ++y) t += red[y][threadIdx.x][j];
            if (n0 + j < N) part[(size_t)blockIdx.x * N + n0 + j] = t;
        }
    }
}

// dU[b][h] = (1/scale) sum_j sum_p G[p][b*W + j][h]   (one block per b; blockDim = (32, 8), 8 columns per thread, j strided over y)
template <int FMT>
__global__ void __launch_bounds__(256) pairs_rowblock_sum_kernel(const uint16_t* __restrict__ planes, long long plane_stride, int W, int H,
                                                                 float* __restrict__ dU, const float* __restrict__ scale) {
    using F = PlaneFmt<FMT>;
    __shared__ float red[8][32][9];
    const int b = blockIdx.x;
    const int h0 = (blockIdx.y * 32 + threadIdx.x) * 8;
    const float inv = 1.0f / ld_scale(scale);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    if (h0 < H) {
        for (int j = threadIdx.y; j < W; j += 8) {
            const size_t o = ((size_t)b * W + j) * H + h0;
#pragma unroll
            for (int p = 0; p < F::P; ++p) F::add8(acc, __ldg(reinterpret_cast<const uint4*>(planes + p * plane_stride + o)));
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[threadIdx.y][threadIdx.x][j] = acc[j];
    __syncthreads();
    if (threadIdx.y == 0 && h0 < H) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float t = 0.f;
#pragma unroll
            for (int y = 0; y < 8; ++y) t += red[y][threadIdx.x][j];
            dU[(size_t)b * H + h0 + j] = t * inv;
        }
    }
}

// dU and the per-chunk partials of dV in ONE pass over the planes of dL/dh1 (|W| <= 64): block = (chunk of <= kPgrMaxB transitions, 256
// columns), thread (x, y) owns 8 columns and the weights j = y, y + 8, ...; the 8 y-partials of dU of every transition of the chunk are
// parked in shared memory and reduced after ONE barrier (same order as pairs_rowblock_sum_kernel), dV[j] accumulates over the
// transitions of the chunk in registers (its scale is removed by the final reduce_partials_kernel).
constexpr int kPgrMaxB = 8;
template <int FMT>
__global__ void __launch_bounds__(256, 2) pairs_grad_reduce_fused_kernel(const uint16_t* __restrict__ planes, long long plane_stride, int B, int W,
                                                                      int H, int b_per_chunk, float* __restrict__ dU, float* __restrict__ partV,
                                                                      const float* __restrict__ scale) {
    pdl_enter();
    using F = PlaneFmt<FMT>;
    extern __shared__ float red_dyn[];  // [kPgrMaxB][8][32][9]
    const int h0 = (blockIdx.y * 32 + threadIdx.x) * 8;
    const int b0 = blockIdx.x * b_per_chunk, b1 = min(B, b0 + b_per_chunk);
    const float inv = 1.0f / ld_scale(scale);
    float accV[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int c = 0; c < 8; ++c) accV[k][c] = 0.f;
    for (int b = b0; b < b1; ++b) {
        float accU[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) accU[c] = 0.f;
        // four weight rows (x P planes) are loaded before any of them is used: with one row at a time the kernel had 32 bytes in flight per
        // thread and ran at a third of the HBM bandwidth (latency bound); predicated loads, no branches, same summation order
#pragma unroll
        for (int kk = 0; kk < 8; kk += 4) {
            uint4 ld[4][F::P];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int j = threadIdx.y + 8 * (kk + q);
                const bool ok = h0 < H && j < W;
                const size_t o = ok ? ((size_t)b * W + j) * H + h0 : 0;
#pragma unroll
                for (int p = 0; p < F::P; ++p)
                    ld[q][p] = ok ? __ldg(reinterpret_cast<const uint4*>(planes + p * plane_stride + o)) : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float v[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) v[c] = 0.f;
#pragma unroll
                for (int p = 0; p < F::P; ++p) F::add8(v, ld[q][p]);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    accU[c] += v[c];
                    accV[kk + q][c] += v[c];
                }
            }
        }
        float* r = red_dyn + (((size_t)(b - b0) * 8 + threadIdx.y) * 32 + threadIdx.x) * 9;
#pragma unroll
        for (int c = 0; c < 8; ++c) r[c] = accU[c];
    }
    __syncthreads();
    if (h0 < H) {
        for (int bl = threadIdx.y; bl < b1 - b0; bl += 8) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float t = 0.f;
#pragma unroll
                for (int y = 0; y < 8; ++y) t += red_dyn[(((size_t)bl * 8 + y) * 32 + threadIdx.x) * 9 + c];
                dU[(size_t)(b0 + bl) * H + h0 + c] = t * inv;
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int j = threadIdx.y + 8 * k;
            if (j < W) {
                float* dst = partV + ((size_t)blockIdx.x * W + j) * H + h0;
                *reinterpret_cast<float4*>(dst) = make_float4(accV[k][0], accV[k][1], accV[k][2], accV[k][3]);
                *reinterpret_cast<float4*>(dst + 4) = make_float4(accV[k][4], accV[k][5], accV[k][6], accV[k][7]);
            }
        }
    }
}

// ---- power-of-two scale of a tensor from its largest magnitude ----------------------------------------------------------------
// scale = 2^(target_exp - e) with amax < 2^e, so that  2^(target_exp-1) <= scale * amax < 2^target_exp  (1 if the tensor is all zero).
__device__ __forceinline__ float scale_from_amax(float amax, int target_exp) {
    if (!(amax > 0.f) || !isfinite(amax)) return 1.0f;
    int e;
    (void)frexpf(amax, &e);
    int k = target_exp - e;
    k = k < -60 ? -60 : (k > 60 ? 60 : k);
    return ldexpf(1.0f, k);
}

// ws[0] = running max (bit pattern of a non-negative float), ws[1] = arrival counter; both zero on entry and zero again on exit
__global__ void __launch_bounds__(256) amax_scale_kernel(const float* __restrict__ src, long long n, int target_exp, float* __restrict__ scale_out,
                                                         unsigned int* __restrict__ ws) {
    pdl_enter();
    __shared__ float red[8];
    float m = 0.f;
    const long long n4 = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) ? (n >> 2) : 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
        m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(__ldg(src + i)));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
        atomicMax(&ws[0], __float_as_uint(m));  // non-negative floats order like their bit patterns; max is order independent
        __threadfence();
        if (atomicAdd(&ws[1], 1u) == gridDim.x - 1) {
            __threadfence();
            const float amax = __uint_as_float(atomicExch(&ws[0], 0u));
            *scale_out = scale_from_amax(amax, target_exp);
            ws[1] = 0u;
        }
    }
}

// ---- fp32 -> planes (operands produced outside the GEMM epilogue: network inputs, weights, gradients) ---------------------------
template <int FMT>
__global__ void __launch_bounds__(256) split_planes_kernel(const float* __restrict__ src, int rows, int cols, int ld_src, int transpose,
                                                           uint16_t* __restrict__ dst, int rows_pad, int ldp, long long plane_stride,
                                                           const float* __restrict__ scale) {
    using F = PlaneFmt<FMT>;
    // dst[p][r][c] for r < rows_pad, c < ldp; source element (r, c) = transpose ? src[c * ld_src + r] : src[r * ld_src + c]
    const long long total = (long long)rows_pad * ldp;
    const float s = ld_scale(scale);
    float amax = 0.f;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(e / ldp), c = (int)(e - (long long)r * ldp);
        float x = 0.f;
        if (r < rows && c < cols) x = (transpose ? src[(size_t)c * ld_src + r] : src[(size_t)r * ld_src + c]) * s;
        uint16_t h[F::P];
        F::split1(x, h, amax);
#pragma unroll
        for (int p = 0; p < F::P; ++p) dst[p * plane_stride + e] = h[p];
    }
    if (FMT == MORL_FMT_F16X2) note_overflow(amax);
}

// non-transposed, ldp % 8 == 0: one thread converts 8 consecutive columns (two 128-bit loads when the source row allows it) and writes one
// 128-bit store per plane -- the gradient seed dL/dQ [65,536 x 24] of every step goes through here
template <int FMT>
__global__ void __launch_bounds__(256) split_planes_vec8_kernel(const float* __restrict__ src, int rows, int cols, int ld_src,
                                                                uint16_t* __restrict__ dst, int rows_pad, int ldp, long long plane_stride,
                                                                const float* __restrict__ scale) {
    pdl_enter();
    using F = PlaneFmt<FMT>;
    const int cpr = ldp >> 3;  // 8-column chunks per row
    const long long total = (long long)rows_pad * cpr;
    const bool vec_ok = (ld_src & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0;
    const float s = ld_scale(scale);
    float amax = 0.f;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(t / cpr), c0 = (int)(t - (long long)r * cpr) << 3;
        float x[8];
        if (r < rows && c0 + 8 <= cols && vec_ok) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * ld_src + c0));
            const float4 b = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * ld_src + c0 + 4));
            x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) x[k] = (r < rows && c0 + k < cols) ? __ldg(src + (size_t)r * ld_src + c0 + k) : 0.f;
        }
        uint32_t pw[F::P][4];
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            uint32_t w[F::P];
            F::split2(x[k] * s, x[k + 1] * s, w, amax);
#pragma unroll
            for (int p = 0; p < F::P; ++p) pw[p][k >> 1] = w[p];
        }
        const size_t e = (size_t)r * ldp + c0;
#pragma unroll
        for (int p = 0; p < F::P; ++p) *reinterpret_cast<uint4*>(dst + p * plane_stride + e) = make_uint4(pw[p][0], pw[p][1], pw[p][2], pw[p][3]);
    }
    if (FMT == MORL_FMT_F16X2) note_overflow(amax);
}

// several small matrices (the weight matrices of a network, plain and transposed) in ONE launch: blockIdx.y selects the job.  Jobs with
// auto_scale != 0 derive their power-of-two scale from the largest |element| of their matrix in a one-block-per-job pre-pass
// (split_amax_multi_kernel, launched right before by the same entry point), which publishes it in *scale.
struct SplitJobs {
    MorlSplitJob job[MORL_SPLIT_MAX_JOBS];
};
__global__ void __launch_bounds__(1024) split_amax_multi_kernel(const __grid_constant__ SplitJobs jobs) {
    pdl_enter();
    __shared__ float red[32];
    const MorlSplitJob& j = jobs.job[blockIdx.x];
    if (!j.auto_scale || !j.scale) return;  // uniform per block
    const float* __restrict__ src = j.src;
    const int n_src = j.transpose ? j.cols : j.rows, k_src = j.transpose ? j.rows : j.cols;  // source matrix [n_src, k_src], row stride ld_src
    float m = 0.f;
    if (j.ld_src == k_src && (k_src & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {  // dense: 128-bit loads
        const int n4 = (n_src * k_src) >> 2;
        for (int e = threadIdx.x; e < n4; e += blockDim.x) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(src) + e);
            m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        }
    } else {
        for (int r = threadIdx.x / 32; r < n_src; r += blockDim.x / 32)
            for (int c = threadIdx.x & 31; c < k_src; c += 32) m = fmaxf(m, fabsf(__ldg(src + (size_t)r * j.ld_src + c)));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = red[threadIdx.x];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
        if (threadIdx.x == 0) *j.scale = scale_from_amax(m, j.target_exp);
    }
}

template <int FMT>
__global__ void __launch_bounds__(256) split_planes_multi_kernel(const __grid_constant__ SplitJobs jobs) {
    pdl_enter();
    using F = PlaneFmt<FMT>;
    const MorlSplitJob& j = jobs.job[blockIdx.y];
    const float* __restrict__ src = j.src;
    uint16_t* __restrict__ dst = static_cast<uint16_t*>(j.dst_planes);
    const float s = j.scale ? *j.scale : 1.0f;  // (auto-scaled jobs: written by the pre-pass)
    const long long total = (long long)j.rows_pad * j.ldp;
    float amax = 0.f;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(e / j.ldp), c = (int)(e - (long long)r * j.ldp);
        float x = 0.f;
        if (r < j.rows && c < j.cols) x = (j.transpose ? src[(size_t)c * j.ld_src + r] : src[(size_t)r * j.ld_src + c]) * s;
        uint16_t h[F::P];
        F::split1(x, h, amax);
#pragma unroll
        for (int p = 0; p < F::P; ++p) dst[p * j.plane_stride + e] = h[p];
    }
    if (FMT == MORL_FMT_F16X2) note_overflow(amax);
}

// ---- separable first layer: h[b*W + j] = relu(u[b] + v[j]) straight into planes ------------------------------------------------
template <int FMT>
__global__ void __launch_bounds__(256) pairs_relu_split_kernel(const float* __restrict__ u, const float* __restrict__ v, int B, int W, int H,
                                                               uint16_t* __restrict__ dst, long long plane_stride, const float* __restrict__ scale,
                                                               uint32_t* __restrict__ bits_out) {
    pdl_enter();
    using F = PlaneFmt<FMT>;
    const int hv = H / 8;  // 8 columns per thread: two float4 loads per operand, one 16-byte store per plane
    const long long total = (long long)B * W * hv;
    const float s = ld_scale(scale);
    float amax = 0.f;
    const int lane = threadIdx.x & 31;
    // warp-uniform trip count (the bit words are assembled with shuffles): e0 = element of lane 0
    for (long long e0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x - lane); e0 < total; e0 += (long long)gridDim.x * blockDim.x) {
        const long long e = e0 + lane;
        const bool ok = e < total;
        const long long ee = ok ? e : 0;
        const int h8 = (int)(ee % hv);
        const long long row = ee / hv;
        const int b = (int)(row / W), j = (int)(row - (long long)b * W);
        const float4* up = reinterpret_cast<const float4*>(u + (size_t)b * H + 8 * h8);
        const float4* vp = reinterpret_cast<const float4*>(v + (size_t)j * H + 8 * h8);
        const float4 u0 = __ldg(up), u1 = __ldg(up + 1), v0 = __ldg(vp), v1 = __ldg(vp + 1);
        const float x[8] = {u0.x + v0.x, u0.y + v0.y, u0.z + v0.z, u0.w + v0.w, u1.x + v1.x, u1.y + v1.y, u1.z + v1.z, u1.w + v1.w};
        uint32_t o[F::P][4];
        uint32_t pos = 0;  // bit t = (column 8 h8 + t is positive)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t w[F::P];
            const float r0 = x[2 * q] < 0.f ? 0.f : x[2 * q], r1 = x[2 * q + 1] < 0.f ? 0.f : x[2 * q + 1];  // NaN-propagating ReLU
            pos |= (r0 > 0.f ? 1u : 0u) << (2 * q) | (r1 > 0.f ? 1u : 0u) << (2 * q + 1);
            F::split2(r0 * s, r1 * s, w, amax);
#pragma unroll
            for (int p = 0; p < F::P; ++p) o[p][q] = w[p];
        }
        if (ok) {
            const long long off = row * H + 8 * h8;
#pragma unroll
            for (int p = 0; p < F::P; ++p) *reinterpret_cast<uint4*>(dst + p * plane_stride + off) = make_uint4(o[p][0], o[p][1], o[p][2], o[p][3]);
        }
        if (bits_out) {
            // four consecutive threads (h8 = 4c .. 4c + 3; H % 32 == 0 keeps them in one aligned lane group) hold one 32-column word
            uint32_t wbits = pos << (8 * (lane & 3));
            wbits |= __shfl_xor_sync(0xffffffffu, wbits, 1);
            wbits |= __shfl_xor_sync(0xffffffffu, wbits, 2);
            if (ok && (lane & 3) == 0) {
                const int chunk = h8 >> 2;
                bits_out[(size_t)row * 8 + (chunk & 1) * 4 + (chunk >> 1)] = wbits;
            }
        }
    }
    if (FMT == MORL_FMT_F16X2) note_overflow(amax);
}

// H = 256 form (the shape of the update): one warp per (transition b, quarter of the weight set), lane = 8 columns.  u[b] stays in
// registers for the warp's rows, v[j] comes from L1 / L2 (64 KB in total), four rows are in flight per iteration: half the load traffic of
// the element-indexed kernel above and no index arithmetic per element -- the kernel is a 67 MB write stream and nothing else.
template <int FMT>
__global__ void __launch_bounds__(256) pairs_relu_split_h256_kernel(const float* __restrict__ u, const float* __restrict__ v, int B, int W,
                                                                    uint16_t* __restrict__ dst, long long plane_stride,
                                                                    const float* __restrict__ scale, uint32_t* __restrict__ bits_out, int jsplit) {
    pdl_enter();
    using F = PlaneFmt<FMT>;
    constexpr int H = 256;
    const int lane = threadIdx.x & 31;
    const long long task = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (task >= (long long)B * jsplit) return;
    const int b = (int)(task / jsplit), js = (int)(task - (long long)b * jsplit);
    const int j0 = (int)((long long)W * js / jsplit), j1 = (int)((long long)W * (js + 1) / jsplit);
    const float s = ld_scale(scale);
    float amax = 0.f;
    const float4 u0 = __ldg(reinterpret_cast<const float4*>(u + (size_t)b * H + 8 * lane)),
                 u1 = __ldg(reinterpret_cast<const float4*>(u + (size_t)b * H + 8 * lane) + 1);
    const float uu[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    for (int jb = j0; jb < j1; jb += 4) {
        float4 va[4], vb[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = min(jb + q, j1 - 1);
            va[q] = __ldg(reinterpret_cast<const float4*>(v + (size_t)j * H + 8 * lane));
            vb[q] = __ldg(reinterpret_cast<const float4*>(v + (size_t)j * H + 8 * lane) + 1);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (jb + q >= j1) break;  // (warp-uniform)
            const float x[8] = {uu[0] + va[q].x, uu[1] + va[q].y, uu[2] + va[q].z, uu[3] + va[q].w,
                                uu[4] + vb[q].x, uu[5] + vb[q].y, uu[6] + vb[q].z, uu[7] + vb[q].w};
            uint32_t o[F::P][4];
            uint32_t pos = 0;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                uint32_t w[F::P];
                const float r0 = x[2 * t] < 0.f ? 0.f : x[2 * t], r1 = x[2 * t + 1] < 0.f ? 0.f : x[2 * t + 1];  // NaN-propagating ReLU
                pos |= (r0 > 0.f ? 1u : 0u) << (2 * t) | (r1 > 0.f ? 1u : 0u) << (2 * t + 1);
                F::split2(r0 * s, r1 * s, w, amax);
#pragma unroll
                for (int p = 0; p < F::P; ++p) o[p][t] = w[p];
            }
            const long long row = (long long)b * W + jb + q;
            const long long off = row * H + 8 * lane;
#pragma unroll
            for (int p = 0; p < F::P; ++p) *reinterpret_cast<uint4*>(dst + p * plane_stride + off) = make_uint4(o[p][0], o[p][1], o[p][2], o[p][3]);
            if (bits_out) {
                uint32_t wbits = pos << (8 * (lane & 3));
                wbits |= __shfl_xor_sync(0xffffffffu, wbits, 1);
                wbits |= __shfl_xor_sync(0xffffffffu, wbits, 2);
                const int chunk = lane >> 2;
                if ((lane & 3) == 0) bits_out[(size_t)row * 8 + (chunk & 1) * 4 + (chunk >> 1)] = wbits;
            }
        }
    }
    if (FMT == MORL_FMT_F16X2) note_overflow(amax);
}



static int make_plane_map_mn(CUtensorMap* map, int fmt, const void* base, int rows, int ld, long long plane_stride_elems) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return -1;
    const cuuint32_t P = (cuuint32_t)fmt_planes(fmt);
    const cuuint64_t dims[3] = {(cuuint64_t)ld, (cuuint64_t)rows, P};
    const cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)plane_stride_elems * 2};
    const cuuint32_t box[3] = {64, (cuuint32_t)kMnKT, P};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(map, fmt_tm_type(fmt), 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)r;
}

static inline bool fmt_ok(int fmt) { return fmt == MORL_FMT_BF16X3 || fmt == MORL_FMT_F16X2; }

// split-K plan of an MN-major product: S splits of rps rows (a multiple of kMnKT) so that n_tiles * S fills the 148 SMs; no split is empty
static inline void mn_split(int M, int n_tiles, int& S, int& rps) {
    S = 148 / n_tiles;
    if (S < 1) S = 1;
    rps = ((M + S - 1) / S + kMnKT - 1) / kMnKT * kMnKT;
    S = (M + rps - 1) / rps;
}

// floats of one job's workspace region: partials [S][g_cols][NB], then the column-sum partials [S][g_cols] (rounded up to 16 bytes)
static inline size_t mn_multi_job_floats(int M, int g_cols, int h_cols) {
    int S, rps;
    mn_split(M, (g_cols + 127) / 128, S, rps);
    const size_t nb = (size_t)((h_cols + 63) / 64 * 64);
    return (size_t)S * g_cols * nb + ((size_t)S * g_cols + 3) / 4 * 4;
}

// Checks job q as job mj.n_jobs of a launch (messages name the entry point `fn`) and appends it: its MnJobArgs and tensor maps, its partials
// at `ws`, its reduction blocks after the first `red_blocks` of the launch.  `ws` and `red_blocks` advance past the job.
static int mn_add_job(const char* fn, int fmt, const MorlMnJob& q, MnMulti& mj, float*& ws, int& red_blocks) {
    const int i = mj.n_jobs, M = mj.M;
    MORL_REQUIRE(q.g_planes && q.h_planes && q.out, MORL_ERR_NULL, "%s: job %d has a NULL pointer", fn, i);
    MORL_REQUIRE(q.g_cols > 0 && q.h_cols > 0 && q.ldg % 64 == 0 && q.ldh % 64 == 0 && q.ldh <= 256 && q.g_cols <= q.ldg && q.h_cols <= q.ldh,
                 MORL_ERR_SHAPE, "%s: job %d: bad shape g_cols=%d ldg=%d h_cols=%d ldh=%d (ld multiples of 64, ldh <= 256)", fn, i, q.g_cols, q.ldg,
                 q.h_cols, q.ldh);
    const int n_tiles = (q.g_cols + 127) / 128;
    MORL_REQUIRE(n_tiles * 128 <= q.ldg || q.ldg % 128 == 0 || n_tiles * 128 - q.ldg <= 64, MORL_ERR_UNSUPPORTED, "%s: job %d: ldg=%d", fn, i, q.ldg);
    MnJobArgs& a = mj.job[i];
    mn_split(M, n_tiles, a.S, a.rows_per_split);  // no split is empty: every unit writes its whole partial tile (the reduction reads all S)
    a.n_tiles = n_tiles;
    a.NB = (q.h_cols + 63) / 64 * 64;
    a.g_cols = q.g_cols; a.h_cols = q.h_cols; a.ld_out = q.ld_out;
    a.unit0 = mj.n_units;
    mj.n_units += n_tiles * a.S;
    a.partial = ws;
    a.colsum_partial = q.colsum_out ? ws + (size_t)a.S * q.g_cols * a.NB : nullptr;
    ws += mn_multi_job_floats(M, q.g_cols, q.h_cols);
    a.out = q.out; a.colsum_out = q.colsum_out; a.g_scale = q.g_scale; a.h_scale = q.h_scale;
    a.red_block0 = red_blocks;
    a.red_main_blocks = (q.g_cols * q.h_cols / 4 + 31) / 32;
    red_blocks += a.red_main_blocks + (q.colsum_out ? (q.g_cols + 31) / 32 : 0);
    int rc = make_plane_map_mn(&mj.tmA[i], fmt, q.g_planes, M, q.ldg, q.g_plane_stride);
    MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "%s: job %d: cuTensorMapEncodeTiled(G) failed (%d)", fn, i, rc);
    rc = make_plane_map_mn(&mj.tmB[i], fmt, q.h_planes, M, q.ldh, q.h_plane_stride);
    MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "%s: job %d: cuTensorMapEncodeTiled(H) failed (%d)", fn, i, rc);
    mj.n_jobs = i + 1;
    return 0;
}

// gemm_planes_mn_multi_kernel over every unit of mj: one CTA per SM, or one per unit when there are fewer units
static int mn_launch(const char* fn, int fmt, const MnMulti& mj, cudaStream_t st) {
    int sms = morl_device_sm_count();
    if (sms <= 0) sms = 148;
    const int grid = mj.n_units < sms ? mj.n_units : sms;
    MORL_DISPATCH_FMT(fmt, {
        constexpr size_t smem = mn_smem_bytes<kFmt>();
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(gemm_planes_mn_multi_kernel<kFmt>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            attr_set = true;
        }
        launch_k(gemm_planes_mn_multi_kernel<kFmt>, dim3(grid), dim3(kGemmThreads), smem, st, mj);
    });
    return check_launch(fn);
}

}  // namespace morl

extern "C" int morl_plane_overflow_count(int reset) {
    using namespace morl;
    unsigned int v = 0;
    cudaDeviceSynchronize();
    if (cudaMemcpyFromSymbol(&v, g_plane_overflow, sizeof(v)) != cudaSuccess) {
        (void)cudaGetLastError();
        set_error("morl_plane_overflow_count: no CUDA device");
        return MORL_ERR_NO_DEVICE;
    }
    if (reset) {
        const unsigned int z = 0;
        cudaMemcpyToSymbol(g_plane_overflow, &z, sizeof(z));
    }
    return (int)(v > 0x7fffffffu ? 0x7fffffffu : v);
}

extern "C" int morl_amax_scale_f32(const float* src, long long n, int target_exp, float* scale_out, void* workspace, void* stream) {
    using namespace morl;
    MORL_REQUIRE(src && scale_out && workspace, MORL_ERR_NULL, "morl_amax_scale_f32: NULL pointer argument");
    MORL_REQUIRE(n > 0 && target_exp >= -14 && target_exp <= 15, MORL_ERR_SHAPE, "morl_amax_scale_f32: bad n=%lld / target_exp=%d", n, target_exp);
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 148) blocks = 148;
    if (blocks < 1) blocks = 1;
    launch_k(amax_scale_kernel, dim3((int)blocks), dim3(256), 0, static_cast<cudaStream_t>(stream), src, n, target_exp, scale_out, static_cast<unsigned int*>(workspace));
    return check_launch("morl_amax_scale_f32");
}

extern "C" size_t morl_gemm_mn_workspace_bytes(int M, int a_cols, int b_cols) {
    if (M <= 0 || a_cols <= 0 || b_cols <= 0) return 0;
    return morl::mn_multi_job_floats(M, a_cols, b_cols) * sizeof(float);
}

extern "C" int morl_gemm_planes_mn_f32(int fmt, const void* g_planes, long long g_plane_stride, int ldg, int g_cols, const float* g_scale,
                                       const void* h_planes, long long h_plane_stride, int ldh, int h_cols, const float* h_scale, int M,
                                       int transpose_out, float* out, int ld_out, float* colsum_out, void* workspace, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_gemm_planes_mn_f32: unknown plane format %d", fmt);
    MORL_REQUIRE(g_planes && h_planes && out && workspace, MORL_ERR_NULL, "morl_gemm_planes_mn_f32: NULL pointer argument");
    MORL_REQUIRE(M > 0 && g_cols > 0 && h_cols > 0, MORL_ERR_SHAPE, "morl_gemm_planes_mn_f32: bad shape M=%d g_cols=%d h_cols=%d", M, g_cols, h_cols);
    MORL_REQUIRE(ldg % 64 == 0 && ldh % 64 == 0 && ldh <= 256 && g_cols <= ldg && h_cols <= ldh, MORL_ERR_UNSUPPORTED,
                 "morl_gemm_planes_mn_f32: plane row lengths must be multiples of 64 (ldg=%d ldh=%d), ldh <= 256", ldg, ldh);
    const int n_tiles = (g_cols + 127) / 128;
    MORL_REQUIRE(n_tiles * 128 <= ldg || ldg % 128 == 0 || n_tiles * 128 - ldg <= 64, MORL_ERR_UNSUPPORTED, "morl_gemm_planes_mn_f32: ldg=%d", ldg);
    MORL_REQUIRE(aligned16(workspace), MORL_ERR_ALIGN, "morl_gemm_planes_mn_f32: workspace must be 16-byte aligned");
    MnMulti mj;
    memset(&mj, 0, sizeof(mj));
    mj.M = M;
    const MorlMnJob q = {g_planes, g_plane_stride, g_scale, h_planes, h_plane_stride, h_scale, out, colsum_out, ldg, g_cols, ldh, h_cols, ld_out};
    float* ws = static_cast<float*>(workspace);
    int red_blocks = 0;
    int rc = mn_add_job("morl_gemm_planes_mn_f32", fmt, q, mj, ws, red_blocks);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = mn_launch("morl_gemm_planes_mn_f32", fmt, mj, st);
    if (rc) return rc;
    if (!transpose_out && h_cols % 4 == 0 && ld_out % 4 == 0 && aligned16(out)) {
        launch_k(reduce_partials_vec4_multi_kernel, dim3(red_blocks), dim3(32, 8), 0, st, mj);
        return check_launch("morl_gemm_planes_mn_f32(reduce)");
    }
    // transposed or odd-width output: the scalar reduction of the same [S][g_cols][NB] partials, summed in the same order
    const MnJobArgs& a = mj.job[0];
    const int main_blocks = (g_cols * h_cols + 31) / 32, vec_blocks = colsum_out ? (g_cols + 31) / 32 : 0;
    launch_k(reduce_partials_kernel, dim3(main_blocks + vec_blocks), dim3(32, 8), 0, st, a.partial, a.S, g_cols, a.NB, g_cols, h_cols, transpose_out, out,
             ld_out, main_blocks, a.colsum_partial, colsum_out, g_scale, h_scale);
    return check_launch("morl_gemm_planes_mn_f32(reduce)");
}

extern "C" size_t morl_gemm_mn_multi_workspace_bytes(const MorlMnJob* jobs, int n_jobs, int M) {
    using namespace morl;
    if (!jobs || n_jobs <= 0 || n_jobs > kMnMaxJobs || M <= 0) return 0;
    size_t floats = 0;
    for (int i = 0; i < n_jobs; ++i) {
        if (jobs[i].g_cols <= 0 || jobs[i].h_cols <= 0) return 0;
        floats += mn_multi_job_floats(M, jobs[i].g_cols, jobs[i].h_cols);
    }
    return floats * sizeof(float);
}

extern "C" int morl_gemm_planes_mn_multi_f32(int fmt, const MorlMnJob* jobs, int n_jobs, int M, void* workspace, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_gemm_planes_mn_multi_f32: unknown plane format %d", fmt);
    MORL_REQUIRE(jobs && workspace, MORL_ERR_NULL, "morl_gemm_planes_mn_multi_f32: NULL pointer argument");
    MORL_REQUIRE(n_jobs >= 1 && n_jobs <= kMnMaxJobs && M > 0, MORL_ERR_SHAPE, "morl_gemm_planes_mn_multi_f32: bad n_jobs=%d / M=%d (1 <= n_jobs <= %d)", n_jobs, M,
                 kMnMaxJobs);
    MORL_REQUIRE(aligned16(workspace), MORL_ERR_ALIGN, "morl_gemm_planes_mn_multi_f32: workspace must be 16-byte aligned");
    MnMulti mj;  // (host staging; copied into the kernel parameters by the launches)
    memset(&mj, 0, sizeof(mj));
    mj.M = M;
    float* ws = static_cast<float*>(workspace);
    int red_blocks = 0;
    for (int i = 0; i < n_jobs; ++i) {
        const MorlMnJob& q = jobs[i];
        const int rc = mn_add_job("morl_gemm_planes_mn_multi_f32", fmt, q, mj, ws, red_blocks);
        if (rc) return rc;
        // the reduction stores four consecutive columns per thread
        MORL_REQUIRE(q.h_cols % 4 == 0 && q.ld_out >= q.h_cols && q.ld_out % 4 == 0 && aligned16(q.out), MORL_ERR_UNSUPPORTED,
                     "morl_gemm_planes_mn_multi_f32: job %d: needs h_cols %% 4 == 0, ld_out %% 4 == 0 (>= h_cols) and a 16-byte aligned output", i);
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rc = mn_launch("morl_gemm_planes_mn_multi_f32", fmt, mj, st);
    if (rc) return rc;
    launch_k(reduce_partials_vec4_multi_kernel, dim3(red_blocks), dim3(32, 8), 0, st, mj);
    return check_launch("morl_gemm_planes_mn_multi_f32(reduce)");
}

extern "C" int morl_colsum_planes(int fmt, const void* planes, long long plane_stride, const float* scale, int M, int ld, int N, float* out,
                                  void* workspace, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_colsum_planes: unknown plane format %d", fmt);
    MORL_REQUIRE(planes && out && workspace, MORL_ERR_NULL, "morl_colsum_planes: NULL pointer argument");
    MORL_REQUIRE(M > 0 && N > 0 && ld >= N && ld % 8 == 0 && plane_stride % 8 == 0, MORL_ERR_SHAPE, "morl_colsum_planes: bad shape M=%d N=%d ld=%d", M, N, ld);
    const int chunks = 296;
    const int rpc = (M + chunks - 1) / chunks;
    const int nch = (M + rpc - 1) / rpc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float* part = static_cast<float*>(workspace);
    MORL_DISPATCH_FMT(fmt, (colsum_planes_kernel<kFmt><<<dim3((unsigned)nch, (unsigned)((ld + 255) / 256)), dim3(32, 8), 0, st>>>(
                               static_cast<const uint16_t*>(planes), plane_stride, M, ld, N, rpc, part)));
    int rc = check_launch("morl_colsum_planes");
    if (rc) return rc;
    launch_k(reduce_partials_kernel, dim3((N + 31) / 32), dim3(dim3(32, 8)), 0, st, part, nch, 1, N, 1, N, 0, out, N, 1 << 30, nullptr, nullptr, scale, nullptr);
    return check_launch("morl_colsum_planes(reduce)");
}

extern "C" int morl_pairs_grad_reduce_planes(int fmt, const void* planes, long long plane_stride, const float* scale, int B, int W, int H, float* dU,
                                             float* dV, void* workspace, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_pairs_grad_reduce_planes: unknown plane format %d", fmt);
    MORL_REQUIRE(planes && dU && dV && workspace, MORL_ERR_NULL, "morl_pairs_grad_reduce_planes: NULL pointer argument");
    MORL_REQUIRE(B > 0 && W > 0 && H > 0 && H % 8 == 0 && plane_stride % 8 == 0, MORL_ERR_SHAPE, "morl_pairs_grad_reduce_planes: bad shape B=%d W=%d H=%d", B, W, H);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const uint16_t* pl = static_cast<const uint16_t*>(planes);
    if (W <= 64) {
        // one pass: dU directly, dV as per-chunk partials [chunks][W*H] reduced in a fixed order
        int bpc = (B + 295) / 296;  // <= 296 chunks (the documented workspace size), at most kPgrMaxB transitions per chunk
        if (bpc > kPgrMaxB) bpc = kPgrMaxB;
        const int nchf = (B + bpc - 1) / bpc;
        if (nchf <= 296) {
            const int Nf = W * H;
            float* partf = static_cast<float*>(workspace);
            const size_t smemf = (size_t)kPgrMaxB * 8 * 32 * 9 * sizeof(float);  // 73,728 B
            MORL_DISPATCH_FMT(fmt, {
                static bool configured = false;
                if (!configured) {
                    cudaFuncSetAttribute(pairs_grad_reduce_fused_kernel<kFmt>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemf);
                    configured = true;
                }
                launch_k(pairs_grad_reduce_fused_kernel<kFmt>, dim3(dim3((unsigned)nchf, (unsigned)((H + 255) / 256))), dim3(dim3(32, 8)), smemf, st, pl, plane_stride, B, W,
                                                                                                                                     H, bpc, dU, partf, scale);
            });
            int rcf = check_launch("morl_pairs_grad_reduce_planes(fused)");
            if (rcf) return rcf;
            launch_k(reduce_partials_kernel, dim3((Nf + 31) / 32), dim3(dim3(32, 8)), 0, st, partf, nchf, 1, Nf, 1, Nf, 0, dV, Nf, 1 << 30, nullptr, nullptr, scale, nullptr);
            return check_launch("morl_pairs_grad_reduce_planes(reduce)");
        }
    }
    // dU[b] = sum over the W rows of transition b
    MORL_DISPATCH_FMT(fmt, (pairs_rowblock_sum_kernel<kFmt><<<dim3((unsigned)B, (unsigned)((H + 255) / 256)), dim3(32, 8), 0, st>>>(pl, plane_stride, W, H,
                                                                                                                                     dU, scale)));
    int rc = check_launch("morl_pairs_grad_reduce_planes(dU)");
    if (rc) return rc;
    // dV[j] = sum over b: column sums of the [B, W*H] view
    const int N = W * H;
    const int chunks = 74;
    const int rpc = (B + chunks - 1) / chunks;
    const int nch = (B + rpc - 1) / rpc;
    float* part = static_cast<float*>(workspace);
    MORL_DISPATCH_FMT(fmt, (colsum_planes_kernel<kFmt><<<dim3((unsigned)nch, (unsigned)((N + 255) / 256)), dim3(32, 8), 0, st>>>(pl, plane_stride, B, N, N,
                                                                                                                                  rpc, part)));
    rc = check_launch("morl_pairs_grad_reduce_planes(dV)");
    if (rc) return rc;
    launch_k(reduce_partials_kernel, dim3((N + 31) / 32), dim3(dim3(32, 8)), 0, st, part, nch, 1, N, 1, N, 0, dV, N, 1 << 30, nullptr, nullptr, scale, nullptr);
    return check_launch("morl_pairs_grad_reduce_planes(reduce)");
}

extern "C" int morl_split_planes(int fmt, const float* src, int rows, int cols, int ld_src, int transpose, void* dst_planes, int rows_pad, int ldp,
                                 long long plane_stride, const float* scale, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_split_planes: unknown plane format %d", fmt);
    MORL_REQUIRE(src && dst_planes, MORL_ERR_NULL, "morl_split_planes: NULL pointer argument");
    MORL_REQUIRE(rows > 0 && cols > 0 && rows_pad >= rows && ldp >= cols && ld_src > 0, MORL_ERR_SHAPE,
                 "morl_split_planes: bad shape rows=%d cols=%d rows_pad=%d ldp=%d", rows, cols, rows_pad, ldp);
    MORL_REQUIRE(plane_stride >= (long long)rows_pad * ldp, MORL_ERR_SHAPE, "morl_split_planes: plane_stride too small");
    const long long total = (long long)rows_pad * ldp;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint16_t* dst = static_cast<uint16_t*>(dst_planes);
    if (!transpose && (ldp & 7) == 0 && (plane_stride & 7) == 0 && (reinterpret_cast<uintptr_t>(dst_planes) & 15u) == 0) {
        const long long chunks = total >> 3;
        long long vb = (chunks + 255) / 256;
        if (vb > 148 * 8) vb = 148 * 8;
        MORL_DISPATCH_FMT(fmt, (launch_k(split_planes_vec8_kernel<kFmt>, dim3((int)vb), dim3(256), 0, st, src, rows, cols, ld_src, dst, rows_pad, ldp, plane_stride, scale)));
        return check_launch("morl_split_planes(vec8)");
    }
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    MORL_DISPATCH_FMT(fmt, (split_planes_kernel<kFmt><<<(int)blocks, 256, 0, st>>>(src, rows, cols, ld_src, transpose, dst, rows_pad, ldp, plane_stride, scale)));
    return check_launch("morl_split_planes");
}

extern "C" int morl_split_planes_multi(int fmt, const MorlSplitJob* jobs, int n_jobs, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_split_planes_multi: unknown plane format %d", fmt);
    MORL_REQUIRE(jobs, MORL_ERR_NULL, "morl_split_planes_multi: NULL pointer argument");
    MORL_REQUIRE(n_jobs > 0 && n_jobs <= MORL_SPLIT_MAX_JOBS, MORL_ERR_SHAPE, "morl_split_planes_multi: n_jobs=%d out of range", n_jobs);
    SplitJobs sj;
    memset(&sj, 0, sizeof(sj));
    long long max_total = 0;
    for (int i = 0; i < n_jobs; ++i) {
        const MorlSplitJob& j = jobs[i];
        MORL_REQUIRE(j.src && j.dst_planes, MORL_ERR_NULL, "morl_split_planes_multi: job %d has a NULL pointer", i);
        MORL_REQUIRE(j.rows > 0 && j.cols > 0 && j.rows_pad >= j.rows && j.ldp >= j.cols && j.ld_src > 0 &&
                         j.plane_stride >= (long long)j.rows_pad * j.ldp,
                     MORL_ERR_SHAPE, "morl_split_planes_multi: job %d bad shape rows=%d cols=%d rows_pad=%d ldp=%d", i, j.rows, j.cols, j.rows_pad, j.ldp);
        MORL_REQUIRE(!j.auto_scale || (j.scale && j.target_exp >= -14 && j.target_exp <= 15), MORL_ERR_SHAPE,
                     "morl_split_planes_multi: job %d auto_scale needs a scale pointer and -14 <= target_exp <= 15 (got %d)", i, j.target_exp);
        sj.job[i] = j;
        const long long t = (long long)j.rows_pad * j.ldp;
        if (t > max_total) max_total = t;
    }
    long long bx = (max_total + 255) / 256;
    if (bx > 148) bx = 148;
    bool any_auto = false;
    for (int i = 0; i < n_jobs; ++i) any_auto = any_auto || (jobs[i].auto_scale && jobs[i].scale);
    if (any_auto) {
        launch_k(split_amax_multi_kernel, dim3(n_jobs), dim3(1024), 0, static_cast<cudaStream_t>(stream), sj);
        int rca = check_launch("morl_split_planes_multi(amax)");
        if (rca) return rca;
    }
    MORL_DISPATCH_FMT(fmt, (launch_k(split_planes_multi_kernel<kFmt>, dim3(dim3((unsigned)bx, (unsigned)n_jobs)), dim3(256), 0, static_cast<cudaStream_t>(stream), sj)));
    return check_launch("morl_split_planes_multi");
}

extern "C" int morl_pairs_relu_split_planes(int fmt, const float* u, const float* v, int B, int W, int H, void* dst_planes, long long plane_stride,
                                            const float* scale, void* relu_bits_out, void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_pairs_relu_split_planes: unknown plane format %d", fmt);
    MORL_REQUIRE(u && v && dst_planes, MORL_ERR_NULL, "morl_pairs_relu_split_planes: NULL pointer argument");
    MORL_REQUIRE(B > 0 && W > 0 && H > 0 && H % 8 == 0 && plane_stride % 8 == 0 && plane_stride >= (long long)B * W * H, MORL_ERR_SHAPE,
                 "morl_pairs_relu_split_planes: bad shape B=%d W=%d H=%d", B, W, H);
    const long long total = (long long)B * W * (H / 8);
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (relu_bits_out)
        MORL_REQUIRE(H % 32 == 0 && H <= 256 && aligned16(relu_bits_out), MORL_ERR_SHAPE,
                     "morl_pairs_relu_split_planes: ReLU bit masks need H %% 32 == 0, H <= 256 (H=%d)", H);
    if (H == 256) {
        const int jsplit = W >= 16 ? 4 : 1;
        const long long tasks = (long long)B * jsplit;
        MORL_DISPATCH_FMT(fmt, (launch_k(pairs_relu_split_h256_kernel<kFmt>, dim3((unsigned)((tasks + 7) / 8)), dim3(256), 0, static_cast<cudaStream_t>(stream),
                                         u, v, B, W, static_cast<uint16_t*>(dst_planes), plane_stride, scale, static_cast<uint32_t*>(relu_bits_out), jsplit)));
        return check_launch("morl_pairs_relu_split_planes(h256)");
    }
    MORL_DISPATCH_FMT(fmt, (launch_k(pairs_relu_split_kernel<kFmt>, dim3((int)blocks), dim3(256), 0, static_cast<cudaStream_t>(stream), 
                               u, v, B, W, H, static_cast<uint16_t*>(dst_planes), plane_stride, scale, static_cast<uint32_t*>(relu_bits_out))));
    return check_launch("morl_pairs_relu_split_planes");
}

// Diagnostics: cycle counters of the K-major GEMM roles, accumulated over all CTAs and launches since the last reset
// (only when MORL_GEMM_STATS=1 was set before the first GEMM call).
extern "C" int morl_debug_gemm_stats(unsigned long long* out8, int reset) {
    using namespace morl;
    MORL_REQUIRE(out8, MORL_ERR_NULL, "morl_debug_gemm_stats: NULL pointer argument");
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out8, g_gemm_stats, 8 * sizeof(unsigned long long));
    if (reset) {
        unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        cudaMemcpyToSymbol(g_gemm_stats, z, sizeof(z));
    }
    return check_launch("morl_debug_gemm_stats");
}

namespace morl {
template <int FMT, int SPLIT>
static int launch_gemm_planes(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmBh, const CUtensorMap& tmC, const GemmArgs& g, bool pair,
                              int sms, cudaStream_t st) {
    constexpr size_t smem1 = KPlan<1, FMT>::kBytes, smem2 = KPlan<2, FMT>::kBytes;
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(gemm_planes_kernel<1, FMT, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
        cudaFuncSetAttribute(gemm_planes_kernel<2, FMT, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
        attr_set = true;
    }
    if (pair) {
        const int n_tiles = (g.M + 2 * kGemmBM - 1) / (2 * kGemmBM);
        const int pairs = n_tiles < sms / 2 ? n_tiles : sms / 2;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(2 * pairs);
        cfg.blockDim = dim3(kGemmThreads);
        cfg.dynamicSmemBytes = smem2;
        cfg.stream = st;
        cudaLaunchAttribute attr[2];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = g.pdl ? 2 : 1;
        cudaLaunchKernelEx(&cfg, gemm_planes_kernel<2, FMT, SPLIT>, tmA, tmB, tmBh, tmC, g);
    } else {
        const int n_tiles = (g.M + kGemmBM - 1) / kGemmBM;
        const int grid = n_tiles < sms ? n_tiles : sms;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kGemmThreads);
        cfg.dynamicSmemBytes = smem1;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = g.pdl ? 1 : 0;
        cudaLaunchKernelEx(&cfg, gemm_planes_kernel<1, FMT, SPLIT>, tmA, tmB, tmBh, tmC, g);
    }
    return check_launch("morl_gemm_planes_f32");
}
}  // namespace morl

extern "C" int morl_gemm_planes_f32(int fmt, const void* a_planes, long long a_plane_stride, const float* a_scale, const void* b_planes,
                                    long long b_plane_stride, const float* b_scale, int M, int N, int N_pad, int K, const float* bias, int relu,
                                    const void* relu_mask_plane0, int ld_mask, float* c_f32, int ldc, void* c_planes, int ldp, long long c_plane_stride,
                                    const float* c_scale, int reverse_tiles, int split_accumulators, const void* relu_bits_in, void* relu_bits_out,
                                    void* stream) {
    using namespace morl;
    MORL_REQUIRE(fmt_ok(fmt), MORL_ERR_UNSUPPORTED, "morl_gemm_planes_f32: unknown plane format %d", fmt);
    MORL_REQUIRE(a_planes && b_planes && (c_f32 || c_planes), MORL_ERR_NULL, "morl_gemm_planes_f32: NULL pointer argument");
    MORL_REQUIRE(M > 0 && N > 0 && K > 0 && N_pad >= N, MORL_ERR_SHAPE, "morl_gemm_planes_f32: bad shape M=%d N=%d N_pad=%d K=%d", M, N, N_pad, K);
    const int BK = fmt == MORL_FMT_F16X2 ? PlaneFmt<MORL_FMT_F16X2>::BK : PlaneFmt<MORL_FMT_BF16X3>::BK;
    MORL_REQUIRE(K % BK == 0 && N_pad % 32 == 0 && N_pad <= 256, MORL_ERR_UNSUPPORTED,
                 "morl_gemm_planes_f32: need K %% %d == 0, N_pad %% 32 == 0, N_pad <= 256 (K=%d N_pad=%d)", BK, K, N_pad);
    MORL_REQUIRE(aligned16(a_planes) && aligned16(b_planes), MORL_ERR_ALIGN, "morl_gemm_planes_f32: operand planes must be 16-byte aligned");
    MORL_REQUIRE(aligned16(relu_bits_in) && aligned16(relu_bits_out), MORL_ERR_ALIGN, "morl_gemm_planes_f32: ReLU bit masks must be 16-byte aligned");
    if (c_planes)
        MORL_REQUIRE(ldp % 32 == 0 && ldp >= N && ldp <= N_pad && aligned16(c_planes) && c_plane_stride % 8 == 0, MORL_ERR_SHAPE,
                     "morl_gemm_planes_f32: ldp=%d must be a multiple of 32 with N <= ldp <= N_pad", ldp);
    int sms = morl_device_sm_count();
    if (sms <= 0) sms = 148;
    // CTA pairs (tcgen05 cta_group::2) whenever there are at least two 128-row tiles; MORL_GEMM_FORCE_1CTA=1 keeps the 1-CTA kernel
    static const bool force_1cta = [] { const char* e = getenv("MORL_GEMM_FORCE_1CTA"); return e && e[0] == '1'; }();
    const bool pair = !force_1cta && M > kGemmBM && sms >= 2;
    const int ncta = pair ? 2 : 1;
    CUtensorMap tmA, tmB;
    int rc = make_plane_map(&tmA, fmt, a_planes, M, K, a_plane_stride, kGemmBM, BK);
    MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_planes_f32: cuTensorMapEncodeTiled(A) failed (%d)", rc);
    rc = make_plane_map(&tmB, fmt, b_planes, N_pad, K, b_plane_stride, N_pad / ncta, BK);
    MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_planes_f32: cuTensorMapEncodeTiled(B) failed (%d)", rc);
    CUtensorMap tmBh = tmB;  // half-width units of the tail split: boxes of N_pad / 4 rows
    if (pair && N_pad % 64 == 0) {
        rc = make_plane_map(&tmBh, fmt, b_planes, N_pad, K, b_plane_stride, N_pad / 4, BK);
        MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_planes_f32: cuTensorMapEncodeTiled(B half) failed (%d)", rc);
    }
    CUtensorMap tmC;
    memset(&tmC, 0, sizeof(tmC));
    if (c_planes) {  // store map of the re-split output: [P][M][ldp], box 32 cols x 32 rows x P planes (64-byte swizzle)
        rc = make_plane_map(&tmC, fmt, c_planes, M, ldp, c_plane_stride, 32, 32);
        MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_planes_f32: cuTensorMapEncodeTiled(C) failed (%d)", rc);
    }
    GemmArgs g;
    g.M = M; g.N = N; g.N_pad = N_pad; g.K = K;
    g.bias = bias; g.c_f32 = c_f32; g.ldc = ldc;
    g.c_planes = c_planes; g.ldp = ldp; g.plane_stride = c_plane_stride;
    g.mask = static_cast<const uint16_t*>(relu_mask_plane0); g.ld_mask = ld_mask; g.relu = relu;
    g.bits_in = static_cast<const uint32_t*>(relu_bits_in); g.bits_out = static_cast<uint32_t*>(relu_bits_out);
    {
        // TMA ring: A box + B box per stage; a narrow B box (the output layer: N_pad = 32) leaves room for a deeper ring, which is what
        // keeps enough bytes in flight per SM when a tile is four A boxes and almost no tensor work
        const uint32_t rowb = (uint32_t)BK * 2u, P = (uint32_t)fmt_planes(fmt);
        const uint32_t a_box = P * (uint32_t)kGemmBM * rowb;
        const uint32_t b_box = (P * (uint32_t)(N_pad / ncta) * rowb + 1023u) & ~1023u;
        const uint32_t room = fmt == MORL_FMT_F16X2 ? (pair ? KPlan<2, MORL_FMT_F16X2>::kOffC : KPlan<1, MORL_FMT_F16X2>::kOffC)
                                                    : (pair ? KPlan<2, MORL_FMT_BF16X3>::kOffC : KPlan<1, MORL_FMT_BF16X3>::kOffC);
        int n_st = (int)(room / (a_box + b_box));
        if (n_st > 8) n_st = 8;
        static const int st_env = [] { const char* e = getenv("MORL_GEMM_STAGES"); return e ? atoi(e) : 0; }();
        if (st_env > 0 && st_env < n_st) n_st = st_env;  // A/B measurements
        g.n_stages = n_st;
        g.b_stage = b_box;
    }
    g.a_scale = a_scale; g.b_scale = b_scale; g.c_scale = c_scale;
    g.reverse = reverse_tiles ? 1 : 0;
    // programmatic dependent launch between consecutive GEMMs of a chain (MORL_GEMM_PDL=0 disables it: A/B in profiles/r02_pdl_ab.txt)
    static const bool want_pdl = [] { const char* e = getenv("MORL_GEMM_PDL"); return !(e && e[0] == '0'); }();
    g.pdl = want_pdl ? 1 : 0;
    static const bool want_skip_b = [] { const char* e = getenv("MORL_GEMM_SKIPB"); return e && e[0] == '1'; }();
    g.skip_b = want_skip_b ? 1 : 0;
    // measured on B200 (profiles/r01_s3_l2hint_ab.txt): the hints do not help, so they are opt-in (MORL_GEMM_L2HINT=1)
    static const bool want_hint = [] { const char* e = getenv("MORL_GEMM_L2HINT"); return e && e[0] == '1'; }();
    g.l2_hint = want_hint ? 1 : 0;
    static const bool want_stats = [] { const char* e = getenv("MORL_GEMM_STATS"); return e && e[0] == '1'; }();
    g.stats = nullptr;
    if (want_stats) {
        void* sp = nullptr;
        cudaGetSymbolAddress(&sp, g_gemm_stats);
        g.stats = static_cast<unsigned long long*>(sp);
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // accumulator mode (see gemm_planes_kernel): per call; MORL_GEMM_SPLIT_ACC=0 / 1 overrides every call (A/B measurements)
    static const int split_env = [] { const char* e = getenv("MORL_GEMM_SPLIT_ACC"); return e ? (e[0] == '0' ? 0 : 1) : -1; }();
    const bool split_acc = split_env >= 0 ? split_env != 0 : split_accumulators != 0;
    if (fmt == MORL_FMT_F16X2)
        return split_acc ? launch_gemm_planes<MORL_FMT_F16X2, 1>(tmA, tmB, tmBh, tmC, g, pair, sms, st)
                         : launch_gemm_planes<MORL_FMT_F16X2, 0>(tmA, tmB, tmBh, tmC, g, pair, sms, st);
    return split_acc ? launch_gemm_planes<MORL_FMT_BF16X3, 1>(tmA, tmB, tmBh, tmC, g, pair, sms, st)
                     : launch_gemm_planes<MORL_FMT_BF16X3, 0>(tmA, tmB, tmBh, tmC, g, pair, sms, st);
}


extern "C" int morl_gemm_chain_supported(int fmt, int M, int K) {
    using namespace morl;
    return fmt_ok(fmt) && M >= 2 * kGemmBM && K == 256;
}

// Several 256-wide hidden layers (Linear + ReLU, planes in / planes out) of one or two networks in ONE persistent launch: job (c, l) computes
// act[c][l+1] = relu(act[c][l] . W[c][l]^T + bias[c][l]) exactly as morl_gemm_planes_f32 does (bit-identical), but a CTA pair takes its row tiles
// through all layers, so intermediate activations are re-read from L2 instead of HBM (csrc: gemm_chain_kernel).
extern "C" int morl_gemm_chain_f32(int fmt, int n_chains, int n_layers, const void* const* act_planes, long long act_plane_stride, const float* act_scale,
                                   const void* const* w_planes, long long w_plane_stride, const float* const* w_scales, const float* const* biases,
                                   int relu, const void* const* relu_bits_in, void* const* relu_bits_out, int M, int K, int k_first, void* stream) {
    using namespace morl;
    MORL_REQUIRE(act_planes && w_planes, MORL_ERR_NULL, "morl_gemm_chain_f32: NULL pointer argument");
    MORL_REQUIRE(n_chains >= 1 && n_chains <= 2 && n_layers >= 1 && n_chains * n_layers <= kChainMaxJobs, MORL_ERR_SHAPE,
                 "morl_gemm_chain_f32: need 1 <= n_chains <= 2 and n_chains * n_layers <= %d (got %d x %d)", kChainMaxJobs, n_chains, n_layers);
    MORL_REQUIRE(morl_gemm_chain_supported(fmt, M, K), MORL_ERR_UNSUPPORTED, "morl_gemm_chain_f32: unsupported configuration fmt=%d M=%d K=%d (256-wide layers, M >= 256)",
                 fmt, M, K);
    const int BK = fmt == MORL_FMT_F16X2 ? PlaneFmt<MORL_FMT_F16X2>::BK : PlaneFmt<MORL_FMT_BF16X3>::BK;
    if (k_first <= 0) k_first = K;
    MORL_REQUIRE(k_first % BK == 0 && k_first <= K, MORL_ERR_SHAPE, "morl_gemm_chain_f32: k_first=%d must be a multiple of %d and <= K", k_first, BK);
    ChainMaps maps;  // (host staging of the 3 x 8 tensor maps on this thread's stack -- the entry point stays re-entrant; copied into the kernel
                     // parameters by the launch)
    ChainArgs g;
    memset(&g, 0, sizeof(g));
    g.M = M; g.K = K; g.k_first = k_first; g.n_chains = n_chains; g.n_layers = n_layers; g.a_scale = act_scale; g.relu = relu ? 1 : 0;
    for (int c = 0; c < n_chains; ++c)
        for (int l = 0; l < n_layers; ++l) {
            const int job = c * n_layers + l;
            const void* a_in = act_planes[c * (n_layers + 1) + l];
            const void* a_out = act_planes[c * (n_layers + 1) + l + 1];
            MORL_REQUIRE(a_in && a_out && w_planes[job] && aligned16(a_in) && aligned16(a_out) && aligned16(w_planes[job]), MORL_ERR_NULL,
                         "morl_gemm_chain_f32: NULL or misaligned plane pointer (chain %d, layer %d)", c, l);
            // layer 0 may read a narrower input [P][M][k_first] (plane stride M * k_first) through weights [P][256][k_first]
            const int kj = l == 0 ? k_first : K;
            const long long a_stride = l == 0 ? (long long)M * k_first : act_plane_stride;
            const long long w_stride = l == 0 ? (long long)256 * k_first : w_plane_stride;
            int rc = make_plane_map(&maps.A[job], fmt, a_in, M, kj, a_stride, kGemmBM, BK);
            MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_chain_f32: cuTensorMapEncodeTiled(A) failed (%d)", rc);
            rc = make_plane_map(&maps.B[job], fmt, w_planes[job], 256, kj, w_stride, 128, BK);
            MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_chain_f32: cuTensorMapEncodeTiled(B) failed (%d)", rc);
            rc = make_plane_map(&maps.C[job], fmt, a_out, M, 256, act_plane_stride, 32, 32);
            MORL_REQUIRE(rc == 0, MORL_ERR_NO_DEVICE, "morl_gemm_chain_f32: cuTensorMapEncodeTiled(C) failed (%d)", rc);
            g.bias[job] = biases ? biases[job] : nullptr;
            g.b_scale[job] = w_scales ? w_scales[job] : nullptr;
            g.bits_out[job] = relu_bits_out ? static_cast<uint32_t*>(relu_bits_out[job]) : nullptr;
            g.bits_in[job] = relu_bits_in ? static_cast<const uint32_t*>(relu_bits_in[job]) : nullptr;
            MORL_REQUIRE(aligned16(g.bits_out[job]) && aligned16(g.bits_in[job]), MORL_ERR_ALIGN, "morl_gemm_chain_f32: ReLU bit masks must be 16-byte aligned");
        }
    g.n_stages = fmt == MORL_FMT_F16X2 ? KPlan<2, MORL_FMT_F16X2>::kStages : KPlan<2, MORL_FMT_BF16X3>::kStages;
    static const bool want_pdl = [] { const char* e = getenv("MORL_GEMM_PDL"); return !(e && e[0] == '0'); }();
    g.pdl = want_pdl ? 1 : 0;
    int sms = morl_device_sm_count();
    if (sms <= 0) sms = 148;
    const int n_tiles = (M + 2 * kGemmBM - 1) / (2 * kGemmBM);
    const int pairs = n_tiles < sms / 2 ? n_tiles : sms / 2;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g.pdl ? 2 : 1;
    if (fmt == MORL_FMT_F16X2) {
        constexpr size_t smem = KPlan<2, MORL_FMT_F16X2>::kBytes;
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(gemm_chain_kernel<MORL_FMT_F16X2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            attr_set = true;
        }
        cfg.dynamicSmemBytes = smem;
        cudaLaunchKernelEx(&cfg, gemm_chain_kernel<MORL_FMT_F16X2>, maps, g);
    } else {
        constexpr size_t smem = KPlan<2, MORL_FMT_BF16X3>::kBytes;
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(gemm_chain_kernel<MORL_FMT_BF16X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            attr_set = true;
        }
        cfg.dynamicSmemBytes = smem;
        cudaLaunchKernelEx(&cfg, gemm_chain_kernel<MORL_FMT_BF16X3>, maps, g);
    }
    return check_launch("morl_gemm_chain_f32");
}

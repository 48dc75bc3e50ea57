// tcgen05 / TMEM / TMA GEMM core with fused layer epilogues (sm_100a only).
//
// D[R, cout] = sum over K segments of A_s[R, K_s] * W_s[cout, K_s]^T, fp32-grade accuracy from
// fp16 tensor-core passes: every operand is stored as two fp16 planes (hi = fp16(v),
// lo = fp16(v - hi)) and each 16-wide k-step issues three MMAs into one TMEM accumulator,
//     Ahi*Whi + Ahi*Wlo + Alo*Whi          (the lo*lo term, ~2^-22 x 2^-22, is dropped),
// in a fixed order, with no split-K: a row's result depends only on that row's inputs, never on
// the tile it shares or on whether the encoder or the decoder computes it (SURVEY.md 7.3 item 2).
//
// CTA = one 128 x bn output tile (bn a multiple of 16, <= 256).  Warp roles:
//   warp 0 lane 0   TMA producer: per 64-wide k-block loads A hi/lo [128x64] and W hi/lo [bn x 64]
//                   (SWIZZLE_128B, K-major) into a multi-stage ring, mbarrier complete_tx
//   warp 1 lane 0   single-thread tcgen05.mma issuer (warp 1 also owns the TMEM allocation);
//                   tcgen05.commit frees stages and finally signals the accumulator
//   all 8 warps     epilogue (two warps per TMEM lane quarter): software-pipelined tcgen05.ld (32 lanes x 16
//                   columns) + operand prefetch -> fused epilogue -> staged in the idle ring -> coalesced stores
#include "epilogue.cuh"
#include "tc_common.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace {

struct TcParams {
    int kb[2];          // k-blocks per segment
    int bn;
    int stages;
    uint32_t tmem_cols;
    uint32_t idesc;
    uint32_t ring_bytes;   // max(stages * stage_bytes, epilogue staging), multiple of 1024
    EpiParams ep;
};

__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA0h, const __grid_constant__ CUtensorMap tmA0l,
               const __grid_constant__ CUtensorMap tmW0h, const __grid_constant__ CUtensorMap tmW0l,
               const __grid_constant__ CUtensorMap tmA1h, const __grid_constant__ CUtensorMap tmA1l,
               const __grid_constant__ CUtensorMap tmW1h, const __grid_constant__ CUtensorMap tmW1l,
               const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t ring = (raw + 1023u) & ~1023u;                     // SWIZZLE_128B needs 1024-B alignment
    const uint32_t w_plane = (uint32_t)p.bn * (BK * 2);
    const uint32_t stage_bytes = 2 * A_PLANE + 2 * w_plane;
    const uint32_t bars = ring + p.ring_bytes;                        // after the ring / staging area
    // barrier block: full[4] | empty[4] | tmem_full | tmem base address
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (MAX_STAGES + s); };
    const uint32_t tmem_full_bar = bars + 8u * (2 * MAX_STAGES);
    const uint32_t tmem_slot = bars + 8u * (2 * MAX_STAGES + 1);
    volatile uint32_t *tmem_slot_ptr =
        reinterpret_cast<volatile uint32_t *>(smem_raw + (tmem_slot - raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * p.bn;
    const int nkb = p.kb[0] + p.kb[1];

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA0h)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW0h)) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                     "r"(p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // every thread helps staging this tile's bias slice (read back by the epilogue from shared memory)
    float *sbias = reinterpret_cast<float *>(smem_raw + (bars + BAR_BLOCK - raw));
    if (p.ep.mode != EPI_RAW)
        for (int i = threadIdx.x; i < p.bn; i += NUM_THREADS) sbias[i] = (n0 + i < p.ep.cout) ? p.ep.bias[n0 + i] : 0.0f;
    fill_scale_tab(reinterpret_cast<float *>(smem_raw + (bars + BAR_BLOCK + 1024 + ROWTAB_BYTES - raw)), p.ep, threadIdx.x);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot_ptr;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch, bias
    // staging of static weights) overlapped the previous kernel's tail; its outputs are only read below.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        // all 32 lanes walk the loop, one elected lane issues (tc_common.cuh: elect_one)
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % p.stages;
            const uint32_t ph = (uint32_t)(kb / p.stages) & 1u;
            mbar_wait(empty_bar(s), ph ^ 1u);
            const uint32_t sa = ring + s * stage_bytes;
            const bool seg1 = kb >= p.kb[0];
            const int kk = (seg1 ? kb - p.kb[0] : kb) * BK;
            if (elect_one()) {
                mbar_expect_tx(full_bar(s), stage_bytes);
                tma_load_2d(sa, seg1 ? &tmA1h : &tmA0h, full_bar(s), kk, m0);
                tma_load_2d(sa + A_PLANE, seg1 ? &tmA1l : &tmA0l, full_bar(s), kk, m0);
                tma_load_2d(sa + 2 * A_PLANE, seg1 ? &tmW1h : &tmW0h, full_bar(s), kk, n0);
                tma_load_2d(sa + 2 * A_PLANE + w_plane, seg1 ? &tmW1l : &tmW0l, full_bar(s), kk, n0);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // all 32 lanes walk the loop, one elected lane issues (tc_common.cuh: elect_one)
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % p.stages;
            const uint32_t ph = (uint32_t)(kb / p.stages) & 1u;
            mbar_wait(full_bar(s), ph);
            tc_fence_after();
            const uint32_t sa = ring + s * stage_bytes;
            const uint64_t a_hi = make_smem_desc(sa);
            const uint64_t a_lo = make_smem_desc(sa + A_PLANE);
            const uint64_t w_hi = make_smem_desc(sa + 2 * A_PLANE);
            const uint64_t w_lo = make_smem_desc(sa + 2 * A_PLANE + w_plane);
            if (elect_one()) {
                // each k16 step advances the start address by 32 B (= 2 in 16-B units)
#pragma unroll
                for (int k = 0; k < BK / 16; ++k)
                    umma_f16(tmem_acc, a_hi + 2 * k, w_hi + 2 * k, p.idesc, (kb | k) != 0 ? 1u : 0u);
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) umma_f16(tmem_acc, a_hi + 2 * k, w_lo + 2 * k, p.idesc, 1u);
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) umma_f16(tmem_acc, a_lo + 2 * k, w_hi + 2 * k, p.idesc, 1u);
                umma_commit(empty_bar(s));   // frees the stage once these MMAs have read it
                if (kb == nkb - 1) umma_commit(tmem_full_bar);      // accumulator complete
            }
            __syncwarp();
        }
    }
    __syncwarp();
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    tile_epilogue(p.ep, sbias, ring, reinterpret_cast<RowTab *>(smem_raw + (bars + BAR_BLOCK + 1024 - raw)), tmem_acc, m0, n0,
                  p.bn, warp, lane);
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(p.tmem_cols)
                     : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;
bool g_use_pdl = true;

}  // namespace

void gemm_set_pdl(int on) { g_use_pdl = on != 0; }
int gemm_get_pdl() { return g_use_pdl ? 1 : 0; }

int gemm_tc_init() {
    static unsigned long long attr_mask = 0;
    if (lbic_first_use_on_device(attr_mask))
        LBIC_CUDA(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    if (g_encode_tiled) return 0;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    LBIC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess)
        return lbic_fail(LBIC_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

// h16 row-major [outer][ld_elems] matrix, logical inner extent `inner`; out-of-bounds box elements
// read as zero.
int make_tmap_2d(CUtensorMap *tm, const void *base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                 uint32_t box_inner, uint32_t box_outer) {
    LBIC_TRY(gemm_tc_init());
    if ((reinterpret_cast<uintptr_t>(base) & 15) || ((ld_elems * 2) & 15))
        return lbic_fail(LBIC_ERR_INVALID, "TMA operand must be 16-byte aligned (base %p, ld %llu)", base,
                         (unsigned long long)ld_elems);
    cuuint64_t gdim[2] = {inner, outer};
    cuuint64_t gstride[1] = {ld_elems * 2};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult rc = g_encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), gdim, gstride, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) return lbic_fail(LBIC_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)rc);
    return 0;
}

int gemm_tc_launch(const GemmCall &g, cudaStream_t st) {
    if (g.R <= 0) return 0;
    LBIC_TRY(gemm_tc_init());
    if (g.bn % 16 || g.bn < 16 || g.bn > 256) return lbic_fail(LBIC_ERR_INVALID, "bad tile N %d", g.bn);
    TcParams p;
    p.kb[0] = (g.K[0] + BK - 1) / BK;
    p.kb[1] = g.nseg > 1 ? (g.K[1] + BK - 1) / BK : 0;
    p.bn = g.bn;
    const int stage_bytes = 2 * A_PLANE + 2 * g.bn * BK * 2;
    int stages = (SMEM_LIMIT - SMEM_SLACK) / stage_bytes;
    if (stages > MAX_STAGES) stages = MAX_STAGES;
    if (stages < 2) return lbic_fail(LBIC_ERR_INVALID, "tile does not fit shared memory");
    p.stages = stages;
    uint32_t cols = 32;
    while ((int)cols < g.bn) cols <<= 1;
    p.tmem_cols = cols;
    // kind::f16 instruction descriptor: D=f32, A=B=h16, both K-major, N=bn, M=128
    p.idesc = (1u << 4) | ((uint32_t)(g.bn >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);   // D=f32, A=B=f16 (format 0), K-major
    p.ep = g.ep;
    const int s1 = g.nseg > 1 ? 1 : 0;
    dim3 grid((g.R + BM - 1) / BM, (g.cout + g.bn - 1) / g.bn);
    size_t ring_bytes = (size_t)stages * stage_bytes;
    if (ring_bytes < (size_t)STG_BYTES) ring_bytes = (STG_BYTES + 1023) / 1024 * 1024;   // epilogue staging lives in the ring
    p.ring_bytes = (uint32_t)ring_bytes;
    const size_t smem = ring_bytes + SMEM_SLACK;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = dim3(NUM_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_use_pdl ? 1 : 0;
    LBIC_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_kernel, *g.A[0].tm_hi, *g.A[0].tm_lo, *g.W[0].tm_hi, *g.W[0].tm_lo,
                                 *g.A[s1].tm_hi, *g.A[s1].tm_lo, *g.W[s1].tm_hi, *g.W[s1].tm_lo, p));
    count_launch(0);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

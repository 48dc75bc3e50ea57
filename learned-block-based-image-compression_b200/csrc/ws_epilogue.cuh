// Device-side pieces shared by the persistent warp-specialised kernels (gemm_ws.cu: the one pipeline body behind
// gemm_ws_kernel and gemm_flow_kernel; gemm_wave.cu: gemm_wave_kernel): shared-memory budget constants, CTA-pair
// helpers, and the epilogue of one 128 x bn tile by the eight epilogue warps (TMEM -> fused layer arithmetic -> staged,
// coalesced row stores).
#pragma once
#include "tc_common.cuh"

namespace {

constexpr int WS_THREADS = 320;
constexpr int WS_EPI_THREADS = 256;
constexpr int WS_MAX_BN = 192;
constexpr int WS_ACC_STRIDE = 256;          // TMEM columns between the two accumulators
constexpr int GC = 32;                      // columns per staged group
// One staging region, reused by two passes per group so that it stays small and the operand ring gets the space
// (the kernel is bound by L2 -> SM bandwidth; a third 64 KiB stage for the 256-wide pair tiles is worth more than a
// barrier):  pass F  = the fp32 plane (128 B per row),  pass HL = hi | lo | CDF-index planes (64 + 64 + 32 B per row).
constexpr int WF_STRIDE = GC * 4 + 16;      // 144 B: rows 16 B apart modulo 128 -> conflict-free 16-byte accesses
constexpr int WHL_STRIDE = 176;             // 128 + 48: 3 * 16 B apart modulo 128, also conflict-free
constexpr int WHL_LO = 64, WHL_IDX = 128;   // byte offsets of the lo / index planes within a pass-HL row
constexpr int WSTG_BYTES = BM * WHL_STRIDE; // 22,528 B
// GDN modes: pass HL needs no index plane (row stride 144 B) and the group's pre-activations (fp32, 128 x 128 B) get
// two cp.async buffers behind it, XOR-swizzled in 16-byte chunks instead of padded.
constexpr int WGDN_STRIDE = 144;
constexpr int WAUX_BUF = BM * GC * 4;       // 16,384 B
constexpr int WGDN_BYTES = BM * WGDN_STRIDE + 2 * WAUX_BUF;   // 51,200 B
constexpr int WS_BAR_BLOCK = 128;           // full[4] empty[4] acc_full[2] acc_empty[2] tmem slot
constexpr int WS_TAIL = WS_BAR_BLOCK + 2 * 1024 + ROWTAB_BYTES + STAB_BYTES;   // barriers, two bias slices, row table, scale table

struct WsParams {
    int kb[2];
    int bn, ntiles_n, total_tiles;
    int stages;
    uint32_t slot_bytes, ring_bytes, stg_bytes;   // stg_bytes: staging region (+ the GDN pre-activation buffer), multiple of 128
    uint32_t idesc;
    EpiParams ep;
};

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// ---- CTA-pair helpers -----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t cta) {
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
        "}" ::"r"(bar), "r"(cta) : "memory");
}
// TMA load issued by either CTA of a pair; the transaction bytes are credited to the LEADER's barrier (the shared
// window of the odd CTA differs from the even one in bit 24 of the cluster address).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap *tm, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// completion of all prior MMAs of the pair -> arrive on the barrier at this offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"((uint16_t)3) : "memory");
}

__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Epilogue of one 128 x bn tile by the eight epilogue warps (warps 2..9 of the CTA): per-tile setup (bias slice, row
// table) while the tile's mainloop is still running, then the accumulator is drained in 32-column groups.
struct EpiCtx {
    uint32_t stg;             // staging region (shared address)
    uint32_t acc_full_bar, acc_empty_bar, full_phase;
    uint32_t tmem_acc;        // TMEM address of this tile's accumulator (column base)
    float *sb;                // this tile's bias slice buffer
    RowTab *rt;
    const float *stab;
    uint32_t rank;            // CTA within its pair (0 = leader)
    // dataflow launch only: the epilogue's own side input (GDN pre-activations) is written by another layer of the same
    // launch; it may be fetched once *dep_cnt >= dep_target (the epilogue warps run ahead of the TMA producer)
    const int *dep_cnt = nullptr;
    int dep_target = 0;
    // second side input written inside the same launch: the entropy parameters (ksi) the QUANT epilogue reads
    const int *dep2_cnt = nullptr;
    int dep2_target = 0;
    unsigned long long *trace_acc = nullptr;   // debug: %globaltimer when the accumulator became available
    // the accumulator was produced by M = 64 MMAs (latency kernel, steps of at most 64 rows): row r sits in TMEM lane
    // 32 (r / 16) + r % 16, i.e. each warp's lanes 0-15 hold rows 16 q .. 16 q + 15 (scripts/mma_m64_layout.cu)
    int m64 = 0;
};

template <bool PAIR>
__device__ __forceinline__ void ws_tile_epilogue(const EpiParams &ep, int bn, int m0, int n0, const EpiCtx &cx) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ew = warp - 2;                 // 0..7
    const int q = warp & 3;                  // TMEM lane quarter (warp id % 4)
    const int sub = ew >> 2;                 // which 16-column chunk of a 32-column group
    const int et = threadIdx.x - 64;         // 0..255
    const int rl = cx.m64 ? q * 16 + (lane & 15) : q * 32 + lane;
    const int mode = ep.mode;
    const bool gdn = (mode == EPI_GDN || mode == EPI_IGDN);
    const uint32_t stg = cx.stg;
    const int r = m0 + rl;
    const bool row_ok = r < ep.R && !(cx.m64 && lane >= 16);
    const int rows_valid = (ep.R - m0) < BM ? (ep.R - m0) : BM;
    float *sb = cx.sb;
    // per-tile setup (overlaps the mainloop of this tile): bias slice, row table
    epi_bar();                           // previous tile's stores have finished reading rt / sbias
    if (mode != EPI_RAW)
        for (int i = et; i < bn; i += WS_EPI_THREADS) sb[i] = (n0 + i < ep.cout) ? ep.bias[n0 + i] : 0.0f;
    if (sub == 0 && row_ok) {
        const EpiRowDst d = epi_row_dst(ep, r);
        cx.rt->f32[rl] = reinterpret_cast<unsigned long long>(epi_f32_ptr(ep, d, n0));
        cx.rt->hilo[rl] = (unsigned long long)(d.hilo + n0);
        cx.rt->idx[rl] = reinterpret_cast<unsigned long long>(mode == EPI_QUANT && ep.idx ? ep.idx + d.blk * ep.M + n0 : nullptr);
    }
    epi_bar();
    const uint32_t lane_base = cx.tmem_acc + ((uint32_t)(q * 32) << 16);
    const int ngroups = (bn + GC - 1) / GC;   // the last group may hold a single 16-column chunk
    // Software pipeline over the 32-column groups: the TMEM load of group g+1 is issued before group g is
    // finished; in the GDN modes each thread also requests its own row's pre-activations of group g+1 (64
    // contiguous bytes) one group ahead, so that global-load latency hides behind a whole group of work.
    const int rsub = lane >> 3, c16 = lane & 7;
    const bool has_f32 = epi_has_f32(mode) && (mode != EPI_QUANT || ep.sym);
    const bool has_hilo = epi_has_hilo(mode);
    auto group_valid = [&](int g) {
        int nv = ep.cout - (n0 + g * GC);
        nv = nv < 0 ? 0 : (nv > GC ? GC : nv);
        return nv > bn - g * GC ? bn - g * GC : nv;
    };
    auto chunk_ok = [&](int g) {
        return row_ok && (n0 + g * GC + sub * 16) < ep.cout && (g * GC + sub * 16) < bn;
    };
    // GDN modes: the group's pre-activations arrive by cp.async with coalesced 16-byte lanes (4 rows x 128 B per
    // warp instruction; a row-per-thread read costs four times the L1 tag lookups and was measurably slower),
    // two groups ahead, into two swizzled buffers behind the staging region: under a saturated L2 a load
    // takes longer than one group of epilogue work.
    const int hl_stride = gdn ? WGDN_STRIDE : WHL_STRIDE;
    const uint32_t aux_base = stg + BM * WGDN_STRIDE;
    auto aux_issue = [&](int g) {
        const int nv = group_valid(g);
        const uint32_t buf = aux_base + (uint32_t)(g & 1) * WAUX_BUF;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int row = ew * 16 + j * 4 + rsub;
            const bool valid = row < rows_valid && c16 * 4 < nv;
            const float *src = valid ? ep.aux + (size_t)(m0 + row) * ep.ld_aux + n0 + g * GC + c16 * 4 : ep.aux;
            const uint32_t dst = buf + row * 128 + ((uint32_t)(c16 ^ (row & 7)) << 4);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // QUANT: the predicted scales (ksi[:, :M]) and means (ksi[:, M:]) of a 32-column group, same coalesced cp.async form,
    // scales into buffer 0 and means into buffer 1.  A row-per-thread read of the two 64-byte pieces costs 32 sectors per
    // warp instruction and made this epilogue 3.4x as long as the GDN one (profiles/r2_epilogue_ablation.log).  Single
    // buffered: the first 4 KiB of buffer 0 are also the tail of the hi / lo staging rows of this mode, which are only
    // written after every thread has read its side inputs (the barrier of pass F lies between).
    const bool quant = (mode == EPI_QUANT);
    auto aux_issue_q = [&](int g) {
        const int nv = group_valid(g);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const uint32_t buf = aux_base + (uint32_t)half * WAUX_BUF;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int row = ew * 16 + j * 4 + rsub;
                const bool valid = row < rows_valid && c16 * 4 < nv;
                const float *src = valid ? ep.aux + (size_t)(m0 + row) * ep.ld_aux + half * ep.M + n0 + g * GC + c16 * 4 : ep.aux;
                const uint32_t dst = buf + row * 128 + ((uint32_t)(c16 ^ (row & 7)) << 4);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    uint32_t accA[16], accB[16];
    if (gdn) {                                       // overlaps the wait for the accumulator
        if (cx.dep_cnt) {
            if (et == 0) {
                uint32_t spins = 0;
                while (ld_acquire_gpu(cx.dep_cnt) < cx.dep_target) {
                    __nanosleep(64);
                    if (++spins > (1u << 24)) __trap();
                }
            }
            epi_bar();
        }
        aux_issue(0);
        if (ngroups > 1) {
            aux_issue(1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        epi_bar();
    }
    if (mode == EPI_QUANT && cx.dep2_cnt) {              // ksi rows of this row block are complete (overlaps the mainloop)
        if (et == 0) {
            uint32_t spins = 0;
            while (ld_acquire_gpu(cx.dep2_cnt) < cx.dep2_target) {
                __nanosleep(32);
                if (++spins > (1u << 24)) __trap();
            }
        }
        epi_bar();
    }
    if (quant) aux_issue_q(0);     // the first group's scales / means travel while the mainloop is still running
    mbar_wait(cx.acc_full_bar, cx.full_phase);
    tc_fence_after();
    if (cx.trace_acc) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(*cx.trace_acc));
    tmem_ld_issue(lane_base + (uint32_t)(sub * 16), accA);
    for (int g = 0; g < ngroups; ++g) {
        const int g0 = g * GC;
        const int nvalid = group_valid(g);
        const bool even = (g & 1) == 0;
        const bool ok = chunk_ok(g);
        EpiOut<16> o;
        if (quant) {                     // (the staging rows are free: barrier at the end of the previous group / tile setup)
            if (g > 0) aux_issue_q(g);
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            epi_bar();
        }
        // phase A: this warp's 16-column chunk of the group
        {
            const int c = n0 + g0 + sub * 16;
            EpiPre<16> pre;
            if (ok) {
                if (gdn) {
                    const uint32_t src = aux_base + (uint32_t)(g & 1) * WAUX_BUF + rl * 128;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint4 v = lds128(src + ((uint32_t)((sub * 4 + i) ^ (rl & 7)) << 4));
                        pre.a[4 * i] = __uint_as_float(v.x); pre.a[4 * i + 1] = __uint_as_float(v.y);
                        pre.a[4 * i + 2] = __uint_as_float(v.z); pre.a[4 * i + 3] = __uint_as_float(v.w);
                    }
                } else if (quant) {
                    const uint32_t src = aux_base + rl * 128;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t off = (uint32_t)((sub * 4 + i) ^ (rl & 7)) << 4;
                        const uint4 va = lds128(src + off), vb = lds128(src + WAUX_BUF + off);
                        pre.a[4 * i] = __uint_as_float(va.x); pre.a[4 * i + 1] = __uint_as_float(va.y);
                        pre.a[4 * i + 2] = __uint_as_float(va.z); pre.a[4 * i + 3] = __uint_as_float(va.w);
                        pre.a2[4 * i] = __uint_as_float(vb.x); pre.a2[4 * i + 1] = __uint_as_float(vb.y);
                        pre.a2[4 * i + 2] = __uint_as_float(vb.z); pre.a2[4 * i + 3] = __uint_as_float(vb.w);
                    }
                } else {
                    epi_prefetch<16>(ep, r, c, pre);
                }
            }
            if (even) tmem_ld_wait(accA); else tmem_ld_wait(accB);
            if (g + 1 < ngroups) {
                if (even) tmem_ld_issue(lane_base + (uint32_t)(g0 + GC + sub * 16), accB);
                else tmem_ld_issue(lane_base + (uint32_t)(g0 + GC + sub * 16), accA);
            } else {
                // all TMEM reads of this accumulator are done: hand it back to the MMA issuer
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (PAIR) mbar_arrive_remote(cx.acc_empty_bar, 0);
                    else mbar_arrive(cx.acc_empty_bar);
                }
            }
            if (ok) {
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(even ? accA[i] : accB[i]);
                epi_compute<16>(ep, sb + g0 + sub * 16, v, pre, o, cx.stab);
            }
        }
        const int gc = sub * 16;
        auto stage_hl = [&]() {
            const uint32_t hrow = stg + rl * hl_stride + gc * 2;
            sts128(hrow, o.hi[0], o.hi[1], o.hi[2], o.hi[3]);
            sts128(hrow + 16, o.hi[4], o.hi[5], o.hi[6], o.hi[7]);
            sts128(hrow + WHL_LO, o.lo[0], o.lo[1], o.lo[2], o.lo[3]);
            sts128(hrow + WHL_LO + 16, o.lo[4], o.lo[5], o.lo[6], o.lo[7]);
            if (mode == EPI_QUANT) sts128(stg + rl * WHL_STRIDE + WHL_IDX + gc, o.idx[0], o.idx[1], o.idx[2], o.idx[3]);
        };
        auto store_hl = [&]() {
            const int c8 = lane & 3;                 // 16-byte chunk within the 64-byte plane row
            const bool is_lo = (lane >> 2) & 1;
            // all shared-memory reads of the four rows first (any row of the staging area / row table may be read; only
            // the stores are predicated), then the stores: four independent load -> store chains instead of one
            if (c8 * 8 < nvalid) {
                h16 *base = (is_lo ? ep.out_lo : ep.out_hi) + g0 + c8 * 8;
                const uint32_t src = stg + (is_lo ? WHL_LO : 0) + c8 * 16;
                uint4 v[4];
                unsigned long long off[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int row = ew * 16 + j * 4 + rsub;
                    v[j] = lds128(src + row * hl_stride);
                    off[j] = cx.rt->hilo[row];
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (ew * 16 + j * 4 + rsub < rows_valid)
                        *reinterpret_cast<uint4 *>(base + off[j]) = v[j];
            }
            if (mode == EPI_QUANT && ep.idx && c16 < 2 && c16 * 16 < nvalid) {      // 2 x 16 B per row
                uint4 v[4];
                unsigned long long dst[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int row = ew * 16 + j * 4 + rsub;
                    v[j] = lds128(stg + row * WHL_STRIDE + WHL_IDX + c16 * 16);
                    dst[j] = cx.rt->idx[row];
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (ew * 16 + j * 4 + rsub < rows_valid)
                        *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(dst[j]) + g0 + c16 * 16) = v[j];
            }
        };
        if (has_f32) {
            // pass F: stage the fp32 plane, then coalesced stores, 4 rows (128 B each) per warp instruction
            if (ok) {
                const uint32_t d = stg + rl * WF_STRIDE + gc * 4;
#pragma unroll
                for (int i = 0; i < 16; i += 4)
                    sts128(d + i * 4, __float_as_uint(o.f[i]), __float_as_uint(o.f[i + 1]),
                           __float_as_uint(o.f[i + 2]), __float_as_uint(o.f[i + 3]));
            }
            epi_bar();
            if (c16 * 4 < nvalid) {
                uint4 v[4];
                unsigned long long dst[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int row = ew * 16 + j * 4 + rsub;
                    v[j] = lds128(stg + row * WF_STRIDE + c16 * 16);
                    dst[j] = cx.rt->f32[row];
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (ew * 16 + j * 4 + rsub < rows_valid)
                        *reinterpret_cast<uint4 *>(reinterpret_cast<float *>(dst[j]) + g0 + c16 * 4) = v[j];
            }
            if (has_hilo) {
                epi_bar();               // the fp32 stores have read the staging area
                if (ok) stage_hl();
                epi_bar();
                if (nvalid > 0) store_hl();
            }
        } else {
            if (ok) stage_hl();
            epi_bar();                   // (GDN: every thread has also read its pre-activations of this group)
            if (gdn && g + 2 < ngroups) aux_issue(g + 2);   // into the buffer this group has just released
            if (nvalid > 0) store_hl();
            if (gdn && g + 1 < ngroups) {                   // this thread's share of group g+1 has landed
                if (g + 2 < ngroups) asm volatile("cp.async.wait_group 1;" ::: "memory");
                else asm volatile("cp.async.wait_group 0;" ::: "memory");
            }
        }
        if (g + 1 < ngroups) epi_bar();   // stores have read the staging area; next pre-activations visible
    }
}

}  // namespace

// Warp-specialised, persistent tcgen05 GEMM: the throughput kernel for large wavefront steps.
//
// profiles/r1_chain_trace.md showed that in gemm_tc_kernel the epilogue (TMEM -> fused math -> staged, coalesced
// stores) takes about as long as the mainloop, and that every tile also pays prologue / pipeline fill / drain.  Here a
// CTA stays resident, loops over output tiles, and runs the three stages of consecutive tiles concurrently:
//
//   warp 0 lane 0   TMA producer: runs ahead over tile boundaries, gated only by the stage ring
//   warp 1 lane 0   tcgen05.mma issuer: accumulates tile i into TMEM buffer (i & 1) as soon as the epilogue has
//                   drained that buffer (acc_empty), tcgen05.commit -> acc_full
//   warps 2..9      epilogue of tile i-1 from the other TMEM buffer, in 32-column groups staged through a small
//                   dedicated shared-memory area (so the ring keeps streaming), then coalesced row stores
//
// Single-CTA tiles are 128 x bn with bn <= 192 (2 stages of 80 KiB + 22 KiB staging, 51 KiB in the GDN modes).  Same
// operand planes, same k order and same epilogue arithmetic as gemm_tc_kernel: results are bit-identical.
//
// PAIR = true is the CTA-pair form (cluster of 2, tcgen05 cta_group::2).  The single-CTA kernel turned out to be bound
// by L2 -> SM bandwidth, not by the tensor pipe: a 128 x 192 tile moves (128 + 192) x 64 x 4 B per k-block for 12 MMAs,
// i.e. 71 B/clk/SM against a chip-wide L2 limit of ~43 B/clk/SM (profiles/r1_l2_bound.md).  A pair computes a 256 x bn
// tile: each CTA loads its own 128 activation rows but only HALF of the weight tile, and the tensor cores of both SMs
// read both halves, which cuts the bytes per flop by 30 %.  The leader CTA (rank 0) issues every MMA; full barriers live
// in the leader, empty / acc_full barriers are signalled in both CTAs by multicast commits, and both epilogues report
// to the leader's acc_empty barrier.  Pair tiles are up to 256 wide with 3 stages of 56-64 KiB.
//
// Both kernels of this file run one device body, ws_pipeline<PAIR, Tiles>.  A tile source says what each tile is:
// LayerTiles walks the tiles of one layer (gemm_ws_kernel, one launch per layer); StepTiles walks the tiles of all
// layers of a wavefront step in one list, with the layers ordered per row block by global counters (gemm_flow_kernel).
#include "ws_epilogue.cuh"

#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace {

// ---------------------------------------------------------------------------------------------------------------
// Dataflow form: ONE launch runs a whole range of layers of a wavefront step.
//
// With one launch per layer every launch ends with the epilogue of its last wave of tiles running alone (~12 us of
// a ~70 us launch), pays a prologue, and rounds its tile count up to whole waves of 74 CTA pairs.  Here the tiles of all
// layers form one list in layer order, the persistent CTA pairs walk it round-robin, and the only synchronisation
// between layers is per 256-row block: a tile of layer l may load its operands once every tile of the layers it reads
// from has been stored for the same row block (a counter per (layer, row block), bumped by each CTA after its stores
// and a __threadfence, polled with ld.acquire by the TMA producer).  A pair only ever waits for tiles with a smaller
// index, and every pair walks the list in order, so the scheme cannot deadlock.  Same tiles, same arithmetic, same
// results as the per-layer launches.
// ---------------------------------------------------------------------------------------------------------------
constexpr int FLOW_MAX_LAYERS = 18;
constexpr int FLOW_SLOT = 2 * A_PLANE + 2 * (WS_MAX_BN / 2) * BK * 2;   // 56 KiB: 128 activation rows + 96 weight rows, hi + lo
constexpr int FLOW_STAGES = 3;
constexpr int FLOW_TAIL = WS_TAIL + 256;    // + the current layer's EpiParams
constexpr int FLOW_THREADS = WS_THREADS + 32;   // + one warp that publishes finished tiles (the gpu-scope release
                                                // waits for the tile's stores to drain; the epilogue warps do not)
constexpr size_t FLOW_SMEM = 1024 + (size_t)FLOW_STAGES * FLOW_SLOT + WGDN_BYTES + FLOW_TAIL;
static_assert(FLOW_SMEM <= (size_t)SMEM_LIMIT, "flow kernel shared memory");
static_assert(sizeof(EpiParams) <= 256, "EpiParams must fit its shared-memory slot");

struct FlowParams {
    const ChainLayer *layers;     // device table indexed by absolute layer id
    int *counters;                // [n_layers][n_rb], zero at launch
    int l0, n_layers, n_rb, R, variant, total_tiles;
    StepDesc step;
    int pre[FLOW_MAX_LAYERS + 1]; // prefix sums of ntn (tiles of one row block over the layers)
    int ntn[FLOW_MAX_LAYERS];     // column tiles per layer
    int dep[FLOW_MAX_LAYERS][2];  // relative layer indices this layer reads from, -1 = none
};

// tile index -> (layer, row block, column tile); the list runs layer by layer, each layer row block by row block
__device__ __forceinline__ void flow_tile(const FlowParams &p, int t, int &li, int &rb, int &nt) {
    li = 0;
    while (t >= p.n_rb * p.pre[li + 1]) ++li;
    const int v = t - p.n_rb * p.pre[li];
    rb = v / p.ntn[li];
    nt = v - rb * p.ntn[li];
}

// ---------------------------------------------------------------------------------------------------------------
// Tile sources.  Each says, per tile, where its operands, width and epilogue parameters come from, and gives the
// stage ring's shape.  Only StepTiles has dependencies between tiles and a publisher warp (DATAFLOW).
// ---------------------------------------------------------------------------------------------------------------
struct WsTile {
    int li, rb, nt, bn;       // layer within the launch, row block (one tile's 128 or 256 rows), column tile, tile width
};
struct WsMaps {
    const CUtensorMap *a_hi, *a_lo, *w_hi, *w_lo;
};

// One layer per launch: operands in the eight __grid_constant__ maps of gemm_ws_kernel, stage count and slot size
// chosen per launch by gemm_ws_launch.
struct LayerTiles {
    static constexpr bool DATAFLOW = false;
    const WsParams &p;
    const CUtensorMap &A0h, &A0l, &W0h, &W0l, &A1h, &A1l, &W1h, &W1l;   // [K segment 0 | 1] x [A hi, A lo, W hi, W lo]

    __device__ __forceinline__ int total_tiles() const { return p.total_tiles; }
    __device__ __forceinline__ int stages() const { return p.stages; }
    __device__ __forceinline__ uint32_t slot_bytes() const { return p.slot_bytes; }
    __device__ __forceinline__ uint32_t ring_bytes() const { return p.ring_bytes; }
    __device__ __forceinline__ uint32_t stg_bytes() const { return p.stg_bytes; }
    __device__ __forceinline__ void load_scale_tab(float *stab) const { fill_scale_tab(stab, p.ep, threadIdx.x); }
    __device__ __forceinline__ void prefetch_maps() const {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&A0h)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&W0h)) : "memory");
    }
    __device__ __forceinline__ WsTile tile(int t) const { return {0, t / p.ntiles_n, t % p.ntiles_n, p.bn}; }
    __device__ __forceinline__ int kb0(const WsTile &) const { return p.kb[0]; }
    __device__ __forceinline__ int nkb(const WsTile &) const { return p.kb[0] + p.kb[1]; }
    __device__ __forceinline__ WsMaps maps(const WsTile &, int seg) const {
        return seg ? WsMaps{&A1h, &A1l, &W1h, &W1l} : WsMaps{&A0h, &A0l, &W0h, &W0l};
    }
    __device__ __forceinline__ uint32_t idesc(const WsTile &) const { return p.idesc; }
    __device__ __forceinline__ const EpiParams &epilogue(const WsTile &, EpiCtx &, EpiParams *, int &) const {
        return p.ep;
    }
};

// The layers [l0, l0 + n_layers) of a wavefront step in one list (gemm_flow_kernel): per-layer maps and tile widths
// from the device ChainLayer table, a fixed ring of FLOW_STAGES x FLOW_SLOT.
template <bool PAIR>
struct StepTiles {
    static constexpr bool DATAFLOW = true;
    static constexpr int CTAS = PAIR ? 2 : 1;          // CTAs that store (and publish) each tile
    const FlowParams &p;

    __device__ __forceinline__ const ChainLayer &layer(int li) const { return p.layers[p.l0 + li]; }
    __device__ __forceinline__ int *counter(int li, int rb) const { return p.counters + (size_t)li * p.n_rb + rb; }

    __device__ __forceinline__ int total_tiles() const { return p.total_tiles; }
    __device__ __forceinline__ static constexpr int stages() { return FLOW_STAGES; }
    __device__ __forceinline__ static constexpr uint32_t slot_bytes() { return FLOW_SLOT; }
    __device__ __forceinline__ static constexpr uint32_t ring_bytes() { return FLOW_STAGES * FLOW_SLOT; }
    __device__ __forceinline__ static constexpr uint32_t stg_bytes() { return WGDN_BYTES; }
    __device__ __forceinline__ void load_scale_tab(float *stab) const {
        const float *gtab = layer(0).ep.scale_tab;
        if (gtab && threadIdx.x < 64) stab[threadIdx.x] = gtab[threadIdx.x];
    }
    __device__ __forceinline__ WsTile tile(int t) const {
        WsTile tl;
        flow_tile(p, t, tl.li, tl.rb, tl.nt);
        tl.bn = layer(tl.li).bn_v[p.variant];
        return tl;
    }
    __device__ __forceinline__ int kb0(const WsTile &tl) const { return layer(tl.li).kb[0]; }
    __device__ __forceinline__ int nkb(const WsTile &tl) const {
        const ChainLayer &L = layer(tl.li);
        return L.kb[0] + (L.nseg > 1 ? L.kb[1] : 0);
    }
    __device__ __forceinline__ WsMaps maps(const WsTile &tl, int seg) const {
        const ChainLayer &L = layer(tl.li);
        return {&L.tmA[seg][0], &L.tmA[seg][1], &L.tmW[p.variant][seg][0], &L.tmW[p.variant][seg][1]};
    }
    __device__ __forceinline__ uint32_t idesc(const WsTile &tl) const {
        return (1u << 4) | ((uint32_t)(tl.bn >> 3) << 17) | ((uint32_t)(CTAS * BM >> 4) << 24);
    }
    // TMA producer: wait until the layers this tile reads from have stored its row block (both CTAs of every pair)
    __device__ __forceinline__ void wait_inputs(const WsTile &tl, int lane) const {
        for (int d = 0; d < 2; ++d) {
            const int dl = p.dep[tl.li][d];
            if (dl < 0) continue;
            const int *cnt = counter(dl, tl.rb);
            const int target = CTAS * p.ntn[dl];
            if (lane == 0) {
                uint32_t spins = 0;
                while (ld_acquire_gpu(cnt) < target) {
                    __nanosleep(64);
                    if (++spins > (1u << 24)) __trap();     // a broken dependency must fail the launch, not hang
                }
            }
            __syncwarp();
        }
        asm volatile("fence.proxy.async;" ::: "memory");   // generic-proxy stores of other CTAs -> our TMA reads
    }
    // Epilogue warps: the tile's side inputs written by other layers of the launch (c.dep*), and its EpiParams.  On a
    // layer change the layer's description, with this launch's row count and step, is copied into shared memory (s_ep;
    // cur: the layer held there).
    __device__ __forceinline__ const EpiParams &epilogue(const WsTile &tl, EpiCtx &c, EpiParams *s_ep, int &cur) const {
        if (tl.li != cur) {
            if (cur >= 0) epi_bar();     // every epilogue thread is past the previous tile (which read the old copy)
            constexpr int NW = (int)(sizeof(EpiParams) / 4);
            constexpr int OFF_R = (int)(offsetof(EpiParams, R) / 4), OFF_STEP = (int)(offsetof(EpiParams, step) / 4);
            constexpr int NSTEP = (int)(sizeof(StepDesc) / 4);
            const int et = threadIdx.x - 64;
            const uint32_t *g = reinterpret_cast<const uint32_t *>(&layer(tl.li).ep);
            const uint32_t *sw = reinterpret_cast<const uint32_t *>(&p.step);
            if (et < NW) {
                uint32_t w = g[et];
                if (et == OFF_R) w = (uint32_t)p.R;
                else if (et >= OFF_STEP && et < OFF_STEP + NSTEP) w = sw[et - OFF_STEP];
                reinterpret_cast<uint32_t *>(s_ep)[et] = w;
            }
            cur = tl.li;
            epi_bar();
        }
        const int dl = p.dep[tl.li][0];
        c.dep_cnt = dl >= 0 ? counter(dl, tl.rb) : nullptr;
        c.dep_target = dl >= 0 ? CTAS * p.ntn[dl] : 0;
        const int dl2 = p.dep[tl.li][1];
        c.dep2_cnt = dl2 >= 0 ? counter(dl2, tl.rb) : nullptr;
        c.dep2_target = dl2 >= 0 ? CTAS * p.ntn[dl2] : 0;
        return *s_ep;
    }
};

// ---------------------------------------------------------------------------------------------------------------
// The persistent pipeline: shared-memory carve-up, barriers, TMEM, and the producer / issuer / epilogue roles (plus,
// for a DATAFLOW tile source, warp 10: the publisher).
// ---------------------------------------------------------------------------------------------------------------
template <bool PAIR, class Tiles>
__device__ __forceinline__ void ws_pipeline(const Tiles &T) {
    constexpr bool FLOW = Tiles::DATAFLOW;
    constexpr int CTAS = PAIR ? 2 : 1;
    constexpr int TILE_ROWS = CTAS * BM;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t ring = (raw + 1023u) & ~1023u;
    const uint32_t stg = ring + T.ring_bytes();                 // dedicated epilogue staging (1024-aligned)
    const uint32_t bars = stg + T.stg_bytes();
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (MAX_STAGES + s); };
    auto acc_full = [&](int a) { return bars + 8u * (2 * MAX_STAGES + a); };
    auto acc_empty = [&](int a) { return bars + 8u * (2 * MAX_STAGES + 2 + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * MAX_STAGES + 4);
    auto tile_done = [&](int a) { return bars + 8u * (2 * MAX_STAGES + 6 + a); };   // DATAFLOW only
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(smem_raw + (tmem_slot - raw));
    float *sbias = reinterpret_cast<float *>(smem_raw + (bars + WS_BAR_BLOCK - raw));        // [2][256]
    RowTab *rt = reinterpret_cast<RowTab *>(smem_raw + (bars + WS_BAR_BLOCK + 2048 - raw));
    float *stab = reinterpret_cast<float *>(rt + 1);
    EpiParams *s_ep = reinterpret_cast<EpiParams *>(stab + 64);   // DATAFLOW only: the current layer's EpiParams
    T.load_scale_tab(stab);                                        // visible after the setup barrier below

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;            // CTA within its pair, 0 = leader
    const int tile_first = (int)(blockIdx.x / CTAS);
    const int tile_stride = (int)(gridDim.x / CTAS);

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < T.stages(); ++s) {
            mbar_init(full_bar(s), CTAS);          // pair: one arrival per CTA's producer, on the leader
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(acc_full(a), 1);
            mbar_init(acc_empty(a), CTAS * (WS_EPI_THREADS / 32));
            if constexpr (FLOW) mbar_init(tile_done(a), WS_EPI_THREADS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if constexpr (!FLOW) T.prefetch_maps();
    }
    if (warp == 1) {
        if (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    asm volatile("griddepcontrol.wait;" ::: "memory");             // PDL: see gemm_tc.cu
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        // all 32 lanes walk the loop, one elected lane issues (tc_common.cuh: elect_one)
        uint32_t it = 0;
        for (int t = tile_first; t < T.total_tiles(); t += tile_stride) {
            const WsTile tl = T.tile(t);
            const int w_rows = PAIR ? tl.bn / 2 : tl.bn;            // weight rows this CTA loads per stage
            const int m0 = tl.rb * TILE_ROWS + (int)rank * BM;
            const int n0 = tl.nt * tl.bn + (int)rank * w_rows;
            if constexpr (FLOW) T.wait_inputs(tl, lane);
            const int kb0 = T.kb0(tl), nkb = T.nkb(tl);
            const uint32_t w_plane = (uint32_t)w_rows * (BK * 2);
            const uint32_t stage_tx = (2 * A_PLANE + 2 * w_plane) * (uint32_t)CTAS;
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % T.stages();
                const uint32_t ph = (it / T.stages()) & 1u;
                mbar_wait(empty_bar(s), ph ^ 1u);
                const uint32_t sa = ring + s * T.slot_bytes();
                const int seg = kb >= kb0 ? 1 : 0;
                const int kk = (seg ? kb - kb0 : kb) * BK;
                if (elect_one()) {
                    const WsMaps m = T.maps(tl, seg);
                    if (PAIR) {
                        if (rank == 0) mbar_expect_tx(full_bar(s), stage_tx);
                        else mbar_arrive_remote(full_bar(s), 0);
                        tma_load_2d_pair(sa, m.a_hi, full_bar(s), kk, m0);
                        tma_load_2d_pair(sa + A_PLANE, m.a_lo, full_bar(s), kk, m0);
                        tma_load_2d_pair(sa + 2 * A_PLANE, m.w_hi, full_bar(s), kk, n0);
                        tma_load_2d_pair(sa + 2 * A_PLANE + w_plane, m.w_lo, full_bar(s), kk, n0);
                    } else {
                        mbar_expect_tx(full_bar(s), stage_tx);
                        tma_load_2d(sa, m.a_hi, full_bar(s), kk, m0);
                        tma_load_2d(sa + A_PLANE, m.a_lo, full_bar(s), kk, m0);
                        tma_load_2d(sa + 2 * A_PLANE, m.w_hi, full_bar(s), kk, n0);
                        tma_load_2d(sa + 2 * A_PLANE + w_plane, m.w_lo, full_bar(s), kk, n0);
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {       // all 32 lanes walk the loop, one elected lane issues (tc_common.cuh: elect_one)
            uint32_t it = 0, ti = 0;
            for (int t = tile_first; t < T.total_tiles(); t += tile_stride, ++ti) {
                const WsTile tl = T.tile(t);
                const int nkb = T.nkb(tl);
                const uint32_t w_plane = (uint32_t)(PAIR ? tl.bn / 2 : tl.bn) * (BK * 2);
                const uint32_t idesc = T.idesc(tl);
                const uint32_t a = ti & 1u;
                mbar_wait(acc_empty(a), ((ti >> 1) & 1u) ^ 1u);      // the epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t tmem_acc = tmem_base + a * WS_ACC_STRIDE;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % T.stages();
                    const uint32_t ph = (it / T.stages()) & 1u;
                    mbar_wait(full_bar(s), ph);
                    tc_fence_after();
                    const uint32_t sa = ring + s * T.slot_bytes();
                    const uint64_t a_hi = make_smem_desc(sa);
                    const uint64_t a_lo = make_smem_desc(sa + A_PLANE);
                    const uint64_t w_hi = make_smem_desc(sa + 2 * A_PLANE);
                    const uint64_t w_lo = make_smem_desc(sa + 2 * A_PLANE + w_plane);
                    auto mma = [&](uint64_t ad, uint64_t wd, uint32_t acc) {
                        if (PAIR) umma_f16_pair(tmem_acc, ad, wd, idesc, acc);
                        else umma_f16(tmem_acc, ad, wd, idesc, acc);
                    };
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) mma(a_hi + 2 * k, w_hi + 2 * k, (kb | k) != 0 ? 1u : 0u);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) mma(a_hi + 2 * k, w_lo + 2 * k, 1u);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) mma(a_lo + 2 * k, w_hi + 2 * k, 1u);
                        if (PAIR) umma_commit_pair(empty_bar(s)); else umma_commit(empty_bar(s));
                        if (kb == nkb - 1) { if (PAIR) umma_commit_pair(acc_full(a)); else umma_commit(acc_full(a)); }
                    }
                    __syncwarp();
                }
            }
        }
    } else if (FLOW && warp == 2 + WS_EPI_THREADS / 32) {
        // ---- publisher: tile (layer, row block) of this CTA is stored -> bump its counter with gpu-scope release ----
        if constexpr (FLOW) {
            if (lane == 0) {
                uint32_t ti = 0;
                for (int t = tile_first; t < T.total_tiles(); t += tile_stride, ++ti) {
                    const WsTile tl = T.tile(t);
                    mbar_wait(tile_done(ti & 1u), (ti >> 1) & 1u);       // all eight epilogue warps have issued their stores
                    asm volatile("fence.proxy.async;" ::: "memory");
                    asm volatile("fence.acq_rel.gpu;" ::: "memory");
                    asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(T.counter(tl.li, tl.rb)) : "memory");
                }
            }
        }
    } else {
        // ---- epilogue warps 2..9 ----------------------------------------------------------------------
        uint32_t ti = 0;
        int cur = -1;
        for (int t = tile_first; t < T.total_tiles(); t += tile_stride, ++ti) {
            const WsTile tl = T.tile(t);
            const uint32_t a = ti & 1u;
            EpiCtx c;
            c.stg = stg; c.acc_full_bar = acc_full(a); c.acc_empty_bar = acc_empty(a); c.full_phase = (ti >> 1) & 1u;
            c.tmem_acc = tmem_base + a * WS_ACC_STRIDE; c.sb = sbias + a * 256; c.rt = rt; c.stab = stab; c.rank = rank;
            const EpiParams &ep = T.epilogue(tl, c, s_ep, cur);
            ws_tile_epilogue<PAIR>(ep, tl.bn, tl.rb * TILE_ROWS + (int)rank * BM, tl.nt * tl.bn, c);
            if constexpr (FLOW) {
                // this CTA's part of tile (layer, row block) is stored: hand it to the publisher warp
                __syncwarp();
                if (lane == 0) mbar_arrive(tile_done(a));
            }
        }
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();   // pair: the peer's shared memory / barriers stay live until both are done
    if (warp == 1) {
        if (PAIR)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// One layer per launch.
template <bool PAIR>
__global__ void __launch_bounds__(WS_THREADS, 1)
gemm_ws_kernel(const __grid_constant__ CUtensorMap tmA0h, const __grid_constant__ CUtensorMap tmA0l,
               const __grid_constant__ CUtensorMap tmW0h, const __grid_constant__ CUtensorMap tmW0l,
               const __grid_constant__ CUtensorMap tmA1h, const __grid_constant__ CUtensorMap tmA1l,
               const __grid_constant__ CUtensorMap tmW1h, const __grid_constant__ CUtensorMap tmW1l,
               const WsParams p) {
    ws_pipeline<PAIR>(LayerTiles{p, tmA0h, tmA0l, tmW0h, tmW0l, tmA1h, tmA1l, tmW1h, tmW1l});
}

// Dataflow launch.  MODE 1: 256-row tiles on CTA pairs (large steps).  MODE 0: 128 x (<= 96) tiles on single CTAs for
// small steps, where a layer has a handful of tiles and what matters is the latency from one layer to the next.
template <int MODE>
__global__ void __launch_bounds__(FLOW_THREADS, 1) gemm_flow_kernel(const FlowParams p) {
    ws_pipeline<MODE == 1>(StepTiles<MODE == 1>{p});
}

unsigned long long g_flow_attr_mask[2] = {0, 0};

unsigned long long g_ws_attr_mask[2] = {0, 0};

// Launch shape of both kernels: one persistent CTA per SM (pair != 0: one cluster of two per two SMs), never more
// CTAs (pairs) than there are tiles.  attr[0] becomes the cluster attribute of a pair launch; returns the number of
// attributes set, after which the caller may add its own.
int ws_launch_config(cudaLaunchConfig_t &cfg, cudaLaunchAttribute *attr, int tiles, int pair, int threads, size_t smem,
                     cudaStream_t st) {
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const int workers = pair ? n_sm / 2 : n_sm;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((pair ? 2 : 1) * (tiles < workers ? tiles : workers), 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 0;
    if (pair) {
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.numAttrs = 1;
    }
    return (int)cfg.numAttrs;
}

}  // namespace

int gemm_ws_max_bn() { return WS_MAX_BN; }
int gemm_pair_max_bn() { return WS_ACC_STRIDE; }

// pair != 0: CTA-pair kernel; g.W[*] tensor maps must then have a box of bn / 2 rows.
int gemm_ws_launch(const GemmCall &g, cudaStream_t st, int pair) {
    if (g.R <= 0) return 0;
    LBIC_TRY(gemm_tc_init());
    pair = pair ? 1 : 0;
    if (g.bn % 16 || g.bn < 16 || g.bn > (pair ? WS_ACC_STRIDE : WS_MAX_BN))
        return lbic_fail(LBIC_ERR_INVALID, "ws kernel: bad tile N %d", g.bn);
    if (lbic_first_use_on_device(g_ws_attr_mask[pair])) {
        if (pair) LBIC_CUDA(cudaFuncSetAttribute(gemm_ws_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        else LBIC_CUDA(cudaFuncSetAttribute(gemm_ws_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    }
    WsParams p;
    const int tile_rows = pair ? 2 * BM : BM;
    const int w_rows = pair ? g.bn / 2 : g.bn;
    p.kb[0] = (g.K[0] + BK - 1) / BK;
    p.kb[1] = g.nseg > 1 ? (g.K[1] + BK - 1) / BK : 0;
    p.bn = g.bn;
    p.ntiles_n = (g.cout + g.bn - 1) / g.bn;
    p.total_tiles = ((g.R + tile_rows - 1) / tile_rows) * p.ntiles_n;
    p.slot_bytes = 2 * A_PLANE + 2 * (uint32_t)w_rows * BK * 2;
    const bool gdn_mode = g.ep.mode == EPI_GDN || g.ep.mode == EPI_IGDN || g.ep.mode == EPI_QUANT;   // modes with side-input buffers
    p.stg_bytes = (uint32_t)(gdn_mode ? WGDN_BYTES : WSTG_BYTES);
    const int avail = SMEM_LIMIT - 1024 - (int)p.stg_bytes - 128 - WS_TAIL;
    int stages = avail / (int)p.slot_bytes;
    stages = stages > MAX_STAGES ? MAX_STAGES : stages;
    if (stages < 2) return lbic_fail(LBIC_ERR_INVALID, "ws kernel: tile does not fit shared memory");
    p.stages = stages;
    p.ring_bytes = (uint32_t)stages * p.slot_bytes;
    p.idesc = (1u << 4) | ((uint32_t)(g.bn >> 3) << 17) | ((uint32_t)(tile_rows >> 4) << 24);
    p.ep = g.ep;
    const int s1 = g.nseg > 1 ? 1 : 0;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[2];
    int na = ws_launch_config(cfg, attr, p.total_tiles, pair, WS_THREADS,
                              1024 + (size_t)p.ring_bytes + p.stg_bytes + WS_TAIL, st);
    if (gemm_get_pdl()) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.numAttrs = na;
    if (pair)
        LBIC_CUDA(cudaLaunchKernelEx(&cfg, gemm_ws_kernel<true>, *g.A[0].tm_hi, *g.A[0].tm_lo, *g.W[0].tm_hi, *g.W[0].tm_lo,
                                     *g.A[s1].tm_hi, *g.A[s1].tm_lo, *g.W[s1].tm_hi, *g.W[s1].tm_lo, p));
    else
        LBIC_CUDA(cudaLaunchKernelEx(&cfg, gemm_ws_kernel<false>, *g.A[0].tm_hi, *g.A[0].tm_lo, *g.W[0].tm_hi, *g.W[0].tm_lo,
                                     *g.A[s1].tm_hi, *g.A[s1].tm_lo, *g.W[s1].tm_hi, *g.W[s1].tm_lo, p));
    count_launch(0);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

// Every CTA pair of the dataflow launch must be resident at once (a pair waits for tiles owned by the others): true on a
// whole B200, not necessarily on a partitioned or shared one.  Checked once; callers fall back to per-layer launches.
int gemm_flow_supported() {
    static int cache[64];
    static bool cache_init = false;
    if (!cache_init) { for (int &c : cache) c = -1; cache_init = true; }
    int cur = 0;
    cudaGetDevice(&cur);
    int &ok = cache[cur & 63];
    if (ok >= 0) return ok;
    ok = 0;
    if (gemm_tc_init() != 0) return ok;
    if (lbic_first_use_on_device(g_flow_attr_mask[1]) &&
        cudaFuncSetAttribute(gemm_flow_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess) {
        cudaGetLastError();
        return ok;
    }
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[1];
    ws_launch_config(cfg, attr, INT_MAX, 1, FLOW_THREADS, FLOW_SMEM, 0);   // a pair on every two SMs
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, gemm_flow_kernel<1>, &cfg) != cudaSuccess) { cudaGetLastError(); nc = 0; }
    ok = (nc * 2 >= (int)cfg.gridDim.x) ? 1 : 0;
    return ok;
}

// Layers [l0, l1) of one wavefront step in a single dataflow launch.  dep: for every absolute layer id the (up to two)
// layer ids it reads from (-1 = none); layers outside [l0, l1) count as already complete.
int gemm_flow_launch(const ChainLayer *d_layers, const ChainLayer *h_layers, int l0, int l1, const int (*dep)[2], int R,
                     const StepDesc &step, int *d_counters, size_t counters_cap, cudaStream_t st, int pair) {
    if (R <= 0 || l1 <= l0) return 0;
    LBIC_TRY(gemm_tc_init());
    const int nl = l1 - l0;
    if (nl > FLOW_MAX_LAYERS) return lbic_fail(LBIC_ERR_INVALID, "flow kernel: too many layers");
    pair = pair ? 1 : 0;     // 0 = single CTAs, 1 = CTA pairs
    if (lbic_first_use_on_device(g_flow_attr_mask[pair])) {
        if (pair) LBIC_CUDA(cudaFuncSetAttribute(gemm_flow_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        else LBIC_CUDA(cudaFuncSetAttribute(gemm_flow_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    }
    const int variant = pair ? LBIC_PAIR_VARIANT : LBIC_SMALL_VARIANT;
    const int tile_rows = pair ? 2 * BM : BM;
    const int max_bn = pair ? WS_MAX_BN : WS_MAX_BN / 2;     // both fill a 56 KiB stage: 2 x 96 weight rows or 1 x 96
    FlowParams p;
    memset(&p, 0, sizeof(p));
    p.layers = d_layers; p.counters = d_counters; p.l0 = l0; p.n_layers = nl; p.R = R; p.step = step;
    p.variant = variant;
    p.n_rb = (R + tile_rows - 1) / tile_rows;
    if ((size_t)nl * p.n_rb > counters_cap) return lbic_fail(LBIC_ERR_INVALID, "flow kernel: counter buffer too small");
    int total = 0;
    for (int i = 0; i < nl; ++i) {
        const ChainLayer &L = h_layers[l0 + i];
        const int bn = L.bn_v[variant];
        if (bn % 16 || bn < 16 || bn > max_bn) return lbic_fail(LBIC_ERR_INVALID, "flow kernel: bad tile N %d", bn);
        p.ntn[i] = (L.cout + bn - 1) / bn;
        p.pre[i] = total;
        total += p.ntn[i];
        for (int d = 0; d < 2; ++d) {
            const int a = dep[l0 + i][d];
            p.dep[i][d] = (a >= l0 && a < l0 + i) ? a - l0 : -1;
        }
    }
    p.pre[nl] = total;
    total *= p.n_rb;
    p.total_tiles = total;
    LBIC_CUDA(cudaMemsetAsync(d_counters, 0, sizeof(int) * (size_t)nl * p.n_rb, st));
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[2];
    const int na = ws_launch_config(cfg, attr, total, pair, FLOW_THREADS, FLOW_SMEM, st);
    // Every CTA (pair) waits for tiles owned by the others, so all of them must be resident at once.  A cooperative
    // launch makes the driver guarantee that or refuse the launch (another kernel holding SMs, MPS / MIG sharing);
    // the occupancy query of gemm_flow_supported() alone cannot see what else is running.  A refused launch is
    // reported as LBIC_FLOW_REFUSED and the caller runs one launch per layer instead.
    // (no programmatic dependent launch here: the counters are zeroed by a memset node right before the kernel)
    static int use_coop = -1;  // 0 after a driver that rejects cooperative + cluster launches outright; LBIC_FLOW_COOP=0 turns
                               // the attribute off (Nsight Compute cannot replay a cooperative cluster launch)
    if (use_coop < 0) { const char *e = getenv("LBIC_FLOW_COOP"); use_coop = (e && atoi(e) == 0) ? 0 : 1; }
    for (int attempt = 0; attempt < 2; ++attempt) {
        int n_attr = na;
        if (use_coop) {
            attr[n_attr].id = cudaLaunchAttributeCooperative;
            attr[n_attr].val.cooperative = 1;
            ++n_attr;
        }
        cfg.numAttrs = n_attr;
        const cudaError_t e = pair ? cudaLaunchKernelEx(&cfg, gemm_flow_kernel<1>, p)
                                   : cudaLaunchKernelEx(&cfg, gemm_flow_kernel<0>, p);
        if (e == cudaSuccess) {
            count_launch(0);
            return 0;
        }
        cudaGetLastError();
        if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorLaunchOutOfResources) return LBIC_FLOW_REFUSED;
        if (!use_coop) return lbic_fail(LBIC_ERR_CUDA, "dataflow launch failed: %s", cudaGetErrorString(e));
        use_coop = 0;          // e.g. cudaErrorNotSupported / invalid value for the attribute combination: plain launch
    }
    return LBIC_FLOW_REFUSED;
}

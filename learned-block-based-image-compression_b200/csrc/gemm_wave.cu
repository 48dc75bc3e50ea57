// The latency kernel: a whole RANGE of wavefront steps of one encode / decode in ONE persistent, cooperative launch.
//
// compress / decompress of a single image (what eval_model calls, agents/blkbsdimgcomp_agent.py:578-599) is a chain of
// dependent small GEMMs: a 768x512 image has 222 wavefront steps (NET:339-357 restated as t = h + 2v) with at most 48
// block rows each, and every step is 14 dependent layers deep (encoder net -> quantisation -> decoder net; the entropy
// net runs beside the encoder net).  One launch per layer costs ~11 us per layer whatever the tile does (launch,
// prologue, TMEM allocation, drain): 48 ms per image, 1 s for the raster-serial reference container.
//
// Here the 148 CTAs stay resident for the whole image.  Every step's work is one list of TILES in a fixed order,
//     GATHER (operand build) | GEMM tiles of every layer, 128 rows x <= 32 columns | RANS (decode only),
// tile j of the list goes to CTA (offset + j) mod 148 (decode launches set 8 CTAs aside for the RANS tiles, KS[1] = 3
// launches a group with a fixed assignment for the entropy chain: wave_for_each_tile), and a tile may start once the tiles it reads from have been
// published through a monotonic counter per (list entry, 128-row block) -- release by a publisher warp after the
// tile's stores, acquire by whoever consumes (the TMA producer before its first load, the epilogue warps before a
// gather / rANS tile or a GDN side input).  Narrow tiles spread a layer over 20-40 SMs so that the tensor time of a
// layer (K / 16 x 3 MMAs of 128 x 32) is ~1 us; the weights stream from L2 (38 MB of fp16 hi/lo planes do not fit the
// 33 MB of shared memory of the chip).  A CTA only ever waits for tiles with a smaller list index and all CTAs are
// co-resident (cooperative launch), so the scheme cannot deadlock; every wait is bounded and traps.
//
// Arithmetic is that of gemm_tc_kernel / gemm_ws_kernel: same operand planes, same k order, one TMEM accumulator per
// output element, same fused epilogues (ws_tile_epilogue) -- results are bit-identical to the per-layer path, which is
// what lets a stream encoded by one path be decoded by the other.
#include "rans_device.cuh"
#include "ws_epilogue.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace {

constexpr int WAVE_MAX_ORD = 24;
constexpr int WAVE_MAX_RB = 32;                  // 128-row blocks per step
// Operand ring: a slot holds one 64-wide k-block = the activation box (hi + lo planes, 16..128 rows: only the rows the
// step has) + 32 weight rows (hi + lo).  A tile's mainloop is bound by the LATENCY of its loads (a layer's K / 64
// k-blocks arrive one L2 round trip after they are requested; the MMAs of a k-block take 0.1 us), so the ring is as deep
// as the staging area of the epilogue leaves room for: 152 KiB = 5 slots of 28 KiB (48 rows + 64 weight rows) for a
// 768x512 image, 2 of 64 KiB for 128 rows x 128 columns (that case is bound by the MMA chain, not by the ring).
constexpr int WAVE_MAX_STAGES = 12;
constexpr int WAVE_RING = 152 * 1024;
constexpr int WAVE_PAD = 16 * 1024;              // the MMA always reads 128 rows of a slot's activation planes: rows past the
                                                 // box are never used, but the last slot's must still be shared memory
constexpr int WAVE_THREADS = WS_THREADS + 32;    // producer | MMA issuer | 8 epilogue warps | publisher
constexpr int WAVE_BAR_BLOCK = 512;              // full[12] empty[12] acc_full[2] acc_empty[2] tile_done[2] pub_free[2] tmem slot
constexpr int WAVE_TAIL = WAVE_BAR_BLOCK + 2 * 1024 + ROWTAB_BYTES + STAB_BYTES + 256;
constexpr int WAVE_SMEM = 1024 + WAVE_RING + WAVE_PAD + WGDN_BYTES + WAVE_TAIL;
constexpr int WAVE_RANS_PARTS = 16;              // rANS tiles per 128-row block: 8 rows each, one warp per row
constexpr int WAVE_ENT_CTAS = 8;                 // decode launches: CTAs that keep the CDF tables in shared memory (rANS tiles only)
static_assert(WAVE_SMEM <= SMEM_LIMIT, "wave kernel shared memory");

// KS[1] = 3 (five-tap second entropy layer): the hidden map g0 = lrelu(E0 T) lives in a position-indexed store that
// includes a one-block ring outside the image (api.cu: run_g0).  A step then also has WK_GATHER_EXT tiles (the four
// zhat taps of the EXTENDED step's rows -- the step's blocks plus the ring positions that become computable), the E0
// layer on those rows (epilogue scatters into the store) and WK_GATHER5 tiles (the five taps of g0 -> operand of E1).
enum WaveKind { WK_GEMM = 0, WK_GATHER = 1, WK_RANS = 2, WK_GATHER_EXT = 3, WK_GATHER5 = 4 };

struct WaveOrd {
    int kind;
    int ext;        // 1: the entry's rows are those of the extended step (KS[1] = 3: WK_GATHER_EXT and the E0 layer)
    int layer;      // ChainLayer index (WK_GEMM)
    int ntn;        // tiles per 128-row block
    int bn;         // tile width (WK_GEMM)
    int dep[2];     // list entries this one reads from, -1 = none
    // WK_GEMM: a dependency that only the k-blocks from kb_late on have (KS[1] = 3: the last of E1's five taps is the only
    // one this step's E0 produces; the chain of the other four -- 4/5 of the layer's K -- starts at the top of the step)
    int dep_late, kb_late;
    int tap0;       // WK_GATHER5: first tap of this entry (its ntn / WAVE_GATHER_PARTS taps)
    int xbase;      // side-chain group: tile nt of this entry belongs to the group's CTA (xbase + nt) mod n_xg
};

struct WaveParams {
    const ChainLayer *layers;
    int *counters;               // [n_ord][WAVE_MAX_RB], zero at launch, never reset: entry (o, rb) counts the tiles of list
                                 // entry o finished for row block rb over all steps of the launch
    int n_ord, tiles_per_rb, recon_ord;
    WaveOrd ord[WAVE_MAX_ORD];
    int pre[WAVE_MAX_ORD + 1];
    int mode;                    // 0: wavefront steps t; 1: raster blocks v * Wb + h (reference container decode)
    int s_begin, s_end;
    int n_img, Hb, Wb;
    int variant;
    int stages;                  // ring depth of this launch
    int kb_group;                // k-blocks the MMA issuer takes per barrier round trip (1..4)
    int kb_adapt;                // 1: only as many of them as have landed when the first one has
    int w_first;                 // a tile's first w_first weight boxes are requested before its dependency wait
    int m64;                     // every step of the launch has at most 64 rows: M = 64 MMAs (40 instead of 52 cycles each)
    uint32_t slot_bytes, a_plane_bytes;   // slot stride; bytes of one activation plane of the launch's largest box
    const float *x_cl, *zhat_cl;
    int Cin, gather_first;       // gather tiles cover segments gather_first .. 4 (0 = x, 1..4 = the four zhat taps)
    h16 *X_hi, *X_lo; int ldX;
    h16 *T_hi, *T_lo; int ldT;
    // KS[1] = 3
    int k3, E1;
    h16 *Text_hi, *Text_lo; int ldText;          // zhat taps of the extended step's rows (operand of E0)
    const h16 *G0_hi, *G0_lo;                    // ring-extended hidden-map store, rows g0_pos_index(), E1 columns
    h16 *H5_hi, *H5_lo; int ldH5;                // five-tap operand of E1
    const int32_t *cdf; int cdf_stride; const int32_t *cdf_len, *offs; const float *scale_tab;
    RansStreamState *states; const uint8_t *const *lane_ptr; int lanes;
    const float *ksi; int ld_ksi; h16 *yq_hi, *yq_lo; int ld_yq; int32_t *sym_out; int M;
    // decode: the last n_ent CTAs are ENTROPY CTAs: they keep the compact 16-bit CDF rows (Tables::cdf16) in shared
    // memory (they need no operand ring) and run the rANS tiles, nothing else; every other tile goes to the other CTAs
    int n_ent, rans_ord;
    int n_xg, xg_e0, xg_e1;      // side-chain CTAs and their list entries [xg_e0, xg_e1) (0 CTAs = no such group)
    const uint16_t *cdf16; const int32_t *cdf16_off; int cdf16_total;
    // debug (LBIC_WAVE_TRACE): %globaltimer stamps of every tile of steps [trace_s0, trace_s0 + trace_ns), 8 words each
    unsigned long long *trace;
    int trace_s0, trace_ns, trace_stride;
};

__device__ __forceinline__ unsigned long long wave_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

struct WaveTile {
    StepDesc sd;
    StepDesc sd_ext;     // KS[1] = 3
    int R_ext;
    int R, n_rb, prev_n_rb;
    int oi, rb, nt;      // list entry, row block, tile within (entry, row block)
    int s, j;            // step, tile index within the step (trace)
};

// trace slot `k` of the tile, or nullptr when the tile is not being traced
__device__ __forceinline__ unsigned long long *wave_trace_slot(const WaveParams &p, const WaveTile &w, int k) {
    if (!p.trace || w.s < p.trace_s0 || w.s >= p.trace_s0 + p.trace_ns || w.j >= p.trace_stride) return nullptr;
    return p.trace + ((size_t)(w.s - p.trace_s0) * p.trace_stride + w.j) * 8 + k;
}
#define WAVE_TRACE(k) do { if (unsigned long long *tp__ = wave_trace_slot(p, w, (k))) *tp__ = wave_now(); } while (0)

// Every role of a CTA walks the same sequence of tiles: tile j of a step belongs to CTA (off + j) mod gridDim.x, where
// off is the number of tiles of all earlier steps.  gen[rb] = number of earlier steps of this launch that had row
// block rb; a dependency on list entry d for row block rb is met once counters[d][rb] >= ord[d].ntn * (gen[rb] + 1).
template <typename F>
__device__ __forceinline__ void wave_for_each_tile(const WaveParams &p, F &&f) {
    int gen[WAVE_MAX_RB];
#pragma unroll 1
    for (int i = 0; i < WAVE_MAX_RB; ++i) gen[i] = 0;
    int off = 0, off_e = 0, prev_n_rb = 0;
    // CTA groups: workers 0 .. Gw-1 | NX CTAs of the side chain (KS[1] = 3: the entropy net, whose E1 tiles are five times
    // as long as any other and must not sit in front of an encoder-net tile in a CTA's queue) | NE entropy CTAs (rANS
    // tiles).  Each group walks its own tiles of the list round-robin; the list positions of a group are contiguous.
    const int NE = p.n_ent, NX = p.n_xg, Gw = (int)gridDim.x - NE - NX;
    const bool is_ent = NE > 0 && (int)blockIdx.x >= Gw + NX;
    const bool is_x = NX > 0 && !is_ent && (int)blockIdx.x >= Gw;
#pragma unroll 1
    for (int s = p.s_begin; s < p.s_end; ++s) {
        WaveTile w;
        if (!step_desc(s, p.mode == 1, p.n_img, p.Hb, p.Wb, w.sd)) continue;
        w.R = w.sd.n_img * w.sd.nv;
        w.R_ext = 0;
        if (p.k3) {              // (one row block per step in this mode: the launch is refused otherwise)
            if (wave_step_ext(s, p.n_img, p.Hb, p.Wb, w.sd_ext)) w.R_ext = w.sd_ext.n_img * w.sd_ext.nv;
        }
        w.n_rb = (w.R + BM - 1) / BM;
        w.prev_n_rb = prev_n_rb;
        w.s = s;
        const int total = w.n_rb * p.tiles_per_rb;
        const int cnt_r = NE > 0 ? w.n_rb * p.ord[p.rans_ord].ntn : 0;     // rANS tiles of the step, a contiguous range
        const int start_r = NE > 0 ? w.n_rb * p.pre[p.rans_ord] : 0;
        const int cnt_x = NX > 0 ? w.n_rb * (p.pre[p.xg_e1] - p.pre[p.xg_e0]) : 0;   // side-chain tiles, contiguous, before the rANS tiles
        const int start_x = NX > 0 ? w.n_rb * p.pre[p.xg_e0] : 0;
        auto locate = [&](int j) {               // list position -> (entry, row block, tile)
            int oi = 0;
            while (j >= w.n_rb * p.pre[oi + 1]) ++oi;
            const int v = j - w.n_rb * p.pre[oi];
            w.oi = oi;
            w.rb = v / p.ord[oi].ntn;
            w.nt = v - w.rb * p.ord[oi].ntn;
            w.j = j;
        };
        // one loop (one copy of every role's code) for the three groups: tile k of the group's share of the step
        int cnt, stride, first, base;
        if (is_ent) { cnt = cnt_r; stride = NE; first = (int)blockIdx.x - Gw - NX - off_e; base = start_r; }
        else if (is_x) { cnt = p.xg_e1 - p.xg_e0; stride = 1; first = 0; base = 0; }     // k = entry: at most one tile of each
        else { cnt = total - cnt_r - cnt_x; stride = Gw; first = (int)blockIdx.x - off; base = 0; }
        if (first < 0) first += stride;
#pragma unroll 1
        for (int k = first; k < cnt; k += stride) {
            if (is_x) {
                // fixed assignment (one row block per step in this mode): the long E1 tiles sit on CTAs that have no E0 tile
                const int oi = p.xg_e0 + k;
                int nt = (int)blockIdx.x - Gw - p.ord[oi].xbase;
                if (nt < 0) nt += NX;
                if (nt >= p.ord[oi].ntn) continue;
                w.oi = oi; w.rb = 0; w.nt = nt; w.j = w.n_rb * p.pre[oi] + nt;
            } else {
                int j = base + k;
                if (!is_ent) {                   // the workers' share is the list without the other groups' ranges
                    if (cnt_x > 0 && j >= start_x) j += cnt_x;
                    if (cnt_r > 0 && j >= start_r) j += cnt_r;
                }
                locate(j);
            }
            f(w, gen);
        }
        off = (off + total - cnt_r - cnt_x) % Gw;
        if (NE > 0) off_e = (off_e + cnt_r) % NE;
        for (int rb = 0; rb < w.n_rb; ++rb) gen[rb]++;
        prev_n_rb = w.n_rb;
    }
}

__device__ __forceinline__ void wave_wait(const int *cnt, int target) {
    uint32_t spins = 0;
    while (ld_acquire_gpu(cnt) < target) {
        __nanosleep(20);
        if (++spins > (1u << 25)) __trap();     // a broken dependency must fail the launch, not hang the GPU
    }
}

// waits for the (up to two) list entries a tile reads from, for the tile's row block
__device__ __forceinline__ void wave_wait_deps(const WaveParams &p, const WaveTile &w, const int *gen) {
    for (int d = 0; d < 2; ++d) {
        const int dl = p.ord[w.oi].dep[d];
        if (dl < 0) continue;
        wave_wait(p.counters + dl * WAVE_MAX_RB + w.rb, p.ord[dl].ntn * (gen[w.rb] + 1));
    }
}

// a gather tile reads zhat blocks of the previous steps: every row block of the previous step's reconstruction layer
// must be complete (all earlier steps then are, each step ends in that layer)
__device__ __forceinline__ void wave_wait_prev_step(const WaveParams &p, const WaveTile &w, const int *gen) {
    for (int rb = 0; rb < w.prev_n_rb; ++rb)
        wave_wait(p.counters + p.recon_ord * WAVE_MAX_RB + rb, p.ord[p.recon_ord].ntn * gen[rb]);
}

// ---- GATHER tile: one K segment (x, or one of the four causal zhat taps) of the step's first-layer operands for a
// quarter (32 rows) of one row block; the arithmetic of gather_kernel (kernels_misc.cu), by the 8 epilogue warps.  The
// rows' source / destination addresses go through the (idle) row table, then every thread converts independent
// (row, 4-channel) items, eight loads in flight at a time.
constexpr int WAVE_GATHER_PARTS = 4;

__device__ __noinline__ void wave_gather_tile(const WaveParams &p, const WaveTile w0, RowTab *rt, int et, int ext) {
    // ext: the four zhat taps of the EXTENDED step's rows -> the operand of E0 (KS[1] = 3); same arithmetic
    WaveTile w = w0;
    if (ext) { w.sd = w0.sd_ext; w.R = w0.R_ext; }
    const int seg = (ext ? 1 : p.gather_first) + w.nt / WAVE_GATHER_PARTS;
    const int part = w.nt % WAVE_GATHER_PARTS;
    const int m0 = w.rb * BM + part * 32;
    int rows = w.R - m0;
    rows = rows < 0 ? 0 : (rows > 32 ? 32 : rows);
    const int c4n = p.Cin >> 2;
    if (et < rows) {
        const int r = m0 + et;
        int img, v, h;
        step_row_to_block(w.sd, r, img, v, h);
        const float *src = nullptr;
        size_t dst;
        if (seg == 0) {
            src = p.x_cl + (((size_t)img * w.sd.Hb + v) * w.sd.Wb + h) * p.Cin;
            dst = (size_t)r * p.ldX;
        } else {
            const int tap = seg - 1;
            const int vv = v + ((tap == 3) ? 0 : -1), hh = h + ((tap == 3) ? -1 : tap - 1);
            if (vv >= 0 && vv < w.sd.Hb && hh >= 0 && hh < w.sd.Wb)
                src = p.zhat_cl + (((size_t)img * w.sd.Hb + vv) * w.sd.Wb + hh) * p.Cin;
            dst = (size_t)r * (ext ? p.ldText : p.ldT) + (size_t)tap * p.Cin;
        }
        rt->f32[et] = reinterpret_cast<unsigned long long>(src);
        rt->hilo[et] = (unsigned long long)dst;
    }
    epi_bar();
    h16 *ph = seg == 0 ? p.X_hi : (ext ? p.Text_hi : p.T_hi), *pl = seg == 0 ? p.X_lo : (ext ? p.Text_lo : p.T_lo);
    const int items = rows * c4n;
    for (int i0 = et; i0 < items; i0 += 8 * WS_EPI_THREADS) {
        float4 val[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * WS_EPI_THREADS;
            val[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < items) {
                const int row = i / c4n, c4 = i - row * c4n;
                const float4 *src = reinterpret_cast<const float4 *>(rt->f32[row]);
                if (src) val[u] = __ldcg(src + c4);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * WS_EPI_THREADS;
            if (i < items) {
                const int row = i / c4n, c4 = i - row * c4n;
                const float f[4] = {val[u].x, val[u].y, val[u].z, val[u].w};
                store_hilo<4>(ph + rt->hilo[row] + c4 * 4, pl + rt->hilo[row] + c4 * 4, f);
            }
        }
    }
}

// ---- GATHER5 tile (KS[1] = 3): one of the five live taps of the 3x3 mask-'B' kernel for a quarter (32 rows) of the row
// block: H5[r, tap * E1 + c] = g0(v + dv, h + dh)[c], both planes, from the ring-extended store (gather5_kernel).
constexpr int WAVE_G5_PARTS = 16;          // 8 rows of one tap per tile (2 x 18 KiB for E1 = 1152): a tile takes ~1 us per row

__device__ __noinline__ void wave_gather5_tile(const WaveParams &p, const WaveTile w, RowTab *rt, int et) {
    const int tap = p.ord[w.oi].tap0 + w.nt / WAVE_G5_PARTS, part = w.nt % WAVE_G5_PARTS;
    const int m0 = w.rb * BM + part * (BM / WAVE_G5_PARTS);
    int rows = w.R - m0;
    rows = rows < 0 ? 0 : (rows > BM / WAVE_G5_PARTS ? BM / WAVE_G5_PARTS : rows);
    if (et < rows) {
        const int r = m0 + et;
        int img, v, h;
        step_row_to_block(w.sd, r, img, v, h);
        const int dv = (tap >= 3) ? 0 : -1;
        const int dh = (tap >= 3) ? tap - 4 : tap - 1;
        rt->f32[et] = (unsigned long long)(g0_pos_index(img, v + dv, h + dh, w.sd.Hb, w.sd.Wb) * (size_t)p.E1);
        rt->hilo[et] = (unsigned long long)((size_t)r * p.ldH5 + (size_t)tap * p.E1);
    }
    epi_bar();
    const int c8n = p.E1 >> 3;                   // 16-byte chunks per plane row
    const int items = rows * c8n * 2;            // (row, chunk, plane)
    for (int i0 = et; i0 < items; i0 += 8 * WS_EPI_THREADS) {
        uint4 val[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * WS_EPI_THREADS;
            val[u] = make_uint4(0u, 0u, 0u, 0u);
            if (i < items) {
                const int pl = i & 1, j = i >> 1;
                const int row = j / c8n, c8 = j - row * c8n;
                const h16 *src = (pl ? p.G0_lo : p.G0_hi) + rt->f32[row] + c8 * 8;
                val[u] = __ldcg(reinterpret_cast<const uint4 *>(src));
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * WS_EPI_THREADS;
            if (i < items) {
                const int pl = i & 1, j = i >> 1;
                const int row = j / c8n, c8 = j - row * c8n;
                h16 *dst = (pl ? p.H5_lo : p.H5_hi) + rt->hilo[row] + c8 * 8;
                *reinterpret_cast<uint4 *>(dst) = val[u];
            }
        }
    }
}

// the staged epilogue of the throughput kernels, compiled as a function of its own (register allocation separate from
// the role loops; the context travels by value)
__device__ __noinline__ void wave_gemm_epilogue(const EpiParams *ep, int bn, int m0, int n0, const EpiCtx cx) {
    ws_tile_epilogue<false>(*ep, bn, m0, n0, cx);
}

// ---- RANS tile: 8 rows of a row block, one warp per row: build_indexes, decode M symbols from the row's stream,
// dequantise -> y_qnt planes.  The symbol chain is serial and sits on the critical path of every decode step, so it
// runs the lean shared-memory decoder of rans_device.cuh on the entropy CTA's copy of the compact CDF rows.
struct WaveEntTables {
    uint32_t cdf16, meta, scratch;     // shared addresses: 16-bit rows | int[3][64] | 8 warps x RANS_ROW_SCRATCH(M)
};

__device__ __noinline__ void wave_rans_tile(const WaveParams &p, const WaveTile w, const WaveEntTables tb, const float *stab,
                                            int ew, int lane) {
    const int r = w.rb * BM + w.nt * 8 + ew;
    if (r >= w.R) return;
    int img, v, h;
    step_row_to_block(w.sd, r, img, v, h);
    const int sidx = p.lanes > 1 ? img * p.lanes + v : img;
    DecCursorW d;
    {
        const uint4 raw = __ldcg(reinterpret_cast<const uint4 *>(p.states + sidx));
        d.x = (unsigned long long)raw.x | ((unsigned long long)raw.y << 32);
        d.pos = raw.z; d.nwords = raw.w;
        d.words = reinterpret_cast<const uint32_t *>(p.lane_ptr[sidx]);
    }
    dec_fill_w(d, lane);
    const float *krow = p.ksi + (size_t)r * p.ld_ksi;
    const int M = p.M;
    const uint32_t scr = tb.scratch + (uint32_t)ew * RANS_ROW_SCRATCH(M);
    rans_decode_row_warp(d, tb.cdf16, tb.meta, scr, krow, stab, M, lane);
    if (lane == 0) {
        uint4 raw;
        raw.x = (uint32_t)d.x; raw.y = (uint32_t)(d.x >> 32); raw.z = d.pos; raw.w = d.nwords;
        __stcg(reinterpret_cast<uint4 *>(p.states + sidx), raw);
    }
    const size_t o = (((size_t)img * w.sd.Hb + v) * w.sd.Wb + h) * M;
    for (int c = lane; c < M; c += 32) {
        const int sym = lds_s32(scr + 8u * M + 4u * c);
        const float yq = (float)sym + __ldcg(krow + M + c);
        h16 hi, lo;
        split_h16(yq, hi, lo);
        p.yq_hi[(size_t)r * p.ld_yq + c] = hi;
        p.yq_lo[(size_t)r * p.ld_yq + c] = lo;
        if (p.sym_out) p.sym_out[o + c] = sym;
    }
}

__global__ void __launch_bounds__(WAVE_THREADS, 1) gemm_wave_kernel(const __grid_constant__ WaveParams p) {
    static_assert(sizeof(EpiParams) <= 256, "EpiParams must fit its shared-memory slot");
    static_assert(sizeof(RansStreamState) == 16, "RansStreamState is moved as one 16-byte word");
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t ring = (raw + 1023u) & ~1023u;
    const uint32_t stg = ring + WAVE_RING + WAVE_PAD;      // epilogue staging (ws_tile_epilogue)
    const uint32_t bars = stg + WGDN_BYTES;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (WAVE_MAX_STAGES + s); };
    auto acc_full = [&](int a) { return bars + 8u * (2 * WAVE_MAX_STAGES + a); };
    auto acc_empty = [&](int a) { return bars + 8u * (2 * WAVE_MAX_STAGES + 2 + a); };
    auto tile_done = [&](int a) { return bars + 8u * (2 * WAVE_MAX_STAGES + 4 + a); };
    auto pub_free = [&](int a) { return bars + 8u * (2 * WAVE_MAX_STAGES + 6 + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * WAVE_MAX_STAGES + 8);
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(smem_raw + (tmem_slot - raw));
    float *sbias = reinterpret_cast<float *>(smem_raw + (bars + WAVE_BAR_BLOCK - raw));        // [2][256]
    RowTab *rt = reinterpret_cast<RowTab *>(smem_raw + (bars + WAVE_BAR_BLOCK + 2048 - raw));
    float *stab = reinterpret_cast<float *>(rt + 1);
    EpiParams *s_ep = reinterpret_cast<EpiParams *>(stab + 64);
    if (p.scale_tab && threadIdx.x < 64) stab[threadIdx.x] = p.scale_tab[threadIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int stages = p.stages;
    WaveEntTables tb;
    tb.cdf16 = 0; tb.meta = 0; tb.scratch = 0;
    if (p.n_ent > 0 && (int)blockIdx.x >= (int)gridDim.x - p.n_ent) {
        // entropy CTA: compact CDF rows | row offsets, lengths, symbol offsets | per-warp scratch, in the (unused) operand ring
        uint8_t *base = smem_raw + (ring - raw);
        uint4 *dst = reinterpret_cast<uint4 *>(base);
        const int nvec = (p.cdf16_total + 7) >> 3;
        for (int i = threadIdx.x; i < nvec; i += WAVE_THREADS) dst[i] = reinterpret_cast<const uint4 *>(p.cdf16)[i];
        int *s_meta = reinterpret_cast<int *>(dst + nvec);
        if (threadIdx.x < 64) {
            s_meta[threadIdx.x] = p.cdf16_off[threadIdx.x];
            s_meta[64 + threadIdx.x] = p.cdf_len[threadIdx.x];
            s_meta[128 + threadIdx.x] = p.offs[threadIdx.x];
        }
        tb.cdf16 = ring;
        tb.meta = ring + 16u * (uint32_t)nvec;
        tb.scratch = tb.meta + 768u;
    }
    // slot layout: activation hi | activation lo (a_plane_bytes each) | weight hi | weight lo
    const uint32_t off_alo = p.a_plane_bytes, off_w = 2 * p.a_plane_bytes;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < WAVE_MAX_STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(acc_full(a), 1);
            mbar_init(acc_empty(a), WS_EPI_THREADS / 32);
            mbar_init(tile_done(a), WS_EPI_THREADS / 32);
            mbar_init(pub_free(a), 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ---- TMA producer: all 32 lanes walk the loop, one elected lane issues (tc_common.cuh: elect_one) ----
        {
            uint32_t it = 0;
            wave_for_each_tile(p, [&](const WaveTile &w, const int *gen) {
                const WaveOrd &o = p.ord[w.oi];
                if (o.kind != WK_GEMM) return;
                const ChainLayer &Lr = p.layers[o.layer];
                const int bn = o.bn;
                const int m0 = w.rb * BM, n0 = w.nt * bn;
                const int R_use = o.ext ? w.R_ext : w.R;
                const int rows = (R_use - m0) < BM ? (R_use - m0) : BM;
                const int cls = lbic_box_class(rows);          // only the rows the step has are loaded
                const int nseg = Lr.nseg > 1 ? 2 : 1;
                // descriptors of this tile's operands into the descriptor cache while the inputs are still being produced
                if (lane == 0) {
                    for (int sg = 0; sg < nseg; ++sg)
                        for (int pl = 0; pl < 2; ++pl) {
                            const CUtensorMap *ta = cls < 4 ? &Lr.tmAs[cls][sg][pl] : &Lr.tmA[sg][pl];
                            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(ta)) : "memory");
                            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&Lr.tmW[p.variant][sg][pl])) : "memory");
                        }
                }
                const int kb0 = Lr.kb[0], nkb = kb0 + (Lr.nseg > 1 ? Lr.kb[1] : 0);
                const uint32_t w_plane = (uint32_t)bn * (BK * 2);
                const uint32_t stage_tx = 2u * (uint32_t)lbic_box_rows(cls) * (BK * 2) + 2 * w_plane;
                // the weights do not depend on the previous layer: the ring's worth of weight boxes goes out BEFORE the
                // dependency wait (the slot's barrier is armed for the whole stage; the activation boxes follow below), so
                // that a tile's first MMAs wait for one L2 round trip of its activations only
                const int npre0 = p.w_first < stages ? p.w_first : stages, npre = nkb < npre0 ? nkb : npre0;
                for (int j = 0; j < npre; ++j) {
                    const uint32_t itj = it + (uint32_t)j;
                    const int s = itj % stages;
                    mbar_wait(empty_bar(s), ((itj / stages) & 1u) ^ 1u);
                    const uint32_t sa = ring + s * p.slot_bytes;
                    const int seg = j >= kb0 ? 1 : 0;
                    const int kk = (seg ? j - kb0 : j) * BK;
                    if (elect_one()) {
                        mbar_expect_tx(full_bar(s), stage_tx);
                        tma_load_2d(sa + off_w, &Lr.tmW[p.variant][seg][0], full_bar(s), kk, n0);
                        tma_load_2d(sa + off_w + w_plane, &Lr.tmW[p.variant][seg][1], full_bar(s), kk, n0);
                    }
                    __syncwarp();
                }
                if (lane == 0) {
                    wave_wait_deps(p, w, gen);
                    WAVE_TRACE(0);
                }
                __syncwarp();
                asm volatile("fence.proxy.async;" ::: "memory");   // generic-proxy stores of other CTAs -> our TMA reads
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    if (o.dep_late >= 0 && kb == o.kb_late) {
                        if (lane == 0) wave_wait(p.counters + o.dep_late * WAVE_MAX_RB + w.rb, p.ord[o.dep_late].ntn * (gen[w.rb] + 1));
                        __syncwarp();
                        asm volatile("fence.proxy.async;" ::: "memory");
                    }
                    const int s = it % stages;
                    const uint32_t ph = (it / stages) & 1u;
                    if (kb >= npre) mbar_wait(empty_bar(s), ph ^ 1u);
                    const uint32_t sa = ring + s * p.slot_bytes;
                    const int seg = kb >= kb0 ? 1 : 0;
                    const int kk = (seg ? kb - kb0 : kb) * BK;
                    if (elect_one()) {
                        if (kb >= npre) mbar_expect_tx(full_bar(s), stage_tx);
                        tma_load_2d(sa, cls < 4 ? &Lr.tmAs[cls][seg][0] : &Lr.tmA[seg][0], full_bar(s), kk, m0);
                        tma_load_2d(sa + off_alo, cls < 4 ? &Lr.tmAs[cls][seg][1] : &Lr.tmA[seg][1], full_bar(s), kk, m0);
                        if (kb >= npre) {
                            tma_load_2d(sa + off_w, &Lr.tmW[p.variant][seg][0], full_bar(s), kk, n0);
                            tma_load_2d(sa + off_w + w_plane, &Lr.tmW[p.variant][seg][1], full_bar(s), kk, n0);
                        }
                    }
                    __syncwarp();
                }
                if (lane == 0) WAVE_TRACE(1);
            });
        }
    } else if (warp == 1) {
        // ---- tcgen05.mma issuer ---------------------------------------------------------------------------
        {   // all 32 lanes walk the loop, one elected lane issues (tc_common.cuh: elect_one)
            uint32_t it = 0, gi = 0;
            wave_for_each_tile(p, [&](const WaveTile &w, const int *) {
                const WaveOrd &o = p.ord[w.oi];
                if (o.kind != WK_GEMM) return;
                const ChainLayer &Lr = p.layers[o.layer];
                const int bn = o.bn;
                const int nkb = Lr.kb[0] + (Lr.nseg > 1 ? Lr.kb[1] : 0);
                const uint32_t w_plane = (uint32_t)bn * (BK * 2);
                const uint32_t idesc = (1u << 4) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)((p.m64 ? 64 : BM) >> 4) << 24);
                const uint32_t a = gi & 1u;
                mbar_wait(acc_empty(a), ((gi >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t tmem_acc = tmem_base + a * WS_ACC_STRIDE;
                // up to four k-blocks per barrier round trip: the issue of an MMA blocks until the tensor core takes it, so the
                // wait / fence / elect sequence between k-blocks is not hidden behind the MMAs (profiles/r2_wave_latency.md)
                const int nb_max = p.kb_group < stages ? p.kb_group : stages;
                uint32_t slot = it % stages, phase = (it / stages) & 1u;        // ring position of the next k-block
                // (starting with a single k-block so that the first MMAs go out as soon as it has landed -- groups of 1, 2, 4, 4 --
                // measured the same: 33.4 / 32.1 against 33.3 / 31.9 ms)
                for (int kb = 0; kb < nkb;) {
                    int nb = nkb - kb < nb_max ? nkb - kb : nb_max;
                    if (p.kb_adapt) {
                        // the next k-block, and as many of the following ones as have already landed: a ring that is only a
                        // little deeper than the group (six slots for KS3311's 64-row boxes) otherwise stalls a whole load
                        // latency per group when the weights come from DRAM
                        const int lim = nb;
                        uint32_t s2 = slot, p2 = phase;
                        mbar_wait(full_bar(s2), p2);
                        nb = 1;
#pragma unroll
                        for (int u = 1; u < 4; ++u) {
                            if (u >= lim) break;
                            if (++s2 == (uint32_t)stages) { s2 = 0; p2 ^= 1u; }
                            if (!__all_sync(0xffffffffu, mbar_test_wait(full_bar(s2), p2))) break;
                            nb = u + 1;
                        }
                    } else {
                        uint32_t s2 = slot, p2 = phase;
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (u < nb) {
                                mbar_wait(full_bar(s2), p2);
                                if (++s2 == (uint32_t)stages) { s2 = 0; p2 ^= 1u; }
                            }
                    }
                    tc_fence_after();
                    if (kb == 0 && lane == 0) WAVE_TRACE(2);
                    if (elect_one()) {
                        uint32_t s2 = slot;
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (u < nb) {
                                const uint32_t sa = ring + s2 * p.slot_bytes;
                                const uint64_t a_hi = make_smem_desc(sa);
                                const uint64_t a_lo = make_smem_desc(sa + off_alo);
                                const uint64_t w_hi = make_smem_desc(sa + off_w);
                                const uint64_t w_lo = make_smem_desc(sa + off_w + w_plane);
#pragma unroll
                                for (int k = 0; k < BK / 16; ++k) umma_f16(tmem_acc, a_hi + 2 * k, w_hi + 2 * k, idesc, ((kb + u) | k) != 0 ? 1u : 0u);
#pragma unroll
                                for (int k = 0; k < BK / 16; ++k) umma_f16(tmem_acc, a_hi + 2 * k, w_lo + 2 * k, idesc, 1u);
#pragma unroll
                                for (int k = 0; k < BK / 16; ++k) umma_f16(tmem_acc, a_lo + 2 * k, w_hi + 2 * k, idesc, 1u);
                                umma_commit(empty_bar(s2));
                                if (++s2 == (uint32_t)stages) s2 = 0;
                            }
                        if (kb + nb == nkb) umma_commit(acc_full(a));
                    }
                    __syncwarp();
                    for (int u = 0; u < nb; ++u)
                        if (++slot == (uint32_t)stages) { slot = 0; phase ^= 1u; }
                    kb += nb;
                    it += nb;
                }
                if (lane == 0) WAVE_TRACE(3);
                ++gi;
            });
        }
    } else if (warp == 10) {
        // ---- publisher: the tile's stores have been issued -> make them visible, bump the tile's counter ----
        if (lane == 0) {
            uint32_t di = 0;
            wave_for_each_tile(p, [&](const WaveTile &w, const int *) {
                const uint32_t a = di & 1u;
                mbar_wait(tile_done(a), (di >> 1) & 1u);
                mbar_arrive(pub_free(a));                           // the epilogue may signal tile di + 2 on this barrier
                asm volatile("fence.proxy.async;" ::: "memory");
                asm volatile("fence.acq_rel.gpu;" ::: "memory");
                asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(p.counters + w.oi * WAVE_MAX_RB + w.rb) : "memory");
                WAVE_TRACE(6);
                if (unsigned long long *tp = wave_trace_slot(p, w, 7))
                    *tp = (unsigned long long)w.oi | ((unsigned long long)w.rb << 8) | ((unsigned long long)w.nt << 16) |
                          ((unsigned long long)blockIdx.x << 32);
                ++di;
            });
        }
    } else {
        // ---- epilogue warps 2..9: GEMM epilogues, gather tiles, rANS tiles ------------------------------------
        const int et = threadIdx.x - 64;
        const int ew = warp - 2;
        uint32_t di = 0, gi = 0;
        wave_for_each_tile(p, [&](const WaveTile &w, const int *gen) {
            const WaveOrd &o = p.ord[w.oi];
            if (o.kind == WK_GEMM) {
                const ChainLayer &Lr = p.layers[o.layer];
                const int bn = o.bn;
                const int m0 = w.rb * BM, n0 = w.nt * bn;
                // this tile's epilogue description: the layer's, with the step and its row count
                epi_bar();     // every epilogue thread is past the previous tile (which read the old copy / the row table)
                {
                    constexpr int NW = (int)(sizeof(EpiParams) / 4);
                    constexpr int OFF_R = (int)(offsetof(EpiParams, R) / 4), OFF_STEP = (int)(offsetof(EpiParams, step) / 4);
                    constexpr int NSTEP = (int)(sizeof(StepDesc) / 4);
                    const uint32_t *g = reinterpret_cast<const uint32_t *>(&Lr.ep);
                    const uint32_t *sw = reinterpret_cast<const uint32_t *>(o.ext ? &w.sd_ext : &w.sd);
                    if (et < NW) {
                        uint32_t wd = g[et];
                        if (et == OFF_R) wd = (uint32_t)(o.ext ? w.R_ext : w.R);
                        else if (et >= OFF_STEP && et < OFF_STEP + NSTEP) wd = sw[et - OFF_STEP];
                        reinterpret_cast<uint32_t *>(s_ep)[et] = wd;
                    }
                }
                epi_bar();
                const uint32_t a = gi & 1u;
                EpiCtx c;
                c.stg = stg; c.acc_full_bar = acc_full(a); c.acc_empty_bar = acc_empty(a); c.full_phase = (gi >> 1) & 1u;
                c.tmem_acc = tmem_base + a * WS_ACC_STRIDE; c.sb = sbias + a * 256; c.rt = rt; c.stab = stab; c.rank = 0;
                const int dl = o.dep[0];
                c.dep_cnt = dl >= 0 ? p.counters + dl * WAVE_MAX_RB + w.rb : nullptr;
                c.dep_target = dl >= 0 ? p.ord[dl].ntn * (gen[w.rb] + 1) : 0;
                const int dl2 = o.dep[1];
                c.dep2_cnt = dl2 >= 0 ? p.counters + dl2 * WAVE_MAX_RB + w.rb : nullptr;
                c.dep2_target = dl2 >= 0 ? p.ord[dl2].ntn * (gen[w.rb] + 1) : 0;
                c.trace_acc = et == 0 ? wave_trace_slot(p, w, 4) : nullptr;
                c.m64 = p.m64;
                wave_gemm_epilogue(s_ep, bn, m0, n0, c);
                ++gi;
            } else {
                // non-GEMM tiles: one thread waits for the inputs, then all eight warps work
                epi_bar();     // the previous tile is done with the row table
                if (et == 0) {
                    if (o.kind == WK_GATHER || o.kind == WK_GATHER_EXT || (o.kind == WK_GATHER5 && o.dep[0] < 0))
                        wave_wait_prev_step(p, w, gen);          // (reconstruction of step t-1 done => its E0 and E1 are too)
                    else wave_wait_deps(p, w, gen);
                    WAVE_TRACE(0);
                }
                epi_bar();
                __syncwarp();  // lane 0 of warp 2 took the branch above: the warp-wide shuffles / votes below want it reconverged
                if (o.kind == WK_GATHER) wave_gather_tile(p, w, rt, et, 0);
                else if (o.kind == WK_GATHER_EXT) wave_gather_tile(p, w, rt, et, 1);
                else if (o.kind == WK_GATHER5) wave_gather5_tile(p, w, rt, et);
                else wave_rans_tile(p, w, tb, stab, ew, lane);
            }
            if (et == 0) WAVE_TRACE(5);
            // this CTA's tile is stored: hand it to the publisher warp (which must have taken tile di - 2 off this barrier)
            __syncwarp();
            if (lane == 0) {
                const uint32_t a = di & 1u;
                mbar_wait(pub_free(a), ((di >> 1) & 1u) ^ 1u);
                mbar_arrive(tile_done(a));
            }
            ++di;
        });
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

unsigned long long g_wave_attr_mask = 0;

int wave_prepare() {
    LBIC_TRY(gemm_tc_init());
    if (lbic_first_use_on_device(g_wave_attr_mask))
        LBIC_CUDA(cudaFuncSetAttribute(gemm_wave_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    return 0;
}

}  // namespace

int gemm_wave_max_rows() { return WAVE_MAX_RB * BM; }

// 1 if one CTA of the wave kernel fits every SM of this device (the launch itself is cooperative, so a busy or shared
// GPU is refused at launch time, not here)
int gemm_wave_supported() {
    static int cache[64];
    static bool cache_init = false;
    if (!cache_init) { for (int &c : cache) c = -1; cache_init = true; }
    int cur = 0;
    cudaGetDevice(&cur);
    int &ok = cache[cur & 63];
    if (ok >= 0) return ok;
    ok = 0;
    if (wave_prepare() != 0) return ok;
    int coop = 0, nb = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, cur);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, gemm_wave_kernel, WAVE_THREADS, WAVE_SMEM) != cudaSuccess) {
        cudaGetLastError();
        nb = 0;
    }
    ok = (coop && nb >= 1) ? 1 : 0;
    return ok;
}

int gemm_wave_launch(const WaveLaunch &w, cudaStream_t st) {
    if (w.s_end <= w.s_begin) return 0;
    LBIC_TRY(wave_prepare());
    WaveParams p;
    memset(&p, 0, sizeof(p));
    p.layers = w.d_layers; p.counters = w.counters;
    p.mode = w.raster ? 1 : 0; p.s_begin = w.s_begin; p.s_end = w.s_end;
    p.n_img = w.n_img; p.Hb = w.Hb; p.Wb = w.Wb;
    p.variant = w.variant;
    p.x_cl = w.x_cl; p.zhat_cl = w.zhat_cl; p.Cin = w.Cin;
    p.X_hi = w.X_hi; p.X_lo = w.X_lo; p.ldX = w.ldX; p.T_hi = w.T_hi; p.T_lo = w.T_lo; p.ldT = w.ldT;
    p.cdf = w.cdf; p.cdf_stride = w.cdf_stride; p.cdf_len = w.cdf_len; p.offs = w.offs; p.scale_tab = w.scale_tab;
    p.states = w.states; p.lane_ptr = w.lane_ptr; p.lanes = w.lanes;
    p.ksi = w.ksi; p.ld_ksi = w.ld_ksi; p.yq_hi = w.yq_hi; p.yq_lo = w.yq_lo; p.ld_yq = w.ld_yq; p.sym_out = w.sym_out; p.M = w.M;
    int max_rows = w.raster ? w.n_img : w.n_img * (w.Hb < (w.Wb + 1) / 2 ? w.Hb : (w.Wb + 1) / 2);
    p.k3 = w.k3 ? 1 : 0;
    if (p.k3) {
        // KS[1] = 3: the extended step has up to two more positions per image (the ring columns); one 128-row block only
        if (w.raster) return lbic_fail(LBIC_ERR_INVALID, "wave kernel: KS[1] = 3 has no raster mode");
        const int nv_ext = (w.Hb < (w.Wb + 3) / 2 + 1 ? w.Hb : (w.Wb + 3) / 2 + 1);
        max_rows = w.n_img * nv_ext;
        if (max_rows > BM) return lbic_fail(LBIC_ERR_INVALID, "wave kernel: KS[1] = 3 steps must fit one row block (%d rows)", max_rows);
        p.E1 = w.E1;
        p.Text_hi = w.Text_hi; p.Text_lo = w.Text_lo; p.ldText = w.ldText;
        p.G0_hi = w.G0_hi; p.G0_lo = w.G0_lo;
        p.H5_hi = w.H5_hi; p.H5_lo = w.H5_lo; p.ldH5 = w.ldH5;
    }
    if (max_rows > WAVE_MAX_RB * BM) return lbic_fail(LBIC_ERR_INVALID, "wave kernel: step of %d rows exceeds %d", max_rows, WAVE_MAX_RB * BM);
    {
        static int m64 = -1;     // LBIC_WAVE_M64=0 keeps M = 128 (tests, measurements)
        if (m64 < 0) { const char *e = getenv("LBIC_WAVE_M64"); m64 = (e && atoi(e) == 0) ? 0 : 1; }
        p.m64 = (m64 && max_rows <= 64) ? 1 : 0;
        static int kbg = -1;     // LBIC_WAVE_KB_GROUP: tuning hook
        if (kbg < 0) { const char *e = getenv("LBIC_WAVE_KB_GROUP"); kbg = e ? atoi(e) : 4; kbg = kbg < 1 ? 1 : (kbg > 4 ? 4 : kbg); }
        p.kb_group = kbg;
        static int kba = -1;     // LBIC_WAVE_KB_ADAPT: tuning hook
        if (kba < 0) { const char *e = getenv("LBIC_WAVE_KB_ADAPT"); kba = e ? atoi(e) : 1; }
        p.kb_adapt = kba ? 1 : 0;
        static int wf = -1;      // LBIC_WAVE_WFIRST: tuning hook
        if (wf < 0) { const char *e = getenv("LBIC_WAVE_WFIRST"); wf = e ? atoi(e) : 0; }
        p.w_first = wf < 0 ? 0 : wf;
    }
    int bn_max = 16;
    for (int i = 0; i < 18; ++i) {
        const int bn = w.h_layers[i].bn_v[w.variant];
        if (bn % 16 || bn < 16 || bn > LBIC_LAT_MAX_BN) return lbic_fail(LBIC_ERR_INVALID, "wave kernel: bad tile N %d", bn);
        bn_max = bn > bn_max ? bn : bn_max;
    }
    {
        const int box = lbic_box_rows(lbic_box_class(max_rows < BM ? max_rows : BM));   // largest activation box of this launch
        p.a_plane_bytes = (uint32_t)box * (BK * 2);
        p.slot_bytes = 2 * p.a_plane_bytes + 2 * (uint32_t)bn_max * (BK * 2);
        // the MMA reads 128 (64) rows of a slot's activation planes whatever the box: only the last slot's over-read needs
        // the pad behind the ring, the rest of it is ring
        const int over = ((p.m64 ? 64 : BM) - box) * (BK * 2);
        p.stages = (WAVE_RING + WAVE_PAD - over) / (int)p.slot_bytes;
        if (p.stages > WAVE_MAX_STAGES) p.stages = WAVE_MAX_STAGES;
        if (p.stages < 2) return lbic_fail(LBIC_ERR_INVALID, "wave kernel: operand slot does not fit the ring");
        static int cap = -1;   // tuning hook: LBIC_WAVE_STAGES caps the ring depth
        if (cap < 0) { const char *e = getenv("LBIC_WAVE_STAGES"); cap = e ? atoi(e) : 0; }
        if (cap >= 2 && p.stages > cap) p.stages = cap;
    }
    // the step's list.  h_layers by LayerId: E..E+3 = entropy net, F..F+6 = encoder net (F0 G0 F1 G1 F2 G2 F3), D..D+6 = decoder net.
    // The encoder net (the critical path of an encode step) comes first so that its tiles are never queued behind the
    // entropy net's in a CTA's own list; the entropy net only has to be done when F3 quantises.
    int n = 0;
    auto add = [&](int kind, int layer, int ntn, int bn, int d0, int d1) {
        p.ord[n].kind = kind; p.ord[n].ext = 0; p.ord[n].layer = layer; p.ord[n].ntn = ntn; p.ord[n].bn = bn;
        p.ord[n].dep[0] = d0; p.ord[n].dep[1] = d1; p.ord[n].dep_late = -1; p.ord[n].kb_late = 0; p.ord[n].tap0 = 0; p.ord[n].xbase = 0;
        return n++;
    };
    auto gemm = [&](int id, int d0, int d1) {
        const ChainLayer &L = w.h_layers[id];
        const int bn = L.bn_v[w.variant];
        return add(WK_GEMM, id, (L.cout + bn - 1) / bn, bn, d0, d1);
    };
    const int E = 0, F = 4, D = 11;
    int n_sm = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    // KS[1] = 3: CTAs the other groups need -- one per tile of the widest encoder / decoder-net layer, the rANS CTAs of a decode
    int main_need = WAVE_GATHER_PARTS * 5;
    for (int i = F; i < D + 7; ++i) {
        if (w.decode && i < D) continue;
        const ChainLayer &L = w.h_layers[i];
        const int bn = L.bn_v[w.variant], nt = (L.cout + bn - 1) / bn;
        main_need = nt > main_need ? nt : main_need;
    }
    const int n_ent_k3 = w.decode ? (max_rows > 8 * WAVE_ENT_CTAS ? 2 * WAVE_ENT_CTAS : WAVE_ENT_CTAS) : 0;
    p.gather_first = w.decode ? 1 : 0;
    const int g = add(WK_GATHER, -1, (w.decode ? 4 : 5) * WAVE_GATHER_PARTS, 0, -1, -1);
    int last_e, last;
    // KS[1] = 3: the entropy net's first layer runs on the extended step's rows and scatters into the g0 store; the
    // second layer reads its five taps from there
    auto ent_k3 = [&]() {
        // taps 0..3 of g0 were produced by earlier steps (gathered first: nothing of this step is needed), tap 4 = (v, h)
        // by this step's E0
        const int g5a = add(WK_GATHER5, -1, 4 * WAVE_G5_PARTS, 0, -1, -1);
        const int gx = add(WK_GATHER_EXT, -1, 4 * WAVE_GATHER_PARTS, 0, -1, -1);
        const int e0 = gemm(E, gx, -1);
        p.ord[gx].ext = 1; p.ord[e0].ext = 1;
        const int g5b = add(WK_GATHER5, -1, 1 * WAVE_G5_PARTS, 0, e0, -1);
        p.ord[g5b].tap0 = 4;
        const int e1 = gemm(E + 1, g5a, -1);
        p.ord[e1].dep_late = g5b;
        p.ord[e1].kb_late = (4 * w.E1) / BK;          // the k-block that holds the first column of tap 4
        const int e2 = gemm(E + 2, e1, -1);
        const int e3 = gemm(E + 3, e2, -1);
        // its own CTAs for this chain, each with at most one tile of every entry: E1 (and g5a, E2, E3) from the group's CTA 0,
        // the E0 sub-chain (gx, E0, g5b) behind E1's CTAs where the grid has room -- an E1 tile then starts as soon as the
        // first four taps are gathered instead of queueing behind an E0 tile of its CTA
        int widest = 0, sub = 0;
        for (int i = g5a; i <= e3; ++i) widest = p.ord[i].ntn > widest ? p.ord[i].ntn : widest;
        for (int i = gx; i <= g5b; ++i) sub = p.ord[i].ntn > sub ? p.ord[i].ntn : sub;
        static int xg = -1;      // LBIC_WAVE_XG: tuning hook (cap of the group; 0 = no side-chain group)
        if (xg < 0) { const char *e = getenv("LBIC_WAVE_XG"); xg = e ? atoi(e) : 1 << 20; }
        int cap = n_sm - main_need - n_ent_k3;
        cap = cap < xg ? cap : xg;
        int nx = p.ord[e1].ntn + sub;
        nx = nx < widest ? widest : nx;
        nx = nx > cap ? cap : nx;
        if (nx < widest) nx = 0;                      // no room for one tile per CTA: the workers take the chain
        p.n_xg = nx;
        p.xg_e0 = g5a; p.xg_e1 = e3 + 1;
        if (nx > 0) {
            const int b = nx - sub < p.ord[e1].ntn ? nx - sub : p.ord[e1].ntn;
            for (int i = gx; i <= g5b; ++i) p.ord[i].xbase = b;
        }
        return e3;
    };
    if (p.k3 && !w.decode) {
        // the entropy net is the longer chain here (E1 has K = 5 E1): its tiles first
        const int f0 = gemm(F, g, -1);
        last_e = ent_k3();
        const int g0 = gemm(F + 1, f0, -1);
        const int f1 = gemm(F + 2, g0, -1);
        const int g1 = gemm(F + 3, f1, -1);
        const int f2 = gemm(F + 4, g1, -1);
        const int g2 = gemm(F + 5, f2, -1);
        last = gemm(F + 6, g2, last_e);
    } else if (p.k3) {
        last_e = ent_k3();
        last = add(WK_RANS, -1, WAVE_RANS_PARTS, 0, last_e, -1);
        p.rans_ord = last;
        p.n_ent = max_rows > 8 * WAVE_ENT_CTAS ? 2 * WAVE_ENT_CTAS : WAVE_ENT_CTAS;   // one warp per row: 64 or 128 rows per round
        p.cdf16 = w.cdf16; p.cdf16_off = w.cdf16_off; p.cdf16_total = w.cdf16_total;
        if (!w.cdf16 || w.cdf16_total <= 0 ||
            (size_t)w.cdf16_total * 2 + 16 + 3 * 64 * 4 + 8 * (size_t)RANS_ROW_SCRATCH(w.M) > (size_t)WAVE_RING)
            return lbic_fail(LBIC_ERR_INVALID, "wave kernel: entropy tables do not fit shared memory");
    } else if (!w.decode) {
        // interleaved: F0 E0 G0 E1 F1 E2 G1 E3 F2 G2 F3 | D0 .. D3
        const int f0 = gemm(F, g, -1);
        const int e0 = gemm(E, g, -1);
        const int g0 = gemm(F + 1, f0, -1);
        const int e1 = gemm(E + 1, e0, -1);
        const int f1 = gemm(F + 2, g0, -1);
        const int e2 = gemm(E + 2, e1, -1);
        const int g1 = gemm(F + 3, f1, -1);
        last_e = gemm(E + 3, e2, -1);
        const int f2 = gemm(F + 4, g1, -1);
        const int g2 = gemm(F + 5, f2, -1);
        last = gemm(F + 6, g2, last_e);            // QUANT: operand from G2, entropy parameters from E3
    } else {
        const int e0 = gemm(E, g, -1);
        const int e1 = gemm(E + 1, e0, -1);
        const int e2 = gemm(E + 2, e1, -1);
        last_e = gemm(E + 3, e2, -1);
        last = add(WK_RANS, -1, WAVE_RANS_PARTS, 0, last_e, -1);
        p.rans_ord = last;
        p.n_ent = max_rows > 8 * WAVE_ENT_CTAS ? 2 * WAVE_ENT_CTAS : WAVE_ENT_CTAS;   // one warp per row: 64 or 128 rows per round
        p.cdf16 = w.cdf16; p.cdf16_off = w.cdf16_off; p.cdf16_total = w.cdf16_total;
        if (!w.cdf16 || w.cdf16_total <= 0 ||
            (size_t)w.cdf16_total * 2 + 16 + 3 * 64 * 4 + 8 * (size_t)RANS_ROW_SCRATCH(w.M) > (size_t)WAVE_RING)
            return lbic_fail(LBIC_ERR_INVALID, "wave kernel: entropy tables do not fit shared memory");
    }
    for (int i = 0; i < 7; ++i) last = gemm(D + i, last, -1);   // D0 IG0 D1 IG1 D2 IG2 D3: each reads the one before
    p.recon_ord = last;
    p.n_ord = n;
    int total = 0;
    for (int i = 0; i < n; ++i) { p.pre[i] = total; total += p.ord[i].ntn; }
    p.pre[n] = total;
    p.tiles_per_rb = total;
    if ((size_t)n * WAVE_MAX_RB > w.counters_cap) return lbic_fail(LBIC_ERR_INVALID, "wave kernel: counter buffer too small");
    LBIC_CUDA(cudaMemsetAsync(w.counters, 0, sizeof(int) * (size_t)n * WAVE_MAX_RB, st));
    // debug: LBIC_WAVE_TRACE=<first step> [LBIC_WAVE_TRACE_STEPS=<n>] dumps per-tile time stamps of one launch to
    // LBIC_WAVE_TRACE_FILE (default gpurun_out/wave_trace.txt); see scripts/wave_trace.py
    static int trace_s0 = -2;
    if (trace_s0 == -2) { const char *e = getenv("LBIC_WAVE_TRACE"); trace_s0 = e ? atoi(e) : -1; }
    static unsigned long long *d_trace = nullptr;
    const bool tracing = trace_s0 >= 0 && trace_s0 >= w.s_begin && trace_s0 < w.s_end;
    size_t trace_words = 0;
    if (tracing) {
        const char *e = getenv("LBIC_WAVE_TRACE_STEPS");
        p.trace_s0 = trace_s0;
        p.trace_ns = e ? atoi(e) : 3;
        p.trace_stride = ((max_rows + BM - 1) / BM) * total;
        trace_words = (size_t)p.trace_ns * p.trace_stride * 8;
        if (d_trace) cudaFree(d_trace);
        LBIC_CUDA(cudaMalloc(&d_trace, trace_words * 8));
        LBIC_CUDA(cudaMemsetAsync(d_trace, 0, trace_words * 8, st));
        p.trace = d_trace;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(n_sm, 1, 1);
    cfg.blockDim = dim3(WAVE_THREADS, 1, 1);
    cfg.dynamicSmemBytes = WAVE_SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;     // all CTAs co-resident, or the launch is refused
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_wave_kernel, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorLaunchOutOfResources || e == cudaErrorNotSupported)
            return LBIC_FLOW_REFUSED;
        return lbic_fail(LBIC_ERR_CUDA, "wave launch failed: %s", cudaGetErrorString(e));
    }
    count_launch(0);
    if (tracing) {
        std::vector<unsigned long long> h(trace_words);
        LBIC_CUDA(cudaStreamSynchronize(st));
        LBIC_CUDA(cudaMemcpy(h.data(), d_trace, trace_words * 8, cudaMemcpyDeviceToHost));
        const char *fn = getenv("LBIC_WAVE_TRACE_FILE");
        FILE *f = fopen(fn ? fn : "gpurun_out/wave_trace.txt", "w");
        if (f) {
            fprintf(f, "# decode=%d raster=%d n_ord=%d; per tile: step j oi kind layer rb nt cta | dep_ready tma_issued first_full mma_issued acc_full epi_done published (ns, %%globaltimer)\n",
                    w.decode, w.raster, n);
            for (int si = 0; si < p.trace_ns; ++si)
                for (int j = 0; j < p.trace_stride; ++j) {
                    const unsigned long long *r = h.data() + ((size_t)si * p.trace_stride + j) * 8;
                    if (!r[6]) continue;
                    const int oi = (int)(r[7] & 0xFF);
                    fprintf(f, "%d %d %d %d %d %d %d %d | %llu %llu %llu %llu %llu %llu %llu\n", trace_s0 + si, j, oi, p.ord[oi].kind,
                            p.ord[oi].layer, (int)((r[7] >> 8) & 0xFF), (int)((r[7] >> 16) & 0xFFFF), (int)(r[7] >> 32), r[0], r[1], r[2],
                            r[3], r[4], r[5], r[6]);
                }
            fclose(f);
        }
        trace_s0 = -1;     // one launch only
    }
    return 0;
}

// Internal declarations shared by the translation units of liblbic_b200.so.
#pragma once

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/lbic.h"

// GEMM operand element: IEEE fp16.  Every fp32 value is stored as two fp16 planes (hi + lo = 22 significand bits);
// see gemm_tc.cu.  (bf16 planes gave 16 bits and ~6x more rounding-boundary symbol flips, DESIGN.md section 2.)
typedef __half h16;

int lbic_fail(int code, const char *fmt, ...);

#define LBIC_CUDA(call)                                                                        \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return lbic_fail(LBIC_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,       \
                             cudaGetErrorString(e__));                                         \
    } while (0)

#define LBIC_TRY(call)                  \
    do {                                \
        int rc__ = (call);              \
        if (rc__ != 0) return rc__;     \
    } while (0)

// ------------------------------------------------------------------------------------------------
// A wavefront step.  Row r of a step's compact activation matrices is block
//   img = r / nv,  v = vmin + r % nv,  h = t - 2 v        (slope-2 wavefront t = h + 2 v)
// The raster-serial decode of the reference container uses nv = 1, vmin = v, t = h + 2 v.
// ------------------------------------------------------------------------------------------------
struct StepDesc {
    int n_img, nv, vmin, t, Hb, Wb;
};

// Row of block position (v,h) of image img in the ring-extended hidden-map store used when KS[1] == 3:
// rows v = -1..Hb-1, columns h = -1..Wb (SURVEY.md A.3: g0 is evaluated on a one-block ring outside the image).
__host__ __device__ inline size_t g0_pos_index(int img, int v, int h, int Hb, int Wb) {
    return ((size_t)img * (Hb + 1) + (v + 1)) * (Wb + 2) + (h + 1);
}

// nv == 0 marks a RASTER chunk (open-loop forward, lbic_forward): row r is block number t + r of the batch in
// (img, v, h) raster order; otherwise the rows are the blocks of wavefront step t (h + 2v = t) of every image.
__host__ __device__ inline void step_row_to_block(const StepDesc &s, int r, int &img, int &v, int &h) {
    if (s.nv == 0) {
        const int hw = s.Hb * s.Wb;
        const int g = s.t + r;
        img = g / hw;
        const int q = g - img * hw;
        v = q / s.Wb;
        h = q - v * s.Wb;
        return;
    }
    img = r / s.nv;
    v = s.vmin + (r - img * s.nv);
    h = s.t - 2 * v;
}

// ------------------------------------------------------------------------------------------------
// Epilogue of a GEMM layer (fused into both GEMM cores).
// ------------------------------------------------------------------------------------------------
enum EpiMode {
    EPI_LRELU = 0,   // v = lrelu(acc+b)                      -> hi/lo           (NET:305-311)
    EPI_PREGDN = 1,  // a = acc+b -> f32; a*a                 -> hi/lo           (GDNF:71 x**2)
    EPI_GDN = 2,     // aux * rsqrt(acc+beta)                 -> hi/lo           (GDNF:71-78)
    EPI_IGDN = 3,    // aux * sqrt(acc+beta)                  -> hi/lo
    EPI_KSI = 4,     // acc+b                                 -> f32 (scales | means, NET:369)
    EPI_QUANT = 5,   // y=acc+b; sym=rint(y-mean); idx; yq    -> hi/lo, sym, idx (NET:371-374)
    EPI_RECON = 6,   // clamp(acc+b, -.5, .5)                 -> zhat (NET:357)
    EPI_RAW = 7,     // acc                                   -> f32 (debug gemm)
    EPI_RESID = 8    // aux + acc + b (optionally clamped)     -> f32 (post-processing net, NET:475-476)
};

struct EpiParams {
    int mode;
    int R;              // valid rows
    int cout;           // valid output columns
    const float *bias;  // [cout] (beta for the GDN modes)
    float acc_scale;    // 2^-k: the layer's weights are stored multiplied by 2^k (fp16 range), undone here exactly
    h16 *out_hi, *out_lo;
    int ld_out;
    int out_pos;        // 1: hi/lo output row = position in the ring-extended g0 store (KS[1]=3), see g0_pos_index
    int no_clamp;       // RECON: 1 = leave the reconstruction unclamped (model.forward returns it so, NET:104-106)
    float *out_f32;
    int ld_f32;
    const float *aux;   // pre-GDN activations (GDN modes) or ksi (QUANT)
    int ld_aux;
    int M;              // latent channels (QUANT)
    const float *scale_tab;   // device, 64 scale levels (QUANT)
    int32_t *sym;       // (n_img,Hb,Wb,M) int32        (QUANT)
    uint8_t *idx;       // (n_img,Hb,Wb,M) uint8        (QUANT)
    float *zhat;        // (n_img,Hb,Wb,Cin) fp32 channel-last   (RECON)
    StepDesc step;
};

// One K segment of a GEMM: A[R,K] (h16 hi/lo planes, row stride ld) times W[cout,K]^T.
struct GemmOperand {
    const h16 *hi, *lo;
    int ld;                 // elements
    const CUtensorMap *tm_hi, *tm_lo;   // host copies of the TMA descriptors
};

struct GemmCall {
    int R, cout, bn;
    int nseg;
    int K[2];
    GemmOperand A[2], W[2];
    EpiParams ep;
};

// One layer as the persistent multi-layer kernels see it (gemm_flow_kernel, gemm_wave_kernel), resident in device memory.
// Tile-width variants per layer, indexed by "split factor" f: the layer's Cout is cut into f * ceil(Cout / (256 f))
// equal tiles (width rounded up to 16), so a cluster of f CTAs gets the same number of tiles per CTA.
constexpr int LBIC_NBN = 14;          // 6 split factors + the warp-specialised kernel's tiling (width <= 192) + its CTA-pair forms + small / latency tilings
constexpr int LBIC_WS_VARIANT = 6;
constexpr int LBIC_PAIR_WIDE = 8;     // CTA-pair form with tiles up to 256 wide (2 pipeline stages instead of 3)
constexpr int LBIC_SMALL_VARIANT = 9;  // tiles of at most 96 columns for the single-CTA dataflow launch of small steps
constexpr int LBIC_LAT_VARIANT = 10;   // tilings of the persistent wavefront (latency) kernel, gemm_wave.cu: at most 32 columns,
constexpr int LBIC_LAT64_VARIANT = 11;  // 64,
constexpr int LBIC_LAT128_VARIANT = 12; // 128 (the time of a tile's MMA chain does not depend on its width up to ~176 columns)
constexpr int LBIC_LAT_MAX_BN = 128;
// rows of the activation TMA box for a tile with `rows` valid rows: class 0..3 = 16 / 32 / 48 / 64, 4 = the full 128
__host__ __device__ inline int lbic_box_class(int rows) { return rows <= 16 ? 0 : rows <= 32 ? 1 : rows <= 48 ? 2 : rows <= 64 ? 3 : 4; }
__host__ __device__ inline int lbic_box_rows(int cls) { return cls < 4 ? 16 * (cls + 1) : 128; }
constexpr int LBIC_QUAD_VARIANT = 13;   // quad form of the dataflow launch: width <= 192 with an EVEN number of column tiles (two pairs
                                        // of a cluster take adjacent tiles); weight TMA box = half the tile
constexpr int LBIC_PAIR_VARIANT = 7;  // same tile width as LBIC_WS_VARIANT; weight TMA box = half the tile (one half per CTA)
__host__ __device__ inline int lbic_split(int i) { return i == 0 ? 1 : i == 1 ? 2 : i == 2 ? 3 : i == 3 ? 4 : i == 4 ? 6 : 8; }
struct alignas(64) ChainLayer {
    CUtensorMap tmA[2][2];              // [segment][hi, lo]   box 64 x 128
    CUtensorMap tmAs[4][2][2];          // [box class][segment][hi, lo]: boxes of 64 k x 16 / 32 / 48 / 64 rows for the latency
                                        // kernel (a step of a single image has at most min(Hb, Wb/2) rows)
    CUtensorMap tmW[LBIC_NBN][2][2];    // [variant][segment][hi, lo]   box 64 x bn_v[variant]
    int kb[2];                          // 64-wide k-blocks per segment
    int nseg;
    int cout;
    int bn_v[LBIC_NBN];
    int n_bn;
    EpiParams ep;                       // R and step are filled in per launch
    // TMA-store epilogue (ws_tile_epilogue): descriptors of the layer's row-indexed OUTPUT planes, boxes of 16 columns x
    // 128 rows: [0] hi, [1] lo (fp16, SWIZZLE_32B), [2] fp32 plane (SWIZZLE_64B).  tma_out = 0: the layer scatters its
    // rows (QUANT symbols / indexes, RECON, the position-indexed g0 store) and keeps the staged copy loops.
    CUtensorMap tmO[6];                 // [3] hi, [4] lo as 64-column boxes (SWIZZLE_128B), [5] fp32 as a 32-column box (SWIZZLE_128B)
    int tma_out;
};

int gemm_ws_launch(const GemmCall &g, cudaStream_t st, int pair = 0);   // persistent warp-specialised kernel (gemm_ws.cu)
int gemm_flow_launch(const ChainLayer *d_layers, const ChainLayer *h_layers, int l0, int l1, const int (*dep)[2], int R,
                     const StepDesc &step, int *d_counters, size_t counters_cap, cudaStream_t st, int pair = 1);
constexpr int LBIC_FLOW_REFUSED = 1000;   // gemm_flow_launch: the (cooperative) launch was refused; use the per-layer path
int gemm_flow_supported();   // 1 if all CTA pairs of the dataflow launch can be co-resident on this device
int gemm_flow_quad_clusters();   // clusters of four of the quad form resident at once (0 = not available)
struct RansStreamState;
// The latency path (gemm_wave.cu): a range of wavefront steps (or raster blocks) of ONE encode / decode in a single
// persistent cooperative launch; gather, GEMM layers and (decode) the rANS step are tiles of one in-kernel work list.
struct WaveLaunch {
    const ChainLayer *d_layers, *h_layers;
    int decode;                 // 0: encode step = gather | entropy net | encoder net + quantisation | decoder net
                                // 1: decode step = gather | entropy net | rANS | decoder net
    int raster;                 // 1: steps are single blocks in raster order (reference container decode)
    int s_begin, s_end;         // wavefront: t in [s_begin, s_end); raster: block number v * Wb + h
    int n_img, Hb, Wb;
    int variant;                // LBIC_LAT*_VARIANT: tile width
    const uint16_t *cdf16; const int32_t *cdf16_off; int cdf16_total;   // compact CDF rows (Tables), decode only
    int ids[20];                // LayerId of E0..E3, F0..F3 (7), D0..D3 (7) in api.cu's LayerId order (18 entries)
    const float *x_cl, *zhat_cl;
    int Cin;
    h16 *X_hi, *X_lo; int ldX;
    h16 *T_hi, *T_lo; int ldT;
    // KS[1] = 3: taps of the extended step (operand of E0), the ring-extended g0 store, the five-tap operand of E1
    int k3, E1;
    h16 *Text_hi, *Text_lo; int ldText;
    const h16 *G0_hi, *G0_lo;
    h16 *H5_hi, *H5_lo; int ldH5;
    // decode only
    const int32_t *cdf; int cdf_stride; const int32_t *cdf_len, *offs; const float *scale_tab;
    RansStreamState *states; const uint8_t *const *lane_ptr; int lanes;
    const float *ksi; int ld_ksi; h16 *yq_hi, *yq_lo; int ld_yq; int32_t *sym_out; int M;
    int *counters; size_t counters_cap;
    int *err_flag;
};
int gemm_wave_launch(const WaveLaunch &w, cudaStream_t st);   // LBIC_FLOW_REFUSED if the cooperative launch is refused
int gemm_wave_supported();
int gemm_wave_max_rows();
int gemm_ws_max_bn();
int gemm_pair_max_bn();
void gemm_set_pdl(int on);   // programmatic dependent launch between consecutive GEMM kernels (default on)
int gemm_get_pdl();
void gemm_set_tma_store(int on);   // dataflow launch: row-indexed layers store their outputs through the TMA engine (default on)
int gemm_get_tma_store();
int gemm_simt_launch(const GemmCall &g, cudaStream_t st);
int gemm_tc_launch(const GemmCall &g, cudaStream_t st);
int gemm_tc_init();   // resolves cuTensorMapEncodeTiled, sets smem attributes
// general form: element size 2 (fp16) or 4 (fp32), swizzle 32 / 64 / 128 bytes
int make_tmap_2d_ex(CUtensorMap *tm, const void *base, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                    uint32_t box_inner, uint32_t box_outer, int swizzle_bytes);
int make_tmap_2d(CUtensorMap *tm, const void *base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                 uint32_t box_inner, uint32_t box_outer);

// ------------------------------------------------------------------------------------------------
// elementwise / layout kernels (kernels_misc.cu)
// ------------------------------------------------------------------------------------------------
int launch_nchw_to_cl(const float *src, float *dst, int n, int C, int HW, cudaStream_t st);
int launch_cl_to_nchw(const float *src, float *dst, int n, int C, int HW, cudaStream_t st);
// band-wise forms (block rows [v0, v1) of every image): the host calls convert while later bands are still in flight
int launch_nchw_to_cl_band(const float *src, float *dst, int n, int C, int Hb, int Wb, int v0, int v1, cudaStream_t st);
int launch_cl_to_nchw_band(const float *src, float *dst, int n, int C, int Hb, int Wb, int v0, int v1, cudaStream_t st);
// 8-bit RGB images (n,3,H,W) <-> channel-last block tensors (pad / crop, +-0.5 and the 8-bit quantisation fused)
int launch_u8_to_xcl(const uint8_t *img, float *x_cl, int n, int H, int W, int Hb, int Wb, int B, int v0, int v1,
                     cudaStream_t st);
int launch_zcl_to_u8(const float *z_cl, uint8_t *img, int n, int H, int W, int Hb, int Wb, int B, int v0, int v1,
                     cudaStream_t st);
int launch_space_to_depth(const float *img, float *blk, int n, int C, int Hb, int Wb, int B, cudaStream_t st);
int launch_depth_to_space(const float *blk, float *img, int n, int C, int Hb, int Wb, int B, cudaStream_t st);
int launch_split_f32(const float *src, h16 *hi, h16 *lo, int64_t n, cudaStream_t st);
// per-step gather of x and the four causal neighbour blocks of zhat (SURVEY.md A.1/A.2)
int launch_gather(const float *x_cl, const float *zhat_cl, int Cin, const StepDesc &s, int R,
                  h16 *X_hi, h16 *X_lo, int ldX, h16 *T_hi, h16 *T_lo, int ldT, cudaStream_t st);
// weight packing
// weight packing: effective fp32 weights (mask folded / taps reordered / GDN reparametrised), their max |w|,
// then the scaled fp16 hi/lo split
int launch_pack_conv(const float *w, const float *mask, int cout, int cin, int kh, int kw,
                     const int *taps_host, int ntaps, float *weff, int ld, cudaStream_t st);
int launch_pack_gdn(const float *gamma, const float *beta, int C, float gbound, float gped, float bbound,
                    float bped, float *weff, int ld, float *beta_out, cudaStream_t st);
int launch_sat_scan(const h16 *hi, int R, int C, int ld, unsigned long long *count, cudaStream_t st);   // *count += clipped elements
int launch_absmax(const float *v, int64_t n, float *out_dev, cudaStream_t st);   // *out_dev = max(*out_dev, max|v|)
int launch_split_scaled(const float *src, h16 *hi, h16 *lo, int64_t n, float scale, cudaStream_t st);
// KS[1]==3: A operand of get_meanscale[2] = the five mask-'B' taps of g0 around each block of the step
// post-processing net (NET:455-476): A operand of its 3x3 conv = all nine taps of the reconstruction around each block
// of a raster chunk, zero outside the image; and the final fix-up: blocks on the image border keep their input
int launch_gather9(const float *z_cl, int Cin, const StepDesc &s, int R, h16 *out_hi, h16 *out_lo, int ld, cudaStream_t st);
int launch_restore_border(const float *z_cl, float *out_cl, int Cin, int n_img, int Hb, int Wb, cudaStream_t st);
int launch_gather5(const h16 *g0_hi, const h16 *g0_lo, int E1, const StepDesc &s, int R, h16 *out_hi, h16 *out_lo,
                   int ld, cudaStream_t st);
int launch_fill_g0_top(const float *bias, int E1, int n_img, int Hb, int Wb, h16 *g_hi, h16 *g_lo, cudaStream_t st);
int launch_add_vec(const float *a, const float *b, float *out, int n, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// entropy model tables + rANS (tables.cu, rans.cu)
// ------------------------------------------------------------------------------------------------
struct Tables {
    int n_levels = 0, stride = 0;
    int32_t *cdf = nullptr;       // device [n_levels][stride]
    int32_t *cdf_length = nullptr;
    int32_t *offset = nullptr;
    float scale_table[64];
    float *d_scale_table = nullptr;   // device copy, 64 floats
    // Compact form for the thread-per-stream decode kernel (rans.cu), which keeps it in shared memory: the rows
    // back to back as 16-bit values without their final 65536 (row l starts at cdf16_off[l]) followed by a
    // 257-entry bucket table per level: lut[l][b] = first k with cdf[l][k] > 256 b, lut[l][256] = len - 1.
    uint16_t *cdf16 = nullptr;        // [cdf16_total] rows | [n_levels][257] bucket table
    int32_t *cdf16_off = nullptr;     // device [65]
    int cdf16_total = 0;              // 0: not available (tables too large for shared memory)
};
int tables_build(Tables &T, const float *scale_table_host, int n_levels, double tail_mass, cudaStream_t st);
int tables_compact(Tables &T, cudaStream_t st);   // (re)builds the compact form from cdf / cdf_length
void tables_free(Tables &T);

struct RansStreamState {   // one per stream, device resident between decode steps
    unsigned long long x;
    uint32_t pos;          // next word index within the stream
    uint32_t nwords;
};

// symbols/indexes: for stream s, symbol k lives at  base + s*stream_stride + k   (elements).
// scratch holds n_streams*scratch_words words followed by start_word[n_streams] and n_words[n_streams];
// out may be NULL (lane mode: launch_lane_pack assembles the containers from the scratch).
int launch_rans_encode(const Tables &T, const int32_t *sym, const uint8_t *idx, int n_streams, int64_t n_sym,
                       int64_t stream_stride, uint32_t *scratch_words, size_t scratch_words_per_stream,
                       uint8_t *out, size_t out_stride, uint32_t *out_len, int *err_flag, cudaStream_t st);
// lane container: merges `lanes` consecutive single streams per image into header|lengths|payload
int launch_lane_pack(const uint32_t *scratch, size_t scratch_words, int n_img, int lanes, uint8_t *out,
                     size_t out_stride, uint32_t *out_len, int *err_flag, cudaStream_t st);
// lanes_container != 0: the streams are 'LBML' lane containers (also when lanes == 1, i.e. a one-block-row image)
int launch_rans_dec_init(const uint8_t *streams, const uint32_t *stream_len, size_t stream_stride, int n_img,
                         int lanes, int lanes_container, RansStreamState *states, const uint8_t **lane_ptr, int *err_flag,
                         cudaStream_t st);
// decode M symbols for every row of a step; writes yq = sym + mean (hi/lo) and optionally symbols
void rans_set_enc_block_max_streams(int n);    // encodes of at most this many streams use the CTA-per-stream kernel (0 = never)
void rans_set_enc_thread_min_streams(int n);   // encodes of at least this many streams use the thread-per-stream kernel
void rans_set_dec_smem_warp(int on);           // 1 (default): warp-per-row decode steps run on shared-memory tables
void rans_set_dec_thread_min_rows(int rows);   // steps with at least this many rows use the thread-per-stream kernel
int launch_rans_dec_step(const Tables &T, RansStreamState *states, const uint8_t *const *lane_ptr, int lanes,
                         const StepDesc &s, int R, int M, const float *ksi, int ld_ksi, h16 *yq_hi, h16 *yq_lo,
                         int ld_yq, int32_t *sym_out, cudaStream_t st);
int launch_selfinfo_step(const StepDesc &s, int R, int M, const float *ksi, int ld_ksi, const int32_t *sym, float *info,
                         cudaStream_t st);
// CDF index of n scales by both routines of the decoders (bisection; hint with bisection fallback), for tests
int launch_scale_index(const float *scales, int n, const float *tab, int32_t *idx_bisect, int32_t *idx_hinted, cudaStream_t st);
int launch_rans_decode_full(const Tables &T, const uint8_t *streams, const uint32_t *stream_len, size_t stream_stride,
                            const uint8_t *idx, int n_streams, int64_t n_sym, int32_t *sym_out, cudaStream_t st);

// image metrics (metrics.cu)
size_t metrics_scratch_bytes(int n, int C, int H, int W);
int launch_image_metrics(const float *x, const float *y, int n, int C, int H, int W, float offset, float range, void *scratch,
                         double *mse_out, double *msssim_out, cudaStream_t st);

// launch bookkeeping
void count_launch(int family);   // 0 = gemm, 1 = other

// Function attributes (opt-in shared memory) are per device: true the first time it is called for (mask, current device).
inline bool lbic_first_use_on_device(unsigned long long &mask) {
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long bit = 1ull << (dev & 63);
    if (mask & bit) return false;
    mask |= bit;
    return true;
}
extern thread_local int64_t *g_launch_counter;   // points into the active model

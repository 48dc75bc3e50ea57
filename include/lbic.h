/*
 * lbic.h -- C ABI of the B200-native closed-loop block codec (liblbic_b200.so).
 *
 * The reference (kamisli-icpl/Learned-block-based-image-compression) has no FFI of its own on
 * this path; its only foreign-function edge is pybind11 into CompressAI.  Each entry point below
 * therefore names the reference *Python* interface it stands behind (paths relative to the
 * reference root; NET = graphs/models/BlockBasedImgCompLossy_net.py,
 * ENT = graphs/layers/entropy_layers_cai.py, AGENT = agents/blkbsdimgcomp_agent.py).
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative lbic_status;
 * the message of the last failure on the calling thread is lbic_last_error(); nothing throws or
 * aborts.  All work is enqueued on the caller's CUDA stream (pass the cudaStream_t as void*;
 * NULL = legacy default stream).  "device pointer" arguments must be device-accessible memory on
 * the model's device; the *_host entry points take ordinary host memory and perform the
 * host<->device copies themselves.  One lbic_model per device; calls on one model are not
 * re-entrant.  Requires an sm_100a GPU: there is no CPU fallback.
 */
#ifndef LBIC_H_
#define LBIC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lbic_model lbic_model;

typedef enum {
    LBIC_OK = 0,
    LBIC_ERR_INVALID = -1,     /* bad argument / unsupported configuration            */
    LBIC_ERR_CUDA = -2,        /* a CUDA runtime or driver call failed                */
    LBIC_ERR_STATE = -3,       /* weights or tables missing (reference: ValueError, ENT:185-204) */
    LBIC_ERR_NOMEM = -4,
    LBIC_ERR_NO_DEVICE = -5,   /* no sm_100 device: the product path refuses to run   */
    LBIC_ERR_OVERFLOW = -6     /* a caller-provided stream buffer was too small       */
} lbic_status;

/* Model hyper-parameters: the four keys the reference model reads from its config JSON
 * (NET:262-302: config.block_size, config.KS, config.N, config.M). */
typedef struct {
    int block_size;            /* B                                  */
    int ks[4];                 /* KS, [3,1,1,1] or [3,3,1,1]         */
    int n;                     /* N                                  */
    int m;                     /* M                                  */
} lbic_config;

/* One state_dict entry (name as in the reference state_dict, SURVEY.md Appendix A.7).
 * data may be a host or a device pointer (fp32, C-contiguous). */
typedef struct {
    const char *name;
    const float *data;
    int ndim;
    int64_t shape[4];
} lbic_tensor_desc;

/* GEMM core selection (lbic_set_option LBIC_OPT_GEMM_CORE):
 *   0 = tcgen05/TMEM/TMA tensor-core tiles, fp16 hi/lo operand split, 3 MMAs per product (product path)
 *   1 = fp32 SIMT evaluation of the same split operands (bring-up / cross-check twin)      */
#define LBIC_OPT_GEMM_CORE 1
#define LBIC_OPT_PAIR 8        /* 1 (default) = CTA-pair (cta_group::2) form of the persistent kernel: 256-row tiles, half the weight traffic per SM */
#define LBIC_OPT_DEC_THREAD_ROWS 9 /* decode steps with >= this many block rows (default 4096) decode one stream per thread, fewer: one per warp (process-wide) */
#define LBIC_OPT_ENC_THREAD_STREAMS 10 /* entropy-encode calls with >= this many streams (default 4096) encode one stream per thread, fewer: one per warp (process-wide) */
#define LBIC_OPT_DEC_SMEM_WARP 20   /* 1 (default): decode steps below LBIC_OPT_DEC_THREAD_ROWS decode one row per warp on shared-memory copies of the compact CDF rows; 0: on the int32 tables in global memory (process-wide) */
#define LBIC_OPT_ENC_BLOCK_STREAMS 17 /* entropy-encode calls with at most this many streams (default 592) encode one stream per CTA: table lookups by seven warps, the serial state chain on one thread (process-wide; 0 = never) */
#define LBIC_OPT_FLOW 11         /* 1 (default) = run each large wavefront step's layers as ONE dataflow launch (row-block dependencies instead of kernel boundaries): on single CTAs below LBIC_OPT_FLOW_PAIR_MIN_ROWS block rows, on CTA pairs from there; 2 = always (pairs); 0 = one launch per layer */
#define LBIC_OPT_FLOW_QUAD 21     /* dataflow launch on clusters of FOUR CTAs: two CTA pairs take adjacent column tiles of one 256-row block and share its activation operand by TMA multicast (each CTA fetches one plane); 0 = CTA pairs only */
#define LBIC_OPT_TMA_STORE 24     /* 1: in the dataflow launch the layers whose output rows are the step's compact rows store through the TMA engine from swizzled staging tiles (full 128-byte lines where the tile allows); 0 (default): staged copy loops; bit-identical, measured equal (process-wide) */
#define LBIC_OPT_CHECK_SATURATION 26 /* 1: count the elements of the fp16 operand planes clipped at +-65504 (lbic_saturation_count); debug, per-layer launches */
#define LBIC_OPT_FLOW_MIN_ROWS 12 /* steps with at least this many block rows take the dataflow launch (default 2560) */
#define LBIC_OPT_FLOW_PAIR_MIN_ROWS 25 /* dataflow steps with fewer block rows than this (default 8192) run on single CTAs with 128 x 96 tiles, larger ones on CTA pairs with 256 x 192 tiles */
#define LBIC_OPT_FLOW_SMALL 13    /* 1 = steps below LBIC_OPT_FLOW_MIN_ROWS also run as one dataflow launch, on single CTAs with 128 x 96 tiles; 0 (default) = one launch per layer there */
#define LBIC_OPT_WAVE 15           /* 1 (default) = calls whose wavefront steps have at most LBIC_OPT_WAVE_MAX_ROWS block rows (single images, small batches; KS[1] = 1) run as ONE persistent cooperative launch per call (gemm_wave.cu): gather, all layers and the rANS decode step are tiles of an in-kernel work list; 0 = one launch per layer */
#define LBIC_OPT_WAVE_MAX_ROWS 16  /* default 1536, at most 4096 */
#define LBIC_OPT_WAVE_DEC_MAX_ROWS 18 /* decode calls take the wave kernel up to this many rows per step (default 64): its rANS tiles run one warp per row on 8 entropy CTAs that keep the CDF tables in shared memory */
#define LBIC_OPT_WAVE_BN 19        /* tuning hook: forced tile width of the wave kernel (32, 64, 128); 0 = 32 */
#define LBIC_OPT_HOST_BANDS 14     /* the *_host entry points move a batch in / out in this many bands of block rows, overlapped with the wavefront (1..16, default 16; 1 = copy, compute, copy) */
#define LBIC_OPT_WS 6          /* 1 (default) = persistent warp-specialised kernel for steps with >= 2 tiles per SM */
#define LBIC_OPT_PDL 7         /* 1 (default) = programmatic dependent launch between consecutive GEMM kernels (process-wide) */
#define LBIC_OPT_FORCE_BN 3    /* tuning hook: force the GEMM tile width (multiple of 16, <= 256); 0 = automatic */

const char *lbic_last_error(void);
const char *lbic_version(void);

/* Model(config) -- NET:259-317.  device = CUDA ordinal. */
int lbic_create(const lbic_config *cfg, int device, lbic_model **out);
void lbic_destroy(lbic_model *m);
int lbic_set_option(lbic_model *m, int option, int value);

/* model.load_state_dict(sd) -- agents/base.py:95-96.  Consumes every `*.weight/bias/mask`,
 * `*.beta/gamma` and GDN reparam buffer of Appendix A.7; folds the masks (NET:381), applies the
 * non-negative reparametrisation (utils/parametrizers.py:45-48) and packs fp16 hi/lo planes (scaled by 2^k per layer) on
 * the device.  The library keeps no reference to the caller's memory. */
int lbic_load_weights(lbic_model *m, const lbic_tensor_desc *tensors, int n_tensors, void *stream);

/* model.update(force=True) -- NET:121-125 -> ENT:579-613 (+ compressai._CXX.pmf_to_quantized_cdf).
 * scale_table: host pointer to the n_levels scale values (NET:13-18); tail_mass as ENT:528.
 * Builds quantized_cdf / cdf_length / offset on the GPU. */
int lbic_build_tables(lbic_model *m, const float *scale_table, int n_levels, double tail_mass, void *stream);
/* Install tables produced elsewhere (e.g. `conditional_gaussian_model._quantized_cdf` buffers
 * found in a reference checkpoint).  Host pointers. */
int lbic_set_tables(lbic_model *m, const float *scale_table, int n_levels, const int32_t *cdf,
                    int cdf_stride, const int32_t *cdf_length, const int32_t *offset);
/* Read the tables back (host pointers; cdf must hold n_levels*cdf_stride ints).  Queries with
 * NULL outputs just return the sizes. */
int lbic_get_tables(lbic_model *m, int *n_levels, int *cdf_stride, int32_t *cdf, int32_t *cdf_length,
                    int32_t *offset);

/* model.compress(x, LRU, chlat) -- NET:319-361, batched over n_img images of identical size.
 *   x          device, (n_img, 3B^2, Hb, Wb) fp32 in [-0.5,0.5]: the layout eval_model passes
 *              (AGENT:588-592)
 *   zhat_out   device, same shape: the encoder-side reconstruction (second return value)
 *   sym_out    device or NULL, (n_img, Hb, Wb, M) int32 quantised latent symbols (NET:353)
 *   idx_out    device or NULL, (n_img, Hb, Wb, M) uint8 CDF indexes (NET:354)
 *   stream_out device, n_img * stream_cap bytes; image i's bitstream starts at i*stream_cap
 *   stream_len device, n_img uint32 byte counts
 *   lanes      1 = the reference container: one rANS64 stream per image, raw words, no header
 *              (NET:359-360);  0 = one lane per block row (container extension, see DESIGN.md)
 * stream_cap >= lbic_stream_bound(...).  stream_out == NULL skips entropy coding. */
int lbic_encode(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out,
                int32_t *sym_out, uint8_t *idx_out, uint8_t *stream_out, size_t stream_cap,
                uint32_t *stream_len, int lanes, void *stream);

/* model.decompress(bitstream, LRU, xshape, chlat, devc) -- NET:400-452, batched.
 *   streams / stream_len / stream_cap as produced by lbic_encode (device pointers)
 *   zhat_out   device, (n_img, 3B^2, Hb, Wb) fp32
 *   sym_out    device or NULL: the decoded symbols */
int lbic_decode(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                int n_img, int Hb, int Wb, float *zhat_out, int32_t *sym_out, int lanes, void *stream);

/* Closed-loop reconstruction WITHOUT entropy coding plus the rate estimate -- the loop of validate_recu_reco_fast
 * (AGENT:491-549): zhat_out as lbic_encode; selfinfo_out device, (n_img, M, Hb, Wb) fp32 = -log2 of the
 * Gaussian-conditional likelihood of every quantised latent (ENT:615-647).  Block windows follow the codec path's
 * border rule (SURVEY.md A.6); for KS[1]=1 that is exactly what model.forward() computes in the reference loop. */
int lbic_validate(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out, float *selfinfo_out,
                  void *stream);

/* model.forward(zhat, x) in eval mode -- NET:90-106, the open-loop pass ACL training-set regeneration runs over
 * every patch (AGENT:643-684): all blocks are independent given the context zhat_in.
 *   zhat_in, x    device, (n_img, 3B^2, Hb, Wb) fp32 (context reconstruction, original)
 *   xhat_out      device, same shape; clamp != 0 applies the caller's clamp_(-0.5, 0.5) (AGENT:667), 0 returns it raw
 *   selfinfo_out  device or NULL, (n_img, M, Hb, Wb) fp32 = -log2 pmf of every quantised latent
 *   sym_out       device or NULL, (n_img, Hb, Wb, M) int32 = round(y - means)
 * Convolutions are zero padded per layer as in the reference's whole-image forward, which for KS[1] = 3 differs from
 * the codec path's block windows at the image border (SURVEY.md A.6). */
int lbic_forward(lbic_model *m, const float *zhat_in, const float *x, int n_img, int Hb, int Wb, float *xhat_out,
                 float *selfinfo_out, int32_t *sym_out, int clamp, void *stream);

/* Kernels cannot return errors: a bitstream buffer that was too small (encode) or a malformed lane container (decode) is
 * flagged on the device; the affected image's stream_len is 0xFFFFFFFF / its lanes decode as empty streams.  This call
 * synchronises `stream` and returns LBIC_ERR_OVERFLOW / LBIC_ERR_INVALID if the last lbic_encode / lbic_decode enqueued on
 * it flagged anything (the *_host entry points below do this themselves). */
int lbic_check_errors(lbic_model *m, void *stream);

/* Same two calls with HOST buffers (pageable or pinned): the copies are part of the call and the
 * call returns after the results are in host memory.  This is what a reference-side binding
 * (INTEGRATION.md) calls from eval_model (AGENT:591-599).  The batch moves over PCIe in bands of block rows while
 * the wavefront runs (LBIC_OPT_HOST_BANDS), so only the first input band and the last output band are exposed. */
int lbic_encode_host(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out,
                     uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes);
int lbic_decode_host(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len,
                     size_t stream_cap, int n_img, int Hb, int Wb, float *zhat_out, int lanes);

/* The per-image body of eval_model for a batch of 8-bit RGB images of identical size (host memory, (n_img, 3, H, W)):
 *   encode: ToTensor (u8 / 255), x - 0.5 (AGENT:581), replicate padding to a multiple of B (AGENT:583-586),
 *           arrange_block_pixels_to_channel_dim (AGENT:588-589) and model.compress (AGENT:592); recon_out (nullable)
 *           receives the encoder-side reconstruction as the reference would save it: arrange_channel_dim_to_block_pixels,
 *           crop, + 0.5 and torchvision save_image's 8-bit quantisation (AGENT:610, 628);
 *   decode: model.decompress (AGENT:598) and the same conversion of the decoder's reconstruction.
 * Same streams as lbic_encode_host on the float tensors eval_model would build from these images. */
int lbic_encode_images_u8_host(lbic_model *m, const uint8_t *img, int n_img, int H, int W, uint8_t *recon_out,
                               uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes);
int lbic_decode_images_u8_host(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                               int n_img, int H, int W, uint8_t *img_out, int lanes);

/* The quality figures eval_model logs (AGENT:611-619), computed on the device: per-image MSE of x vs y ((n, C, H, W)
 * fp32 device tensors; PSNR = -10 log10(mse) for the unit-range images the agent compares) and, if msssim_out != NULL,
 * pytorch_msssim.ms_ssim(x + offset, y + offset, data_range) per image (the agent passes offset 0.5, data_range 1.0;
 * the smaller image side must exceed 160).  mse_out / msssim_out: HOST arrays of n doubles; the call synchronises. */
int lbic_image_metrics(lbic_model *m, const float *x, const float *y, int n, int C, int H, int W, float offset,
                       float data_range, double *mse_out, double *msssim_out, void *stream);

/* The optional post-processing module -- BlkBasedPostProcessing (NET:455-476), `use_postpm` in the config JSON,
 * applied by eval_model to the block tensor of the reconstruction (AGENT:604-606).
 *   lbic_load_postpm_weights   the module's state_dict: res_net.0.{weight (4C, C, 3, 3), bias}, res_net.2.{weight (C, 4C, 1, 1), bias}, C = 3B^2
 *   lbic_postprocess           z, out: device (n_img, 3B^2, Hb, Wb) fp32; clamp != 0 applies the caller's clamp_(-0.5, 0.5) */
int lbic_load_postpm_weights(lbic_model *m, const lbic_tensor_desc *tensors, int n_tensors, void *stream);
int lbic_postprocess(lbic_model *m, const float *z, int n_img, int Hb, int Wb, float *out, int clamp, void *stream);

/* Block-row bands: ONE large image split over several GPUs (BASELINE.json config 5).  A rank owns block rows [v0, v1)
 * and runs every wavefront step t = h + 2 v (NET:339-357 restated) restricted to them; the only exchange is the halo:
 * after step t the owner of row v1-1 passes zhat(v1-1, t - 2 (v1-1)) to the rank below before its step t+1 (the caller
 * moves it, e.g. torch.distributed send / recv on views of lbic_band_zhat; lbic_b200/band.py).  KS[1] = 1 only.
 *   lbic_band_begin  x: device (n_img, 3B^2, Hb, Wb) to encode, or NULL with `streams` = lane containers to decode
 *   lbic_band_zhat   device pointer to the working reconstruction, channel-last (n_img, Hb, Wb, 3B^2)
 *   lbic_band_step   step t for block rows [v0, v1)
 *   lbic_band_end    the band's rows of the reconstruction (channel-last) and, after an encode, one rANS stream per
 *                    owned block row (the lanes of the 'LBML' container: n_img * (v1-v0) slots of lane_cap bytes) */
int lbic_band_begin(lbic_model *m, const float *x, int n_img, int Hb, int Wb, const uint8_t *streams,
                    const uint32_t *stream_len, size_t stream_cap, void *stream);
float *lbic_band_zhat(lbic_model *m);
int lbic_band_step(lbic_model *m, int t, int v0, int v1, void *stream);
int lbic_band_end(lbic_model *m, int v0, int v1, float *zhat_rows_out, uint8_t *lane_out, size_t lane_cap,
                  uint32_t *lane_len, void *stream);

/* Worst-case size in bytes of one image's bitstream for the given grid (8 bytes per symbol + 64 per rANS stream + the
 * lane-container header): a buffer of this size cannot overflow, whatever the symbols.  Typical streams are far smaller;
 * callers that size stream_cap from experience must check stream_len / lbic_check_errors. */
size_t lbic_stream_bound(const lbic_model *m, int Hb, int Wb, int lanes);

/* arrange_block_pixels_to_channel_dim / arrange_channel_dim_to_block_pixels -- AGENT:853-873.
 * img: (n, C, Hb*B, Wb*B); blk: (n, C*B*B, Hb, Wb), channel (v*B+h)*C + c.  Device pointers. */
int lbic_space_to_depth(const float *img, float *blk, int n, int C, int Hb, int Wb, int B, void *stream);
int lbic_depth_to_space(const float *blk, float *img, int n, int C, int Hb, int Wb, int B, void *stream);

/* The entropy coder on its own: compressai.ans.BufferedRansEncoder.encode_with_indexes + flush
 * (NET:359-360) and RansDecoder.set_stream + decode_stream (NET:409-410,439) for n_streams
 * independent streams of n_sym symbols each.  Device pointers; symbols int32, indexes uint8. */
int lbic_rans_encode(lbic_model *m, const int32_t *symbols, const uint8_t *indexes, int n_streams,
                     int64_t n_sym, uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len,
                     void *stream);
int lbic_rans_decode(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                     const uint8_t *indexes, int n_streams, int64_t n_sym, int32_t *symbols_out,
                     void *stream);

/* Bring-up / test hook: D[R,cout] = A[R,K] * W[cout,K]^T with fp32 host-visible results, through
 * the selected GEMM core (A, W, D device fp32; the split into fp16 hi/lo planes happens inside). */
int lbic_debug_gemm(lbic_model *m, const float *A, const float *W, float *D, int R, int K, int cout,
                    void *stream);

/* Test hook: ONE fused GEMM layer, D = A0 W0^T (+ A1 W1^T), through an explicitly chosen core form and epilogue, on
 * operands the caller gives in fp32 (split into fp16 hi/lo planes on the device as activations are; the weights are NOT
 * rescaled: pass them as the layer would store them and undo that with acc_scale).  Row r of the step is block r (QUANT /
 * RECON outputs land at row r).  Allocates per call and synchronises `stream`.  With LBIC_OPT_CHECK_SATURATION set, the
 * hi plane is scanned afterwards as a product layer's is (lbic_saturation_count). */
typedef struct {
    int mode;                  /* epilogue: 0 LRELU, 1 PREGDN, 2 GDN, 3 IGDN, 4 KSI, 5 QUANT, 6 RECON, 7 RAW, 8 RESID   */
    int core;                  /* 0 SIMT twin, 1 per-tile tcgen05 kernel, 2 persistent kernel, 3 its CTA-pair form
                                  (tiles <= 192 wide), 4 CTA pair with tiles <= 256 wide                               */
    int force_bn;              /* core 1: tile width (multiple of 16, <= 256); 0 = the automatic width                   */
    int R, cout, nseg;         /* rows, output channels (multiple of 16), K segments (1 or 2)                           */
    int K[2];                  /* segment widths (multiples of 8)                                                         */
    const float *A[2];         /* device, (R, K[s]) fp32 row-major                                                        */
    const float *W[2];         /* device, (cout, K[s]) fp32 row-major                                                     */
    const float *bias;         /* device [cout] (beta for GDN / IGDN), NULL = zeros                                       */
    const float *aux;          /* device: pre-GDN activation (GDN, IGDN), ksi = scales | means (QUANT), residual (RESID) */
    int ld_aux;                /* row stride of aux in elements                                                          */
    float acc_scale;           /* the epilogue computes acc * acc_scale + bias                                            */
    int M;                     /* QUANT: means at aux[r * ld_aux + M + c], symbols / indexes with row stride M (>= cout)  */
    const float *scale_table;  /* QUANT: device, 64 increasing scale levels; NULL = the model's installed table          */
    int no_clamp;              /* RECON / RESID: 1 = no clamp to [-0.5, 0.5]                                              */
    float *out_f32;            /* RAW, PREGDN, KSI, RECON, RESID: (R, cout) fp32; QUANT: (R, M) int32 symbols            */
    uint16_t *out_hi, *out_lo; /* LRELU, PREGDN, GDN, IGDN, QUANT: (R, cout) fp16 bit patterns                           */
    uint8_t *out_idx;          /* QUANT: (R, M) CDF indexes                                                               */
} lbic_debug_layer_args;
int lbic_debug_layer(lbic_model *m, const lbic_debug_layer_args *args, void *stream);

/* Test hook: the rate estimate of lbic_validate for R rows of M channels (row r = block r): ksi (R, ld_ksi) device
 * fp32 with the scales in columns [0, M), sym (R, M) int32, info (R, M) fp32 = -log2 likelihood.  Synchronises. */
int lbic_debug_selfinfo(lbic_model *m, const float *ksi, int ld_ksi, const int32_t *sym, int R, int M, float *info,
                        void *stream);

/* Test hook: the CDF index of n scales (device fp32) as the decoders compute it from `scale_table` (device, 64 levels):
 * idx_bisect[i] by bisection, idx_hinted[i] by the logarithmic hint with its bisection fallback.  Synchronises. */
int lbic_debug_scale_index(lbic_model *m, const float *scales, int n, const float *scale_table, int32_t *idx_bisect,
                           int32_t *idx_hinted, void *stream);

/* Tuning hook: times `iters` back-to-back launches of the D = A W^T tile kernel (EPI_RAW or a PREGDN-style
 * epilogue when with_epilogue != 0) on synthetic operands with CUDA events; returns the mean ms per launch. */
int lbic_debug_gemm_bench(lbic_model *m, int R, int K, int cout, int with_epilogue, int iters, double *ms_per_launch);

/* Number of kernels this library has launched on behalf of `m` since creation. */
/* Debug aid for the fp16 operand planes: every activation is stored as hi + lo fp16 planes, which CLIP at +-65504
 * instead of overflowing (the squares of the GDN layers clip for |x| > 255.9).  With LBIC_OPT_CHECK_SATURATION set, every
 * GEMM layer's hi plane is scanned after the layer (one launch per layer; the dataflow and wave kernels are bypassed,
 * results unchanged) and the clipped elements are counted; this call synchronises `stream` and returns the total since
 * the last reset.  A non-zero count means rate / distortion may deviate from the reference for these weights. */
int lbic_saturation_count(lbic_model *m, void *stream, int64_t *count, int reset);
int64_t lbic_launch_count(const lbic_model *m);
/* Per-kernel-family launch counts and (if timing is enabled) accumulated device milliseconds for
 * the GEMM family; used by bench.py for the roofline line. */
int lbic_set_profiling(lbic_model *m, int enabled);
int lbic_get_profile(lbic_model *m, int64_t *gemm_launches, double *gemm_ms, double *gemm_flops);
/* The same records split by layer, in the order E0 E1 E2 E3 | F0 G0 F1 G1 F2 G2 F3 | D0 IG0 D1 IG1 D2 IG2 D3
 * (get_meanscale / prtr_forward* / prtr_inverse* of graphs/models/BlockBasedImgCompLossy_net.py:262-302; G = the GDN
 * gamma product).  Fills at most max_layers entries of each array and returns the number filled (18), or < 0. */
int lbic_get_layer_profile(lbic_model *m, int max_layers, int64_t *launches, double *ms, double *flops);

#ifdef __cplusplus
}
#endif
#endif /* LBIC_H_ */

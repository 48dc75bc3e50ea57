// C ABI (include/lbic.h): model management, weight packing, workspace, and the wavefront drivers for
// encode (NET:319-361) and decode (NET:400-452).
#include <math.h>
#include <cmath>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "epilogue.cuh"   // epi_has_f32 / epi_has_hilo (lbic_debug_layer)
#include "lbic_internal.h"

// ------------------------------------------------------------------------------------------------
// errors, launch accounting
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
thread_local int64_t *g_launch_counter = nullptr;

int lbic_fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch(int family) {
    if (g_launch_counter) g_launch_counter[family]++;
}

extern "C" const char *lbic_last_error(void) { return g_err; }
extern "C" const char *lbic_version(void) { return "lbic_b200 0.1 (sm_100a; tcgen05 fp16 hi/lo x3 + SIMT twin)"; }

// ------------------------------------------------------------------------------------------------
// model
// ------------------------------------------------------------------------------------------------
namespace {

enum LayerId {
    L_E0, L_E1, L_E2, L_E3,                       // entropy-parameter net (get_meanscale.{0,2,4,6})
    L_F0, L_G0, L_F1, L_G1, L_F2, L_G2, L_F3,     // encoder: prtr_forward1+2, prtr_forward3.{0..5}
    L_D0, L_IG0, L_D1, L_IG1, L_D2, L_IG2, L_D3,  // decoder: prtr_inverse1+2, prtr_inverse3.{0..5}
    L_COUNT
};

constexpr int NBN = LBIC_NBN;

struct PackedSeg {
    int K = 0;
    float *weff = nullptr;   // effective fp32 weights (temporary, freed after the scaled split)
    h16 *hi = nullptr, *lo = nullptr;
    CUtensorMap tm_hi[NBN], tm_lo[NBN];   // TMA box = 64 x bn_v[i]
};

struct PackedLayer {
    int cout = 0, bn = 0, nseg = 0;
    int bn_v[NBN] = {};
    int n_bn = 0;
    PackedSeg seg[2];
    float *bias = nullptr;
    float acc_scale = 1.0f;   // 2^-k, see finish_layer
};

struct ActBuf {
    h16 *hi = nullptr, *lo = nullptr;
    int ld = 0;
};

struct ActView {   // an activation buffer seen as a GEMM A operand of logical width K
    const ActBuf *buf = nullptr;
    int K = 0;
    CUtensorMap tm_hi, tm_lo;         // box 64 k x 128 rows
    CUtensorMap tm_small[4][2];       // boxes of 64 k x 16 / 32 / 48 / 64 rows, [class][hi, lo] (latency kernel)
};

struct Workspace {
    int n_img = 0, Hb = 0, Wb = 0, R_cap = 0;
    float *x_cl = nullptr, *zhat_cl = nullptr;
    ActBuf X, T, YQ, H1, H2, H3, S, U;
    float *A32 = nullptr, *KSI = nullptr;
    int ldA32 = 0, ldKSI = 0;
    ActView vX, vT, vYQ, vH1, vH2, vH3, vS[3], vU[3];
    // KS[1] == 3 only: ring-extended hidden map g0, its per-step tap gather, and the taps of the ring-extended rows
    int R_ext_cap = 0;
    ActBuf G0, H1x5, Text;
    ActView vH1x5, vText;
    int32_t *sym = nullptr;
    uint8_t *idx = nullptr;
    uint32_t *rans_scratch = nullptr;
    size_t rans_scratch_words = 0;   // total words allocated
    RansStreamState *dec_states = nullptr;
    const uint8_t **lane_ptr = nullptr;
    std::vector<ChainLayer> h_chain;   // host copy of the per-layer chain descriptors (indexed by LayerId)
    ChainLayer *d_chain = nullptr;
    int *flow_counters = nullptr;      // (layer, 256-row block) completion counters of the dataflow launch
    size_t flow_counters_cap = 0;
    int *wave_counters = nullptr;      // (list entry, 128-row block) counters of the persistent wavefront kernel
    size_t wave_counters_cap = 0;
    std::vector<void *> allocs;
};

constexpr int LBIC_MAX_BANDS = 16;   // host calls move images in at most this many bands of block rows

struct ProfRec {
    cudaEvent_t a, b;
    double flops;
    int layer;     // LayerId, or -1 for a chain launch covering several layers
};

}  // namespace

struct lbic_model {
    lbic_config cfg;
    int device = 0;
    int Cin = 0, N = 0, C2 = 0, C3 = 0, M = 0, E1 = 0, E2 = 0, E3 = 0, EO = 0, k1 = 1;
    PackedLayer L[L_COUNT];
    bool weights_loaded = false;
    // optional post-processing net (BlkBasedPostProcessing, NET:455-476): 3x3 conv (all nine taps) -> lrelu -> 1x1 conv
    PackedLayer PP[2];
    bool postpm_loaded = false;
    std::vector<void *> pp_allocs;       // its packed weights
    ActBuf PPA, PPH;                     // nine-tap operand (9 * 3B^2 wide) and hidden activations (4 * 3B^2)
    ActView vPPA, vPPH;
    int pp_rcap = 0;
    std::vector<void *> pp_ws_allocs;
    std::vector<void *> weight_allocs;
    Tables tables;
    Workspace ws;
    int gemm_core = 0;
    int force_bn = 0;
    int use_ws = 1;        // warp-specialised persistent kernel for large steps
    int use_pair = 1;      // CTA-pair (cta_group::2) form of the persistent kernel
    int use_flow = 1;      // dataflow launch of a whole layer range per step (1 = steps with >= flow_min_rows rows, 2 = always)
    int flow_min_rows = 2560;       // (profiles/r2_midsize.log: 2048 gains 4-8 % at 128-256 images and loses 2 % at 48)
    int flow_pair_min_rows = 8192;   // dataflow steps below this many rows run on single CTAs (128 x 96 tiles), from it on CTA pairs
    int flow_quad = 0;     // large steps: dataflow launch on clusters of four (activation operand shared by TMA multicast)
    int flow_small = 0;    // steps below flow_min_rows: 1 = single-CTA dataflow launch with 96-wide tiles, 0 = one launch per
                           // layer (default: the counter hand-off costs as much as a PDL-chained launch, profiles/r1_dataflow.md)
    int flow_max_rows = 1 << 30;
    int use_wave = 1;      // persistent wavefront (latency) kernel for steps of at most wave_max_rows rows (KS[1] == 1)
    int wave_max_rows = 1536;
    int wave_dec_max_rows = 64;    // decode: the rANS tiles run one warp per row on 8 entropy CTAs (64 rows at a time)
    int wave_bn = 0;               // forced tile width of the wave kernel (32 / 64 / 128), 0 = by rows per step
    float *selfinfo_cl = nullptr;   // set by lbic_validate for the duration of the call: (n,Hb,Wb,M) self-information
    cudaStream_t hs[3] = {nullptr, nullptr, nullptr};   // host-call pipeline: copies in, compute, copies out
    cudaEvent_t hev[2 * LBIC_MAX_BANDS] = {};            // band b copied in / band b ready to copy out
    // grow-only device temporaries of lbic_validate / lbic_forward (channel-last self-information, reconstruction)
    float *aux[3] = {nullptr, nullptr, nullptr};     // [2]: scratch of lbic_image_metrics
    size_t aux_bytes[3] = {0, 0, 0};
    int host_bands = LBIC_MAX_BANDS;   // host calls: bands of block rows per batch (copy / compute overlap granularity)
    float *recon_cl = nullptr;      // set by lbic_forward: the decoder net writes here instead of the zhat feedback buffer
    int recon_no_clamp = 0;
    // block-row-band mode (one large image over several GPUs): geometry of the call in progress
    int band_n = 0, band_Hb = 0, band_Wb = 0, band_decode = 0;
    int64_t launches[2] = {0, 0};
    int *err_flag = nullptr;
    // debug: count the elements of every fp16 operand plane a GEMM layer writes that were clipped at +-65504
    // (LBIC_OPT_CHECK_SATURATION: per-layer launches only, one scan per layer; lbic_saturation_count reads the total)
    int check_sat = 0;
    unsigned long long *d_sat = nullptr;
    // the workspace is shared by all calls on this model: a call on another stream than the previous one waits for it
    cudaEvent_t ws_event = nullptr;
    cudaStream_t ws_stream = nullptr;
    bool ws_used = false;
    // host-call staging
    void *io_dev = nullptr;
    size_t io_bytes = 0;
    // profiling
    int profiling = 0;
    std::vector<ProfRec> prof;
};

namespace {

struct Active {   // routes launch counting to the model for the duration of an API call
    explicit Active(lbic_model *m) {
        g_launch_counter = m ? m->launches : nullptr;
        if (m) cudaSetDevice(m->device);
    }
    ~Active() { g_launch_counter = nullptr; }
};

int dev_alloc(std::vector<void *> &list, void **p, size_t bytes, bool zero = false) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) return lbic_fail(LBIC_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    list.push_back(*p);
    if (zero) LBIC_CUDA(cudaMemset(*p, 0, bytes));
    return 0;
}

void free_all(std::vector<void *> &list) {
    for (void *p : list) cudaFree(p);
    list.clear();
}

// tile-width variants of a layer, one per split factor (lbic_split): widest first
int bn_variants(int cout, int *out) {
    for (int i = 0; i < NBN; ++i) {
        if (i == LBIC_QUAD_VARIANT) {
            int nt = (cout + gemm_ws_max_bn() - 1) / gemm_ws_max_bn();
            nt += nt & 1;
            out[i] = ((cout + nt - 1) / nt + 15) / 16 * 16;
            continue;
        }
        if (i >= LBIC_WS_VARIANT) {
            const int wmax = i == LBIC_PAIR_WIDE ? gemm_pair_max_bn()
                             : i == LBIC_SMALL_VARIANT ? gemm_ws_max_bn() / 2
                             : i == LBIC_LAT_VARIANT ? 32 : i == LBIC_LAT64_VARIANT ? 64 : i == LBIC_LAT128_VARIANT ? 128
                             : gemm_ws_max_bn();
            const int nt = (cout + wmax - 1) / wmax;
            out[i] = ((cout + nt - 1) / nt + 15) / 16 * 16;
            continue;
        }
        const int f = lbic_split(i);
        const int ntiles = f * ((cout + 256 * f - 1) / (256 * f));
        int bn = ((cout + ntiles - 1) / ntiles + 15) / 16 * 16;
        out[i] = bn < 16 ? 16 : bn;
    }
    return NBN;
}

int pick_bn(int cout) {
    const int ntiles = (cout + 255) / 256;
    int bn = (cout + ntiles - 1) / ntiles;
    bn = (bn + 15) / 16 * 16;
    return bn;
}

// ---- weight loading ---------------------------------------------------------------------------
struct SdView {
    std::map<std::string, const lbic_tensor_desc *> by_name;
    const lbic_tensor_desc *find(const std::string &k) const {
        auto it = by_name.find(k);
        return it == by_name.end() ? nullptr : it->second;
    }
};

int64_t numel(const lbic_tensor_desc *t) {
    int64_t n = 1;
    for (int i = 0; i < t->ndim; ++i) n *= t->shape[i];
    return n;
}

// copies a state_dict tensor to a temporary device buffer (host or device source)
int stage(const SdView &sd, const std::string &name, int64_t expect, std::vector<void *> &tmp, float **out,
          cudaStream_t st) {
    const lbic_tensor_desc *t = sd.find(name);
    if (!t) return lbic_fail(LBIC_ERR_STATE, "state_dict is missing key '%s'", name.c_str());
    if (numel(t) != expect)
        return lbic_fail(LBIC_ERR_INVALID, "state_dict['%s'] has %lld elements, expected %lld", name.c_str(),
                         (long long)numel(t), (long long)expect);
    LBIC_TRY(dev_alloc(tmp, (void **)out, sizeof(float) * (size_t)expect));
    LBIC_CUDA(cudaMemcpyAsync(*out, t->data, sizeof(float) * (size_t)expect, cudaMemcpyDefault, st));
    return 0;
}

int scalar(const SdView &sd, const std::string &name, float fallback, float *out) {
    const lbic_tensor_desc *t = sd.find(name);
    *out = fallback;
    if (t && numel(t) == 1) LBIC_CUDA(cudaMemcpy(out, t->data, sizeof(float), cudaMemcpyDefault));
    return 0;
}

const int TAPS_A[8] = {0, 0, 0, 1, 0, 2, 1, 0};            // 3x3 mask 'A' live taps (kh,kw)  MC:12-17
const int TAPS_B[10] = {0, 0, 0, 1, 0, 2, 1, 0, 1, 1};     // 3x3 mask 'B' adds the centre
const int TAPS_1[2] = {0, 0};
const int TAPS_9[18] = {0, 0, 0, 1, 0, 2, 1, 0, 1, 1, 1, 2, 2, 0, 2, 1, 2, 2};   // plain 3x3 conv (post-processing net)

int pack_conv_seg(lbic_model *m, const SdView &sd, const std::string &prefix, int cout, int cin, int k,
                  const int *taps, int ntaps, int bn, PackedSeg &seg, float **bias_tmp, std::vector<void *> &tmp,
                  cudaStream_t st) {
    float *w = nullptr, *mask = nullptr;
    const int64_t nw = (int64_t)cout * cin * k * k;
    LBIC_TRY(stage(sd, prefix + ".weight", nw, tmp, &w, st));
    if (sd.find(prefix + ".mask")) LBIC_TRY(stage(sd, prefix + ".mask", nw, tmp, &mask, st));
    LBIC_TRY(stage(sd, prefix + ".bias", cout, tmp, bias_tmp, st));
    seg.K = ntaps * cin;
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&seg.hi, sizeof(h16) * (size_t)cout * seg.K));
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&seg.lo, sizeof(h16) * (size_t)cout * seg.K));
    LBIC_TRY(dev_alloc(tmp, (void **)&seg.weff, sizeof(float) * (size_t)cout * seg.K));
    LBIC_TRY(launch_pack_conv(w, mask, cout, cin, k, k, taps, ntaps, seg.weff, seg.K, st));
    int bnv[NBN];
    const int nb = bn_variants(cout, bnv);
    (void)bn;
    for (int i = 0; i < nb; ++i) {
        const int box = (i == LBIC_PAIR_VARIANT || i == LBIC_PAIR_WIDE || i == LBIC_QUAD_VARIANT) ? bnv[i] / 2 : bnv[i];   // a CTA pair loads half the tile per CTA
        LBIC_TRY(make_tmap_2d(&seg.tm_hi[i], seg.hi, seg.K, cout, seg.K, 64, box));
        LBIC_TRY(make_tmap_2d(&seg.tm_lo[i], seg.lo, seg.K, cout, seg.K, 64, box));
    }
    return 0;
}

// fp16 operand planes need the weights inside fp16's normal range: scale the layer's effective weights by 2^k so
// that max |w| lands in [2^9, 2^10), split into hi/lo, and undo the scale exactly in the epilogue (acc_scale = 2^-k).
int finish_layer(lbic_model *m, PackedLayer &L, cudaStream_t st) {
    float *d_max = nullptr;
    std::vector<void *> tmp;
    LBIC_TRY(dev_alloc(tmp, (void **)&d_max, sizeof(float), true));
    for (int s = 0; s < L.nseg; ++s) LBIC_TRY(launch_absmax(L.seg[s].weff, (int64_t)L.cout * L.seg[s].K, d_max, st));
    float mx = 0.0f;
    LBIC_CUDA(cudaMemcpyAsync(&mx, d_max, sizeof(float), cudaMemcpyDeviceToHost, st));
    LBIC_CUDA(cudaStreamSynchronize(st));
    free_all(tmp);
    int k = 0;
    if (mx > 0.0f && std::isfinite(mx)) k = 9 - (int)floorf(log2f(mx));
    k = k > 24 ? 24 : (k < -24 ? -24 : k);
    const float scale = ldexpf(1.0f, k);
    L.acc_scale = ldexpf(1.0f, -k);
    for (int s = 0; s < L.nseg; ++s)
        LBIC_TRY(launch_split_scaled(L.seg[s].weff, L.seg[s].hi, L.seg[s].lo, (int64_t)L.cout * L.seg[s].K, scale, st));
    (void)m;
    return 0;
}

int pack_linear_into(lbic_model *m, PackedLayer &L, const SdView &sd, const std::string &prefix, int cout, int cin, int k,
                     const int *taps, int ntaps, std::vector<void *> &tmp, cudaStream_t st);
int pack_linear(lbic_model *m, const SdView &sd, int id, const std::string &prefix, int cout, int cin, int k,
                const int *taps, int ntaps, std::vector<void *> &tmp, cudaStream_t st) {
    return pack_linear_into(m, m->L[id], sd, prefix, cout, cin, k, taps, ntaps, tmp, st);
}
int pack_linear_into(lbic_model *m, PackedLayer &L, const SdView &sd, const std::string &prefix, int cout, int cin, int k,
                     const int *taps, int ntaps, std::vector<void *> &tmp, cudaStream_t st) {
    L.cout = cout;
    L.bn = pick_bn(cout);
    L.n_bn = bn_variants(cout, L.bn_v);
    L.nseg = 1;
    float *b = nullptr;
    LBIC_TRY(pack_conv_seg(m, sd, prefix, cout, cin, k, taps, ntaps, L.bn, L.seg[0], &b, tmp, st));
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&L.bias, sizeof(float) * cout));
    LBIC_TRY(launch_add_vec(b, nullptr, L.bias, cout, st));
    return finish_layer(m, L, st);
}

// first layer of the encoder / decoder nets: 1x1 conv on x (or y_qnt) plus masked 3x3 conv on zhat, summed
int pack_dual(lbic_model *m, const SdView &sd, int id, const std::string &p1, int cin1, const std::string &p2,
              int cout, std::vector<void *> &tmp, cudaStream_t st) {
    PackedLayer &L = m->L[id];
    L.cout = cout;
    L.bn = pick_bn(cout);
    L.n_bn = bn_variants(cout, L.bn_v);
    L.nseg = 2;
    float *b1 = nullptr, *b2 = nullptr;
    LBIC_TRY(pack_conv_seg(m, sd, p1, cout, cin1, 1, TAPS_1, 1, L.bn, L.seg[0], &b1, tmp, st));
    LBIC_TRY(pack_conv_seg(m, sd, p2, cout, m->Cin, 3, TAPS_A, 4, L.bn, L.seg[1], &b2, tmp, st));
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&L.bias, sizeof(float) * cout));
    LBIC_TRY(launch_add_vec(b1, b2, L.bias, cout, st));
    return finish_layer(m, L, st);
}

int pack_gdn(lbic_model *m, const SdView &sd, int id, const std::string &prefix, int C, std::vector<void *> &tmp,
             cudaStream_t st) {
    PackedLayer &L = m->L[id];
    L.cout = C;
    L.bn = pick_bn(C);
    L.n_bn = bn_variants(C, L.bn_v);
    L.nseg = 1;
    float *g = nullptr, *b = nullptr;
    LBIC_TRY(stage(sd, prefix + ".gamma", (int64_t)C * C, tmp, &g, st));
    LBIC_TRY(stage(sd, prefix + ".beta", C, tmp, &b, st));
    // defaults = NonNegativeParametrizer constants (utils/parametrizers.py:33-40, GDNF:55-61)
    const float ped = (float)pow(2.0, -36.0);
    float gped, gbound, bped, bbound;
    LBIC_TRY(scalar(sd, prefix + ".gamma_reparam.pedestal", ped, &gped));
    LBIC_TRY(scalar(sd, prefix + ".gamma_reparam.lower_bound.bound", (float)sqrt(0.0 + pow(2.0, -36.0)), &gbound));
    LBIC_TRY(scalar(sd, prefix + ".beta_reparam.pedestal", ped, &bped));
    LBIC_TRY(scalar(sd, prefix + ".beta_reparam.lower_bound.bound", (float)sqrt(1e-6 + pow(2.0, -36.0)), &bbound));
    PackedSeg &seg = L.seg[0];
    seg.K = C;
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&seg.hi, sizeof(h16) * (size_t)C * C));
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&seg.lo, sizeof(h16) * (size_t)C * C));
    LBIC_TRY(dev_alloc(m->weight_allocs, (void **)&L.bias, sizeof(float) * C));
    LBIC_TRY(dev_alloc(tmp, (void **)&seg.weff, sizeof(float) * (size_t)C * C));
    LBIC_TRY(launch_pack_gdn(g, b, C, gbound, gped, bbound, bped, seg.weff, C, L.bias, st));
    for (int i = 0; i < L.n_bn; ++i) {
        const int box = (i == LBIC_PAIR_VARIANT || i == LBIC_PAIR_WIDE || i == LBIC_QUAD_VARIANT) ? L.bn_v[i] / 2 : L.bn_v[i];
        LBIC_TRY(make_tmap_2d(&seg.tm_hi[i], seg.hi, C, C, C, 64, box));
        LBIC_TRY(make_tmap_2d(&seg.tm_lo[i], seg.lo, C, C, C, 64, box));
    }
    return finish_layer(m, L, st);
}

// ---- workspace ----------------------------------------------------------------------------------
int alloc_act(Workspace &ws, ActBuf &b, int ld) {
    b.ld = ld;
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&b.hi, sizeof(h16) * (size_t)ws.R_cap * ld, true));
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&b.lo, sizeof(h16) * (size_t)ws.R_cap * ld, true));
    return 0;
}

int make_view(Workspace &ws, ActView &v, const ActBuf &b, int K) {
    v.buf = &b;
    v.K = K;
    LBIC_TRY(make_tmap_2d(&v.tm_hi, b.hi, K, ws.R_cap, b.ld, 64, 128));
    LBIC_TRY(make_tmap_2d(&v.tm_lo, b.lo, K, ws.R_cap, b.ld, 64, 128));
    for (int c = 0; c < 4; ++c) {
        LBIC_TRY(make_tmap_2d(&v.tm_small[c][0], b.hi, K, ws.R_cap, b.ld, 64, lbic_box_rows(c)));
        LBIC_TRY(make_tmap_2d(&v.tm_small[c][1], b.lo, K, ws.R_cap, b.ld, 64, lbic_box_rows(c)));
    }
    return 0;
}

int build_chain(lbic_model *m);
EpiParams epi(int mode, const StepDesc &sd);
EpiParams epi_hilo(int mode, const StepDesc &sd, const ActBuf &out);
EpiParams epi_pregdn(lbic_model *m, const StepDesc &sd);

int ensure_workspace(lbic_model *m, int n_img, int Hb, int Wb) {
    Workspace &ws = m->ws;
    if (ws.n_img >= n_img && ws.Hb == Hb && ws.Wb == Wb) return 0;
    LBIC_CUDA(cudaDeviceSynchronize());
    free_all(ws.allocs);
    ws = Workspace();
    ws.n_img = n_img; ws.Hb = Hb; ws.Wb = Wb;
    const int max_nv = Hb < (Wb + 1) / 2 ? Hb : (Wb + 1) / 2;
    ws.R_cap = ((n_img * max_nv) + 127) / 128 * 128;
    const size_t nblk = (size_t)n_img * Hb * Wb;
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.x_cl, sizeof(float) * nblk * m->Cin));
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.zhat_cl, sizeof(float) * nblk * m->Cin));
    LBIC_TRY(alloc_act(ws, ws.X, m->Cin));
    LBIC_TRY(alloc_act(ws, ws.T, 4 * m->Cin));
    LBIC_TRY(alloc_act(ws, ws.YQ, m->M));
    LBIC_TRY(alloc_act(ws, ws.H1, m->E1));
    if (m->k1 == 3) {
        ws.R_ext_cap = ((n_img * (max_nv + 2)) + 127) / 128 * 128;
        const size_t npos = (size_t)n_img * (Hb + 1) * (Wb + 2);
        ws.G0.ld = m->E1;
        LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.G0.hi, sizeof(h16) * npos * m->E1, true));
        LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.G0.lo, sizeof(h16) * npos * m->E1, true));
        LBIC_TRY(alloc_act(ws, ws.H1x5, 5 * m->E1));
        ws.Text.ld = 4 * m->Cin;
        LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.Text.hi, sizeof(h16) * (size_t)ws.R_ext_cap * ws.Text.ld, true));
        LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.Text.lo, sizeof(h16) * (size_t)ws.R_ext_cap * ws.Text.ld, true));
    }
    LBIC_TRY(alloc_act(ws, ws.H2, m->E2));
    LBIC_TRY(alloc_act(ws, ws.H3, m->E3));
    LBIC_TRY(alloc_act(ws, ws.S, m->N));
    LBIC_TRY(alloc_act(ws, ws.U, m->N));
    ws.ldA32 = m->N; ws.ldKSI = m->EO;
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.A32, sizeof(float) * (size_t)ws.R_cap * ws.ldA32, true));
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.KSI, sizeof(float) * (size_t)ws.R_cap * ws.ldKSI, true));
    LBIC_TRY(make_view(ws, ws.vX, ws.X, m->Cin));
    LBIC_TRY(make_view(ws, ws.vT, ws.T, 4 * m->Cin));
    LBIC_TRY(make_view(ws, ws.vYQ, ws.YQ, m->M));
    LBIC_TRY(make_view(ws, ws.vH1, ws.H1, m->E1));
    if (m->k1 == 3) {
        LBIC_TRY(make_view(ws, ws.vH1x5, ws.H1x5, 5 * m->E1));
        ws.vText.buf = &ws.Text; ws.vText.K = 4 * m->Cin;
        LBIC_TRY(make_tmap_2d(&ws.vText.tm_hi, ws.Text.hi, 4 * m->Cin, ws.R_ext_cap, ws.Text.ld, 64, 128));
        LBIC_TRY(make_tmap_2d(&ws.vText.tm_lo, ws.Text.lo, 4 * m->Cin, ws.R_ext_cap, ws.Text.ld, 64, 128));
        for (int c = 0; c < 4; ++c) {
            LBIC_TRY(make_tmap_2d(&ws.vText.tm_small[c][0], ws.Text.hi, 4 * m->Cin, ws.R_ext_cap, ws.Text.ld, 64, lbic_box_rows(c)));
            LBIC_TRY(make_tmap_2d(&ws.vText.tm_small[c][1], ws.Text.lo, 4 * m->Cin, ws.R_ext_cap, ws.Text.ld, 64, lbic_box_rows(c)));
        }
    }
    LBIC_TRY(make_view(ws, ws.vH2, ws.H2, m->E2));
    LBIC_TRY(make_view(ws, ws.vH3, ws.H3, m->E3));
    const int wd[3] = {m->N, m->C2, m->C3};
    for (int i = 0; i < 3; ++i) {
        LBIC_TRY(make_view(ws, ws.vS[i], ws.S, wd[i]));
        LBIC_TRY(make_view(ws, ws.vU[i], ws.U, wd[i]));
    }
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.sym, sizeof(int32_t) * nblk * m->M));
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.idx, nblk * m->M));
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.dec_states, sizeof(RansStreamState) * (size_t)n_img * Hb));
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.lane_ptr, sizeof(void *) * (size_t)n_img * Hb));
    LBIC_TRY(build_chain(m));
    ws.flow_counters_cap = (size_t)L_COUNT * ((ws.R_cap + 127) / 128 + 1);
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.flow_counters, sizeof(int) * ws.flow_counters_cap, true));
    ws.wave_counters_cap = 24 * 32;
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.wave_counters, sizeof(int) * ws.wave_counters_cap, true));
    return 0;
}

// Per-layer descriptors of the persistent chain kernel: the same operand views and epilogues run_ent / run_enc /
// run_dec pass to the per-layer path, indexed by LayerId (so [L_E0, L_COUNT) is a whole encode step).
int build_chain(lbic_model *m) {
    Workspace &ws = m->ws;
    ws.h_chain.assign(L_COUNT, ChainLayer());
    StepDesc none;
    memset(&none, 0, sizeof(none));
    auto set = [&](int id, const ActView *a0, const ActView *a1, EpiParams ep) {
        ChainLayer &c = ws.h_chain[id];
        const PackedLayer &L = m->L[id];
        memset(&c, 0, sizeof(c));
        c.nseg = L.nseg; c.cout = L.cout; c.n_bn = L.n_bn;
        const ActView *av[2] = {a0, a1};
        for (int s = 0; s < L.nseg; ++s) {
            c.kb[s] = (L.seg[s].K + 63) / 64;
            c.tmA[s][0] = av[s]->tm_hi; c.tmA[s][1] = av[s]->tm_lo;
            for (int b = 0; b < 4; ++b) { c.tmAs[b][s][0] = av[s]->tm_small[b][0]; c.tmAs[b][s][1] = av[s]->tm_small[b][1]; }
            for (int v = 0; v < L.n_bn; ++v) { c.tmW[v][s][0] = L.seg[s].tm_hi[v]; c.tmW[v][s][1] = L.seg[s].tm_lo[v]; }
        }
        for (int v = 0; v < L.n_bn; ++v) c.bn_v[v] = L.bn_v[v];
        ep.cout = L.cout; ep.bias = L.bias; ep.scale_tab = m->tables.d_scale_table; ep.acc_scale = L.acc_scale;
        c.ep = ep;
        // output descriptors for the TMA-store epilogue: layers whose output rows are the step's compact rows
        const bool row_indexed = (ep.mode == EPI_LRELU && !ep.out_pos && !(id == L_E0 && m->k1 == 3)) || ep.mode == EPI_PREGDN || ep.mode == EPI_GDN ||
                                 ep.mode == EPI_IGDN || ep.mode == EPI_KSI;
        c.tma_out = 0;
        if (row_indexed) {
            bool ok = true;
            const bool has_hilo = ep.mode != EPI_KSI, has_f32 = ep.mode == EPI_PREGDN || ep.mode == EPI_KSI;
            if (has_hilo)
                ok = make_tmap_2d_ex(&c.tmO[0], ep.out_hi, 2, L.cout, ws.R_cap, ep.ld_out, 16, 128, 32) == 0 &&
                     make_tmap_2d_ex(&c.tmO[1], ep.out_lo, 2, L.cout, ws.R_cap, ep.ld_out, 16, 128, 32) == 0;
            if (ok && has_hilo)
                ok = make_tmap_2d_ex(&c.tmO[3], ep.out_hi, 2, L.cout, ws.R_cap, ep.ld_out, 64, 128, 128) == 0 &&
                     make_tmap_2d_ex(&c.tmO[4], ep.out_lo, 2, L.cout, ws.R_cap, ep.ld_out, 64, 128, 128) == 0;
            if (ok && has_f32)
                ok = make_tmap_2d_ex(&c.tmO[2], ep.out_f32, 4, L.cout, ws.R_cap, ep.ld_f32, 16, 128, 64) == 0 &&
                     make_tmap_2d_ex(&c.tmO[5], ep.out_f32, 4, L.cout, ws.R_cap, ep.ld_f32, 32, 128, 128) == 0;
            c.tma_out = ok ? 1 : 0;
        }
    };
    auto pre = [&]() { return epi_pregdn(m, none); };
    auto gdn = [&](bool inv) {
        EpiParams e = epi_hilo(inv ? EPI_IGDN : EPI_GDN, none, ws.U);
        e.aux = ws.A32; e.ld_aux = ws.ldA32;
        return e;
    };
    if (m->k1 == 3) {
        {
            EpiParams e0 = epi_hilo(EPI_LRELU, none, ws.G0);                // rows of the EXTENDED step, scattered into the g0
            e0.out_pos = 1;                                                 // store (wave kernel; the dataflow launch starts at E1)
            set(L_E0, &ws.vText, nullptr, e0);
        }
        set(L_E1, &ws.vH1x5, nullptr, epi_hilo(EPI_LRELU, none, ws.H2));
    } else {
        set(L_E0, &ws.vT, nullptr, epi_hilo(EPI_LRELU, none, ws.H1));
        set(L_E1, &ws.vH1, nullptr, epi_hilo(EPI_LRELU, none, ws.H2));
    }
    set(L_E2, &ws.vH2, nullptr, epi_hilo(EPI_LRELU, none, ws.H3));
    {
        EpiParams e = epi(EPI_KSI, none);
        e.out_f32 = ws.KSI; e.ld_f32 = ws.ldKSI;
        set(L_E3, &ws.vH3, nullptr, e);
    }
    set(L_F0, &ws.vX, &ws.vT, pre());
    set(L_G0, &ws.vS[0], nullptr, gdn(false));
    set(L_F1, &ws.vU[0], nullptr, pre());
    set(L_G1, &ws.vS[1], nullptr, gdn(false));
    set(L_F2, &ws.vU[1], nullptr, pre());
    set(L_G2, &ws.vS[2], nullptr, gdn(false));
    {
        EpiParams e = epi_hilo(EPI_QUANT, none, ws.YQ);
        e.aux = ws.KSI; e.ld_aux = ws.ldKSI; e.M = m->M; e.sym = ws.sym; e.idx = ws.idx;
        set(L_F3, &ws.vU[2], nullptr, e);
    }
    set(L_D0, &ws.vYQ, &ws.vT, pre());
    set(L_IG0, &ws.vS[0], nullptr, gdn(true));
    set(L_D1, &ws.vU[0], nullptr, pre());
    set(L_IG1, &ws.vS[1], nullptr, gdn(true));
    set(L_D2, &ws.vU[1], nullptr, pre());
    set(L_IG2, &ws.vS[2], nullptr, gdn(true));
    {
        EpiParams e = epi(EPI_RECON, none);
        e.zhat = ws.zhat_cl;
        set(L_D3, &ws.vU[2], nullptr, e);
    }
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.d_chain, sizeof(ChainLayer) * L_COUNT));
    LBIC_CUDA(cudaMemcpy(ws.d_chain, ws.h_chain.data(), sizeof(ChainLayer) * L_COUNT, cudaMemcpyHostToDevice));
    return 0;
}

// which layers each layer reads from (operands and epilogue side inputs), by LayerId; -1 = inputs of the step
const int FLOW_DEP[L_COUNT][2] = {
    {-1, -1}, {L_E0, -1}, {L_E1, -1}, {L_E2, -1},                                              // E0..E3
    {-1, -1}, {L_F0, -1}, {L_G0, -1}, {L_F1, -1}, {L_G1, -1}, {L_F2, -1}, {L_G2, L_E3},          // F0 G0 F1 G1 F2 G2 F3 (ksi)
    {L_F3, -1}, {L_D0, -1}, {L_IG0, -1}, {L_D1, -1}, {L_IG1, -1}, {L_D2, -1}, {L_IG2, -1}};     // D0 IG0 D1 IG1 D2 IG2 D3

// 0: one launch per layer; 1: dataflow launch on CTA pairs (large steps); 2: dataflow launch on single CTAs (small steps)
int flow_applies(const lbic_model *m, int R) {
    if (m->check_sat) return 0;
    if (m->gemm_core != 0 || !m->use_pair || !m->use_flow || m->force_bn || !gemm_flow_supported()) return 0;
    if (m->use_flow == 2) return 1;
    // mid-size steps: the single-CTA form has twice the tiles per worker (128 x 96 on 148 CTAs against 256 x 192 on 74
    // pairs), which is what a step of 4-8 k rows needs to keep the workers busy across layer boundaries; from ~8 k rows
    // the pair form's smaller operand traffic wins (profiles/r2_midsize.log)
    // (the threshold is quoted for 768-wide layers and scales with the tiles per row block, i.e. inversely with N).
    // KS[1] = 3 topologies (five-tap second entropy layer, K = 5 E1) measure no gain from the single-CTA window
    // (B8_highrate at 64 / 128 / 256 images: 110 / 153 / 187 against 112 / 152 / 189 Mpixel/s): pairs from 4096 rows as before.
    if (m->k1 == 3) return (R >= (m->flow_min_rows > 4096 ? m->flow_min_rows : 4096) && R <= m->flow_max_rows) ? 1 : ((m->flow_small && R < m->flow_min_rows) ? 2 : 0);
    if (R >= m->flow_min_rows && R <= m->flow_max_rows)
        return (long)R * (m->N > 0 ? m->N : 768) >= (long)m->flow_pair_min_rows * 768 ? 1 : 2;
    return (m->flow_small && R < m->flow_min_rows) ? 2 : 0;
}

int run_flow(lbic_model *m, int l0, int l1, const StepDesc &sd, int R, cudaStream_t st) {
    Workspace &ws = m->ws;
    ProfRec rec;
    if (m->profiling) {
        double fl = 0;
        for (int l = l0; l < l1; ++l)
            for (int s = 0; s < m->L[l].nseg; ++s) fl += 2.0 * R * (double)m->L[l].seg[s].K * m->L[l].cout;
        cudaEventCreate(&rec.a); cudaEventCreate(&rec.b);
        rec.flops = fl;
        rec.layer = -1;
        cudaEventRecord(rec.a, st);
    }
    const int mode = flow_applies(m, R) == 1 ? 1 : 0;
    int rc = LBIC_FLOW_REFUSED;
    if (mode == 1 && m->flow_quad) {
        rc = gemm_flow_launch(ws.d_chain, ws.h_chain.data(), l0, l1, FLOW_DEP, R, sd, ws.flow_counters, ws.flow_counters_cap, st, 2);
        if (rc == LBIC_FLOW_REFUSED) m->flow_quad = 0;       // no clusters of four on this device: CTA pairs from now on
    }
    if (rc == LBIC_FLOW_REFUSED)
        rc = gemm_flow_launch(ws.d_chain, ws.h_chain.data(), l0, l1, FLOW_DEP, R, sd, ws.flow_counters, ws.flow_counters_cap, st,
                              mode);
    if (m->profiling) {
        cudaEventRecord(rec.b, st);
        m->prof.push_back(rec);
    }
    return rc;
}

int ensure_rans_scratch(lbic_model *m, size_t words) {
    Workspace &ws = m->ws;
    if (ws.rans_scratch_words >= words) return 0;
    // (old block stays in ws.allocs until the workspace is rebuilt; growth is rare)
    LBIC_TRY(dev_alloc(ws.allocs, (void **)&ws.rans_scratch, sizeof(uint32_t) * words));
    ws.rans_scratch_words = words;
    return 0;
}

// ---- GEMM dispatch --------------------------------------------------------------------------------
int run_gemm_layer(lbic_model *m, const PackedLayer &L, int id, int R, const ActView *a0, const ActView *a1, EpiParams ep,
                   cudaStream_t st);
int run_gemm(lbic_model *m, int id, int R, const ActView *a0, const ActView *a1, EpiParams ep, cudaStream_t st) {
    return run_gemm_layer(m, m->L[id], id, R, a0, a1, ep, st);
}
int run_gemm_layer(lbic_model *m, const PackedLayer &L, int id, int R, const ActView *a0, const ActView *a1, EpiParams ep,
                   cudaStream_t st) {
    GemmCall g;
    // Tile width: the widest variant that still gives about one CTA per SM; small steps (few rows) take narrower
    // tiles so that more SMs share the layer -- the result does not depend on the choice (no split-K, fixed k order).
    int vi = 0;
    bool ws = false;
    const int row_tiles = (R + 127) / 128;
    if (m->force_bn) {
        for (int i = 0; i < L.n_bn && i < LBIC_PAIR_VARIANT; ++i)
            if (L.bn_v[i] == m->force_bn) vi = i;
    } else if (m->gemm_core == 0 && m->use_ws &&
               (m->use_ws == 2 ||
                row_tiles * ((L.cout + L.bn_v[LBIC_WS_VARIANT] - 1) / L.bn_v[LBIC_WS_VARIANT]) >= 148)) {
        // at least one tile per SM: the persistent kernel overlaps each tile's epilogue with the next mainloop
        vi = LBIC_WS_VARIANT;
        ws = true;
        if (m->use_pair) {
            // Both pair tilings are L2-bandwidth bound: pick the one that moves fewer bytes per SM over the launch,
            // rounds of tiles (74 clusters) x bytes per tile (operand loads of one CTA + its output rows).
            int ktot = 0;
            for (int s = 0; s < L.nseg; ++s) ktot += (L.seg[s].K + 63) / 64 * 64;
            const int md = ep.mode;   // bytes per output element: fp32 plane, hi+lo planes, (GDN) pre-activation read back
            const int out_b = ((md == EPI_RAW || md == EPI_PREGDN || md == EPI_KSI || md == EPI_RECON || md == EPI_QUANT || md == EPI_RESID) ? 4 : 0) +
                              ((md == EPI_LRELU || md == EPI_PREGDN || md == EPI_GDN || md == EPI_IGDN || md == EPI_QUANT) ? 4 : 0) +
                              ((md == EPI_GDN || md == EPI_IGDN) ? 4 : 0);
            const int rt2 = (R + 255) / 256;
            double best = 0;
            const int cand[2] = {LBIC_PAIR_VARIANT, LBIC_PAIR_WIDE};
            for (int c = 0; c < (m->use_pair == 2 ? 1 : 2); ++c) {
                const int bnc = L.bn_v[cand[c]];
                const int tiles = rt2 * ((L.cout + bnc - 1) / bnc);
                const double cost = (double)((tiles + 73) / 74) * ((double)ktot * (128 + bnc / 2) * 4 + 128.0 * bnc * out_b);
                if (c == 0 || cost < best) { best = cost; vi = cand[c]; }
            }
        }
    } else {
        while (vi + 1 < LBIC_WS_VARIANT && row_tiles * ((L.cout + L.bn_v[vi] - 1) / L.bn_v[vi]) < 132) ++vi;
    }
    g.R = R; g.cout = L.cout; g.bn = L.bn_v[vi]; g.nseg = L.nseg;
    const ActView *av[2] = {a0, a1};
    double flops = 0;
    for (int s = 0; s < L.nseg; ++s) {
        if (!av[s] || av[s]->K != L.seg[s].K)
            return lbic_fail(LBIC_ERR_INVALID, "internal: layer %d segment %d K mismatch", id, s);
        g.K[s] = L.seg[s].K;
        g.A[s].hi = av[s]->buf->hi; g.A[s].lo = av[s]->buf->lo; g.A[s].ld = av[s]->buf->ld;
        g.A[s].tm_hi = &av[s]->tm_hi; g.A[s].tm_lo = &av[s]->tm_lo;
        g.W[s].hi = L.seg[s].hi; g.W[s].lo = L.seg[s].lo; g.W[s].ld = L.seg[s].K;
        g.W[s].tm_hi = &L.seg[s].tm_hi[vi]; g.W[s].tm_lo = &L.seg[s].tm_lo[vi];
        flops += 2.0 * R * (double)L.seg[s].K * L.cout;
    }
    ep.R = R; ep.cout = L.cout; ep.bias = L.bias; ep.acc_scale = L.acc_scale;
    ep.scale_tab = m->tables.d_scale_table;
    g.ep = ep;
    ProfRec rec;
    if (m->profiling) {
        cudaEventCreate(&rec.a); cudaEventCreate(&rec.b);
        rec.flops = flops;
        rec.layer = id;
        cudaEventRecord(rec.a, st);
    }
    const int rc = m->gemm_core == 1 ? gemm_simt_launch(g, st)
                                     : (ws ? gemm_ws_launch(g, st, vi >= LBIC_PAIR_VARIANT) : gemm_tc_launch(g, st));
    if (m->profiling) {
        cudaEventRecord(rec.b, st);
        m->prof.push_back(rec);
    }
    if (rc == 0 && m->check_sat && m->d_sat && !ep.out_pos &&
        (ep.mode == EPI_LRELU || ep.mode == EPI_PREGDN || ep.mode == EPI_GDN || ep.mode == EPI_IGDN || ep.mode == EPI_QUANT))
        return launch_sat_scan(ep.out_hi, R, L.cout, ep.ld_out, m->d_sat, st);
    return rc;
}

EpiParams epi(int mode, const StepDesc &sd) {
    EpiParams e;
    memset(&e, 0, sizeof(e));
    e.mode = mode;
    e.step = sd;
    return e;
}

EpiParams epi_hilo(int mode, const StepDesc &sd, const ActBuf &out) {
    EpiParams e = epi(mode, sd);
    e.out_hi = out.hi; e.out_lo = out.lo; e.ld_out = out.ld;
    return e;
}

// KS[1] == 3: hidden map g0 = lrelu(E0(zhat taps)) at the ring-extended positions `ext` (single-position or
// diagonal steps with h in [-1, Wb]), scattered into the position-indexed store (SURVEY.md A.3 / A.6).
int run_g0(lbic_model *m, const StepDesc &ext, int R_ext, cudaStream_t st) {
    Workspace &ws = m->ws;
    if (R_ext <= 0) return 0;
    if (R_ext > ws.R_ext_cap) return lbic_fail(LBIC_ERR_INVALID, "internal: extended step exceeds its workspace");
    LBIC_TRY(launch_gather(nullptr, ws.zhat_cl, m->Cin, ext, R_ext, nullptr, nullptr, 0, ws.Text.hi, ws.Text.lo,
                           ws.Text.ld, st));
    EpiParams e = epi_hilo(EPI_LRELU, ext, ws.G0);
    e.out_pos = 1;
    return run_gemm(m, L_E0, R_ext, &ws.vText, nullptr, e, st);
}

// entropy-parameter net: T (or the g0 store) -> ksi   (get_meanscale_fast, NET:389-398)
int run_ent(lbic_model *m, const StepDesc &sd, int R, cudaStream_t st) {
    Workspace &ws = m->ws;
    if (m->k1 == 3) {
        LBIC_TRY(launch_gather5(ws.G0.hi, ws.G0.lo, m->E1, sd, R, ws.H1x5.hi, ws.H1x5.lo, ws.H1x5.ld, st));
        LBIC_TRY(run_gemm(m, L_E1, R, &ws.vH1x5, nullptr, epi_hilo(EPI_LRELU, sd, ws.H2), st));
    } else {
        LBIC_TRY(run_gemm(m, L_E0, R, &ws.vT, nullptr, epi_hilo(EPI_LRELU, sd, ws.H1), st));
        LBIC_TRY(run_gemm(m, L_E1, R, &ws.vH1, nullptr, epi_hilo(EPI_LRELU, sd, ws.H2), st));
    }
    LBIC_TRY(run_gemm(m, L_E2, R, &ws.vH2, nullptr, epi_hilo(EPI_LRELU, sd, ws.H3), st));
    EpiParams e = epi(EPI_KSI, sd);
    e.out_f32 = ws.KSI; e.ld_f32 = ws.ldKSI;
    LBIC_TRY(run_gemm(m, L_E3, R, &ws.vH3, nullptr, e, st));
    return 0;
}

// GDN / IGDN stage i (widths N, C2, C3): S (squares) -> U
int run_gdn(lbic_model *m, int id, int i, bool inverse, const StepDesc &sd, int R, cudaStream_t st) {
    Workspace &ws = m->ws;
    EpiParams e = epi_hilo(inverse ? EPI_IGDN : EPI_GDN, sd, ws.U);
    e.aux = ws.A32; e.ld_aux = ws.ldA32;
    return run_gemm(m, id, R, &ws.vS[i], nullptr, e, st);
}

EpiParams epi_pregdn(lbic_model *m, const StepDesc &sd) {
    Workspace &ws = m->ws;
    EpiParams e = epi_hilo(EPI_PREGDN, sd, ws.S);
    e.out_f32 = ws.A32; e.ld_f32 = ws.ldA32;
    return e;
}

// encoder net + quantisation: X, T, ksi -> symbols, indexes, y_qnt   (forward_prtr_fast NET:379-382, NET:371-374)
int run_enc(lbic_model *m, const StepDesc &sd, int R, int32_t *sym, uint8_t *idx, cudaStream_t st) {
    Workspace &ws = m->ws;
    LBIC_TRY(run_gemm(m, L_F0, R, &ws.vX, &ws.vT, epi_pregdn(m, sd), st));
    LBIC_TRY(run_gdn(m, L_G0, 0, false, sd, R, st));
    LBIC_TRY(run_gemm(m, L_F1, R, &ws.vU[0], nullptr, epi_pregdn(m, sd), st));
    LBIC_TRY(run_gdn(m, L_G1, 1, false, sd, R, st));
    LBIC_TRY(run_gemm(m, L_F2, R, &ws.vU[1], nullptr, epi_pregdn(m, sd), st));
    LBIC_TRY(run_gdn(m, L_G2, 2, false, sd, R, st));
    EpiParams e = epi_hilo(EPI_QUANT, sd, ws.YQ);
    e.aux = ws.KSI; e.ld_aux = ws.ldKSI; e.M = m->M;
    e.sym = sym; e.idx = idx;
    LBIC_TRY(run_gemm(m, L_F3, R, &ws.vU[2], nullptr, e, st));
    return 0;
}

// decoder net: y_qnt, T -> zhat block, clamped   (inverse_prtr_fast NET:384-387, NET:357)
int run_dec(lbic_model *m, const StepDesc &sd, int R, cudaStream_t st) {
    Workspace &ws = m->ws;
    LBIC_TRY(run_gemm(m, L_D0, R, &ws.vYQ, &ws.vT, epi_pregdn(m, sd), st));
    LBIC_TRY(run_gdn(m, L_IG0, 0, true, sd, R, st));
    LBIC_TRY(run_gemm(m, L_D1, R, &ws.vU[0], nullptr, epi_pregdn(m, sd), st));
    LBIC_TRY(run_gdn(m, L_IG1, 1, true, sd, R, st));
    LBIC_TRY(run_gemm(m, L_D2, R, &ws.vU[1], nullptr, epi_pregdn(m, sd), st));
    LBIC_TRY(run_gdn(m, L_IG2, 2, true, sd, R, st));
    EpiParams e = epi(EPI_RECON, sd);
    e.zhat = m->recon_cl ? m->recon_cl : ws.zhat_cl;
    e.no_clamp = m->recon_no_clamp;
    LBIC_TRY(run_gemm(m, L_D3, R, &ws.vU[2], nullptr, e, st));
    return 0;
}

int floor_div2(int a) { return a >= 0 ? a / 2 : -((-a + 1) / 2); }

// ring-extended diagonal of step t (KS[1] == 3): positions (v, h = t - 2v) with v in [0, Hb-1], h in [-1, Wb]
bool wave_step_ext(int t, int n_img, int Hb, int Wb, StepDesc &sd) {
    int vmin = floor_div2(t - Wb + 1);   // ceil((t - Wb) / 2)
    if (vmin < 0) vmin = 0;
    int vmax = floor_div2(t + 1);
    if (vmax > Hb - 1) vmax = Hb - 1;
    if (vmax < vmin) return false;
    sd.n_img = n_img; sd.nv = vmax - vmin + 1; sd.vmin = vmin; sd.t = t; sd.Hb = Hb; sd.Wb = Wb;
    return true;
}

bool wave_step(int t, int n_img, int Hb, int Wb, StepDesc &sd) {
    if (t < 0) return false;
    int vmin = t - (Wb - 1) <= 0 ? 0 : (t - (Wb - 1) + 1) / 2;
    int vmax = t / 2 < Hb - 1 ? t / 2 : Hb - 1;
    if (vmax < vmin) return false;
    sd.n_img = n_img; sd.nv = vmax - vmin + 1; sd.vmin = vmin; sd.t = t; sd.Hb = Hb; sd.Wb = Wb;
    return true;
}

int check_ready(lbic_model *m, bool need_tables) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    if (!m->weights_loaded) return lbic_fail(LBIC_ERR_STATE, "weights not loaded: call lbic_load_weights first");
    if (need_tables && !m->tables.cdf) return lbic_fail(LBIC_ERR_STATE, "Uninitialized CDFs. Run update() first");
    if (!m->tables.d_scale_table) return lbic_fail(LBIC_ERR_STATE, "Uninitialized scale table. Run update() first");
    return 0;
}

// Worst case of one rANS64 stream of n_sym symbols: a table symbol costs at most 16 bits, an escaped one at most
// 16 (tail bin) + 4 (nibble count) + 32 (eight 4-bit nibbles of the 32-bit raw value) = 52 bits, plus the 64-bit final
// state and one word of renormalisation slack: 8 bytes per symbol + 64 can never overflow.  (CompressAI's flush() sizes
// its buffer as one 32-bit word per PUSHED entry, bypass nibbles included; this is the same bound per worst-case symbol.)
size_t lane_bound(size_t n_sym) { return 8 * n_sym + 64; }

// is_lane_container: 'LBML' | lanes | len[lanes] | payloads  (one lane per block row), else the raw reference stream
size_t stream_bound(const lbic_model *m, int Hb, int Wb, bool is_lane_container) {
    if (!is_lane_container) return lane_bound((size_t)Hb * Wb * m->M);
    return 8 + 4 * (size_t)Hb + (size_t)Hb * lane_bound((size_t)Wb * m->M);
}

// Host-side callbacks of the wavefront drivers: the *_host entry points use them to move the batch in and out in bands
// of block rows while the wavefront is running (block row v is first read by step 2v and final after step Wb-1+2v).
struct RowHooks {
    void *ctx = nullptr;
    int (*need_rows)(void *ctx, int v_hi, cudaStream_t st) = nullptr;    // x_cl block rows [0, v_hi] are read by what is enqueued next
    int (*rows_done)(void *ctx, int v_done, cudaStream_t st) = nullptr;  // zhat_cl block rows [0, v_done) are final after what has been enqueued
    // would the matching call enqueue anything?  (the latency path batches steps into one launch and only cuts the
    // launch where a hook has work to put between two steps)
    bool (*will_need)(void *ctx, int v_hi) = nullptr;
    bool (*will_done)(void *ctx, int v_done) = nullptr;
};

// The persistent wavefront kernel (gemm_wave.cu) takes over when every step of the call has at most wave_max_rows rows.
bool wave_applies(const lbic_model *m, int n_img, int Hb, int Wb, bool raster, bool decode) {
    if (!m->use_wave || m->gemm_core != 0 || m->force_bn || m->profiling || m->check_sat || m->selfinfo_cl ||
        m->recon_cl || !gemm_wave_supported())
        return false;
    const int max_nv = Hb < (Wb + 1) / 2 ? Hb : (Wb + 1) / 2;
    if (m->k1 == 3) {
        // five-tap topologies: wavefront calls whose EXTENDED steps (two ring positions more per image) fit one row block
        const int nv_ext = Hb < (Wb + 3) / 2 + 1 ? Hb : (Wb + 3) / 2 + 1;
        // (a one-column image has steps with ring positions but no block of the image: those stay on the per-layer path)
        if (raster || Wb < 2 || (long)n_img * nv_ext > 128) return false;
        if (decode && (m->tables.cdf16_total <= 0 || (long)n_img * nv_ext > m->wave_dec_max_rows)) return false;
        return true;
    }
    const long rows = raster ? n_img : (long)n_img * max_nv;
    int cap = m->wave_max_rows < gemm_wave_max_rows() ? m->wave_max_rows : gemm_wave_max_rows();
    if (decode) {
        if (m->tables.cdf16_total <= 0) return false;      // the entropy CTAs need the compact tables
        cap = cap < m->wave_dec_max_rows ? cap : m->wave_dec_max_rows;
    }
    return rows <= cap;
}

int run_wave(lbic_model *m, bool decode, bool raster, int s_begin, int s_end, int n_img, int Hb, int Wb, int lanes_L,
             int32_t *sym_out, cudaStream_t st) {
    Workspace &ws = m->ws;
    WaveLaunch w;
    memset(&w, 0, sizeof(w));
    w.d_layers = ws.d_chain; w.h_layers = ws.h_chain.data();
    w.decode = decode ? 1 : 0; w.raster = raster ? 1 : 0;
    w.s_begin = s_begin; w.s_end = s_end; w.n_img = n_img; w.Hb = Hb; w.Wb = Wb;
    for (int i = 0; i < L_COUNT; ++i) w.ids[i] = i;
    {
        // tile width: 32 columns.  The MMA chain of a tile takes the same time for any width up to ~176 columns (it is
        // bound by the latency of dependent accumulations), but the staged epilogue grows with the width (1.5 us per 32
        // columns) and sits on the layer-to-layer critical path: profiles/r2_wave_latency.md.  64 / 128 stay selectable.
        w.variant = m->wave_bn == 64 ? LBIC_LAT64_VARIANT : m->wave_bn == 128 ? LBIC_LAT128_VARIANT : LBIC_LAT_VARIANT;
    }
    w.x_cl = ws.x_cl; w.zhat_cl = ws.zhat_cl; w.Cin = m->Cin;
    w.X_hi = ws.X.hi; w.X_lo = ws.X.lo; w.ldX = ws.X.ld;
    w.T_hi = ws.T.hi; w.T_lo = ws.T.lo; w.ldT = ws.T.ld;
    w.scale_tab = m->tables.d_scale_table;
    if (m->k1 == 3) {
        w.k3 = 1; w.E1 = m->E1;
        w.Text_hi = ws.Text.hi; w.Text_lo = ws.Text.lo; w.ldText = ws.Text.ld;
        w.G0_hi = ws.G0.hi; w.G0_lo = ws.G0.lo;
        w.H5_hi = ws.H1x5.hi; w.H5_lo = ws.H1x5.lo; w.ldH5 = ws.H1x5.ld;
    }
    if (decode) {
        const Tables &T = m->tables;
        w.cdf = T.cdf; w.cdf_stride = T.stride; w.cdf_len = T.cdf_length; w.offs = T.offset;
        w.states = ws.dec_states; w.lane_ptr = ws.lane_ptr; w.lanes = lanes_L;
        w.ksi = ws.KSI; w.ld_ksi = ws.ldKSI; w.yq_hi = ws.YQ.hi; w.yq_lo = ws.YQ.lo; w.ld_yq = ws.YQ.ld;
        w.sym_out = sym_out; w.M = m->M;
        w.cdf16 = T.cdf16; w.cdf16_off = T.cdf16_off; w.cdf16_total = T.cdf16_total;
    }
    w.counters = ws.wave_counters; w.counters_cap = ws.wave_counters_cap;
    w.err_flag = m->err_flag;
    return gemm_wave_launch(w, st);
}


int ws_acquire(lbic_model *m, cudaStream_t st) {
    if (m->ws_used && st != m->ws_stream) LBIC_CUDA(cudaStreamWaitEvent(st, m->ws_event, 0));
    return 0;
}
int ws_release(lbic_model *m, cudaStream_t st) {
    LBIC_CUDA(cudaEventRecord(m->ws_event, st));
    m->ws_stream = st;
    m->ws_used = true;
    return 0;
}

int ensure_aux(lbic_model *m, int which, size_t bytes, float **out) {
    if (m->aux_bytes[which] < bytes) {
        if (m->aux[which]) { LBIC_CUDA(cudaDeviceSynchronize()); cudaFree(m->aux[which]); m->aux[which] = nullptr; m->aux_bytes[which] = 0; }
        cudaError_t e = cudaMalloc(&m->aux[which], bytes);
        if (e != cudaSuccess) return lbic_fail(LBIC_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        m->aux_bytes[which] = bytes;
    }
    *out = m->aux[which];
    return 0;
}

int encode_impl(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out, int32_t *sym_out,
                uint8_t *idx_out, uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes,
                cudaStream_t st, const RowHooks *hk);
int decode_impl(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap, int n_img, int Hb,
                int Wb, float *zhat_out, int32_t *sym_out, int lanes, cudaStream_t st, const RowHooks *hk);

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int lbic_create(const lbic_config *cfg, int device, lbic_model **out) {
    if (!cfg || !out) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return lbic_fail(LBIC_ERR_NO_DEVICE, "no CUDA device: liblbic_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return lbic_fail(LBIC_ERR_INVALID, "device %d out of range", device);
    cudaDeviceProp prop;
    LBIC_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return lbic_fail(LBIC_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                         prop.major, prop.minor);
    if (cfg->ks[0] != 3 || (cfg->ks[1] != 1 && cfg->ks[1] != 3) || cfg->ks[2] != 1 || cfg->ks[3] != 1)
        return lbic_fail(LBIC_ERR_INVALID, "unsupported KS [%d,%d,%d,%d]", cfg->ks[0], cfg->ks[1], cfg->ks[2], cfg->ks[3]);
    if (cfg->block_size < 1 || cfg->n % 8 || cfg->n < 16 || cfg->m % 16 || cfg->m < 16 || cfg->m > 256 ||
        (3 * cfg->block_size * cfg->block_size) % 16)
        return lbic_fail(LBIC_ERR_INVALID, "unsupported sizes B=%d N=%d M=%d (need 3B^2, M multiples of 16)",
                         cfg->block_size, cfg->n, cfg->m);
    LBIC_CUDA(cudaSetDevice(device));
    lbic_model *m = new lbic_model();
    // tuning hooks for benchmarking without code changes (the same switches as lbic_set_option)
    if (const char *e = getenv("LBIC_FLOW")) m->use_flow = atoi(e) < 0 ? 0 : (atoi(e) > 2 ? 2 : atoi(e));
    if (const char *e = getenv("LBIC_FLOW_MIN_ROWS")) m->flow_min_rows = atoi(e) < 1 ? 1 : atoi(e);
    if (const char *e = getenv("LBIC_FLOW_MAX_ROWS")) m->flow_max_rows = atoi(e) < 1 ? 1 : atoi(e);
    if (const char *e = getenv("LBIC_FLOW_SMALL")) m->flow_small = atoi(e) ? 1 : 0;
    if (const char *e = getenv("LBIC_FLOW_PAIR_MIN_ROWS")) m->flow_pair_min_rows = atoi(e) < 1 ? 1 : atoi(e);
    if (const char *e = getenv("LBIC_FLOW_QUAD")) m->flow_quad = atoi(e) ? 1 : 0;
    if (const char *e = getenv("LBIC_WAVE")) m->use_wave = atoi(e) ? 1 : 0;
    if (const char *e = getenv("LBIC_WAVE_MAX_ROWS")) m->wave_max_rows = atoi(e) < 1 ? 1 : atoi(e);
    if (const char *e = getenv("LBIC_WAVE_DEC_MAX_ROWS")) m->wave_dec_max_rows = atoi(e) < 1 ? 1 : atoi(e);
    if (const char *e = getenv("LBIC_WAVE_BN")) m->wave_bn = atoi(e);
    m->cfg = *cfg;
    m->device = device;
    m->Cin = 3 * cfg->block_size * cfg->block_size;
    m->N = cfg->n; m->C2 = cfg->n / 8 * 7; m->C3 = cfg->n / 8 * 6; m->M = cfg->m;
    m->E1 = cfg->n / 8 * 12; m->E2 = cfg->n / 8 * 10; m->E3 = cfg->n / 8 * 8; m->EO = 2 * cfg->m;
    m->k1 = cfg->ks[1];
    const int dims[] = {m->N, m->C2, m->C3, m->E1, m->E2, m->E3};
    for (int d : dims)
        if (d % 16) {
            delete m;
            return lbic_fail(LBIC_ERR_INVALID, "channel width %d is not a multiple of 16", d);
        }
    if (cudaMalloc(&m->err_flag, sizeof(int)) != cudaSuccess) {
        delete m;
        return lbic_fail(LBIC_ERR_NOMEM, "cudaMalloc failed");
    }
    cudaMemset(m->err_flag, 0, sizeof(int));
    if (cudaMalloc(&m->d_sat, sizeof(unsigned long long)) == cudaSuccess) cudaMemset(m->d_sat, 0, sizeof(unsigned long long));
    if (cudaEventCreateWithFlags(&m->ws_event, cudaEventDisableTiming) != cudaSuccess) {
        cudaFree(m->err_flag);
        delete m;
        return lbic_fail(LBIC_ERR_CUDA, "cudaEventCreate failed");
    }
    const char *core = getenv("LBIC_GEMM_CORE");
    if (core && !strcmp(core, "simt")) m->gemm_core = 1;
    *out = m;
    return 0;
}

extern "C" void lbic_destroy(lbic_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    free_all(m->ws.allocs);
    free_all(m->weight_allocs);
    free_all(m->pp_allocs);
    free_all(m->pp_ws_allocs);
    tables_free(m->tables);
    if (m->tables.d_scale_table) cudaFree(m->tables.d_scale_table);
    if (m->err_flag) cudaFree(m->err_flag);
    if (m->d_sat) cudaFree(m->d_sat);
    if (m->ws_event) cudaEventDestroy(m->ws_event);
    if (m->io_dev) cudaFree(m->io_dev);
    for (auto &a : m->aux) if (a) cudaFree(a);
    for (auto &h : m->hs) if (h) cudaStreamDestroy(h);
    for (auto &ev : m->hev) if (ev) cudaEventDestroy(ev);
    for (auto &r : m->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    delete m;
}

extern "C" int lbic_set_option(lbic_model *m, int option, int value) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    switch (option) {
    case LBIC_OPT_GEMM_CORE:
        if (value != 0 && value != 1) return lbic_fail(LBIC_ERR_INVALID, "gemm core must be 0 or 1");
        m->gemm_core = value;
        return 0;
    case LBIC_OPT_PDL:
        gemm_set_pdl(value);
        return 0;
    case LBIC_OPT_WS:
        m->use_ws = value < 0 ? 0 : (value > 2 ? 2 : value);   // 2 = always (testing)
        return 0;
    case LBIC_OPT_DEC_THREAD_ROWS:
        rans_set_dec_thread_min_rows(value);
        return 0;
    case LBIC_OPT_ENC_THREAD_STREAMS:
        rans_set_enc_thread_min_streams(value);
        return 0;
    case LBIC_OPT_DEC_SMEM_WARP:
        rans_set_dec_smem_warp(value);
        return 0;
    case LBIC_OPT_ENC_BLOCK_STREAMS:
        rans_set_enc_block_max_streams(value);
        return 0;
    case LBIC_OPT_FLOW:
        m->use_flow = value < 0 ? 0 : (value > 2 ? 2 : value);
        return 0;
    case LBIC_OPT_FLOW_MIN_ROWS:
        m->flow_min_rows = value < 1 ? 1 : value;
        return 0;
    case LBIC_OPT_WAVE:
        m->use_wave = value ? 1 : 0;
        return 0;
    case LBIC_OPT_WAVE_MAX_ROWS:
        m->wave_max_rows = value < 1 ? 1 : (value > gemm_wave_max_rows() ? gemm_wave_max_rows() : value);
        return 0;
    case LBIC_OPT_WAVE_DEC_MAX_ROWS:
        m->wave_dec_max_rows = value < 1 ? 1 : value;
        return 0;
    case LBIC_OPT_WAVE_BN:
        if (value != 0 && value != 32 && value != 64 && value != 128) return lbic_fail(LBIC_ERR_INVALID, "wave tile width must be 0, 32, 64 or 128");
        m->wave_bn = value;
        return 0;
    case LBIC_OPT_HOST_BANDS:
        m->host_bands = value < 1 ? 1 : (value > LBIC_MAX_BANDS ? LBIC_MAX_BANDS : value);
        return 0;
    case LBIC_OPT_FLOW_SMALL:
        m->flow_small = value ? 1 : 0;
        return 0;
    case LBIC_OPT_FLOW_QUAD:
        m->flow_quad = value ? 1 : 0;
        return 0;
    case LBIC_OPT_CHECK_SATURATION:
        m->check_sat = value ? 1 : 0;
        return 0;
    case LBIC_OPT_FLOW_PAIR_MIN_ROWS:
        m->flow_pair_min_rows = value < 1 ? 1 : value;
        return 0;
    case LBIC_OPT_TMA_STORE:
        gemm_set_tma_store(value);
        return 0;
    case LBIC_OPT_PAIR:
        m->use_pair = value < 0 ? 0 : (value > 3 ? 3 : value);   // 2 = narrow (<= 192) tiles only, 3 = wide (<= 256) in the microbench
        return 0;
    case LBIC_OPT_FORCE_BN:
        if (value != 0 && (value % 16 || value < 16 || value > 256)) return lbic_fail(LBIC_ERR_INVALID, "bad tile width");
        m->force_bn = value;
        return 0;
    default:
        return lbic_fail(LBIC_ERR_INVALID, "unknown option %d", option);
    }
}

extern "C" int lbic_load_weights(lbic_model *m, const lbic_tensor_desc *tensors, int n_tensors, void *stream) {
    if (!m || !tensors) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(gemm_tc_init());
    SdView sd;
    for (int i = 0; i < n_tensors; ++i)
        if (tensors[i].name && tensors[i].data) sd.by_name[tensors[i].name] = &tensors[i];
    LBIC_CUDA(cudaDeviceSynchronize());
    free_all(m->weight_allocs);
    m->weights_loaded = false;
    std::vector<void *> tmp;
    int rc = 0;
    do {
        const int Cin = m->Cin, N = m->N, C2 = m->C2, C3 = m->C3, M = m->M;
#define P(call) if ((rc = (call)) != 0) break
        P(pack_linear(m, sd, L_E0, "get_meanscale.0", m->E1, Cin, 3, TAPS_A, 4, tmp, st));
        if (m->k1 == 3) {
            P(pack_linear(m, sd, L_E1, "get_meanscale.2", m->E2, m->E1, 3, TAPS_B, 5, tmp, st));
        } else {
            P(pack_linear(m, sd, L_E1, "get_meanscale.2", m->E2, m->E1, 1, TAPS_1, 1, tmp, st));
        }
        P(pack_linear(m, sd, L_E2, "get_meanscale.4", m->E3, m->E2, 1, TAPS_1, 1, tmp, st));
        P(pack_linear(m, sd, L_E3, "get_meanscale.6", m->EO, m->E3, 1, TAPS_1, 1, tmp, st));
        P(pack_dual(m, sd, L_F0, "prtr_forward1", Cin, "prtr_forward2", N, tmp, st));
        P(pack_gdn(m, sd, L_G0, "prtr_forward3.0", N, tmp, st));
        P(pack_linear(m, sd, L_F1, "prtr_forward3.1", C2, N, 1, TAPS_1, 1, tmp, st));
        P(pack_gdn(m, sd, L_G1, "prtr_forward3.2", C2, tmp, st));
        P(pack_linear(m, sd, L_F2, "prtr_forward3.3", C3, C2, 1, TAPS_1, 1, tmp, st));
        P(pack_gdn(m, sd, L_G2, "prtr_forward3.4", C3, tmp, st));
        P(pack_linear(m, sd, L_F3, "prtr_forward3.5", M, C3, 1, TAPS_1, 1, tmp, st));
        P(pack_dual(m, sd, L_D0, "prtr_inverse1", M, "prtr_inverse2", N, tmp, st));
        P(pack_gdn(m, sd, L_IG0, "prtr_inverse3.0", N, tmp, st));
        P(pack_linear(m, sd, L_D1, "prtr_inverse3.1", C2, N, 1, TAPS_1, 1, tmp, st));
        P(pack_gdn(m, sd, L_IG1, "prtr_inverse3.2", C2, tmp, st));
        P(pack_linear(m, sd, L_D2, "prtr_inverse3.3", C3, C2, 1, TAPS_1, 1, tmp, st));
        P(pack_gdn(m, sd, L_IG2, "prtr_inverse3.4", C3, tmp, st));
        P(pack_linear(m, sd, L_D3, "prtr_inverse3.5", Cin, C3, 1, TAPS_1, 1, tmp, st));
#undef P
    } while (0);
    cudaError_t e = cudaStreamSynchronize(st);
    free_all(tmp);
    if (rc) return rc;
    if (e != cudaSuccess) return lbic_fail(LBIC_ERR_CUDA, "weight packing failed: %s", cudaGetErrorString(e));
    m->weights_loaded = true;
    return 0;
}

extern "C" int lbic_build_tables(lbic_model *m, const float *scale_table, int n_levels, double tail_mass,
                                 void *stream) {
    if (!m || !scale_table) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    if (n_levels != 64) return lbic_fail(LBIC_ERR_INVALID, "the codec path uses a 64-level scale table (NET:13-18)");
    Active act(m);
    return tables_build(m->tables, scale_table, n_levels, tail_mass, (cudaStream_t)stream);
}

extern "C" int lbic_set_tables(lbic_model *m, const float *scale_table, int n_levels, const int32_t *cdf,
                               int cdf_stride, const int32_t *cdf_length, const int32_t *offset) {
    if (!m || !scale_table || !cdf || !cdf_length || !offset) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    if (n_levels != 64 || cdf_stride < 3) return lbic_fail(LBIC_ERR_INVALID, "bad table shape");
    Active act(m);
    Tables &T = m->tables;
    LBIC_CUDA(cudaDeviceSynchronize());
    tables_free(T);
    LBIC_CUDA(cudaMalloc(&T.cdf, sizeof(int32_t) * (size_t)n_levels * cdf_stride));
    LBIC_CUDA(cudaMalloc(&T.cdf_length, sizeof(int32_t) * 64));
    LBIC_CUDA(cudaMalloc(&T.offset, sizeof(int32_t) * 64));
    LBIC_CUDA(cudaMemcpy(T.cdf, cdf, sizeof(int32_t) * (size_t)n_levels * cdf_stride, cudaMemcpyHostToDevice));
    LBIC_CUDA(cudaMemcpy(T.cdf_length, cdf_length, sizeof(int32_t) * n_levels, cudaMemcpyHostToDevice));
    LBIC_CUDA(cudaMemcpy(T.offset, offset, sizeof(int32_t) * n_levels, cudaMemcpyHostToDevice));
    T.n_levels = n_levels; T.stride = cdf_stride;
    for (int i = 0; i < 64; ++i) T.scale_table[i] = scale_table[i];
    if (!T.d_scale_table) LBIC_CUDA(cudaMalloc(&T.d_scale_table, sizeof(float) * 64));
    LBIC_CUDA(cudaMemcpy(T.d_scale_table, T.scale_table, sizeof(float) * 64, cudaMemcpyHostToDevice));
    return tables_compact(T, 0);
}

extern "C" int lbic_get_tables(lbic_model *m, int *n_levels, int *cdf_stride, int32_t *cdf, int32_t *cdf_length,
                               int32_t *offset) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    Tables &T = m->tables;
    if (!T.cdf) return lbic_fail(LBIC_ERR_STATE, "Uninitialized CDFs. Run update() first");
    Active act(m);
    if (n_levels) *n_levels = T.n_levels;
    if (cdf_stride) *cdf_stride = T.stride;
    LBIC_CUDA(cudaDeviceSynchronize());
    if (cdf) LBIC_CUDA(cudaMemcpy(cdf, T.cdf, sizeof(int32_t) * (size_t)T.n_levels * T.stride, cudaMemcpyDeviceToHost));
    if (cdf_length) LBIC_CUDA(cudaMemcpy(cdf_length, T.cdf_length, sizeof(int32_t) * T.n_levels, cudaMemcpyDeviceToHost));
    if (offset) LBIC_CUDA(cudaMemcpy(offset, T.offset, sizeof(int32_t) * T.n_levels, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" size_t lbic_stream_bound(const lbic_model *m, int Hb, int Wb, int lanes) {
    if (!m || Hb < 1 || Wb < 1) return 0;
    return stream_bound(m, Hb, Wb, lanes != 1);
}

extern "C" int lbic_encode(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out,
                           int32_t *sym_out, uint8_t *idx_out, uint8_t *stream_out, size_t stream_cap,
                           uint32_t *stream_len, int lanes, void *stream) {
    if (!x) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    return encode_impl(m, x, n_img, Hb, Wb, zhat_out, sym_out, idx_out, stream_out, stream_cap, stream_len, lanes,
                       (cudaStream_t)stream, nullptr);
}

namespace {
// One encode-side wavefront step: entropy net, encoder net + quantisation, decoder net for the R rows of `sd`
// (NET:363-377 for every block of the diagonal at once).  The gather of the step's operands has been enqueued.
int encode_step(lbic_model *m, const StepDesc &sd, int R, bool want_syms, cudaStream_t st) {
    Workspace &ws = m->ws;
    if (flow_applies(m, R) && !m->recon_cl) {
        // the whole step as one dataflow launch; if the launch itself is refused (no co-residency: a shared or
        // partitioned GPU) the per-layer path below takes over for good
        if (m->k1 == 3) LBIC_TRY(launch_gather5(ws.G0.hi, ws.G0.lo, m->E1, sd, R, ws.H1x5.hi, ws.H1x5.lo, ws.H1x5.ld, st));
        const int rc = run_flow(m, m->k1 == 3 ? L_E1 : L_E0, L_COUNT, sd, R, st);
        if (rc != LBIC_FLOW_REFUSED) return rc;
        m->use_flow = 0;
    }
    LBIC_TRY(run_ent(m, sd, R, st));
    LBIC_TRY(run_enc(m, sd, R, want_syms ? ws.sym : nullptr, want_syms ? ws.idx : nullptr, st));
    return run_dec(m, sd, R, st);
}

int encode_impl(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out, int32_t *sym_out,
                uint8_t *idx_out, uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes,
                cudaStream_t st, const RowHooks *hk) {
    LBIC_TRY(check_ready(m, stream_out != nullptr));
    if ((!x && !(hk && hk->need_rows)) || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    if (lanes != 0 && lanes != 1) return lbic_fail(LBIC_ERR_INVALID, "lanes must be 1 (reference) or 0 (per block row)");
    if (stream_out && (!stream_len || stream_cap % 4)) return lbic_fail(LBIC_ERR_INVALID, "stream_cap must be a multiple of 4");
    Active act(m);
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    Workspace &ws = m->ws;
    const int HW = Hb * Wb;
    const size_t nblk = (size_t)n_img * HW;
    LBIC_TRY(ws_acquire(m, st));
    LBIC_CUDA(cudaMemsetAsync(m->err_flag, 0, sizeof(int), st));
    if (x) LBIC_TRY(launch_nchw_to_cl(x, ws.x_cl, n_img, m->Cin, HW, st));
    LBIC_CUDA(cudaMemsetAsync(ws.zhat_cl, 0, sizeof(float) * nblk * m->Cin, st));   // NET:336
    const bool want_syms = sym_out || idx_out || stream_out || m->selfinfo_cl;
    const int T_steps = Wb + 2 * (Hb - 1);
    if (m->k1 == 3) LBIC_TRY(launch_fill_g0_top(m->L[L_E0].bias, m->E1, n_img, Hb, Wb, ws.G0.hi, ws.G0.lo, st));
    // one step through the per-layer / dataflow launches
    auto launch_step = [&](int t) -> int {
        StepDesc sd, ext;
        if (m->k1 == 3 && wave_step_ext(t, n_img, Hb, Wb, ext)) LBIC_TRY(run_g0(m, ext, n_img * ext.nv, st));
        if (!wave_step(t, n_img, Hb, Wb, sd)) return 0;
        const int R = n_img * sd.nv;
        LBIC_TRY(launch_gather(ws.x_cl, ws.zhat_cl, m->Cin, sd, R, ws.X.hi, ws.X.lo, ws.X.ld, ws.T.hi, ws.T.lo, ws.T.ld, st));
        LBIC_TRY(encode_step(m, sd, R, want_syms, st));
        if (m->selfinfo_cl)
            LBIC_TRY(launch_selfinfo_step(sd, R, m->M, ws.KSI, ws.ldKSI, ws.sym, m->selfinfo_cl, st));
        return 0;
    };
    // Small steps (single images, small batches): consecutive steps are collected into ONE launch of the persistent
    // wavefront kernel, cut only where a host hook has copies or conversions to put between two steps.
    bool wave = wave_applies(m, n_img, Hb, Wb, false, false);
    int pend = -1;                                   // steps [pend, t) wait to be launched
    auto flush = [&](int t_end) -> int {
        if (pend < 0) return 0;
        const int b = pend;
        pend = -1;
        const int rc = run_wave(m, false, false, b, t_end, n_img, Hb, Wb, 0, nullptr, st);
        if (rc != LBIC_FLOW_REFUSED) return rc;
        m->use_wave = 0;                             // no co-residency on this device: per-layer launches from now on
        wave = false;
        for (int t = b; t < t_end; ++t) LBIC_TRY(launch_step(t));
        return 0;
    };
    for (int t = (m->k1 == 3 ? -1 : 0); t < T_steps; ++t) {
        StepDesc sd;
        const bool has = wave_step(t, n_img, Hb, Wb, sd);
        if (has && hk && hk->need_rows) {
            const int v_hi = sd.vmin + sd.nv - 1;
            if (!wave || !hk->will_need || hk->will_need(hk->ctx, v_hi)) {
                LBIC_TRY(flush(t));
                LBIC_TRY(hk->need_rows(hk->ctx, v_hi, st));
            }
        }
        if (wave) {
            if (!has) LBIC_TRY(launch_step(t));      // KS[1] = 3: step -1 has ring positions only (one small GEMM, per-layer path)
            else if (pend < 0) pend = t;
        } else {
            LBIC_TRY(launch_step(t));
        }
        if (has && hk && hk->rows_done && t >= Wb - 1) {
            int done = (t - (Wb - 1)) / 2 + 1;
            done = done < Hb ? done : Hb;
            if (!wave || !hk->will_done || hk->will_done(hk->ctx, done)) {
                LBIC_TRY(flush(t + 1));
                LBIC_TRY(hk->rows_done(hk->ctx, done, st));
            }
        }
    }
    LBIC_TRY(flush(T_steps));
    if (zhat_out) LBIC_TRY(launch_cl_to_nchw(ws.zhat_cl, zhat_out, n_img, m->Cin, HW, st));
    if (sym_out) LBIC_CUDA(cudaMemcpyAsync(sym_out, ws.sym, sizeof(int32_t) * nblk * m->M, cudaMemcpyDeviceToDevice, st));
    if (idx_out) LBIC_CUDA(cudaMemcpyAsync(idx_out, ws.idx, nblk * m->M, cudaMemcpyDeviceToDevice, st));
    if (stream_out) {
        const int L = lanes == 1 ? 1 : Hb;
        const int n_streams = n_img * L;
        const int64_t n_sym = (int64_t)HW * m->M / L;
        // scratch words per stream: the reference container is coded straight into the caller's slot size; a lane gets
        // its worst case (lane_bound), so only the caller's stream_cap can ever be the limit
        const size_t per = (lanes == 1 ? stream_cap : lane_bound((size_t)n_sym)) / 4;
        LBIC_TRY(ensure_rans_scratch(m, (size_t)n_streams * per + 2 * (size_t)n_streams));
        LBIC_TRY(launch_rans_encode(m->tables, ws.sym, ws.idx, n_streams, n_sym, n_sym, ws.rans_scratch, per,
                                    lanes == 1 ? stream_out : nullptr, stream_cap, stream_len, m->err_flag, st));
        if (lanes != 1)
            LBIC_TRY(launch_lane_pack(ws.rans_scratch, per, n_img, L, stream_out, stream_cap, stream_len, m->err_flag, st));
    }
    return ws_release(m, st);
}
}  // namespace

extern "C" int lbic_validate(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out,
                             float *selfinfo_out, void *stream) {
    LBIC_TRY(check_ready(m, false));
    if (!x || !selfinfo_out || n_img < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    float *cl = nullptr;
    LBIC_TRY(ensure_aux(m, 0, sizeof(float) * (size_t)n_img * Hb * Wb * m->M, &cl));
    m->selfinfo_cl = cl;
    int rc = lbic_encode(m, x, n_img, Hb, Wb, zhat_out, nullptr, nullptr, nullptr, 0, nullptr, 1, stream);
    m->selfinfo_cl = nullptr;
    Active act2(m);
    if (rc == 0) rc = launch_cl_to_nchw(cl, selfinfo_out, n_img, m->M, Hb * Wb, st);   // -> (n, M, Hb, Wb) as AGENT:509
    if (rc == 0) rc = ws_release(m, st);
    return rc;
}

// Open-loop forward = the reference's model.forward(zhat, x) in eval mode (NET:90-106): every block of the batch is
// independent given the context zhat, so the whole batch is processed as raster chunks of up to R_cap rows through the
// same gather / GEMM / epilogue kernels (no wavefront).  KS[1] = 3: the second entropy layer is zero padded in this
// whole-image form, so the hidden-map ring is zero here (the codec path computes it, SURVEY.md A.6); the hidden map
// of ALL blocks is produced first, then the rest of the nets.
extern "C" int lbic_forward(lbic_model *m, const float *zhat_in, const float *x, int n_img, int Hb, int Wb,
                            float *xhat_out, float *selfinfo_out, int32_t *sym_out, int clamp, void *stream) {
    LBIC_TRY(check_ready(m, false));
    if (!zhat_in || !x || !xhat_out || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    Workspace &ws = m->ws;
    const int HW = Hb * Wb;
    const long nblk = (long)n_img * HW;
    float *xhat_cl = nullptr, *info_cl = nullptr;
    int rc = 0;
    do {
#define P(call) if ((rc = (call)) != 0) break
        P(ws_acquire(m, st));
        P(ensure_aux(m, 1, sizeof(float) * (size_t)nblk * m->Cin, &xhat_cl));
        if (selfinfo_out) P(ensure_aux(m, 0, sizeof(float) * (size_t)nblk * m->M, &info_cl));
        P(launch_nchw_to_cl(x, ws.x_cl, n_img, m->Cin, HW, st));
        P(launch_nchw_to_cl(zhat_in, ws.zhat_cl, n_img, m->Cin, HW, st));
        const int chunk = ws.R_cap;
        if (m->k1 == 3) {
            const size_t npos = (size_t)n_img * (Hb + 1) * (Wb + 2);
            if (cudaMemsetAsync(ws.G0.hi, 0, sizeof(h16) * npos * m->E1, st) != cudaSuccess ||
                cudaMemsetAsync(ws.G0.lo, 0, sizeof(h16) * npos * m->E1, st) != cudaSuccess) {
                rc = lbic_fail(LBIC_ERR_CUDA, "memset failed");
                break;
            }
            for (long r0 = 0; r0 < nblk && rc == 0; r0 += chunk) {
                const int R = (int)(nblk - r0 < chunk ? nblk - r0 : chunk);
                const StepDesc sd{n_img, 0, 0, (int)r0, Hb, Wb};
                P(launch_gather(nullptr, ws.zhat_cl, m->Cin, sd, R, nullptr, nullptr, 0, ws.T.hi, ws.T.lo, ws.T.ld, st));
                EpiParams e = epi_hilo(EPI_LRELU, sd, ws.G0);
                e.out_pos = 1;
                P(run_gemm(m, L_E0, R, &ws.vT, nullptr, e, st));
            }
            if (rc) break;
        }
        m->recon_cl = xhat_cl;
        m->recon_no_clamp = clamp ? 0 : 1;
        for (long r0 = 0; r0 < nblk && rc == 0; r0 += chunk) {
            const int R = (int)(nblk - r0 < chunk ? nblk - r0 : chunk);
            const StepDesc sd{n_img, 0, 0, (int)r0, Hb, Wb};
            P(launch_gather(ws.x_cl, ws.zhat_cl, m->Cin, sd, R, ws.X.hi, ws.X.lo, ws.X.ld, ws.T.hi, ws.T.lo, ws.T.ld, st));
            P(run_ent(m, sd, R, st));
            P(run_enc(m, sd, R, ws.sym, ws.idx, st));
            P(run_dec(m, sd, R, st));
            if (info_cl) P(launch_selfinfo_step(sd, R, m->M, ws.KSI, ws.ldKSI, ws.sym, info_cl, st));
        }
        m->recon_cl = nullptr;
        m->recon_no_clamp = 0;
        if (rc) break;
        P(launch_cl_to_nchw(xhat_cl, xhat_out, n_img, m->Cin, HW, st));
        if (info_cl) P(launch_cl_to_nchw(info_cl, selfinfo_out, n_img, m->M, HW, st));
        if (sym_out && cudaMemcpyAsync(sym_out, ws.sym, sizeof(int32_t) * (size_t)nblk * m->M, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            rc = lbic_fail(LBIC_ERR_CUDA, "copy failed");
        if (rc == 0) rc = ws_release(m, st);
#undef P
    } while (0);
    m->recon_cl = nullptr;
    m->recon_no_clamp = 0;
    return rc;
}

extern "C" int lbic_decode(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                           int n_img, int Hb, int Wb, float *zhat_out, int32_t *sym_out, int lanes, void *stream) {
    return decode_impl(m, streams, stream_len, stream_cap, n_img, Hb, Wb, zhat_out, sym_out, lanes, (cudaStream_t)stream,
                       nullptr);
}

// Synchronises `stream` and reports what the kernels enqueued on it flagged since the last encode / decode started:
// a stream buffer that was too small (LBIC_ERR_OVERFLOW) or a malformed lane container (LBIC_ERR_INVALID).
extern "C" int lbic_check_errors(lbic_model *m, void *stream) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    Active act(m);
    LBIC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    int flag = 0;
    LBIC_CUDA(cudaMemcpy(&flag, m->err_flag, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        cudaMemset(m->err_flag, 0, sizeof(int));
        return lbic_fail(flag == 1 ? LBIC_ERR_OVERFLOW : LBIC_ERR_INVALID,
                         flag == 1 ? "bitstream buffer too small (stream_cap)" : "malformed lane container");
    }
    return 0;
}

namespace {
int decode_impl(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap, int n_img, int Hb,
                int Wb, float *zhat_out, int32_t *sym_out, int lanes, cudaStream_t st, const RowHooks *hk) {
    LBIC_TRY(check_ready(m, true));
    if (!streams || !stream_len || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    if (lanes != 0 && lanes != 1) return lbic_fail(LBIC_ERR_INVALID, "lanes must be 1 (reference) or 0 (per block row)");
    if (stream_cap % 4) return lbic_fail(LBIC_ERR_INVALID, "stream_cap must be a multiple of 4");
    Active act(m);
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    Workspace &ws = m->ws;
    const int HW = Hb * Wb;
    const size_t nblk = (size_t)n_img * HW;
    const int L = lanes == 1 ? 1 : Hb;
    LBIC_TRY(ws_acquire(m, st));
    LBIC_CUDA(cudaMemsetAsync(m->err_flag, 0, sizeof(int), st));
    LBIC_CUDA(cudaMemsetAsync(ws.zhat_cl, 0, sizeof(float) * nblk * m->Cin, st));   // NET:417
    LBIC_TRY(launch_rans_dec_init(streams, stream_len, stream_cap, n_img, L, lanes != 1, ws.dec_states, ws.lane_ptr,
                                  m->err_flag, st));
    auto one_step = [&](const StepDesc &sd, int R) -> int {
        LBIC_TRY(launch_gather(nullptr, ws.zhat_cl, m->Cin, sd, R, nullptr, nullptr, 0, ws.T.hi, ws.T.lo, ws.T.ld, st));
        bool flow = flow_applies(m, R) != 0;
        bool ent_done = false;
        if (flow) {
            if (m->k1 == 3) LBIC_TRY(launch_gather5(ws.G0.hi, ws.G0.lo, m->E1, sd, R, ws.H1x5.hi, ws.H1x5.lo, ws.H1x5.ld, st));
            const int rc = run_flow(m, m->k1 == 3 ? L_E1 : L_E0, L_F0, sd, R, st);
            if (rc == LBIC_FLOW_REFUSED) { m->use_flow = 0; flow = false; }
            else if (rc) return rc;
            else ent_done = true;
        }
        if (!ent_done) LBIC_TRY(run_ent(m, sd, R, st));
        LBIC_TRY(launch_rans_dec_step(m->tables, ws.dec_states, ws.lane_ptr, L, sd, R, m->M, ws.KSI, ws.ldKSI, ws.YQ.hi,
                                      ws.YQ.lo, ws.YQ.ld, sym_out ? ws.sym : nullptr, st));
        if (flow) {
            const int rc = run_flow(m, L_D0, L_COUNT, sd, R, st);
            if (rc != LBIC_FLOW_REFUSED) return rc;
            m->use_flow = 0;
        }
        return run_dec(m, sd, R, st);
    };
    if (m->k1 == 3) LBIC_TRY(launch_fill_g0_top(m->L[L_E0].bias, m->E1, n_img, Hb, Wb, ws.G0.hi, ws.G0.lo, st));
    const bool raster = (L == 1 && lanes == 1);      // reference container: the rANS state threads through the blocks in
                                                     // raster order (NET:420-450), one block of every image per step
    // raster step s = v * Wb + h; wavefront step s = t
    auto launch_step = [&](int s) -> int {
        if (raster) {
            const int v = s / Wb, h = s - v * Wb;
            if (m->k1 == 3) {
                // hidden-map positions that become computable now: the ring columns of the row start, then (v,h)
                if (h == 0) {
                    if (v >= 1) { StepDesc e{n_img, 1, v - 1, Wb + 2 * (v - 1), Hb, Wb}; LBIC_TRY(run_g0(m, e, n_img, st)); }
                    StepDesc e{n_img, 1, v, -1 + 2 * v, Hb, Wb};
                    LBIC_TRY(run_g0(m, e, n_img, st));
                }
                StepDesc e{n_img, 1, v, h + 2 * v, Hb, Wb};
                LBIC_TRY(run_g0(m, e, n_img, st));
            }
            StepDesc sd{n_img, 1, v, h + 2 * v, Hb, Wb};
            return one_step(sd, n_img);
        }
        StepDesc sd, ext;
        if (m->k1 == 3 && wave_step_ext(s, n_img, Hb, Wb, ext)) LBIC_TRY(run_g0(m, ext, n_img * ext.nv, st));
        if (!wave_step(s, n_img, Hb, Wb, sd)) return 0;
        return one_step(sd, n_img * sd.nv);
    };
    bool wave = wave_applies(m, n_img, Hb, Wb, raster, true);
    int pend = -1;
    auto flush = [&](int s_end) -> int {
        if (pend < 0) return 0;
        const int b = pend;
        pend = -1;
        const int rc = run_wave(m, true, raster, b, s_end, n_img, Hb, Wb, L, sym_out ? ws.sym : nullptr, st);
        if (rc != LBIC_FLOW_REFUSED) return rc;
        m->use_wave = 0;
        wave = false;
        for (int s = b; s < s_end; ++s) LBIC_TRY(launch_step(s));
        return 0;
    };
    const int s_first = raster ? 0 : (m->k1 == 3 ? -1 : 0);
    const int s_last = raster ? Hb * Wb : Wb + 2 * (Hb - 1);
    for (int s = s_first; s < s_last; ++s) {
        if (wave) {
            if (s < 0) LBIC_TRY(launch_step(s));     // KS[1] = 3: step -1 has ring positions only
            else if (pend < 0) pend = s;
        } else {
            LBIC_TRY(launch_step(s));
        }
        if (hk && hk->rows_done) {
            int done = -1;
            if (raster) {
                if ((s + 1) % Wb == 0) done = (s + 1) / Wb;
            } else if (s >= Wb - 1) {
                done = (s - (Wb - 1)) / 2 + 1;
                done = done < Hb ? done : Hb;
            }
            if (done > 0 && (!wave || !hk->will_done || hk->will_done(hk->ctx, done))) {
                LBIC_TRY(flush(s + 1));
                LBIC_TRY(hk->rows_done(hk->ctx, done, st));
            }
        }
    }
    LBIC_TRY(flush(s_last));
    if (zhat_out) LBIC_TRY(launch_cl_to_nchw(ws.zhat_cl, zhat_out, n_img, m->Cin, HW, st));
    if (sym_out) LBIC_CUDA(cudaMemcpyAsync(sym_out, ws.sym, sizeof(int32_t) * nblk * m->M, cudaMemcpyDeviceToDevice, st));
    return ws_release(m, st);
}

int ensure_io(lbic_model *m, size_t bytes) {
    if (m->io_bytes >= bytes) return 0;
    if (m->io_dev) { cudaDeviceSynchronize(); cudaFree(m->io_dev); m->io_dev = nullptr; m->io_bytes = 0; }
    cudaError_t e = cudaMalloc(&m->io_dev, bytes);
    if (e != cudaSuccess) return lbic_fail(LBIC_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    m->io_bytes = bytes;
    return 0;
}
size_t align256(size_t v) { return (v + 255) / 256 * 256; }

int check_async(lbic_model *m) {
    int flag = 0;
    LBIC_CUDA(cudaMemcpy(&flag, m->err_flag, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        cudaMemset(m->err_flag, 0, sizeof(int));
        return lbic_fail(flag == 1 ? LBIC_ERR_OVERFLOW : LBIC_ERR_INVALID,
                         flag == 1 ? "bitstream buffer too small (stream_cap)" : "malformed lane container");
    }
    return 0;
}

// ---- host-buffer calls -----------------------------------------------------------------------------------------
// The wavefront reads block row v of the input for the first time at step 2v and writes block row v of the
// reconstruction for the last time at step Wb-1+2v, so a host call moves the batch in BANDS of block rows: all input
// bands are queued on a copy stream up front and the compute stream waits for band b only right before the first step
// that touches it (converting it to the channel-last working layout then); every finished band of the reconstruction is
// converted and handed to a second copy stream at once.  The whole batch stays ONE batch for the GEMMs, and all but the
// first input band and the last output band of the PCIe time hides behind the wavefront.
int host_pipeline_init(lbic_model *m) {
    if (m->hs[0]) return 0;
    for (int i = 0; i < 3; ++i) LBIC_CUDA(cudaStreamCreateWithFlags(&m->hs[i], cudaStreamNonBlocking));
    for (auto &ev : m->hev) LBIC_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    return 0;
}

struct BandPipe {
    lbic_model *m = nullptr;
    int n = 0, Hb = 0, Wb = 0;
    int nb = 0, vb[LBIC_MAX_BANDS + 1] = {};      // band b = block rows [vb[b], vb[b+1])
    int next_in = 0, next_out = 0;
    int fmt = 0;                                  // 0: fp32 (n, Cin, Hb, Wb) block tensors, 1: u8 (n, 3, H, W) images
    int H = 0, W = 0, B = 0;                      // fmt 1
    const uint8_t *h_in = nullptr; uint8_t *d_in = nullptr;
    uint8_t *h_out = nullptr; uint8_t *d_out = nullptr;
    int rc = 0;

    void plan(lbic_model *model, int n_img, int hb, int wb) {
        m = model; n = n_img; Hb = hb; Wb = wb;
        nb = hb < m->host_bands ? hb : m->host_bands;
        for (int b = 0; b <= nb; ++b) vb[b] = (int)((long)hb * b / nb);
    }
    // plane geometry of a band for the 2-D copies: `planes` rows of `pitch` bytes, the band is bytes [off, off + width)
    void geom(int b, size_t &planes, size_t &pitch, size_t &off, size_t &width) const {
        if (fmt == 0) {
            planes = (size_t)n * m->Cin; pitch = sizeof(float) * (size_t)Hb * Wb;
            off = sizeof(float) * (size_t)vb[b] * Wb; width = sizeof(float) * (size_t)(vb[b + 1] - vb[b]) * Wb;
        } else {
            const int y0 = vb[b] * B, y1 = vb[b + 1] * B < H ? vb[b + 1] * B : H;
            planes = (size_t)n * 3; pitch = (size_t)H * W;
            off = (size_t)y0 * W; width = y1 > y0 ? (size_t)(y1 - y0) * W : 0;
        }
    }
    int queue_inputs() {
        for (int b = 0; b < nb; ++b) {
            size_t planes, pitch, off, width;
            geom(b, planes, pitch, off, width);
            if (width) LBIC_CUDA(cudaMemcpy2DAsync(d_in + off, pitch, h_in + off, pitch, width, planes, cudaMemcpyHostToDevice, m->hs[0]));
            LBIC_CUDA(cudaEventRecord(m->hev[b], m->hs[0]));
        }
        return 0;
    }
    static bool will_need(void *ctx, int v_hi) {
        const BandPipe *p = (const BandPipe *)ctx;
        return p->next_in < p->nb && p->vb[p->next_in] <= v_hi;
    }
    static bool will_done(void *ctx, int v_done) {
        const BandPipe *p = (const BandPipe *)ctx;
        return p->next_out < p->nb && p->vb[p->next_out + 1] <= v_done;
    }
    static int need_rows(void *ctx, int v_hi, cudaStream_t st) {
        BandPipe *p = (BandPipe *)ctx;
        while (p->next_in < p->nb && p->vb[p->next_in] <= v_hi) {
            const int b = p->next_in++;
            LBIC_CUDA(cudaStreamWaitEvent(st, p->m->hev[b], 0));
            if (p->fmt == 0)
                LBIC_TRY(launch_nchw_to_cl_band((const float *)p->d_in, p->m->ws.x_cl, p->n, p->m->Cin, p->Hb, p->Wb, p->vb[b], p->vb[b + 1], st));
            else
                LBIC_TRY(launch_u8_to_xcl(p->d_in, p->m->ws.x_cl, p->n, p->H, p->W, p->Hb, p->Wb, p->B, p->vb[b], p->vb[b + 1], st));
        }
        return 0;
    }
    static int rows_done(void *ctx, int v_done, cudaStream_t st) {
        BandPipe *p = (BandPipe *)ctx;
        while (p->next_out < p->nb && p->vb[p->next_out + 1] <= v_done) {
            const int b = p->next_out++;
            if (p->fmt == 0)
                LBIC_TRY(launch_cl_to_nchw_band(p->m->ws.zhat_cl, (float *)p->d_out, p->n, p->m->Cin, p->Hb, p->Wb, p->vb[b], p->vb[b + 1], st));
            else
                LBIC_TRY(launch_zcl_to_u8(p->m->ws.zhat_cl, p->d_out, p->n, p->H, p->W, p->Hb, p->Wb, p->B, p->vb[b], p->vb[b + 1], st));
            LBIC_CUDA(cudaEventRecord(p->m->hev[LBIC_MAX_BANDS + b], st));
            LBIC_CUDA(cudaStreamWaitEvent(p->m->hs[2], p->m->hev[LBIC_MAX_BANDS + b], 0));
            size_t planes, pitch, off, width;
            p->geom(b, planes, pitch, off, width);
            if (width) LBIC_CUDA(cudaMemcpy2DAsync(p->h_out + off, pitch, p->d_out + off, pitch, width, planes, cudaMemcpyDeviceToHost, p->m->hs[2]));
        }
        return 0;
    }
};

// fmt 0: x / zhat are fp32 (n, 3B^2, Hb, Wb) block tensors; fmt 1: 8-bit (n, 3, H, W) images (pad / crop fused)
int encode_host_impl(lbic_model *m, int fmt, const void *in, int n_img, int H, int W, int Hb, int Wb, void *recon_out,
                     uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes) {
    LBIC_TRY(check_ready(m, stream_out != nullptr));
    if (!in || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    if (stream_out && (!stream_len || stream_cap % 4)) return lbic_fail(LBIC_ERR_INVALID, "stream_cap must be a multiple of 4");
    Active act(m);
    LBIC_TRY(host_pipeline_init(m));
    const size_t nin = fmt == 0 ? sizeof(float) * (size_t)m->Cin * Hb * Wb * n_img : (size_t)n_img * 3 * H * W;
    const size_t o_in = 0, o_out = align256(nin), o_len = o_out + (recon_out ? align256(nin) : 0),
                 o_s = o_len + align256(4 * (size_t)n_img);
    LBIC_TRY(ensure_io(m, o_s + (stream_out ? (size_t)n_img * stream_cap : 0)));
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    uint8_t *io = (uint8_t *)m->io_dev;
    cudaStream_t s_cmp = m->hs[1], s_out = m->hs[2];
    BandPipe bp;
    bp.plan(m, n_img, Hb, Wb);
    bp.fmt = fmt; bp.H = H; bp.W = W; bp.B = m->cfg.block_size;
    bp.h_in = (const uint8_t *)in; bp.d_in = io + o_in;
    bp.h_out = (uint8_t *)recon_out; bp.d_out = io + o_out;
    LBIC_TRY(bp.queue_inputs());
    RowHooks hk;
    hk.ctx = &bp; hk.need_rows = BandPipe::need_rows; hk.rows_done = recon_out ? BandPipe::rows_done : nullptr;
    hk.will_need = BandPipe::will_need; hk.will_done = BandPipe::will_done;
    int rc = encode_impl(m, nullptr, n_img, Hb, Wb, nullptr, nullptr, nullptr, stream_out ? io + o_s : nullptr, stream_cap,
                         (uint32_t *)(io + o_len), lanes, s_cmp, &hk);
    Active act2(m);
    if (rc == 0 && stream_out && cudaMemcpyAsync(stream_len, io + o_len, 4 * (size_t)n_img, cudaMemcpyDeviceToHost, s_cmp) != cudaSuccess)
        rc = lbic_fail(LBIC_ERR_CUDA, "copy failed");
    cudaError_t e0 = cudaStreamSynchronize(m->hs[0]), e1 = cudaStreamSynchronize(s_cmp);
    if (rc == 0 && (e0 != cudaSuccess || e1 != cudaSuccess))
        rc = lbic_fail(LBIC_ERR_CUDA, "encode failed: %s", cudaGetErrorString(e0 != cudaSuccess ? e0 : e1));
    if (rc == 0 && stream_out) rc = check_async(m);
    if (rc == 0 && stream_out) {
        // one strided copy for all bitstreams: every image's slot up to the longest stream of the batch
        size_t longest = 0;
        for (int i = 0; i < n_img; ++i) longest = stream_len[i] > longest ? stream_len[i] : longest;
        if (longest > stream_cap) rc = lbic_fail(LBIC_ERR_OVERFLOW, "bitstream buffer too small (stream_cap)");
        else if (longest && cudaMemcpy2DAsync(stream_out, stream_cap, io + o_s, stream_cap, longest, n_img, cudaMemcpyDeviceToHost, s_cmp) != cudaSuccess)
            rc = lbic_fail(LBIC_ERR_CUDA, "copy failed");
        if (cudaStreamSynchronize(s_cmp) != cudaSuccess && rc == 0) rc = lbic_fail(LBIC_ERR_CUDA, "stream copy failed");
    }
    cudaError_t e2 = cudaStreamSynchronize(s_out);
    if (rc == 0 && e2 != cudaSuccess) rc = lbic_fail(LBIC_ERR_CUDA, "encode failed: %s", cudaGetErrorString(e2));
    return rc;
}

int decode_host_impl(lbic_model *m, int fmt, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                     int n_img, int H, int W, int Hb, int Wb, void *out, int lanes) {
    LBIC_TRY(check_ready(m, true));
    if (!streams || !stream_len || !out || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    if (stream_cap % 4) return lbic_fail(LBIC_ERR_INVALID, "stream_cap must be a multiple of 4");
    Active act(m);
    LBIC_TRY(host_pipeline_init(m));
    const size_t nout = fmt == 0 ? sizeof(float) * (size_t)m->Cin * Hb * Wb * n_img : (size_t)n_img * 3 * H * W;
    const size_t o_out = 0, o_len = align256(nout), o_s = o_len + align256(4 * (size_t)n_img);
    LBIC_TRY(ensure_io(m, o_s + (size_t)n_img * stream_cap));
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    uint8_t *io = (uint8_t *)m->io_dev;
    cudaStream_t s_cmp = m->hs[1], s_out = m->hs[2];
    size_t longest = 0;
    for (int i = 0; i < n_img; ++i) {
        if (stream_len[i] > stream_cap) return lbic_fail(LBIC_ERR_INVALID, "stream %d longer than stream_cap", i);
        longest = stream_len[i] > longest ? stream_len[i] : longest;
    }
    LBIC_CUDA(cudaMemcpyAsync(io + o_len, stream_len, 4 * (size_t)n_img, cudaMemcpyHostToDevice, s_cmp));
    if (longest) LBIC_CUDA(cudaMemcpy2DAsync(io + o_s, stream_cap, streams, stream_cap, longest, n_img, cudaMemcpyHostToDevice, s_cmp));
    BandPipe bp;
    bp.plan(m, n_img, Hb, Wb);
    bp.fmt = fmt; bp.H = H; bp.W = W; bp.B = m->cfg.block_size;
    bp.h_out = (uint8_t *)out; bp.d_out = io + o_out;
    RowHooks hk;
    hk.ctx = &bp; hk.rows_done = BandPipe::rows_done; hk.will_done = BandPipe::will_done;
    int rc = decode_impl(m, io + o_s, (const uint32_t *)(io + o_len), stream_cap, n_img, Hb, Wb, nullptr, nullptr, lanes,
                         s_cmp, &hk);
    Active act2(m);
    cudaError_t e1 = cudaStreamSynchronize(s_cmp), e2 = cudaStreamSynchronize(s_out);
    if (rc) return rc;
    if (e1 != cudaSuccess || e2 != cudaSuccess)
        return lbic_fail(LBIC_ERR_CUDA, "decode failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
    return check_async(m);
}
}  // namespace

extern "C" int lbic_encode_host(lbic_model *m, const float *x, int n_img, int Hb, int Wb, float *zhat_out,
                                uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes) {
    return encode_host_impl(m, 0, x, n_img, 0, 0, Hb, Wb, zhat_out, stream_out, stream_cap, stream_len, lanes);
}

extern "C" int lbic_decode_host(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                                int n_img, int Hb, int Wb, float *zhat_out, int lanes) {
    return decode_host_impl(m, 0, streams, stream_len, stream_cap, n_img, 0, 0, Hb, Wb, zhat_out, lanes);
}

extern "C" int lbic_encode_images_u8_host(lbic_model *m, const uint8_t *img, int n_img, int H, int W, uint8_t *recon_out,
                                          uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len, int lanes) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    if (H < 1 || W < 1) return lbic_fail(LBIC_ERR_INVALID, "bad image size");
    const int B = m->cfg.block_size;
    return encode_host_impl(m, 1, img, n_img, H, W, (H + B - 1) / B, (W + B - 1) / B, recon_out, stream_out, stream_cap,
                            stream_len, lanes);
}

extern "C" int lbic_decode_images_u8_host(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len,
                                          size_t stream_cap, int n_img, int H, int W, uint8_t *img_out, int lanes) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    if (H < 1 || W < 1) return lbic_fail(LBIC_ERR_INVALID, "bad image size");
    const int B = m->cfg.block_size;
    return decode_host_impl(m, 1, streams, stream_len, stream_cap, n_img, H, W, (H + B - 1) / B, (W + B - 1) / B, img_out,
                            lanes);
}

// ------------------------------------------------------------------------------------------------
// eval_model's quality figures on the GPU (SURVEY.md 8(f) rank 4; AGENT:611-619): per-image MSE and MS-SSIM.
// ------------------------------------------------------------------------------------------------
extern "C" int lbic_image_metrics(lbic_model *m, const float *x, const float *y, int n, int C, int H, int W, float offset,
                                  float data_range, double *mse_out, double *msssim_out, void *stream) {
    if (!m || !x || !y || !mse_out) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    Active act(m);
    float *scratch = nullptr;
    LBIC_TRY(ensure_aux(m, 2, metrics_scratch_bytes(n, C, H, W), &scratch));
    return launch_image_metrics(x, y, n, C, H, W, offset, data_range, scratch, mse_out, msssim_out, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// Post-processing net (SURVEY.md 8(f) rank 4): BlkBasedPostProcessing, NET:455-476, applied to the block tensor of a
// reconstruction when `use_postpm` is set (AGENT:604-606).  x + pad(conv1x1(lrelu(conv3x3_valid(x)))): two GEMMs over
// all blocks of the batch in raster chunks (nothing is recursive here), the residual add and the caller's clamp fused
// into the second epilogue; blocks on the image border keep their input (the residual is zero padded).
// ------------------------------------------------------------------------------------------------
extern "C" int lbic_load_postpm_weights(lbic_model *m, const lbic_tensor_desc *tensors, int n_tensors, void *stream) {
    if (!m || !tensors) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(gemm_tc_init());
    SdView sd;
    for (int i = 0; i < n_tensors; ++i)
        if (tensors[i].name && tensors[i].data) sd.by_name[tensors[i].name] = &tensors[i];
    LBIC_CUDA(cudaDeviceSynchronize());
    free_all(m->pp_allocs);
    m->postpm_loaded = false;
    std::vector<void *> tmp;
    std::swap(m->weight_allocs, m->pp_allocs);          // the packers allocate into weight_allocs
    int rc = pack_linear_into(m, m->PP[0], sd, "res_net.0", 4 * m->Cin, m->Cin, 3, TAPS_9, 9, tmp, st);
    if (rc == 0) rc = pack_linear_into(m, m->PP[1], sd, "res_net.2", m->Cin, 4 * m->Cin, 1, TAPS_1, 1, tmp, st);
    std::swap(m->weight_allocs, m->pp_allocs);
    cudaError_t e = cudaStreamSynchronize(st);
    free_all(tmp);
    if (rc) return rc;
    if (e != cudaSuccess) return lbic_fail(LBIC_ERR_CUDA, "weight packing failed: %s", cudaGetErrorString(e));
    m->postpm_loaded = true;
    return 0;
}

extern "C" int lbic_postprocess(lbic_model *m, const float *z, int n_img, int Hb, int Wb, float *out, int clamp, void *stream) {
    if (!m || !z || !out || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    if (!m->postpm_loaded) return lbic_fail(LBIC_ERR_STATE, "post-processing weights not loaded: call lbic_load_postpm_weights first");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    Workspace &ws = m->ws;
    if (m->pp_rcap != ws.R_cap) {                       // operand buffers of the two layers, sized like the workspace's
        LBIC_CUDA(cudaDeviceSynchronize());
        free_all(m->pp_ws_allocs);
        m->PPA.ld = 9 * m->Cin; m->PPH.ld = 4 * m->Cin;
        for (ActBuf *b : {&m->PPA, &m->PPH}) {
            LBIC_TRY(dev_alloc(m->pp_ws_allocs, (void **)&b->hi, sizeof(h16) * (size_t)ws.R_cap * b->ld, true));
            LBIC_TRY(dev_alloc(m->pp_ws_allocs, (void **)&b->lo, sizeof(h16) * (size_t)ws.R_cap * b->ld, true));
        }
        LBIC_TRY(make_view(ws, m->vPPA, m->PPA, 9 * m->Cin));
        LBIC_TRY(make_view(ws, m->vPPH, m->PPH, 4 * m->Cin));
        m->pp_rcap = ws.R_cap;
    }
    const int HW = Hb * Wb;
    const long nblk = (long)n_img * HW;
    float *out_cl = nullptr;
    LBIC_TRY(ws_acquire(m, st));
    LBIC_TRY(ensure_aux(m, 1, sizeof(float) * (size_t)nblk * m->Cin, &out_cl));
    LBIC_TRY(launch_nchw_to_cl(z, ws.zhat_cl, n_img, m->Cin, HW, st));
    const int chunk = ws.R_cap;
    for (long r0 = 0; r0 < nblk; r0 += chunk) {
        const int R = (int)(nblk - r0 < chunk ? nblk - r0 : chunk);
        const StepDesc sd{n_img, 0, 0, (int)r0, Hb, Wb};                       // raster chunk: row r = block r0 + r
        LBIC_TRY(launch_gather9(ws.zhat_cl, m->Cin, sd, R, m->PPA.hi, m->PPA.lo, m->PPA.ld, st));
        LBIC_TRY(run_gemm_layer(m, m->PP[0], -1, R, &m->vPPA, nullptr, epi_hilo(EPI_LRELU, sd, m->PPH), st));
        EpiParams e = epi(EPI_RESID, sd);
        e.out_f32 = out_cl + (size_t)r0 * m->Cin; e.ld_f32 = m->Cin;
        e.aux = ws.zhat_cl + (size_t)r0 * m->Cin; e.ld_aux = m->Cin;
        e.no_clamp = clamp ? 0 : 1;
        LBIC_TRY(run_gemm_layer(m, m->PP[1], -1, R, &m->vPPH, nullptr, e, st));
    }
    LBIC_TRY(launch_restore_border(ws.zhat_cl, out_cl, m->Cin, n_img, Hb, Wb, st));
    LBIC_TRY(launch_cl_to_nchw(out_cl, out, n_img, m->Cin, HW, st));
    return ws_release(m, st);
}

// ------------------------------------------------------------------------------------------------
// Block-row bands: ONE large image over several GPUs (BASELINE config 5).
//
// Dependencies cross a horizontal cut only downwards: block (v, h) reads zhat of row v-1 at columns h-1 .. h+1
// (KS[1] = 1), and (v-1, h+1) belongs to wavefront step t-1.  Rank g owns block rows [v0, v1) and runs every step
// restricted to them; after step t it owes the rank below ONE block, zhat(v1-1, t - 2 (v1-1)), before that rank's step
// t+1.  The library runs the steps and exposes the reconstruction buffer; the caller (band.py, torch.distributed
// send / recv over NVLink) moves the halo blocks -- the only exchange on the data path.  Each band is entropy-coded as
// the lanes of its own block rows (the lane container holds one rANS stream per block row), so the bands' payloads
// concatenate into the same container a single GPU writes.
// ------------------------------------------------------------------------------------------------
extern "C" int lbic_band_begin(lbic_model *m, const float *x, int n_img, int Hb, int Wb, const uint8_t *streams,
                               const uint32_t *stream_len, size_t stream_cap, void *stream) {
    const bool decode = streams != nullptr;
    LBIC_TRY(check_ready(m, decode));
    if ((!x && !decode) || (decode && !stream_len) || n_img < 1 || Hb < 1 || Wb < 1) return lbic_fail(LBIC_ERR_INVALID, "bad arguments");
    if (m->k1 != 1) return lbic_fail(LBIC_ERR_INVALID, "band mode supports KS[1] = 1 (one halo block per step)");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(ensure_workspace(m, n_img, Hb, Wb));
    Workspace &ws = m->ws;
    const size_t nblk = (size_t)n_img * Hb * Wb;
    LBIC_TRY(ws_acquire(m, st));
    LBIC_CUDA(cudaMemsetAsync(m->err_flag, 0, sizeof(int), st));
    LBIC_CUDA(cudaMemsetAsync(ws.zhat_cl, 0, sizeof(float) * nblk * m->Cin, st));
    if (decode) {
        if (stream_cap % 4) return lbic_fail(LBIC_ERR_INVALID, "stream_cap must be a multiple of 4");
        LBIC_TRY(launch_rans_dec_init(streams, stream_len, stream_cap, n_img, Hb, 1, ws.dec_states, ws.lane_ptr, m->err_flag, st));
    } else {
        LBIC_TRY(launch_nchw_to_cl(x, ws.x_cl, n_img, m->Cin, Hb * Wb, st));
    }
    m->band_n = n_img; m->band_Hb = Hb; m->band_Wb = Wb; m->band_decode = decode ? 1 : 0;
    return 0;
}

extern "C" float *lbic_band_zhat(lbic_model *m) { return (m && m->band_n) ? m->ws.zhat_cl : nullptr; }

// wavefront step t restricted to block rows [v0, v1)
extern "C" int lbic_band_step(lbic_model *m, int t, int v0, int v1, void *stream) {
    if (!m || !m->band_n) return lbic_fail(LBIC_ERR_STATE, "lbic_band_begin has not been called");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    Workspace &ws = m->ws;
    const int n_img = m->band_n, Hb = m->band_Hb, Wb = m->band_Wb;
    StepDesc sd;
    if (!wave_step(t, n_img, Hb, Wb, sd)) return 0;
    const int lo = sd.vmin > v0 ? sd.vmin : v0;
    const int hi = (sd.vmin + sd.nv) < v1 ? (sd.vmin + sd.nv) : v1;
    if (hi <= lo) return 0;
    sd.vmin = lo; sd.nv = hi - lo;
    const int R = n_img * sd.nv;
    if (m->band_decode) {
        LBIC_TRY(launch_gather(nullptr, ws.zhat_cl, m->Cin, sd, R, nullptr, nullptr, 0, ws.T.hi, ws.T.lo, ws.T.ld, st));
        LBIC_TRY(run_ent(m, sd, R, st));
        LBIC_TRY(launch_rans_dec_step(m->tables, ws.dec_states, ws.lane_ptr, Hb, sd, R, m->M, ws.KSI, ws.ldKSI, ws.YQ.hi,
                                      ws.YQ.lo, ws.YQ.ld, nullptr, st));
        return run_dec(m, sd, R, st);
    }
    LBIC_TRY(launch_gather(ws.x_cl, ws.zhat_cl, m->Cin, sd, R, ws.X.hi, ws.X.lo, ws.X.ld, ws.T.hi, ws.T.lo, ws.T.ld, st));
    return encode_step(m, sd, R, true, st);
}

// Ends the call for block rows [v0, v1): the band's reconstruction (channel-last rows, (n_img, v1-v0, Wb, 3B^2)) and,
// after an encode, its lanes: lane_out holds n_img * (v1-v0) slots of lane_cap bytes, lane_len their byte counts.
extern "C" int lbic_band_end(lbic_model *m, int v0, int v1, float *zhat_rows_out, uint8_t *lane_out, size_t lane_cap,
                             uint32_t *lane_len, void *stream) {
    if (!m || !m->band_n) return lbic_fail(LBIC_ERR_STATE, "lbic_band_begin has not been called");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    Workspace &ws = m->ws;
    const int n_img = m->band_n, Hb = m->band_Hb, Wb = m->band_Wb, nr = v1 - v0;
    if (v0 < 0 || v1 > Hb || nr <= 0) return lbic_fail(LBIC_ERR_INVALID, "bad band");
    const size_t row_f = (size_t)Wb * m->Cin;
    if (zhat_rows_out)
        LBIC_CUDA(cudaMemcpy2DAsync(zhat_rows_out, sizeof(float) * row_f * nr, ws.zhat_cl + (size_t)v0 * row_f,
                                    sizeof(float) * row_f * Hb, sizeof(float) * row_f * nr, n_img, cudaMemcpyDeviceToDevice, st));
    if (lane_out && !m->band_decode) {
        if (!lane_len || lane_cap % 4) return lbic_fail(LBIC_ERR_INVALID, "lane_cap must be a multiple of 4");
        const int64_t n_sym = (int64_t)Wb * m->M;
        const size_t per = lane_cap / 4;
        LBIC_TRY(ensure_rans_scratch(m, (size_t)nr * per + 2 * (size_t)nr));
        for (int i = 0; i < n_img; ++i) {
            const size_t o = ((size_t)i * Hb + v0) * Wb * m->M;
            LBIC_TRY(launch_rans_encode(m->tables, ws.sym + o, ws.idx + o, nr, n_sym, n_sym, ws.rans_scratch, per,
                                        lane_out + (size_t)i * nr * lane_cap, lane_cap, lane_len + (size_t)i * nr, m->err_flag, st));
        }
    }
    m->band_n = 0;
    return ws_release(m, st);
}

extern "C" int lbic_space_to_depth(const float *img, float *blk, int n, int C, int Hb, int Wb, int B, void *stream) {
    if (!img || !blk) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    return launch_space_to_depth(img, blk, n, C, Hb, Wb, B, (cudaStream_t)stream);
}

extern "C" int lbic_depth_to_space(const float *blk, float *img, int n, int C, int Hb, int Wb, int B, void *stream) {
    if (!img || !blk) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    return launch_depth_to_space(blk, img, n, C, Hb, Wb, B, (cudaStream_t)stream);
}

extern "C" int lbic_rans_encode(lbic_model *m, const int32_t *symbols, const uint8_t *indexes, int n_streams,
                                int64_t n_sym, uint8_t *stream_out, size_t stream_cap, uint32_t *stream_len,
                                void *stream) {
    if (!m || !symbols || !indexes || !stream_out || !stream_len) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    if (!m->tables.cdf) return lbic_fail(LBIC_ERR_STATE, "Uninitialized CDFs. Run update() first");
    if (stream_cap % 4) return lbic_fail(LBIC_ERR_INVALID, "stream_cap must be a multiple of 4");
    Active act(m);
    if (m->ws.n_img == 0) LBIC_TRY(ensure_workspace(m, 1, 1, 2));
    const size_t per = stream_cap / 4;
    LBIC_TRY(ensure_rans_scratch(m, (size_t)n_streams * per + 2 * (size_t)n_streams));
    return launch_rans_encode(m->tables, symbols, indexes, n_streams, n_sym, n_sym, m->ws.rans_scratch, per, stream_out,
                              stream_cap, stream_len, m->err_flag, (cudaStream_t)stream);
}

extern "C" int lbic_rans_decode(lbic_model *m, const uint8_t *streams, const uint32_t *stream_len, size_t stream_cap,
                                const uint8_t *indexes, int n_streams, int64_t n_sym, int32_t *symbols_out,
                                void *stream) {
    if (!m || !streams || !stream_len || !indexes || !symbols_out) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    Active act(m);
    return launch_rans_decode_full(m->tables, streams, stream_len, stream_cap, indexes, n_streams, n_sym, symbols_out,
                                   (cudaStream_t)stream);
}

extern "C" int lbic_debug_gemm(lbic_model *m, const float *A, const float *W, float *D, int R, int K, int cout,
                               void *stream) {
    if (!m || !A || !W || !D) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    if (K % 8 || cout % 16) return lbic_fail(LBIC_ERR_INVALID, "debug gemm needs K %% 8 == 0 and cout %% 16 == 0");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<void *> tmp;
    h16 *ah, *al, *wh, *wl;
    int rc = 0;
    do {
#define P(call) if ((rc = (call)) != 0) break
        P(dev_alloc(tmp, (void **)&ah, sizeof(h16) * (size_t)R * K));
        P(dev_alloc(tmp, (void **)&al, sizeof(h16) * (size_t)R * K));
        P(dev_alloc(tmp, (void **)&wh, sizeof(h16) * (size_t)cout * K));
        P(dev_alloc(tmp, (void **)&wl, sizeof(h16) * (size_t)cout * K));
        P(launch_split_f32(A, ah, al, (int64_t)R * K, st));
        P(launch_split_f32(W, wh, wl, (int64_t)cout * K, st));
        GemmCall g;
        memset(&g, 0, sizeof(g));
        g.R = R; g.cout = cout; g.bn = pick_bn(cout); g.nseg = 1; g.K[0] = K;
        const bool ws = m->gemm_core == 0 && m->use_ws == 2;   // forced persistent kernel (optionally its CTA-pair form)
        const int pair = ws && m->use_pair;
        if (ws) {
            const int wmax = (pair && m->use_pair == 3) ? gemm_pair_max_bn() : gemm_ws_max_bn();
            const int nt = (cout + wmax - 1) / wmax;
            g.bn = ((cout + nt - 1) / nt + 15) / 16 * 16;
        }
        CUtensorMap ta_h, ta_l, tw_h, tw_l;
        P(make_tmap_2d(&ta_h, ah, K, R, K, 64, 128));
        P(make_tmap_2d(&ta_l, al, K, R, K, 64, 128));
        P(make_tmap_2d(&tw_h, wh, K, cout, K, 64, pair ? g.bn / 2 : g.bn));
        P(make_tmap_2d(&tw_l, wl, K, cout, K, 64, pair ? g.bn / 2 : g.bn));
        g.A[0].hi = ah; g.A[0].lo = al; g.A[0].ld = K; g.A[0].tm_hi = &ta_h; g.A[0].tm_lo = &ta_l;
        g.W[0].hi = wh; g.W[0].lo = wl; g.W[0].ld = K; g.W[0].tm_hi = &tw_h; g.W[0].tm_lo = &tw_l;
        g.ep.mode = EPI_RAW; g.ep.R = R; g.ep.cout = cout; g.ep.out_f32 = D; g.ep.ld_f32 = cout; g.ep.acc_scale = 1.0f;
        P(m->gemm_core == 1 ? gemm_simt_launch(g, st) : (ws ? gemm_ws_launch(g, st, pair) : gemm_tc_launch(g, st)));
#undef P
    } while (0);
    cudaError_t e = cudaStreamSynchronize(st);
    free_all(tmp);
    if (rc) return rc;
    if (e != cudaSuccess) return lbic_fail(LBIC_ERR_CUDA, "debug gemm failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int lbic_debug_layer(lbic_model *m, const lbic_debug_layer_args *a, void *stream) {
    if (!m || !a) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    const int md = a->mode;
    if (md < EPI_LRELU || md > EPI_RESID || a->core < 0 || a->core > 4 || a->R < 1 || a->cout < 16 || a->cout % 16 ||
        a->nseg < 1 || a->nseg > 2)
        return lbic_fail(LBIC_ERR_INVALID, "debug layer: bad mode / core / shape");
    for (int s = 0; s < a->nseg; ++s)
        if (!a->A[s] || !a->W[s] || a->K[s] < 8 || a->K[s] % 8)
            return lbic_fail(LBIC_ERR_INVALID, "debug layer: segment %d needs A, W and K %% 8 == 0", s);
    const bool needs_aux = md == EPI_GDN || md == EPI_IGDN || md == EPI_QUANT || md == EPI_RESID;
    if ((epi_has_f32(md) && !a->out_f32) || (epi_has_hilo(md) && (!a->out_hi || !a->out_lo)) ||
        (md == EPI_QUANT && !a->out_idx) || (needs_aux && !a->aux))
        return lbic_fail(LBIC_ERR_INVALID, "debug layer: an output or side input of mode %d is missing", md);
    if (md == EPI_QUANT && (a->M < a->cout || a->ld_aux < a->M + a->cout || (!a->scale_table && !m->tables.d_scale_table)))
        return lbic_fail(LBIC_ERR_INVALID, "debug layer: QUANT needs M >= cout, ld_aux >= M + cout and a scale table");
    if (a->core == 1 && a->force_bn && (a->force_bn % 16 || a->force_bn > 256))
        return lbic_fail(LBIC_ERR_INVALID, "debug layer: bad tile width %d", a->force_bn);
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    std::vector<void *> tmp;
    int rc = 0;
    do {
#define P(call) if ((rc = (call)) != 0) break
        GemmCall g;
        memset(&g, 0, sizeof(g));
        const int pair = a->core >= 3;
        // activation planes cover whole (pair) tiles, zero beyond row R, as the workspace buffers do (R_cap rows)
        const int Rp = (a->R + 255) / 256 * 256;
        g.R = a->R; g.cout = a->cout; g.nseg = a->nseg;
        if (a->core >= 2) {
            const int wmax = a->core == 4 ? gemm_pair_max_bn() : gemm_ws_max_bn();
            const int nt = (a->cout + wmax - 1) / wmax;
            g.bn = ((a->cout + nt - 1) / nt + 15) / 16 * 16;
        } else {
            g.bn = a->force_bn ? a->force_bn : pick_bn(a->cout);
        }
        CUtensorMap tm[2][4];   // [segment][A hi, A lo, W hi, W lo]
        for (int s = 0; s < a->nseg && rc == 0; ++s) {
            const int K = a->K[s];
            h16 *ah, *al, *wh, *wl;
            P(dev_alloc(tmp, (void **)&ah, sizeof(h16) * (size_t)Rp * K, true));
            P(dev_alloc(tmp, (void **)&al, sizeof(h16) * (size_t)Rp * K, true));
            P(dev_alloc(tmp, (void **)&wh, sizeof(h16) * (size_t)a->cout * K));
            P(dev_alloc(tmp, (void **)&wl, sizeof(h16) * (size_t)a->cout * K));
            P(launch_split_f32(a->A[s], ah, al, (int64_t)a->R * K, st));
            P(launch_split_f32(a->W[s], wh, wl, (int64_t)a->cout * K, st));
            // the maps make_view and pack_conv_seg build: 64 k x 128 rows, 64 k x tile width (half of it per CTA of a pair)
            P(make_tmap_2d(&tm[s][0], ah, K, Rp, K, 64, 128));
            P(make_tmap_2d(&tm[s][1], al, K, Rp, K, 64, 128));
            P(make_tmap_2d(&tm[s][2], wh, K, a->cout, K, 64, pair ? g.bn / 2 : g.bn));
            P(make_tmap_2d(&tm[s][3], wl, K, a->cout, K, 64, pair ? g.bn / 2 : g.bn));
            g.K[s] = K;
            g.A[s].hi = ah; g.A[s].lo = al; g.A[s].ld = K; g.A[s].tm_hi = &tm[s][0]; g.A[s].tm_lo = &tm[s][1];
            g.W[s].hi = wh; g.W[s].lo = wl; g.W[s].ld = K; g.W[s].tm_hi = &tm[s][2]; g.W[s].tm_lo = &tm[s][3];
        }
        if (rc) break;
        float *bias = const_cast<float *>(a->bias);
        if (!bias) P(dev_alloc(tmp, (void **)&bias, sizeof(float) * a->cout, true));
        StepDesc raster = {1, 0, 0, 0, a->R, 1};   // raster chunk of one image of R x 1 blocks: row r -> block r
        EpiParams &e = g.ep;
        e = epi(md, raster);
        e.R = a->R; e.cout = a->cout; e.bias = bias; e.acc_scale = a->acc_scale;
        e.no_clamp = a->no_clamp;
        e.aux = a->aux; e.ld_aux = a->ld_aux; e.M = a->M;
        e.scale_tab = a->scale_table ? a->scale_table : m->tables.d_scale_table;
        e.out_hi = reinterpret_cast<h16 *>(a->out_hi); e.out_lo = reinterpret_cast<h16 *>(a->out_lo); e.ld_out = a->cout;
        if (md == EPI_QUANT) {
            e.sym = reinterpret_cast<int32_t *>(a->out_f32);
            e.idx = a->out_idx;
        } else if (md == EPI_RECON) {
            e.zhat = a->out_f32;
        } else {
            e.out_f32 = a->out_f32; e.ld_f32 = a->cout;
        }
        P(a->core == 0 ? gemm_simt_launch(g, st) : a->core == 1 ? gemm_tc_launch(g, st) : gemm_ws_launch(g, st, pair));
        if (m->check_sat && m->d_sat && epi_has_hilo(md)) P(launch_sat_scan(e.out_hi, a->R, a->cout, e.ld_out, m->d_sat, st));
#undef P
    } while (0);
    cudaError_t ce = cudaStreamSynchronize(st);
    free_all(tmp);
    if (rc) return rc;
    if (ce != cudaSuccess) return lbic_fail(LBIC_ERR_CUDA, "debug layer failed: %s", cudaGetErrorString(ce));
    return 0;
}

extern "C" int lbic_debug_selfinfo(lbic_model *m, const float *ksi, int ld_ksi, const int32_t *sym, int R, int M,
                                   float *info, void *stream) {
    if (!m || !ksi || !sym || !info || R < 1 || M < 1 || ld_ksi < M) return lbic_fail(LBIC_ERR_INVALID, "bad argument");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    const StepDesc raster = {1, 0, 0, 0, R, 1};
    LBIC_TRY(launch_selfinfo_step(raster, R, M, ksi, ld_ksi, sym, info, st));
    LBIC_CUDA(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int lbic_debug_scale_index(lbic_model *m, const float *scales, int n, const float *scale_table,
                                      int32_t *idx_bisect, int32_t *idx_hinted, void *stream) {
    if (!m || !scales || !scale_table || !idx_bisect || !idx_hinted || n < 1) return lbic_fail(LBIC_ERR_INVALID, "bad argument");
    Active act(m);
    cudaStream_t st = (cudaStream_t)stream;
    LBIC_TRY(launch_scale_index(scales, n, scale_table, idx_bisect, idx_hinted, st));
    LBIC_CUDA(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int lbic_debug_gemm_bench(lbic_model *m, int R, int K, int cout, int with_epilogue, int iters,
                                     double *ms_per_launch) {
    if (!m || !ms_per_launch || R < 1 || K % 8 || cout % 16 || iters < 1) return lbic_fail(LBIC_ERR_INVALID, "bad argument");
    Active act(m);
    cudaStream_t st = 0;
    std::vector<void *> tmp;
    int rc = 0;
    *ms_per_launch = 0;
    do {
#define P(call) if ((rc = (call)) != 0) break
        const int Rp = (R + 127) / 128 * 128;
        h16 *ah, *al, *wh, *wl, *oh, *ol;
        float *A, *W, *D, *bias;
        P(dev_alloc(tmp, (void **)&A, sizeof(float) * (size_t)Rp * K, true));
        P(dev_alloc(tmp, (void **)&W, sizeof(float) * (size_t)cout * K, true));
        P(dev_alloc(tmp, (void **)&D, sizeof(float) * (size_t)Rp * cout, true));
        P(dev_alloc(tmp, (void **)&bias, sizeof(float) * cout, true));
        P(dev_alloc(tmp, (void **)&ah, sizeof(h16) * (size_t)Rp * K, true));
        P(dev_alloc(tmp, (void **)&al, sizeof(h16) * (size_t)Rp * K, true));
        P(dev_alloc(tmp, (void **)&wh, sizeof(h16) * (size_t)cout * K, true));
        P(dev_alloc(tmp, (void **)&wl, sizeof(h16) * (size_t)cout * K, true));
        P(dev_alloc(tmp, (void **)&oh, sizeof(h16) * (size_t)Rp * cout, true));
        P(dev_alloc(tmp, (void **)&ol, sizeof(h16) * (size_t)Rp * cout, true));
        GemmCall g;
        memset(&g, 0, sizeof(g));
        const bool ws = m->use_ws == 2;
        const int pair = ws && m->use_pair;
        g.R = R; g.cout = cout; g.bn = m->force_bn ? m->force_bn : pick_bn(cout); g.nseg = 1; g.K[0] = K;
        if (ws && !m->force_bn) {
            const int wmax = (pair && m->use_pair == 3) ? gemm_pair_max_bn() : gemm_ws_max_bn();
            const int nt = (cout + wmax - 1) / wmax;
            g.bn = ((cout + nt - 1) / nt + 15) / 16 * 16;
        }
        CUtensorMap ta_h, ta_l, tw_h, tw_l;
        P(make_tmap_2d(&ta_h, ah, K, Rp, K, 64, 128));
        P(make_tmap_2d(&ta_l, al, K, Rp, K, 64, 128));
        P(make_tmap_2d(&tw_h, wh, K, cout, K, 64, pair ? g.bn / 2 : g.bn));
        P(make_tmap_2d(&tw_l, wl, K, cout, K, 64, pair ? g.bn / 2 : g.bn));
        g.A[0].hi = ah; g.A[0].lo = al; g.A[0].ld = K; g.A[0].tm_hi = &ta_h; g.A[0].tm_lo = &ta_l;
        g.W[0].hi = wh; g.W[0].lo = wl; g.W[0].ld = K; g.W[0].tm_hi = &tw_h; g.W[0].tm_lo = &tw_l;
        g.ep.R = R; g.ep.cout = cout; g.ep.acc_scale = 1.0f;
        // with_epilogue: 0 RAW, 1 PREGDN, 2 GDN, 3 QUANT, 4 LRELU, 5 KSI, 6 RECON  (synthetic operands; row r = block r)
        g.ep.bias = bias; g.ep.scale_tab = m->tables.d_scale_table;
        g.ep.step.n_img = R; g.ep.step.nv = 1; g.ep.step.vmin = 0; g.ep.step.t = 0; g.ep.step.Hb = 1; g.ep.step.Wb = 1;
        switch (with_epilogue) {
        case 0: g.ep.mode = EPI_RAW; g.ep.out_f32 = D; g.ep.ld_f32 = cout; break;
        case 1:
            g.ep.mode = EPI_PREGDN; g.ep.out_hi = oh; g.ep.out_lo = ol; g.ep.ld_out = cout;
            g.ep.out_f32 = D; g.ep.ld_f32 = cout;
            break;
        case 2: g.ep.mode = EPI_GDN; g.ep.out_hi = oh; g.ep.out_lo = ol; g.ep.ld_out = cout; g.ep.aux = D; g.ep.ld_aux = cout; break;
        case 3: {
            float *ksi; int32_t *sym; uint8_t *idx;
            P(dev_alloc(tmp, (void **)&ksi, sizeof(float) * (size_t)Rp * 2 * cout, true));
            P(dev_alloc(tmp, (void **)&sym, sizeof(int32_t) * (size_t)Rp * cout, true));
            P(dev_alloc(tmp, (void **)&idx, (size_t)Rp * cout, true));
            if (!m->tables.d_scale_table) { rc = lbic_fail(LBIC_ERR_INVALID, "QUANT bench needs entropy tables (call update first)"); break; }
            g.ep.mode = EPI_QUANT; g.ep.out_hi = oh; g.ep.out_lo = ol; g.ep.ld_out = cout;
            g.ep.aux = ksi; g.ep.ld_aux = 2 * cout; g.ep.M = cout; g.ep.sym = sym; g.ep.idx = idx;
        } break;
        case 4: g.ep.mode = EPI_LRELU; g.ep.out_hi = oh; g.ep.out_lo = ol; g.ep.ld_out = cout; break;
        case 5: g.ep.mode = EPI_KSI; g.ep.out_f32 = D; g.ep.ld_f32 = cout; break;
        case 6: g.ep.mode = EPI_RECON; g.ep.zhat = D; break;
        default: rc = lbic_fail(LBIC_ERR_INVALID, "unknown epilogue selector"); break;
        }
        if (rc) break;
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        for (int i = 0; i < 3 && rc == 0; ++i) rc = m->gemm_core == 1 ? gemm_simt_launch(g, st) : (ws ? gemm_ws_launch(g, st, pair) : gemm_tc_launch(g, st));
        if (rc) break;
        cudaEventRecord(e0, st);
        for (int i = 0; i < iters && rc == 0; ++i) rc = m->gemm_core == 1 ? gemm_simt_launch(g, st) : (ws ? gemm_ws_launch(g, st, pair) : gemm_tc_launch(g, st));
        cudaEventRecord(e1, st);
        cudaError_t e = cudaStreamSynchronize(st);
        if (rc == 0 && e != cudaSuccess) rc = lbic_fail(LBIC_ERR_CUDA, "gemm bench failed: %s", cudaGetErrorString(e));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        *ms_per_launch = ms / iters;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
#undef P
    } while (0);
    cudaDeviceSynchronize();
    free_all(tmp);
    return rc;
}

extern "C" int lbic_get_layer_profile(lbic_model *m, int max_layers, int64_t *launches, double *ms, double *flops) {
    if (!m || !launches || !ms || !flops || max_layers < 0) return lbic_fail(LBIC_ERR_INVALID, "bad argument");
    cudaSetDevice(m->device);
    LBIC_CUDA(cudaDeviceSynchronize());
    const int n = max_layers < L_COUNT ? max_layers : L_COUNT;
    for (int i = 0; i < n; ++i) { launches[i] = 0; ms[i] = 0; flops[i] = 0; }
    for (auto &r : m->prof) {
        if (r.layer < 0 || r.layer >= n) continue;
        float t = 0;
        LBIC_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
        launches[r.layer] += 1; ms[r.layer] += t; flops[r.layer] += r.flops;
    }
    return n;
}

extern "C" int lbic_saturation_count(lbic_model *m, void *stream, int64_t *count, int reset) {
    if (!m || !count) return lbic_fail(LBIC_ERR_INVALID, "null argument");
    Active act(m);
    *count = 0;
    if (!m->d_sat) return 0;
    LBIC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    unsigned long long v = 0;
    LBIC_CUDA(cudaMemcpy(&v, m->d_sat, sizeof(v), cudaMemcpyDeviceToHost));
    if (reset) LBIC_CUDA(cudaMemset(m->d_sat, 0, sizeof(v)));
    *count = (int64_t)v;
    return 0;
}

extern "C" int64_t lbic_launch_count(const lbic_model *m) { return m ? m->launches[0] + m->launches[1] : 0; }

extern "C" int lbic_set_profiling(lbic_model *m, int enabled) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    for (auto &r : m->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    m->prof.clear();
    m->profiling = enabled ? 1 : 0;
    return 0;
}

extern "C" int lbic_get_profile(lbic_model *m, int64_t *gemm_launches, double *gemm_ms, double *gemm_flops) {
    if (!m) return lbic_fail(LBIC_ERR_INVALID, "null model");
    cudaSetDevice(m->device);
    LBIC_CUDA(cudaDeviceSynchronize());
    double ms = 0, fl = 0;
    for (auto &r : m->prof) {
        float t = 0;
        LBIC_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
        ms += t;
        fl += r.flops;
    }
    if (gemm_launches) *gemm_launches = (int64_t)m->prof.size();
    if (gemm_ms) *gemm_ms = ms;
    if (gemm_flops) *gemm_flops = fl;
    return 0;
}

// Layout, gather and weight-packing kernels (HBM-bound byte movers around the GEMM chain).
#include "epilogue.cuh"

namespace {

// ---- (n, C, HW) <-> (n, HW, C) transposes -----------------------------------------------------
__global__ void transpose_kernel(const float *__restrict__ src, float *__restrict__ dst, int rows, int cols) {
    // src: [batch][rows][cols] -> dst: [batch][cols][rows]
    __shared__ float tile[32][33];
    const size_t base = (size_t)blockIdx.z * rows * cols;
    int c = blockIdx.x * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        int r = blockIdx.y * 32 + j;
        if (r < rows && c < cols) tile[j][threadIdx.x] = src[base + (size_t)r * cols + c];
    }
    __syncthreads();
    int r2 = blockIdx.y * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        int c2 = blockIdx.x * 32 + j;
        if (r2 < rows && c2 < cols) dst[base + (size_t)c2 * rows + r2] = tile[threadIdx.x][j];
    }
}

// ---- arrange_block_pixels_to_channel_dim / inverse (AGENT:853-873) ------------------------------
// blk[n][(bv*B+bh)*C + c][v][h] = img[n][c][v*B+bv][h*B+bh]
template <bool TO_DEPTH>
__global__ void space_depth_kernel(const float *__restrict__ src, float *__restrict__ dst, int n, int C, int Hb, int Wb,
                                   int B) {
    const size_t total = (size_t)n * C * Hb * B * Wb * B;
    const int W = Wb * B, H = Hb * B;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        // i indexes the image tensor (n, C, H, W)
        int x = (int)(i % W);
        size_t t = i / W;
        int y = (int)(t % H);
        t /= H;
        int c = (int)(t % C);
        int b = (int)(t / C);
        int v = y / B, bv = y % B, h = x / B, bh = x % B;
        size_t j = (((size_t)b * (C * B * B) + (size_t)(bv * B + bh) * C + c) * Hb + v) * Wb + h;
        if (TO_DEPTH) dst[j] = src[i]; else dst[i] = src[j];
    }
}

// ---- 8-bit image <-> channel-last block tensors (eval_model's per-image body, AGENT:581-589 and 610-628) ---------
// The kernels are templated on where an image's pixels and blocks are:
//   U8Batch: n images of one size, block rows [v0, v1) of each, so that the host wrappers can convert band by band
//            while the rest of the batch is still in flight over PCIe; image b's planes at b * 3HW, its blocks from
//            b * Hb * Wb in x_cl and zhat_cl;
//   U8Mixed: the whole images of a mixed-size call (a host list, MixedSpan), their planes at the packed byte offsets
//            (MixedPix), x_cl in packed block order and zhat_cl in schedule order (MixedGeo).
// Both number their work items image after image: begin_*() gives the count (and fixes what one geometry shares across
// images), at(i) resolves item i to its image and the item within that image's part.
struct U8Img {
    int b, H, W;       // image, pixel size
    int Wp, W4;        // padded width (to x_cl), quads of output pixels per row (to u8)
    bool vec;          // (to u8) rows of whole 4-byte words
    size_t q;          // work item within the image's part of the band
    long long off;     // (mixed) byte offset of the image's planes
    int P, Wb;         // (mixed) first packed block and block columns of the image
};
struct U8Batch {
    int n, H, W, Hb, Wb, B, v0, v1;
    size_t per_img;
    int Wp, W4;
    bool vec;
    __device__ size_t begin_xcl() {
        Wp = Wb * B;
        per_img = (size_t)(v1 - v0) * B * Wp;
        return (size_t)n * per_img;
    }
    __device__ size_t begin_u8() {
        const int y0 = v0 * B, y1 = (v1 * B < H) ? v1 * B : H;
        if (y1 <= y0) return 0;
        W4 = (W + 3) >> 2;
        per_img = (size_t)(y1 - y0) * W4;
        vec = (W & 3) == 0 && (B & 3) == 0;
        return (size_t)n * per_img;
    }
    __device__ U8Img at(size_t i) const {
        U8Img p;
        p.b = (int)(i / per_img);
        p.q = i - (size_t)p.b * per_img;
        p.H = H; p.W = W; p.Wp = Wp; p.W4 = W4; p.vec = vec;
        return p;
    }
    __device__ size_t plane(const U8Img &p, int c, int y) const { return (((size_t)p.b * 3 + c) * H + y) * W; }
    __device__ size_t x_block(const U8Img &p, int v, int h) const { return ((size_t)p.b * Hb + v) * Wb + h; }
    __device__ size_t z_block(const U8Img &p, int v, int h) const { return ((size_t)p.b * Hb + v) * Wb + h; }
};
struct U8Mixed {
    MixedGeo g;
    const MixedPix *__restrict__ pix;
    const MixedSpan *__restrict__ span;
    int n_span, B, v0;
    long long n_items;
    __device__ size_t begin_xcl() const { return (size_t)n_items; }
    __device__ size_t begin_u8() const { return (size_t)n_items; }
    __device__ U8Img at(size_t i) const {
        int lo = 0, hi = n_span - 1;   // the last image whose first item is <= i
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if ((size_t)span[mid].item0 <= i) lo = mid; else hi = mid - 1;
        }
        const MixedSpan s = span[lo];
        const MixedPix px = pix[s.img];
        const int4 gi = g.img[s.img];
        U8Img p;
        p.b = s.img; p.q = i - (size_t)s.item0;
        p.H = px.H; p.W = px.W;
        p.Wp = gi.y * B; p.W4 = (px.W + 3) >> 2;
        // whole 4-byte words only where the image's planes start on one: packed offsets are 3 * sum H_j W_j
        p.vec = (px.W & 3) == 0 && (B & 3) == 0 && (px.off & 3) == 0;
        p.off = px.off; p.P = gi.z; p.Wb = gi.y;
        return p;
    }
    __device__ size_t plane(const U8Img &p, int c, int y) const { return (size_t)p.off + ((size_t)c * p.H + y) * p.W; }
    __device__ size_t x_block(const U8Img &p, int v, int h) const { return (size_t)p.P + v * p.Wb + h; }
    __device__ size_t z_block(const U8Img &p, int v, int h) const { return (size_t)g.sched[p.P + v * p.Wb + h]; }
};

//   x_cl[(img, v, h)][(bv*B + bh)*3 + c] = img[c][min(v*B+bv, H-1)][min(h*B+bh, W-1)] / 255 - 0.5
// = ToTensor() (u8 / 255 in fp32), `x - 0.5` (AGENT:581), replicate padding to a multiple of B (AGENT:583-586) and
// arrange_block_pixels_to_channel_dim (AGENT:853-860) in one pass.  One thread per padded pixel, bh fastest.
template <class Geo>
__global__ void u8_to_xcl_kernel(const uint8_t *__restrict__ img, float *__restrict__ x_cl, Geo g) {
    const int B = g.B, v0 = g.v0;
    const size_t total = g.begin_xcl();
    const int Cin = 3 * B * B;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const U8Img p = g.at(i);
        const int yy = (int)(p.q / p.Wp), x = (int)(p.q - (size_t)yy * p.Wp);
        const int y = v0 * B + yy;
        const int v = y / B, bv = y - v * B, h = x / B, bh = x - h * B;
        const int ys = y < p.H ? y : p.H - 1, xs = x < p.W ? x : p.W - 1;
        const uint8_t *src = img + g.plane(p, 0, ys) + xs;
        float *dst = x_cl + g.x_block(p, v, h) * Cin + (bv * B + bh) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c)
            dst[c] = __fsub_rn(__fdiv_rn((float)src[(size_t)c * p.H * p.W], 255.0f), 0.5f);
    }
}

// out[c][y][x] = uint8(clamp((z + 0.5) * 255 + 0.5, 0, 255)) for y < H, x < W: arrange_channel_dim_to_block_pixels
// (AGENT:863-873), the crop of the padding, `+ 0.5` (AGENT:628) and torchvision's save_image quantisation
// (mul(255).add_(0.5).clamp_(0, 255).to(uint8)) in one pass.  One thread per 4 horizontally adjacent pixels.
template <class Geo>
__global__ void zcl_to_u8_kernel(const float *__restrict__ z_cl, uint8_t *__restrict__ out, Geo g) {
    const int B = g.B, v0 = g.v0;
    const size_t total = g.begin_u8();
    if (total == 0) return;
    const int y0 = v0 * B;
    const int Cin = 3 * B * B;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const U8Img p = g.at(i);
        const int W = p.W, W4 = p.W4;
        const int yy = (int)(p.q / W4), x4 = (int)(p.q - (size_t)yy * W4) << 2;
        const int y = y0 + yy, v = y / B, bv = y - v * B;
        uint8_t px[3][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int x = x4 + j < W ? x4 + j : W - 1;
            const int h = x / B, bh = x - h * B;
            const float *src = z_cl + g.z_block(p, v, h) * Cin + (bv * B + bh) * 3;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float t = __fadd_rn(__fmul_rn(__fadd_rn(src[c], 0.5f), 255.0f), 0.5f);
                t = fminf(fmaxf(t, 0.0f), 255.0f);
                px[c][j] = (uint8_t)t;
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            uint8_t *dst = out + g.plane(p, c, y) + x4;
            if (p.vec) {
                *reinterpret_cast<uchar4 *>(dst) = make_uchar4(px[c][0], px[c][1], px[c][2], px[c][3]);
            } else {
                for (int j = 0; j < 4 && x4 + j < W; ++j) dst[j] = px[c][j];
            }
        }
    }
}

// (n, C, Hb, Wb) fp32 -> channel-last, block rows [v0, v1) only (band-wise form of transpose_kernel for the host calls)
__global__ void nchw_to_cl_band_kernel(const float *__restrict__ src, float *__restrict__ dst, int C, int Hb, int Wb,
                                       int v0, int v1) {
    __shared__ float tile[32][33];
    const int HW = Hb * Wb, p0 = v0 * Wb, np = (v1 - v0) * Wb;
    const size_t base = (size_t)blockIdx.z * C * HW;
    const int p = blockIdx.x * 32 + threadIdx.x;         // position within the band
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = blockIdx.y * 32 + j;
        if (c < C && p < np) tile[j][threadIdx.x] = src[base + (size_t)c * HW + p0 + p];
    }
    __syncthreads();
    const int c2 = blockIdx.y * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int p2 = blockIdx.x * 32 + j;
        if (c2 < C && p2 < np) dst[base + (size_t)(p0 + p2) * C + c2] = tile[threadIdx.x][j];
    }
}

__global__ void cl_to_nchw_band_kernel(const float *__restrict__ src, float *__restrict__ dst, int C, int Hb, int Wb,
                                       int v0, int v1) {
    __shared__ float tile[32][33];
    const int HW = Hb * Wb, p0 = v0 * Wb, np = (v1 - v0) * Wb;
    const size_t base = (size_t)blockIdx.z * C * HW;
    const int c = blockIdx.x * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int p = blockIdx.y * 32 + j;
        if (c < C && p < np) tile[j][threadIdx.x] = src[base + (size_t)(p0 + p) * C + c];
    }
    __syncthreads();
    const int p2 = blockIdx.y * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c2 = blockIdx.x * 32 + j;
        if (c2 < C && p2 < np) dst[base + (size_t)c2 * HW + p0 + p2] = tile[threadIdx.x][j];
    }
}

__global__ void split_kernel(const float *__restrict__ src, h16 *__restrict__ hi, h16 *__restrict__ lo, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        h16 h, l;
        split_h16(src[i], h, l);
        hi[i] = h;
        lo[i] = l;
    }
}

// ---- per-step gathers -----------------------------------------------------------------------------
// Row sources: row_at(s, r) resolves row r of a step once; the row then answers where its x block is, where its zhat
// neighbour (dv, dh) is (false: outside the image) and which row of the g0 store its tap (dv, dh) reads.
//   StepDesc: one geometry, the closed form (x_cl and zhat_cl by block, the g0 store by ring position, g0_pos_index).
//   MixedRows: the R row records of a mixed-size step (schedule rows, or the ring-extended rows of E0, which have no x
//   block); x_cl is in packed block order, zhat_cl and the g0 store in schedule order, the borders those of the row's
//   own image.
struct StepRow {
    int img, v, h, Hb, Wb;
    __device__ size_t x_block() const { return ((size_t)img * Hb + v) * Wb + h; }
    __device__ bool zhat_block(int dv, int dh, size_t &b) const {
        const int vv = v + dv, hh = h + dh;
        if (!(vv >= 0 && vv < Hb && hh >= 0 && hh < Wb)) return false;
        b = ((size_t)img * Hb + vv) * Wb + hh;
        return true;
    }
    __device__ size_t g0_row(int dv, int dh) const { return g0_pos_index(img, v + dv, h + dh, Hb, Wb); }
};
__device__ __forceinline__ StepRow row_at(const StepDesc &s, int r) {
    StepRow q;
    step_row_to_block(s, r, q.img, q.v, q.h);
    q.Hb = s.Hb; q.Wb = s.Wb;
    return q;
}

struct MixedRows {
    MixedGeo g;
    const int4 *__restrict__ rows;
};
struct MixedRow {
    int4 rec, gi;   // {img, v, h, packed block}, the image's {Hb, Wb, P, G}
    const int *sched, *g0row;
    __device__ size_t x_block() const { return (size_t)rec.w; }
    __device__ bool zhat_block(int dv, int dh, size_t &b) const {
        const int vv = rec.y + dv, hh = rec.z + dh;
        if (!(vv >= 0 && vv < gi.x && hh >= 0 && hh < gi.y)) return false;
        b = (size_t)sched[gi.z + vv * gi.y + hh];
        return true;
    }
    __device__ size_t g0_row(int dv, int dh) const {
        return (size_t)g0row[gi.w + (rec.y + dv + 1) * (gi.y + 2) + (rec.z + dh + 1)];
    }
};
__device__ __forceinline__ MixedRow row_at(const MixedRows &s, int r) {
    MixedRow q;
    q.rec = s.rows[r];
    q.gi = s.g.img[q.rec.x];
    q.sched = s.g.sched; q.g0row = s.g.g0row;
    return q;
}

// Row r of the step.  X[r, :] = x(v,h); T[r, tap*Cin + c] = zhat(v+dv, h+dh)[c] for the four live taps of a 3x3
// mask-'A' kernel, (dv,dh) = (-1,-1), (-1,0), (-1,+1), (0,-1) (masked_conv2d.py:12-17), zero outside the image
// (NET:349).
template <class Rows>
__global__ void gather_kernel(const float *__restrict__ x_cl, const float *__restrict__ zhat_cl, int Cin, Rows s,
                              int R, h16 *__restrict__ X_hi, h16 *__restrict__ X_lo, int ldX,
                              h16 *__restrict__ T_hi, h16 *__restrict__ T_lo, int ldT) {
    const int r = blockIdx.x;
    if (r >= R) return;
    const auto q = row_at(s, r);
    const int c4n = Cin >> 2;
    const int first = X_hi ? 0 : 1;
    for (int e = threadIdx.x + first * c4n; e < 5 * c4n; e += blockDim.x) {
        const int seg = e / c4n, c = (e - seg * c4n) << 2;
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        h16 *ph, *pl;
        if (seg == 0) {
            val = *reinterpret_cast<const float4 *>(x_cl + q.x_block() * Cin + c);
            ph = X_hi + (size_t)r * ldX + c;
            pl = X_lo + (size_t)r * ldX + c;
        } else {
            const int tap = seg - 1;
            const int dv = (tap == 3) ? 0 : -1;
            const int dh = (tap == 3) ? -1 : tap - 1;
            size_t b;
            if (q.zhat_block(dv, dh, b)) val = *reinterpret_cast<const float4 *>(zhat_cl + b * Cin + c);
            ph = T_hi + (size_t)r * ldT + tap * Cin + c;
            pl = T_lo + (size_t)r * ldT + tap * Cin + c;
        }
        const float f[4] = {val.x, val.y, val.z, val.w};
        store_hilo<4>(ph, pl, f);
    }
}

// KS[1] == 3: out[r, tap*E1 + c] = g0(v+dv, h+dh)[c] for the five live taps of a 3x3 mask-'B' kernel,
// (dv,dh) = (-1,-1), (-1,0), (-1,+1), (0,-1), (0,0); every such position lies inside the ring-extended store.
template <class Rows>
__global__ void gather5_kernel(const h16 *__restrict__ g_hi, const h16 *__restrict__ g_lo, int E1, Rows s, int R,
                               h16 *__restrict__ o_hi, h16 *__restrict__ o_lo, int ld) {
    const int r = blockIdx.x;
    if (r >= R) return;
    const auto q = row_at(s, r);
    const int c8n = E1 >> 3;   // 16-byte chunks per plane row
    for (int e = threadIdx.x; e < 5 * c8n; e += blockDim.x) {
        const int tap = e / c8n, c = (e - tap * c8n) << 3;
        const int dv = (tap >= 3) ? 0 : -1;
        const int dh = (tap >= 3) ? tap - 4 : tap - 1;
        const size_t src = q.g0_row(dv, dh) * E1 + c;
        const size_t dst = (size_t)r * ld + (size_t)tap * E1 + c;
        *reinterpret_cast<uint4 *>(o_hi + dst) = *reinterpret_cast<const uint4 *>(g_hi + src);
        *reinterpret_cast<uint4 *>(o_lo + dst) = *reinterpret_cast<const uint4 *>(g_lo + src);
    }
}

// Post-processing net (NET:462-463: nn.Conv2d(C1, 4 C1, 3, padding=0), no mask): out[r, tap*Cin + c] = z(v+dv, h+dh)[c]
// for all nine taps (dv, dh) in raster order of the kernel, zero outside the image (only interior blocks keep the
// result, NET:476 pads the residual back with zeros).
__global__ void gather9_kernel(const float *__restrict__ z_cl, int Cin, StepDesc s, int R, h16 *__restrict__ o_hi,
                               h16 *__restrict__ o_lo, int ld) {
    const int r = blockIdx.x;
    if (r >= R) return;
    int img, v, h;
    step_row_to_block(s, r, img, v, h);
    const int c4n = Cin >> 2;
    for (int e = threadIdx.x; e < 9 * c4n; e += blockDim.x) {
        const int tap = e / c4n, c = (e - tap * c4n) << 2;
        const int vv = v + tap / 3 - 1, hh = h + tap % 3 - 1;
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        if (vv >= 0 && vv < s.Hb && hh >= 0 && hh < s.Wb)
            val = *reinterpret_cast<const float4 *>(z_cl + (((size_t)img * s.Hb + vv) * s.Wb + hh) * Cin + c);
        const float f[4] = {val.x, val.y, val.z, val.w};
        store_hilo<4>(o_hi + (size_t)r * ld + (size_t)tap * Cin + c, o_lo + (size_t)r * ld + (size_t)tap * Cin + c, f);
    }
}

// blocks on the image border: the zero-padded residual leaves them unchanged (NET:476)
__global__ void restore_border_kernel(const float *__restrict__ z_cl, float *__restrict__ out_cl, int Cin, int n_img, int Hb,
                                      int Wb) {
    const int per = 2 * Wb + 2 * (Hb > 2 ? Hb - 2 : 0);        // border blocks of one image (Hb, Wb >= 1)
    const int b = blockIdx.x;
    const int img = b / per, q = b - img * per;
    int v, h;
    if (q < Wb) { v = 0; h = q; }
    else if (q < 2 * Wb) { v = Hb - 1; h = q - Wb; }
    else { const int k = q - 2 * Wb; v = 1 + (k >> 1); h = (k & 1) ? Wb - 1 : 0; }
    if (v >= Hb) return;
    const size_t o = (((size_t)img * Hb + v) * Wb + h) * Cin;
    for (int c = threadIdx.x; c < Cin; c += blockDim.x) out_cl[o + c] = z_cl[o + c];
}

// KS[1] == 3: row v = -1 of the hidden map sees only zero padding, so g0(-1, h) = lrelu(0 + b_e0) for every h --
// bit-identical to what the E0 GEMM epilogue produces from an all-zero accumulator.
__global__ void fill_g0_top_kernel(const float *__restrict__ bias, int E1, int n_img, int Hb, int Wb,
                                   h16 *__restrict__ g_hi, h16 *__restrict__ g_lo) {
    const int pos = blockIdx.x;                 // img * (Wb+2) + (h+1)
    const int img = pos / (Wb + 2), hp = pos - img * (Wb + 2);
    const size_t row = g0_pos_index(img, -1, hp - 1, Hb, Wb);
    for (int c = threadIdx.x; c < E1; c += blockDim.x) {
        float v = 0.0f + bias[c];
        v = v > 0.0f ? v : v * 0.01f;
        h16 h, l;
        split_h16(v, h, l);
        g_hi[row * E1 + c] = h;
        g_lo[row * E1 + c] = l;
    }
}

// ---- mixed-size batches (MixedGeo): x_cl is in packed block order, zhat_cl in schedule order ------------------------
// Packed NCHW (image i at C * P_i, (C, Hb_i, Wb_i) within) <-> channel-last rows, 32 blocks x 32 channels per tile.
// TO_CL: row = packed block; otherwise row = the block's schedule row.
template <bool TO_CL>
__global__ void nchw_cl_mixed_kernel(const float *__restrict__ src, float *__restrict__ dst, int C, MixedGeo g, int nblk) {
    __shared__ float tile[32][33];
    const int b0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int b = b0 + threadIdx.x;
    size_t pl = 0, hw = 0;   // this thread's block: offset in its image's NCHW planes, plane size
    size_t row = 0;
    if (b < nblk) {
        const int4 gi = g.img[g.blk_img[b]];
        hw = (size_t)gi.x * gi.y;
        pl = (size_t)C * gi.z + (size_t)(b - gi.z);
        row = TO_CL ? (size_t)b : (size_t)g.sched[b];
    }
    if (TO_CL) {
        for (int j = threadIdx.y; j < 32; j += 8)
            if (b < nblk && c0 + j < C) tile[j][threadIdx.x] = src[pl + (size_t)(c0 + j) * hw];
        __syncthreads();
        const int c = c0 + threadIdx.x;
        for (int j = threadIdx.y; j < 32; j += 8)
            if (b0 + j < nblk && c < C) dst[(size_t)(b0 + j) * C + c] = tile[threadIdx.x][j];
    } else {
        __shared__ size_t srow[32];
        if (threadIdx.y == 0) srow[threadIdx.x] = row;
        __syncthreads();
        const int c = c0 + threadIdx.x;
        for (int j = threadIdx.y; j < 32; j += 8)
            if (b0 + j < nblk && c < C) tile[j][threadIdx.x] = src[srow[j] * C + c];
        __syncthreads();
        for (int j = threadIdx.y; j < 32; j += 8)
            if (b < nblk && c0 + j < C) dst[pl + (size_t)(c0 + j) * hw] = tile[threadIdx.x][j];
    }
}

// dst[b * C + c] = src[sched[b] * C + c]: a schedule-ordered (block, C) array in packed block order
template <class T>
__global__ void unschedule_kernel(const T *__restrict__ src, T *__restrict__ dst, int C, MixedGeo g, int nblk) {
    const size_t total = (size_t)nblk * C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / C), c = (int)(i - (size_t)b * C);
        dst[i] = src[(size_t)g.sched[b] * C + c];
    }
}

// ---- weight packing -------------------------------------------------------------------------------
struct TapList {
    int n;
    int kh[9], kw[9];      // up to a full 3x3 kernel (post-processing net); the masked convs use 1, 4 or 5
};

// weff[co][t*cin + ci] = w[co][ci][kh_t][kw_t] * mask[co][ci][kh_t][kw_t]      (NET:381 weight * mask)
__global__ void pack_conv_kernel(const float *__restrict__ w, const float *__restrict__ mask, int cout, int cin, int KH,
                                 int KW, TapList taps, float *__restrict__ weff, int ld) {
    const size_t total = (size_t)cout * taps.n * cin;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ci = (int)(i % cin);
        const int t = (int)((i / cin) % taps.n);
        const int co = (int)(i / ((size_t)cin * taps.n));
        const size_t src = (((size_t)co * cin + ci) * KH + taps.kh[t]) * KW + taps.kw[t];
        weff[(size_t)co * ld + (size_t)t * cin + ci] = w[src] * (mask ? mask[src] : 1.0f);
    }
}

// NonNegativeParametrizer.forward: max(p, bound)^2 - pedestal   (utils/parametrizers.py:45-48)
__global__ void pack_gdn_kernel(const float *__restrict__ gamma, const float *__restrict__ beta, int C, float gbound,
                                float gped, float bbound, float bped, float *__restrict__ weff, int ld,
                                float *__restrict__ beta_out) {
    const size_t total = (size_t)C * C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int rI = (int)(i / C), cI = (int)(i % C);
        const float g = fmaxf(gamma[i], gbound);
        weff[(size_t)rI * ld + cI] = g * g - gped;
        if (i < (size_t)C) {
            const float b = fmaxf(beta[i], bbound);
            beta_out[i] = b * b - bped;
        }
    }
}

__global__ void absmax_kernel(const float *__restrict__ v, size_t n, float *__restrict__ out) {
    float m = 0.0f;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(v[i]));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int *>(out), __float_as_uint(m));   // m >= 0
}

__global__ void split_scaled_kernel(const float *__restrict__ src, h16 *__restrict__ hi, h16 *__restrict__ lo, size_t n,
                                    float scale) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        h16 h, l;
        split_h16(src[i] * scale, h, l);
        hi[i] = h;
        lo[i] = l;
    }
}

__global__ void add_vec_kernel(const float *a, const float *b, float *out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] + (b ? b[i] : 0.0f);
}

inline int grid_for(size_t total, int block) {
    size_t g = (total + block - 1) / block;
    if (g > 148 * 16) g = 148 * 16;   // grid-stride loops; a multiple of the SM count
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace

int launch_nchw_to_cl(const float *src, float *dst, int C, const CallImages &c, cudaStream_t st) {
    if (c.geo) {
        dim3 grid((unsigned)((c.nblk + 31) / 32), (C + 31) / 32), block(32, 8);
        nchw_cl_mixed_kernel<true><<<grid, block, 0, st>>>(src, dst, C, *c.geo, (int)c.nblk);
    } else {
        const int HW = c.Hb * c.Wb;
        dim3 grid((HW + 31) / 32, (C + 31) / 32, c.n_img), block(32, 8);
        transpose_kernel<<<grid, block, 0, st>>>(src, dst, C, HW);
    }
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_cl_to_nchw(const float *src, float *dst, int C, const CallImages &c, cudaStream_t st) {
    if (c.geo) {
        dim3 grid((unsigned)((c.nblk + 31) / 32), (C + 31) / 32), block(32, 8);
        nchw_cl_mixed_kernel<false><<<grid, block, 0, st>>>(src, dst, C, *c.geo, (int)c.nblk);
    } else {
        const int HW = c.Hb * c.Wb;
        dim3 grid((C + 31) / 32, (HW + 31) / 32, c.n_img), block(32, 8);
        transpose_kernel<<<grid, block, 0, st>>>(src, dst, HW, C);
    }
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

// (a mixed-size call converts its whole images: v0 = 0 in the kernels, the band arguments are not used)
int launch_u8_to_xcl(const uint8_t *img, float *x_cl, const CallImages &c, int B, int v0, int v1, cudaStream_t st) {
    if (c.geo) {
        const long long total = c.u8_items[0];
        if (c.n_img < 1 || total < 1) return 0;
        u8_to_xcl_kernel<<<grid_for((size_t)total, 256), 256, 0, st>>>(
            img, x_cl, U8Mixed{*c.geo, c.pix, c.span, c.n_img, B, 0, total});
    } else {
        if (v1 <= v0) return 0;
        const size_t total = (size_t)c.n_img * (v1 - v0) * B * c.Wb * B;
        u8_to_xcl_kernel<<<grid_for(total, 256), 256, 0, st>>>(img, x_cl,
                                                               U8Batch{c.n_img, c.H, c.W, c.Hb, c.Wb, B, v0, v1});
    }
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_zcl_to_u8(const float *z_cl, uint8_t *img, const CallImages &c, int B, int v0, int v1, cudaStream_t st) {
    if (c.geo) {
        const long long total = c.u8_items[1];
        if (c.n_img < 1 || total < 1) return 0;
        zcl_to_u8_kernel<<<grid_for((size_t)total, 256), 256, 0, st>>>(
            z_cl, img, U8Mixed{*c.geo, c.pix, c.span + c.n_img, c.n_img, B, 0, total});
    } else {
        if (v1 <= v0 || v0 * B >= c.H) return 0;
        const size_t total = (size_t)c.n_img * ((size_t)(v1 - v0) * B) * ((c.W + 3) / 4);
        zcl_to_u8_kernel<<<grid_for(total, 256), 256, 0, st>>>(z_cl, img,
                                                               U8Batch{c.n_img, c.H, c.W, c.Hb, c.Wb, B, v0, v1});
    }
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_nchw_to_cl_band(const float *src, float *dst, int n, int C, int Hb, int Wb, int v0, int v1, cudaStream_t st) {
    if (v1 <= v0) return 0;
    dim3 grid(((v1 - v0) * Wb + 31) / 32, (C + 31) / 32, n), block(32, 8);
    nchw_to_cl_band_kernel<<<grid, block, 0, st>>>(src, dst, C, Hb, Wb, v0, v1);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_cl_to_nchw_band(const float *src, float *dst, int n, int C, int Hb, int Wb, int v0, int v1, cudaStream_t st) {
    if (v1 <= v0) return 0;
    dim3 grid((C + 31) / 32, ((v1 - v0) * Wb + 31) / 32, n), block(32, 8);
    cl_to_nchw_band_kernel<<<grid, block, 0, st>>>(src, dst, C, Hb, Wb, v0, v1);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_space_to_depth(const float *img, float *blk, int n, int C, int Hb, int Wb, int B, cudaStream_t st) {
    const size_t total = (size_t)n * C * Hb * B * Wb * B;
    space_depth_kernel<true><<<grid_for(total, 256), 256, 0, st>>>(img, blk, n, C, Hb, Wb, B);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_depth_to_space(const float *blk, float *img, int n, int C, int Hb, int Wb, int B, cudaStream_t st) {
    const size_t total = (size_t)n * C * Hb * B * Wb * B;
    space_depth_kernel<false><<<grid_for(total, 256), 256, 0, st>>>(blk, img, n, C, Hb, Wb, B);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_split_f32(const float *src, h16 *hi, h16 *lo, int64_t n, cudaStream_t st) {
    split_kernel<<<grid_for((size_t)n, 256), 256, 0, st>>>(src, hi, lo, (size_t)n);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

// The gathers of a step: the closed form of s.sd, or (mixed-size step) the step's row records.
int launch_gather(const float *x_cl, const float *zhat_cl, int Cin, const StepRows &s, h16 *X_hi, h16 *X_lo, int ldX,
                  h16 *T_hi, h16 *T_lo, int ldT, cudaStream_t st) {
    if (s.R <= 0) return 0;
    int threads = 5 * (Cin / 4);
    threads = threads > 256 ? 256 : ((threads + 31) / 32) * 32;
    if (s.geo)
        gather_kernel<<<s.R, threads, 0, st>>>(x_cl, zhat_cl, Cin, MixedRows{*s.geo, s.rows}, s.R, X_hi, X_lo, ldX, T_hi,
                                               T_lo, ldT);
    else
        gather_kernel<<<s.R, threads, 0, st>>>(x_cl, zhat_cl, Cin, s.sd, s.R, X_hi, X_lo, ldX, T_hi, T_lo, ldT);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_gather5(const h16 *g0_hi, const h16 *g0_lo, int E1, const StepRows &s, h16 *out_hi, h16 *out_lo, int ld,
                   cudaStream_t st) {
    if (s.R <= 0) return 0;
    if (s.geo)
        gather5_kernel<<<s.R, 256, 0, st>>>(g0_hi, g0_lo, E1, MixedRows{*s.geo, s.rows}, s.R, out_hi, out_lo, ld);
    else
        gather5_kernel<<<s.R, 256, 0, st>>>(g0_hi, g0_lo, E1, s.sd, s.R, out_hi, out_lo, ld);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_gather9(const float *z_cl, int Cin, const StepRows &s, h16 *out_hi, h16 *out_lo, int ld, cudaStream_t st) {
    if (s.R <= 0) return 0;
    gather9_kernel<<<s.R, 256, 0, st>>>(z_cl, Cin, s.sd, s.R, out_hi, out_lo, ld);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_restore_border(const float *z_cl, float *out_cl, int Cin, int n_img, int Hb, int Wb, cudaStream_t st) {
    const int per = 2 * Wb + 2 * (Hb > 2 ? Hb - 2 : 0);
    restore_border_kernel<<<n_img * per, 128, 0, st>>>(z_cl, out_cl, Cin, n_img, Hb, Wb);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_fill_g0_top(const float *bias, int E1, int n_img, int Hb, int Wb, h16 *g_hi, h16 *g_lo, cudaStream_t st) {
    fill_g0_top_kernel<<<n_img * (Wb + 2), 256, 0, st>>>(bias, E1, n_img, Hb, Wb, g_hi, g_lo);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

template <class T>
int launch_packed_order(const T *src, T *dst, int C, const CallImages &c, cudaStream_t st) {
    if (!c.geo) {   // one geometry: the schedule order is the packed order
        LBIC_CUDA(cudaMemcpyAsync(dst, src, sizeof(T) * c.nblk * C, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    unschedule_kernel<T><<<grid_for(c.nblk * C, 256), 256, 0, st>>>(src, dst, C, *c.geo, (int)c.nblk);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}
template int launch_packed_order<int32_t>(const int32_t *, int32_t *, int, const CallImages &, cudaStream_t);
template int launch_packed_order<uint8_t>(const uint8_t *, uint8_t *, int, const CallImages &, cudaStream_t);

int launch_pack_conv(const float *w, const float *mask, int cout, int cin, int kh, int kw, const int *taps_host,
                     int ntaps, float *weff, int ld, cudaStream_t st) {
    if (ntaps < 1 || ntaps > 9) return lbic_fail(LBIC_ERR_INVALID, "pack_conv: %d taps", ntaps);
    TapList tl;
    tl.n = ntaps;
    for (int i = 0; i < ntaps; ++i) {
        tl.kh[i] = taps_host[2 * i];
        tl.kw[i] = taps_host[2 * i + 1];
    }
    const size_t total = (size_t)cout * ntaps * cin;
    pack_conv_kernel<<<grid_for(total, 256), 256, 0, st>>>(w, mask, cout, cin, kh, kw, tl, weff, ld);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_pack_gdn(const float *gamma, const float *beta, int C, float gbound, float gped, float bbound, float bped,
                    float *weff, int ld, float *beta_out, cudaStream_t st) {
    pack_gdn_kernel<<<grid_for((size_t)C * C, 256), 256, 0, st>>>(gamma, beta, C, gbound, gped, bbound, bped, weff, ld,
                                                                beta_out);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

// Saturation check of an fp16 operand plane (debug option LBIC_OPT_CHECK_SATURATION): the hi planes clip at +-65504
// instead of overflowing (epilogue.cuh: pack_hilo), silently; this counts the clipped elements of rows [0, R) x columns
// [0, C) of a plane with row stride ld.
__global__ void sat_scan_kernel(const h16 *__restrict__ hi, int R, int C, int ld, unsigned long long *__restrict__ count) {
    const long long n = (long long)R * C;
    unsigned int local = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / C), c = (int)(i - (long long)r * C);
        const unsigned short bits = __half_as_ushort(hi[(size_t)r * ld + c]);
        local += ((bits & 0x7FFFu) >= 0x7BFFu) ? 1u : 0u;           // |x| = 65504 (the clip value), inf or nan
    }
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, (unsigned long long)local);
}

int launch_sat_scan(const h16 *hi, int R, int C, int ld, unsigned long long *count, cudaStream_t st) {
    if (R <= 0 || C <= 0) return 0;
    const long long n = (long long)R * C;
    const int blocks = (int)((n + 1023) / 1024 < 1184 ? (n + 1023) / 1024 : 1184);
    sat_scan_kernel<<<blocks, 256, 0, st>>>(hi, R, C, ld, count);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_absmax(const float *v, int64_t n, float *out_dev, cudaStream_t st) {
    absmax_kernel<<<grid_for((size_t)n, 256), 256, 0, st>>>(v, (size_t)n, out_dev);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_split_scaled(const float *src, h16 *hi, h16 *lo, int64_t n, float scale, cudaStream_t st) {
    split_scaled_kernel<<<grid_for((size_t)n, 256), 256, 0, st>>>(src, hi, lo, (size_t)n, scale);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_add_vec(const float *a, const float *b, float *out, int n, cudaStream_t st) {
    add_vec_kernel<<<(n + 255) / 256, 256, 0, st>>>(a, b, out, n);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

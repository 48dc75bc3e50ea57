// K5 / K6: rANS64 entropy coder on the GPU.
//
// Bit-compatible with the coder the reference binds from CompressAI (compressai.ans:
// BufferedRansEncoder.encode_with_indexes + flush, RansDecoder.set_stream + decode_stream; call sites
// graphs/models/BlockBasedImgCompLossy_net.py:328,359-360,409-410,439): one 64-bit state per stream,
// RANS64_L = 2^31, 32-bit renormalisation words, 16-bit probabilities, 4-bit bypass escape for values outside
// the table.  A stream's bytes are  [state lo][state hi][renorm words in decode order].
//
// Lanes: the reference container is ONE stream per image (symbols in raster block order, channels inner), so
// its decode is serial in raster order.  The lane container (extension) holds one such stream per block row:
//   u32 'LBML' | u32 lanes | u32 len[lanes] | lane 0 bytes | lane 1 bytes | ...
// which lets the decoder follow the same slope-2 wavefront as the encoder.
#include "rans_device.cuh"

namespace {

constexpr uint32_t LANE_MAGIC = 0x4C4D424Cu;   // "LBML"

// Where the encoder finds the symbols of stream s: equal streams of n_sym symbols every `stride` elements (one
// geometry per call), or the segments [seg[s], seg[s+1]) of a mixed-size batch.
struct EqualSegs {
    long n_sym, stride;
    __device__ __forceinline__ size_t start(int s) const { return (size_t)s * stride; }
    __device__ __forceinline__ long count(int) const { return n_sym; }
};
struct MixedSegs {
    const int64_t *seg;
    __device__ __forceinline__ size_t start(int s) const { return (size_t)seg[s]; }
    __device__ __forceinline__ long count(int s) const { return (long)(seg[s + 1] - seg[s]); }
};
// The lanes of image img: `lanes` per image, or lane0[img] .. lane0[img+1] - 1 (mixed-size batch).
struct EqualLanes {
    int lanes;
    __device__ __forceinline__ size_t first(int img) const { return (size_t)img * lanes; }
    __device__ __forceinline__ int count(int) const { return lanes; }
    __device__ __forceinline__ int total(int n_img) const { return n_img * lanes; }
    __device__ __forceinline__ void lane_of(int i, int n_img, int &img, int &l) const { img = i / lanes; l = i - img * lanes; }
};
struct MixedLanes {
    const int *lane0;
    __device__ __forceinline__ size_t first(int img) const { return (size_t)lane0[img]; }
    __device__ __forceinline__ int count(int img) const { return lane0[img + 1] - lane0[img]; }
    __device__ __forceinline__ int total(int n_img) const { return lane0[n_img]; }
    __device__ __forceinline__ void lane_of(int i, int n_img, int &img, int &l) const {
        int lo = 0, hi = n_img - 1;                 // last image whose first lane is <= i
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (lane0[mid] <= i) lo = mid; else hi = mid - 1;
        }
        img = lo; l = i - lane0[lo];
    }
};

// ---------------------------------------------------------------------------------------------
// encoder: one thread per stream walks its symbols backwards (flush() pops the pushed symbols in
// reverse) and writes renormalisation words from the end of its scratch region towards the front.
// ---------------------------------------------------------------------------------------------
struct EncCursor {
    unsigned long long x;
    uint32_t *base;   // scratch region start
    long pos;         // next free slot + 1 (we write base[--pos])
    bool overflow;
};

__device__ __forceinline__ void enc_emit(EncCursor &c) {
    if (c.pos <= 0) { c.overflow = true; return; }
    c.base[--c.pos] = (uint32_t)c.x;
    c.x >>= 32;
}

// warp-uniform variant: every lane tracks the same cursor, lane 0 performs the store
__device__ __forceinline__ void enc_emit_w(EncCursor &c, int lane) {
    if (c.pos <= 0) { c.overflow = true; return; }
    --c.pos;
    if (lane == 0) c.base[c.pos] = (uint32_t)c.x;
    c.x >>= 32;
}

__device__ __forceinline__ void enc_put(EncCursor &c, uint32_t start, uint32_t range) {
    const unsigned long long x_max = ((RANS_L >> PREC) << 32) * (unsigned long long)range;
    if (c.x >= x_max) enc_emit(c);
    c.x = ((c.x / range) << PREC) + (c.x % range) + start;
}

__device__ __forceinline__ void enc_put_bits(EncCursor &c, uint32_t val) {
    const unsigned long long x_max = ((RANS_L >> PREC) << 32) * (unsigned long long)(1u << (PREC - BYPASS));
    if (c.x >= x_max) enc_emit(c);
    c.x = (c.x << BYPASS) | val;
}

// One warp per stream.  The state update is inherently serial, so the warp splits the work in two:
//   * in parallel, each lane prepares one of the next 32 symbols: table lookups (start, range), the escape
//     decision, and the exact reciprocal of `range` (Granlund-Montgomery / ryg_rans Rans64EncSymbolInit:
//     rcp = ceil(2^(63+s) / range), s = ceil(log2 range); floor(x / range) = mulhi64(x, rcp) >> (s - 1) for every
//     x < 2^63, which covers x < x_max = range << 47);
//   * then all lanes replay the 32 prepared symbols in order (records broadcast with shuffles, every lane holds the
//     same state, lane 0 writes the renormalisation words), so no memory latency or division sits on the serial chain.
template <class Segs>
__global__ void rans_encode_kernel(const int32_t *__restrict__ cdf, int cdf_stride, const int32_t *__restrict__ cdf_len,
                                   const int32_t *__restrict__ offs, const int32_t *__restrict__ sym,
                                   const uint8_t *__restrict__ idx, int n_streams, Segs seg,
                                   uint32_t *__restrict__ scratch, long scratch_words, uint32_t *__restrict__ start_word,
                                   uint32_t *__restrict__ n_words, int *__restrict__ err) {
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= n_streams) return;
    EncCursor c;
    c.x = RANS_L;
    c.base = scratch + (size_t)s * scratch_words;
    c.pos = scratch_words;
    c.overflow = false;
    const int32_t *ps = sym + seg.start(s);
    const uint8_t *pi = idx + seg.start(s);
    const long n_sym = seg.count(s);
    for (long top = n_sym; top > 0; top -= 32) {
        // lane j prepares symbol top-1-j (the coder walks the symbols backwards)
        const long k = top - 1 - lane;
        uint32_t sr = 0, raw = 0, flags = 0;       // sr = start | range << 16; flags: bit0 escape, bits 8.. rcp shift
        unsigned long long rcp = 0;
        if (k >= 0) {
            const int ci = pi[k];
            const int32_t *row = cdf + (size_t)ci * cdf_stride;
            const int max_value = __ldg(cdf_len + ci) - 2;
            int value = ps[k] - __ldg(offs + ci);
            if (value < 0) {
                raw = (uint32_t)(-2 * value - 1);
                value = max_value;
            } else if (value >= max_value) {
                raw = (uint32_t)(2 * (value - max_value));
                value = max_value;
            }
            const uint32_t start = (uint32_t)__ldg(row + value);
            const uint32_t range = (uint32_t)__ldg(row + value + 1) - start;
            sr = start | (range << 16);
            uint32_t shift = 0;
            while (range > (1u << shift)) ++shift;
            if (range >= 2) {
                // ((1 << (shift + 63)) + range - 1) / range as two 64-bit divides
                unsigned long long x0 = range - 1;
                const unsigned long long x1 = 1ull << (shift + 31);
                const unsigned long long t1 = x1 / range;
                x0 += (x1 % range) << 32;
                rcp = x0 / range + (t1 << 32);
            }
            flags = (value == max_value ? 1u : 0u) | (shift << 8);
        }
        const int cnt = top < 32 ? (int)top : 32;
        for (int j = 0; j < cnt; ++j) {
            const uint32_t b_sr = __shfl_sync(0xffffffffu, sr, j);
            const uint32_t b_fl = __shfl_sync(0xffffffffu, flags, j);
            const uint32_t r_lo = __shfl_sync(0xffffffffu, (uint32_t)rcp, j);
            const uint32_t r_hi = __shfl_sync(0xffffffffu, (uint32_t)(rcp >> 32), j);
            if (b_fl & 1u) {
                // escape: pushed order is main, count (15,15,...,rem), nibbles LSB first -> popped in reverse
                const uint32_t b_raw = __shfl_sync(0xffffffffu, raw, j);
                int nb = 0;
                while (nb < 8 && (b_raw >> (nb * BYPASS)) != 0) ++nb;
                for (int q = nb - 1; q >= 0; --q) {
                    const unsigned long long x_max = ((RANS_L >> PREC) << 32) * (unsigned long long)(1u << (PREC - BYPASS));
                    if (c.x >= x_max) enc_emit_w(c, lane);
                    c.x = (c.x << BYPASS) | ((b_raw >> (q * BYPASS)) & MAX_BYPASS);
                }
                const int qn = nb / MAX_BYPASS, rem = nb - qn * MAX_BYPASS;
                for (int q = 0; q <= qn; ++q) {
                    const unsigned long long x_max = ((RANS_L >> PREC) << 32) * (unsigned long long)(1u << (PREC - BYPASS));
                    if (c.x >= x_max) enc_emit_w(c, lane);
                    c.x = (c.x << BYPASS) | (uint32_t)(q == 0 ? rem : MAX_BYPASS);
                }
            }
            const uint32_t start = b_sr & 0xFFFFu, range = b_sr >> 16;
            const unsigned long long x_max = ((RANS_L >> PREC) << 32) * (unsigned long long)range;
            if (c.x >= x_max) enc_emit_w(c, lane);
            unsigned long long q;
            if (range >= 2) {
                const unsigned long long r64 = (unsigned long long)r_lo | ((unsigned long long)r_hi << 32);
                q = __umul64hi(c.x, r64) >> ((b_fl >> 8) - 1);
            } else {
                q = c.x;
            }
            c.x = (q << PREC) + (c.x - q * range) + start;
        }
    }
    // Rans64EncFlush: two words, low half first in memory
    if (c.pos < 2) c.overflow = true;
    if (lane == 0) {
        if (!c.overflow) {
            c.base[--c.pos] = (uint32_t)(c.x >> 32);
            c.base[--c.pos] = (uint32_t)(c.x);
        }
        if (c.overflow) {
            atomicExch(err, 1);
            start_word[s] = 0;
            n_words[s] = 0xFFFFFFFFu;
        } else {
            start_word[s] = (uint32_t)c.pos;
            n_words[s] = (uint32_t)(scratch_words - c.pos);
        }
    }
}

// ---- CTA-per-stream form of the encoder ----------------------------------------------------------------
// Few, long streams: the reference container of a single image is ONE stream of Hb*Wb*M symbols (589 824 for a
// 768x512 image), and its state update is a serial chain.  One CTA per stream splits the work by warp: warps 1..7
// prepare the next chunk of 1024 symbols in parallel (table lookups, escape decision, exact reciprocal of the range,
// exactly as the warp kernel above) into shared memory while lane 0 of warp 0 replays the previous chunk; the serial
// chain then consists of one 16-byte shared-memory load (independent of the state, so the unrolled loop keeps several
// in flight), a compare, a 64-bit mulhi and a few adds per symbol: ~25 ns instead of ~150 ns in the warp kernel,
// where every lane steps through the chain and the records travel by shuffles.  Same arithmetic, same words.
constexpr int ENC_B_THREADS = 256;
constexpr int ENC_B_CHUNK = 1024;

__global__ void __launch_bounds__(ENC_B_THREADS)
rans_encode_block_kernel(const int32_t *__restrict__ cdf, int cdf_stride, const int32_t *__restrict__ cdf_len,
                         const int32_t *__restrict__ offs, const int32_t *__restrict__ sym,
                         const uint8_t *__restrict__ idx, int n_streams, long n_sym, long stream_stride,
                         uint32_t *__restrict__ scratch, long scratch_words, uint32_t *__restrict__ start_word,
                         uint32_t *__restrict__ n_words, int *__restrict__ err) {
    __shared__ uint4 rec[2][ENC_B_CHUNK];        // start | range << 16, escape | shift << 8, rcp lo, rcp hi
    __shared__ uint32_t raws[2][ENC_B_CHUNK];    // raw value of an escaped symbol
    const int s = blockIdx.x;
    if (s >= n_streams) return;
    const int32_t *ps = sym + (size_t)s * stream_stride;
    const uint8_t *pi = idx + (size_t)s * stream_stride;
    const long nchunks = (n_sym + ENC_B_CHUNK - 1) / ENC_B_CHUNK;
    // element e of chunk c is symbol n_sym - 1 - (c * CHUNK + e): the coder walks the symbols backwards
    auto prepare = [&](long c, int buf, int first, int stride) {
        for (int e = first; e < ENC_B_CHUNK; e += stride) {
            const long k = n_sym - 1 - (c * ENC_B_CHUNK + e);
            if (k < 0) break;
            const int ci = pi[k];
            const int32_t *row = cdf + (size_t)ci * cdf_stride;
            const int max_value = __ldg(cdf_len + ci) - 2;
            int value = ps[k] - __ldg(offs + ci);
            uint32_t raw = 0;
            if (value < 0) {
                raw = (uint32_t)(-2 * value - 1);
                value = max_value;
            } else if (value >= max_value) {
                raw = (uint32_t)(2 * (value - max_value));
                value = max_value;
            }
            const uint32_t start = (uint32_t)__ldg(row + value);
            const uint32_t range = (uint32_t)__ldg(row + value + 1) - start;
            uint32_t shift = 0;
            while (range > (1u << shift)) ++shift;
            unsigned long long rcp = 0;
            if (range >= 2) {
                unsigned long long x0 = range - 1;
                const unsigned long long x1 = 1ull << (shift + 31);
                const unsigned long long t1 = x1 / range;
                x0 += (x1 % range) << 32;
                rcp = x0 / range + (t1 << 32);
            }
            rec[buf][e] = make_uint4(start | (range << 16), (value == max_value ? 1u : 0u) | (shift << 8), (uint32_t)rcp,
                                     (uint32_t)(rcp >> 32));
            raws[buf][e] = raw;
        }
    };
    prepare(0, 0, threadIdx.x, ENC_B_THREADS);
    __syncthreads();
    EncCursor c;
    c.x = RANS_L;
    c.base = scratch + (size_t)s * scratch_words;
    c.pos = scratch_words;
    c.overflow = false;
    for (long ch = 0; ch < nchunks; ++ch) {
        const int buf = (int)(ch & 1);
        if (threadIdx.x >= 32) {
            if (ch + 1 < nchunks) prepare(ch + 1, buf ^ 1, threadIdx.x - 32, ENC_B_THREADS - 32);
        } else if (threadIdx.x == 0) {
            const long left = n_sym - ch * ENC_B_CHUNK;
            const int cnt = left < ENC_B_CHUNK ? (int)left : ENC_B_CHUNK;
#pragma unroll 4
            for (int e = 0; e < cnt; ++e) {
                const uint4 r = rec[buf][e];
                if (r.y & 1u) {
                    // escape: pushed order is main, count (15,15,...,rem), nibbles LSB first -> popped in reverse
                    const uint32_t raw = raws[buf][e];
                    int nb = 0;
                    while (nb < 8 && (raw >> (nb * BYPASS)) != 0) ++nb;
                    for (int q = nb - 1; q >= 0; --q) enc_put_bits(c, (raw >> (q * BYPASS)) & MAX_BYPASS);
                    const int qn = nb / MAX_BYPASS, rem = nb - qn * MAX_BYPASS;
                    for (int q = 0; q <= qn; ++q) enc_put_bits(c, (uint32_t)(q == 0 ? rem : MAX_BYPASS));
                }
                const uint32_t start = r.x & 0xFFFFu, range = r.x >> 16;
                const unsigned long long x_max = ((RANS_L >> PREC) << 32) * (unsigned long long)range;
                if (c.x >= x_max) enc_emit(c);
                unsigned long long q;
                if (range >= 2) {
                    const unsigned long long r64 = (unsigned long long)r.z | ((unsigned long long)r.w << 32);
                    q = __umul64hi(c.x, r64) >> ((r.y >> 8) - 1);
                } else {
                    q = c.x;
                }
                c.x = (q << PREC) + (c.x - q * range) + start;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // Rans64EncFlush: two words, low half first in memory
        if (c.pos < 2) c.overflow = true;
        if (!c.overflow) {
            c.base[--c.pos] = (uint32_t)(c.x >> 32);
            c.base[--c.pos] = (uint32_t)(c.x);
            start_word[s] = (uint32_t)c.pos;
            n_words[s] = (uint32_t)(scratch_words - c.pos);
        } else {
            atomicExch(err, 1);
            start_word[s] = 0;
            n_words[s] = 0xFFFFFFFFu;
        }
    }
}

// ---- thread-per-stream form of the encoder --------------------------------------------------------
// A batch holds tens of thousands of independent streams (one per block row per image in the lane container), so
// one THREAD per stream keeps every lane busy where the warp kernel above replays its serial chain on 32 lanes.
// The table lookups hit the compact 16-bit rows in shared memory (Tables::cdf16); the division is the plain 64-bit
// one (its ~100 instructions are cheap next to a warp per stream).  Same arithmetic as enc_put / the warp kernel,
// hence the same words.
constexpr int ENC_T_THREADS = 128;

__device__ __forceinline__ void enc_symbol_thread(EncCursor &c, int symbol, int ci, const uint16_t *__restrict__ s_cdf,
                                                  const int *__restrict__ s_off, const int *__restrict__ s_len,
                                                  const int *__restrict__ s_offs) {
    const uint16_t *row = s_cdf + s_off[ci];
    const int len = s_len[ci];
    const int max_value = len - 2;
    int value = symbol - s_offs[ci];
    uint32_t raw = 0;
    if (value < 0) {
        raw = (uint32_t)(-2 * value - 1);
        value = max_value;
    } else if (value >= max_value) {
        raw = (uint32_t)(2 * (value - max_value));
        value = max_value;
    }
    const uint32_t start = row[value];
    const uint32_t range = ((value + 1 == len - 1) ? 65536u : (uint32_t)row[value + 1]) - start;
    if (value == max_value) {
        // escape: pushed order is main, count (15,15,...,rem), nibbles LSB first -> popped in reverse
        int nb = 0;
        while (nb < 8 && (raw >> (nb * BYPASS)) != 0) ++nb;
        for (int q = nb - 1; q >= 0; --q) enc_put_bits(c, (raw >> (q * BYPASS)) & MAX_BYPASS);
        const int qn = nb / MAX_BYPASS, rem = nb - qn * MAX_BYPASS;
        for (int q = 0; q <= qn; ++q) enc_put_bits(c, (uint32_t)(q == 0 ? rem : MAX_BYPASS));
    }
    enc_put(c, start, range);
}

template <class Segs>
__global__ void __launch_bounds__(ENC_T_THREADS)
rans_encode_thread_kernel(const uint16_t *__restrict__ cdf16, const int32_t *__restrict__ off16, int total,
                          const int32_t *__restrict__ cdf_len, const int32_t *__restrict__ offs,
                          const int32_t *__restrict__ sym, const uint8_t *__restrict__ idx, int n_streams, Segs seg, uint32_t *__restrict__ scratch, long scratch_words,
                          uint32_t *__restrict__ start_word, uint32_t *__restrict__ n_words, int *__restrict__ err) {
    extern __shared__ uint4 enc_smem[];
    const int nvec = (total + 7) >> 3;
    for (int i = threadIdx.x; i < nvec; i += blockDim.x) enc_smem[i] = reinterpret_cast<const uint4 *>(cdf16)[i];
    int *s_off = reinterpret_cast<int *>(enc_smem + nvec);
    int *s_len = s_off + 64, *s_offs = s_len + 64;
    if (threadIdx.x < 64) {
        s_off[threadIdx.x] = off16[threadIdx.x];
        s_len[threadIdx.x] = cdf_len[threadIdx.x];
        s_offs[threadIdx.x] = offs[threadIdx.x];
    }
    __syncthreads();
    const uint16_t *s_cdf = reinterpret_cast<const uint16_t *>(enc_smem);
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    EncCursor c;
    c.x = RANS_L;
    c.base = scratch + (size_t)s * scratch_words;
    c.pos = scratch_words;
    c.overflow = false;
    const int32_t *ps = sym + seg.start(s);
    const uint8_t *pi = idx + seg.start(s);
    // the coder walks the symbols backwards, four at a time (stream lengths and starts are multiples of 4)
    for (long k = seg.count(s) - 4; k >= 0; k -= 4) {
        const int4 v = *reinterpret_cast<const int4 *>(ps + k);
        const uchar4 ci = *reinterpret_cast<const uchar4 *>(pi + k);
        enc_symbol_thread(c, v.w, ci.w, s_cdf, s_off, s_len, s_offs);
        enc_symbol_thread(c, v.z, ci.z, s_cdf, s_off, s_len, s_offs);
        enc_symbol_thread(c, v.y, ci.y, s_cdf, s_off, s_len, s_offs);
        enc_symbol_thread(c, v.x, ci.x, s_cdf, s_off, s_len, s_offs);
    }
    // Rans64EncFlush: two words, low half first in memory
    if (c.pos < 2) c.overflow = true;
    if (!c.overflow) {
        c.base[--c.pos] = (uint32_t)(c.x >> 32);
        c.base[--c.pos] = (uint32_t)(c.x);
        start_word[s] = (uint32_t)c.pos;
        n_words[s] = (uint32_t)(scratch_words - c.pos);
    } else {
        atomicExch(err, 1);
        start_word[s] = 0;
        n_words[s] = 0xFFFFFFFFu;
    }
}

// move each stream's words to the front of its output slot (coalesced, one CTA per stream)
__global__ void rans_compact_kernel(const uint32_t *__restrict__ scratch, long scratch_words,
                                    const uint32_t *__restrict__ start_word, const uint32_t *__restrict__ n_words,
                                    uint8_t *__restrict__ out, size_t out_stride, uint32_t *__restrict__ out_len,
                                    int *__restrict__ err) {
    const int s = blockIdx.x;
    const uint32_t nw = n_words[s];
    if (nw == 0xFFFFFFFFu || (size_t)nw * 4 > out_stride) {
        if (threadIdx.x == 0) { out_len[s] = 0xFFFFFFFFu; atomicExch(err, 1); }
        return;
    }
    const uint32_t *src = scratch + (size_t)s * scratch_words + start_word[s];
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + (size_t)s * out_stride);
    for (uint32_t i = threadIdx.x; i < nw; i += blockDim.x) dst[i] = src[i];
    if (threadIdx.x == 0) out_len[s] = nw * 4;
}

// lane container assembly: one CTA per image
template <class Lanes>
__global__ void lane_pack_kernel(const uint32_t *__restrict__ scratch, long scratch_words,
                                 const uint32_t *__restrict__ start_word, const uint32_t *__restrict__ n_words,
                                 Lanes lm, uint8_t *__restrict__ out, size_t out_stride, uint32_t *__restrict__ out_len,
                                 int *__restrict__ err) {
    extern __shared__ uint32_t lane_off[];   // lanes + 1 word offsets
    const int img = blockIdx.x;
    const int lanes = lm.count(img);
    __shared__ int bad;
    if (threadIdx.x == 0) {
        bad = 0;
        uint32_t run = 2 + (uint32_t)lanes;
        for (int l = 0; l < lanes; ++l) {
            lane_off[l] = run;
            const uint32_t nw = n_words[lm.first(img) + l];
            if (nw == 0xFFFFFFFFu) bad = 1; else run += nw;
        }
        lane_off[lanes] = run;
        if ((size_t)run * 4 > out_stride) bad = 1;
    }
    __syncthreads();
    if (bad) {
        if (threadIdx.x == 0) { out_len[img] = 0xFFFFFFFFu; atomicExch(err, 1); }
        return;
    }
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + (size_t)img * out_stride);
    if (threadIdx.x == 0) { dst[0] = LANE_MAGIC; dst[1] = (uint32_t)lanes; out_len[img] = lane_off[lanes] * 4; }
    for (int l = threadIdx.x; l < lanes; l += blockDim.x) dst[2 + l] = n_words[lm.first(img) + l] * 4;
    for (int l = 0; l < lanes; ++l) {
        const size_t s = lm.first(img) + l;
        const uint32_t *src = scratch + s * scratch_words + start_word[s];
        const uint32_t nw = n_words[s];
        for (uint32_t i = threadIdx.x; i < nw; i += blockDim.x) dst[lane_off[l] + i] = src[i];
    }
}

// Parses the per-image container(s) and initialises one decoder state per lane.
template <class Lanes>
__global__ void rans_dec_init_kernel(const uint8_t *__restrict__ streams, const uint32_t *__restrict__ stream_len,
                                     size_t stream_stride, int n_img, Lanes lm, int lanes_container,
                                     RansStreamState *__restrict__ states, const uint8_t **__restrict__ lane_ptr,
                                     int *__restrict__ err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= lm.total(n_img)) return;
    int img, l;
    lm.lane_of(i, n_img, img, l);
    const int lanes = lm.count(img);
    const uint8_t *base = streams + (size_t)img * stream_stride;
    const uint32_t total = stream_len[img];
    const uint8_t *p = base;
    uint32_t nbytes = total;
    // The container comes from the caller (possibly from an untrusted file): every length is checked in 64-bit
    // arithmetic against what is left of the image's slot, lane payloads must be whole 32-bit words, and a stream
    // may not be longer than its slot.  A rejected container decodes as an empty stream (all reads return zero).
    if ((size_t)total > stream_stride || (total & 3u)) {
        atomicExch(err, 2);
        nbytes = 0;
    } else if (lanes_container) {
        const uint32_t *hdr = reinterpret_cast<const uint32_t *>(base);
        const unsigned long long hdr_bytes = 8ull + 4ull * (unsigned long long)lanes;
        if ((unsigned long long)total < hdr_bytes || hdr[0] != LANE_MAGIC || hdr[1] != (uint32_t)lanes) {
            atomicExch(err, 2);
            nbytes = 0;
        } else {
            unsigned long long o = hdr_bytes;
            bool ok = true;
            for (int j = 0; j <= l && ok; ++j) {
                const uint32_t len_j = hdr[2 + j];
                ok = !(len_j & 3u) && (unsigned long long)len_j <= (unsigned long long)total - o;
                if (ok && j < l) o += len_j;
            }
            if (ok) {
                nbytes = hdr[2 + l];
                p = base + o;
            } else {
                atomicExch(err, 2);
                nbytes = 0;
            }
        }
    }
    RansStreamState st;
    st.nwords = nbytes / 4;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(p);
    const unsigned long long lo = st.nwords > 0 ? w[0] : 0u, hi = st.nwords > 1 ? w[1] : 0u;
    st.x = lo | (hi << 32);
    st.pos = 2;
    states[i] = st;
    lane_ptr[i] = p;
}

// The rows of a decode step: a StepDesc (one geometry; row r -> block (img, v, h), stream img * lanes + v with lanes,
// img without), or the schedule rows [row0, row0 + R) of a mixed-size batch with a stream per row.  row_at() resolves
// the row's stream, row_out() where its M symbols go in the (block, M) symbol array.
struct MixedDecRows {
    const int *stream;
    int row0;
};
struct DecRow {
    int img, v, h;
};
__device__ __forceinline__ int row_at(const StepDesc &sd, int lanes, int r, DecRow &q) {
    step_row_to_block(sd, r, q.img, q.v, q.h);
    return lanes > 1 ? q.img * lanes + q.v : q.img;
}
__device__ __forceinline__ size_t row_out(const StepDesc &sd, int, const DecRow &q, int M) {
    return (((size_t)q.img * sd.Hb + q.v) * sd.Wb + q.h) * M;
}
__device__ __forceinline__ int row_at(const MixedDecRows &mr, int, int r, DecRow &) { return mr.stream[r]; }
__device__ __forceinline__ size_t row_out(const MixedDecRows &mr, int r, const DecRow &, int M) {
    return (size_t)(mr.row0 + r) * M;
}

// One warp per row of the step: build_indexes from the predicted scales, decode M symbols from the row's
// lane, dequantise (sym + mean, ENT:159-168) and emit the decoder-net input as h16 hi/lo planes.
template <class Rows>
__global__ void rans_dec_step_kernel(const int32_t *__restrict__ cdf, int cdf_stride,
                                     const int32_t *__restrict__ cdf_len, const int32_t *__restrict__ offs,
                                     const float *__restrict__ scale_tab, RansStreamState *__restrict__ states,
                                     const uint8_t *const *__restrict__ lane_ptr, int lanes, Rows sd, int R, int M,
                                     const float *__restrict__ ksi, int ld_ksi, h16 *__restrict__ yq_hi,
                                     h16 *__restrict__ yq_lo, int ld_yq, int32_t *__restrict__ sym_out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= R) return;
    DecRow q;
    const int sidx = row_at(sd, lanes, warp, q);
    DecCursor d;
    {
        const RansStreamState st = states[sidx];
        d.x = st.x; d.pos = st.pos; d.nwords = st.nwords;
        d.words = reinterpret_cast<const uint32_t *>(lane_ptr[sidx]);
    }
    const float *krow = ksi + (size_t)warp * ld_ksi;
    int my_idx[8];
    int my_sym[8];
    const int per = (M + 31) >> 5;   // M <= 256
    for (int j = 0; j < per; ++j) {
        const int c = j * 32 + lane;
        my_idx[j] = c < M ? scale_to_index(krow[c], scale_tab) : 0;
        my_sym[j] = 0;
    }
    for (int c = 0; c < M; ++c) {
        const int ci = __shfl_sync(0xffffffffu, my_idx[c >> 5], c & 31);
        const int sym = dec_symbol_warp(d, cdf + (size_t)ci * cdf_stride, cdf_len[ci], offs[ci], lane);
        if (lane == (c & 31)) my_sym[c >> 5] = sym;
    }
    if (lane == 0) {
        RansStreamState st;
        st.x = d.x; st.pos = d.pos; st.nwords = d.nwords;
        states[sidx] = st;
    }
    const size_t o = row_out(sd, warp, q, M);
    for (int j = 0; j < per; ++j) {
        const int c = j * 32 + lane;
        if (c < M) {
            const float yq = (float)my_sym[j] + krow[M + c];
            h16 hi, lo;
            split_h16(yq, hi, lo);
            yq_hi[(size_t)warp * ld_yq + c] = hi;
            yq_lo[(size_t)warp * ld_yq + c] = lo;
            if (sym_out) sym_out[o + c] = my_sym[j];
        }
    }
}

// ---- warp-per-row decode step on shared-memory tables ---------------------------------------------------------
// The decode step of small batches (fewer rows than the thread-per-stream kernel wants): a block of eight warps
// copies the compact 16-bit CDF rows (Tables::cdf16, 54 KB for the reference's scale table) into shared memory once
// and each warp decodes one row with the lean decoder of rans_device.cuh -- ~3x faster per row than
// rans_dec_step_kernel, whose every symbol waits for two dependent L2 round trips (row lookups) and ~150 instructions.
constexpr int DEC_S_WARPS = 8;

template <class Rows>
__global__ void __launch_bounds__(DEC_S_WARPS * 32)
rans_dec_step_smem_kernel(const uint16_t *__restrict__ cdf16, const int32_t *__restrict__ off16, int total,
                          const int32_t *__restrict__ cdf_len, const int32_t *__restrict__ offs,
                          const float *__restrict__ scale_tab, RansStreamState *__restrict__ states,
                          const uint8_t *const *__restrict__ lane_ptr, int lanes, Rows sd, int R, int M,
                          const float *__restrict__ ksi, int ld_ksi, h16 *__restrict__ yq_hi, h16 *__restrict__ yq_lo,
                          int ld_yq, int32_t *__restrict__ sym_out) {
    extern __shared__ uint4 dsm[];
    const int nvec = (total + 7) >> 3;
    for (int i = threadIdx.x; i < nvec; i += blockDim.x) dsm[i] = reinterpret_cast<const uint4 *>(cdf16)[i];
    int *s_meta = reinterpret_cast<int *>(dsm + nvec);
    float *s_tab = reinterpret_cast<float *>(s_meta + 192);
    if (threadIdx.x < 64) {
        s_meta[threadIdx.x] = off16[threadIdx.x];
        s_meta[64 + threadIdx.x] = cdf_len[threadIdx.x];
        s_meta[128 + threadIdx.x] = offs[threadIdx.x];
        s_tab[threadIdx.x] = scale_tab[threadIdx.x];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * DEC_S_WARPS + warp;
    if (r >= R) return;
    const uint32_t s_cdf = (uint32_t)__cvta_generic_to_shared(dsm);
    const uint32_t s_met = s_cdf + 16u * (uint32_t)nvec;
    const uint32_t scr = s_met + 1024u + (uint32_t)warp * RANS_ROW_SCRATCH(M);
    DecRow q;
    const int sidx = row_at(sd, lanes, r, q);
    DecCursorW d;
    {
        const RansStreamState st = states[sidx];
        d.x = st.x; d.pos = st.pos; d.nwords = st.nwords;
        d.words = reinterpret_cast<const uint32_t *>(lane_ptr[sidx]);
    }
    dec_fill_w(d, lane);
    const float *krow = ksi + (size_t)r * ld_ksi;
    rans_decode_row_warp(d, s_cdf, s_met, scr, krow, s_tab, M, lane);
    if (lane == 0) {
        RansStreamState st;
        st.x = d.x; st.pos = d.pos; st.nwords = d.nwords;
        states[sidx] = st;
    }
    const size_t o = row_out(sd, r, q, M);
    for (int c = lane; c < M; c += 32) {
        const int sym = lds_s32(scr + 8u * M + 4u * c);
        h16 hi, lo;
        split_h16((float)sym + krow[M + c], hi, lo);
        yq_hi[(size_t)r * ld_yq + c] = hi;
        yq_lo[(size_t)r * ld_yq + c] = lo;
        if (sym_out) sym_out[o + c] = sym;
    }
}

// ---- thread-per-stream form of the decode step ---------------------------------------------------
// With hundreds of images in flight a step has tens of thousands of independent streams, so one THREAD per stream
// (instead of one warp) keeps every lane busy; what makes that affordable is that all probes of the CDF search hit
// shared memory: the CTA holds the compact 16-bit tables (Tables::cdf16, ~88 KiB for the reference's scale table)
// and each symbol costs one bucket lookup plus a bisection over the few entries of that bucket.  Same symbols as
// dec_symbol_warp by construction: both return (first k with cdf[k] > slot) - 1.
constexpr int DEC_T_THREADS = 256;

// Per-thread cursor with the next stream word already in a register: lanes of a warp need a new word at different
// symbols, and a load issued only when needed would stall the whole warp for a memory round trip at nearly every
// symbol.  The word is requested right after the previous one is consumed and is not needed for ~4 symbols.
struct DecCursorT {
    unsigned long long x;
    const uint32_t *words;
    uint32_t pos, nwords, w_next;
};
__device__ __forceinline__ uint32_t dec_word_t(DecCursorT &d) {
    const uint32_t w = d.w_next;
    d.pos++;
    d.w_next = d.pos < d.nwords ? __ldg(d.words + d.pos) : 0u;   // a corrupt stream stays finite
    return w;
}
__device__ __forceinline__ int dec_bits_t(DecCursorT &d) {
    const int val = (int)(d.x & MAX_BYPASS);
    d.x >>= BYPASS;
    if (d.x < RANS_L) d.x = (d.x << 32) | dec_word_t(d);
    return val;
}

__device__ __forceinline__ int dec_symbol_thread(DecCursorT &d, const uint16_t *__restrict__ row,
                                                 const uint16_t *__restrict__ lut, int len, int off) {
    const uint32_t cf = (uint32_t)(d.x & 0xFFFFu);
    const int max_value = len - 2;
    const uint32_t b = cf >> 8;
    int lo = lut[b], hi = lut[b + 1];           // first k with row[k] > 256 b  /  > 256 (b + 1)   (<= len - 1)
    while (lo < hi) {                            // mid < hi <= len - 1, so row[mid] is a stored (16-bit) entry
        const int mid = (lo + hi) >> 1;
        if ((uint32_t)row[mid] > cf) hi = mid; else lo = mid + 1;
    }
    const int s = lo - 1;
    const uint32_t start = row[s];
    const uint32_t next = (s + 1 == len - 1) ? 65536u : (uint32_t)row[s + 1];
    d.x = (unsigned long long)(next - start) * (d.x >> PREC) + cf - start;
    if (d.x < RANS_L) d.x = (d.x << 32) | dec_word_t(d);
    int value = s;
    if (value == max_value) {
        int val = dec_bits_t(d);
        int nb = val;
        while (val == MAX_BYPASS) {
            val = dec_bits_t(d);
            nb += val;
        }
        int raw = 0;
        for (int j = 0; j < nb; ++j) {
            val = dec_bits_t(d);
            raw |= val << (j * BYPASS);
        }
        value = raw >> 1;
        if (raw & 1) value = -value - 1; else value += max_value;
    }
    return value + off;
}

template <class Rows>
__global__ void __launch_bounds__(DEC_T_THREADS)
rans_dec_step_thread_kernel(const uint16_t *__restrict__ cdf16, const int32_t *__restrict__ off16, int total,
                            const int32_t *__restrict__ cdf_len, const int32_t *__restrict__ offs,
                            const float *__restrict__ scale_tab, RansStreamState *__restrict__ states,
                            const uint8_t *const *__restrict__ lane_ptr, int lanes, Rows sd, int R, int M,
                            const float *__restrict__ ksi, int ld_ksi, h16 *__restrict__ yq_hi,
                            h16 *__restrict__ yq_lo, int ld_yq, int32_t *__restrict__ sym_out) {
    extern __shared__ uint4 dec_smem[];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = r < R;
    // this thread's stream state and first operands are requested before the table copy so their latency overlaps it
    DecRow q = {0, 0, 0};
    int sidx = 0;
    DecCursorT d;
    d.x = 0; d.words = nullptr; d.pos = 0; d.nwords = 0; d.w_next = 0;
    const float *krow = ksi;
    float4 sc = make_float4(0.f, 0.f, 0.f, 0.f), mu = sc;
    if (active) {
        sidx = row_at(sd, lanes, r, q);
        const RansStreamState st = states[sidx];
        d.x = st.x; d.pos = st.pos; d.nwords = st.nwords;
        d.words = reinterpret_cast<const uint32_t *>(lane_ptr[sidx]);
        d.w_next = d.pos < d.nwords ? __ldg(d.words + d.pos) : 0u;
        krow = ksi + (size_t)r * ld_ksi;
        sc = *reinterpret_cast<const float4 *>(krow);
        mu = *reinterpret_cast<const float4 *>(krow + M);
    }
    const int nvec = (total + 64 * 257 + 7) >> 3;          // 16-byte units (the allocation is padded accordingly)
    for (int i = threadIdx.x; i < nvec; i += blockDim.x) dec_smem[i] = reinterpret_cast<const uint4 *>(cdf16)[i];
    int *s_off = reinterpret_cast<int *>(dec_smem + nvec);
    int *s_len = s_off + 64, *s_offs = s_len + 64;
    float *s_tab = reinterpret_cast<float *>(s_offs + 64);
    if (threadIdx.x < 64) {
        s_off[threadIdx.x] = off16[threadIdx.x];
        s_len[threadIdx.x] = cdf_len[threadIdx.x];
        s_offs[threadIdx.x] = offs[threadIdx.x];
        s_tab[threadIdx.x] = scale_tab[threadIdx.x];
    }
    __syncthreads();
    if (!active) return;
    const uint16_t *s_cdf = reinterpret_cast<const uint16_t *>(dec_smem);
    const uint16_t *s_lut = s_cdf + total;
    const size_t o = row_out(sd, r, q, M);
    const ScaleHint hint = scale_hint(s_tab);
    for (int c0 = 0; c0 < M; c0 += 4) {
        const float scs[4] = {sc.x, sc.y, sc.z, sc.w};
        const float mus[4] = {mu.x, mu.y, mu.z, mu.w};
        if (c0 + 4 < M) {                       // next four channels' entropy parameters, one iteration ahead
            sc = *reinterpret_cast<const float4 *>(krow + c0 + 4);
            mu = *reinterpret_cast<const float4 *>(krow + M + c0 + 4);
        }
        int sym[4];
        h16 hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float sj = fmaxf(scs[j], LBIC_SCALES_MIN);
            bool ok;
            int ci = scale_to_index_hinted(sj, s_tab, hint, &ok);
            if (!ok) ci = scale_to_index_bisect(sj, s_tab);
            sym[j] = dec_symbol_thread(d, s_cdf + s_off[ci], s_lut + ci * 257, s_len[ci], s_offs[ci]);
            split_h16((float)sym[j] + mus[j], hi[j], lo[j]);
        }
        uint2 uh, ul;
        uh.x = (uint32_t)__half_as_ushort(hi[0]) | ((uint32_t)__half_as_ushort(hi[1]) << 16);
        uh.y = (uint32_t)__half_as_ushort(hi[2]) | ((uint32_t)__half_as_ushort(hi[3]) << 16);
        ul.x = (uint32_t)__half_as_ushort(lo[0]) | ((uint32_t)__half_as_ushort(lo[1]) << 16);
        ul.y = (uint32_t)__half_as_ushort(lo[2]) | ((uint32_t)__half_as_ushort(lo[3]) << 16);
        *reinterpret_cast<uint2 *>(yq_hi + (size_t)r * ld_yq + c0) = uh;
        *reinterpret_cast<uint2 *>(yq_lo + (size_t)r * ld_yq + c0) = ul;
        if (sym_out) *reinterpret_cast<int4 *>(sym_out + o + c0) = make_int4(sym[0], sym[1], sym[2], sym[3]);
    }
    RansStreamState st;
    st.x = d.x; st.pos = d.pos; st.nwords = d.nwords;
    states[sidx] = st;
}

// Closed-loop validation without entropy coding (AGENT:491-549 validate_recu_reco_fast): the rate is estimated as
// -log2 of the Gaussian-conditional likelihood of each quantised latent (ENT:615-647, eval mode: values = |sym|,
// scales lower-bounded at 0.11, likelihood lower-bounded at 1e-9).  One thread per (row, channel) of the step.
__global__ void selfinfo_step_kernel(StepDesc sd, int R, int M, const float *__restrict__ ksi, int ld_ksi,
                                     const int32_t *__restrict__ sym, float *__restrict__ info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * M) return;
    const int r = i / M, c = i - r * M;
    int img, v, h;
    step_row_to_block(sd, r, img, v, h);
    const size_t o = (((size_t)img * sd.Hb + v) * sd.Wb + h) * M + c;
    const float s = fmaxf(ksi[(size_t)r * ld_ksi + c], LBIC_SCALES_MIN);
    const float val = fabsf((float)sym[o]);
    const float k = (float)(-0.70710678118654752440);
    const float upper = 0.5f * erfcf(k * ((0.5f - val) / s));
    const float lower = 0.5f * erfcf(k * ((-0.5f - val) / s));
    const float lik = fmaxf(upper - lower, 1e-9f);
    info[o] = -log2f(lik);
}

// Whole-stream decode with given indexes (lbic_rans_decode): one warp per stream.
__global__ void rans_decode_full_kernel(const int32_t *__restrict__ cdf, int cdf_stride,
                                        const int32_t *__restrict__ cdf_len, const int32_t *__restrict__ offs,
                                        const uint8_t *__restrict__ streams, const uint32_t *__restrict__ stream_len,
                                        size_t stream_stride, const uint8_t *__restrict__ idx, int n_streams, long n_sym,
                                        int32_t *__restrict__ sym_out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_streams) return;
    DecCursor d;
    d.words = reinterpret_cast<const uint32_t *>(streams + (size_t)warp * stream_stride);
    d.nwords = stream_len[warp] / 4;
    d.x = (unsigned long long)(d.nwords > 0 ? d.words[0] : 0u) | ((unsigned long long)(d.nwords > 1 ? d.words[1] : 0u) << 32);
    d.pos = 2;
    const uint8_t *pi = idx + (size_t)warp * n_sym;
    int32_t *po = sym_out + (size_t)warp * n_sym;
    for (long k = 0; k < n_sym; ++k) {
        const int ci = pi[k];
        const int sym = dec_symbol_warp(d, cdf + (size_t)ci * cdf_stride, cdf_len[ci], offs[ci], lane);
        if (lane == 0) po[k] = sym;
    }
}

}  // namespace

static int g_enc_thread_min_streams = 4096;
static int g_enc_block_max_streams = 592;     // up to 4 CTAs per SM: one CTA per stream; more (and short) streams: one warp each

// scratch layout: [n_streams * scratch_words] words, then start_word[n_streams], n_words[n_streams]
// (`aligned`: every stream starts and ends on a multiple of 4 symbols and the arrays are 16 / 4-byte aligned;
// `min_sym`: the shortest stream)
// (`block_form`: streams of block_n_sym symbols back to back may take the CTA-per-stream form)
// (`form`: 0 = by the policy below; 1 warp, 2 CTA, 3 thread per stream = that form, LBIC_ERR_INVALID if it does not apply)
template <class Segs>
int rans_encode_any(const Tables &T, const int32_t *sym, const uint8_t *idx, int n_streams, Segs seg, bool aligned,
                    int64_t min_sym, bool block_form, long block_n_sym, uint32_t *scratch, size_t scratch_words, uint8_t *out, size_t out_stride,
                    uint32_t *out_len, int *err_flag, cudaStream_t st, int form = 0) {
    if (!T.cdf) return lbic_fail(LBIC_ERR_STATE, "Uninitialized CDFs. Run update() first");
    uint32_t *start_word = scratch + (size_t)n_streams * scratch_words;
    uint32_t *n_words = start_word + n_streams;
    const bool thread_ok = T.cdf16_total > 0 && aligned && (reinterpret_cast<uintptr_t>(sym) & 15) == 0 &&
                           (reinterpret_cast<uintptr_t>(idx) & 3) == 0;
    if (form < 0 || form > 3 || (form == 3 && !thread_ok) || (form == 2 && !block_form))
        return lbic_fail(LBIC_ERR_INVALID, "rANS encoder form %d does not apply to these streams", form);
    // many streams: one thread per stream with the tables in shared memory; few (single images): one warp per stream
    if (form == 0)
        form = thread_ok && n_streams >= g_enc_thread_min_streams                          ? 3
               : block_form && n_streams <= g_enc_block_max_streams && min_sym >= 256 ? 2
                                                                                        : 1;
    if (form == 3) {
        const size_t smem = 16 * (((size_t)T.cdf16_total + 7) / 8) + 3 * 64 * 4;
        static unsigned long long attr_mask = 0;
        if (lbic_first_use_on_device(attr_mask))
            LBIC_CUDA(cudaFuncSetAttribute(rans_encode_thread_kernel<Segs>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        rans_encode_thread_kernel<Segs><<<(n_streams + ENC_T_THREADS - 1) / ENC_T_THREADS, ENC_T_THREADS, smem, st>>>(
            T.cdf16, T.cdf16_off, T.cdf16_total, T.cdf_length, T.offset, sym, idx, n_streams, seg, scratch,
            (long)scratch_words, start_word, n_words, err_flag);
    } else if (form == 2) {
        // few long streams (single images, the reference container): one CTA per stream, serial chain on one thread
        rans_encode_block_kernel<<<n_streams, ENC_B_THREADS, 0, st>>>(
            T.cdf, T.stride, T.cdf_length, T.offset, sym, idx, n_streams, block_n_sym, block_n_sym, scratch,
            (long)scratch_words, start_word, n_words, err_flag);
    } else {
        const int warps_per_block = 4;
        rans_encode_kernel<Segs><<<(n_streams + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(
            T.cdf, T.stride, T.cdf_length, T.offset, sym, idx, n_streams, seg, scratch, (long)scratch_words, start_word,
            n_words, err_flag);
    }
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    if (out) {
        rans_compact_kernel<<<n_streams, 256, 0, st>>>(scratch, (long)scratch_words, start_word, n_words, out,
                                                       out_stride, out_len, err_flag);
        count_launch(1);
        LBIC_CUDA(cudaGetLastError());
    }
    return 0;
}

int launch_rans_encode(const Tables &T, const int32_t *sym, const uint8_t *idx, const CallImages &c, uint32_t *scratch,
                       size_t scratch_words, uint8_t *out, size_t out_stride, uint32_t *out_len, int *err_flag,
                       cudaStream_t st) {
    // (mixed: every stream is a whole number of blocks of M symbols, M a multiple of 16; the streams differ in length,
    // so the CTA-per-stream form, which is for few long streams of one size, is not used)
    if (c.geo)
        return rans_encode_any(T, sym, idx, c.n_streams, MixedSegs{c.seg}, true, c.min_sym, false, 0L, scratch,
                               scratch_words, out, out_stride, out_len, err_flag, st);
    const long n_sym = (long)c.min_sym;
    return rans_encode_any(T, sym, idx, c.n_streams, EqualSegs{n_sym, n_sym}, n_sym % 4 == 0, n_sym, true, n_sym, scratch,
                           scratch_words, out, out_stride, out_len, err_flag, st);
}

int launch_rans_encode_form(const Tables &T, const int32_t *sym, const uint8_t *idx, int n_streams, const int64_t *seg,
                            const int64_t *seg_host, int form, uint32_t *scratch, size_t scratch_words, uint8_t *out,
                            size_t out_stride, uint32_t *out_len, int *err_flag, cudaStream_t st) {
    const int64_t n0 = seg_host[1] - seg_host[0];
    bool equal = seg_host[0] == 0, aligned = true;
    int64_t min_sym = n0;
    for (int s = 0; s < n_streams; ++s) {
        const int64_t n = seg_host[s + 1] - seg_host[s];
        equal = equal && n == n0;
        aligned = aligned && n % 4 == 0 && seg_host[s] % 4 == 0;
        min_sym = n < min_sym ? n : min_sym;
    }
    // equal streams back to back take the closed form, as an equal-size call codes them; any others the segment table
    if (equal)
        return rans_encode_any(T, sym, idx, n_streams, EqualSegs{(long)n0, (long)n0}, aligned, min_sym, true, (long)n0,
                               scratch, scratch_words, out, out_stride, out_len, err_flag, st, form);
    return rans_encode_any(T, sym, idx, n_streams, MixedSegs{seg}, aligned, min_sym, false, 0L, scratch, scratch_words, out,
                           out_stride, out_len, err_flag, st, form);
}

int launch_lane_pack(const uint32_t *scratch, size_t scratch_words, const CallImages &c, uint8_t *out, size_t out_stride,
                     uint32_t *out_len, int *err_flag, cudaStream_t st) {
    const uint32_t *start_word = scratch + (size_t)c.n_streams * scratch_words;
    const uint32_t *n_words = start_word + (size_t)c.n_streams;
    const size_t smem = sizeof(uint32_t) * (c.max_lanes + 1);
    if (c.geo)
        lane_pack_kernel<MixedLanes><<<c.n_img, 256, smem, st>>>(scratch, (long)scratch_words, start_word, n_words,
                                                                 MixedLanes{c.lane0}, out, out_stride, out_len, err_flag);
    else
        lane_pack_kernel<EqualLanes><<<c.n_img, 256, smem, st>>>(scratch, (long)scratch_words, start_word, n_words,
                                                                 EqualLanes{c.lanes}, out, out_stride, out_len, err_flag);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_rans_dec_init(const uint8_t *streams, const uint32_t *stream_len, size_t stream_stride, const CallImages &c,
                         RansStreamState *states, const uint8_t **lane_ptr, int *err_flag, cudaStream_t st) {
    const int grid = (c.n_streams + 127) / 128, container = c.lane_container ? 1 : 0;
    if (c.geo)
        rans_dec_init_kernel<MixedLanes><<<grid, 128, 0, st>>>(streams, stream_len, stream_stride, c.n_img,
                                                               MixedLanes{c.lane0}, container, states, lane_ptr, err_flag);
    else
        rans_dec_init_kernel<EqualLanes><<<grid, 128, 0, st>>>(streams, stream_len, stream_stride, c.n_img,
                                                               EqualLanes{c.lanes}, container, states, lane_ptr, err_flag);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

static int g_dec_thread_min_rows = 4096;
static int g_dec_smem_warp = 1;     // warp-per-row steps use the shared-memory decoder (0: the global-memory one; tests)
void rans_set_dec_smem_warp(int on) { g_dec_smem_warp = on ? 1 : 0; }
void rans_set_dec_thread_min_rows(int rows) { g_dec_thread_min_rows = rows < 1 ? 1 : rows; }
void rans_set_enc_thread_min_streams(int n) { g_enc_thread_min_streams = n < 1 ? 1 : n; }
void rans_set_enc_block_max_streams(int n) { g_enc_block_max_streams = n < 0 ? 0 : n; }

// (`form`: 0 = by the policy below; 1 warp per row on the int32 tables, 2 warp per row on shared-memory tables, 3 thread per
// row = that form, LBIC_ERR_INVALID if it does not apply)
template <class Rows>
int rans_dec_step_any(const Tables &T, RansStreamState *states, const uint8_t *const *lane_ptr, int lanes, const Rows &s,
                      int R, int M, const float *ksi, int ld_ksi, h16 *yq_hi, h16 *yq_lo, int ld_yq, int32_t *sym_out,
                      cudaStream_t st, int form) {
    if (R <= 0) return 0;
    if (M > 256) return lbic_fail(LBIC_ERR_INVALID, "M > 256 unsupported by the decode step");
    const bool thread_ok = T.cdf16_total > 0 && M % 4 == 0 && ld_ksi % 4 == 0 && ld_yq % 4 == 0;
    const size_t smem_s = 16 * (((size_t)T.cdf16_total + 7) / 8) + 1024 + (size_t)DEC_S_WARPS * RANS_ROW_SCRATCH(M);
    const bool smem_ok = T.cdf16_total > 0 && smem_s <= 200 * 1024;
    if (form < 0 || form > 3 || (form == 3 && !thread_ok) || (form == 2 && !smem_ok))
        return lbic_fail(LBIC_ERR_INVALID, "rANS decode step form %d does not apply", form);
    // many streams: one thread per stream with the tables in shared memory; few (single images): one warp per stream
    if (form == 0) form = thread_ok && R >= g_dec_thread_min_rows ? 3 : smem_ok && g_dec_smem_warp ? 2 : 1;
    if (form == 3) {
        const size_t smem = 16 * (((size_t)T.cdf16_total + 64 * 257 + 7) / 8) + 4 * 64 * 4;
        static unsigned long long attr_mask = 0;
        if (lbic_first_use_on_device(attr_mask))
            LBIC_CUDA(cudaFuncSetAttribute(rans_dec_step_thread_kernel<Rows>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        rans_dec_step_thread_kernel<Rows><<<(R + DEC_T_THREADS - 1) / DEC_T_THREADS, DEC_T_THREADS, smem, st>>>(
            T.cdf16, T.cdf16_off, T.cdf16_total, T.cdf_length, T.offset, T.d_scale_table, states, lane_ptr, lanes, s, R, M,
            ksi, ld_ksi, yq_hi, yq_lo, ld_yq, sym_out);
        count_launch(1);
        LBIC_CUDA(cudaGetLastError());
        return 0;
    }
    if (form == 2) {
        // few rows: one warp per row on shared-memory tables
        static unsigned long long attr_mask2 = 0;
        if (lbic_first_use_on_device(attr_mask2))
            LBIC_CUDA(cudaFuncSetAttribute(rans_dec_step_smem_kernel<Rows>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        rans_dec_step_smem_kernel<Rows><<<(R + DEC_S_WARPS - 1) / DEC_S_WARPS, DEC_S_WARPS * 32, smem_s, st>>>(
            T.cdf16, T.cdf16_off, T.cdf16_total, T.cdf_length, T.offset, T.d_scale_table, states, lane_ptr, lanes, s, R, M,
            ksi, ld_ksi, yq_hi, yq_lo, ld_yq, sym_out);
        count_launch(1);
        LBIC_CUDA(cudaGetLastError());
        return 0;
    }
    const int warps_per_block = 4;
    rans_dec_step_kernel<Rows><<<(R + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(
        T.cdf, T.stride, T.cdf_length, T.offset, T.d_scale_table, states, lane_ptr, lanes, s, R, M, ksi, ld_ksi, yq_hi, yq_lo,
        ld_yq, sym_out);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_rans_dec_step(const Tables &T, RansStreamState *states, const uint8_t *const *lane_ptr, int lanes,
                         const StepRows &s, int M, const float *ksi, int ld_ksi, h16 *yq_hi, h16 *yq_lo, int ld_yq,
                         int32_t *sym_out, cudaStream_t st, int form) {
    if (s.geo)   // schedule rows [sd.t, sd.t + R)
        return rans_dec_step_any(T, states, lane_ptr, 0, MixedDecRows{s.geo->stream + s.sd.t, s.sd.t}, s.R, M, ksi,
                                 ld_ksi, yq_hi, yq_lo, ld_yq, sym_out, st, form);
    return rans_dec_step_any(T, states, lane_ptr, lanes, s.sd, s.R, M, ksi, ld_ksi, yq_hi, yq_lo, ld_yq, sym_out, st, form);
}

int launch_selfinfo_step(const StepDesc &s, int R, int M, const float *ksi, int ld_ksi, const int32_t *sym, float *info,
                         cudaStream_t st) {
    if (R <= 0) return 0;
    const int n = R * M;
    selfinfo_step_kernel<<<(n + 255) / 256, 256, 0, st>>>(s, R, M, ksi, ld_ksi, sym, info);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

// The two index routines of the decoders on given scales: scale_to_index as the warp-per-row decoders and the wave
// kernel call it, and the hinted lookup with its bisection fallback as the thread-per-stream decoder does.
__global__ void scale_index_kernel(const float *__restrict__ scales, int n, const float *__restrict__ tab,
                                   int32_t *__restrict__ idx_bisect, int32_t *__restrict__ idx_hinted) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    idx_bisect[i] = scale_to_index(scales[i], tab);
    const float s = fmaxf(scales[i], LBIC_SCALES_MIN);
    const ScaleHint hint = scale_hint(tab);
    bool ok;
    int ci = scale_to_index_hinted(s, tab, hint, &ok);
    if (!ok) ci = scale_to_index_bisect(s, tab);
    idx_hinted[i] = ci;
}

int launch_scale_index(const float *scales, int n, const float *tab, int32_t *idx_bisect, int32_t *idx_hinted, cudaStream_t st) {
    if (n <= 0) return 0;
    scale_index_kernel<<<(n + 255) / 256, 256, 0, st>>>(scales, n, tab, idx_bisect, idx_hinted);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

int launch_rans_decode_full(const Tables &T, const uint8_t *streams, const uint32_t *stream_len, size_t stream_stride,
                            const uint8_t *idx, int n_streams, int64_t n_sym, int32_t *sym_out, cudaStream_t st) {
    if (!T.cdf) return lbic_fail(LBIC_ERR_STATE, "Uninitialized CDFs. Run update() first");
    const int warps_per_block = 4;
    rans_decode_full_kernel<<<(n_streams + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, st>>>(
        T.cdf, T.stride, T.cdf_length, T.offset, streams, stream_len, stream_stride, idx, n_streams, (long)n_sym,
        sym_out);
    count_launch(1);
    LBIC_CUDA(cudaGetLastError());
    return 0;
}

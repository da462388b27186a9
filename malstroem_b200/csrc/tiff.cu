// tiff.cu — SURVEY.md §8(f3): the raster codec of malstroem/io.py on the device.
//
// The reference reads and writes its rasters through GDAL's GeoTIFF driver (io.py:52-72 RasterReader.read,
// io.py:112-139 RasterWriter.write: tiled='yes', compress='deflate', predictor 2 for float32 / int32 / uint8).  With
// the algorithms on the GPU, zlib on one core is what `malstroem complete` would spend its time in (five full
// rasters per run), so the two halves that touch every byte are kernels here; the container (header, tag directory,
// tile offsets) is a few hundred bytes and is handled on the host side (malstroem_b200/io.py).
//
// ENCODE (k_tiff_encode): one CTA per 256 x 256 tile, one thread per tile row.  The horizontal predictor (TIFF
// predictor 2: each sample minus its left neighbour, in the sample's own width, wrapping) is applied on the fly, the
// row is tokenised as run-length LZ77 at sample granularity (a sample equal to its predecessor extends a match with
// distance = sample size: flat areas and constant slopes become zeros after differencing and collapse to a few bits),
// and the tokens go out as ONE fixed-Huffman deflate block (RFC 1951 3.2.6) wrapped as a zlib stream (RFC 1950: 0x78
// 0x9C ... Adler-32), which is what TIFF compression 8 holds.  Two passes over the row: count bits (+ Adler-32
// partials), block-wide exclusive scan, then write the bits at the row's offset (64-bit accumulator, whole words
// stored plainly, the two shared words at the ends with atomicOr into the zeroed slot).
//
// DECODE (k_tiff_inflate + k_tiff_unpack): any conforming deflate stream (stored, fixed and dynamic Huffman blocks -
// GDAL / zlib write dynamic ones), one warp per tile or strip with lane 0 decoding (canonical-code walk, RFC 1951
// 3.2.2) and the whole warp copying matches; then the predictor is undone per row, the block is cropped into the raster
// and the nodata substitution of RasterReader.read (io.py:69-71: isnan / isclose) is applied on the way.
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace ms {

constexpr int TT = 256;                 // tile edge (GDAL's default block size for TILED=YES)

__device__ __forceinline__ unsigned rev_bits(unsigned code, int n) { return __brev(code) >> (32 - n); }

// length -> (symbol - 257, extra bits, extra value) of RFC 1951 3.2.5
__device__ __forceinline__ void length_code(int len, int &sym, int &ebits, int &eval) {
    if (len == 258) { sym = 28; ebits = 0; eval = 0; return; }
    int l = len - 3;
    if (l < 8) { sym = l; ebits = 0; eval = 0; return; }
    int g = 31 - __clz(l);              // l in [2^g, 2^(g+1))
    ebits = g - 2;
    sym = 4 * ebits + 4 + ((l >> ebits) & 3);
    eval = l & ((1 << ebits) - 1);
}

struct BitSink {
    unsigned *out;          // zeroed slot, word addressed
    size_t word;            // next word to write
    unsigned long long acc;
    int nacc;
    bool first;
    __device__ void init(unsigned *o, size_t bitpos) { out = o; word = bitpos >> 5; acc = 0; nacc = (int)(bitpos & 31); first = true; }
    __device__ __forceinline__ void put(unsigned v, int n) {
        acc |= (unsigned long long)v << nacc;
        nacc += n;
        if (nacc >= 32) {
            if (first) { atomicOr(out + word, (unsigned)acc); first = false; }
            else out[word] = (unsigned)acc;
            word++;
            acc >>= 32;
            nacc -= 32;
        }
    }
    __device__ void finish() { if (nacc > 0) atomicOr(out + word, (unsigned)acc); }
};

// fixed Huffman codes (RFC 1951 3.2.6), bit-reversed for the LSB-first stream
__device__ __forceinline__ int lit_bits(unsigned v) { return v < 144 ? 8 : 9; }
__device__ __forceinline__ void put_literal(BitSink &s, unsigned v) {
    if (v < 144) s.put(rev_bits(0x30 + v, 8), 8);
    else s.put(rev_bits(0x190 + (v - 144), 9), 9);
}
template <int ES> __device__ __forceinline__ int match_bits(int len) {
    int sym, eb, ev;
    length_code(len, sym, eb, ev);
    return (sym < 23 ? 7 : 8) + eb + 5 + (ES == 8 ? 1 : 0);
}
template <int ES> __device__ __forceinline__ void put_match(BitSink &s, int len) {
    int sym, eb, ev;
    length_code(len, sym, eb, ev);
    if (sym < 23) s.put(rev_bits(sym + 1, 7), 7);               // symbols 257..279: 7-bit codes 0000001..
    else s.put(rev_bits(0xC0 + (sym - 23), 8), 8);              // 280..287: 8-bit codes 11000000..
    if (eb) s.put((unsigned)ev, eb);
    // distance = ES: codes 0 (1), 1 (2), 3 (4), 5 (7-8, one extra bit)
    const int dcode = ES == 1 ? 0 : (ES == 2 ? 1 : (ES == 4 ? 3 : 5));
    s.put(rev_bits(dcode, 5), 5);
    if (ES == 8) s.put(1u, 1);
}

template <int ES> struct SampleT;
template <> struct SampleT<1> { typedef unsigned char T; };
template <> struct SampleT<2> { typedef unsigned short T; };
template <> struct SampleT<4> { typedef unsigned int T; };
template <> struct SampleT<8> { typedef unsigned long long T; };

// Walk one tile row: calls lit(value) for a sample that goes out as ES literal bytes and run(nsamples) for a run of
// samples equal to their predecessor.  `prev` = the value before the row's first sample in the stream (hasprev).
template <int ES, class FL, class FR>
__device__ __forceinline__ void walk_row(const typename SampleT<ES>::T *row, int valid, bool predictor,
                                         unsigned long long prev, bool hasprev, FL lit, FR run) {
    typedef typename SampleT<ES>::T T;
    constexpr int MINRUN = ES >= 4 ? 1 : (ES == 2 ? 2 : 3);      // a match is at least 3 bytes
    T left = 0;
    unsigned long long pv = prev;
    int pending = 0;                     // samples equal to pv not yet emitted
    bool have = hasprev;
    for (int x = 0; x < TT; x++) {
        T sample = x < valid ? row[x] : (T)0;
        T v = predictor ? (T)(sample - left) : sample;
        left = sample;
        if (have && (unsigned long long)v == pv) { pending++; continue; }
        if (pending) {
            if (pending >= MINRUN) run(pending);
            else for (int k = 0; k < pending; k++) lit(pv);
            pending = 0;
        }
        lit((unsigned long long)v);
        pv = v;
        have = true;
    }
    if (pending) {
        if (pending >= MINRUN) run(pending);
        else for (int k = 0; k < pending; k++) lit(pv);
    }
}

// a run of n samples as matches of at most 258 bytes, none shorter than 3, each a whole number of samples
template <int ES, class F> __device__ __forceinline__ void split_run(int nsamples, F emit) {
    constexpr int MAXL = 258 - (258 % ES);
    int len = nsamples * ES;
    while (len > 0) {
        int l = len < MAXL ? len : MAXL;
        const int rest = len - l;
        if (rest > 0 && rest < 3) {          // only for 1- and 2-byte samples: leave at least 3 bytes for the last piece
            int need = 3 - rest;
            if (ES == 2 && (need & 1)) need++;
            l -= need;
        }
        emit(l);
        len -= l;
    }
}

template <int ES>
__global__ void __launch_bounds__(TT) k_tiff_encode(const unsigned char *__restrict__ data, int rows, int cols, int tiles_x,
                                                    int predictor, unsigned char *out, size_t slot, unsigned *sizes) {
    typedef typename SampleT<ES>::T T;
    __shared__ unsigned s_bits[TT], s_a[TT], s_b[TT], s_warp[TT / 32];
    const int tile = blockIdx.x, ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = ty * TT + tid, c0 = tx * TT;
    const int valid = r < rows ? min(TT, cols - c0) : 0;
    const T *row = reinterpret_cast<const T *>(data) + (size_t)(r < rows ? r : 0) * cols + c0;
    // the value that precedes this row in the tile's byte stream: the last value of the previous tile row
    unsigned long long prev = 0;
    bool hasprev = tid > 0;
    if (hasprev) {
        const int pr = r - 1;
        const int pvalid = pr < rows ? min(TT, cols - c0) : 0;
        const T *prow = reinterpret_cast<const T *>(data) + (size_t)(pr < rows ? pr : 0) * cols + c0;
        T last = TT - 1 < pvalid ? prow[TT - 1] : (T)0, before = TT - 2 < pvalid ? prow[TT - 2] : (T)0;
        prev = predictor ? (unsigned long long)(T)(last - before) : (unsigned long long)last;
    }
    // ---- pass 1: bits and Adler-32 partials of this row
    unsigned nbits = 0, a = 0, b = 0;
    walk_row<ES>(row, valid, predictor != 0, prev, hasprev,
        [&](unsigned long long v) {
#pragma unroll
            for (int k = 0; k < ES; k++) nbits += lit_bits((unsigned)(v >> (8 * k)) & 255u);
        },
        [&](int n) { split_run<ES>(n, [&](int l) { nbits += match_bits<ES>(l); }); });
    // Adler-32 partials (sum of the bytes, sum of the running sums) over the row's value stream
    {
        T left = 0;
        for (int x = 0; x < TT; x++) {
            T sample = x < valid ? row[x] : (T)0;
            T v = predictor ? (T)(sample - left) : sample;
            left = sample;
#pragma unroll
            for (int k = 0; k < ES; k++) { a += (unsigned)((unsigned long long)v >> (8 * k)) & 255u; b += a; }
        }
    }
    s_bits[tid] = nbits;
    s_a[tid] = a % 65521u;
    s_b[tid] = b % 65521u;
    // ---- exclusive scan of the bit counts over the 256 rows
    unsigned inc = nbits;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    unsigned base = 0;
    for (int w = 0; w < warp; w++) base += s_warp[w];
    const unsigned total = s_warp[0] + s_warp[1] + s_warp[2] + s_warp[3] + s_warp[4] + s_warp[5] + s_warp[6] + s_warp[7];
    const size_t start = 19 + (size_t)base + inc - nbits;      // 16 bits zlib header + 3 bits block header
    unsigned *dst = reinterpret_cast<unsigned *>(out + (size_t)tile * slot);
    // ---- pass 2: the bits
    BitSink sink;
    sink.init(dst, tid == 0 ? 0 : start);
    if (tid == 0) {
        sink.put(0x9C78u, 16);      // CMF 0x78 (deflate, 32 K window), FLG 0x9C
        sink.put(3u, 3);            // BFINAL = 1, BTYPE = 01 (fixed Huffman)
    }
    walk_row<ES>(row, valid, predictor != 0, prev, hasprev,
        [&](unsigned long long v) {
#pragma unroll
            for (int k = 0; k < ES; k++) put_literal(sink, (unsigned)(v >> (8 * k)) & 255u);
        },
        [&](int n) { split_run<ES>(n, [&](int l) { put_match<ES>(sink, l); }); });
    if (tid == TT - 1) {
        sink.put(0u, 7);            // end of block (symbol 256: 0000000)
        // pad to a byte, then Adler-32 (big-endian) of the uncompressed tile
        const size_t endbit = 19 + (size_t)total + 7;
        const int pad = (int)((8 - (endbit & 7)) & 7);
        if (pad) sink.put(0u, pad);
        unsigned A = 1, B = 0;
        const unsigned nrow = TT * ES;
        for (int k = 0; k < TT; k++) {
            B = (unsigned)(((unsigned long long)B + (unsigned long long)nrow * A + s_b[k]) % 65521ull);
            A = (A + s_a[k]) % 65521u;
        }
        unsigned ad = (B << 16) | A;
        sink.put((ad >> 24) & 255u, 8); sink.put((ad >> 16) & 255u, 8); sink.put((ad >> 8) & 255u, 8); sink.put(ad & 255u, 8);
        sizes[tile] = (unsigned)((endbit + pad) / 8 + 4);
    }
    sink.finish();
}

// ---- inflate -----------------------------------------------------------------------------------------------------------
struct BitSrc {
    const unsigned char *p, *end;
    unsigned long long acc;
    int nacc;
    __device__ void init(const unsigned char *b, const unsigned char *e) { p = b; end = e; acc = 0; nacc = 0; }
    __device__ __forceinline__ void fill() {
        while (nacc <= 56 && p < end) { acc |= (unsigned long long)(*p++) << nacc; nacc += 8; }
    }
    __device__ __forceinline__ unsigned bits(int n) {
        if (nacc < n) fill();
        unsigned v = (unsigned)(acc & ((1ull << n) - 1ull));
        acc >>= n;
        nacc -= n;
        return v;
    }
};

struct Huff {
    unsigned short count[16];
    unsigned short symbol[288];
};

// canonical code from code lengths (RFC 1951 3.2.2); returns false for an over-subscribed set
__device__ bool huff_build(Huff &h, const unsigned char *length, int n) {
    for (int l = 0; l < 16; l++) h.count[l] = 0;
    for (int s = 0; s < n; s++) h.count[length[s]]++;
    int left = 1;
    for (int l = 1; l < 16; l++) {
        left <<= 1;
        left -= h.count[l];
        if (left < 0) return false;
    }
    unsigned short offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; l++) offs[l + 1] = offs[l] + h.count[l];
    for (int s = 0; s < n; s++)
        if (length[s]) h.symbol[offs[length[s]]++] = (unsigned short)s;
    return true;
}

__device__ __forceinline__ int huff_decode(BitSrc &b, const Huff &h) {
    int code = 0, first = 0, index = 0;
    if (b.nacc < 16) b.fill();
    for (int len = 1; len < 16; len++) {
        code |= (int)(b.acc & 1ull);
        b.acc >>= 1;
        b.nacc--;
        int count = h.count[len];
        if (code - count < first) return h.symbol[index + (code - first)];
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

__constant__ unsigned short c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ unsigned char c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ unsigned short c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ unsigned char c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ unsigned char c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// One warp per stream.  Lane 0 decodes; literals are written by lane 0, matches are copied by the whole warp.
// in_off / in_len: the zlib stream of block k inside `in`; out: k * out_stride, out_len bytes expected.  err: set to
// the (1 + stream index) of a malformed stream.
__global__ void __launch_bounds__(128) k_tiff_inflate(const unsigned char *__restrict__ in, const unsigned long long *__restrict__ in_off,
                                                      const unsigned *__restrict__ in_len, int nstreams, unsigned char *out,
                                                      size_t out_stride, unsigned out_len, unsigned last_len, int *err) {
    __shared__ Huff s_lc[4], s_dc[4];
    __shared__ unsigned char s_len[4][320];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = blockIdx.x * 4 + w;
    if (k >= nstreams) return;
    Huff &lc = s_lc[w], &dc = s_dc[w];
    unsigned char *lens = s_len[w];
    unsigned char *dst = out + (size_t)k * out_stride;
    BitSrc b;
    b.init(in + in_off[k], in + in_off[k] + in_len[k]);
    unsigned pos = 0;
    int bad = 0, last = 0;
    if (lane == 0) {
        unsigned cmf = b.bits(8), flg = b.bits(8);
        if ((cmf & 15u) != 8u || ((cmf << 8) | flg) % 31u != 0u || (flg & 32u)) bad = 1;
    }
    bad = __shfl_sync(0xffffffffu, bad, 0);
    while (!bad && !last) {
        int type = 0;
        if (lane == 0) { last = (int)b.bits(1); type = (int)b.bits(2); }
        last = __shfl_sync(0xffffffffu, last, 0);
        type = __shfl_sync(0xffffffffu, type, 0);
        if (type == 0) {
            // stored block: byte aligned LEN, NLEN, then LEN bytes
            unsigned len = 0;
            const unsigned char *src = nullptr;
            if (lane == 0) {
                int drop = b.nacc & 7;
                b.acc >>= drop; b.nacc -= drop;
                unsigned l = b.bits(16), nl = b.bits(16);
                if ((l ^ 0xffffu) != nl) bad = 1;
                len = l;
                // bytes still in the accumulator belong to the block
                src = b.p - (b.nacc >> 3);
                if (src + len > b.end) bad = 1;
            }
            bad = __shfl_sync(0xffffffffu, bad, 0);
            len = __shfl_sync(0xffffffffu, len, 0);
            unsigned long long sp = __shfl_sync(0xffffffffu, (unsigned long long)(size_t)src, 0);
            if (bad) break;
            if (pos + len > out_len) { bad = 1; break; }
            const unsigned char *s8 = (const unsigned char *)(size_t)sp;
            for (unsigned i = lane; i < len; i += 32) dst[pos + i] = s8[i];
            pos += len;
            if (lane == 0) { b.p = s8 + len; b.acc = 0; b.nacc = 0; }
            __syncwarp();
            continue;
        }
        if (type == 3) { bad = 1; break; }
        if (lane == 0) {
            if (type == 1) {
                for (int s = 0; s < 144; s++) lens[s] = 8;
                for (int s = 144; s < 256; s++) lens[s] = 9;
                for (int s = 256; s < 280; s++) lens[s] = 7;
                for (int s = 280; s < 288; s++) lens[s] = 8;
                huff_build(lc, lens, 288);
                for (int s = 0; s < 30; s++) lens[s] = 5;
                huff_build(dc, lens, 30);
            } else {
                int nlen = (int)b.bits(5) + 257, ndist = (int)b.bits(5) + 1, ncode = (int)b.bits(4) + 4;
                if (nlen > 286 || ndist > 30) bad = 1;
                else {
                    for (int i = 0; i < 19; i++) lens[i] = 0;
                    for (int i = 0; i < ncode; i++) lens[c_clorder[i]] = (unsigned char)b.bits(3);
                    if (!huff_build(lc, lens, 19)) bad = 1;
                    int idx = 0;
                    while (!bad && idx < nlen + ndist) {
                        int sym = huff_decode(b, lc);
                        if (sym < 0) { bad = 1; break; }
                        if (sym < 16) lens[idx++ + 0] = (unsigned char)sym;
                        else {
                            int rep, val = 0;
                            if (sym == 16) { if (idx == 0) { bad = 1; break; } val = lens[idx - 1]; rep = 3 + (int)b.bits(2); }
                            else if (sym == 17) rep = 3 + (int)b.bits(3);
                            else rep = 11 + (int)b.bits(7);
                            if (idx + rep > nlen + ndist) { bad = 1; break; }
                            while (rep--) lens[idx++] = (unsigned char)val;
                        }
                    }
                    // lens holds the literal/length lengths followed by the distance lengths; the code-length code is
                    // done with (lc is rebuilt from lens, which huff_build only reads)
                    if (!bad) {
                        if (lens[256] == 0) bad = 1;
                        unsigned char dl[32];
                        for (int i = 0; i < ndist; i++) dl[i] = lens[nlen + i];
                        if (!huff_build(lc, lens, nlen)) bad = 1;
                        if (!huff_build(dc, dl, ndist)) bad = 1;
                    }
                }
            }
        }
        bad = __shfl_sync(0xffffffffu, bad, 0);
        if (bad) break;
        // ---- the block's symbols
        for (;;) {
            int len = 0, dist = 0, stop = 0;
            if (lane == 0) {
                // literals are written as they come; a match or the end of the block is handed to the warp
                for (;;) {
                    int sym = huff_decode(b, lc);
                    if (sym < 0) { bad = 1; stop = 1; break; }
                    if (sym < 256) {
                        if (pos >= out_len) { bad = 1; stop = 1; break; }
                        dst[pos++] = (unsigned char)sym;
                        continue;
                    }
                    if (sym == 256) { stop = 1; break; }
                    sym -= 257;
                    if (sym >= 29) { bad = 1; stop = 1; break; }
                    len = c_lbase[sym] + (int)b.bits(c_lext[sym]);
                    int ds = huff_decode(b, dc);
                    if (ds < 0 || ds >= 30) { bad = 1; stop = 1; break; }
                    dist = c_dbase[ds] + (int)b.bits(c_dext[ds]);
                    if ((unsigned)dist > pos || pos + len > out_len) { bad = 1; stop = 1; }
                    break;
                }
            }
            bad = __shfl_sync(0xffffffffu, bad, 0);
            stop = __shfl_sync(0xffffffffu, stop, 0);
            pos = __shfl_sync(0xffffffffu, pos, 0);
            if (stop) break;
            len = __shfl_sync(0xffffffffu, len, 0);
            dist = __shfl_sync(0xffffffffu, dist, 0);
            __syncwarp();
            // copy `len` bytes from `dist` back: overlapping copies repeat the last `dist` bytes
            if (dist >= len || dist >= 32) {
                for (int base = 0; base < len; base += min(dist, 32)) {
                    int n = min(min(dist, 32), len - base);
                    unsigned char v = 0;
                    if (lane < n) v = dst[pos + base + lane - dist];
                    __syncwarp();
                    if (lane < n) dst[pos + base + lane] = v;
                    __syncwarp();
                }
            } else {
                // short period: every byte is a function of the first `dist` source bytes
                for (int i = lane; i < len; i += 32) dst[pos + i] = dst[pos - dist + (i % dist)];
                __syncwarp();
            }
            pos += len;
        }
        if (bad) break;
    }
    // (the last strip of a striped file only holds the rows that are left)
    if (lane == 0 && (bad || (pos != out_len && !(k == nstreams - 1 && pos == last_len)))) atomicCAS(err, 0, k + 1);
}

// Undo the predictor per block row, crop into the raster, substitute nodata (io.py:69-71).  block = bw x bh samples
// (tiles: 256 x 256; strips: image width x rows per strip), one thread per block row.  Block k of the call sits in
// block row block_row0 + k / blocks_x of the file; only file rows [out_row0, out_row0 + out_rows) are written, file row
// r to raster row r - out_row0.
template <int ES>
__global__ void __launch_bounds__(128) k_tiff_unpack(const unsigned char *__restrict__ blocks, size_t block_stride, int bw, int bh,
                                                     int blocks_x, int nblocks, int predictor, unsigned char *raster, int rows,
                                                     int cols, int block_row0, int out_row0, int out_rows, int fmt,
                                                     int subst_mode, double nodata, double subst) {
    typedef typename SampleT<ES>::T T;
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (long long)nblocks * bh) return;
    int blk = (int)(g / bh), br = (int)(g - (long long)blk * bh);
    int by = blk / blocks_x, bx = blk - by * blocks_x;
    int r = (block_row0 + by) * bh + br, c0 = bx * bw;
    if (r >= rows || r < out_row0 || r >= out_row0 + out_rows) return;
    const T *src = reinterpret_cast<const T *>(blocks + (size_t)blk * block_stride) + (size_t)br * bw;
    T *dst = reinterpret_cast<T *>(raster) + (size_t)(r - out_row0) * cols + c0;
    int n = min(bw, cols - c0);
    T acc = 0;
    for (int x = 0; x < n; x++) {
        T v = src[x];
        if (predictor == 2) { acc = (T)(acc + v); v = acc; }
        if (subst_mode) {
            // fmt: 1 unsigned, 2 signed, 3 float
            double d;
            if (fmt == 3) d = ES == 4 ? (double)__uint_as_float((unsigned)v) : __longlong_as_double((long long)v);
            else if (fmt == 2) d = ES == 1 ? (double)(signed char)v : (ES == 2 ? (double)(short)v : (ES == 4 ? (double)(int)v : (double)(long long)v));
            else d = (double)v;
            bool hit = subst_mode == 2 ? isnan(d) : (fabs(d - nodata) <= 1e-8 + 1e-5 * fabs(nodata));      // np.isclose defaults
            if (hit) {
                if (fmt == 3) v = ES == 4 ? (T)__float_as_uint((float)subst) : (T)__double_as_longlong(subst);
                else v = (T)(long long)subst;
            }
        }
        dst[x] = v;
    }
}

// the encoded tiles, one after the other: tile k's sizes[k] bytes from its slot to packed + offs[k]
__global__ void __launch_bounds__(256) k_tiff_pack(const unsigned char *__restrict__ slots, size_t slot,
                                                   const unsigned *__restrict__ sizes, const unsigned long long *__restrict__ offs,
                                                   unsigned char *__restrict__ packed) {
    const int k = blockIdx.x;
    const unsigned n = sizes[k];
    const unsigned char *src = slots + (size_t)k * slot;
    unsigned char *dst = packed + offs[k];
    // word copies where both sides allow it (slots are 256-byte aligned; the destination rarely is)
    for (unsigned i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

}  // namespace ms

extern "C" {

/* tile k's sizes[k] bytes (slot k of `slots`) -> packed + offs[k]  (all device) */
int ms_tiff_pack_dev(const void *slots, int64_t slot, const uint32_t *sizes, const uint64_t *offs, int64_t ntiles,
                     void *packed, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!slots || !sizes || !offs || !packed || ntiles < 1) { set_error("tiff pack: bad argument"); return MS_ERR_ARG; }
    MS_LAUNCH(k_tiff_pack, (int)ntiles, 256, 0, (cudaStream_t)stream, (const unsigned char *)slots, (size_t)slot, sizes,
              (const unsigned long long *)offs, (unsigned char *)packed);
    return MS_OK;
}

/* Worst-case size of one encoded 256 x 256 tile of `sample_bytes`-wide samples (slot size for ms_tiff_encode_dev) */
int64_t ms_tiff_tile_slot(int sample_bytes) {
    int64_t raw = (int64_t)ms::TT * ms::TT * sample_bytes;
    return ((raw * 9 + 7) / 8 + 64 + 255) & ~(int64_t)255;
}

/* RasterWriter.write (io.py:112-139), the part that touches every byte: the raster (device, row major, sample_bytes
 * 1 / 2 / 4 / 8) as zlib streams of its 256 x 256 tiles in row-major tile order, tile k at out + k * slot
 * (slot = ms_tiff_tile_slot), sizes[k] bytes long.  predictor: 1 none, 2 horizontal differencing. */
int ms_tiff_encode_dev(const void *raster, int sample_bytes, int64_t rows, int64_t cols, int predictor, void *out,
                       int64_t slot, uint32_t *sizes, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!raster || !out || !sizes || rows < 1 || cols < 1 || (predictor != 1 && predictor != 2) ||
        slot < ms_tiff_tile_slot(sample_bytes)) {
        set_error("tiff encode: bad argument");
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    int tiles_x = (int)cdiv(cols, TT), tiles_y = (int)cdiv(rows, TT);
    int ntiles = tiles_x * tiles_y;
    MS_CUDA(cudaMemsetAsync(out, 0, (size_t)ntiles * (size_t)slot, s));
    prof_units(rows * cols);
    const unsigned char *d = (const unsigned char *)raster;
    unsigned char *o = (unsigned char *)out;
    int pr = predictor == 2 ? 1 : 0;
    switch (sample_bytes) {
        case 1: MS_LAUNCH(k_tiff_encode<1>, ntiles, TT, 0, s, d, (int)rows, (int)cols, tiles_x, pr, o, (size_t)slot, sizes); break;
        case 2: MS_LAUNCH(k_tiff_encode<2>, ntiles, TT, 0, s, d, (int)rows, (int)cols, tiles_x, pr, o, (size_t)slot, sizes); break;
        case 4: MS_LAUNCH(k_tiff_encode<4>, ntiles, TT, 0, s, d, (int)rows, (int)cols, tiles_x, pr, o, (size_t)slot, sizes); break;
        case 8: MS_LAUNCH(k_tiff_encode<8>, ntiles, TT, 0, s, d, (int)rows, (int)cols, tiles_x, pr, o, (size_t)slot, sizes); break;
        default: set_error("tiff encode: sample size %d", sample_bytes); return MS_ERR_ARG;
    }
    return MS_OK;
}

/* RasterReader.read_rows: the window of file rows [out_row0, out_row0 + out_rows) of ms_tiff_decode_dev.  The nblocks
 * streams are the whole block rows from block row block_row0 on (k * blocks_x tiles, or k strips) and must cover the
 * window; `raster` is out_rows x cols and receives the window, `rows` is the file's row count.  The last strip of a
 * striped file may be short only when the call holds the file's last block row. */
int ms_tiff_decode_rows_dev(const void *in, const uint64_t *in_off, const uint32_t *in_len, int64_t nblocks,
                            int block_w, int block_h, int sample_bytes, int sample_format, int predictor, void *scratch,
                            void *raster, int64_t rows, int64_t cols, int64_t block_row0, int64_t out_row0,
                            int64_t out_rows, int subst_mode, double nodata, double subst, int compressed, void *stream) {
    using namespace ms;
    MS_TRY(ensure_init());
    if (!in || !in_off || !in_len || !scratch || !raster || nblocks < 1 || block_w < 1 || block_h < 1 || rows < 1 ||
        cols < 1 || (predictor != 1 && predictor != 2)) {
        set_error("tiff decode: bad argument");
        return MS_ERR_ARG;
    }
    const int64_t blocks_x = cdiv(cols, block_w), block_rows = cdiv(rows, block_h), k = nblocks / blocks_x;
    if (nblocks % blocks_x || block_row0 < 0 || block_row0 + k > block_rows || out_rows < 1 || out_row0 < block_row0 * block_h ||
        out_row0 + out_rows > min(rows, (block_row0 + k) * block_h)) {
        set_error("tiff decode: %lld blocks from block row %lld do not cover rows [%lld, %lld) of %lld",
                  (long long)nblocks, (long long)block_row0, (long long)out_row0, (long long)(out_row0 + out_rows),
                  (long long)rows);
        return MS_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    size_t block_bytes = (size_t)block_w * block_h * sample_bytes;
    // strips (block_w == cols): the file's last one holds the remaining rows only; tiles are always whole
    int64_t last_rows = rows - (block_rows - 1) * block_h;
    size_t last_bytes = block_w >= cols && block_row0 + k == block_rows ? (size_t)block_w * (size_t)last_rows * sample_bytes
                                                                        : block_bytes;
    const unsigned char *blocks = (const unsigned char *)scratch;
    if (compressed) {
        DevBuf<int> err;
        MS_TRY(err.alloc(1, s));
        MS_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), s));
        prof_units(out_rows * cols);
        MS_LAUNCH(k_tiff_inflate, cdiv(nblocks, 4), 128, 0, s, (const unsigned char *)in, (const unsigned long long *)in_off,
                  in_len, (int)nblocks, (unsigned char *)scratch, block_bytes, (unsigned)block_bytes, (unsigned)last_bytes, err.p);
        int *h = (int *)host_flags().h;
        MS_TRY(ms::readback(h, err.p, sizeof(int), s));
        MS_TRY(ms::stream_sync(s));
        if (*h) { set_error("tiff decode: stream %d is not a valid zlib stream of %zu bytes", *h - 1, block_bytes); return MS_ERR_ARG; }
    }
    int64_t nthreads = nblocks * block_h;
    unsigned char *r8 = (unsigned char *)raster;
#define MS_UNPACK(ES)                                                                                                    \
    MS_LAUNCH(k_tiff_unpack<ES>, cdiv(nthreads, 128), 128, 0, s, blocks, block_bytes, block_w, block_h, (int)blocks_x,     \
              (int)nblocks, predictor, r8, (int)rows, (int)cols, (int)block_row0, (int)out_row0, (int)out_rows,          \
              sample_format, subst_mode, nodata, subst)
    switch (sample_bytes) {
        case 1: MS_UNPACK(1); break;
        case 2: MS_UNPACK(2); break;
        case 4: MS_UNPACK(4); break;
        case 8: MS_UNPACK(8); break;
        default: set_error("tiff decode: sample size %d", sample_bytes); return MS_ERR_ARG;
    }
#undef MS_UNPACK
    return MS_OK;
}

/* RasterReader.read (io.py:52-72), the part that touches every byte: nblocks zlib streams (`in` + in_off[k], in_len[k]
 * bytes; all device) of blocks of block_w x block_h samples (tiles, or strips with block_w = cols) are inflated into
 * `scratch` (nblocks * block_w * block_h * sample_bytes bytes), the predictor is undone, the blocks are cropped into
 * the rows x cols raster and samples that are the file's nodata value (subst_mode 1: isclose(nodata); 2: isnan) are
 * replaced by `subst` (subst_mode 0: none).  sample_format: 1 unsigned, 2 signed, 3 float.  MS_ERR_ARG with the
 * index of the stream in the message when a stream is malformed.  The whole file: the window (0, 0, rows) of
 * ms_tiff_decode_rows_dev. */
int ms_tiff_decode_dev(const void *in, const uint64_t *in_off, const uint32_t *in_len, int64_t nblocks, int block_w,
                       int block_h, int sample_bytes, int sample_format, int predictor, void *scratch, void *raster,
                       int64_t rows, int64_t cols, int subst_mode, double nodata, double subst, int compressed,
                       void *stream) {
    return ms_tiff_decode_rows_dev(in, in_off, in_len, nblocks, block_w, block_h, sample_bytes, sample_format, predictor,
                                   scratch, raster, rows, cols, 0, 0, rows, subst_mode, nodata, subst, compressed, stream);
}

}  // extern "C"

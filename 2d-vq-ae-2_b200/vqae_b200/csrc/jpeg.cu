// Baseline JPEG tiles of a uint8 RGB canvas level (include/vqae_b200.h, vqae_jpeg_tiles; DESIGN.md 4.16).
//
// Each tile is encoded as the baseline sequential JFIF file libjpeg(-turbo) writes with the standard
// Annex K Huffman tables: jccolor.c fixed-point colour conversion, 4:4:4 or 4:2:0 (edge replication,
// (sum + 1|2) >> 2 downsampling), jfdctint islow FDCT, rounding-to-nearest quantisation by 8 Q[k],
// dummy blocks at the right and bottom edges, one scan with the DC predictors running over the whole
// tile, 0xFF stuffing and 1-bit padding.  The headers come from the host (vqae_b200/jpeg.py) and are
// copied in front of each scan.  Integer arithmetic only and no atomics: a tile's bytes depend on its
// pixels, the quality tables and the subsampling, nothing else.
//
// Tile (c, r) of a level W x H with tile size T and overlap o (0 <= o < T) covers x in [max(0, cT - o),
// min(W, (c+1)T + o)) and likewise in y.  A call encodes the tile rows [row0, row0 + nrows), all columns,
// row-major.
//
// Two passes of one CTA per tile and a scan between them:
//   jpeg_tile_kernel   one thread per MCU loads its clamped window, converts colour, downsamples, runs the
//                      FDCT and quantises, storing 64 zigzag int16 per block; then a CTA scan gives every
//                      block its bit offset (DC differences included); then one thread per block writes
//                      its code words: words wholly inside the block directly, its first and last
//                      (shared) word to a side array, from which the first block touching each shared
//                      word assembles it.  Finally it counts the 0xFF bytes of the scan: the tile size.
//   jpeg_offsets_kernel  the int64 exclusive scan of the tile sizes (offsets[0] = 0).
//   jpeg_write_kernel  header, stuffed scan and EOI of each tile at its offset of the payload.
#include <algorithm>

#include "common.cuh"
#include "kernels.cuh"

namespace vqae {

constexpr int JP_THREADS = 256;
constexpr int JP_SCAN_THREADS = 1024;
constexpr int JP_BLOCK_BITS = 1664;            // >= 22 DC bits + 63 x (16 + 10) AC bits, a whole word count
constexpr int JP_BLOCK_WORDS = JP_BLOCK_BITS / 32;
constexpr int JP_CHUNK = 16;                   // scan bytes per thread and round in the write kernel
constexpr int JP_HEADER_SHAPES = 16;           // (row class, column class), see axis_class

// natural (row-major) index -> zigzag position
__constant__ uint8_t c_unzigzag[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42,
                                       3,  8,  12, 17, 25, 30, 41, 43, 9,  11, 18, 24, 31, 40, 44, 53,
                                       10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60,
                                       21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

// Huffman codes as (length << 16) | code, table 0 luminance, 1 chrominance; quantisers 8 Q
struct JpegTables {
    uint32_t dc[2][12];
    uint32_t ac[2][256];
    uint16_t qdiv[2][64];                 // natural order
};

struct JpegGeom {
    int64_t ext_w, ext_h;                      // level extent
    int64_t row0, ncols;                       // first tile row of the call, tile columns
    int64_t pitch;                             // canvas row pitch in bytes
    int tile, overlap, sub420, header_len;
};

// tile span along one axis: start and length of tile i of an axis of extent ext
__host__ __device__ inline void tile_span(int64_t i, int64_t ext, int T, int o, int64_t* start, int64_t* len) {
    const int64_t a = i * T - o < 0 ? 0 : i * T - o;
    const int64_t b = (i + 1) * T + o > ext ? ext : (i + 1) * T + o;
    *start = a;
    *len = b - a;
}

__host__ __device__ inline int64_t mcus_of(int64_t len, int sub420) {
    return sub420 ? (len + 15) / 16 : (len + 7) / 8;
}

// Tiles 1 .. n-3 of an axis all span T + 2o (o < T, so only tiles n-2 and n-1 can reach the extent and only
// tile 0 starts at it); tiles 0, n-2 and n-1 are taken one by one.  The four classes of an axis: 0 the first,
// 1 a middle, 2 the second-to-last, 3 the last tile (smaller n: the lower class of a tile that is several).
__host__ __device__ inline int axis_class(int64_t i, int64_t n) {
    return i == 0 ? 0 : (i == n - 1 ? 3 : (i == n - 2 ? 2 : 1));
}

// sum of the MCU counts of tiles 0 .. i-1 of an axis of n tiles
__host__ __device__ inline int64_t axis_mcu_prefix(int64_t i, int64_t n, int64_t ext, int T, int o, int sub420) {
    int64_t st, len, sum = 0;
    const int64_t regular = i - 1 < n - 3 ? i - 1 : n - 3;      // tiles 1 .. min(i - 1, n - 3)
    if (regular > 0) {
        tile_span(1, ext, T, o, &st, &len);
        sum += regular * mcus_of(len, sub420);
    }
    const int64_t special[3] = {0, n - 2 >= 1 ? n - 2 : -1, n - 1 >= 1 ? n - 1 : -1};
    for (int k = 0; k < 3; ++k) {
        if (special[k] < 0 || special[k] >= i) continue;
        tile_span(special[k], ext, T, o, &st, &len);
        sum += mcus_of(len, sub420);
    }
    return sum;
}

// first block of tile (r, c) among the call's tiles (row-major)
__host__ __device__ inline int64_t tile_block_base(const JpegGeom& g, int64_t r, int64_t c) {
    const int nb = g.sub420 ? 6 : 3;
    const int64_t n_rows_total = (g.ext_h + g.tile - 1) / g.tile;
    const int64_t row_mcus = axis_mcu_prefix(g.ncols, g.ncols, g.ext_w, g.tile, g.overlap, g.sub420);
    const int64_t rows_before = axis_mcu_prefix(r, n_rows_total, g.ext_h, g.tile, g.overlap, g.sub420) -
                                axis_mcu_prefix(g.row0, n_rows_total, g.ext_h, g.tile, g.overlap, g.sub420);
    int64_t st, th;
    tile_span(r, g.ext_h, g.tile, g.overlap, &st, &th);
    return (int64_t)nb * (rows_before * row_mcus + mcus_of(th, g.sub420) *
                          axis_mcu_prefix(c, g.ncols, g.ext_w, g.tile, g.overlap, g.sub420));
}

// ---- CTA helpers --------------------------------------------------------------------------------------------
// exclusive scan over the CTA (blockDim.x == JP_THREADS); returns the exclusive prefix, sets *total
__device__ int64_t cta_scan(int64_t v, int64_t* total, int64_t* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t u = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += u;
    }
    if (lane == 31) sh[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int64_t w = lane < JP_THREADS / 32 ? sh[lane] : 0;
        int64_t s = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t u = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += u;
        }
        if (lane < JP_THREADS / 32) sh[lane] = s - w;
        if (lane == JP_THREADS / 32 - 1) sh[JP_THREADS / 32] = s;
    }
    __syncthreads();
    const int64_t out = sh[warp] + incl - v;
    *total = sh[JP_THREADS / 32];
    __syncthreads();
    return out;
}

// ---- colour, FDCT, quantisation -----------------------------------------------------------------------------
__device__ __forceinline__ int ycc(int r, int g, int b, int comp) {
    if (comp == 0) return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    if (comp == 1) return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// jfdctint.c (islow), CONST_BITS 13, PASS1_BITS 2; in place on 8 values with stride `st`
template <bool PASS1>
__device__ __forceinline__ void fdct_1d(int* d, int st) {
    constexpr int CB = 13, P1 = 2, SH = PASS1 ? CB - P1 : CB + P1;
    const int t0 = d[0] + d[7 * st], t7 = d[0] - d[7 * st];
    const int t1 = d[st] + d[6 * st], t6 = d[st] - d[6 * st];
    const int t2 = d[2 * st] + d[5 * st], t5 = d[2 * st] - d[5 * st];
    const int t3 = d[3 * st] + d[4 * st], t4 = d[3 * st] - d[4 * st];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    if (PASS1) {
        d[0] = (t10 + t11) << P1;
        d[4 * st] = (t10 - t11) << P1;
    } else {
        d[0] = descale(t10 + t11, P1);
        d[4 * st] = descale(t10 - t11, P1);
    }
    int z1 = (t12 + t13) * 4433;                                   // FIX(0.541196100)
    d[2 * st] = descale(z1 + t13 * 6270, SH);                      // FIX(0.765366865)
    d[6 * st] = descale(z1 - t12 * 15137, SH);                     // FIX(1.847759065)
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * 9633;                               // FIX(1.175875602)
    const int a4 = t4 * 2446, a5 = t5 * 16819, a6 = t6 * 25172, a7 = t7 * 12299;
    z1 *= -7373;                                                   // FIX(0.899976223)
    z2 *= -20995;                                                  // FIX(2.562915447)
    z3 = z3 * -16069 + z5;                                         // FIX(1.961570560)
    z4 = z4 * -3196 + z5;                                          // FIX(0.390180644)
    d[7 * st] = descale(a4 + z1 + z3, SH);
    d[5 * st] = descale(a5 + z2 + z4, SH);
    d[3 * st] = descale(a6 + z2 + z3, SH);
    d[st] = descale(a7 + z1 + z4, SH);
}

// category (bit length) of |v|
__device__ __forceinline__ int category(int v) { return v == 0 ? 0 : 32 - __clz(v < 0 ? -v : v); }

// bit k set for every nonzero zigzag coefficient k of a block
__device__ __forceinline__ uint64_t nonzero_mask(const int16_t* zz) {
    const int4* p = reinterpret_cast<const int4*>(zz);
    uint64_t m = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int4 w = p[i];
        const int v[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            if (v[h] & 0xffff) m |= 1ull << (8 * i + 2 * h);
            if (v[h] >> 16) m |= 1ull << (8 * i + 2 * h + 1);
        }
    }
    return m;
}

// the DC difference and AC symbols of one block (zigzag coefficients `zz`) into `put(code, len)`
template <typename Put>
__device__ __forceinline__ void block_symbols(const int16_t* zz, int diff, const uint32_t* dc, const uint32_t* ac,
                                              Put&& put) {
    const int cat = category(diff);
    put(dc[cat] & 0xffffu, dc[cat] >> 16);
    put((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << cat) - 1), cat);
    uint64_t nz = nonzero_mask(zz) & ~1ull;
    int last = 0;
    while (nz) {
        const int k = __ffsll((long long)nz) - 1;
        nz &= nz - 1;
        int run = k - last - 1;
        for (; run > 15; run -= 16) put(ac[0xF0] & 0xffffu, ac[0xF0] >> 16);
        const int v = zz[k], s = category(v);
        const uint32_t h = ac[(run << 4) | s];
        put(h & 0xffffu, h >> 16);
        put((uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1), s);
        last = k;
    }
    if (last != 63) put(ac[0] & 0xffffu, ac[0] >> 16);
}

// ---- pass 1: blocks, bit offsets, code words, 0xFF count -----------------------------------------------------
struct JpegScratch {
    int16_t* coef;        // [blocks][64] zigzag
    int64_t* boff;        // [blocks] tile-relative bit offset
    uint32_t* edge;       // [blocks][2] first / last word contribution
    uint32_t* words;      // [blocks * JP_BLOCK_WORDS] tile streams, big-endian bytes, word-aligned per tile
    int64_t* tile_bits;   // [tiles]
    int64_t* sizes;       // [tiles] file bytes
};

// the previous block of the same component in MCU order, -1 for the first
__device__ __forceinline__ int64_t pred_block(int64_t b, int nb) {
    const int64_t m = b / nb;
    const int j = (int)(b - m * nb);
    if (nb == 3) return m == 0 ? -1 : b - 3;
    if (j >= 1 && j <= 3) return b - 1;
    if (m == 0) return -1;
    return j == 0 ? b - 3 : b - 6;
}

__device__ __forceinline__ int block_table(int64_t b, int nb) {
    const int j = (int)(b % nb);
    return (nb == 3 ? j > 0 : j >= 4) ? 1 : 0;
}

__device__ __forceinline__ uint32_t bswap(uint32_t w) { return __byte_perm(w, 0, 0x0123); }

__global__ void __launch_bounds__(JP_THREADS)
jpeg_tile_kernel(const uint8_t* __restrict__ canvas, const JpegGeom g, const __grid_constant__ JpegTables tabs,
                 JpegScratch s) {
    __shared__ uint32_t sh_dc[2][12], sh_ac[2][256];
    __shared__ uint16_t sh_q[2][64];
    __shared__ uint8_t sh_unzz[64];
    __shared__ int64_t sh_scan[JP_THREADS / 32 + 1];
    __shared__ int16_t sh_rows[64 * JP_THREADS];                  // pass-1 output, |v| <= 8 * 128 * 4 * sqrt(2)
    int16_t* rows = sh_rows + threadIdx.x;
    for (int i = threadIdx.x; i < 2 * 256; i += JP_THREADS) (&sh_ac[0][0])[i] = (&tabs.ac[0][0])[i];
    if (threadIdx.x < 24) (&sh_dc[0][0])[threadIdx.x] = (&tabs.dc[0][0])[threadIdx.x];
    if (threadIdx.x < 128) (&sh_q[0][0])[threadIdx.x] = (&tabs.qdiv[0][0])[threadIdx.x];
    if (threadIdx.x < 64) sh_unzz[threadIdx.x] = c_unzigzag[threadIdx.x];
    __syncthreads();

    const int64_t t = blockIdx.x, r = g.row0 + t / g.ncols, c = t % g.ncols;
    int64_t y0, x0, th, tw;
    tile_span(r, g.ext_h, g.tile, g.overlap, &y0, &th);
    tile_span(c, g.ext_w, g.tile, g.overlap, &x0, &tw);
    const int sub = g.sub420, nb = sub ? 6 : 3, msz = sub ? 16 : 8;
    const int64_t mw = (tw + msz - 1) / msz, mh = (th + msz - 1) / msz, nblk = nb * mw * mh;
    const int64_t ybw = (tw + 7) / 8, ybh = (th + 7) / 8;
    const int64_t chh = (th + 1) / 2;                              // chroma rows before replication
    const int64_t base = tile_block_base(g, r, c);
    int16_t* coef = s.coef + base * 64;
    int64_t* boff = s.boff + base;
    uint32_t* edge = s.edge + base * 2;
    uint32_t* words = s.words + base * JP_BLOCK_WORDS;
    const uint8_t* img = canvas + y0 * g.pitch + x0 * 3;

    // 1. blocks: one thread per MCU
    for (int64_t m = threadIdx.x; m < mw * mh; m += JP_THREADS) {
        const int64_t my = m / mw, mx = m % mw;
        int prev_dc = 0;
        for (int j = 0; j < nb; ++j) {
            const int comp = sub ? (j < 4 ? 0 : j - 3) : j;
            const int tab = comp ? 1 : 0;
            int16_t* zz = coef + (m * nb + j) * 64;
            int64_t by = my, bx = mx;
            if (sub && j < 4) {
                by = 2 * my + (j >> 1);
                bx = 2 * mx + (j & 1);
            }
            if (comp == 0 && (by >= ybh || bx >= ybw)) {        // dummy block: zero AC, DC of the block before
                int4* dst = reinterpret_cast<int4*>(zz);
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = make_int4(i ? 0 : prev_dc & 0xffff, 0, 0, 0);
                continue;
            }
            // pass 1 row by row into the thread's column of `rows`, pass 2 and quantisation column by column
#pragma unroll 1
            for (int yy = 0; yy < 8; ++yy) {
                int d[8];
#pragma unroll
                for (int xx = 0; xx < 8; ++xx) {
                    int v;
                    if (!sub || comp == 0) {
                        const int64_t py = min(by * 8 + yy, th - 1), px = min(bx * 8 + xx, tw - 1);
                        const uint8_t* p = img + py * g.pitch + px * 3;
                        v = ycc(p[0], p[1], p[2], comp);
                    } else {
                        const int64_t cy = min(by * 8 + yy, chh - 1), cx = bx * 8 + xx;
                        int sum = 0;
#pragma unroll
                        for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
                            for (int dx = 0; dx < 2; ++dx) {
                                const int64_t py = min(2 * cy + dy, th - 1), px = min(2 * cx + dx, tw - 1);
                                const uint8_t* p = img + py * g.pitch + px * 3;
                                sum += ycc(p[0], p[1], p[2], comp);
                            }
                        }
                        v = (sum + 1 + (xx & 1)) >> 2;
                    }
                    d[xx] = v - 128;
                }
                fdct_1d<true>(d, 1);
#pragma unroll
                for (int xx = 0; xx < 8; ++xx) rows[(yy * 8 + xx) * JP_THREADS] = (int16_t)d[xx];
            }
#pragma unroll 1
            for (int xx = 0; xx < 8; ++xx) {
                int d[8];
#pragma unroll
                for (int yy = 0; yy < 8; ++yy) d[yy] = rows[(yy * 8 + xx) * JP_THREADS];
                fdct_1d<false>(d, 1);
#pragma unroll
                for (int yy = 0; yy < 8; ++yy) {
                    const int i = yy * 8 + xx, v = d[yy], qd = sh_q[tab][i];
                    const int a = ((v < 0 ? -v : v) + (qd >> 1)) / qd;
                    zz[sh_unzz[i]] = (int16_t)(v < 0 ? -a : a);
                }
            }
            prev_dc = zz[0];
        }
    }
    __syncthreads();

    // 2. bit offsets of the blocks, in fixed block order
    int64_t carry = 0;
    for (int64_t b0 = 0; b0 < nblk; b0 += JP_THREADS) {
        const int64_t b = b0 + threadIdx.x;
        int64_t mine = 0;
        if (b < nblk) {
            const int64_t p = pred_block(b, nb);
            const int tab = block_table(b, nb);
            const int diff = coef[b * 64] - (p < 0 ? 0 : coef[p * 64]);
            uint32_t n = 0;
            block_symbols(coef + b * 64, diff, sh_dc[tab], sh_ac[tab], [&](uint32_t, uint32_t len) { n += len; });
            mine = n;
        }
        int64_t total;
        const int64_t ex = cta_scan(mine, &total, sh_scan);
        if (b < nblk) boff[b] = carry + ex;
        carry += total;
    }
    const int64_t tbits = carry;
    if (threadIdx.x == 0) s.tile_bits[t] = tbits;
    __syncthreads();

    // 3. code words: the words inside a block directly, its first and last word to `edge`
    for (int64_t b = threadIdx.x; b < nblk; b += JP_THREADS) {
        const int64_t p = pred_block(b, nb);
        const int tab = block_table(b, nb);
        const int64_t start = boff[b], end = b + 1 < nblk ? boff[b + 1] : tbits;
        const int64_t head_word = start >> 5, last_word = (end - 1) >> 5;
        int64_t cur = head_word;                 // the word the accumulator fills
        uint64_t acc = 0;
        int nacc = (int)(start & 31);            // bits in `acc`; the leading ones belong to earlier blocks
        uint32_t head = 0, last = 0;
        auto flush = [&](uint32_t w) {
            if (cur == head_word) head = w;
            else if (cur == last_word) last = w;
            else words[cur] = bswap(w);
            ++cur;
        };
        auto put = [&](uint32_t code, uint32_t len) {
            acc = (acc << len) | code;
            nacc += len;
            if (nacc >= 32) {
                nacc -= 32;
                flush((uint32_t)(acc >> nacc));
                acc &= (1ull << nacc) - 1;
            }
        };
        const int diff = coef[b * 64] - (p < 0 ? 0 : coef[p * 64]);
        block_symbols(coef + b * 64, diff, sh_dc[tab], sh_ac[tab], put);
        if (nacc) flush((uint32_t)(acc << (32 - nacc)));
        edge[2 * b] = head;
        edge[2 * b + 1] = last;
    }
    __syncthreads();

    // 4. shared words, each assembled by the first block touching it
    for (int64_t b = threadIdx.x; b < nblk; b += JP_THREADS) {
        const int64_t start = boff[b], end = b + 1 < nblk ? boff[b + 1] : tbits;
        const int64_t hw = start >> 5, lw = (end - 1) >> 5;
        for (int side = 0; side < 2; ++side) {
            int64_t w;
            if (side == 0) {
                if (start & 31) continue;                       // an earlier block owns the first word
                w = hw;
            } else {
                if (lw == hw) continue;
                w = lw;
            }
            uint32_t v = edge[2 * b + side];
            for (int64_t b2 = b + 1; b2 < nblk && (boff[b2] >> 5) == w; ++b2) v |= edge[2 * b2];
            words[w] = bswap(v);
        }
    }
    __syncthreads();

    // 5. the tile's file size: header + scan bytes + stuffed zeros + EOI
    const int64_t nbytes = (tbits + 7) >> 3;
    const uint8_t* sb = reinterpret_cast<const uint8_t*>(words);
    int64_t ff = 0;
    for (int64_t i = threadIdx.x; i < nbytes; i += JP_THREADS) {
        uint32_t v = sb[i];
        if (i == nbytes - 1 && (tbits & 7)) v |= (1u << (8 - (tbits & 7))) - 1;
        ff += v == 0xFF;
    }
    int64_t total;
    cta_scan(ff, &total, sh_scan);
    if (threadIdx.x == 0) s.sizes[t] = g.header_len + nbytes + total + 2;
}

// ---- offsets ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(JP_SCAN_THREADS)
jpeg_offsets_kernel(const int64_t* __restrict__ sizes, int64_t n, int64_t* __restrict__ offsets) {
    __shared__ int64_t warp_sum[JP_SCAN_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t per = (n + JP_SCAN_THREADS - 1) / JP_SCAN_THREADS;
    const int64_t lo = min(n, tid * per), hi = min(n, lo + per);
    int64_t mine = 0;
    for (int64_t i = lo; i < hi; ++i) mine += sizes[i];
    int64_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int64_t v = warp_sum[lane];
        int64_t s = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t u = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += u;
        }
        warp_sum[lane] = s - v;
    }
    __syncthreads();
    int64_t run = warp_sum[warp] + incl - mine;
    if (tid == 0) offsets[0] = 0;
    for (int64_t i = lo; i < hi; ++i) {
        run += sizes[i];
        offsets[i + 1] = run;
    }
}

// ---- pass 2: header, stuffed scan, EOI ----------------------------------------------------------------------
__global__ void __launch_bounds__(JP_THREADS)
jpeg_write_kernel(const JpegGeom g, const uint8_t* __restrict__ headers, const JpegScratch s,
                  const int64_t* __restrict__ offsets, uint8_t* __restrict__ payload) {
    __shared__ int64_t sh_scan[JP_THREADS / 32 + 1];
    const int64_t t = blockIdx.x, r = g.row0 + t / g.ncols, c = t % g.ncols;
    const int64_t n_rows_total = (g.ext_h + g.tile - 1) / g.tile;
    const uint8_t* hdr = headers + (int64_t)(4 * axis_class(r, n_rows_total) + axis_class(c, g.ncols)) * g.header_len;
    uint8_t* out = payload + offsets[t];
    for (int i = threadIdx.x; i < g.header_len; i += JP_THREADS) out[i] = hdr[i];
    out += g.header_len;
    const int64_t tbits = s.tile_bits[t], nbytes = (tbits + 7) >> 3;
    const uint8_t* sb = reinterpret_cast<const uint8_t*>(s.words + tile_block_base(g, r, c) * JP_BLOCK_WORDS);
    int64_t carry = 0;
    for (int64_t i0 = 0; i0 < nbytes; i0 += (int64_t)JP_THREADS * JP_CHUNK) {
        const int64_t lo = i0 + (int64_t)threadIdx.x * JP_CHUNK;
        uint8_t v[JP_CHUNK];
        int ff = 0;
#pragma unroll
        for (int k = 0; k < JP_CHUNK; ++k) {
            const int64_t i = lo + k;
            uint32_t b = i < nbytes ? sb[i] : 0;
            if (i == nbytes - 1 && (tbits & 7)) b |= (1u << (8 - (tbits & 7))) - 1;
            v[k] = (uint8_t)b;
            ff += i < nbytes && b == 0xFF;
        }
        int64_t total;
        int64_t pos = carry + lo + cta_scan(ff, &total, sh_scan);
#pragma unroll
        for (int k = 0; k < JP_CHUNK; ++k) {
            if (lo + k >= nbytes) break;
            out[pos++] = v[k];
            if (v[k] == 0xFF) out[pos++] = 0;
        }
        carry += total;
    }
    if (threadIdx.x == 0) {
        out[nbytes + carry] = 0xFF;
        out[nbytes + carry + 1] = 0xD9;
    }
}

// ---- host ---------------------------------------------------------------------------------------------------
// Annex K.3 tables: code-length counts (16) and symbols
static const uint8_t kDcBits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
                                       {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
static const uint8_t kAcBits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
                                       {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
static const uint8_t kAcVals[2][162] = {
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
     0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
     0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
     0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
     0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
     0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
     0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
     0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
     0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
     0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
     0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
     0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
     0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
     0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
     0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
     0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
     0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};

// canonical codes (Annex C) of a (bits, values) table as (length << 16) | code
static void huff_codes(const uint8_t* nbits, const uint8_t* vals, uint32_t* out) {
    uint32_t code = 0;
    int k = 0;
    for (int len = 1; len <= 16; ++len) {
        for (int i = 0; i < nbits[len - 1]; ++i, ++k) out[vals[k]] = ((uint32_t)len << 16) | code++;
        code <<= 1;
    }
}

struct JpegPlan {
    JpegGeom g;
    int64_t ntiles, nblocks;
};

static int jpeg_plan(int64_t ext_h, int64_t ext_w, int tile, int overlap, int64_t row0, int64_t nrows,
                     int subsampling, JpegPlan* p) {
    // overlap < tile: the tile spans of axis_mcu_prefix
    if (ext_h <= 0 || ext_w <= 0 || tile <= 0 || overlap < 0 || overlap >= tile || nrows <= 0 || row0 < 0)
        return VQAE_ERR_BAD_ARG;
    const int64_t n_rows_total = (ext_h + tile - 1) / tile, ncols = (ext_w + tile - 1) / tile;
    if (row0 + nrows > n_rows_total) return VQAE_ERR_BAD_ARG;
    if (subsampling != 0 && subsampling != 2) return VQAE_ERR_UNSUPPORTED;
    int64_t s, l, max_h = 0, max_w = 0;
    for (int64_t i : {(int64_t)0, std::min<int64_t>(1, n_rows_total - 1), std::max<int64_t>(0, n_rows_total - 2),
                      n_rows_total - 1}) {
        tile_span(i, ext_h, tile, overlap, &s, &l);
        max_h = std::max(max_h, l);
    }
    for (int64_t i : {(int64_t)0, std::min<int64_t>(1, ncols - 1), std::max<int64_t>(0, ncols - 2), ncols - 1}) {
        tile_span(i, ext_w, tile, overlap, &s, &l);
        max_w = std::max(max_w, l);
    }
    if (max_h > 65535 || max_w > 65535) return VQAE_ERR_UNSUPPORTED;
    JpegGeom& g = p->g;
    g.ext_w = ext_w;
    g.ext_h = ext_h;
    g.row0 = row0;
    g.ncols = ncols;
    g.pitch = 0;
    g.tile = tile;
    g.overlap = overlap;
    g.sub420 = subsampling == 2;
    g.header_len = 0;
    p->ntiles = nrows * ncols;
    if (p->ntiles > INT32_MAX) return VQAE_ERR_UNSUPPORTED;
    p->nblocks = (int64_t)(g.sub420 ? 6 : 3) *
                 (axis_mcu_prefix(row0 + nrows, n_rows_total, ext_h, tile, overlap, g.sub420) -
                  axis_mcu_prefix(row0, n_rows_total, ext_h, tile, overlap, g.sub420)) *
                 axis_mcu_prefix(ncols, ncols, ext_w, tile, overlap, g.sub420);
    return VQAE_OK;
}

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

static size_t jpeg_scratch_layout(const JpegPlan& p, int header_len, size_t* off) {  // off[7]
    const size_t nb = (size_t)p.nblocks, nt = (size_t)p.ntiles;
    const size_t sz[7] = {nb * 64 * sizeof(int16_t), nb * sizeof(int64_t), nb * 2 * sizeof(uint32_t),
                          nb * JP_BLOCK_WORDS * sizeof(uint32_t), nt * sizeof(int64_t), nt * sizeof(int64_t),
                          (size_t)JP_HEADER_SHAPES * header_len};
    size_t total = 0;
    for (int i = 0; i < 7; ++i) {
        off[i] = total;
        total += align256(sz[i]);
    }
    return total;
}

size_t jpeg_tiles_scratch_bytes(int64_t ext_h, int64_t ext_w, int tile, int overlap, int64_t row0, int64_t nrows,
                                int subsampling, int header_len) {
    JpegPlan p;
    if (jpeg_plan(ext_h, ext_w, tile, overlap, row0, nrows, subsampling, &p) || header_len <= 0) return 0;
    size_t off[7];
    return jpeg_scratch_layout(p, header_len, off);
}

int64_t jpeg_tiles_worst_bytes(int64_t ext_h, int64_t ext_w, int tile, int overlap, int64_t row0, int64_t nrows,
                               int subsampling, int header_len) {
    JpegPlan p;
    if (jpeg_plan(ext_h, ext_w, tile, overlap, row0, nrows, subsampling, &p) || header_len <= 0) return -1;
    // every scan byte may be followed by a stuffed zero
    return p.ntiles * (header_len + 2) + p.nblocks * (2 * JP_BLOCK_BITS / 8);
}

int jpeg_tiles(const uint8_t* canvas, int64_t pitch, int64_t ext_h, int64_t ext_w, int tile, int overlap,
               int64_t row0, int64_t nrows, int quality, int subsampling, const uint8_t* headers_host,
               int header_len, const uint16_t* qtables_host, int64_t* offsets, uint8_t* payload,
               int64_t payload_capacity, void* scratch, size_t scratch_bytes, cudaStream_t stream) {
    JpegPlan p;
    if (int rc = jpeg_plan(ext_h, ext_w, tile, overlap, row0, nrows, subsampling, &p)) return rc;
    if (quality < 1 || quality > 100) return VQAE_ERR_UNSUPPORTED;
    if (!canvas || !headers_host || !qtables_host || !offsets || !payload || !scratch) return VQAE_ERR_BAD_ARG;
    if (header_len <= 0 || pitch < 3 * ext_w) return VQAE_ERR_BAD_ARG;
    if (payload_capacity < p.ntiles * (header_len + 2) + p.nblocks * (2 * JP_BLOCK_BITS / 8)) return VQAE_ERR_BAD_ARG;
    size_t off[7];
    if (scratch_bytes < jpeg_scratch_layout(p, header_len, off)) return VQAE_ERR_SCRATCH;
    JpegTables tabs;
    static const uint8_t zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                       12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                       35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                       58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    for (int t = 0; t < 2; ++t) {
        for (int k = 0; k < 64; ++k) {
            const uint16_t q = qtables_host[64 * t + k];
            if (q < 1 || q > 255) return VQAE_ERR_BAD_ARG;
            tabs.qdiv[t][zigzag[k]] = (uint16_t)(8 * q);
        }
    }
    static const uint8_t dc_vals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
    for (int t = 0; t < 2; ++t) {
        std::fill(tabs.ac[t], tabs.ac[t] + 256, 0u);
        huff_codes(kDcBits[t], dc_vals, tabs.dc[t]);
        huff_codes(kAcBits[t], kAcVals[t], tabs.ac[t]);
    }
    p.g.pitch = pitch;
    p.g.header_len = header_len;
    uint8_t* base = static_cast<uint8_t*>(scratch);
    JpegScratch s;
    s.coef = reinterpret_cast<int16_t*>(base + off[0]);
    s.boff = reinterpret_cast<int64_t*>(base + off[1]);
    s.edge = reinterpret_cast<uint32_t*>(base + off[2]);
    s.words = reinterpret_cast<uint32_t*>(base + off[3]);
    s.tile_bits = reinterpret_cast<int64_t*>(base + off[4]);
    s.sizes = reinterpret_cast<int64_t*>(base + off[5]);
    uint8_t* headers = base + off[6];
    VQAE_CUDA_TRY(cudaMemcpyAsync(headers, headers_host, (size_t)JP_HEADER_SHAPES * header_len,
                                  cudaMemcpyHostToDevice, stream));
    const unsigned grid = (unsigned)p.ntiles;
    jpeg_tile_kernel<<<grid, JP_THREADS, 0, stream>>>(canvas, p.g, tabs, s);
    if (int rc = check_launch()) return rc;
    jpeg_offsets_kernel<<<1, JP_SCAN_THREADS, 0, stream>>>(s.sizes, p.ntiles, offsets);
    if (int rc = check_launch()) return rc;
    jpeg_write_kernel<<<grid, JP_THREADS, 0, stream>>>(p.g, headers, s, offsets, payload);
    return check_launch();
}

}  // namespace vqae

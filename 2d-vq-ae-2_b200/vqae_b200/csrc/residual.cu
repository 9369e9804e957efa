// Near-lossless residual layer of stored code maps, version 1 (DESIGN.md section 4.15; include/vqae_b200.h,
// vqae_residual_stats / vqae_residual_tables / vqae_residual_encode / vqae_residual_apply).
//
// Per byte of an H x W x 3 patch (n = 3 H W bytes in canvas order: row-major, channel innermost), with x the
// original, xh the base decode and d = x - xh:
//   e = 0:  s = d & 255,                                  x' = (xh + s) & 255  (= x)
//   e >= 1: k = sign(d) floor((|d| + e) / (2e + 1)),      x' = clamp(xh + k (2e + 1), 0, 255), |x - x'| <= e
//           s = k & 255 (|k| <= 85; the decoder sign-extends s)
// Each patch is one chunk: its own 256-entry table (total 2^14, packing.quantise_frequencies of the patch's
// exact symbol counts), 32 interleaved rANS lanes (symbol i -> lane i mod 32, the coder of rans.cuh, symbols
// coded last to first), laid out as 256 x u16 frequencies | 32 x u32 lane word counts | 32 x u32 final lane
// states | the words of lane 0 in decoder order, lane 1, ..., lane 31; 768 + 2 sum(w) bytes.
//
// Kernels (patch t of a call sits at the canvas position of vqae_quality_u8's addressing tuple; all offsets
// 64-bit; integer arithmetic only and no atomics, so results are bitwise reproducible):
//   residual_stats_kernel   one CTA per patch (grid-strided): reads x and xh once, per-warp histograms in
//                           shared memory updated by one lane per distinct symbol (__match_any_sync), both
//                           Adler-32 sums (of xh and x') as 64-bit partials reduced in a fixed order
//   residual_tables_kernel  one CTA per patch: quantise_frequencies, the (count desc, symbol asc) order as a
//                           rank sort of the 256 keys, an excess settled pass by pass with a CTA scan
//   residual_encode_kernel  one warp per patch, lane j = rANS lane j: rounds of RR steps (32 RR bytes) staged
//                           in shared memory, coded backwards; each round's words are flushed coalesced to
//                           the end of the lane's worst-case region of the patch's slot; at the end the
//                           warp moves the lanes' words together into the chunk layout, and the shared
//                           offsets scan + compaction of rans.cuh builds the payload
//   residual_apply_kernel   one warp per patch: slot -> symbol table in shared memory, per round the next RR
//                           words of every lane and the RR x 32 base bytes staged in shared memory, decoded,
//                           and x' written over xh in place; both Adler values and the flags
// Bounds by construction (apply): reads of a chunk are clamped to its own [off[p], off[p + 1]) range of the
// payload, lane word counts to the lane's symbol count, and a lane decodes at most one word per symbol from
// its staged window, so a damaged chunk gives wrong pixels and a flag, never an access outside its buffers.
#include "common.cuh"
#include "kernels.cuh"
#include "rans.cuh"

namespace vqae {

namespace {

constexpr int RL_LANES = 32;
constexpr int RL_SYMS = 256;
constexpr int RL_S = 14;
constexpr uint32_t RL_M = 1u << RL_S;
constexpr int RL_HEADER = 768;                  // 256 x u16 + 32 x u32 + 32 x u32
constexpr int RL_RR = 128;                      // steps (symbols per lane) staged per round
constexpr int RL_WSTRIDE = RL_RR + 2;           // staged words per lane: an odd number of 32-bit words
constexpr int RL_WARPS = 2;                     // patches (warps) per CTA of the encode / apply kernels
constexpr int RL_STATS_THREADS = 256;
constexpr int64_t RL_MAX_PIXELS = 1 << 20;      // H W
constexpr uint32_t ADLER_MOD = 65521;

struct Canvas {                   // patch t: grid position (r0 + q / rc, c0 + q % rc), q = first + t
    uint8_t* p;
    int64_t cols, r0, c0, rc, first;
    __device__ uint8_t* patch(int64_t t, int H, int W) const {
        const int64_t q = first + t;
        const int64_t pr = r0 + q / rc, pc = c0 + q % rc;
        return p + ((pr * H) * cols + pc * W) * 3;
    }
};

__device__ __forceinline__ uint32_t res_symbol(int x, int xh, int e, int q) {
    const int d = x - xh;
    if (e == 0) return (uint32_t)d & 255u;
    const int k = (abs(d) + e) / q;
    return (uint32_t)(d < 0 ? -k : k) & 255u;
}

__device__ __forceinline__ uint32_t res_apply(int xh, uint32_t s, int e, int q) {
    if (e == 0) return (uint32_t)(xh + (int)s) & 255u;
    const int v = xh + (int)(int8_t)(uint8_t)s * q;
    return (uint32_t)min(max(v, 0), 255);
}

// byte i -> (row, byte within the row) walking in steps of `step` bytes
struct RowWalk {
    int y, r;
    __device__ void start(int64_t i, int rowb) { y = (int)(i / rowb); r = (int)(i - (int64_t)y * rowb); }
    __device__ void advance(int step, int rowb) {
        r += step;
        while (r >= rowb) { r -= rowb; ++y; }
    }
};

__device__ __forceinline__ uint32_t adler_of(uint64_t a, uint64_t b, int64_t n) {
    const uint32_t A = (uint32_t)((1 + a) % ADLER_MOD), B = (uint32_t)(((uint64_t)n + b) % ADLER_MOD);
    return (B << 16) | A;
}

__device__ __forceinline__ uint64_t warp_sum64(uint64_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    return v;
}

// exclusive prefix over the warp's lanes, and the warp total
__device__ __forceinline__ uint32_t warp_excl_scan(uint32_t v, uint32_t* total) {
    const int lane = threadIdx.x & 31;
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += u;
    }
    *total = __shfl_sync(0xffffffffu, incl, 31);
    return incl - v;
}

// ---- stats: symbol histograms and both Adler-32 values, one CTA per patch -----------------------------
__global__ void __launch_bounds__(RL_STATS_THREADS)
residual_stats_kernel(Canvas xs, Canvas bs, int64_t batch, int H, int W, int e, int64_t* __restrict__ hist,
                      uint32_t* __restrict__ adler) {
    __shared__ uint32_t wh[RL_STATS_THREADS / 32][RL_SYMS];
    __shared__ uint64_t red[RL_STATS_THREADS / 32][4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rowb = 3 * W, q = 2 * e + 1;
    const int64_t n = (int64_t)H * rowb;
    for (int64_t t = blockIdx.x; t < batch; t += gridDim.x) {
        __syncthreads();                                     // the previous patch is done with wh / red
        for (int i = tid; i < (RL_STATS_THREADS / 32) * RL_SYMS; i += RL_STATS_THREADS) (&wh[0][0])[i] = 0;
        __syncthreads();
        const uint8_t* px = xs.patch(t, H, W);
        const uint8_t* pb = bs.patch(t, H, W);
        uint64_t ba = 0, bb = 0, oa = 0, ob = 0;
        RowWalk rw;
        rw.start(tid, rowb);
        for (int64_t i = tid; i < n; i += RL_STATS_THREADS) {
            const int a = __ldg(px + (int64_t)rw.y * xs.cols * 3 + rw.r);
            const int b = __ldg(pb + (int64_t)rw.y * bs.cols * 3 + rw.r);
            const uint32_t s = res_symbol(a, b, e, q);
            const uint32_t o = res_apply(b, s, e, q);
            const uint64_t wt = (uint64_t)(n - i);
            ba += b; bb += wt * b; oa += o; ob += wt * o;
            const unsigned act = __activemask();
            const unsigned same = __match_any_sync(act, s);
            if (lane == __ffs(same) - 1) wh[warp][s] += __popc(same);   // one lane per distinct symbol
            __syncwarp(act);
            rw.advance(RL_STATS_THREADS, rowb);
        }
        ba = warp_sum64(ba); bb = warp_sum64(bb); oa = warp_sum64(oa); ob = warp_sum64(ob);
        if (lane == 0) { red[warp][0] = ba; red[warp][1] = bb; red[warp][2] = oa; red[warp][3] = ob; }
        __syncthreads();
        uint64_t c = 0;                                      // tid = symbol
        for (int w = 0; w < RL_STATS_THREADS / 32; ++w) c += wh[w][tid];
        hist[t * RL_SYMS + tid] = (int64_t)c;
        if (tid == 0) {
            uint64_t s[4] = {0, 0, 0, 0};
            for (int w = 0; w < RL_STATS_THREADS / 32; ++w)
                for (int k = 0; k < 4; ++k) s[k] += red[w][k];
            adler[t * 2] = adler_of(s[0], s[1], n);
            adler[t * 2 + 1] = adler_of(s[2], s[3], n);
        }
    }
}

// ---- tables: packing.quantise_frequencies per patch, one CTA (256 threads = symbols) per patch ---------
__device__ int block_excl_scan(int v, int* warp_tot, int* total) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t wt;
    const int ex = (int)warp_excl_scan((uint32_t)v, &wt);
    __syncthreads();
    if (lane == 0) warp_tot[warp] = (int)wt;
    __syncthreads();
    int before = 0, all = 0;
    for (int w = 0; w < RL_SYMS / 32; ++w) {
        if (w < warp) before += warp_tot[w];
        all += warp_tot[w];
    }
    *total = all;
    return before + ex;
}

__global__ void __launch_bounds__(RL_SYMS)
residual_tables_kernel(const int64_t* __restrict__ hist, int64_t batch, int32_t* __restrict__ freq) {
    __shared__ int64_t cnt[RL_SYMS];
    __shared__ int by_rank[RL_SYMS];
    __shared__ int64_t red64[RL_SYMS / 32];
    __shared__ int warp_tot[RL_SYMS / 32];
    const int s = threadIdx.x, lane = s & 31, warp = s >> 5;
    for (int64_t t = blockIdx.x; t < batch; t += gridDim.x) {
        __syncthreads();
        const int64_t ns = hist[t * RL_SYMS + s];
        cnt[s] = ns;
        uint64_t v = warp_sum64((uint64_t)ns);
        if (lane == 0) red64[warp] = (int64_t)v;
        __syncthreads();
        int64_t total = 0;
        for (int w = 0; w < RL_SYMS / 32; ++w) total += red64[w];
        const bool present = ns > 0;
        int rank = 0;                                        // (count descending, symbol ascending)
        for (int u = 0; u < RL_SYMS; ++u) {
            const int64_t nu = cnt[u];
            rank += (nu > ns) || (nu == ns && u < s);
        }
        int64_t f = 0;
        if (present && total > 0) f = max((int64_t)1, (ns << RL_S) / total);
        int m, fsum;
        block_excl_scan(present ? 1 : 0, warp_tot, &m);
        block_excl_scan((int)f, warp_tot, &fsum);
        int d = (int)RL_M - fsum;
        if (d > 0 && present) f += d / m + (rank < d % m ? 1 : 0);
        while (d < 0) {                                      // uniform over the CTA
            by_rank[s] = 0;
            __syncthreads();
            if (present) by_rank[rank] = f > 1 ? 1 : 0;
            __syncthreads();
            int elig;
            const int before = block_excl_scan(by_rank[s], warp_tot, &elig);   // thread s: rank s
            __syncthreads();
            by_rank[s] = before;
            __syncthreads();
            const int take = min(-d, elig);
            if (present && f > 1 && by_rank[rank] < take) f -= 1;
            d += take;
            if (take == 0) break;                            // not reached: an excess implies f > 1 somewhere
            __syncthreads();
        }
        freq[t * RL_SYMS + s] = (int32_t)f;
    }
}

// ---- encode: one warp per patch ------------------------------------------------------------------------
__global__ void __launch_bounds__(RL_WARPS * 32)
residual_encode_kernel(Canvas xs, Canvas bs, int64_t batch, int H, int W, int e,
                       const int32_t* __restrict__ freq, uint8_t* __restrict__ slots, int64_t slot_bytes,
                       uint32_t* __restrict__ sizes) {
    __shared__ uint32_t fc_all[RL_WARPS][RL_SYMS];                 // f | c << 16
    __shared__ uint8_t sx_all[RL_WARPS][RL_LANES * RL_RR];
    __shared__ uint16_t wb_all[RL_WARPS][RL_LANES * RL_WSTRIDE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* fc = fc_all[warp];
    uint8_t* sx = sx_all[warp];
    uint16_t* wb = wb_all[warp];
    const int rowb = 3 * W, q = 2 * e + 1;
    const int n = H * rowb;
    const int nsteps = (n + RL_LANES - 1) / RL_LANES, rounds = (nsteps + RL_RR - 1) / RL_RR;
    const int nq = n / RL_LANES, nrem = n % RL_LANES;
    const int nj = nq + (lane < nrem ? 1 : 0);                     // this lane's symbols
    const int end_j = lane * nq + min(lane, nrem) + nj;            // end of its worst-case word region

    for (int64_t t = (int64_t)blockIdx.x * RL_WARPS + warp; t < batch; t += (int64_t)gridDim.x * RL_WARPS) {
        const uint8_t* px = xs.patch(t, H, W);
        const uint8_t* pb = bs.patch(t, H, W);
        uint8_t* slot = slots + t * slot_bytes;
        uint16_t* sw = reinterpret_cast<uint16_t*>(slot + RL_HEADER);
        // table: lane owns symbols 8 lane .. 8 lane + 7
        uint32_t f8[8], fl = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            f8[k] = (uint32_t)freq[t * RL_SYMS + lane * 8 + k];
            fl += f8[k];
        }
        uint32_t ftot;
        uint32_t c = warp_excl_scan(fl, &ftot);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            fc[lane * 8 + k] = f8[k] | (c << 16);
            reinterpret_cast<uint16_t*>(slot)[lane * 8 + k] = (uint16_t)f8[k];
            c += f8[k];
        }
        __syncwarp();

        uint32_t x = RANS_L;
        int w = 0;
        bool bad = ftot != RL_M;
        for (int r = rounds - 1; r >= 0; --r) {
            const int s0 = r * RL_RR, s1 = min(nsteps, s0 + RL_RR);
            const int64_t b0 = (int64_t)s0 * RL_LANES;
            const int nb = (int)min((int64_t)(s1 - s0) * RL_LANES, n - b0);
            RowWalk rw;
            rw.start(b0 + lane, rowb);
            for (int b = lane; b < nb; b += RL_LANES) {
                const int a = __ldg(px + (int64_t)rw.y * xs.cols * 3 + rw.r);
                const int h = __ldg(pb + (int64_t)rw.y * bs.cols * 3 + rw.r);
                sx[b] = (uint8_t)res_symbol(a, h, e, q);
                rw.advance(RL_LANES, rowb);
            }
            __syncwarp();
            int ew = 0;
            for (int st = s1 - 1; st >= s0; --st) {
                const int i = st * RL_LANES + lane;
                if (i >= n) continue;
                const uint32_t ent = fc[sx[(st - s0) * RL_LANES + lane]];
                uint32_t f = ent & 0xffffu, cs = ent >> 16;
                if (f == 0) {                                      // not encodable: keep the state valid
                    bad = true;
                    f = RL_M;
                    cs = 0;
                }
                uint16_t word;
                if (rans_encode(x, f, cs, RL_S, word)) wb[lane * RL_WSTRIDE + ew++] = word;
            }
            __syncwarp();
            for (int l = 0; l < RL_LANES; ++l) {                    // flush: lane l's words, coalesced
                const int el = __shfl_sync(0xffffffffu, ew, l), wl = __shfl_sync(0xffffffffu, w, l);
                const int endl = __shfl_sync(0xffffffffu, end_j, l);
                for (int k = lane; k < el; k += RL_LANES) sw[endl - 1 - wl - k] = wb[l * RL_WSTRIDE + k];
            }
            w += ew;
            __syncwarp();
        }
        // lanes' words [end_j - w_j, end_j) -> [pre_j, pre_j + w_j): every target lies at or below its source
        uint32_t wtot;
        const int pre = (int)warp_excl_scan((uint32_t)w, &wtot);
        for (int l = 0; l < RL_LANES; ++l) {
            const int wl = __shfl_sync(0xffffffffu, w, l), pl = __shfl_sync(0xffffffffu, pre, l);
            const int src = __shfl_sync(0xffffffffu, end_j, l) - wl;
            for (int k0 = 0; k0 < wl; k0 += RL_LANES) {
                const int k = k0 + lane;
                const uint16_t v = k < wl ? sw[src + k] : 0;
                __syncwarp();
                if (k < wl) sw[pl + k] = v;
                __syncwarp();
            }
        }
        uint32_t* hdr = reinterpret_cast<uint32_t*>(slot + 2 * RL_SYMS);
        hdr[lane] = (uint32_t)w;
        hdr[RL_LANES + lane] = x;
        const bool any_bad = __any_sync(0xffffffffu, bad);
        if (lane == 0) sizes[t] = any_bad ? 0u : (uint32_t)RL_HEADER + 2u * wtot;
        __syncwarp();
    }
}

// ---- apply: one warp per patch, decodes in place --------------------------------------------------------
struct ApplyWarpSmem {
    uint32_t f[RL_SYMS], c[RL_SYMS];
    uint8_t sym[RL_M];
    uint8_t sx[RL_LANES * RL_RR];
    uint16_t wb[RL_LANES * RL_WSTRIDE];
};

__global__ void __launch_bounds__(RL_WARPS * 32)
residual_apply_kernel(const uint8_t* __restrict__ payload, int64_t payload_bytes,
                      const int64_t* __restrict__ offsets, const uint32_t* __restrict__ adler, int64_t grid_cols,
                      int64_t lr0, int64_t lc0, int64_t lrc, int64_t lfirst, Canvas cv, int64_t batch, int H,
                      int W, int e, uint8_t* __restrict__ flags) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ApplyWarpSmem& sm = reinterpret_cast<ApplyWarpSmem*>(smem_raw)[warp];
    const int rowb = 3 * W, q = 2 * e + 1;
    const int n = H * rowb;
    const int nsteps = (n + RL_LANES - 1) / RL_LANES, rounds = (nsteps + RL_RR - 1) / RL_RR;
    const int nq = n / RL_LANES, nrem = n % RL_LANES;
    const int nj = nq + (lane < nrem ? 1 : 0);

    for (int64_t t = (int64_t)blockIdx.x * RL_WARPS + warp; t < batch; t += (int64_t)gridDim.x * RL_WARPS) {
        const int64_t lq = lfirst + t;
        const int64_t p = (lr0 + lq / lrc) * grid_cols + lc0 + lq % lrc;
        int64_t a = offsets[p], b = offsets[p + 1];
        a = min(max(a, (int64_t)0), payload_bytes);
        b = min(max(b, a), payload_bytes);
        const int64_t len = b - a;
        const uint8_t* ch = payload + a;
        auto rd8 = [&](int64_t k) -> uint32_t { return k < len ? (uint32_t)__ldg(ch + k) : 0u; };
        auto rd16 = [&](int64_t k) -> uint32_t { return rd8(k) | (rd8(k + 1) << 8); };
        auto rd32 = [&](int64_t k) -> uint32_t { return rd16(k) | (rd16(k + 2) << 16); };

        uint32_t f8[8], fl = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            f8[k] = rd16(2 * (lane * 8 + k));
            fl += f8[k];
        }
        uint32_t ftot;
        uint32_t c = warp_excl_scan(fl, &ftot);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            sm.f[lane * 8 + k] = f8[k];
            sm.c[lane * 8 + k] = c;
            c += f8[k];
        }
        __syncwarp();
        for (uint32_t slot = lane; slot < RL_M; slot += RL_LANES) {   // largest s with c[s] <= slot
            int lo = 0, hi = RL_SYMS - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (sm.c[mid] <= slot) lo = mid; else hi = mid - 1;
            }
            sm.sym[slot] = (uint8_t)lo;
        }
        const uint32_t w_raw = rd32(2 * RL_SYMS + 4 * lane);
        uint32_t x = rd32(2 * RL_SYMS + 4 * RL_LANES + 4 * lane);
        const int wj = (int)min(w_raw, (uint32_t)nj);
        uint32_t wsum;
        const int pre = (int)warp_excl_scan((uint32_t)wj, &wsum);
        uint64_t wraw_sum = w_raw;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) wraw_sum += __shfl_xor_sync(0xffffffffu, wraw_sum, d);
        __syncwarp();

        uint8_t* pc = cv.patch(t, H, W);
        uint64_t ba = 0, bb = 0, oa = 0, ob = 0;
        int k = 0;                                                   // words consumed by this lane
        for (int r = 0; r < rounds; ++r) {
            const int s0 = r * RL_RR, s1 = min(nsteps, s0 + RL_RR);
            const int64_t b0 = (int64_t)s0 * RL_LANES;
            const int nb = (int)min((int64_t)(s1 - s0) * RL_LANES, n - b0);
            RowWalk rw;
            rw.start(b0 + lane, rowb);
            for (int bi = lane; bi < nb; bi += RL_LANES) {
                const uint32_t h = pc[(int64_t)rw.y * cv.cols * 3 + rw.r];
                sm.sx[bi] = (uint8_t)h;
                const uint64_t wt = (uint64_t)(n - (b0 + bi));
                ba += h; bb += wt * h;
                rw.advance(RL_LANES, rowb);
            }
            for (int l = 0; l < RL_LANES; ++l) {                    // the next RR words of every lane
                const int kl = __shfl_sync(0xffffffffu, k, l), wl = __shfl_sync(0xffffffffu, wj, l);
                const int pl = __shfl_sync(0xffffffffu, pre, l);
                for (int u = lane; u < RL_RR; u += RL_LANES) {
                    const int idx = kl + u;
                    sm.wb[l * RL_WSTRIDE + u] =
                        idx < wl ? (uint16_t)rd16(RL_HEADER + 2 * ((int64_t)pl + idx)) : (uint16_t)0;
                }
            }
            __syncwarp();
            const int k0 = k;
            for (int st = s0; st < s1; ++st) {
                const int i = st * RL_LANES + lane;
                if (i >= n) break;
                const uint32_t slot = x & (RL_M - 1);
                const uint32_t s = sm.sym[slot];
                x = sm.f[s] * (x >> RL_S) + slot - sm.c[s];
                if (x < RANS_L) {                                    // at most one word per step: k - k0 < RR
                    x = (x << 16) | sm.wb[lane * RL_WSTRIDE + (k - k0)];
                    ++k;
                }
                uint8_t& v = sm.sx[(st - s0) * RL_LANES + lane];
                v = (uint8_t)res_apply(v, s, e, q);
            }
            __syncwarp();
            rw.start(b0 + lane, rowb);
            for (int bi = lane; bi < nb; bi += RL_LANES) {
                const uint32_t o = sm.sx[bi];
                pc[(int64_t)rw.y * cv.cols * 3 + rw.r] = (uint8_t)o;
                const uint64_t wt = (uint64_t)(n - (b0 + bi));
                oa += o; ob += wt * o;
                rw.advance(RL_LANES, rowb);
            }
            __syncwarp();
        }
        ba = warp_sum64(ba); bb = warp_sum64(bb); oa = warp_sum64(oa); ob = warp_sum64(ob);
        const bool lane_bad = x != RANS_L || (uint32_t)k != w_raw;
        const bool stream_bad = __any_sync(0xffffffffu, lane_bad) || ftot != RL_M || len < RL_HEADER ||
                                len != RL_HEADER + 2 * (int64_t)wraw_sum;
        if (lane == 0) {
            const bool base_bad = adler_of(ba, bb, n) != adler[p * 2];
            const bool out_bad = adler_of(oa, ob, n) != adler[p * 2 + 1];
            flags[t] = (uint8_t)((stream_bad ? 1 : 0) | (base_bad ? 2 : 0) | (out_bad ? 4 : 0));
        }
        __syncwarp();
    }
}

inline size_t align256r(size_t v) { return (v + 255) & ~(size_t)255; }
inline int64_t chunk_worst(int H, int W) { return RL_HEADER + 2 * (int64_t)H * W * 3; }
inline int64_t slot_bytes_r(int H, int W) { return (chunk_worst(H, W) + 15) & ~(int64_t)15; }

// placement of a batch of H x W patches inside a canvas [rows, cols, 3] (VQAE_OK / VQAE_ERR_BAD_ARG)
int check_canvas(const uint8_t* p, int64_t rows, int64_t cols, int64_t r0, int64_t c0, int64_t rc, int64_t first,
                 int64_t batch, int H, int W) {
    if (!p || rows <= 0 || cols <= 0 || r0 < 0 || c0 < 0 || rc <= 0 || first < 0) return VQAE_ERR_BAD_ARG;
    const int64_t last = first + batch - 1;
    if ((r0 + last / rc + 1) * H > rows || (c0 + rc) * W > cols) return VQAE_ERR_BAD_ARG;
    return VQAE_OK;
}

int check_shape(int64_t batch, int H, int W, int e) {
    if (batch <= 0 || H <= 0 || W <= 0 || e < 0) return VQAE_ERR_BAD_ARG;
    if ((int64_t)H * W > RL_MAX_PIXELS || e > 127) return VQAE_ERR_UNSUPPORTED;
    return VQAE_OK;
}

int grid_cap(int per_sm, int64_t units, unsigned* grid) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    const int64_t cap = (int64_t)sm_count * per_sm;
    *grid = (unsigned)(units < cap ? units : cap);
    return VQAE_OK;
}

}  // namespace

int residual_stats(const uint8_t* x, int64_t x_rows, int64_t x_cols, int64_t x_r0, int64_t x_c0, int64_t x_rc,
                   int64_t x_first, const uint8_t* base, int64_t b_rows, int64_t b_cols, int64_t b_r0, int64_t b_c0,
                   int64_t b_rc, int64_t b_first, int64_t batch, int H, int W, int e, int64_t* hist,
                   uint32_t* adler, cudaStream_t stream) {
    if (!hist || !adler) return VQAE_ERR_BAD_ARG;
    if (int rc = check_shape(batch, H, W, e)) return rc;
    if (int rc = check_canvas(x, x_rows, x_cols, x_r0, x_c0, x_rc, x_first, batch, H, W)) return rc;
    if (int rc = check_canvas(base, b_rows, b_cols, b_r0, b_c0, b_rc, b_first, batch, H, W)) return rc;
    if (x_first + batch - 1 > 0x7fffffff || b_first + batch - 1 > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    unsigned grid;
    if (int rc = grid_cap(8, batch, &grid)) return rc;
    const Canvas a{const_cast<uint8_t*>(x), x_cols, x_r0, x_c0, x_rc, x_first};
    const Canvas b{const_cast<uint8_t*>(base), b_cols, b_r0, b_c0, b_rc, b_first};
    residual_stats_kernel<<<grid, RL_STATS_THREADS, 0, stream>>>(a, b, batch, H, W, e, hist, adler);
    return check_launch();
}

int residual_tables(const int64_t* hist, int64_t batch, int32_t* freq, cudaStream_t stream) {
    if (!hist || !freq || batch <= 0) return VQAE_ERR_BAD_ARG;
    unsigned grid;
    if (int rc = grid_cap(8, batch, &grid)) return rc;
    residual_tables_kernel<<<grid, RL_SYMS, 0, stream>>>(hist, batch, freq);
    return check_launch();
}

size_t residual_encode_scratch_bytes(int64_t batch, int H, int W) {
    if (check_shape(batch, H, W, 0)) return 0;
    return align256r((size_t)batch * slot_bytes_r(H, W)) + align256r((size_t)batch * sizeof(uint32_t));
}

int residual_encode(const uint8_t* x, int64_t x_rows, int64_t x_cols, int64_t x_r0, int64_t x_c0, int64_t x_rc,
                    int64_t x_first, const uint8_t* base, int64_t b_rows, int64_t b_cols, int64_t b_r0,
                    int64_t b_c0, int64_t b_rc, int64_t b_first, int64_t batch, int H, int W, int e,
                    const int32_t* freq, int64_t* offsets, uint8_t* payload, int64_t payload_capacity,
                    void* scratch, size_t scratch_bytes, cudaStream_t stream) {
    if (!freq || !offsets || !payload) return VQAE_ERR_BAD_ARG;
    if (int rc = check_shape(batch, H, W, e)) return rc;
    if (int rc = check_canvas(x, x_rows, x_cols, x_r0, x_c0, x_rc, x_first, batch, H, W)) return rc;
    if (int rc = check_canvas(base, b_rows, b_cols, b_r0, b_c0, b_rc, b_first, batch, H, W)) return rc;
    if (x_first + batch - 1 > 0x7fffffff || b_first + batch - 1 > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    if (payload_capacity < batch * chunk_worst(H, W)) return VQAE_ERR_BAD_ARG;
    if (!scratch || scratch_bytes < residual_encode_scratch_bytes(batch, H, W)) return VQAE_ERR_SCRATCH;
    const int64_t sb = slot_bytes_r(H, W);
    uint8_t* slots = static_cast<uint8_t*>(scratch);
    uint32_t* sizes = reinterpret_cast<uint32_t*>(slots + align256r((size_t)batch * sb));
    unsigned grid;
    if (int rc = grid_cap(8, (batch + RL_WARPS - 1) / RL_WARPS, &grid)) return rc;
    const Canvas a{const_cast<uint8_t*>(x), x_cols, x_r0, x_c0, x_rc, x_first};
    const Canvas b{const_cast<uint8_t*>(base), b_cols, b_r0, b_c0, b_rc, b_first};
    residual_encode_kernel<<<grid, RL_WARPS * 32, 0, stream>>>(a, b, batch, H, W, e, freq, slots, sb, sizes);
    if (int rc = check_launch()) return rc;
    return rans_offsets_and_compact(sizes, batch, slots, sb, offsets, payload, payload_capacity, stream);
}

int residual_apply(const uint8_t* payload, int64_t payload_bytes, const int64_t* offsets_host,
                   const int64_t* offsets, const uint32_t* adler, int64_t grid_rows, int64_t grid_cols,
                   int64_t l_r0, int64_t l_c0, int64_t l_rc, int64_t l_first, uint8_t* canvas, int64_t rows,
                   int64_t cols, int64_t r0, int64_t c0, int64_t rc_, int64_t first, int64_t batch, int H, int W,
                   int e, uint8_t* flags, cudaStream_t stream) {
    if (!payload || !offsets_host || !offsets || !adler || !flags) return VQAE_ERR_BAD_ARG;
    if (int rc = check_shape(batch, H, W, e)) return rc;
    if (int rc = check_canvas(canvas, rows, cols, r0, c0, rc_, first, batch, H, W)) return rc;
    if (grid_rows <= 0 || grid_cols <= 0 || l_r0 < 0 || l_c0 < 0 || l_rc <= 0 || l_first < 0) return VQAE_ERR_BAD_ARG;
    if (l_r0 + (l_first + batch - 1) / l_rc + 1 > grid_rows || l_c0 + l_rc > grid_cols) return VQAE_ERR_BAD_ARG;
    if (first + batch - 1 > 0x7fffffff || l_first + batch - 1 > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    const int64_t P = grid_rows * grid_cols, worst = chunk_worst(H, W);
    if (offsets_host[0] != 0 || offsets_host[P] != payload_bytes) return VQAE_ERR_BAD_ARG;
    for (int64_t p = 0; p < P; ++p) {
        const int64_t len = offsets_host[p + 1] - offsets_host[p];
        if (len < RL_HEADER || len > worst || (len & 1)) return VQAE_ERR_BAD_ARG;
    }
    unsigned grid;
    if (int rc = grid_cap(3, (batch + RL_WARPS - 1) / RL_WARPS, &grid)) return rc;
    const size_t smem = RL_WARPS * sizeof(ApplyWarpSmem);
    VQAE_CUDA_TRY(cudaFuncSetAttribute(residual_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const Canvas cv{canvas, cols, r0, c0, rc_, first};
    residual_apply_kernel<<<grid, RL_WARPS * 32, smem, stream>>>(payload, payload_bytes, offsets, adler, grid_cols,
                                                                 l_r0, l_c0, l_rc, l_first, cv, batch, H, W, e,
                                                                 flags);
    return check_launch();
}

}  // namespace vqae

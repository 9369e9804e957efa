// Box-filtered overview levels of uint8 RGB patches (include/vqae_b200.h, vqae_pyramid_u8).
//
// Level k (factor f = 2^k, 1 <= k <= 9, f dividing the patch height H and width W): per channel,
//     out = (S + f^2 / 2) >> 2k,   S = the exact integer sum of the f x f source pixels,
// the box mean rounded half up -- PIL.Image.reduce(f).  Every level is rounded once, from the exact
// sum of the original pixels; no level is derived from a rounded one.
//
// Work unit: a T x T square of one patch, T = the largest power of two <= 64 that divides H and W
// (T >= min(2^k_max, 64) because 2^k_max divides both).  The CTA reads the square once (16-byte loads
// when the canvas allows), forms the exact 2 x 2 sums in shared memory and from them, level by level,
// the 2^j x 2^j sums for j <= log2 T, writing each requested level as it goes.  Levels coarser than 64
// need sums across units: each unit then stores its three 64 x 64 sums to scratch [n, H/64, W/64, 3]
// and pyramid_coarse_kernel adds (f/64)^2 of them per output pixel.  Sums are uint32 (512^2 * 255 <
// 2^32), integer arithmetic throughout and no atomics: the result depends on the pixels only, not on
// the batch, the grid or a patch's position, so it is bitwise reproducible.  Canvas offsets are 64-bit.
#include "common.cuh"
#include "kernels.cuh"

namespace vqae {

constexpr int PY_THREADS = 128;
constexpr int PY_MAX_T = 64;                  // the largest square a unit stages (level 6)
constexpr int PY_MIN_CTAS = 6;
constexpr int PY_CHUNK = 16;                  // pixels per 16-byte-load item (3 x 16 B per row)
constexpr int PY_LEVELS = 10;                // k = 0 .. 9 (k = 0 unused)

struct PyrSrc {                               // patch t at grid (r0 + q / rc, c0 + q % rc), q = first + t,
    const uint8_t* p;                         // of a canvas uint8 [rows, cols, 3]
    int64_t cols, r0, c0, rc, first;
};
struct PyrDst {                               // level k: canvas p[k] with cols[k] pixels per row
    uint8_t* p[PY_LEVELS];
    int64_t cols[PY_LEVELS];
    int64_t r0, c0, rc, first;
};

// byte offset of pixel (y, x) of patch t in a canvas of `cols` pixels per row with h x w patches
static __device__ __forceinline__ int64_t patch_px(int64_t t, int64_t first, int64_t r0, int64_t c0,
                                                   int64_t rc, int64_t cols, int h, int w, int y, int x) {
    const int64_t q = first + t;
    const int64_t pr = r0 + q / rc, pc = c0 + q % rc;
    return ((pr * h + y) * cols + pc * w + x) * 3;
}

static __device__ __forceinline__ uint32_t byte_of(const uint4& v, int n) {
    const uint32_t w = n < 4 ? v.x : n < 8 ? v.y : n < 12 ? v.z : v.w;
    return (w >> (8 * (n & 3))) & 0xffu;
}

// level j's sums of one unit (n x n pixels, 3 channels) from level j - 1's (2n x 2n) in shared memory;
// writes the level when requested
static __device__ __forceinline__ void pyr_level(const uint32_t* __restrict__ prev, uint32_t* __restrict__ cur,
                                                 int n, int j, bool emit, uint8_t* __restrict__ dst,
                                                 int64_t dst_cols) {
    const int n2 = 2 * n;
    const uint32_t half = 1u << (2 * j - 1);
    for (int i = threadIdx.x; i < n * n * 3; i += PY_THREADS) {
        const int c = i % 3, px = i / 3, y = px / n, x = px - y * n;
        const uint32_t* a = prev + ((2 * y) * n2 + 2 * x) * 3 + c;
        const uint32_t s = a[0] + a[3] + a[n2 * 3] + a[n2 * 3 + 3];
        cur[i] = s;
        if (emit) dst[(int64_t)y * dst_cols * 3 + x * 3 + c] = (uint8_t)((s + half) >> (2 * j));
    }
}

__global__ void __launch_bounds__(PY_THREADS, PY_MIN_CTAS)
pyramid_tiles_kernel(PyrSrc src, PyrDst dst, int64_t units, int H, int W, int T, int top, int mask,
                     int vec, uint32_t* __restrict__ scratch) {
    __shared__ uint32_t buf_a[(PY_MAX_T / 2) * (PY_MAX_T / 2) * 3];   // levels 1, 3, 5
    __shared__ uint32_t buf_b[(PY_MAX_T / 4) * (PY_MAX_T / 4) * 3];   // levels 2, 4, 6
    const int tpr = W / T, tiles = (H / T) * tpr;
    const int n1 = T / 2;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int64_t t = u / tiles;
        const int tile = (int)(u - t * tiles);
        const int ty = (tile / tpr) * T, tx = (tile % tpr) * T;      // the unit's origin in the patch
        const uint8_t* sp = src.p + patch_px(t, src.first, src.r0, src.c0, src.rc, src.cols, H, W, ty, tx);
        const int64_t srow = src.cols * 3;

        __syncthreads();                       // the previous unit is done with buf_a / buf_b
        // level 1: exact 2 x 2 sums of the staged square
        if (vec) {                             // item: 2 rows x 16 pixels (3 x 16 B each) -> 8 sums x 3
            const int cpr = T / PY_CHUNK;
            for (int i = threadIdx.x; i < n1 * cpr; i += PY_THREADS) {
                const int y = i / cpr, ch = i - y * cpr;
                const uint4* ra = reinterpret_cast<const uint4*>(sp + (int64_t)(2 * y) * srow + ch * PY_CHUNK * 3);
                const uint4* rb = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(ra) + srow);
                uint4 a[3], b[3];
#pragma unroll
                for (int q = 0; q < 3; ++q) { a[q] = __ldg(ra + q); b[q] = __ldg(rb + q); }
                uint32_t* o = buf_a + (y * n1 + ch * (PY_CHUNK / 2)) * 3;
#pragma unroll
                for (int m = 0; m < PY_CHUNK * 3 / 2; ++m) {        // output byte m: pixel m / 3, channel m % 3
                    const int n0 = (m / 3) * 6 + m % 3;             // source bytes n0, n0 + 3 of both rows
                    o[m] = byte_of(a[n0 / 16], n0 % 16) + byte_of(a[(n0 + 3) / 16], (n0 + 3) % 16) +
                           byte_of(b[n0 / 16], n0 % 16) + byte_of(b[(n0 + 3) / 16], (n0 + 3) % 16);
                }
            }
        } else {                               // item: one 2 x 2 block, byte loads
            for (int i = threadIdx.x; i < n1 * n1; i += PY_THREADS) {
                const int y = i / n1, x = i - y * n1;
                const uint8_t* pa = sp + (int64_t)(2 * y) * srow + 2 * x * 3;
                const uint8_t* pb = pa + srow;
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    buf_a[i * 3 + c] = (uint32_t)__ldg(pa + c) + __ldg(pa + 3 + c) + __ldg(pb + c) + __ldg(pb + 3 + c);
            }
        }
        __syncthreads();
        // the requested levels j <= top; level j + 1 is summed from level j.  Unrolled so that dst.p[j]
        // and dst.cols[j] are constant indices (no copy of the parameters to local memory)
        if ((mask >> 1) & 1) {
            uint8_t* d = dst.p[1] + patch_px(t, dst.first, dst.r0, dst.c0, dst.rc, dst.cols[1], H >> 1, W >> 1,
                                             ty >> 1, tx >> 1);
            for (int i = threadIdx.x; i < n1 * n1 * 3; i += PY_THREADS) {
                const int px = i / 3, y = px / n1, x = px - y * n1;
                d[(int64_t)y * dst.cols[1] * 3 + x * 3 + i % 3] = (uint8_t)((buf_a[i] + 2u) >> 2);
            }
        }
        uint32_t* cur = buf_a;
        uint32_t* nxt = buf_b;
#pragma unroll
        for (int j = 2; j <= 6; ++j) {
            if (j > top) break;
            const bool emit = (mask >> j) & 1;
            uint8_t* d = emit ? dst.p[j] + patch_px(t, dst.first, dst.r0, dst.c0, dst.rc, dst.cols[j], H >> j,
                                                    W >> j, ty >> j, tx >> j)
                              : nullptr;
            pyr_level(cur, nxt, T >> j, j, emit, d, dst.cols[j]);
            __syncthreads();
            uint32_t* s = cur; cur = nxt; nxt = s;
        }
        // levels coarser than 64: this unit's three 64 x 64 sums (top == 6, cur holds 1 x 1 x 3)
        if (mask >> 7 && threadIdx.x < 3) {
            const int64_t g = (t * (H / PY_MAX_T) + ty / PY_MAX_T) * (W / PY_MAX_T) + tx / PY_MAX_T;
            scratch[g * 3 + threadIdx.x] = cur[threadIdx.x];
        }
    }
}

// levels 7 .. 9 (blockIdx.y = k - 7): output pixel = (f/64)^2 unit sums from scratch, rounded once
__global__ void __launch_bounds__(PY_THREADS)
pyramid_coarse_kernel(const uint32_t* __restrict__ scratch, PyrDst dst, int64_t batch, int H, int W, int mask) {
    const int k = 7 + blockIdx.y;
    if (!((mask >> k) & 1)) return;
    const int f = 1 << k, m = f / PY_MAX_T, gh = H / PY_MAX_T, gw = W / PY_MAX_T;
    const int oh = H / f, ow = W / f;
    const int64_t i = (int64_t)blockIdx.x * PY_THREADS + threadIdx.x;
    if (i >= batch * oh * ow) return;
    const int64_t t = i / (oh * ow);
    const int px = (int)(i - t * oh * ow), oy = px / ow, ox = px - oy * ow;
    uint32_t s0 = 0, s1 = 0, s2 = 0;
    for (int r = 0; r < m; ++r) {
        const uint32_t* row = scratch + ((t * gh + oy * m + r) * gw + ox * m) * 3;
        for (int x = 0; x < m; ++x) { s0 += row[3 * x]; s1 += row[3 * x + 1]; s2 += row[3 * x + 2]; }
    }
    uint8_t* const p = k == 7 ? dst.p[7] : k == 8 ? dst.p[8] : dst.p[9];        // constant indices
    const int64_t cols = k == 7 ? dst.cols[7] : k == 8 ? dst.cols[8] : dst.cols[9];
    uint8_t* d = p + patch_px(t, dst.first, dst.r0, dst.c0, dst.rc, cols, oh, ow, oy, ox);
    const uint32_t half = 1u << (2 * k - 1);
    d[0] = (uint8_t)((s0 + half) >> (2 * k));
    d[1] = (uint8_t)((s1 + half) >> (2 * k));
    d[2] = (uint8_t)((s2 + half) >> (2 * k));
}

static size_t align256p(size_t v) { return (v + 255) & ~(size_t)255; }

static bool pyramid_shape_ok(int H, int W, int mask) {
    if (mask <= 0 || (mask & ~0x3fe)) return false;               // bits 1 .. 9 only
    for (int k = 1; k < PY_LEVELS; ++k)
        if (((mask >> k) & 1) && ((H % (1 << k)) || (W % (1 << k)))) return false;
    return true;
}

size_t pyramid_u8_scratch_bytes(int64_t batch, int H, int W, int mask) {
    if (batch <= 0 || H <= 0 || W <= 0 || !pyramid_shape_ok(H, W, mask) || !(mask >> 7)) return 0;
    return align256p((size_t)batch * (H / PY_MAX_T) * (W / PY_MAX_T) * 3 * sizeof(uint32_t));
}

// a batch of h x w patches at (r0 + (first + t) / rc, c0 + (first + t) % rc) inside a canvas
// [rows, cols, 3]; first + batch <= 2^31 is checked before, so nothing here overflows
static bool placement_ok(int64_t rows, int64_t cols, int64_t r0, int64_t c0, int64_t rc, int64_t first,
                         int64_t batch, int h, int w) {
    if (rows <= 0 || cols <= 0 || r0 < 0 || c0 < 0 || rc <= 0) return false;
    const int64_t gr = rows / h, gc = cols / w;                  // whole patches the canvas holds
    return r0 < gr && (first + batch - 1) / rc < gr - r0 && c0 < gc && rc <= gc - c0;
}

int pyramid_u8(const uint8_t* src, int64_t src_rows, int64_t src_cols, int64_t src_r0, int64_t src_c0,
               int64_t src_rc, int64_t src_first, int64_t batch, int H, int W, int mask,
               uint8_t* const* dst, const int64_t* dst_rows, const int64_t* dst_cols, int64_t dst_r0,
               int64_t dst_c0, int64_t dst_rc, int64_t dst_first, void* scratch, size_t scratch_bytes,
               cudaStream_t stream) {
    if (!src || !dst || !dst_rows || !dst_cols || batch <= 0 || H <= 0 || W <= 0 || mask == 0 ||
        src_first < 0 || dst_first < 0)
        return VQAE_ERR_BAD_ARG;
    if (mask & ~0x3fe) return VQAE_ERR_UNSUPPORTED;
    for (int k = 1; k < PY_LEVELS; ++k)
        if (((mask >> k) & 1) && !dst[k]) return VQAE_ERR_BAD_ARG;
    if (!pyramid_shape_ok(H, W, mask)) return VQAE_ERR_UNSUPPORTED;
    if (src_first > 0x7fffffff - batch + 1 || dst_first > 0x7fffffff - batch + 1) return VQAE_ERR_UNSUPPORTED;
    if (!placement_ok(src_rows, src_cols, src_r0, src_c0, src_rc, src_first, batch, H, W)) return VQAE_ERR_BAD_ARG;
    PyrDst d{};
    for (int k = 1; k < PY_LEVELS; ++k) {
        if (!((mask >> k) & 1)) continue;
        if (!placement_ok(dst_rows[k], dst_cols[k], dst_r0, dst_c0, dst_rc, dst_first, batch, H >> k, W >> k))
            return VQAE_ERR_BAD_ARG;
        d.p[k] = dst[k];
        d.cols[k] = dst_cols[k];
    }
    d.r0 = dst_r0; d.c0 = dst_c0; d.rc = dst_rc; d.first = dst_first;
    const size_t need = pyramid_u8_scratch_bytes(batch, H, W, mask);
    if (need && (!scratch || scratch_bytes < need)) return VQAE_ERR_SCRATCH;
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;

    int log_t = 0;                                               // T = 2^log_t: 64 or the 2-power of H, W
    while (log_t < 6 && H % (2 << log_t) == 0 && W % (2 << log_t) == 0) ++log_t;
    const int T = 1 << log_t;
    int kmax = 9;
    while (!((mask >> kmax) & 1)) --kmax;
    const int top = kmax < log_t ? kmax : log_t;                 // the last level a unit sums
    const PyrSrc s{src, src_cols, src_r0, src_c0, src_rc, src_first};
    // 16-byte loads: each 16-pixel chunk of a row starts on a 16-byte boundary
    const int vec = T >= PY_CHUNK && (reinterpret_cast<uintptr_t>(src) & 15) == 0 && src_cols % 16 == 0;
    const int64_t units = batch * (H / T) * (W / T);
    const int64_t cap = (int64_t)sm_count * PY_MIN_CTAS;
    const unsigned grid = (unsigned)(units < cap ? units : cap);
    pyramid_tiles_kernel<<<grid, PY_THREADS, 0, stream>>>(s, d, units, H, W, T, top, mask, vec,
                                                          reinterpret_cast<uint32_t*>(scratch));
    if (int rc = check_launch()) return rc;
    if (!(mask >> 7)) return VQAE_OK;
    const int64_t most = batch * (H / 128) * (W / 128);          // level 7 has the most pixels
    pyramid_coarse_kernel<<<dim3(ceil_div_u(most, PY_THREADS), 3), PY_THREADS, 0, stream>>>(
        reinterpret_cast<const uint32_t*>(scratch), d, batch, H, W, mask);
    return check_launch();
}

}  // namespace vqae

// Reconstruction quality of uint8 RGB patches: exact per-channel SSE and the mean SSIM of each patch
// (include/vqae_b200.h, vqae_quality_u8).
//
// SSIM (Wang et al. 2004) as skimage.metrics.structural_similarity(gaussian_weights=True, sigma=1.5,
// use_sample_covariance=False, data_range=255, channel_axis=-1) defines it: per channel, 11 x 11
// Gaussian window w = g g^T (g: 11 taps, sigma 1.5, normalised to sum 1 in float64, rounded once to
// fp32), population moments
//     mu_x = sum w x,  s_xx = sum w x^2 - mu_x^2,  s_yy likewise,  s_xy = sum w x y - mu_x mu_y,
//     ssim = (2 mu_x mu_y + C1)(2 s_xy + C2) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)),
// C1 = (0.01 * 255)^2, C2 = (0.03 * 255)^2, averaged over the 3 channels and the (H - 10)(W - 10) window
// positions that lie inside the patch.
//
// Work unit: a QT_Y x QT_X tile of window positions of one patch plus the pixels it owns for the SSE
// (rows [oy0, oy0 + QT_Y), the last tile row of a patch also owns the 10 rows below it; columns alike),
// so every pixel is counted once and every window position once for any H, W >= 11.  The CTA stages
// the tile's halo (QT_Y + 10) x (QT_X + 10) of both images as uint8 in shared memory, then per channel
// runs the horizontal 11-tap pass for the five moments into shared memory and the vertical pass from
// there, evaluating SSIM at each position.  Nothing image-sized reaches global memory: one SSIM partial
// and three SSE partials per (patch, tile) go to scratch, and quality_finish_kernel sums them per patch
// in tile order.  A patch's result depends on its pixels only -- not on its place in the batch, the
// batch size or the grid -- and no atomics are involved, so results are bitwise reproducible.
//
// Accuracy: the moments are accumulated in fp64.  s_xx = E[x^2] - mu_x^2 cancels: in fp32, even with
// a per-tile shift subtracted from the pixels (which makes a flat tile exact), the flat part of a tile
// that straddles a flat / textured edge keeps pixels up to d = 255 levels away from the shift, and 22
// fp32 roundings of sums near d^2 = 65025 leave |error| in s_xx up to ~22 * 2^-24 * d^2 ~ 0.09 against
// C2 = 58.5, i.e. ~1e-3 of that window's SSIM and ~1e-4 of a patch mean when an eighth of its tiles
// straddle such an edge.  In fp64 the products w * x^2 (24 + 16 significant bits) are exact and each sum
// rounds at 2^-53 relative: |error| in s_xx stays below 65025 * 30 * 2^-53 < 3e-10, 5e-12 of C2, with
// no shift needed.  B200 runs fp64 FMAs at half the fp32 rate; the kernel stays CUDA-core bound.
#include "common.cuh"
#include "kernels.cuh"

#include <cmath>

namespace vqae {

constexpr int QT_X = 32, QT_Y = 16;                    // window positions per tile
constexpr int QT_R = 5, QT_TAPS = 2 * QT_R + 1;        // 11-tap window
constexpr int QT_HX = QT_X + 2 * QT_R, QT_HY = QT_Y + 2 * QT_R;
constexpr int QT_THREADS = 256;
constexpr int QT_MIN_CTAS = 3;
constexpr int QT_HG = 4;                               // output columns per horizontal-pass item
constexpr int QT_VG = QT_Y / (QT_THREADS / QT_X);      // output rows per vertical-pass item (2)
static_assert(QT_X % QT_HG == 0 && QT_THREADS % QT_X == 0 && QT_Y % (QT_THREADS / QT_X) == 0, "tiling");

struct QualityImage {                 // patch t of the call: grid position (r0 + q / rc, c0 + q % rc),
    const uint8_t* p;                 // q = first + t, of a canvas uint8 [rows, cols, 3]
    int64_t cols, r0, c0, rc, first;
    __device__ const uint8_t* patch(int64_t t, int H, int W) const {
        const int64_t q = first + t;
        const int64_t pr = r0 + q / rc, pc = c0 + q % rc;
        return p + ((pr * H) * cols + pc * W) * 3;
    }
};
struct QualityWeights { float w[QT_TAPS]; };

static __device__ __forceinline__ double ssim_at(double mx, double my, double exx, double eyy, double exy) {
    constexpr double C1 = (0.01 * 255) * (0.01 * 255), C2 = (0.03 * 255) * (0.03 * 255);
    const double sxx = exx - mx * mx, syy = eyy - my * my, sxy = exy - mx * my;
    return ((2.0 * mx * my + C1) * (2.0 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2));
}

__global__ void __launch_bounds__(QT_THREADS, QT_MIN_CTAS)
quality_ssim_tiles_kernel(QualityImage ref, QualityImage rec, int64_t units, int H, int W, int ntx,
                          int tiles, QualityWeights wt, double* __restrict__ ssim_part,
                          uint32_t* __restrict__ sse_part) {
    __shared__ uint8_t sx[QT_HY * QT_HX * 3], sy[QT_HY * QT_HX * 3];
    __shared__ double hm[5][QT_HY][QT_X];             // horizontal pass: x, y, x^2, y^2, x y
    __shared__ double red_s[QT_THREADS / 32];
    __shared__ uint32_t red_e[QT_THREADS / 32][3];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Hv = H - 2 * QT_R, Wv = W - 2 * QT_R;    // valid window positions
    double w[QT_TAPS];
#pragma unroll
    for (int k = 0; k < QT_TAPS; ++k) w[k] = (double)wt.w[k];

    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int64_t t = u / tiles;
        const int tile = (int)(u - t * tiles);
        const int ty = tile / ntx, tx = tile - ty * ntx;
        const int oy0 = ty * QT_Y, ox0 = tx * QT_X;
        const int ny = min(QT_Y, Hv - oy0), nx = min(QT_X, Wv - ox0);
        const int hy = ny + 2 * QT_R, hx = nx + 2 * QT_R;
        // pixels this tile owns for the SSE (relative to (oy0, ox0))
        const int own_y = oy0 + QT_Y >= Hv ? H - oy0 : QT_Y;
        const int own_x = ox0 + QT_X >= Wv ? W - ox0 : QT_X;
        const uint8_t* pa = ref.patch(t, H, W) + ((int64_t)oy0 * ref.cols + ox0) * 3;
        const uint8_t* pb = rec.patch(t, H, W) + ((int64_t)oy0 * rec.cols + ox0) * 3;

        __syncthreads();                               // the previous unit is done with sx / sy / hm
        uint32_t e0 = 0, e1 = 0, e2 = 0;
        for (int i = tid; i < QT_HY * QT_HX; i += QT_THREADS) {
            const int r = i / QT_HX, c = i - r * QT_HX;
            uint8_t a0 = 0, a1 = 0, a2 = 0, b0 = 0, b1 = 0, b2 = 0;
            if (r < hy && c < hx) {
                const uint8_t* qa = pa + ((int64_t)r * ref.cols + c) * 3;
                const uint8_t* qb = pb + ((int64_t)r * rec.cols + c) * 3;
                a0 = __ldg(qa); a1 = __ldg(qa + 1); a2 = __ldg(qa + 2);
                b0 = __ldg(qb); b1 = __ldg(qb + 1); b2 = __ldg(qb + 2);
                if (r < own_y && c < own_x) {
                    const int d0 = a0 - b0, d1 = a1 - b1, d2 = a2 - b2;
                    e0 += d0 * d0; e1 += d1 * d1; e2 += d2 * d2;
                }
            }
            sx[i * 3] = a0; sx[i * 3 + 1] = a1; sx[i * 3 + 2] = a2;
            sy[i * 3] = b0; sy[i * 3 + 1] = b1; sy[i * 3 + 2] = b2;
        }
        double acc = 0.0;                              // this thread's SSIM sum, fixed order
        for (int ch = 0; ch < 3; ++ch) {
            __syncthreads();                           // staging done / previous channel's vertical pass done
            // horizontal pass: item = (halo row r, QT_HG output columns)
            for (int i = tid; i < QT_HY * (QT_X / QT_HG); i += QT_THREADS) {
                const int r = i / (QT_X / QT_HG), c0 = (i - r * (QT_X / QT_HG)) * QT_HG;
                if (r >= hy || c0 >= nx) continue;
                double m[5][QT_HG];
#pragma unroll
                for (int o = 0; o < QT_HG; ++o)
#pragma unroll
                    for (int q = 0; q < 5; ++q) m[q][o] = 0.0;
#pragma unroll
                for (int k = 0; k < QT_HG + 2 * QT_R; ++k) {
                    const int s = (r * QT_HX + c0 + k) * 3 + ch;
                    const double x = (double)sx[s], y = (double)sy[s];
                    const double xx = x * x, yy = y * y, xy = x * y;
#pragma unroll
                    for (int o = 0; o < QT_HG; ++o) {
                        const int j = k - o;
                        if (j >= 0 && j < QT_TAPS) {
                            m[0][o] = fma(w[j], x, m[0][o]);
                            m[1][o] = fma(w[j], y, m[1][o]);
                            m[2][o] = fma(w[j], xx, m[2][o]);
                            m[3][o] = fma(w[j], yy, m[3][o]);
                            m[4][o] = fma(w[j], xy, m[4][o]);
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < 5; ++q)
#pragma unroll
                    for (int o = 0; o < QT_HG; ++o) hm[q][r][c0 + o] = m[q][o];
            }
            __syncthreads();
            // vertical pass: item = (output column, QT_VG output rows); one warp per row group
            {
                const int c = lane, r0 = warp * QT_VG;
                double m[5][QT_VG];
#pragma unroll
                for (int o = 0; o < QT_VG; ++o)
#pragma unroll
                    for (int q = 0; q < 5; ++q) m[q][o] = 0.0;
                if (c < nx && r0 < ny) {
#pragma unroll
                    for (int k = 0; k < QT_VG + 2 * QT_R; ++k) {
                        double v[5];
#pragma unroll
                        for (int q = 0; q < 5; ++q) v[q] = hm[q][r0 + k][c];
#pragma unroll
                        for (int o = 0; o < QT_VG; ++o) {
                            const int j = k - o;
                            if (j >= 0 && j < QT_TAPS) {
#pragma unroll
                                for (int q = 0; q < 5; ++q) m[q][o] = fma(w[j], v[q], m[q][o]);
                            }
                        }
                    }
#pragma unroll
                    for (int o = 0; o < QT_VG; ++o)
                        if (r0 + o < ny) acc += ssim_at(m[0][o], m[1][o], m[2][o], m[3][o], m[4][o]);
                }
            }
        }
        // CTA reduction in a fixed order: warp trees, then the warps in order
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            acc += __shfl_down_sync(0xffffffffu, acc, s);
            e0 += __shfl_down_sync(0xffffffffu, e0, s);
            e1 += __shfl_down_sync(0xffffffffu, e1, s);
            e2 += __shfl_down_sync(0xffffffffu, e2, s);
        }
        if (lane == 0) {
            red_s[warp] = acc;
            red_e[warp][0] = e0; red_e[warp][1] = e1; red_e[warp][2] = e2;
        }
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            uint32_t f0 = 0, f1 = 0, f2 = 0;
            for (int i = 0; i < QT_THREADS / 32; ++i) {
                s += red_s[i];
                f0 += red_e[i][0]; f1 += red_e[i][1]; f2 += red_e[i][2];
            }
            ssim_part[u] = s;
            sse_part[u * 3] = f0; sse_part[u * 3 + 1] = f1; sse_part[u * 3 + 2] = f2;
        }
    }
}

// per patch: the tile partials in tile order (fp64 for SSIM, int64 for SSE)
__global__ void __launch_bounds__(128)
quality_finish_kernel(const double* __restrict__ ssim_part, const uint32_t* __restrict__ sse_part,
                      int64_t batch, int tiles, double inv_count, int64_t* __restrict__ sse,
                      double* __restrict__ ssim) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= batch) return;
    const double* ps = ssim_part + t * tiles;
    const uint32_t* pe = sse_part + t * tiles * 3;
    double s = 0.0;
    int64_t e0 = 0, e1 = 0, e2 = 0;
    for (int i = 0; i < tiles; ++i) {
        s += ps[i];
        e0 += pe[i * 3]; e1 += pe[i * 3 + 1]; e2 += pe[i * 3 + 2];
    }
    ssim[t] = s * inv_count;
    sse[t * 3] = e0; sse[t * 3 + 1] = e1; sse[t * 3 + 2] = e2;
}

static int64_t quality_tiles(int H, int W) {
    return (int64_t)((H - 2 * QT_R + QT_Y - 1) / QT_Y) * ((W - 2 * QT_R + QT_X - 1) / QT_X);
}

static size_t align256q(size_t v) { return (v + 255) & ~(size_t)255; }

// placement of a batch of H x W patches inside a canvas [rows, cols, 3] (VQAE_OK / VQAE_ERR_BAD_ARG)
static int check_placement(const uint8_t* p, int64_t rows, int64_t cols, int64_t r0, int64_t c0, int64_t rc,
                    int64_t first, int64_t batch, int H, int W) {
    if (!p || rows <= 0 || cols <= 0 || r0 < 0 || c0 < 0 || rc <= 0 || first < 0) return VQAE_ERR_BAD_ARG;
    const int64_t last = first + batch - 1;
    if ((r0 + last / rc + 1) * H > rows || (c0 + rc) * W > cols) return VQAE_ERR_BAD_ARG;
    return VQAE_OK;
}

size_t quality_u8_scratch_bytes(int64_t batch, int H, int W) {
    if (batch <= 0 || H < QT_TAPS || W < QT_TAPS) return 0;
    const size_t units = (size_t)batch * quality_tiles(H, W);
    return align256q(units * sizeof(double)) + align256q(units * 3 * sizeof(uint32_t));
}

int quality_u8(const uint8_t* ref, int64_t ref_rows, int64_t ref_cols, int64_t ref_r0, int64_t ref_c0,
               int64_t ref_rc, int64_t ref_first, const uint8_t* rec, int64_t rec_rows, int64_t rec_cols,
               int64_t rec_r0, int64_t rec_c0, int64_t rec_rc, int64_t rec_first, int64_t batch, int H,
               int W, int64_t* sse, double* ssim, void* scratch, size_t scratch_bytes,
               cudaStream_t stream) {
    if (!sse || !ssim || batch <= 0 || H <= 0 || W <= 0) return VQAE_ERR_BAD_ARG;
    if (int rc = check_placement(ref, ref_rows, ref_cols, ref_r0, ref_c0, ref_rc, ref_first, batch, H, W))
        return rc;
    if (int rc = check_placement(rec, rec_rows, rec_cols, rec_r0, rec_c0, rec_rc, rec_first, batch, H, W))
        return rc;
    if (H < QT_TAPS || W < QT_TAPS) return VQAE_ERR_UNSUPPORTED;
    if (ref_first + batch - 1 > 0x7fffffff || rec_first + batch - 1 > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    const size_t need = quality_u8_scratch_bytes(batch, H, W);
    if (!scratch || scratch_bytes < need) return VQAE_ERR_SCRATCH;
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;

    // the Gaussian taps: formed in float64, rounded once to fp32
    QualityWeights wt{};
    double g[QT_TAPS], sum = 0.0;
    for (int k = 0; k < QT_TAPS; ++k) {
        const double d = (double)(k - QT_R);
        g[k] = std::exp(-d * d / (2.0 * 1.5 * 1.5));
        sum += g[k];
    }
    for (int k = 0; k < QT_TAPS; ++k) wt.w[k] = (float)(g[k] / sum);

    const int ntx = (W - 2 * QT_R + QT_X - 1) / QT_X;
    const int tiles = (int)quality_tiles(H, W);
    const int64_t units = batch * tiles;
    double* ssim_part = reinterpret_cast<double*>(scratch);
    uint32_t* sse_part = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(scratch) +
                                                     align256q((size_t)units * sizeof(double)));
    const QualityImage a{ref, ref_cols, ref_r0, ref_c0, ref_rc, ref_first};
    const QualityImage b{rec, rec_cols, rec_r0, rec_c0, rec_rc, rec_first};
    const int64_t cap = (int64_t)sm_count * QT_MIN_CTAS;
    const unsigned grid = (unsigned)(units < cap ? units : cap);
    quality_ssim_tiles_kernel<<<grid, QT_THREADS, 0, stream>>>(a, b, units, H, W, ntx, tiles, wt, ssim_part,
                                                               sse_part);
    if (int rc = check_launch()) return rc;
    const double inv_count = 1.0 / (3.0 * (double)(H - 2 * QT_R) * (double)(W - 2 * QT_R));
    quality_finish_kernel<<<ceil_div_u(batch, 128), 128, 0, stream>>>(ssim_part, sse_part, batch, tiles,
                                                                      inv_count, sse, ssim);
    return check_launch();
}

}  // namespace vqae

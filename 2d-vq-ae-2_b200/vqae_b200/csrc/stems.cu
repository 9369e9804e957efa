// Input normalisation and the two stem convolutions (HBM-bound, CUDA cores).
//   normalize_u8   : albumentations Normalize + ToTensorV2
//                    (conf/transforms/camelyon16_transforms.yaml:1-23, transforms/normalize.yaml)
//   stem_in_f32    : Encoder.in_stem  (vq_ae/model.py:141,198)  3x3, zero pad, bias, 3 -> 8
//   stem_out_f32   : Decoder.out_stem (vq_ae/model.py:291)      3x3, zero pad, bias, 8 -> 3
//   stem_out_u8    : the same with de-normalised uint8 RGB output placed into a slide canvas
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.cuh"

namespace vqae {
namespace {

struct Norm3 {
    float sub[3];  // 255 * mean_c
    float mul[3];  // 1 / (255 * std_c)
};

// same operation order as the reference's numpy code: (x - mean255) * (1 / std255), no FMA
__device__ __forceinline__ float norm_px(uint8_t v, float sub, float mul) {
    return __fmul_rn(__fsub_rn((float)v, sub), mul);
}

inline Norm3 make_norm(const float* mean, const float* stdv) {
    Norm3 n;
    for (int c = 0; c < 3; ++c) {
        n.sub[c] = mean[c] * 255.0f;
        n.mul[c] = 1.0f / (stdv[c] * 255.0f);
    }
    return n;
}

__global__ void __launch_bounds__(256)
normalize_u8_kernel(const uint8_t* __restrict__ img, float* __restrict__ out, int64_t npix,
                    int64_t hw, Norm3 n, int out_layout) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const uint8_t* s = img + p * 3;
    const float r = norm_px(s[0], n.sub[0], n.mul[0]);
    const float g = norm_px(s[1], n.sub[1], n.mul[1]);
    const float b = norm_px(s[2], n.sub[2], n.mul[2]);
    if (out_layout == VQAE_LAYOUT_NHWC) {
        out[p * 3 + 0] = r;
        out[p * 3 + 1] = g;
        out[p * 3 + 2] = b;
    } else {
        const int64_t bi = p / hw, q = p % hw;
        float* o = out + bi * 3 * hw + q;
        o[0] = r;
        o[hw] = g;
        o[2 * hw] = b;
    }
}

// XKIND: 0 = fp32 NCHW, 1 = fp32 NHWC, 2 = u8 NHWC (normalised on the fly)
template <int XKIND>
__global__ void __launch_bounds__(256)
stem_in_kernel(const void* __restrict__ xv, const float* __restrict__ w_oihw,
               const float* __restrict__ bias, float* __restrict__ out, int64_t npix, int H,
               int W, Norm3 n) {
    __shared__ float ws[27][8];  // [(c*9 + ky*3 + kx)][o]
    __shared__ float bs[8];
    for (int i = threadIdx.x; i < 27 * 8; i += blockDim.x) {
        const int o = i / 27, r = i % 27;  // OIHW: o*27 + c*9 + ky*3 + kx
        ws[r][o] = w_oihw[i];
    }
    if (threadIdx.x < 8) bs[threadIdx.x] = bias[threadIdx.x];
    __syncthreads();

    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const int x = (int)(p % W);
    const int64_t r = p / W;
    const int y = (int)(r % H);
    const int64_t b = r / H;
    const int64_t hw = (int64_t)H * W;

    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = bs[o];

#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int iy = y + ky - 1;
        if (iy < 0 || iy >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int ix = x + kx - 1;
            if (ix < 0 || ix >= W) continue;
            float v[3];
            if (XKIND == 0) {
                const float* s = reinterpret_cast<const float*>(xv) + b * 3 * hw +
                                 (int64_t)iy * W + ix;
                v[0] = __ldg(s);
                v[1] = __ldg(s + hw);
                v[2] = __ldg(s + 2 * hw);
            } else if (XKIND == 1) {
                const float* s =
                    reinterpret_cast<const float*>(xv) + (b * hw + (int64_t)iy * W + ix) * 3;
                v[0] = __ldg(s);
                v[1] = __ldg(s + 1);
                v[2] = __ldg(s + 2);
            } else {
                const uint8_t* s =
                    reinterpret_cast<const uint8_t*>(xv) + (b * hw + (int64_t)iy * W + ix) * 3;
                v[0] = norm_px(__ldg(s), n.sub[0], n.mul[0]);
                v[1] = norm_px(__ldg(s + 1), n.sub[1], n.mul[1]);
                v[2] = norm_px(__ldg(s + 2), n.sub[2], n.mul[2]);
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float* wr = ws[c * 9 + ky * 3 + kx];
#pragma unroll
                for (int o = 0; o < 8; ++o) acc[o] = fmaf(v[c], wr[o], acc[o]);
            }
        }
    }
    float4* o4 = reinterpret_cast<float4*>(out + p * 8);
    o4[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    o4[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

// Tiled form of the same convolution for W % 128 == 0, H % 8 == 0: one CTA = 8 rows x 128 columns,
// one thread = 4 adjacent pixels.  The (normalised) input tile with its zero-padded halo is staged
// once in shared memory as fp32 planes [c][row][col + 3] (so a thread's 6-column window lies in two
// aligned 128-bit loads), every broadcast weight load feeds 4 pixels, and a thread writes 128
// contiguous bytes.  Accumulation order per output is that of stem_in_kernel (bias, then ky, kx, c).
constexpr int ST_TH = 8, ST_TW = 128, ST_PW = ST_TW + 8;      // padded row pitch (floats)

template <int XKIND, bool HALF_OUT>
__global__ void __launch_bounds__(256)
stem_in_tiled_kernel(const void* __restrict__ xv, const float* __restrict__ w_oihw,
                     const float* __restrict__ bias, void* __restrict__ outv, int H, int W,
                     int tiles_x, int tiles_y, Norm3 n) {
    float* out = reinterpret_cast<float*>(outv);
    // input tile [c][row][col] first, output staging [row][4-px group][8 + 1 float4] afterwards
    __shared__ __align__(16) float ostage[ST_TH * 32 * 9 * 4];
    float (*tile)[ST_TH + 2][ST_PW] = reinterpret_cast<float (*)[ST_TH + 2][ST_PW]>(ostage);
    static_assert(sizeof(float) * 3 * (ST_TH + 2) * ST_PW <= sizeof(float) * ST_TH * 32 * 9 * 4, "tile fits");
    __shared__ __align__(16) float ws[27][8];  // [(ky*3 + kx)*3 + c][o]
    __shared__ float bs[8];
    const int tid = threadIdx.x;
    for (int i = tid; i < 27 * 8; i += 256) {
        const int o = i / 27, r = i % 27;        // OIHW: o*27 + c*9 + ky*3 + kx
        const int c = r / 9, t = r % 9;
        ws[t * 3 + c][o] = w_oihw[i];
    }
    if (tid < 8) bs[tid] = bias[tid];
    const int tx = blockIdx.x % tiles_x;
    const int ty = (blockIdx.x / tiles_x) % tiles_y;
    const int64_t b = blockIdx.x / (tiles_x * tiles_y);
    const int x0 = tx * ST_TW, y0 = ty * ST_TH;
    const int64_t hw = (int64_t)H * W;
    // stage rows y0-1 .. y0+8, columns x0-1 .. x0+128 -> tile[c][r][col - x0 + 3]
    for (int i = tid; i < (ST_TH + 2) * (ST_TW + 2); i += 256) {
        const int r = i / (ST_TW + 2), cc = i % (ST_TW + 2);
        const int iy = y0 - 1 + r, ix = x0 - 1 + cc;
        float v0 = 0.f, v1 = 0.f, v2 = 0.f;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
            if (XKIND == 0) {
                const float* s = reinterpret_cast<const float*>(xv) + b * 3 * hw + (int64_t)iy * W + ix;
                v0 = __ldg(s); v1 = __ldg(s + hw); v2 = __ldg(s + 2 * hw);
            } else if (XKIND == 1) {
                const float* s = reinterpret_cast<const float*>(xv) + (b * hw + (int64_t)iy * W + ix) * 3;
                v0 = __ldg(s); v1 = __ldg(s + 1); v2 = __ldg(s + 2);
            } else {
                const uint8_t* s = reinterpret_cast<const uint8_t*>(xv) + (b * hw + (int64_t)iy * W + ix) * 3;
                v0 = norm_px(__ldg(s), n.sub[0], n.mul[0]);
                v1 = norm_px(__ldg(s + 1), n.sub[1], n.mul[1]);
                v2 = norm_px(__ldg(s + 2), n.sub[2], n.mul[2]);
            }
        }
        tile[0][r][cc + 2] = v0;
        tile[1][r][cc + 2] = v1;
        tile[2][r][cc + 2] = v2;
    }
    __syncthreads();

    const int gx = tid & 31, gy = tid >> 5;      // 4-pixel group, row in tile
    float2 acc[4][4];                            // packed fp32x2 FMAs: the same per-output fmaf chains
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int o = 0; o < 4; ++o) acc[p][o] = make_float2(bs[2 * o], bs[2 * o + 1]);
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        float win[3][8];                         // padded columns 4gx .. 4gx+7 = image x-3 .. x+4
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float4 a = *reinterpret_cast<const float4*>(&tile[c][gy + ky][4 * gx]);
            const float4 d = *reinterpret_cast<const float4*>(&tile[c][gy + ky][4 * gx + 4]);
            win[c][0] = a.x; win[c][1] = a.y; win[c][2] = a.z; win[c][3] = a.w;
            win[c][4] = d.x; win[c][5] = d.y; win[c][6] = d.z; win[c][7] = d.w;
        }
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float4 w0 = *reinterpret_cast<const float4*>(&ws[(ky * 3 + kx) * 3 + c][0]);
                const float4 w1 = *reinterpret_cast<const float4*>(&ws[(ky * 3 + kx) * 3 + c][4]);
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    const float v = win[c][p + kx + 2];          // image column x + p + kx - 1
                    const float2 vv = make_float2(v, v);
                    acc[p][0] = __ffma2_rn(vv, make_float2(w0.x, w0.y), acc[p][0]);
                    acc[p][1] = __ffma2_rn(vv, make_float2(w0.z, w0.w), acc[p][1]);
                    acc[p][2] = __ffma2_rn(vv, make_float2(w1.x, w1.y), acc[p][2]);
                    acc[p][3] = __ffma2_rn(vv, make_float2(w1.z, w1.w), acc[p][3]);
                }
            }
    }
    // stage the 8 x 128 x 8 output tile in shared memory (pitch 33 float4 per 4-pixel group row keeps
    // the 128-byte-strided writes conflict-free), then store whole 512-byte lines per warp instruction
    float4* stage = reinterpret_cast<float4*>(ostage);
    __syncthreads();                             // every thread is done reading the input tile
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        stage[(gy * 32 + gx) * 9 + 2 * p] = make_float4(acc[p][0].x, acc[p][0].y, acc[p][1].x, acc[p][1].y);
        stage[(gy * 32 + gx) * 9 + 2 * p + 1] = make_float4(acc[p][2].x, acc[p][2].y, acc[p][3].x, acc[p][3].y);
    }
    __syncthreads();
    if constexpr (HALF_OUT) {
        // fp16 stream: one pixel (8 channels = 16 bytes) per thread and step, 2 KB rows
        __half* outh = reinterpret_cast<__half*>(outv);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = tid + 256 * k;         // pixel index in the tile: row (i >> 7), 128 per row
            const int r = i >> 7, j = i & 127;   // j = 4 * group + pixel of the group
            const float4 lo = stage[(r * 32 + (j >> 2)) * 9 + 2 * (j & 3)];
            const float4 hi = stage[(r * 32 + (j >> 2)) * 9 + 2 * (j & 3) + 1];
            const __half2 h0 = __floats2half2_rn(lo.x, lo.y), h1 = __floats2half2_rn(lo.z, lo.w);
            const __half2 h2 = __floats2half2_rn(hi.x, hi.y), h3 = __floats2half2_rn(hi.z, hi.w);
            uint4 u;
            u.x = *reinterpret_cast<const uint32_t*>(&h0); u.y = *reinterpret_cast<const uint32_t*>(&h1);
            u.z = *reinterpret_cast<const uint32_t*>(&h2); u.w = *reinterpret_cast<const uint32_t*>(&h3);
            uint4* dst = reinterpret_cast<uint4*>(outh + ((b * H + y0 + r) * (int64_t)W + x0) * 8);
            dst[j] = u;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int i = tid + 256 * k;         // float4 index in the tile: row (i >> 8), 256 per row
            const int r = i >> 8, j = i & 255;   // j = 8 * group + chunk
            float4* dst = reinterpret_cast<float4*>(out + ((b * H + y0 + r) * (int64_t)W + x0) * 8);
            dst[j] = stage[(r * 32 + (j >> 3)) * 9 + (j & 7)];
        }
    }
}

// U8: the de-normalising uint8 epilogue (u8_store, common.cuh) placing image b at patch
// first_patch + b of a canvas; a warp's 32 pixels (one row segment when W % 32 == 0) are staged in
// shared memory and leave as six 16-byte stores.  The arithmetic up to the stored value is shared.
template <int CIN, bool U8>
__global__ void __launch_bounds__(256)
stem_out_kernel(const float* __restrict__ x, const float* __restrict__ w_oihw,
                const float* __restrict__ bias, float* __restrict__ out, int out_layout,
                int64_t npix, int H, int W, U8Canvas cv) {
    __shared__ float ws[9 * CIN][3];  // [(ky*3+kx)*CIN + c][o]
    __shared__ float bs[3];
    for (int i = threadIdx.x; i < 3 * CIN * 9; i += blockDim.x) {
        const int o = i / (CIN * 9);
        const int c = (i / 9) % CIN;
        const int t = i % 9;
        ws[t * CIN + c][o] = w_oihw[i];
    }
    if (threadIdx.x < 3) bs[threadIdx.x] = bias[threadIdx.x];
    __syncthreads();

    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const int xx = (int)(p % W);
    const int64_t r = p / W;
    const int y = (int)(r % H);
    const int64_t b = r / H;
    const int64_t hw = (int64_t)H * W;

    float a0 = bs[0], a1 = bs[1], a2 = bs[2];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int iy = y + ky - 1;
        if (iy < 0 || iy >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int ix = xx + kx - 1;
            if (ix < 0 || ix >= W) continue;
            const float4* s =
                reinterpret_cast<const float4*>(x + (b * hw + (int64_t)iy * W + ix) * CIN);
#pragma unroll
            for (int c4 = 0; c4 < CIN / 4; ++c4) {
                const float4 v = __ldg(s + c4);
                const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float* wr = ws[(ky * 3 + kx) * CIN + c4 * 4 + j];
                    a0 = fmaf(vv[j], wr[0], a0);
                    a1 = fmaf(vv[j], wr[1], a1);
                    a2 = fmaf(vv[j], wr[2], a2);
                }
            }
        }
    }
    if constexpr (U8) {
        __shared__ __align__(16) uint8_t st[8][96];                 // one 32-pixel segment per warp
        const int q = (int)cv.first_patch + (int)b;                 // first_patch + B < 2^31
        const int prow = q / cv.grid_cols, pcol = q - prow * cv.grid_cols;
        uint8_t* dst = cv.canvas + (((int64_t)prow * H + y) * cv.canvas_cols + (int64_t)pcol * W + xx) * 3;
        const uint8_t r8 = u8_store(a0, cv.s[0], cv.o[0]), g8 = u8_store(a1, cv.s[1], cv.o[1]),
                      b8 = u8_store(a2, cv.s[2], cv.o[2]);
        if (!cv.vec) {
            dst[0] = r8; dst[1] = g8; dst[2] = b8;
            return;
        }
        // vec: W % 32 == 0, so a warp's 32 pixels are one 96-byte segment of an image row (and
        // npix % 32 == 0: no warp is cut by the early return above)
        const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
        st[wp][lane * 3] = r8; st[wp][lane * 3 + 1] = g8; st[wp][lane * 3 + 2] = b8;
        __syncwarp();
        uint8_t* seg = dst - lane * 3;                               // the segment's first byte
        if (lane < 6)
            reinterpret_cast<uint4*>(seg)[lane] = reinterpret_cast<const uint4*>(st[wp])[lane];
        return;
    }
    if (out_layout == VQAE_LAYOUT_NHWC) {
        out[p * 3 + 0] = a0;
        out[p * 3 + 1] = a1;
        out[p * 3 + 2] = a2;
    } else {
        float* o = out + b * 3 * hw + (int64_t)y * W + xx;
        o[0] = a0;
        o[hw] = a1;
        o[2 * hw] = a2;
    }
}

}  // namespace

int normalize_u8(const uint8_t* img, float* out, int64_t B, int H, int W, const float* mean,
                 const float* stdv, int out_layout, cudaStream_t stream) {
    if (!img || !out || !mean || !stdv || B <= 0 || H <= 0 || W <= 0) return VQAE_ERR_BAD_ARG;
    const int64_t hw = (int64_t)H * W, npix = B * hw;
    normalize_u8_kernel<<<ceil_div_u(npix, 256), 256, 0, stream>>>(img, out, npix, hw,
                                                                   make_norm(mean, stdv),
                                                                   out_layout);
    return check_launch();
}

int stem_in_f32(const void* x, int x_dtype, int x_layout, const float* w, const float* bias,
                void* outv, int out_dtype, int64_t B, int H, int W, int c_out, const float* mean,
                const float* stdv, cudaStream_t stream) {
    if (!x || !w || !bias || !outv || B <= 0 || H <= 0 || W <= 0) return VQAE_ERR_BAD_ARG;
    if (c_out != 8) return VQAE_ERR_UNSUPPORTED;
    const int64_t npix = B * H * W;
    const unsigned grid = ceil_div_u(npix, 256);
    const bool tiled = (W % ST_TW == 0) && (H % ST_TH == 0) &&
                       B * (H / ST_TH) * (W / ST_TW) <= 0x7fffffff;
    const int txs = W / ST_TW, tys = H / ST_TH;
    const unsigned tgrid = tiled ? (unsigned)(B * txs * tys) : 0u;
    // the fp16 stream output exists in the tiled form (W % 128 == 0, H % 8 == 0)
    const bool half_out = out_dtype == VQAE_DT_F16;
    if ((half_out && !tiled) || (!half_out && out_dtype != VQAE_DT_F32)) return VQAE_ERR_UNSUPPORTED;
    float* out = reinterpret_cast<float*>(outv);
    Norm3 n{};
    int kind;
    if (x_dtype == VQAE_DT_U8) {
        if (!mean || !stdv) return VQAE_ERR_BAD_ARG;
        if (x_layout != VQAE_LAYOUT_NHWC) return VQAE_ERR_UNSUPPORTED;
        n = make_norm(mean, stdv);
        kind = 2;
    } else if (x_dtype == VQAE_DT_F32) {
        kind = x_layout == VQAE_LAYOUT_NCHW ? 0 : 1;
    } else {
        return VQAE_ERR_UNSUPPORTED;
    }
#define STEM_TILED(K, HO) stem_in_tiled_kernel<K, HO><<<tgrid, 256, 0, stream>>>(x, w, bias, outv, H, W, txs, tys, n)
    if (tiled && half_out) {
        if (kind == 2) STEM_TILED(2, true); else if (kind == 0) STEM_TILED(0, true); else STEM_TILED(1, true);
    } else if (tiled) {
        if (kind == 2) STEM_TILED(2, false); else if (kind == 0) STEM_TILED(0, false); else STEM_TILED(1, false);
    } else {
        if (kind == 2) stem_in_kernel<2><<<grid, 256, 0, stream>>>(x, w, bias, out, npix, H, W, n);
        else if (kind == 0) stem_in_kernel<0><<<grid, 256, 0, stream>>>(x, w, bias, out, npix, H, W, n);
        else stem_in_kernel<1><<<grid, 256, 0, stream>>>(x, w, bias, out, npix, H, W, n);
    }
#undef STEM_TILED
    return check_launch();
}

int stem_out_f32(const float* x, const float* w, const float* bias, float* out, int out_layout,
                 int64_t B, int H, int W, int c_in, cudaStream_t stream) {
    if (!x || !w || !bias || !out || B <= 0 || H <= 0 || W <= 0) return VQAE_ERR_BAD_ARG;
    if (c_in != 8) return VQAE_ERR_UNSUPPORTED;
    const int64_t npix = B * H * W;
    stem_out_kernel<8, false><<<ceil_div_u(npix, 256), 256, 0, stream>>>(x, w, bias, out, out_layout,
                                                                         npix, H, W, U8Canvas{});
    return check_launch();
}

int make_u8_canvas(uint8_t* canvas, int64_t canvas_rows, int64_t canvas_cols, int64_t first_patch,
                   int grid_cols, int64_t B, int H, int W, const float* mean, const float* stdv,
                   U8Canvas* cv) {
    if (!canvas || !mean || !stdv || B <= 0 || H <= 0 || W <= 0 || canvas_rows <= 0 ||
        canvas_cols <= 0 || grid_cols <= 0 || first_patch < 0)
        return VQAE_ERR_BAD_ARG;
    const int64_t last = first_patch + B - 1;
    if ((int64_t)grid_cols * W > canvas_cols || (last / grid_cols + 1) * H > canvas_rows)
        return VQAE_ERR_BAD_ARG;
    if (last > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;           // patch indices are 32-bit in the kernels
    cv->canvas = canvas;
    cv->canvas_cols = canvas_cols;
    cv->first_patch = first_patch;
    cv->grid_cols = grid_cols;
    cv->vec = W % 32 == 0 && canvas_cols % 16 == 0 && (reinterpret_cast<uintptr_t>(canvas) & 15u) == 0;
    for (int c = 0; c < 3; ++c) {
        cv->s[c] = 255.0f * stdv[c];           // the fp32 products of the normalisation
        cv->o[c] = 255.0f * mean[c];
    }
    return VQAE_OK;
}

int stem_out_u8(const float* x, const float* w, const float* bias, const U8Canvas& cv, int64_t B,
                int H, int W, int c_in, cudaStream_t stream) {
    if (!x || !w || !bias) return VQAE_ERR_BAD_ARG;
    if (c_in != 8) return VQAE_ERR_UNSUPPORTED;
    const int64_t npix = B * H * W;
    stem_out_kernel<8, true><<<ceil_div_u(npix, 256), 256, 0, stream>>>(x, w, bias, nullptr,
                                                                        VQAE_LAYOUT_NHWC, npix, H, W, cv);
    return check_launch();
}

}  // namespace vqae

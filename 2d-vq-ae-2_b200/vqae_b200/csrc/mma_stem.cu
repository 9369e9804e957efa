// The two stem convolutions on warp-level tensor-core MMAs with split fp16 operands (fp32-accurate).
//
// Encoder.in_stem (vq_ae/model.py:141,198: 3x3 conv, zero padding, bias, 3 -> 8, with the u8
// normalisation of conf/transforms/camelyon16_transforms.yaml fused): the input window is staged as
// split fp16 pixels (hi R, G, B, 0 | lo R, G, B, 0 = 16 bytes), and per kernel row ky ONE m16n8k16 MMA
// covers K = 4 window pixels x 4 halves -- lane t of a fragment row owns window pixel kx = t, so its hi
// and lo operand registers are one 128-bit load; weights are zero on the 4th pixel and channel.  Nine
// MMAs per 16 pixels instead of 3456 FMAs: 320 -> ~150 us at batch 256 of 256^2 (HBM floor 90 us).
//
// Decoder.out_stem (vq_ae/model.py:291: 3x3 conv, zero padding, bias, 8 -> 3) on warp-level tensor-core
// MMAs, fp32-accurate: the nine taps are nine K = 8 GEMM steps over a staged tile whose pixels are 16-byte
// rows of fp16 channels, so a tap is a row shift of the ldmatrix address (the scheme of stage 2 in
// mma_same.cu); operands are split hi + lo (three MMAs per product, see tc_split.cu) because this is
// the layer that produces the reconstruction.  The CUDA-core kernel it replaces (stems.cu) reads its
// 3x3 x 8-channel window straight from global memory and runs at 98 % of the L1 data-pipe
// (524 us at batch 256 of 256^2 against an HBM floor of 112 us); here every input pixel is read once.
// Used by the "fp16" and "fp32tc" paths; "fp32" keeps the exact fp32 kernel.
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"
#include "mma_common.cuh"
#include "tc_common.cuh"

namespace vqae {
namespace {

using namespace mma;

constexpr int SO_TH = 16, SO_TW = 32, SO_PW = SO_TW + 2;
constexpr int SO_NPAD = (SO_TH + 2) * SO_PW;           // 612 pixels of tile + ring
constexpr int SO_ROWS = SO_NPAD + 12;                  // + slack for the last ldmatrix rows
constexpr int SO_MT = SO_TH * SO_TW / 16;              // 32 M-tiles
constexpr int SO_THREADS = 256, SO_WARPS = 8;
constexpr uint32_t SO_PLANE = SO_ROWS * 16;
constexpr uint32_t SO_SMEM = 2 * SO_PLANE;

struct StemOutArgs {
    const float* x;          // NHWC fp32 [B,H,W,8]
    const float* w;          // OIHW [3,8,3,3]
    const float* bias;       // [3]
    float* out;              // NCHW [B,3,H,W] or NHWC [B,H,W,3] (fp32 form)
    int n_tiles, H, W, tiles_x, tiles_per_img, nhwc_out;
    U8Canvas cv;             // uint8 form
};

__device__ __forceinline__ void so_split2(float f0, float f1, uint32_t& hi, uint32_t& lo) {
    const __half2 hh = __floats2half2_rn(f0, f1);
    const float2 hf = __half22float2(hh);
    const __half2 ll = __floats2half2_rn(f0 - hf.x, f1 - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&hh);
    lo = *reinterpret_cast<const uint32_t*>(&ll);
}

// U8: the de-normalising uint8 epilogue (u8_store) placing image b at patch first_patch + b of a
// canvas.  A warp covers four 16-pixel row segments of a tile (48 bytes each, 16-byte aligned: tiles
// start at multiples of 32 pixels = 96 bytes); their bytes are staged in the warp's 192 bytes of shared
// memory and leave after its MMA steps as twelve 16-byte stores.  Everything up to the stored value is
// the fp32 form's arithmetic.
template <bool U8>
__global__ void __launch_bounds__(SO_THREADS, 3)
stem_out_mma_kernel(StemOutArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = tc::smem_u32(smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;

    // B fragments of the nine taps: B[k = channel][n = output], n < 3 real; hi / lo
    uint32_t bh[9], bl[9];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        float w0 = 0.f, w1 = 0.f;
        if (g < 3) {
            w0 = __ldg(a.w + (g * 8 + 2 * t) * 9 + tap);
            w1 = __ldg(a.w + (g * 8 + 2 * t + 1) * 9 + tap);
        }
        so_split2(w0, w1, bh[tap], bl[tap]);
    }
    const float bias0 = 2 * t < 3 ? __ldg(a.bias + 2 * t) : 0.f;
    const float bias1 = 2 * t + 1 < 3 ? __ldg(a.bias + 2 * t + 1) : 0.f;
    for (int i = tid; i < (int)(SO_SMEM / 16); i += SO_THREADS)
        *reinterpret_cast<uint4*>(smem + i * 16) = make_uint4(0, 0, 0, 0);
    __syncthreads();
    const size_t plane = (size_t)a.H * a.W;

    // a thread stages the same (up to three) ring'd-tile pixels of every tile; the NEXT tile's pixels are
    // loaded into registers before the current tile is computed, so their latency hides behind the MMAs
    constexpr int PPT = (SO_NPAD + SO_THREADS - 1) / SO_THREADS;
    float4 pv[PPT][2];
    auto fetch = [&](int tile) {
        const int img = tile / a.tiles_per_img;
        const int trem = tile - img * a.tiles_per_img;
        const int r0 = (trem / a.tiles_x) * SO_TH, c0 = (trem % a.tiles_x) * SO_TW;
        const float* ximg = a.x + (size_t)img * plane * 8;
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            const int q = tid + k * SO_THREADS;
            const int lr = q / SO_PW, lc = q - lr * SO_PW;
            const int y = r0 - 1 + lr, x = c0 - 1 + lc;
            pv[k][0] = pv[k][1] = make_float4(0.f, 0.f, 0.f, 0.f);           // zero padding
            if (q < SO_NPAD && y >= 0 && y < a.H && x >= 0 && x < a.W) {
                const float4* p = reinterpret_cast<const float4*>(ximg + ((size_t)y * a.W + x) * 8);
                pv[k][0] = __ldg(p);
                pv[k][1] = __ldg(p + 1);
            }
        }
    };
    if ((int)blockIdx.x < a.n_tiles) fetch(blockIdx.x);

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int img = tile / a.tiles_per_img;
        const int trem = tile - img * a.tiles_per_img;
        const int r0 = (trem / a.tiles_x) * SO_TH, c0 = (trem % a.tiles_x) * SO_TW;

        // ---- stage tile + ring as fp16 hi / lo rows of 8 channels ----
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            const int q = tid + k * SO_THREADS;
            if (q < SO_NPAD) {
                uint4 hi, lo;
                so_split2(pv[k][0].x, pv[k][0].y, hi.x, lo.x);
                so_split2(pv[k][0].z, pv[k][0].w, hi.y, lo.y);
                so_split2(pv[k][1].x, pv[k][1].y, hi.z, lo.z);
                so_split2(pv[k][1].z, pv[k][1].w, hi.w, lo.w);
                *reinterpret_cast<uint4*>(smem + q * 16) = hi;
                *reinterpret_cast<uint4*>(smem + SO_PLANE + q * 16) = lo;
            }
        }
        __syncthreads();
        if (tile + (int)gridDim.x < a.n_tiles) fetch(tile + gridDim.x);

        // u8: the tile's first canvas byte (32-bit patch arithmetic: first_patch + B < 2^31)
        uint8_t* tile_dst = nullptr;
        const int64_t row_bytes = a.cv.canvas_cols * 3;
        if constexpr (U8) {
            const int q = (int)a.cv.first_patch + img;
            const int prow = q / a.cv.grid_cols, pcol = q - prow * a.cv.grid_cols;
            tile_dst = a.cv.canvas + ((int64_t)prow * a.H + r0) * row_bytes + ((int64_t)pcol * a.W + c0) * 3;
        }
        // ---- nine shifted K = 8 GEMM steps per M-tile (16 pixels of a row), two M-tiles per warp step
        const int lrow = (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll 1
        for (int mt0 = warp; mt0 < SO_MT; mt0 += 2 * SO_WARPS) {
            float d[2][4];
            uint32_t lbase[2];
            int rr[2], cb[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int mt = mt0 + u * SO_WARPS;
                rr[u] = mt >> 1;
                cb[u] = (mt & 1) * 16;
                lbase[u] = sbase + (uint32_t)((rr[u] + 1) * SO_PW + cb[u] + 1 + lrow) * 16;
                d[u][0] = d[u][2] = bias0;
                d[u][1] = d[u][3] = bias1;
            }
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
                const int shift = (tap / 3 - 1) * SO_PW + (tap % 3 - 1);
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    uint32_t h0, h1, l0, l1;
                    ldmatrix_x2(h0, h1, lbase[u] + shift * 16);
                    ldmatrix_x2(l0, l1, lbase[u] + SO_PLANE + shift * 16);
                    mma_1688(d[u], l0, l1, bh[tap]);
                    mma_1688(d[u], h0, h1, bl[tap]);
                    mma_1688(d[u], h0, h1, bh[tap]);
                }
            }
            if constexpr (U8) {
                // lane (g, t): t = 0 holds channels 0, 1 and t = 1 channel 2 of pixels g and g + 8;
                // the warp's four 16-pixel segments of the tile go to its 192 staging bytes
                uint8_t* st = smem + SO_SMEM + warp * 192 + (mt0 >> 4) * 96;
                if (t < 2) {
                    const float s0 = t ? a.cv.s[2] : a.cv.s[0], o0 = t ? a.cv.o[2] : a.cv.o[0];
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        uint8_t* sp = st + u * 48 + g * 3 + 2 * t;
                        sp[0] = u8_store(d[u][0], s0, o0);
                        sp[24] = u8_store(d[u][2], s0, o0);
                        if (t == 0) {
                            sp[1] = u8_store(d[u][1], a.cv.s[1], a.cv.o[1]);
                            sp[25] = u8_store(d[u][3], a.cv.s[1], a.cv.o[1]);
                        }
                    }
                }
                continue;
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int y = r0 + rr[u], x = c0 + cb[u] + g;
                if (a.nhwc_out) {
                    float* o = a.out + ((size_t)img * plane + (size_t)y * a.W + x) * 3;
                    if (t == 0) {
                        o[0] = d[u][0]; o[1] = d[u][1];
                        o[24] = d[u][2]; o[25] = d[u][3];
                    } else if (t == 1) {
                        o[2] = d[u][0];
                        o[26] = d[u][2];
                    }
                } else {
                    float* o = a.out + (size_t)img * 3 * plane + (size_t)y * a.W + x;
                    if (t == 0) {
                        o[0] = d[u][0]; o[8] = d[u][2];
                        o[plane] = d[u][1]; o[plane + 8] = d[u][3];
                    } else if (t == 1) {
                        o[2 * plane] = d[u][0]; o[2 * plane + 8] = d[u][2];
                    }
                }
            }
        }
        if constexpr (U8) {
            // segment (j, u) of this warp is M-tile warp + 16 j + 8 u: tile row (mt >> 1), columns 16 (warp & 1)
            __syncwarp();
            const uint8_t* st = smem + SO_SMEM + warp * 192;
            if (a.cv.vec) {
                if (lane < 12) {
                    const int seg = lane / 3, k = lane - 3 * seg;
                    const int mt = warp + 16 * (seg >> 1) + 8 * (seg & 1);
                    uint8_t* dst = tile_dst + (int64_t)(mt >> 1) * row_bytes + (mt & 1) * 48;
                    reinterpret_cast<uint4*>(dst)[k] = reinterpret_cast<const uint4*>(st + seg * 48)[k];
                }
            } else {
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    const int seg = 2 * pass + (lane >> 4), px = lane & 15;
                    const int mt = warp + 16 * pass + 8 * (lane >> 4);
                    uint8_t* dst = tile_dst + (int64_t)(mt >> 1) * row_bytes + ((mt & 1) * 16 + px) * 3;
                    dst[0] = st[seg * 48 + px * 3];
                    dst[1] = st[seg * 48 + px * 3 + 1];
                    dst[2] = st[seg * 48 + px * 3 + 2];
                }
            }
            // the staging is rewritten only after the next tile's first barrier
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// in_stem
// ------------------------------------------------------------------------------------------------
constexpr int SI_TH = 16, SI_TW = 32;
constexpr int SI_SROWS = SI_TH + 2, SI_SPW = SI_TW + 4;       // 34 real pixels + 2 zero per staged row
constexpr int SI_SREAL_C = SI_TW + 2;
constexpr int SI_MT = SI_TH * SI_TW / 16;
constexpr uint32_t SI_SMEM = SI_SROWS * SI_SPW * 16;

struct SiNorm { float sub[3], mul[3]; };
struct StemInArgs {
    const void* x;           // u8 NHWC [B,H,W,3] | fp32 NHWC | fp32 NCHW
    const float* w;          // OIHW [8,3,3,3]
    const float* bias;       // [8]
    float* out;              // NHWC fp32 [B,H,W,8]
    int n_tiles, H, W, tiles_x, tiles_per_img;
    SiNorm n;
};

// XKIND: 0 = fp32 NCHW, 1 = fp32 NHWC, 2 = u8 NHWC (normalised like normalize_u8 / stem_in_kernel)
template <int XKIND>
__global__ void __launch_bounds__(SO_THREADS, 4)
stem_in_mma_kernel(StemInArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    // B fragments: k-slots (2t, 2t + 1) [h = 0] and (2t + 8, 2t + 9) [h = 1] of this lane stand for
    // window pixel kx = t, channels (0, 1) and (2, pad); n = g
    uint32_t bh[3][2], bl[3][2];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float w[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = 2 * h + e;
                w[e] = (t < 3 && c < 3) ? __ldg(a.w + g * 27 + c * 9 + ky * 3 + t) : 0.f;
            }
            so_split2(w[0], w[1], bh[ky][h], bl[ky][h]);
        }
    const float bias0 = __ldg(a.bias + 2 * t), bias1 = __ldg(a.bias + 2 * t + 1);
    for (int i = tid; i < (int)(SI_SMEM / 16); i += SO_THREADS)
        *reinterpret_cast<uint4*>(smem + i * 16) = make_uint4(0, 0, 0, 0);
    __syncthreads();
    const int64_t hw = (int64_t)a.H * a.W;

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int img = tile / a.tiles_per_img;
        const int trem = tile - img * a.tiles_per_img;
        const int r0 = (trem / a.tiles_x) * SI_TH, c0 = (trem % a.tiles_x) * SI_TW;
        // ---- stage the window: 18 x 34 pixels, zero outside the image (= the conv's padding) ----
        for (int i = tid; i < SI_SROWS * SI_SREAL_C; i += SO_THREADS) {
            const int si = i / SI_SREAL_C, sj = i - si * SI_SREAL_C;
            const int iy = r0 - 1 + si, ix = c0 - 1 + sj;
            float v0 = 0.f, v1 = 0.f, v2 = 0.f;
            if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W) {
                if (XKIND == 0) {
                    const float* s = reinterpret_cast<const float*>(a.x) + (int64_t)img * 3 * hw + (int64_t)iy * a.W + ix;
                    v0 = __ldg(s); v1 = __ldg(s + hw); v2 = __ldg(s + 2 * hw);
                } else if (XKIND == 1) {
                    const float* s = reinterpret_cast<const float*>(a.x) + ((int64_t)img * hw + (int64_t)iy * a.W + ix) * 3;
                    v0 = __ldg(s); v1 = __ldg(s + 1); v2 = __ldg(s + 2);
                } else {
                    const uint8_t* s = reinterpret_cast<const uint8_t*>(a.x) + ((int64_t)img * hw + (int64_t)iy * a.W + ix) * 3;
                    v0 = __fmul_rn(__fsub_rn((float)__ldg(s), a.n.sub[0]), a.n.mul[0]);
                    v1 = __fmul_rn(__fsub_rn((float)__ldg(s + 1), a.n.sub[1]), a.n.mul[1]);
                    v2 = __fmul_rn(__fsub_rn((float)__ldg(s + 2), a.n.sub[2]), a.n.mul[2]);
                }
            }
            uint4 px;                                      // hi01, hi2-, lo01, lo2-
            so_split2(v0, v1, px.x, px.z);
            so_split2(v2, 0.f, px.y, px.w);
            *reinterpret_cast<uint4*>(smem + (uint32_t)(si * SI_SPW + sj) * 16) = px;
        }
        __syncthreads();
        // ---- 32 M-tiles of 16 pixels of a row, two per warp step ----
        float* oimg = a.out + (size_t)img * hw * 8;
#pragma unroll 1
        for (int mt0 = warp; mt0 < SI_MT; mt0 += 2 * SO_WARPS) {
            float d[2][4];
            const uint8_t* p0[2];
            int rr[2], cb[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int mt = mt0 + u * SO_WARPS;
                rr[u] = mt >> 1;
                cb[u] = (mt & 1) * 16;
                // pixel (r, c) of the tile = staged (r + 1, c + 1); its window starts at staged (r + ky, c)
                p0[u] = smem + (uint32_t)(rr[u] * SI_SPW + cb[u] + g + t) * 16;
                d[u][0] = d[u][2] = bias0;
                d[u][1] = d[u][3] = bias1;
            }
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const uint4 u0 = *reinterpret_cast<const uint4*>(p0[u] + ky * SI_SPW * 16);
                    const uint4 u1 = *reinterpret_cast<const uint4*>(p0[u] + ky * SI_SPW * 16 + 8 * 16);
                    const uint32_t ah[4] = {u0.x, u1.x, u0.y, u1.y}, al[4] = {u0.z, u1.z, u0.w, u1.w};
                    mma_16816(d[u], al, bh[ky][0], bh[ky][1]);
                    mma_16816(d[u], ah, bl[ky][0], bl[ky][1]);
                    mma_16816(d[u], ah, bh[ky][0], bh[ky][1]);
                }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                float* o = oimg + ((size_t)(r0 + rr[u]) * a.W + c0 + cb[u] + g) * 8 + 2 * t;
                *reinterpret_cast<float2*>(o) = make_float2(d[u][0], d[u][1]);
                *reinterpret_cast<float2*>(o + 64) = make_float2(d[u][2], d[u][3]);
            }
        }
        __syncthreads();
    }
}

// ---- in_stem on uint8 tiles ------------------------------------------------------------------------
// A uint8 pixel value is EXACT in fp16, so the activation side needs no hi / lo split: the
// normalisation (u8 - 255 mean_c) / (255 std_c) is folded into the weights,
//     sum_c,tap W (u8 - sub_c) mul_c  =  sum W' u8  +  sum Wm inside,      W' = W mul_c,  Wm = -sum_c W mul_c sub_c,
// with `inside` (1 inside the image, 0 in the zero padding, which pads the NORMALISED tensor) as a fourth
// input channel in the slot the fp32 form pads with zero.  Only the weights are split (hi + lo, scaled by
// the power of two that moves the largest of them into (2^13, 2^14]): two MMAs per kernel row instead
// of three, 8-byte pixel records, and the window is staged from aligned 32-bit loads issued one tile
// ahead (the fp32 form spends a third of its time waiting for three byte loads per pixel).
constexpr int SU_RAW_W = 26;                                  // raw words per staged row: bytes -4 .. 99 of the row
constexpr uint32_t SU_REC = SI_SROWS * SI_SPW * 8;            // fp16 records (R, G | B, inside), 8 B each
constexpr int SU_NRAW = SI_SROWS * SU_RAW_W;
constexpr uint32_t SU_SMEM = SU_REC + SU_NRAW * 4;

__global__ void __launch_bounds__(SO_THREADS, 4)
stem_in_u8_mma_kernel(StemInArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ float wq[8 * 3 * 3 * 4];                       // [g][ky][kx][c]: W' (c < 3), Wm (c = 3)
    __shared__ int wmax_bits;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    if (tid == 0) wmax_bits = 0;
    for (int i = tid; i < (int)(SU_REC / 16); i += SO_THREADS)
        *reinterpret_cast<uint4*>(smem + i * 16) = make_uint4(0, 0, 0, 0);
    __syncthreads();
    for (int i = tid; i < 8 * 36; i += SO_THREADS) {
        const int gg = i / 36, r = i - gg * 36, ky = r / 12, kx = (r - ky * 12) >> 2, c = r & 3;
        float v;
        if (c < 3) {
            const float mul = c == 0 ? a.n.mul[0] : (c == 1 ? a.n.mul[1] : a.n.mul[2]);   // no dynamic
            v = __fmul_rn(__ldg(a.w + gg * 27 + c * 9 + ky * 3 + kx), mul);               // parameter index
        } else {
            v = 0.f;
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
                v = fmaf(-__fmul_rn(__ldg(a.w + gg * 27 + cc * 9 + ky * 3 + kx), a.n.mul[cc]), a.n.sub[cc], v);
        }
        wq[i] = v;
        atomicMax(&wmax_bits, __float_as_int(fabsf(v)));      // non-negative floats order like their bits
    }
    __syncthreads();
    // scale = 2^(14 - e) with max|w| = m 2^e, m in [0.5, 1): the largest scaled weight lies in [2^13, 2^14)
    const float wmax = __int_as_float(wmax_bits);
    int e = 0;
    if (wmax > 0.f && wmax < INFINITY) (void)frexpf(wmax, &e);
    const float scale = wmax > 0.f ? ldexpf(1.f, 14 - e) : 1.f, inv = wmax > 0.f ? ldexpf(1.f, e - 14) : 1.f;
    uint32_t bh[3][2], bl[3][2];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float w[2];
#pragma unroll
            for (int e2 = 0; e2 < 2; ++e2)
                w[e2] = t < 3 ? wq[((g * 3 + ky) * 3 + t) * 4 + 2 * h + e2] * scale : 0.f;
            so_split2(w[0], w[1], bh[ky][h], bl[ky][h]);
        }
    const float bias0 = __ldg(a.bias + 2 * t), bias1 = __ldg(a.bias + 2 * t + 1);
    uint32_t* raw = reinterpret_cast<uint32_t*>(smem + SU_REC);
    const uint8_t* rawb = smem + SU_REC;
    const int64_t hw = (int64_t)a.H * a.W;

    // the raw words of a tile's window: word wi of staged row si covers bytes 4 wi - 4 .. 4 wi - 1 counted from
    // the first byte of pixel (r0 - 1 + si, c0); pixel (., c0 - 1 + sj) sits at raw bytes 1 + 3 sj .. 3 + 3 sj
    constexpr int PPT = (SU_NRAW + SO_THREADS - 1) / SO_THREADS;
    // Tile coordinates advance incrementally (a tile is only 512 pixels: two run-time divisions per
    // tile and thread were a quarter of all instructions): tile = (img, ty, tx), step = gridDim.x tiles.
    const int tiles_y = a.tiles_per_img / a.tiles_x;
    const int st_img = (int)gridDim.x / a.tiles_per_img, st_rem = (int)gridDim.x - st_img * a.tiles_per_img;
    const int st_ty = st_rem / a.tiles_x, st_tx = st_rem - st_ty * a.tiles_x;
    int n_img, n_ty, n_tx;                                     // the tile whose window is being fetched
    // the (up to PPT) raw words and (up to 3) records a thread handles sit at the same window positions in
    // every tile
    int raw_si[PPT], raw_wi[PPT];
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        const int q = tid + k * SO_THREADS;
        raw_si[k] = q / SU_RAW_W;
        raw_wi[k] = q - raw_si[k] * SU_RAW_W;
    }
    constexpr int RROWS = SO_THREADS / SI_SPW;                // record rows per pass (7 of 18)
    const int rec_si = tid / SI_SPW, rec_sj = tid - rec_si * SI_SPW;
    const bool rec_on = rec_si < RROWS && rec_sj < SI_SREAL_C;
    uint32_t rv[PPT];
    auto fetch = [&]() {
        const int r0 = n_ty * SI_TH, c0 = n_tx * SI_TW;
        const uint8_t* base = reinterpret_cast<const uint8_t*>(a.x) + ((int64_t)n_img * hw + c0) * 3 - 4;
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            rv[k] = 0u;
            if (tid + k * SO_THREADS < SU_NRAW) {
                const int iy = r0 - 1 + raw_si[k];
                // the first / last word reach into the neighbouring row at the image's left / right edge
                const bool ok = iy >= 0 && iy < a.H && !(raw_wi[k] == 0 && c0 == 0) &&
                                !(raw_wi[k] == SU_RAW_W - 1 && c0 + SI_TW == a.W);
                if (ok)
                    rv[k] = __ldg(reinterpret_cast<const uint32_t*>(base + (int64_t)iy * a.W * 3) + raw_wi[k]);
            }
        }
    };
    n_img = (int)blockIdx.x / a.tiles_per_img;
    {
        const int trem = (int)blockIdx.x - n_img * a.tiles_per_img;
        n_ty = trem / a.tiles_x;
        n_tx = trem - n_ty * a.tiles_x;
    }
    if ((int)blockIdx.x < a.n_tiles) fetch();
    // per-warp constants of the MMA phase: M-tile mt = warp + 8 j (j = 0 .. 3) is pixels cb .. cb + 15 of
    // tile row (warp >> 1) + 4 j, cb = 16 (warp & 1)
    const int cb = (warp & 1) * 16, rr0 = warp >> 1;
    const uint8_t* pw = smem + (uint32_t)(rr0 * SI_SPW + cb + g + t) * 8;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int r0 = n_ty * SI_TH, c0 = n_tx * SI_TW;
        const int img = n_img;
#pragma unroll
        for (int k = 0; k < PPT; ++k)
            if (tid + k * SO_THREADS < SU_NRAW) raw[tid + k * SO_THREADS] = rv[k];
        __syncthreads();
        n_img += st_img; n_ty += st_ty; n_tx += st_tx;                       // the next tile of this CTA
        if (n_tx >= a.tiles_x) { n_tx -= a.tiles_x; ++n_ty; }
        if (n_ty >= tiles_y) { n_ty -= tiles_y; ++n_img; }
        if (tile + (int)gridDim.x < a.n_tiles) fetch();                      // in flight during this tile
        // ---- records: (R, G | B, inside) as fp16, zero outside the image (= the conv's padding) ----
        if (rec_on) {
            const int ix = c0 - 1 + rec_sj;
            const bool col_in = ix >= 0 && ix < a.W;
#pragma unroll
            for (int pass = 0; pass < (SI_SROWS + RROWS - 1) / RROWS; ++pass) {
                const int si = pass * RROWS + rec_si;
                if (si < SI_SROWS) {
                    const int iy = r0 - 1 + si;
                    uint2 rec = make_uint2(0u, 0u);
                    if (col_in && iy >= 0 && iy < a.H) {
                        const uint8_t* b = rawb + si * (SU_RAW_W * 4) + 1 + 3 * rec_sj;
                        // 0x6400 | n is the fp16 number 1024 + n (n < 1024): subtracting 1024 leaves n exactly
                        const uint32_t p01 = 0x64006400u | (uint32_t)b[0] | ((uint32_t)b[1] << 16);
                        const uint32_t p2m = 0x3C006400u | (uint32_t)b[2];             // high half: 1.0 = inside
                        const __half2 h01 = __hsub2(*reinterpret_cast<const __half2*>(&p01),
                                                    __floats2half2_rn(1024.f, 1024.f));
                        const __half2 h2m = __hsub2(*reinterpret_cast<const __half2*>(&p2m),
                                                    __floats2half2_rn(1024.f, 0.f));
                        rec.x = *reinterpret_cast<const uint32_t*>(&h01);
                        rec.y = *reinterpret_cast<const uint32_t*>(&h2m);
                    }
                    *reinterpret_cast<uint2*>(smem + (uint32_t)(si * SI_SPW + rec_sj) * 8) = rec;
                }
            }
        }
        __syncthreads();
        // ---- 32 M-tiles of 16 pixels of a row: four per warp, two at a time ----
        float* ow = a.out + (((size_t)img * a.H + r0 + rr0) * a.W + c0 + cb + g) * 8 + 2 * t;
        const size_t orow4 = (size_t)4 * a.W * 8;                 // four tile rows further
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
            float d[2][4];
#pragma unroll
            for (int u = 0; u < 2; ++u) d[u][0] = d[u][1] = d[u][2] = d[u][3] = 0.f;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const uint8_t* p = pw + ((2 * jj + u) * 4 + ky) * SI_SPW * 8;
                    const uint2 u0 = *reinterpret_cast<const uint2*>(p);
                    const uint2 u1 = *reinterpret_cast<const uint2*>(p + 8 * 8);
                    const uint32_t av[4] = {u0.x, u1.x, u0.y, u1.y};
                    mma_16816(d[u], av, bl[ky][0], bl[ky][1]);
                    mma_16816(d[u], av, bh[ky][0], bh[ky][1]);
                }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                float* o = ow + (2 * jj + u) * orow4;
                *reinterpret_cast<float2*>(o) = make_float2(fmaf(d[u][0], inv, bias0), fmaf(d[u][1], inv, bias1));
                *reinterpret_cast<float2*>(o + 64) = make_float2(fmaf(d[u][2], inv, bias0), fmaf(d[u][3], inv, bias1));
            }
        }
        __syncthreads();
    }
}

template <int XKIND>
int launch_stem_in_mma(const StemInArgs& a, int sm_count, cudaStream_t stream) {
    const int cap = sm_count * 4;
    const int grid = a.n_tiles < cap ? a.n_tiles : cap;
    stem_in_mma_kernel<XKIND><<<grid, SO_THREADS, SI_SMEM, stream>>>(a);
    return check_launch();
}

}  // namespace

bool stem_in_mma_supported(int H, int W, int c_out) {
    return c_out == 8 && H >= SI_TH && W >= SI_TW && H % SI_TH == 0 && W % SI_TW == 0;
}

int stem_in_mma(const void* x, int x_dtype, int x_layout, const float* w, const float* bias, float* out,
                int64_t B, int H, int W, int c_out, const float* mean, const float* stdv, int sm_count,
                cudaStream_t stream) {
    if (!x || !w || !bias || !out || B <= 0) return VQAE_ERR_BAD_ARG;
    if (!stem_in_mma_supported(H, W, c_out)) return VQAE_ERR_UNSUPPORTED;
    StemInArgs a{};
    a.x = x; a.w = w; a.bias = bias; a.out = out; a.H = H; a.W = W;
    a.tiles_x = W / SI_TW; a.tiles_per_img = (H / SI_TH) * a.tiles_x;
    const int64_t nt = B * a.tiles_per_img;
    if (nt > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    a.n_tiles = (int)nt;
    if (x_dtype == VQAE_DT_U8) {
        if (!mean || !stdv) return VQAE_ERR_BAD_ARG;
        if (x_layout != VQAE_LAYOUT_NHWC) return VQAE_ERR_UNSUPPORTED;
        for (int c = 0; c < 3; ++c) {
            a.n.sub[c] = mean[c] * 255.0f;
            a.n.mul[c] = 1.0f / (stdv[c] * 255.0f);
        }
        if ((reinterpret_cast<uintptr_t>(x) & 3u) == 0) {            // 32-bit window loads
            const int cap = sm_count * 4;
            const int grid = a.n_tiles < cap ? a.n_tiles : cap;
            stem_in_u8_mma_kernel<<<grid, SO_THREADS, SU_SMEM, stream>>>(a);
            return check_launch();
        }
        return launch_stem_in_mma<2>(a, sm_count, stream);
    }
    if (x_dtype != VQAE_DT_F32) return VQAE_ERR_UNSUPPORTED;
    return x_layout == VQAE_LAYOUT_NCHW ? launch_stem_in_mma<0>(a, sm_count, stream)
                                        : launch_stem_in_mma<1>(a, sm_count, stream);
}

bool stem_out_mma_supported(int H, int W, int c_in) {
    return c_in == 8 && H >= SO_TH && W >= SO_TW && H % SO_TH == 0 && W % SO_TW == 0;
}

int stem_out_mma(const float* x, const float* w, const float* bias, float* out, int out_layout,
                 int64_t B, int H, int W, int c_in, int sm_count, cudaStream_t stream) {
    if (!x || !w || !bias || !out || B <= 0) return VQAE_ERR_BAD_ARG;
    if (!stem_out_mma_supported(H, W, c_in)) return VQAE_ERR_UNSUPPORTED;
    if (out_layout != VQAE_LAYOUT_NCHW && out_layout != VQAE_LAYOUT_NHWC) return VQAE_ERR_BAD_ARG;
    StemOutArgs a;
    a.x = x; a.w = w; a.bias = bias; a.out = out; a.H = H; a.W = W;
    a.nhwc_out = out_layout == VQAE_LAYOUT_NHWC;
    a.tiles_x = W / SO_TW; a.tiles_per_img = (H / SO_TH) * a.tiles_x;
    const int64_t nt = B * a.tiles_per_img;
    if (nt > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    a.n_tiles = (int)nt;
    const int cap = sm_count * 3;
    const int grid = a.n_tiles < cap ? a.n_tiles : cap;
    stem_out_mma_kernel<false><<<grid, SO_THREADS, SO_SMEM, stream>>>(a);
    return check_launch();
}

int stem_out_mma_u8(const float* x, const float* w, const float* bias, const U8Canvas& cv, int64_t B,
                    int H, int W, int c_in, int sm_count, cudaStream_t stream) {
    if (!x || !w || !bias) return VQAE_ERR_BAD_ARG;
    if (!stem_out_mma_supported(H, W, c_in)) return VQAE_ERR_UNSUPPORTED;
    StemOutArgs a{};
    a.x = x; a.w = w; a.bias = bias; a.out = nullptr; a.H = H; a.W = W; a.cv = cv;
    a.tiles_x = W / SO_TW; a.tiles_per_img = (H / SO_TH) * a.tiles_x;
    const int64_t nt = B * a.tiles_per_img;
    if (nt > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    a.n_tiles = (int)nt;
    const int cap = sm_count * 3;
    const int grid = a.n_tiles < cap ? a.n_tiles : cap;
    stem_out_mma_kernel<true><<<grid, SO_THREADS, SO_SMEM + SO_WARPS * 192, stream>>>(a);
    return check_launch();
}

}  // namespace vqae

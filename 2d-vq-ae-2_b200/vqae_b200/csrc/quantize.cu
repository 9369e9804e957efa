// Fused quantiser (exact fp32 CUDA-core form) + code gather + code-map placement.
//
// Reference: ProjectedEMAVectorQuantizer2d.forward / EMAVectorQuantizer.forward in eval mode
// (vq_ae/layers/vq.py:96-154,185-192).  One kernel does, per latent vector,
//   z   = proj_in(x)                                   (vq.py:191, 1x1 conv C -> D, bias)
//   idx = argmin_k sum_d ((z_d - e_kd)^2)^2            (vq.py:121-129: cdist with p = ndim = 4;
//                                                       the 4th root is monotone and is dropped)
//   out = E'[idx],  E' = proj_out(embed)               (vq.py:130,192 -- gather of a
//                                                       precomputed [K][C] table)
//   loss partial = sum_d (z_d - e_idx,d)^2             (vq.py:143)
// without materialising the N x K distance matrix.  Ties resolve to the lowest index
// (strict '<' while scanning k upward), like torch.argmin.
#include "common.cuh"
#include "kernels.cuh"

namespace vqae {
namespace {

constexpr int QT = 128;  // vectors (= threads) per CTA
constexpr int QD = 8;    // distance-space dimension

struct QArgs {
    const float* x;
    float* out;
    int64_t* idx;
    float* partial;  // [gridDim.x] per-CTA loss partial sums
    uint32_t* near_ties;
    float* z_out;
    const float* embed;
    const float* w_in;
    const float* b_in;
    const float* table;
    int64_t N, S;
    int K, C;
    float tie_rel_gap;
};

// XL / OL: layout of x / out (0 NCHW, 1 NHWC);  PROJ: proj_in present
template <int XL, int OL, bool PROJ>
__global__ void __launch_bounds__(QT) quantize_kernel(QArgs a) {
    extern __shared__ __align__(16) float smem[];
    float* cb = smem;                                   // [K][8]
    float* wi = cb + a.K * QD;                          // [C][8]  (PROJ only)
    float* bi = wi + (PROJ ? a.C * QD : 0);             // [8]
    float* stage = bi + QD;                             // [QT][C + 4]  (PROJ && NHWC only)
    __shared__ int sidx[QT];
    __shared__ float sred[QT / 32];

    const int tid = threadIdx.x;
    const int64_t n0 = (int64_t)blockIdx.x * QT;
    const int64_t n = n0 + tid;
    const bool ok = n < a.N;
    const int C = a.C;

    for (int i = tid; i < a.K * QD / 4; i += QT)
        reinterpret_cast<float4*>(cb)[i] = __ldg(reinterpret_cast<const float4*>(a.embed) + i);
    if (PROJ) {
        // w_in is [D][C] (OIHW, 1x1) -> wi[c][d]
        for (int i = tid; i < C * QD; i += QT) {
            const int d = i / C, c = i % C;
            wi[c * QD + d] = __ldg(a.w_in + i);
        }
        if (tid < QD) bi[tid] = __ldg(a.b_in + tid);
    }
    const int LDS_ = C + 4;
    if (PROJ && XL == VQAE_LAYOUT_NHWC) {
        // coalesced copy of the contiguous [QT][C] tile
        const int c4n = C / 4;
        const int64_t tile_f4 = (int64_t)QT * c4n;
        const int64_t lim_f4 = (a.N - n0) * c4n;
        const float4* src = reinterpret_cast<const float4*>(a.x) + n0 * c4n;
        for (int64_t i = tid; i < tile_f4 && i < lim_f4; i += QT) {
            const int row = (int)(i / c4n), c4 = (int)(i % c4n);
            *reinterpret_cast<float4*>(stage + row * LDS_ + c4 * 4) = __ldg(src + i);
        }
    }
    __syncthreads();

    // ---- z = proj_in(x) (or x itself) ----
    float z[QD];
#pragma unroll
    for (int d = 0; d < QD; ++d) z[d] = 0.f;
    int64_t b = 0, s = 0;
    if (ok) {
        b = n / a.S;
        s = n - b * a.S;
    }
    if (ok) {
        if (PROJ) {
            if (XL == VQAE_LAYOUT_NHWC) {
                const float* row = stage + tid * LDS_;
                for (int c = 0; c < C; c += 4) {
                    const float4 v = *reinterpret_cast<const float4*>(row + c);
                    const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 w0 = *reinterpret_cast<const float4*>(wi + (c + j) * QD);
                        const float4 w1 = *reinterpret_cast<const float4*>(wi + (c + j) * QD + 4);
                        z[0] = fmaf(vv[j], w0.x, z[0]); z[1] = fmaf(vv[j], w0.y, z[1]);
                        z[2] = fmaf(vv[j], w0.z, z[2]); z[3] = fmaf(vv[j], w0.w, z[3]);
                        z[4] = fmaf(vv[j], w1.x, z[4]); z[5] = fmaf(vv[j], w1.y, z[5]);
                        z[6] = fmaf(vv[j], w1.z, z[6]); z[7] = fmaf(vv[j], w1.w, z[7]);
                    }
                }
            } else {
                const float* px = a.x + b * C * a.S + s;
#pragma unroll 4
                for (int c = 0; c < C; ++c) {
                    const float v = __ldg(px + (int64_t)c * a.S);
                    const float4 w0 = *reinterpret_cast<const float4*>(wi + c * QD);
                    const float4 w1 = *reinterpret_cast<const float4*>(wi + c * QD + 4);
                    z[0] = fmaf(v, w0.x, z[0]); z[1] = fmaf(v, w0.y, z[1]);
                    z[2] = fmaf(v, w0.z, z[2]); z[3] = fmaf(v, w0.w, z[3]);
                    z[4] = fmaf(v, w1.x, z[4]); z[5] = fmaf(v, w1.y, z[5]);
                    z[6] = fmaf(v, w1.z, z[6]); z[7] = fmaf(v, w1.w, z[7]);
                }
            }
#pragma unroll
            for (int d = 0; d < QD; ++d) z[d] += bi[d];
        } else {
            if (XL == VQAE_LAYOUT_NHWC) {
                const float4 v0 = __ldg(reinterpret_cast<const float4*>(a.x + n * QD));
                const float4 v1 = __ldg(reinterpret_cast<const float4*>(a.x + n * QD) + 1);
                z[0] = v0.x; z[1] = v0.y; z[2] = v0.z; z[3] = v0.w;
                z[4] = v1.x; z[5] = v1.y; z[6] = v1.z; z[7] = v1.w;
            } else {
#pragma unroll
                for (int d = 0; d < QD; ++d) z[d] = __ldg(a.x + (b * QD + d) * a.S + s);
            }
        }
    }

    // ---- L4 argmin over the SMEM codebook, d-ordered fp32 accumulation ----
    float best = INFINITY, second = INFINITY;
    int bidx = 0;
#pragma unroll 4
    for (int k = 0; k < a.K; ++k) {
        const float4 e0 = *reinterpret_cast<const float4*>(cb + k * QD);
        const float4 e1 = *reinterpret_cast<const float4*>(cb + k * QD + 4);
        float d, q, acc;
        d = z[0] - e0.x; q = d * d; acc = q * q;
        d = z[1] - e0.y; q = d * d; acc = fmaf(q, q, acc);
        d = z[2] - e0.z; q = d * d; acc = fmaf(q, q, acc);
        d = z[3] - e0.w; q = d * d; acc = fmaf(q, q, acc);
        d = z[4] - e1.x; q = d * d; acc = fmaf(q, q, acc);
        d = z[5] - e1.y; q = d * d; acc = fmaf(q, q, acc);
        d = z[6] - e1.z; q = d * d; acc = fmaf(q, q, acc);
        d = z[7] - e1.w; q = d * d; acc = fmaf(q, q, acc);
        if (acc < best) {
            second = best;
            best = acc;
            bidx = k;
        } else if (acc < second) {
            second = acc;
        }
    }

    // ---- per-vector outputs ----
    float sq = 0.f;
    bool tie = false;
    if (ok) {
        const float* e = cb + bidx * QD;
#pragma unroll
        for (int d = 0; d < QD; ++d) {
            const float df = z[d] - e[d];
            sq = fmaf(df, df, sq);
        }
        a.idx[n] = bidx;
        tie = (second - best) < a.tie_rel_gap * second;
        if (!PROJ && a.out != nullptr) {
            // bare quantiser: the reference returns inputs + (quantized - inputs) (straight-through
            // estimator, vq.py:146), which differs from the codebook row by up to one ulp
            float o[QD];
#pragma unroll
            for (int d = 0; d < QD; ++d) o[d] = __fadd_rn(z[d], __fsub_rn(e[d], z[d]));
            if (OL == VQAE_LAYOUT_NHWC) {
                float4* po = reinterpret_cast<float4*>(a.out + n * QD);
                po[0] = make_float4(o[0], o[1], o[2], o[3]);
                po[1] = make_float4(o[4], o[5], o[6], o[7]);
            } else {
#pragma unroll
                for (int d = 0; d < QD; ++d) a.out[(b * QD + d) * a.S + s] = o[d];
            }
        }
        if (a.z_out) {
            float4* zo = reinterpret_cast<float4*>(a.z_out + n * QD);
            zo[0] = make_float4(z[0], z[1], z[2], z[3]);
            zo[1] = make_float4(z[4], z[5], z[6], z[7]);
        }
    }
    sidx[tid] = bidx;

    // loss partial: deterministic in-CTA tree, one slot per CTA
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((tid & 31) == 0) sred[tid >> 5] = sq;
    if (a.near_ties) {
        const unsigned m = __ballot_sync(0xffffffffu, tie);
        if ((tid & 31) == 0 && m) atomicAdd(a.near_ties, (uint32_t)__popc(m));
    }
    __syncthreads();
    if (tid == 0) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < QT / 32; ++w) t += sred[w];
        a.partial[blockIdx.x] = t;
    }

    // ---- out rows = table[idx] ----
    if (a.out == nullptr || !PROJ) return;
    if (OL == VQAE_LAYOUT_NHWC) {
        const int c4n = C / 4;
        const int64_t tile_f4 = (int64_t)QT * c4n;
        const int64_t lim_f4 = (a.N - n0) * c4n;
        float4* dst = reinterpret_cast<float4*>(a.out) + n0 * c4n;
        const float4* tab = reinterpret_cast<const float4*>(a.table);
        for (int64_t i = tid; i < tile_f4 && i < lim_f4; i += QT) {
            const int row = (int)(i / c4n), c4 = (int)(i % c4n);
            dst[i] = __ldg(tab + (int64_t)sidx[row] * c4n + c4);
        }
    } else if (ok) {
        const float4* trow = reinterpret_cast<const float4*>(a.table + (int64_t)bidx * C);
        float* po = a.out + b * C * a.S + s;
        for (int c4 = 0; c4 < C / 4; ++c4) {
            const float4 v = __ldg(trow + c4);
            po[(int64_t)(c4 * 4 + 0) * a.S] = v.x;
            po[(int64_t)(c4 * 4 + 1) * a.S] = v.y;
            po[(int64_t)(c4 * 4 + 2) * a.S] = v.z;
            po[(int64_t)(c4 * 4 + 3) * a.S] = v.w;
        }
    }
}

// loss = sum(partials) / (N * D) * commitment_cost, summed in a fixed order in fp64
__global__ void __launch_bounds__(256)
loss_finalize_kernel(const float* __restrict__ partial, int nparts, double inv_count, float cc,
                     float* __restrict__ loss) {
    __shared__ double sh[256];
    double t = 0.0;
    for (int i = threadIdx.x; i < nparts; i += 256) t += (double)partial[i];
    sh[threadIdx.x] = t;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *loss = (float)(sh[0] * inv_count) * cc;
}

// table[k][c] = b_out[c] + sum_d w_out[c][d] * embed[k][d]   (proj_out of every code)
__global__ void __launch_bounds__(256)
table_kernel(const float* __restrict__ embed, const float* __restrict__ w_out,
             const float* __restrict__ b_out, float* __restrict__ table, int K, int D, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * C) return;
    const int k = i / C, c = i % C;
    if (w_out == nullptr) {
        table[i] = embed[k * D + c];
        return;
    }
    float acc = 0.f;
    for (int d = 0; d < D; ++d) acc = fmaf(w_out[c * D + d], embed[k * D + d], acc);
    table[i] = acc + (b_out ? b_out[c] : 0.f);
}

template <bool U8>
__global__ void __launch_bounds__(256)
embed_codes_kernel(const void* __restrict__ indices, const float* __restrict__ table, int K,
                   int C, float* __restrict__ out, int out_layout, int64_t N, int64_t S) {
    const int c4n = C / 4;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * c4n) return;
    const float4* tab = reinterpret_cast<const float4*>(table);
    if (out_layout == VQAE_LAYOUT_NHWC) {
        const int64_t n = i / c4n;
        const int c4 = (int)(i % c4n);
        int64_t k = U8 ? (int64_t) reinterpret_cast<const uint8_t*>(indices)[n]
                       : reinterpret_cast<const int64_t*>(indices)[n];
        k = k < 0 ? 0 : (k >= K ? K - 1 : k);
        reinterpret_cast<float4*>(out)[i] = __ldg(tab + k * c4n + c4);
    } else {
        // thread = (b, c4, s): consecutive threads walk s -> coalesced plane writes
        const int64_t s = i % S;
        const int64_t r = i / S;
        const int c4 = (int)(r % c4n);
        const int64_t b = r / c4n;
        const int64_t n = b * S + s;
        int64_t k = U8 ? (int64_t) reinterpret_cast<const uint8_t*>(indices)[n]
                       : reinterpret_cast<const int64_t*>(indices)[n];
        k = k < 0 ? 0 : (k >= K ? K - 1 : k);
        const float4 v = __ldg(tab + k * c4n + c4);
        float* po = out + (b * C + c4 * 4) * S + s;
        po[0] = v.x;
        po[S] = v.y;
        po[2 * S] = v.z;
        po[3 * S] = v.w;
    }
}

// embed_codes on a window of a stored code map: patch t of the call is region patch first_patch + t
// (region_cols patches per region row, region origin (r0, c0) in patches), code (y, x) of it sits at
// map[((r0 + pr) th + y) map_cols + (c0 + pc) tw + x].  Thread j of image row blockIdx.y writes float4
// j of the patch's NHWC rows: consecutive threads read consecutive codes of one map row (each code
// once per C / 4 threads) and write consecutive output float4s.
template <bool U8>
__global__ void __launch_bounds__(256)
embed_codemap_kernel(const void* __restrict__ map, int64_t map_cols, int th, int tw, int64_t r0,
                     int64_t c0, int64_t region_cols, int64_t first_patch, int64_t n,
                     const float4* __restrict__ tab, int K, int c4n, float4* __restrict__ out) {
    const int per_patch = th * tw * c4n;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= per_patch) return;
    const int pix = j / c4n, c4 = j - pix * c4n;
    const int y = pix / tw, x = pix - y * tw;
    for (int64_t t = blockIdx.y; t < n; t += gridDim.y) {
        const int64_t q = first_patch + t;
        const int64_t pr = q / region_cols, pc = q - pr * region_cols;
        const int64_t m = ((r0 + pr) * th + y) * map_cols + (c0 + pc) * tw + x;
        int64_t k = U8 ? (int64_t) reinterpret_cast<const uint8_t*>(map)[m]
                       : reinterpret_cast<const int64_t*>(map)[m];
        k = k < 0 ? 0 : (k >= K ? K - 1 : k);                   // embed_codes_kernel's clamping
        out[t * per_patch + j] = __ldg(tab + k * c4n + c4);
    }
}

template <typename MapT>
__global__ void __launch_bounds__(256)
codemap_place_kernel(const int64_t* __restrict__ tiles, int64_t total, int th, int tw,
                     int64_t first_patch, int grid_cols, MapT* __restrict__ map,
                     int64_t map_cols) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int x = (int)(i % tw);
    const int64_t r = i / tw;
    const int y = (int)(r % th);
    const int64_t t = r / th;
    const int64_t patch = first_patch + t;
    const int64_t prow = patch / grid_cols, pcol = patch % grid_cols;
    map[(prow * th + y) * map_cols + pcol * tw + x] = (MapT)tiles[i];
}

}  // namespace

int quantizer_prepare_f32(const float* embed, int K, int D, const float* w_out,
                          const float* b_out, int C, float* table, cudaStream_t stream) {
    if (!embed || !table || K <= 0 || D <= 0 || C <= 0) return VQAE_ERR_BAD_ARG;
    if (w_out == nullptr && C != D) return VQAE_ERR_DIM_MISMATCH;
    table_kernel<<<ceil_div_u((int64_t)K * C, 256), 256, 0, stream>>>(embed, w_out, b_out, table,
                                                                      K, D, C);
    return check_launch();
}

size_t quantizer_scratch_bytes(int64_t n) {
    if (n <= 0) return 0;
    const size_t a = (size_t)((n + QT - 1) / QT) * sizeof(float), b = quantize_tc_scratch_bytes(n);
    return a > b ? a : b;
}

template <int XL, int OL, bool PROJ>
static int launch_q(const QArgs& a, size_t smem, unsigned grid, cudaStream_t stream) {
    auto kern = quantize_kernel<XL, OL, PROJ>;
    if (smem > 48 * 1024)
        VQAE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)smem));
    kern<<<grid, QT, smem, stream>>>(a);
    return check_launch();
}

bool quantize_supported(const vqae_quantizer_params* p, int x_dtype, int x_layout, int out_dtype,
                        int out_layout, bool has_out, int kernel) {
    if (!p) return false;
    const bool f32 = x_dtype == VQAE_DT_F32 && (!has_out || out_dtype == VQAE_DT_F32);
    const bool io_ok = (x_dtype == VQAE_DT_F32 || x_dtype == VQAE_DT_BF16 || x_dtype == VQAE_DT_F16) &&
                       (!has_out || out_dtype == x_dtype);
    const bool tc = io_ok && quantize_tc_supported(p, x_layout, out_layout, has_out);
    const bool cc = f32 && p->dim == QD && p->num_codes > 0 && p->num_codes <= 1024;
    if (kernel == VQAE_QUANT_TENSOR_CORE) return tc;
    if (kernel == VQAE_QUANT_CUDA_CORE) return cc;
    return tc || cc;
}

int quantize_any(const vqae_quantizer_params* p, const void* x, int x_dtype, int x_layout, void* out,
                 int out_dtype, int out_layout, int64_t* indices, float* loss, uint32_t* near_ties,
                 float tie_rel_gap, float* z_out, void* scratch, size_t scratch_bytes, int64_t B,
                 int64_t S, int kernel, cudaStream_t stream) {
    if (!p) return VQAE_ERR_BAD_ARG;
    if (kernel < VQAE_QUANT_AUTO || kernel > VQAE_QUANT_TENSOR_CORE) return VQAE_ERR_BAD_ARG;
    if (!quantize_supported(p, x_dtype, x_layout, out_dtype, out_layout, out != nullptr, kernel))
        return VQAE_ERR_UNSUPPORTED;
    if (x_dtype != VQAE_DT_F32) {
        // 16-bit I/O exists on the tcgen05 kernel only (fp32 distance arithmetic inside)
        if (!x || !indices || !loss || !p->embed || B <= 0 || S <= 0) return VQAE_ERR_BAD_ARG;
        if (out && !p->table) return VQAE_ERR_BAD_ARG;
        const int64_t N = B * S;
        if (!scratch || scratch_bytes < quantizer_scratch_bytes(N)) return VQAE_ERR_SCRATCH;
        int sm_count = 0;
        if (int rc = device_sm_count(&sm_count)) return rc;
        return quantize_tc(p, x, out, x_dtype, indices, loss, scratch, near_ties, tie_rel_gap, z_out,
                           nullptr, N, sm_count, stream);
    }
    return quantize_f32(p, reinterpret_cast<const float*>(x), x_layout, reinterpret_cast<float*>(out),
                        out_layout, indices, loss, near_ties, tie_rel_gap, z_out, scratch,
                        scratch_bytes, B, S, stream, kernel);
}

int quantize_f32(const vqae_quantizer_params* p, const float* x, int x_layout, float* out,
                 int out_layout, int64_t* indices, float* loss, uint32_t* near_ties,
                 float tie_rel_gap, float* z_out, void* scratch, size_t scratch_bytes, int64_t B,
                 int64_t S, cudaStream_t stream, int kernel) {
    if (!p || !x || !indices || !loss || !p->embed || B <= 0 || S <= 0) return VQAE_ERR_BAD_ARG;
    if (out && !p->table) return VQAE_ERR_BAD_ARG;
    if (p->dim != QD) return VQAE_ERR_UNSUPPORTED;
    if (p->num_codes <= 0 || p->num_codes > 1024) return VQAE_ERR_UNSUPPORTED;
    const bool proj = p->w_in != nullptr;
    if (!proj && p->c != p->dim) return VQAE_ERR_DIM_MISMATCH;  // vq.py:100-104
    if (proj && (!p->b_in || p->c % 4 != 0 || p->c > 512)) return VQAE_ERR_UNSUPPORTED;
    const int64_t N = B * S;
    const size_t need = quantizer_scratch_bytes(N);
    if (!scratch || scratch_bytes < need) return VQAE_ERR_SCRATCH;

    QArgs a;
    a.x = x; a.out = out; a.idx = indices; a.partial = reinterpret_cast<float*>(scratch);
    a.near_ties = near_ties; a.z_out = z_out; a.embed = p->embed; a.w_in = p->w_in;
    a.b_in = p->b_in; a.table = p->table; a.N = N; a.S = S; a.K = p->num_codes; a.C = p->c;
    a.tie_rel_gap = tie_rel_gap;

    if (kernel != VQAE_QUANT_CUDA_CORE && quantize_tc_supported(p, x_layout, out_layout, out != nullptr)) {
        // fused kernel: loss and near-tie totals are reduced by its last CTA (no memset / finalize)
        int sm_count = 0;
        if (int rc = device_sm_count(&sm_count)) return rc;
        return quantize_tc_f32(p, x, out, indices, loss, scratch, near_ties, tie_rel_gap, z_out,
                               nullptr, N, sm_count, stream);
    }
    if (near_ties) VQAE_CUDA_TRY(cudaMemsetAsync(near_ties, 0, sizeof(uint32_t), stream));

    const unsigned grid = ceil_div_u(N, QT);
    size_t smem = ((size_t)p->num_codes * QD + QD) * sizeof(float);
    if (proj) smem += (size_t)p->c * QD * sizeof(float);
    if (proj && x_layout == VQAE_LAYOUT_NHWC) smem += (size_t)QT * (p->c + 4) * sizeof(float);
    if (smem > 227 * 1024) return VQAE_ERR_UNSUPPORTED;

    int rc;
    const int xl = x_layout == VQAE_LAYOUT_NHWC, ol = out_layout == VQAE_LAYOUT_NHWC;
#define VQ_DISPATCH(XL, OL)                                                   \
    (proj ? launch_q<XL, OL, true>(a, smem, grid, stream)                     \
          : launch_q<XL, OL, false>(a, smem, grid, stream))
    if (xl && ol) rc = VQ_DISPATCH(1, 1);
    else if (xl) rc = VQ_DISPATCH(1, 0);
    else if (ol) rc = VQ_DISPATCH(0, 1);
    else rc = VQ_DISPATCH(0, 0);
#undef VQ_DISPATCH
    if (rc != VQAE_OK) return rc;

    loss_finalize_kernel<<<1, 256, 0, stream>>>(a.partial, (int)grid,
                                                1.0 / ((double)N * (double)QD),
                                                p->commitment_cost, loss);
    return check_launch();
}

int embed_codes_f32(const void* indices, int idx_is_u8, const float* table, int K, int C,
                    float* out, int out_layout, int64_t B, int64_t S, cudaStream_t stream) {
    if (!indices || !table || !out || B <= 0 || S <= 0 || K <= 0) return VQAE_ERR_BAD_ARG;
    if (C % 4 != 0) return VQAE_ERR_UNSUPPORTED;
    const int64_t total = B * S * (C / 4);
    const unsigned grid = ceil_div_u(total, 256);
    if (idx_is_u8)
        embed_codes_kernel<true><<<grid, 256, 0, stream>>>(indices, table, K, C, out, out_layout,
                                                           B * S, S);
    else
        embed_codes_kernel<false><<<grid, 256, 0, stream>>>(indices, table, K, C, out, out_layout,
                                                            B * S, S);
    return check_launch();
}

int embed_codemap_f32(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int th,
                      int tw, int64_t r0, int64_t c0, int64_t region_cols, int64_t first_patch,
                      int64_t n, const float* table, int K, int C, float* out, cudaStream_t stream) {
    if (!map || !table || !out || map_rows <= 0 || map_cols <= 0 || th <= 0 || tw <= 0 || n <= 0 ||
        region_cols <= 0 || K <= 0 || C <= 0 || r0 < 0 || c0 < 0 || first_patch < 0)
        return VQAE_ERR_BAD_ARG;
    const int64_t last = first_patch + n - 1;               // the window must lie inside the map
    if ((r0 + last / region_cols + 1) * th > map_rows || (c0 + region_cols) * tw > map_cols)
        return VQAE_ERR_BAD_ARG;
    if (C % 4 != 0 || (int64_t)th * tw * (C / 4) > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    const int c4n = C / 4;
    const dim3 grid(ceil_div_u((int64_t)th * tw * c4n, 256), (unsigned)(n < 65535 ? n : 65535));
    const float4* tab = reinterpret_cast<const float4*>(table);
    float4* o4 = reinterpret_cast<float4*>(out);
    if (map_is_u8)
        embed_codemap_kernel<true><<<grid, 256, 0, stream>>>(map, map_cols, th, tw, r0, c0, region_cols,
                                                             first_patch, n, tab, K, c4n, o4);
    else
        embed_codemap_kernel<false><<<grid, 256, 0, stream>>>(map, map_cols, th, tw, r0, c0, region_cols,
                                                              first_patch, n, tab, K, c4n, o4);
    return check_launch();
}

template <typename MapT>
static int codemap_place(const int64_t* tiles, int64_t n_tiles, int th, int tw, int64_t first_patch,
                         int grid_cols, MapT* map, int64_t map_rows, int64_t map_cols,
                         cudaStream_t stream) {
    if (!tiles || !map || n_tiles <= 0 || th <= 0 || tw <= 0 || grid_cols <= 0)
        return VQAE_ERR_BAD_ARG;
    const int64_t last = first_patch + n_tiles - 1;
    if (first_patch < 0 || (last / grid_cols + 1) * th > map_rows ||
        (int64_t)grid_cols * tw > map_cols)
        return VQAE_ERR_BAD_ARG;
    const int64_t total = n_tiles * th * tw;
    codemap_place_kernel<MapT><<<ceil_div_u(total, 256), 256, 0, stream>>>(
        tiles, total, th, tw, first_patch, grid_cols, map, map_cols);
    return check_launch();
}

int codemap_place_u8(const int64_t* tiles, int64_t n_tiles, int th, int tw, int64_t first_patch,
                     int grid_cols, uint8_t* map, int64_t map_rows, int64_t map_cols,
                     cudaStream_t stream) {
    return codemap_place<uint8_t>(tiles, n_tiles, th, tw, first_patch, grid_cols, map, map_rows,
                                  map_cols, stream);
}

int codemap_place_i64(const int64_t* tiles, int64_t n_tiles, int th, int tw, int64_t first_patch,
                      int grid_cols, int64_t* map, int64_t map_rows, int64_t map_cols,
                      cudaStream_t stream) {
    return codemap_place<int64_t>(tiles, n_tiles, th, tw, first_patch, grid_cols, map, map_rows,
                                  map_cols, stream);
}

}  // namespace vqae

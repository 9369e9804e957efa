// extern "C" boundary (include/vqae_b200.h): argument checks, block composition, launch counting.
#include <atomic>

#include "common.cuh"
#include "kernels.cuh"

namespace vqae {

static thread_local cudaError_t g_last_error = cudaSuccess;
static std::atomic<uint64_t> g_launches{0};

void set_last_cuda_error(cudaError_t e) { g_last_error = e; }
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct FixupScratch {
    size_t t1, t2, t3, skip, total;  // byte offsets
};

// byte layout of the scratch buffer of one block call
static FixupScratch fixup_layout(const vqae_fixup_params* p, int64_t B, int H, int W) {
    FixupScratch s{};
    const size_t px = (size_t)B * H * W;
    const size_t cb = (size_t)p->c_branch, co = (size_t)p->c_out;
    size_t off = 0;
    auto take = [&](size_t elems) {
        size_t o = off;
        off += align256(elems * sizeof(float));
        return o;
    };
    if (p->mode == VQAE_MODE_SAME) {
        s.t1 = take(px * cb);
        s.t2 = take(px * cb);
    } else if (p->mode == VQAE_MODE_DOWN) {
        s.t1 = take(px * cb);
        s.t2 = take(px / 4 * cb);
        s.skip = take(px / 4 * co);
    } else {
        // branch_conv1 output, low res; the low-res skip conv output (c_out channels) reuses it
        // after branch_conv2 has consumed it, so it must hold the wider of the two
        s.t1 = take(px * (cb > co ? cb : co));
        s.t2 = take(px * cb);        // 1x1 of branch_conv2 applied at low res
        s.t3 = take(px * 4 * cb);    // ... upsampled
        s.skip = take(px * 4 * co);  // upsampled skip
    }
    s.total = off;
    return s;
}

}  // namespace vqae

using namespace vqae;

extern "C" {

int vqae_abi_version(void) { return VQAE_ABI_VERSION; }

const char* vqae_error_string(int code) {
    switch (code) {
        case VQAE_OK: return "ok";
        case VQAE_ERR_BAD_ARG: return "bad argument (null pointer or non-positive extent)";
        case VQAE_ERR_UNSUPPORTED: return "shape/dtype/layout not supported by the sm_100a kernels";
        case VQAE_ERR_DIM_MISMATCH: return "VQ dim != channel dim not supported";
        case VQAE_ERR_CUDA: return "CUDA runtime error";
        case VQAE_ERR_SCRATCH: return "scratch buffer missing or too small";
    }
    return "unknown error";
}

const char* vqae_last_cuda_error(void) { return cudaGetErrorString(g_last_error); }

uint64_t vqae_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int vqae_normalize_u8(const uint8_t* img, float* out, int64_t batch, int height, int width,
                      const float* mean_host, const float* std_host, int out_layout,
                      void* stream) {
    return normalize_u8(img, out, batch, height, width, mean_host, std_host, out_layout,
                        (cudaStream_t)stream);
}

int vqae_pack_conv_weight_f32(const float* w_oihw, float* packed, int out_ch, int in_ch, int kh,
                              int kw, void* stream) {
    return pack_conv_weight_f32(w_oihw, packed, out_ch, in_ch, kh * kw, (cudaStream_t)stream);
}

size_t vqae_pack_elems(int kind, int c_in, int c_out, int taps) {
    return pack_elems(kind, c_in, c_out, taps);
}

int vqae_pack_batched(const vqae_pack_desc* descs_device, int n_descs, int max_elems, void* stream) {
    return pack_batched(descs_device, n_descs, max_elems, (cudaStream_t)stream);
}

int vqae_stem_in_f32(const void* x, int x_dtype, int x_layout, const float* w_oihw,
                     const float* bias, float* out, int64_t batch, int height, int width,
                     int c_out, const float* mean_host, const float* std_host, void* stream) {
    return stem_in_f32(x, x_dtype, x_layout, w_oihw, bias, out, VQAE_DT_F32, batch, height, width,
                       c_out, mean_host, std_host, (cudaStream_t)stream);
}

int vqae_stem_in(const void* x, int x_dtype, int x_layout, const float* w_oihw, const float* bias,
                 void* out, int out_dtype, int64_t batch, int height, int width, int c_out,
                 const float* mean_host, const float* std_host, void* stream) {
    return stem_in_f32(x, x_dtype, x_layout, w_oihw, bias, out, out_dtype, batch, height, width,
                       c_out, mean_host, std_host, (cudaStream_t)stream);
}

int vqae_stem_out_f32(const float* x, const float* w_oihw, const float* bias, float* out,
                      int out_layout, int64_t batch, int height, int width, int c_in,
                      void* stream) {
    return stem_out_f32(x, w_oihw, bias, out, out_layout, batch, height, width, c_in,
                        (cudaStream_t)stream);
}

int vqae_conv_f32(int kind, const float* x, const float* w_packed, float* out,
                  const float* residual, int64_t batch, int height, int width, int c_in,
                  int c_out, float pre_add, int pre_elu, float post_add, float scale, float bias,
                  void* stream) {
    if (kind < CONV_1x1 || kind > CONV_3x3_CIRC) return VQAE_ERR_BAD_ARG;
    return conv_f32(kind, x, w_packed, out, residual, batch, height, width, c_in, c_out,
                    PreOp{pre_add, post_add, pre_elu}, scale, bias, (cudaStream_t)stream);
}

int vqae_bicubic_up2_f32(const float* x, float* out, int64_t batch, int height, int width, int c,
                         float bias, void* stream) {
    return bicubic_up2_f32(x, out, batch, height, width, c, bias, (cudaStream_t)stream);
}

size_t vqae_fixup_block_scratch_bytes(const vqae_fixup_params* p, int64_t batch, int height,
                                      int width) {
    if (!p || batch <= 0 || height <= 0 || width <= 0) return 0;
    return fixup_layout(p, batch, height, width).total;
}

int vqae_fixup_block_f32(const vqae_fixup_params* p, const float* x, float* out, void* scratch,
                         size_t scratch_bytes, int64_t B, int H, int W, void* stream_) {
    if (!p || !x || !out || !p->w1 || !p->w2 || !p->w3 || B <= 0 || H <= 0 || W <= 0)
        return VQAE_ERR_BAD_ARG;
    if (x == out) return VQAE_ERR_BAD_ARG;
    cudaStream_t stream = (cudaStream_t)stream_;
    const FixupScratch L = fixup_layout(p, B, H, W);
    if (!scratch || scratch_bytes < L.total) return VQAE_ERR_SCRATCH;
    char* base = reinterpret_cast<char*>(scratch);
    float* t1 = reinterpret_cast<float*>(base + L.t1);
    float* t2 = reinterpret_cast<float*>(base + L.t2);
    const int ci = p->c_in, co = p->c_out, cb = p->c_branch;
    const PreOp pre1{p->bias1a, p->bias1b, 1};
    const PreOp pre2{p->bias2a, p->bias2b, 1};
    const PreOp pre3{p->bias3a, p->bias3b, 1};
    const PreOp pre_skip{p->bias1c, 0.f, 0};
    int rc;

    // 'up' block in two kernels: the three low-resolution 1x1 convs (up_head.cu: t2 and the low-res
    // skip into t1), then both upsamples + branch_conv3 + residual sum (up_tail.cu); same arithmetic as
    // the six launches further down
    if (p->mode == VQAE_MODE_UP && p->w_skip && up_head_supported(B * H * W, ci, cb, co) &&
        up_tail_supported(B, H, W, cb, co)) {
        rc = up_head_f32(x, p->w1, p->w2, p->w_skip, t2, t1, B * H * W, ci, cb, co, p->bias1a,
                         p->bias1b, p->bias2a, p->bias2b, p->bias1c, stream);
        if (rc) return rc;
        return up_tail_f32(t2, t1, p->w3, out, B, H, W, cb, co, p->bias3a, p->bias3b, p->scale,
                           p->bias4, p->bias1d, stream);
    }

    // branch_conv1(act(x + bias1a) + bias1b)                      conv_block.py:199-200
    rc = conv_f32(CONV_1x1, x, p->w1, t1, nullptr, B, H, W, ci, cb, pre1, 1.f, 0.f, stream);
    if (rc) return rc;

    if (p->mode == VQAE_MODE_SAME) {
        if (ci != co || p->w_skip) return VQAE_ERR_UNSUPPORTED;
        // branch_conv2: 3x3 circular                              conv_block.py:202-203
        rc = conv_f32(CONV_3x3_CIRC, t1, p->w2, t2, nullptr, B, H, W, cb, cb, pre2, 1.f, 0.f,
                      stream);
        if (rc) return rc;
        // branch_conv3, * scale + bias4, + inp                    conv_block.py:205-214
        return conv_f32(CONV_1x1, t2, p->w3, out, x, B, H, W, cb, co, pre3, p->scale, p->bias4,
                        stream);
    }
    if (!p->w_skip) return VQAE_ERR_BAD_ARG;
    float* skip = reinterpret_cast<float*>(base + L.skip);

    if (p->mode == VQAE_MODE_DOWN) {
        if ((H | W) & 1) return VQAE_ERR_UNSUPPORTED;
        rc = conv_f32(CONV_2x2S2, t1, p->w2, t2, nullptr, B, H, W, cb, cb, pre2, 1.f, 0.f, stream);
        if (rc) return rc;
        // skip_conv(inp + bias1c) + bias1d                        conv_block.py:211-213
        rc = conv_f32(CONV_2x2S2, x, p->w_skip, skip, nullptr, B, H, W, ci, co, pre_skip, 1.f,
                      p->bias1d, stream);
        if (rc) return rc;
        return conv_f32(CONV_1x1, t2, p->w3, out, skip, B, H / 2, W / 2, cb, co, pre3, p->scale,
                        p->bias4, stream);
    }
    if (p->mode == VQAE_MODE_UP) {
        // ResizeConv2D = conv1x1(bicubic_up2(.)) (layers/conv.py:10-11).  Both maps are linear and
        // the conv has no bias, so the 1x1 runs at low resolution and the upsample follows.
        float* t3 = reinterpret_cast<float*>(base + L.t3);
        rc = conv_f32(CONV_1x1, t1, p->w2, t2, nullptr, B, H, W, cb, cb, pre2, 1.f, 0.f, stream);
        if (rc) return rc;
        // skip: conv1x1(inp + bias1c) at low res (into t1, now free)
        rc = conv_f32(CONV_1x1, x, p->w_skip, t1, nullptr, B, H, W, ci, co, pre_skip, 1.f, 0.f,
                      stream);
        if (rc) return rc;
        // both upsamples, the pre-activation, branch_conv3 and the residual sum in ONE kernel: the
        // upsampled tensors never reach HBM (same arithmetic as the three launches below); reached
        // when only the tail is built for the shape (c_branch = 64)
        if (up_tail_supported(B, H, W, cb, co))
            return up_tail_f32(t2, t1, p->w3, out, B, H, W, cb, co, p->bias3a, p->bias3b, p->scale,
                               p->bias4, p->bias1d, stream);
        rc = bicubic_up2_f32(t2, t3, B, H, W, cb, 0.f, stream);
        if (rc) return rc;
        rc = bicubic_up2_f32(t1, skip, B, H, W, co, p->bias1d, stream);
        if (rc) return rc;
        return conv_f32(CONV_1x1, t3, p->w3, out, skip, B, 2 * H, 2 * W, cb, co, pre3, p->scale,
                        p->bias4, stream);
    }
    return VQAE_ERR_BAD_ARG;
}

int vqae_pack_same_block_f16(const float* w1_oihw, const float* w2_oihw, const float* w3_oihw,
                              int c, void* packed, void* stream) {
    return pack_same_block_f16(w1_oihw, w2_oihw, w3_oihw, c, packed, (cudaStream_t)stream);
}

}  // extern "C"
namespace vqae {
int device_sm_count(int* out) {
    static PerDevice<int> sm_count_dev{};
    int& sm_count = sm_count_dev.cur();
    if (sm_count == 0) {
        int dev = 0;
        VQAE_CUDA_TRY(cudaGetDevice(&dev));
        VQAE_CUDA_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));
    }
    *out = sm_count;
    return VQAE_OK;
}
}  // namespace vqae
extern "C" {

int vqae_same_block_f16(const void* x, void* out, int io_dtype, const void* w_packed,
                         const float* scalars8_host, int64_t batch, int height, int width, int c,
                         void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return same_block_tc(x, out, io_dtype, w_packed, scalars8_host, batch, height, width, c, sm_count,
                         nullptr, (cudaStream_t)stream);
}

int vqae_same_block_mma_supported(int height, int width, int c) {
    return same_block_mma_supported(height, width, c) ? 1 : 0;
}

int vqae_same_block_mma_f16(const float* x, float* out, const void* w_packed,
                            const float* scalars8_host, int64_t batch, int height, int width, int c,
                            void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return same_block_mma(x, out, w_packed, scalars8_host, batch, height, width, c, sm_count,
                          (cudaStream_t)stream);
}

int vqae_down_block_mma_supported(int height, int width, int c_in) {
    return down_block_mma_supported(height, width, c_in) ? 1 : 0;
}

int vqae_down_block_mma_f16(const float* x, float* out, const void* w_packed,
                            const float* scalars8_host, int64_t batch, int height, int width,
                            int c_in, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return down_block_mma(x, out, w_packed, scalars8_host, batch, height, width, c_in, sm_count,
                          (cudaStream_t)stream);
}

int vqae_same_block_mma_split_supported(int height, int width, int c) {
    return same_block_mma_split_supported(height, width, c) ? 1 : 0;
}

int vqae_same_block_mma_split_f16(const float* x, float* out, const void* w_hi, const void* w_lo,
                                  const float* scalars8_host, const float* premul3_host,
                                  int64_t batch, int height, int width, int c, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return same_block_mma_split(x, out, w_hi, w_lo, scalars8_host, premul3_host, batch, height, width,
                                c, sm_count, (cudaStream_t)stream);
}

int vqae_same_block_split_supported(int height, int width, int c) {
    return same_block_split_supported(height, width, c) ? 1 : 0;
}

int vqae_same_block_split_f16(const float* x, float* out, const void* w_hi, const void* w_lo,
                              const float* scalars8_host, const float* premul3_host, int64_t batch,
                              int height, int width, int c, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return same_block_split(x, out, w_hi, w_lo, scalars8_host, premul3_host, batch, height, width, c,
                            sm_count, (cudaStream_t)stream);
}

int vqae_down_block_split_f16(const float* x, float* out, const void* w_hi, const void* w_lo,
                              const float* scalars8_host, const float* premul3_host, int64_t batch,
                              int height, int width, int c_in, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return down_block_split(x, out, w_hi, w_lo, scalars8_host, premul3_host, batch, height, width,
                            c_in, sm_count, (cudaStream_t)stream);
}

int vqae_stem_in_mma_supported(int height, int width, int c_out) {
    return stem_in_mma_supported(height, width, c_out) ? 1 : 0;
}

int vqae_stem_in_mma_f32(const void* x, int x_dtype, int x_layout, const float* w_oihw,
                         const float* bias, float* out, int64_t batch, int height, int width,
                         int c_out, const float* mean_host, const float* std_host, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return stem_in_mma(x, x_dtype, x_layout, w_oihw, bias, out, batch, height, width, c_out,
                       mean_host, std_host, sm_count, (cudaStream_t)stream);
}

int vqae_stem_out_mma_supported(int height, int width, int c_in) {
    return stem_out_mma_supported(height, width, c_in) ? 1 : 0;
}

int vqae_stem_out_mma_f32(const float* x, const float* w_oihw, const float* bias, float* out,
                          int out_layout, int64_t batch, int height, int width, int c_in,
                          void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return stem_out_mma(x, w_oihw, bias, out, out_layout, batch, height, width, c_in, sm_count,
                        (cudaStream_t)stream);
}

int vqae_stem_out_u8_supported(int height, int width, int c_in, int kernel) {
    if (kernel == VQAE_STEM_OUT_TENSOR_CORE) return stem_out_mma_supported(height, width, c_in) ? 1 : 0;
    return kernel == VQAE_STEM_OUT_EXACT && height > 0 && width > 0 && c_in == 8 ? 1 : 0;
}

int vqae_stem_out_u8(const float* x, const float* w_oihw, const float* bias, const float* mean_host,
                     const float* std_host, uint8_t* canvas, int64_t canvas_rows, int64_t canvas_cols,
                     int64_t first_patch, int grid_cols, int64_t batch, int height, int width, int c_in,
                     int kernel, void* stream) {
    if (!x || !w_oihw || !bias) return VQAE_ERR_BAD_ARG;
    U8Canvas cv{};
    if (int rc = make_u8_canvas(canvas, canvas_rows, canvas_cols, first_patch, grid_cols, batch, height,
                                width, mean_host, std_host, &cv))
        return rc;
    if (kernel == VQAE_STEM_OUT_EXACT)
        return stem_out_u8(x, w_oihw, bias, cv, batch, height, width, c_in, (cudaStream_t)stream);
    if (kernel != VQAE_STEM_OUT_TENSOR_CORE) return VQAE_ERR_BAD_ARG;
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return stem_out_mma_u8(x, w_oihw, bias, cv, batch, height, width, c_in, sm_count,
                           (cudaStream_t)stream);
}

int vqae_front_fused_supported(int height, int width) {
    return front_fused_supported(height, width) ? 1 : 0;
}

int vqae_front_fused_f16(const void* x, int x_dtype, int x_layout, const float* stem_w,
                         const float* stem_bias, const float* mean_host, const float* std_host,
                         const void* same_w_packed, const float* same_scalars8_host,
                         const void* down_w_packed, const float* down_scalars8_host, float* out,
                         int64_t batch, int height, int width, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return front_fused(x, x_dtype, x_layout, stem_w, stem_bias, mean_host, std_host, same_w_packed,
                       same_scalars8_host, down_w_packed, down_scalars8_host, out, batch, height,
                       width, sm_count, (cudaStream_t)stream);
}

int vqae_up_block_mma_supported(int height, int width, int c_in) {
    return up_block_mma_supported(height, width, c_in) ? 1 : 0;
}

size_t vqae_up_block_mma_scratch_bytes(int64_t batch, int height, int width, int c_in) {
    return up_block_mma_scratch_bytes(batch, height, width, c_in);
}

int vqae_up_block_mma_f16(const float* x, float* out, const void* w_packed,
                          const float* scalars8_host, void* scratch, size_t scratch_bytes,
                          int64_t batch, int height, int width, int c_in, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return up_block_mma(x, out, w_packed, scalars8_host, scratch, scratch_bytes, batch, height, width,
                        c_in, sm_count, (cudaStream_t)stream);
}

size_t vqae_same_chain_flag_bytes(int n_blocks, int64_t batch) {
    return same_chain_flag_bytes(n_blocks, batch);
}

int vqae_same_chain_supported(int64_t batch, int height, int width, int c) {
    int sm_count = 0;
    if (device_sm_count(&sm_count)) return 0;
    return same_chain_supported(batch, height, width, c, sm_count) ? 1 : 0;
}

int vqae_same_chain_f16(const float* x, float* buf_a, float* buf_b, const void* w_packed_all,
                         const float* scalars_dev, void* flags, size_t flag_bytes, int n_blocks,
                         int64_t batch, int height, int width, int c, void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return same_chain_tc(x, buf_a, buf_b, w_packed_all, scalars_dev, flags, flag_bytes, n_blocks,
                         batch, height, width, c, sm_count, (cudaStream_t)stream);
}

int vqae_trunk_resident_max_clusters(void) {
    int n = 0;
    return trunk_resident_max_clusters(&n) == VQAE_OK ? n : -1;
}

int vqae_trunk_resident_supported(int64_t batch, int height, int width, int c) {
    return trunk_resident_supported(batch, height, width, c) ? 1 : 0;
}

int vqae_pack_resident_block_f16(const float* w1_oihw, const float* w2_oihw, const float* w3_oihw,
                                  int c, float scale, void* packed, void* stream) {
    return pack_resident_block_f16(w1_oihw, w2_oihw, w3_oihw, c, scale, packed,
                                    (cudaStream_t)stream);
}

int vqae_trunk_resident_f16(const void* x, void* out, int io_dtype, const void* w_packed_all,
                             const float* scalars_dev, int n_blocks, int64_t batch, int height,
                             int width, int c, void* stream) {
    return trunk_resident_tc(x, out, io_dtype, w_packed_all, scalars_dev, n_blocks, batch, height, width, c,
                             (cudaStream_t)stream);
}

size_t vqae_down_block_pack_elems(int c_in) { return down_block_pack_elems(c_in); }

int vqae_pack_down_block_f16(const float* w1_oihw, const float* w2_oihw, const float* w3_oihw,
                              const float* wskip_oihw, int c_in, float scale, void* packed,
                              void* stream) {
    return pack_down_block_f16(w1_oihw, w2_oihw, w3_oihw, wskip_oihw, c_in, scale, packed,
                                (cudaStream_t)stream);
}

int vqae_down_block_f16(const void* x, void* out, int io_dtype, const void* w_packed,
                         const float* scalars8_host, int64_t batch, int height, int width, int c_in,
                         void* stream) {
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    if (c_in == 64) {                  // the wide block of the 512-model: streamed weights (tc_down128.cu)
        if (io_dtype != VQAE_DT_F32) return VQAE_ERR_UNSUPPORTED;
        return down128_tc(reinterpret_cast<const float*>(x), reinterpret_cast<float*>(out), w_packed,
                          scalars8_host, batch, height, width, c_in, sm_count, (cudaStream_t)stream);
    }
    return down_block_tc(x, out, io_dtype, w_packed, scalars8_host, batch, height, width, c_in, sm_count,
                         (cudaStream_t)stream);
}

int vqae_quantizer_prepare_f32(const float* embed, int num_codes, int dim, const float* w_out,
                               const float* b_out, int c, float* table, void* stream) {
    return quantizer_prepare_f32(embed, num_codes, dim, w_out, b_out, c, table,
                                 (cudaStream_t)stream);
}

size_t vqae_quantizer_scratch_bytes(int64_t n_vectors) {
    return quantizer_scratch_bytes(n_vectors);
}

int vqae_quantize_f32(const vqae_quantizer_params* p, const float* x, int x_layout, float* out,
                      int out_layout, int64_t* indices, float* loss, uint32_t* near_ties,
                      float tie_rel_gap, float* z_out, void* scratch, size_t scratch_bytes,
                      int64_t batch, int64_t spatial, void* stream) {
    return quantize_f32(p, x, x_layout, out, out_layout, indices, loss, near_ties, tie_rel_gap,
                        z_out, scratch, scratch_bytes, batch, spatial, (cudaStream_t)stream);
}

int vqae_quantize_supported(const vqae_quantizer_params* p, int x_dtype, int x_layout,
                            int out_dtype, int out_layout, int has_out, int kernel) {
    return quantize_supported(p, x_dtype, x_layout, out_dtype, out_layout, has_out != 0, kernel) ? 1 : 0;
}

int vqae_quantize(const vqae_quantizer_params* p, const void* x, int x_dtype, int x_layout,
                  void* out, int out_dtype, int out_layout, int64_t* indices, float* loss,
                  uint32_t* near_ties, float tie_rel_gap, float* z_out, void* scratch,
                  size_t scratch_bytes, int64_t batch, int64_t spatial, int kernel, void* stream) {
    return quantize_any(p, x, x_dtype, x_layout, out, out_dtype, out_layout, indices, loss,
                        near_ties, tie_rel_gap, z_out, scratch, scratch_bytes, batch, spatial,
                        kernel, (cudaStream_t)stream);
}

int vqae_quantize_tc_supported(const vqae_quantizer_params* p, int x_layout, int out_layout,
                               int has_out) {
    return p && quantize_tc_supported(p, x_layout, out_layout, has_out != 0) ? 1 : 0;
}

int vqae_quantize_tc_f32(const vqae_quantizer_params* p, const float* x, float* out,
                         int64_t* indices, float* loss, uint32_t* near_ties, float tie_rel_gap,
                         float* z_out, float* diag, void* scratch, size_t scratch_bytes,
                         int64_t batch, int64_t spatial, void* stream_) {
    if (!p || !x || !indices || !loss || !p->embed || batch <= 0 || spatial <= 0)
        return VQAE_ERR_BAD_ARG;
    if (out && !p->table) return VQAE_ERR_BAD_ARG;
    if (!quantize_tc_supported(p, VQAE_LAYOUT_NHWC, VQAE_LAYOUT_NHWC, out != nullptr))
        return VQAE_ERR_UNSUPPORTED;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t N = batch * spatial;
    if (!scratch || scratch_bytes < quantizer_scratch_bytes(N)) return VQAE_ERR_SCRATCH;
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    return quantize_tc_f32(p, x, out, indices, loss, scratch, near_ties, tie_rel_gap, z_out, diag, N,
                           sm_count, stream);
}

int vqae_embed_codes_f32(const void* indices, int idx_is_u8, const float* table, int num_codes,
                         int c, float* out, int out_layout, int64_t batch, int64_t spatial,
                         void* stream) {
    return embed_codes_f32(indices, idx_is_u8, table, num_codes, c, out, out_layout, batch,
                           spatial, (cudaStream_t)stream);
}

int vqae_embed_codemap_f32(const void* code_map, int map_is_u8, int64_t map_rows, int64_t map_cols,
                           int th, int tw, int64_t r0, int64_t c0, int64_t region_cols,
                           int64_t first_patch, int64_t n, const float* table, int num_codes, int c,
                           float* out, void* stream) {
    return embed_codemap_f32(code_map, map_is_u8, map_rows, map_cols, th, tw, r0, c0, region_cols,
                             first_patch, n, table, num_codes, c, out, (cudaStream_t)stream);
}

int vqae_codemap_place_u8(const int64_t* tiles, int64_t n_tiles, int th, int tw,
                          int64_t first_patch, int grid_cols, uint8_t* map, int64_t map_rows,
                          int64_t map_cols, void* stream) {
    return codemap_place_u8(tiles, n_tiles, th, tw, first_patch, grid_cols, map, map_rows,
                            map_cols, (cudaStream_t)stream);
}

int vqae_codemap_place_i64(const int64_t* tiles, int64_t n_tiles, int th, int tw,
                           int64_t first_patch, int grid_cols, int64_t* map, int64_t map_rows,
                           int64_t map_cols, void* stream) {
    return codemap_place_i64(tiles, n_tiles, th, tw, first_patch, grid_cols, map, map_rows,
                             map_cols, (cudaStream_t)stream);
}

size_t vqae_quality_u8_scratch_bytes(int64_t batch, int height, int width) {
    return quality_u8_scratch_bytes(batch, height, width);
}

int vqae_quality_u8(const uint8_t* ref, int64_t ref_rows, int64_t ref_cols, int64_t ref_r0, int64_t ref_c0,
                    int64_t ref_region_cols, int64_t ref_first, const uint8_t* rec, int64_t rec_rows,
                    int64_t rec_cols, int64_t rec_r0, int64_t rec_c0, int64_t rec_region_cols,
                    int64_t rec_first, int64_t batch, int height, int width, int64_t* sse, double* ssim,
                    void* scratch, size_t scratch_bytes, void* stream) {
    return quality_u8(ref, ref_rows, ref_cols, ref_r0, ref_c0, ref_region_cols, ref_first, rec, rec_rows,
                      rec_cols, rec_r0, rec_c0, rec_region_cols, rec_first, batch, height, width, sse, ssim,
                      scratch, scratch_bytes, (cudaStream_t)stream);
}

int vqae_codemap_histogram(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int64_t r0,
                           int64_t c0, int64_t nr, int64_t nc, int num_codes, int64_t* counts, void* stream) {
    return codemap_histogram(map, map_is_u8, map_rows, map_cols, r0, c0, nr, nc, num_codes, counts,
                             (cudaStream_t)stream);
}

size_t vqae_codemap_pack_scratch_bytes(int64_t n_patches, int th, int tw) {
    return codemap_pack_scratch_bytes(n_patches, th, tw);
}

int64_t vqae_codemap_pack_worst_bytes(int64_t n_patches, int th, int tw) {
    return codemap_pack_worst_bytes(n_patches, th, tw);
}

int vqae_codemap_pack(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int th, int tw,
                      const uint32_t* freq_host, int num_codes, int scale_bits, int64_t* offsets,
                      uint8_t* payload, int64_t payload_capacity, void* scratch, size_t scratch_bytes,
                      void* stream) {
    return codemap_pack(map, map_is_u8, map_rows, map_cols, th, tw, freq_host, num_codes, scale_bits, offsets,
                        payload, payload_capacity, scratch, scratch_bytes, (cudaStream_t)stream);
}

int vqae_codemap_unpack(const uint8_t* payload, int64_t payload_bytes, const int64_t* offsets_host,
                        const int64_t* offsets, int64_t map_rows, int64_t map_cols, int th, int tw,
                        const uint32_t* freq_host, int num_codes, int scale_bits, int64_t r0, int64_t c0,
                        int64_t nr, int64_t nc, void* out, int out_is_u8, uint8_t* flags, void* stream) {
    return codemap_unpack(payload, payload_bytes, offsets_host, offsets, map_rows, map_cols, th, tw, freq_host,
                          num_codes, scale_bits, r0, c0, nr, nc, out, out_is_u8, flags, (cudaStream_t)stream);
}

}  // extern "C"

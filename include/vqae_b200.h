/* vqae_b200.h -- C-ABI of the B200-native (sm_100a) inference hot path of 2D-VQ-AE-2.
 *
 * The reference (sara-nl/2D-VQ-AE-2) has no FFI of its own: every FLOP of its hot path is a
 * PyTorch/cuDNN library call made from vq_ae/model.py and vq_ae/layers/*.py.  This header is
 * therefore the boundary a maintainer would bind (ctypes, see INTEGRATION.md) to replace those
 * library calls.  Each entry point cites the reference call site(s) it replaces; paths are
 * relative to the reference checkout.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - activations inside the path are NHWC ("channels last"), fp32 or bf16;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every call returns 0 on success or a VQAE_ERR_* code; nothing is thrown, nothing is
 *     synchronised; kernels are only enqueued on `stream`;
 *   - there is no CPU fallback anywhere behind this ABI.
 */
#ifndef VQAE_B200_H_
#define VQAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQAE_ABI_VERSION 4

enum {
    VQAE_OK = 0,
    VQAE_ERR_BAD_ARG = 1,        /* null pointer / non-positive extent                          */
    VQAE_ERR_UNSUPPORTED = 2,    /* shape outside what the kernels are built for                */
    VQAE_ERR_DIM_MISMATCH = 3,   /* mirrors NotImplementedError of layers/vq.py:100-104         */
    VQAE_ERR_CUDA = 4,           /* a CUDA runtime call / launch failed (see vqae_last_cuda_error) */
    VQAE_ERR_SCRATCH = 5         /* scratch buffer too small                                    */
};

/* layouts of tensors crossing the boundary */
enum { VQAE_LAYOUT_NCHW = 0, VQAE_LAYOUT_NHWC = 1 };
/* element types crossing the boundary */
enum { VQAE_DT_F32 = 0, VQAE_DT_BF16 = 1, VQAE_DT_U8 = 2, VQAE_DT_F16 = 3 };
/* PreActFixupResBlock modes (layers/conv_block.py:147) */
enum { VQAE_MODE_SAME = 0, VQAE_MODE_DOWN = 1, VQAE_MODE_UP = 2 };

int vqae_abi_version(void);
const char* vqae_error_string(int code);
/* cudaGetErrorString of the last CUDA error seen by this library on the calling thread */
const char* vqae_last_cuda_error(void);
/* number of kernels this library has launched since load (for bench.py's gpu_launches) */
uint64_t vqae_launch_count(void);

/* ---- a-N  input normalisation ------------------------------------------------------------
 * Replaces albumentations Normalize + ToTensorV2 (conf/transforms/camelyon16_transforms.yaml:1-23,
 * conf/transforms/normalize.yaml:1-11):  out = (u8 - 255*mean_c) * (1 / (255*std_c)).
 * img: [B,H,W,3] u8;  out: fp32 [B,3,H,W] (NCHW) or [B,H,W,3] (NHWC).  mean/std: host float[3]. */
int vqae_normalize_u8(const uint8_t* img, float* out, int64_t batch, int height, int width,
                      const float* mean_host, const float* std_host, int out_layout, void* stream);

/* ---- weight packing (once after load_state_dict()/eval()) ---------------------------------
 * OIHW fp32 conv weight -> [KH*KW][I][O] fp32 ("tap-major, output-channel fastest").        */
int vqae_pack_conv_weight_f32(const float* w_oihw, float* packed, int out_ch, int in_ch, int kh,
                              int kw, void* stream);

/* Batched form: every weight layout of this library, any number of matrices / blocks, ONE launch.
 * A descriptor names the OIHW fp32 sources of one conv (F32_CONV: src[0]) or of one
 * PreActFixupResBlock (SAME / RESIDENT: src = {branch_conv1, branch_conv2, branch_conv3};
 * DOWN: + skip_conv) and the destination; c_in / c_out are the block's channel counts (F32_CONV:
 * the conv's, with `taps` = kh*kw); `scale` is the Fixup scale folded into branch_conv3 by the
 * RESIDENT and DOWN layouts.  kind | VQAE_PACK_LO writes f16(w - f16(w)), the low half of the
 * split operands of precision "fp32tc" (vqae_same_block_split_f16, vqae_down_block_split_f16), where
 * premul[] scales the matrices first.  n_elems = vqae_pack_elems(kind, c_in, c_out, taps).
 * descs_device: the table in DEVICE memory; max_elems: the largest n_elems in it.             */
enum { VQAE_PACK_F32_CONV = 0, VQAE_PACK_SAME_F16 = 1, VQAE_PACK_RESIDENT_F16 = 2,
       VQAE_PACK_DOWN_F16 = 3, VQAE_PACK_SAME_MMA_F16 = 4, VQAE_PACK_DOWN_MMA_F16 = 5,
       VQAE_PACK_UP_MMA_F16 = 6, VQAE_PACK_LO = 0x100 };
typedef struct vqae_pack_desc {
    int32_t kind, c_in, c_out, taps;
    float scale;
    int32_t n_elems;
    const void* src[4];
    void* dst;
    float premul[4];   /* powers of two applied to branch_conv1, 2, 3, skip before rounding (0 = 1):
                          the split-operand packs of the fp32-accurate tensor-core mode */
} vqae_pack_desc;
size_t vqae_pack_elems(int kind, int c_in, int c_out, int taps);
int vqae_pack_batched(const vqae_pack_desc* descs_device, int n_descs, int max_elems, void* stream);

/* ---- a-S  stems --------------------------------------------------------------------------
 * in_stem  (vq_ae/model.py:141,198; conv_layer/same2d.yaml: 3x3, zero pad, bias) 3 -> c_out.
 * x is one of: fp32 NCHW [B,3,H,W], fp32 NHWC [B,H,W,3], u8 NHWC [B,H,W,3] (normalised on the
 * fly with mean/std as in vqae_normalize_u8; mean/std may be NULL otherwise).
 * w: OIHW [c_out,3,3,3] fp32, bias [c_out];  out: NHWC fp32 [B,H,W,c_out], c_out == 8.      */
int vqae_stem_in_f32(const void* x, int x_dtype, int x_layout, const float* w_oihw,
                     const float* bias, float* out, int64_t batch, int height, int width,
                     int c_out, const float* mean_host, const float* std_host, void* stream);
/* the same with the output element type chosen: VQAE_DT_F32, or VQAE_DT_F16 -- the activation
 * stream of the reduced-precision path (needs width % 128 == 0, height % 8 == 0)              */
int vqae_stem_in(const void* x, int x_dtype, int x_layout, const float* w_oihw, const float* bias,
                 void* out, int out_dtype, int64_t batch, int height, int width, int c_out,
                 const float* mean_host, const float* std_host, void* stream);
/* out_stem (vq_ae/model.py:291): 3x3, zero pad, bias, c_in(8) -> 3.
 * x NHWC fp32 [B,H,W,c_in];  out fp32 NCHW [B,3,H,W] or NHWC [B,H,W,3].                     */
int vqae_stem_out_f32(const float* x, const float* w_oihw, const float* bias, float* out,
                      int out_layout, int64_t batch, int height, int width, int c_in,
                      void* stream);

/* ---- building blocks of a-R, exported for per-piece parity tests and ResizeConv2D ----------
 * One branch/skip conv of PreActFixupResBlock with its Fixup pre-activation and epilogue fused:
 *   out = conv_kind( act?(x + pre_add) + post_add ) * scale + bias (+ residual)
 * kind: 0 = 1x1 (proj2d.yaml), 1 = 2x2 stride 2 (down2d.yaml), 2 = 3x3 circular pad 1
 * (same2d.yaml with padding_mode circular, pre_activation_fixup.yaml:40,60).
 * x NHWC fp32 [B,H,W,c_in]; w packed [taps][c_in][c_out]; out/residual NHWC [B,H',W',c_out];
 * c_in, c_out multiples of 8 (c_out in {8,16,32} or a multiple of 64).                       */
int vqae_conv_f32(int kind, const float* x, const float* w_packed, float* out,
                  const float* residual, int64_t batch, int height, int width, int c_in,
                  int c_out, float pre_add, int pre_elu, float post_add, float scale, float bias,
                  void* stream);
/* nn.Upsample(mode='bicubic', scale_factor=2, align_corners=False) (layers/conv.py:8) + bias:
 * x NHWC fp32 [B,H,W,c] -> out NHWC [B,2H,2W,c], c multiple of 4.                            */
int vqae_bicubic_up2_f32(const float* x, float* out, int64_t batch, int height, int width, int c,
                         float bias, void* stream);

/* ---- a-R  PreActFixupResBlock.forward (layers/conv_block.py:196-216) ------------------------
 * Weights are the packed form of vqae_pack_conv_weight_f32.  Scalars are the (1,)-shaped
 * parameters bias1a..bias4, scale, bias1c, bias1d read to the host once at pack time.       */
typedef struct vqae_fixup_params {
    int mode;        /* VQAE_MODE_*                                                          */
    int c_in, c_out, c_branch;
    const float* w1;     /* branch_conv1: [1][c_in][c_branch]                                */
    const float* w2;     /* branch_conv2: same [9][cb][cb] (3x3 circular), down [4][cb][cb]
                            (2x2 stride 2), up [1][cb][cb] (1x1 after bicubic x2)            */
    const float* w3;     /* branch_conv3: [1][c_branch][c_out]                               */
    const float* w_skip; /* skip_conv: down [4][c_in][c_out], up [1][c_in][c_out], else NULL */
    float bias1a, bias1b, bias2a, bias2b, bias3a, bias3b, bias4, scale, bias1c, bias1d;
} vqae_fixup_params;

/* bytes of scratch one block call needs for an input of [batch, height, width, c_in] */
size_t vqae_fixup_block_scratch_bytes(const vqae_fixup_params* p, int64_t batch, int height,
                                      int width);
/* x: NHWC fp32 [B,H,W,c_in];  out: NHWC fp32 [B,H',W',c_out] (H' = H, H/2 or 2H by mode);
 * x and out must not alias.                                                                 */
int vqae_fixup_block_f32(const vqae_fixup_params* p, const float* x, float* out, void* scratch,
                         size_t scratch_bytes, int64_t batch, int height, int width,
                         void* stream);

/* ---- a-T / a-R on tensor cores (tcgen05, fp16 operands, fp32 accumulate + fp32 residual) -------
 * Activation stream: every kernel below reads x and writes out as NHWC tensors of element type
 * io_dtype = VQAE_DT_F32 or VQAE_DT_F16 (both the same).  The arithmetic between load and store
 * is identical (operands rounded to fp16 for the GEMMs, fp32 accumulation, fp32 residual add);
 * the fp16 stream halves the HBM bytes of the block-boundary tensors and is what the
 * reduced-precision plan uses (the reference's own autocast run stores fp16 between ops too).
 * One PreActFixupResBlock in mode 'same' (layers/conv_block.py:196-216) per call, all three
 * convs and their pre-activations fused in one kernel; c in {8, 16, 32, 64} (8 runs zero-padded
 * as 16), height % 16 == 0, width % 32 == 0 -- every 'same' block of the shipped encoder and
 * decoder (DownBlock/UpBlock pre/post layers and the 50-block trunks, model.py:150-153,240-263).
 * w_packed comes from vqae_pack_same_block_f16 (11 * cp * cp bf16, cp = max(c, 16));
 * scalars8_host = {bias1a, bias1b, bias2a, bias2b, bias3a, bias3b, bias4, scale} on the HOST.
 * x, out: NHWC fp32 [B,H,W,c], must not alias.                                               */
int vqae_pack_same_block_f16(const float* w1_oihw, const float* w2_oihw, const float* w3_oihw,
                              int c, void* packed, void* stream);
int vqae_same_block_f16(const void* x, void* out, int io_dtype, const void* w_packed,
                        const float* scalars8_host, int64_t batch, int height, int width, int c,
                        void* stream);
/* The same block at LOW channel counts (c in {8, 16, 32}: the full-resolution pyramid levels) on
 * warp-level tensor-core MMAs with the three GEMMs chained through registers (csrc/mma_same.cu):
 * for N = c <= 32 the activation arithmetic and the memory stream are the cost, not the GEMMs, and
 * many independent warps beat one 512-pixel tile per CTA behind tensor-memory round trips.
 * w_packed: 11 * c * c fp16 from vqae_pack_batched(VQAE_PACK_SAME_MMA_F16); scalars8_host as for
 * vqae_same_block_f16; x, out: NHWC fp32, must not alias; height % 16 == 0, width % 32 == 0.   */
int vqae_same_block_mma_supported(int height, int width, int c);
int vqae_same_block_mma_f16(const float* x, float* out, const void* w_packed,
                            const float* scalars8_host, int64_t batch, int height, int width, int c,
                            void* stream);
/* 'down' block (c_in in {8, 16, 32} -> 2 c_in) on warp-level MMAs, every intermediate in registers
 * (csrc/mma_down.cu; a 2x2 stride-2 conv has no halo).  w_packed: vqae_pack_batched(
 * VQAE_PACK_DOWN_MMA_F16); scalars8_host as for vqae_down_block_f16; x: NHWC fp32 [B,H,W,c_in],
 * out: NHWC fp32 [B,H/2,W/2,2 c_in]; height % 2 == 0, width % 32 == 0.                        */
int vqae_down_block_mma_supported(int height, int width, int c_in);
int vqae_down_block_mma_f16(const float* x, float* out, const void* w_packed,
                            const float* scalars8_host, int64_t batch, int height, int width,
                            int c_in, void* stream);
/* in_stem on warp-level tensor-core MMAs with split fp16 operands (csrc/mma_stem.cu): fp32-accurate
 * (not bit-identical to vqae_stem_in_f32), nine MMAs per 16 pixels; c_out == 8, height % 16 == 0,
 * width % 32 == 0.  Same arguments as vqae_stem_in_f32.                                        */
int vqae_stem_in_mma_supported(int height, int width, int c_out);
int vqae_stem_in_mma_f32(const void* x, int x_dtype, int x_layout, const float* w_oihw,
                         const float* bias, float* out, int64_t batch, int height, int width,
                         int c_out, const float* mean_host, const float* std_host, void* stream);
/* out_stem on warp-level tensor-core MMAs with split fp16 operands (csrc/mma_stem.cu): fp32-accurate
 * (not bit-identical to vqae_stem_out_f32), every input pixel read once; c_in == 8,
 * height % 16 == 0, width % 32 == 0.  Same arguments as vqae_stem_out_f32.                     */
int vqae_stem_out_mma_supported(int height, int width, int c_in);
int vqae_stem_out_mma_f32(const float* x, const float* w_oihw, const float* bias, float* out,
                          int out_layout, int64_t batch, int height, int width, int c_in,
                          void* stream);
/* out_stem with the uint8 output of a decoded slide: the exact inverse of vqae_normalize_u8,
 *     u8 = min(max(rint(fma(v, 255 std_c, 255 mean_c)), 0), 255)     (round half to even; NaN -> 0)
 * with v the fp32 value the fp32 form of the same kernel stores and the two products formed in fp32
 * on the host.  Image b of the batch is written as patch q = first_patch + b of a canvas uint8
 * [canvas_rows, canvas_cols, 3] (NHWC RGB, the layout vqae_stem_in reads) holding a grid of
 * height x width patches, grid_cols per row: at canvas pixel ((q / grid_cols) height,
 * (q % grid_cols) width) -- the addressing of vqae_codemap_place_u8.  grid_cols = 1 and
 * first_patch = 0 on a [batch * height, width, 3] canvas is the plain [B,H,W,3] batch.
 * kernel: VQAE_STEM_OUT_EXACT (the CUDA-core kernel of vqae_stem_out_f32, bit-identical values before
 * the conversion) or VQAE_STEM_OUT_TENSOR_CORE (that of vqae_stem_out_mma_f32; height % 16 == 0,
 * width % 32 == 0).  Rows leave as 16-byte stores when width % 32 == 0, canvas_cols % 16 == 0 and
 * the canvas is 16-byte aligned.  x NHWC fp32 [B,H,W,c_in], c_in == 8; mean/std: host float[3].
 * VQAE_ERR_BAD_ARG for a null pointer, a non-positive extent or a placement outside the canvas,
 * checked before anything is launched; VQAE_ERR_UNSUPPORTED when first_patch + batch > 2^31.       */
enum { VQAE_STEM_OUT_EXACT = 0, VQAE_STEM_OUT_TENSOR_CORE = 1 };
int vqae_stem_out_u8_supported(int height, int width, int c_in, int kernel);
int vqae_stem_out_u8(const float* x, const float* w_oihw, const float* bias, const float* mean_host,
                     const float* std_host, uint8_t* canvas, int64_t canvas_rows, int64_t canvas_cols,
                     int64_t first_patch, int grid_cols, int64_t batch, int height, int width, int c_in,
                     int kernel, void* stream);
/* The encoder's FRONT END in one launch (csrc/mma_front.cu): in_stem (with the u8 normalisation of
 * vqae_stem_in) + the C = 8 'same' block + the 'down' block 8 -> 16 of the first DownBlock
 * (model.py:141,144-148,198-199) -- the input image is read once, the 16-channel half-resolution
 * tensor written once, the two 8-channel full-resolution tensors in between never reach memory.
 * Arithmetic of the "fp16" path: vqae_stem_in (fp32-accurate; split-operand tensor-core MMAs) ->
 * vqae_same_block_mma_f16 -> vqae_down_block_mma_f16, same packed weights and host scalars as those
 * calls.  x as for vqae_stem_in; out: NHWC fp32 [B,H/2,W/2,16]; height % 16 == 0, width % 32 == 0. */
int vqae_front_fused_supported(int height, int width);
int vqae_front_fused_f16(const void* x, int x_dtype, int x_layout, const float* stem_w_oihw,
                         const float* stem_bias, const float* mean_host, const float* std_host,
                         const void* same_w_packed, const float* same_scalars8_host,
                         const void* down_w_packed, const float* down_scalars8_host, float* out,
                         int64_t batch, int height, int width, void* stream);
/* fp32-ACCURATE tensor-core forms (precision "fp32tc"): every GEMM operand is a pair hi + lo of fp16
 * numbers (22 significand bits), every product three tensor-core products hi.hi + lo.hi + hi.lo with
 * fp32 accumulation, the activation is the fp32 path's expm1f -- the reference's fp32 index contract
 * (vq.py:121-129) holds outside reported near-ties at tensor-core speed.
 * 'same' block (csrc/tc_split.cu, tcgen05, 8 x 32 pixel tiles): c in {8, 16, 32, 64}, height % 8 == 0,
 * width % 32 == 0.  w_hi / w_lo: vqae_pack_batched(VQAE_PACK_SAME_F16 [| VQAE_PACK_LO]) with
 * premul = premul3_host (powers of two for branch_conv1, 2, 3: 2^(14 - ceil(log2 max|w|)) keeps every
 * low half a normal fp16 number); scalars8_host as for vqae_same_block_f16.  fp32 NHWC in and out.
 * 'down' block (csrc/mma_down.cu, SPLIT instantiation, register-resident): c_in in {8, 16, 32};
 * w_hi / w_lo: VQAE_PACK_DOWN_MMA_F16 [| VQAE_PACK_LO] with premul = {p1, p2, p3, p3} (branch_conv3
 * and skip_conv share an accumulator, hence a factor); scalars8_host as for vqae_down_block_f16. */
 /* the same contract at c in {8, 16} on register-chained warp-level MMAs (csrc/mma_same_split.cu;
 * w_hi / w_lo: VQAE_PACK_SAME_MMA_F16 [| VQAE_PACK_LO] with premul) */
int vqae_same_block_mma_split_supported(int height, int width, int c);
int vqae_same_block_mma_split_f16(const float* x, float* out, const void* w_hi, const void* w_lo,
                                  const float* scalars8_host, const float* premul3_host,
                                  int64_t batch, int height, int width, int c, void* stream);
int vqae_same_block_split_supported(int height, int width, int c);
int vqae_same_block_split_f16(const float* x, float* out, const void* w_hi, const void* w_lo,
                              const float* scalars8_host, const float* premul3_host, int64_t batch,
                              int height, int width, int c, void* stream);
int vqae_down_block_split_f16(const float* x, float* out, const void* w_hi, const void* w_lo,
                              const float* scalars8_host, const float* premul3_host, int64_t batch,
                              int height, int width, int c_in, void* stream);
/* 'up' block (c_in in {16, 32, 64, 128} -> c_in / 2, x2 bicubic; conv_block.py:196-216 with ResizeConv2D,
 * conv.py:4-11) on warp-level MMAs in two kernels (csrc/mma_up.cu): the three 1x1 convs that
 * commute with the upsample at LOW resolution (register-resident), then bicubic interpolation
 * (index-clamped, separable) + branch_conv3 + skip sum at high resolution.  w_packed:
 * vqae_pack_batched(VQAE_PACK_UP_MMA_F16, c_in, c_in / 2); scalars8_host = {bias1a, bias1b, bias2a,
 * bias2b, bias3a, bias3b, bias1c, bias4 + bias1d}; x: NHWC fp32 [B,H,W,c_in], out: NHWC fp32
 * [B,2H,2W,c_in/2]; height % 4 == 0, width % 16 == 0; scratch >= vqae_up_block_mma_scratch_bytes. */
int vqae_up_block_mma_supported(int height, int width, int c_in);
size_t vqae_up_block_mma_scratch_bytes(int64_t batch, int height, int width, int c_in);
int vqae_up_block_mma_f16(const float* x, float* out, const void* w_packed,
                          const float* scalars8_host, void* scratch, size_t scratch_bytes,
                          int64_t batch, int height, int width, int c_in, void* stream);
/* A run of n_blocks consecutive 'same' blocks of equal width in ONE persistent launch (the 50-block
 * trunks model.py:150-153,240-263 and the post layers of DownBlock/UpBlock): every (block, tile)
 * task is scheduled round-robin over the resident CTAs and ordered by per-(block, image) completion
 * counters, so no SM idles at block boundaries.  Results are bit-identical to n_blocks calls of
 * vqae_same_block_f16.  w_packed_all: the blocks' vqae_pack_same_block_f16 outputs back to back;
 * scalars_dev: DEVICE float [n_blocks][8] in the order of scalars8_host above; block i reads
 * (i ? buf[(i-1)&1] : x) and writes buf[i&1] with buf = {buf_a, buf_b}: the result is in
 * buf[(n_blocks-1)&1]; flags: DEVICE scratch of vqae_same_chain_flag_bytes(n_blocks, batch).    */
size_t vqae_same_chain_flag_bytes(int n_blocks, int64_t batch);
/* 1 if the persistent form is built for this shape on the current device: c == 64 and at least
 * SM-count + tiles-per-image tiles per block (the scheduling argument in csrc/tc_chain.cu needs
 * that); otherwise run the blocks one by one with vqae_same_block_f16.                       */
int vqae_same_chain_supported(int64_t batch, int height, int width, int c);
int vqae_same_chain_f16(const float* x, float* buf_a, float* buf_b, const void* w_packed_all,
                         const float* scalars_dev, void* flags, size_t flag_bytes, int n_blocks,
                         int64_t batch, int height, int width, int c, void* stream);
/* The same run with the fp32 residual stream RESIDENT ON THE SM (c in {64, 128} at 32 x 32: the
 * 50-block trunks model.py:150-153,240-263 plus the adjacent post/pre layers; c == 32 at 64 x 64: the
 * five-block runs of the pyramids): a cluster of height / 8 CTAs owns an image, the residual lives in
 * tensor memory and branch_conv3 accumulates straight into it, halo rows travel through distributed
 * shared memory; the only global traffic is the first load and the last store of each image.  The
 * launch is persistent (at most as many clusters as the device holds at once; each works through
 * its share of the batch), any batch size.  w_packed_all: vqae_pack_resident_block_f16 outputs back
 * to back (11 * c * c bf16 per block, branch_conv3 pre-multiplied by the Fixup `scale`, so bias4 and
 * scale are applied as  x += (scale W3) v;  the bias4 terms are summed and added on the way out);
 * scalars_dev as for vqae_same_chain_f16.  x, out: NHWC fp32 [B,H,W,c]; out may alias x.
 * Deterministic (repeated launches are bit-identical).  Not bit-identical to vqae_same_block_f16
 * (rounding of scale*W3, accumulation order): agrees within the bf16 tolerance
 * (tests/test_gpu_tc.py).                                                                       */
/* 4-CTA clusters of the c == 64 resident kernel the current device holds at once (one image pair
 * each at a time); -1 on error.  Batches that are a multiple of twice this number keep every
 * cluster busy to the end.                                                                      */
int vqae_trunk_resident_max_clusters(void);
int vqae_trunk_resident_supported(int64_t batch, int height, int width, int c);
int vqae_pack_resident_block_f16(const float* w1_oihw, const float* w2_oihw, const float* w3_oihw,
                                  int c, float scale, void* packed, void* stream);
int vqae_trunk_resident_f16(const void* x, void* out, int io_dtype, const void* w_packed_all,
                            const float* scalars_dev, int n_blocks, int64_t batch, int height,
                            int width, int c, void* stream);
/* PreActFixupResBlock in mode 'down' (conv specs pre_activation_fixup.yaml:35-45): c_in ->
 * 2*c_in, stride 2, branch + skip fused in one tcgen05 kernel; c_in in {8, 16, 32} (csrc/tc_down.cu:
 * weights and all four parity planes resident in shared memory) and c_in == 64 (csrc/tc_down128.cu,
 * the 64 -> 128 block of the 512-model: planes one at a time, the 288 KB of weights per tile streamed
 * through a bulk-copy ring; fp32 I/O only); height % 16 == 0, width % 32 == 0.
 * w_packed: vqae_down_block_pack_elems(c_in) fp16 from vqae_pack_down_block_f16 /
 * vqae_pack_batched(VQAE_PACK_DOWN_F16) (scale is folded into branch_conv3 there);
 * scalars8_host = {bias1a, bias1b, bias2a, bias2b, bias3a, bias3b, bias1c, bias4 + bias1d}.
 * x: NHWC fp32 [B,H,W,c_in];  out: NHWC fp32 [B,H/2,W/2,2*c_in].                             */
size_t vqae_down_block_pack_elems(int c_in);
int vqae_pack_down_block_f16(const float* w1_oihw, const float* w2_oihw, const float* w3_oihw,
                              const float* wskip_oihw, int c_in, float scale, void* packed,
                              void* stream);
int vqae_down_block_f16(const void* x, void* out, int io_dtype, const void* w_packed,
                        const float* scalars8_host, int64_t batch, int height, int width, int c_in,
                        void* stream);

/* ---- a-P / a-Q / a-G  quantiser -------------------------------------------------------------
 * ProjectedEMAVectorQuantizer2d.forward + EMAVectorQuantizer.forward in eval mode
 * (layers/vq.py:96-154, 185-192):  z = proj_in(x);  idx = argmin_k sum_d (z_d - e_kd)^4
 * (torch.cdist with p = inputs.dim() = 4, first index wins ties);  q = embed[idx];
 * loss = mean((z - q)^2) * commitment_cost;  out = proj_out(q).
 *
 * vqae_quantizer_prepare builds the output table E' = proj_out(embed) ([K][c] fp32) once.
 * If w_in == NULL the call is the bare EMAVectorQuantizer on c == dim inputs and the output
 * rows are embed[idx] itself (table == embed).                                              */
int vqae_quantizer_prepare_f32(const float* embed, int num_codes, int dim,
                               const float* w_out /*[c][dim]*/, const float* b_out /*[c]*/,
                               int c, float* table /*[num_codes][c]*/, void* stream);

typedef struct vqae_quantizer_params {
    int num_codes;          /* K (256)                                                       */
    int dim;                /* D (8): distance space                                         */
    int c;                  /* channel count of x / out (64 or 128; == dim when bare)        */
    const float* embed;     /* [K][D]                                                        */
    const float* w_in;      /* proj_in weight [D][c] (OIHW with 1x1 taps), or NULL           */
    const float* b_in;      /* [D] or NULL                                                   */
    const float* table;     /* [K][c] from vqae_quantizer_prepare_f32                        */
    float commitment_cost;
} vqae_quantizer_params;

size_t vqae_quantizer_scratch_bytes(int64_t n_vectors);
/* x: fp32, [B,c,S] (NCHW, S = prod(spatial)) or [B,S,c] (NHWC);  out: same shape, layout
 * out_layout;  indices: int64 [B,S];  loss: 1 fp32;  near_ties: 1 uint32 (may be NULL) =
 * number of vectors whose top-2 relative gap of the un-rooted L4 sums is < tie_rel_gap.
 * z_out (may be NULL): fp32 [B*S][D] projected latents, for diagnostics/parity tests.      */
int vqae_quantize_f32(const vqae_quantizer_params* p, const float* x, int x_layout, float* out,
                      int out_layout, int64_t* indices, float* loss, uint32_t* near_ties,
                      float tie_rel_gap, float* z_out, void* scratch, size_t scratch_bytes,
                      int64_t batch, int64_t spatial, void* stream);

/* The tcgen05 form of the same call, taken automatically by vqae_quantize_f32 when
 * vqae_quantize_tc_supported() is 1 (proj_in present, K = 256, D = 8, c = 64,
 * NHWC in/out; env VQAE_QUANT_TC=0 disables it).  The tensor cores evaluate the quartic expansion
 * of sum_d (z_d - e_kd)^4 from bf16 hi/lo splits as a candidate filter; indices, loss and the
 * near-tie count come from the same exact fp32 evaluation as the CUDA-core kernel and are
 * bit-identical to it.  diag (may be NULL): fp32 [N][4] = {min approximate distance (offset by
 * -sum z^4), error scale T, number of candidates, 1 if the row took the full exact scan}.      */
int vqae_quantize_tc_supported(const vqae_quantizer_params* p, int x_layout, int out_layout,
                               int has_out);
/* General form: x / out in x_dtype / out_dtype (VQAE_DT_F32, VQAE_DT_BF16 or VQAE_DT_F16 -- the
 * distance arithmetic is fp32 whatever the I/O type, like torch.cdist under autocast), and an
 * explicit kernel choice instead of any environment switch: VQAE_QUANT_AUTO takes the tcgen05
 * kernel where vqae_quantize_supported(..., VQAE_QUANT_TENSOR_CORE) is 1 and the CUDA-core kernel
 * (fp32 I/O only) elsewhere; the other two values force one of them (VQAE_ERR_UNSUPPORTED if it
 * is not built for the shape).                                                                 */
enum { VQAE_QUANT_AUTO = 0, VQAE_QUANT_CUDA_CORE = 1, VQAE_QUANT_TENSOR_CORE = 2 };
int vqae_quantize_supported(const vqae_quantizer_params* p, int x_dtype, int x_layout,
                            int out_dtype, int out_layout, int has_out, int kernel);
int vqae_quantize(const vqae_quantizer_params* p, const void* x, int x_dtype, int x_layout,
                  void* out, int out_dtype, int out_layout, int64_t* indices, float* loss,
                  uint32_t* near_ties, float tie_rel_gap, float* z_out, void* scratch,
                  size_t scratch_bytes, int64_t batch, int64_t spatial, int kernel, void* stream);
int vqae_quantize_tc_f32(const vqae_quantizer_params* p, const float* x, float* out,
                         int64_t* indices, float* loss, uint32_t* near_ties, float tie_rel_gap,
                         float* z_out, float* diag, void* scratch, size_t scratch_bytes,
                         int64_t batch, int64_t spatial, void* stream);

/* embed_code -> proj_out (layers/vq.py:44-45,192): out[n,:] = table[idx[n],:].
 * indices: int64 or u8 (idx_dtype VQAE_DT_U8 / anything else = int64); out NHWC/NCHW fp32. */
int vqae_embed_codes_f32(const void* indices, int idx_is_u8, const float* table, int num_codes,
                         int c, float* out, int out_layout, int64_t batch, int64_t spatial,
                         void* stream);

/* vqae_embed_codes_f32 straight out of a stored code map: code_map u8 (map_is_u8 = 1) or int64
 * [map_rows, map_cols] made of th x tw code tiles; a region of region_cols patches per row starts at
 * patch (r0, c0); patch t = 0 .. n-1 of the call is region patch first_patch + t, i.e. map patch
 * (r0 + (first_patch + t) / region_cols, c0 + (first_patch + t) % region_cols).  out: NHWC fp32
 * [n, th, tw, c] = table[code] (codes clamped to [0, num_codes) like vqae_embed_codes_f32).
 * VQAE_ERR_BAD_ARG for a null pointer, a non-positive extent or a window outside the map.      */
int vqae_embed_codemap_f32(const void* code_map, int map_is_u8, int64_t map_rows, int64_t map_cols,
                           int th, int tw, int64_t r0, int64_t c0, int64_t region_cols,
                           int64_t first_patch, int64_t n, const float* table, int num_codes, int c,
                           float* out, void* stream);

/* ---- a-X  code-map placement (scripts/extract_embeddings/extract_embeddings.py:47-59,75-89) -
 * Places n_tiles [th,tw] int64 code tiles at (row*th, col*tw) of a u8 map [rows*th, cols*tw];
 * tile t has row-major patch index first_patch + t (datamodules/camelyon16.py:184-190).     */
int vqae_codemap_place_u8(const int64_t* tiles, int64_t n_tiles, int th, int tw,
                          int64_t first_patch, int grid_cols, uint8_t* map, int64_t map_rows,
                          int64_t map_cols, void* stream);
/* the same into an int64 map: the reference assembles slides in the encoder's index dtype and
 * narrows with cast_to_lowest_dtype only when a slide is complete (extract_embeddings.py:54-59,
 * 75-89), which is what codebooks of more than 256 entries need.                            */
int vqae_codemap_place_i64(const int64_t* tiles, int64_t n_tiles, int th, int tw,
                           int64_t first_patch, int grid_cols, int64_t* map, int64_t map_rows,
                           int64_t map_cols, void* stream);

/* ---- reconstruction quality of uint8 RGB patches (csrc/quality.cu) ---------------------------
 * The reference publishes reconstruction MSE (README.md:35,40) and validation MSE / PSNR / SSIM per
 * codebook size (scripts/extract_validation_metrics/results.md:3-6, eval.py:13-45, torchmetrics).
 * This call scores an original patch x against its reconstruction y, both uint8 H x W x 3:
 *   sse[b, c]  = sum over the patch of (x - y)^2 in channel c, exact (integer arithmetic), int64;
 *   ssim[b]    = mean over the 3 channels and the (H - 10)(W - 10) valid window positions (no padding)
 *                of (2 mu_x mu_y + C1)(2 s_xy + C2) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)),
 *                11 x 11 Gaussian window (sigma 1.5, the 11 taps normalised to sum 1 in float64 and
 *                rounded once to fp32), population moments, C1 = (0.01 * 255)^2, C2 = (0.03 * 255)^2;
 *                float64, moments accumulated in float64.
 * This is skimage.metrics.structural_similarity(gaussian_weights=True, sigma=1.5,
 * use_sample_covariance=False, data_range=255, channel_axis=-1).  Each input is a canvas uint8
 * [rows, cols, 3] holding a grid of height x width patches; patch t of the call sits at grid position
 * (r0 + (first + t) / region_cols, c0 + (first + t) % region_cols) -- the addressing of
 * vqae_embed_codemap_f32; region_cols = 1 on a [batch * height, width, 3] canvas is a plain batch.
 * Results depend on each patch's pixels only (not on its position in the batch, the batch size or the
 * grid): bitwise reproducible.  Checked before anything is launched: VQAE_ERR_BAD_ARG for a null
 * pointer, a non-positive extent or a placement outside either canvas; VQAE_ERR_UNSUPPORTED for
 * height or width < 11 or first + batch > 2^31; VQAE_ERR_SCRATCH when scratch is missing or smaller
 * than vqae_quality_u8_scratch_bytes (0 for an unsupported shape).                                */
size_t vqae_quality_u8_scratch_bytes(int64_t batch, int height, int width);
int vqae_quality_u8(const uint8_t* ref, int64_t ref_rows, int64_t ref_cols, int64_t ref_r0, int64_t ref_c0,
                    int64_t ref_region_cols, int64_t ref_first,
                    const uint8_t* rec, int64_t rec_rows, int64_t rec_cols, int64_t rec_r0, int64_t rec_c0,
                    int64_t rec_region_cols, int64_t rec_first,
                    int64_t batch, int height, int width, int64_t* sse, double* ssim,
                    void* scratch, size_t scratch_bytes, void* stream);

/* ---- packed code maps: per-patch rANS entropy coding (csrc/codemap_pack.cu, DESIGN.md 4.13) ---
 * A code map [map_rows, map_cols] (uint8 when map_is_u8 / out_is_u8, else int64) is a grid of th x tw
 * code tiles; patch p = row-major patch index.  Format version 1: one static table of num_codes (K)
 * frequencies freq_host[s] summing to 2^scale_bits (S), one rANS stream per patch (32-bit state,
 * L = 2^16, 16-bit words): the final encoder state (4 bytes LE), then the words in decoder order (2 bytes
 * LE each); 4 <= stream bytes <= 4 + 2 th tw, always even.  offsets [P + 1] (int64): stream p is
 * payload[offsets[p], offsets[p + 1]), offsets[0] = 0, offsets[P] = payload bytes.
 *
 * vqae_codemap_histogram   counts[K + 1] (int64): counts[s] = #codes equal to s in the window
 *                          rows [r0, r0 + nr) x cols [c0, c0 + nc) of the map (in codes), counts[K] = #codes
 *                          outside [0, K).  Exact (integer atomics), independent of the grid.
 * vqae_codemap_pack        codes every patch of the whole map with the table: writes offsets and the
 *                          payload (payload_capacity >= vqae_codemap_pack_worst_bytes).  A patch holding a
 *                          code outside [0, K) or with frequency 0 gets a 0-byte stream (offsets show it).
 * vqae_codemap_unpack      decodes the patches of the region (r0, c0, nr, nc) (in patches) into out
 *                          [nr th, nc tw] (patch t of the region, row-major, at (t / nc, t % nc) -- the
 *                          addressing of vqae_codemap_place_u8 with grid_cols = nc) and writes flags[nr nc]:
 *                          bit 0 the final state is not L, bit 1 the words were not exactly consumed,
 *                          bit 2 the stream length is not even within [4, 4 + 2 th tw].  offsets_host and
 *                          offsets hold the same P + 1 values (host copy validated, device copy read).
 *                          Every read of patch p stays inside its own [offsets[p], offsets[p + 1]) range
 *                          clamped to the payload; past its end a stream reads zero words.
 * Checked before anything is launched: VQAE_ERR_BAD_ARG for a null pointer, a non-positive extent, a
 * map that is not a grid of tiles, a window or region outside the map, frequencies not summing to 2^S,
 * offsets that do not start at 0, end at payload_bytes and step by an even 4 .. 4 + 2 th tw, or a short
 * payload_capacity; VQAE_ERR_UNSUPPORTED for K outside [1, 1024], S outside [1, 14], th tw > 16384,
 * more than 2^31 - 1 patches, or a uint8 output with K > 256; VQAE_ERR_SCRATCH when scratch is missing
 * or smaller than vqae_codemap_pack_scratch_bytes.                                                 */
int vqae_codemap_histogram(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int64_t r0,
                           int64_t c0, int64_t nr, int64_t nc, int num_codes, int64_t* counts, void* stream);
size_t vqae_codemap_pack_scratch_bytes(int64_t n_patches, int th, int tw);
int64_t vqae_codemap_pack_worst_bytes(int64_t n_patches, int th, int tw);
int vqae_codemap_pack(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int th, int tw,
                      const uint32_t* freq_host, int num_codes, int scale_bits, int64_t* offsets,
                      uint8_t* payload, int64_t payload_capacity, void* scratch, size_t scratch_bytes,
                      void* stream);
int vqae_codemap_unpack(const uint8_t* payload, int64_t payload_bytes, const int64_t* offsets_host,
                        const int64_t* offsets, int64_t map_rows, int64_t map_cols, int th, int tw,
                        const uint32_t* freq_host, int num_codes, int scale_bits, int64_t r0, int64_t c0,
                        int64_t nr, int64_t nc, void* out, int out_is_u8, uint8_t* flags, void* stream);

/* ---- box-filtered pyramid levels of uint8 RGB patches (csrc/pyramid.cu, DESIGN.md 4.14) ----------
 * Level k of the bit mask level_mask (bit k: factor f = 2^k, 1 <= k <= 9, f dividing height and width)
 * is, per channel, out = (S + f^2 / 2) >> 2k with S the exact integer sum of the f x f source pixels:
 * the box mean rounded half up (PIL.Image.reduce(f)), every level rounded once from the original
 * pixels.  The source is a canvas uint8 [src_rows, src_cols, 3] of height x width patches; patch t of the
 * call sits at grid position (r0 + (first + t) / region_cols, c0 + (first + t) % region_cols) -- the
 * addressing of vqae_quality_u8.  Level k goes to the canvas dst[k] uint8 [dst_rows[k], dst_cols[k], 3]
 * of (height / f) x (width / f) patches, at the position the dst_* tuple (shared by all levels) gives
 * patch t.  dst, dst_rows and dst_cols are host arrays of 10 entries indexed by k; entries of levels
 * not in the mask are not read.  Each source pixel is read once; integer arithmetic, no atomics: bitwise
 * reproducible, independent of the batch and the grid.  Checked before anything is launched:
 * VQAE_ERR_BAD_ARG for a null pointer (src, the arrays, dst[k] of a requested level), a non-positive
 * extent, an empty mask, a negative first or a placement outside any canvas; VQAE_ERR_UNSUPPORTED for
 * mask bits outside 1 .. 9, a factor not dividing height or width, or first + batch > 2^31;
 * VQAE_ERR_SCRATCH when vqae_pyramid_u8_scratch_bytes is nonzero (levels with f >= 128) and scratch is
 * missing or smaller (0 for an unsupported shape).                                                   */
size_t vqae_pyramid_u8_scratch_bytes(int64_t batch, int height, int width, int level_mask);
int vqae_pyramid_u8(const uint8_t* src, int64_t src_rows, int64_t src_cols, int64_t src_r0, int64_t src_c0,
                    int64_t src_region_cols, int64_t src_first, int64_t batch, int height, int width,
                    int level_mask, uint8_t* const* dst, const int64_t* dst_rows, const int64_t* dst_cols,
                    int64_t dst_r0, int64_t dst_c0, int64_t dst_region_cols, int64_t dst_first,
                    void* scratch, size_t scratch_bytes, void* stream);

/* ---- baseline JPEG tiles of a uint8 RGB canvas level (csrc/jpeg.cu, DESIGN.md 4.16) ---------------------
 * The level is ext_h x ext_w pixels of the canvas uint8 [.., pitch] (row y, column x, channel ch at
 * canvas[y * pitch + 3 x + ch]).  With tile size `tile` and `overlap`, tile (c, r) covers x in
 * [max(0, c tile - overlap), min(ext_w, (c + 1) tile + overlap)) and likewise y; the call encodes the tile
 * rows [row0, row0 + nrows), every column, row-major.  Each tile becomes the baseline JFIF file libjpeg
 * writes for quality `quality` and subsampling 0 (4:4:4) or 2 (4:2:0) with the standard Huffman tables:
 * headers_host (host) holds 16 headers of header_len bytes, header (4 row class + column class) for the
 * tiles of that class (class 0: the first row / column, 1: the middle ones, 2: the second-to-last, 3: the
 * last; in a grid of n < 4 tiles the lower class of a tile that is several); qtables_host (host)
 * the luminance and chrominance tables of that quality, 2 x 64 in zigzag order as in the DQT segments.
 * The files go back to back into `payload`, file i at [offsets[i], offsets[i + 1]) (offsets: device,
 * nrows * ncols + 1 int64, offsets[0] = 0).  Integer arithmetic, no atomics: each file depends on its
 * pixels, the tables and the subsampling only.  Checked before anything is launched: VQAE_ERR_BAD_ARG for
 * a null pointer, a non-positive extent, tile <= 0, overlap < 0, overlap >= tile, rows outside the tile
 * grid, pitch < 3 ext_w, a table entry outside [1, 255] or payload_capacity < vqae_jpeg_tiles_worst_bytes;
 * VQAE_ERR_UNSUPPORTED for quality outside 1 .. 100, subsampling not 0 or 2, or a tile side over 65535;
 * VQAE_ERR_SCRATCH when scratch_bytes < vqae_jpeg_tiles_scratch_bytes.  The two size queries return 0 /
 * -1 for arguments the encoder rejects.                                                                */
size_t vqae_jpeg_tiles_scratch_bytes(int64_t ext_h, int64_t ext_w, int tile, int overlap, int64_t row0,
                                     int64_t nrows, int subsampling, int header_len);
int64_t vqae_jpeg_tiles_worst_bytes(int64_t ext_h, int64_t ext_w, int tile, int overlap, int64_t row0,
                                    int64_t nrows, int subsampling, int header_len);
int vqae_jpeg_tiles(const uint8_t* canvas, int64_t pitch, int64_t ext_h, int64_t ext_w, int tile, int overlap,
                    int64_t row0, int64_t nrows, int quality, int subsampling, const uint8_t* headers_host,
                    int header_len, const uint16_t* qtables_host, int64_t* offsets, uint8_t* payload,
                    int64_t payload_capacity, void* scratch, size_t scratch_bytes, void* stream);

/* ---- near-lossless residual layer of stored code maps (csrc/residual.cu, DESIGN.md 4.15) ----------
 * Patches are height x width x 3 uint8, n = 3 height width bytes in canvas order (row-major, channel
 * innermost); x the original, base the decode of the map, e = max_error in [0, 127], d = x - base:
 *   e = 0:  symbol s = d & 255,  x' = (base + s) & 255 = x;
 *   e >= 1: k = sign(d) floor((|d| + e) / (2e + 1)), s = k & 255, x' = clamp(base + k (2e + 1), 0, 255),
 *           |x - x'| <= e.
 * A chunk per patch: 256 x u16 frequencies (total 2^14), 32 x u32 lane word counts, 32 x u32 final lane
 * states, then the 16-bit words of lanes 0 .. 31 in decoder order, little-endian; symbol i is coded by rANS
 * lane i mod 32 (32-bit state, L = 2^16, at most one word per symbol); 768 + 2 sum(w) bytes, at most
 * 768 + 2 n.  Adler-32 values are zlib.adler32 of a patch's bytes in canvas order, (B << 16) | A.
 * Every canvas is uint8 [rows, cols, 3] with the addressing tuple of vqae_quality_u8.
 *
 * vqae_residual_stats      hist[batch][256] (int64): exact symbol counts per patch; adler[batch][2]: the
 *                          Adler-32 of base and of x'.
 * vqae_residual_tables     freq[batch][256] (int32) from hist: packing.quantise_frequencies with S = 14.
 * vqae_residual_encode     codes each patch of the call with its row of freq into offsets[batch + 1] and
 *                          the payload (payload_capacity >= batch (768 + 2 n)).  A patch with a symbol of
 *                          frequency 0 (freq not made from these pixels) gets a 0-byte chunk.
 * vqae_residual_apply      decodes the chunks of patches (layer_r0 + q / layer_region_cols) grid_cols +
 *                          layer_c0 + q % layer_region_cols, q = layer_first + t, of a layer of grid_rows x
 *                          grid_cols patches and replaces the base pixels of patch t of the canvas with x'
 *                          in place; adler holds the layer's [P][2] stored values.  flags[batch]: bit 0 the
 *                          chunk failed (a lane not back at L with its words exactly consumed, a table not
 *                          summing to 2^14, a length that disagrees with the word counts), bit 1 the base
 *                          Adler differs, bit 2 the output Adler differs.  Reads of a chunk stay inside its
 *                          own [offsets[p], offsets[p + 1]) range clamped to the payload.
 * Integer arithmetic, no atomics: bitwise reproducible, independent of the batch and the grid.  Checked
 * before anything is launched: VQAE_ERR_BAD_ARG for a null pointer, a non-positive extent, a negative e or
 * first, a placement outside a canvas or the layer grid, a short payload_capacity, or offsets_host (the
 * P + 1 offsets on the host) not starting at 0, ending at payload_bytes and stepping by an even
 * 768 .. 768 + 2 n; VQAE_ERR_UNSUPPORTED for e > 127, height x width > 2^20 or first + batch > 2^31;
 * VQAE_ERR_SCRATCH when scratch is missing or smaller than vqae_residual_encode_scratch_bytes.        */
int vqae_residual_stats(const uint8_t* x, int64_t x_rows, int64_t x_cols, int64_t x_r0, int64_t x_c0,
                        int64_t x_region_cols, int64_t x_first, const uint8_t* base, int64_t base_rows,
                        int64_t base_cols, int64_t base_r0, int64_t base_c0, int64_t base_region_cols,
                        int64_t base_first, int64_t batch, int height, int width, int max_error, int64_t* hist,
                        uint32_t* adler, void* stream);
int vqae_residual_tables(const int64_t* hist, int64_t batch, int32_t* freq, void* stream);
size_t vqae_residual_encode_scratch_bytes(int64_t batch, int height, int width);
int vqae_residual_encode(const uint8_t* x, int64_t x_rows, int64_t x_cols, int64_t x_r0, int64_t x_c0,
                         int64_t x_region_cols, int64_t x_first, const uint8_t* base, int64_t base_rows,
                         int64_t base_cols, int64_t base_r0, int64_t base_c0, int64_t base_region_cols,
                         int64_t base_first, int64_t batch, int height, int width, int max_error,
                         const int32_t* freq, int64_t* offsets, uint8_t* payload, int64_t payload_capacity,
                         void* scratch, size_t scratch_bytes, void* stream);
int vqae_residual_apply(const uint8_t* payload, int64_t payload_bytes, const int64_t* offsets_host,
                        const int64_t* offsets, const uint32_t* adler, int64_t grid_rows, int64_t grid_cols,
                        int64_t layer_r0, int64_t layer_c0, int64_t layer_region_cols, int64_t layer_first,
                        uint8_t* canvas, int64_t rows, int64_t cols, int64_t r0, int64_t c0, int64_t region_cols,
                        int64_t first, int64_t batch, int height, int width, int max_error, uint8_t* flags,
                        void* stream);

/* ---- f-4  training-mode codebook maintenance (layers/vq.py:47-94) -----------------------------
 * EMAVectorQuantizer._update_ema / _init_ema without the N x K one-hot matrix of the reference:
 *   vqae_ema_accumulate_f32   counts[k] = #{n : idx[n] = k},  dw[k,:] = sum of z[n,:] over those n
 *                             (vq.py:49-54: one_hot.sum(0), one_hot.T @ flat_input); deterministic
 *                             (fixed summation order, no atomics).  The all-reduce of counts / dw
 *                             across ranks (vq.py:56-58) is the caller's, between this and the update.
 *   vqae_ema_update_f32       vq.py:60-74: EMA of cluster_size / embed_avg, Laplace smoothing,
 *                             embed = embed_avg / smoothed cluster size; all three buffers in place.
 *   vqae_column_stats_f32     mean and unbiased std of z over its rows (vq.py:77-78)
 *   vqae_ema_init_f32         vq.py:90-94: embed = embed * std + mean, embed_avg = embed,
 *                             cluster_size += cluster_add  (= N * world_size / K)
 * z: [n, dim] fp32 row-major (the `z_out` of vqae_quantize), indices: int64 [n].                 */
size_t vqae_ema_scratch_bytes(int64_t n, int num_codes, int dim);
int vqae_ema_accumulate_f32(const float* z, const int64_t* indices, int64_t n, int num_codes, int dim,
                            float* counts, float* dw, void* scratch, size_t scratch_bytes,
                            void* stream);
int vqae_ema_update_f32(float* embed, float* embed_avg, float* cluster_size, const float* counts,
                        const float* dw, int num_codes, int dim, float decay, float laplace_alpha,
                        void* stream);
int vqae_column_stats_f32(const float* z, int64_t n, int dim, float* mean, float* std_unbiased,
                          void* scratch, size_t scratch_bytes, void* stream);
int vqae_ema_init_f32(float* embed, float* embed_avg, float* cluster_size, const float* mean,
                      const float* std_unbiased, int num_codes, int dim, float cluster_add,
                      void* stream);

/* out = a + b over n fp32 elements (16-byte aligned pointers): the level sums of the multi-level
 * hierarchy, `down + shortcut(aux)` (model.py:208) and `shortcut(aux) + enc`, `prev_up + ...`
 * (model.py:283-288).  out may alias a or b.                                                     */
int vqae_add_f32(const float* a, const float* b, float* out, int64_t n, void* stream);

/* ---- f-4  MBConv (layers/conv_block.py:240-321) and SELayer (layers/misc.py:7-30), eval mode --------
 * The block is  out = BN3(W3 . (t2 * gate)) + skip(x),  t2 = SiLU(BN2(depthwise(SiLU(BN1(W1 . x))))),
 * gate = SELayer(t2); BatchNorm in eval mode arrives folded as per-channel (scale, shift).  NHWC fp32.
 *
 * vqae_pointwise_conv_f32: a full conv as a GEMM over pixels with a fused epilogue
 *     out[p, n] = act(scale[n] * sum_k A[p, k] w[n, k] + shift[n]) + res[p, n]
 *   mode 0: 1x1 conv, A = the input rows, K = c_in                         (nn.Conv2d k=1; proj2d.yaml)
 *   mode 1: 2x2 stride-2 conv, A = space-to-depth rows, K = 4 c_in,        (down2d.yaml)
 *           w[n][(dy*2+dx)*c_in + ci]
 *   mode 2: 2x2 stride-2 transposed conv, w = [4][n_out][c_in], one matrix (up2d.yaml, ConvTranspose2d)
 *           per output parity (dy, dx); out is [B, 2 hi, 2 wi, n_out]
 *   scale / shift / gate ([B, c_in], mode 0 only: A[p, k] *= gate[image(p), k]) / res may be NULL.
 * vqae_depthwise_conv_f32: one filter per channel, w_taps = [taps][c]; mode 0: 3x3 circular, 1: 2x2 stride 2,
 *   2: 2x2 stride-2 transposed; then affine + SiLU; row_sums [B, rows_out, c] (or NULL) receives each
 *   output row's channel sums for the squeeze of the SELayer (fixed summation order).
 * vqae_se_gate_f32: gate[b, :] = sigmoid(w2 . SiLU(w1 . mean + b1) + b2), mean = sum of row_sums / pixels. */
int vqae_pointwise_conv_f32(const float* a, const float* w, const float* scale, const float* shift,
                            const float* gate, const float* res, float* out, int64_t batch, int hi, int wi,
                            int c_in, int n_out, int mode, int act_silu, void* stream);
int vqae_depthwise_conv_f32(const float* in, const float* w_taps, const float* scale, const float* shift,
                            float* out, float* row_sums, int64_t batch, int hi, int wi, int c, int mode,
                            void* stream);
int vqae_se_gate_f32(const float* row_sums, int64_t batch, int rows, int pixels_per_image, int c,
                     const float* w1, const float* b1, const float* w2, const float* b2, int c_hidden,
                     float* gate, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VQAE_B200_H_ */

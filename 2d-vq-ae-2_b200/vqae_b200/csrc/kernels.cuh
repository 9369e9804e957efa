// Internal (C++) launch interface between the C-ABI in abi.cu and the kernel files.
#pragma once
#include "common.cuh"

namespace vqae {

enum ConvKind { CONV_1x1 = 0, CONV_2x2S2 = 1, CONV_3x3_CIRC = 2 };

// conv_f32.cu
int conv_f32(int kind, const float* in, const float* w, float* out, const float* res, int64_t B,
             int Hi, int Wi, int Cin, int Cout, PreOp pre, float scale, float bias,
             cudaStream_t stream);
int bicubic_up2_f32(const float* in, float* out, int64_t B, int H, int W, int C, float bias,
                    cudaStream_t stream);
int pack_conv_weight_f32(const float* w, float* packed, int O, int I, int taps,
                         cudaStream_t stream);

// pack.cu (every weight layout; one launch for a whole model's convs)
size_t pack_elems(int kind, int c_in, int c_out, int taps);
int pack_one(vqae_pack_desc d, cudaStream_t stream);
int pack_batched(const vqae_pack_desc* descs_dev, int n_descs, int max_elems, cudaStream_t stream);

// up_head.cu (low-resolution half of an 'up' block: the three 1x1 convs in one pointwise kernel)
bool up_head_supported(int64_t P, int ci, int cb, int co);
int up_head_f32(const float* x, const float* w1, const float* w2, const float* ws, float* t2, float* s1,
                int64_t P, int ci, int cb, int co, float b1a, float b1b, float b2a, float b2b, float b1c,
                cudaStream_t stream);

// up_tail.cu (high-resolution half of an 'up' block in one kernel)
bool up_tail_supported(int64_t B, int H, int W, int cb, int co);
int up_tail_f32(const float* t2, const float* s1, const float* w3, float* out, int64_t B, int H, int W,
                int cb, int co, float b3a, float b3b, float scale, float b4, float b1d,
                cudaStream_t stream);

// stems.cu
int normalize_u8(const uint8_t* img, float* out, int64_t B, int H, int W, const float* mean,
                 const float* stdv, int out_layout, cudaStream_t stream);
int stem_in_f32(const void* x, int x_dtype, int x_layout, const float* w, const float* bias,
                void* out, int out_dtype, int64_t B, int H, int W, int c_out, const float* mean,
                const float* stdv, cudaStream_t stream);
int stem_out_f32(const float* x, const float* w, const float* bias, float* out, int out_layout,
                 int64_t B, int H, int W, int c_in, cudaStream_t stream);
int stem_out_u8(const float* x, const float* w, const float* bias, const U8Canvas& cv, int64_t B,
                int H, int W, int c_in, cudaStream_t stream);

// quantize.cu
int quantizer_prepare_f32(const float* embed, int K, int D, const float* w_out,
                          const float* b_out, int C, float* table, cudaStream_t stream);
size_t quantizer_scratch_bytes(int64_t n);
int quantize_f32(const vqae_quantizer_params* p, const float* x, int x_layout, float* out,
                 int out_layout, int64_t* indices, float* loss, uint32_t* near_ties,
                 float tie_rel_gap, float* z_out, void* scratch, size_t scratch_bytes,
                 int64_t B, int64_t S, cudaStream_t stream, int kernel = VQAE_QUANT_AUTO);
bool quantize_supported(const vqae_quantizer_params* p, int x_dtype, int x_layout, int out_dtype,
                        int out_layout, bool has_out, int kernel);
int quantize_any(const vqae_quantizer_params* p, const void* x, int x_dtype, int x_layout, void* out,
                 int out_dtype, int out_layout, int64_t* indices, float* loss, uint32_t* near_ties,
                 float tie_rel_gap, float* z_out, void* scratch, size_t scratch_bytes, int64_t B,
                 int64_t S, int kernel, cudaStream_t stream);
int embed_codes_f32(const void* indices, int idx_is_u8, const float* table, int K, int C,
                    float* out, int out_layout, int64_t B, int64_t S, cudaStream_t stream);
int embed_codemap_f32(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int th,
                      int tw, int64_t r0, int64_t c0, int64_t region_cols, int64_t first_patch,
                      int64_t n, const float* table, int K, int C, float* out, cudaStream_t stream);
int codemap_place_u8(const int64_t* tiles, int64_t n_tiles, int th, int tw, int64_t first_patch,
                     int grid_cols, uint8_t* map, int64_t map_rows, int64_t map_cols,
                     cudaStream_t stream);
int codemap_place_i64(const int64_t* tiles, int64_t n_tiles, int th, int tw, int64_t first_patch,
                      int grid_cols, int64_t* map, int64_t map_rows, int64_t map_cols,
                      cudaStream_t stream);

// quantize_tc.cu (tcgen05 candidate filter + exact fp32 argmin)
bool quantize_tc_supported(const vqae_quantizer_params* p, int x_layout, int out_layout,
                           bool has_out);
int quantize_tc_f32(const vqae_quantizer_params* p, const float* x, float* out, int64_t* indices,
                    float* loss, void* scratch, uint32_t* near_ties, float tie_rel_gap,
                    float* z_out, float* diag, int64_t N, int sm_count, cudaStream_t stream);
int quantize_tc(const vqae_quantizer_params* p, const void* x, void* out, int dtype,
                int64_t* indices, float* loss, void* scratch, uint32_t* near_ties,
                float tie_rel_gap, float* z_out, float* diag, int64_t N, int sm_count,
                cudaStream_t stream);
size_t quantize_tc_scratch_bytes(int64_t n);
void quantize_tc_set_prof(long long* dev_ptr);
int device_sm_count(int* out);

// tc_kernels.cu (tcgen05 bf16 path)
int same_block_tc(const void* x, void* out, int io_dtype, const void* w_packed,
                  const float* scalars8, int64_t B, int H, int W, int C, int sm_count,
                  long long* prof, cudaStream_t stream);
int pack_same_block_f16(const float* w1, const float* w2, const float* w3, int C, void* packed,
                         cudaStream_t stream);

// mma_same.cu (low-channel 'same' blocks on warp-level MMAs)
bool same_block_mma_supported(int H, int W, int C);
int same_block_mma(const float* x, float* out, const void* w_packed, const float* scalars8,
                   int64_t B, int H, int W, int C, int sm_count, cudaStream_t stream);

// mma_down.cu ('down' blocks on warp-level MMAs, register-resident)
bool down_block_mma_supported(int H, int W, int CI);
int down_block_mma(const float* x, float* out, const void* w_packed, const float* scalars8,
                   int64_t B, int H, int W, int CI, int sm_count, cudaStream_t stream);

int down_block_split(const float* x, float* out, const void* w_hi, const void* w_lo,
                     const float* scalars8, const float* premul3, int64_t B, int H, int W, int CI,
                     int sm_count, cudaStream_t stream);

// mma_same_split.cu (fp32-accurate 'same' block at C = 8, 16: split fp16 operands on warp-level MMAs)
bool same_block_mma_split_supported(int H, int W, int C);
int same_block_mma_split(const float* x, float* out, const void* w_hi, const void* w_lo,
                         const float* scalars8, const float* premul3, int64_t B, int H, int W, int C,
                         int sm_count, cudaStream_t stream);

// tc_split.cu (fp32-accurate 'same' block: split fp16 operands on tcgen05)
bool same_block_split_supported(int H, int W, int C);
int same_block_split(const float* x, float* out, const void* w_hi, const void* w_lo,
                     const float* scalars8, const float* premul3, int64_t B, int H, int W, int C,
                     int sm_count, cudaStream_t stream);

// mma_front.cu (in_stem + 'same' C = 8 + 'down' 8 -> 16 in one kernel)
bool front_fused_supported(int H, int W);
int front_fused(const void* x, int x_dtype, int x_layout, const float* stem_w, const float* stem_b,
                const float* mean, const float* stdv, const void* same_w, const float* same_scalars8,
                const void* down_w, const float* down_scalars8, float* out, int64_t B, int H, int W,
                int sm_count, cudaStream_t stream);

// tc_down128.cu ('down' 64 -> 128 on tcgen05 with streamed weights)
bool down128_tc_supported(int H, int W, int CI);
int down128_tc(const float* x, float* out, const void* w_packed, const float* scalars8, int64_t B,
               int H, int W, int CI, int sm_count, cudaStream_t stream);

// mma_stem.cu (in_stem / out_stem on split-operand MMAs)
bool stem_in_mma_supported(int H, int W, int c_out);
int stem_in_mma(const void* x, int x_dtype, int x_layout, const float* w, const float* bias, float* out,
                int64_t B, int H, int W, int c_out, const float* mean, const float* stdv, int sm_count,
                cudaStream_t stream);
bool stem_out_mma_supported(int H, int W, int c_in);
int stem_out_mma_u8(const float* x, const float* w, const float* bias, const U8Canvas& cv, int64_t B,
                    int H, int W, int c_in, int sm_count, cudaStream_t stream);
int stem_out_mma(const float* x, const float* w, const float* bias, float* out, int out_layout,
                 int64_t B, int H, int W, int c_in, int sm_count, cudaStream_t stream);

// mma_up.cu ('up' blocks on warp-level MMAs: low-resolution head + high-resolution tail)
bool up_block_mma_supported(int H, int W, int CI);
size_t up_block_mma_scratch_bytes(int64_t B, int H, int W, int CI);
int up_block_mma(const float* x, float* out, const void* w_packed, const float* scalars8,
                 void* scratch, size_t scratch_bytes, int64_t B, int H, int W, int CI, int sm_count,
                 cudaStream_t stream);

// tc_chain.cu (persistent multi-block 'same' chain)
size_t same_chain_flag_bytes(int n_blocks, int64_t B);
bool same_chain_supported(int64_t B, int H, int W, int C, int sm_count);
int same_chain_tc(const float* x, float* buf_a, float* buf_b, const void* w_packed_all,
                  const float* scalars_dev, void* flags, size_t flag_bytes, int n_blocks, int64_t B,
                  int H, int W, int C, int sm_count, cudaStream_t stream);

// tc_resident.cu (image-resident trunk: residual stream in tensor memory, 4-CTA clusters)
bool trunk_resident_supported(int64_t B, int H, int W, int C);
int pack_resident_block_f16(const float* w1, const float* w2, const float* w3, int C, float scale,
                             void* packed, cudaStream_t stream);
int trunk_resident_max_clusters(int* out);
void trunk_resident_set_prof(long long* dev_ptr);
int trunk_resident_tc(const void* x, void* out, int io_dtype, const void* w_packed_all,
                      const float* scalars_dev, int n_blocks, int64_t B, int H, int W, int C,
                      cudaStream_t stream);

// tc_bench.cu
int tc_mma_bench2(int M, int N, int reps, int n_issuers, int ctas_per_sm, int mode, long long* out,
                  cudaStream_t stream);
// tc_down.cu
size_t down_block_pack_elems(int CI);
int pack_down_block_f16(const float* w1, const float* w2, const float* w3, const float* ws, int CI,
                         float scale, void* packed, cudaStream_t stream);
int down_block_tc(const void* x, void* out, int io_dtype, const void* w_packed,
                  const float* scalars8, int64_t B, int H, int W, int CI, int sm_count,
                  cudaStream_t stream);

// quality.cu (per-patch SSE and SSIM of two uint8 RGB images)
size_t quality_u8_scratch_bytes(int64_t batch, int H, int W);
int quality_u8(const uint8_t* ref, int64_t ref_rows, int64_t ref_cols, int64_t ref_r0, int64_t ref_c0,
               int64_t ref_rc, int64_t ref_first, const uint8_t* rec, int64_t rec_rows, int64_t rec_cols,
               int64_t rec_r0, int64_t rec_c0, int64_t rec_rc, int64_t rec_first, int64_t batch, int H,
               int W, int64_t* sse, double* ssim, void* scratch, size_t scratch_bytes,
               cudaStream_t stream);

// codemap_pack.cu (packed code maps: histogram, rANS pack, region unpack)
int codemap_histogram(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int64_t r0,
                      int64_t c0, int64_t nr, int64_t nc, int K, int64_t* counts, cudaStream_t stream);
size_t codemap_pack_scratch_bytes(int64_t n_patches, int th, int tw);
int64_t codemap_pack_worst_bytes(int64_t n_patches, int th, int tw);
int codemap_pack(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int th, int tw,
                 const uint32_t* freq_host, int K, int S, int64_t* offsets, uint8_t* payload,
                 int64_t payload_capacity, void* scratch, size_t scratch_bytes, cudaStream_t stream);
int codemap_unpack(const uint8_t* payload, int64_t payload_bytes, const int64_t* offsets_host,
                   const int64_t* offsets, int64_t map_rows, int64_t map_cols, int th, int tw,
                   const uint32_t* freq_host, int K, int S, int64_t r0, int64_t c0, int64_t nr, int64_t nc,
                   void* out, int out_is_u8, uint8_t* flags, cudaStream_t stream);

}  // namespace vqae

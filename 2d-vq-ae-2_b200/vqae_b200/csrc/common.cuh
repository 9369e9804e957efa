// Shared helpers for the sm_100a kernels of the VQ-AE inference path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "vqae_b200.h"

namespace vqae {

// thread-local record of the last CUDA error (vqae_last_cuda_error)
void set_last_cuda_error(cudaError_t e);
void count_launch(int n = 1);

inline int check_launch() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_cuda_error(e);
        return VQAE_ERR_CUDA;
    }
    count_launch();
    return VQAE_OK;
}

#define VQAE_CUDA_TRY(expr)                         \
    do {                                            \
        cudaError_t _e = (expr);                    \
        if (_e != cudaSuccess) {                    \
            ::vqae::set_last_cuda_error(_e);        \
            return VQAE_ERR_CUDA;                   \
        }                                           \
    } while (0)

// nn.ELU(alpha=1) (conf/model/layers/activation/elu.yaml): x > 0 ? x : expm1(x)
__device__ __forceinline__ float elu1(float x) { return x > 0.0f ? x : expm1f(x); }

// ELU of the fp32-accurate tensor-core mode ("fp32tc"): expm1f costs ~25 instructions per element and the
// split-operand kernels are bound by exactly that arithmetic.  For x <= 0:
//   |x| < 1/4 : expm1(x) = x (1 + x/2 + x^2/6 + ... + x^6/5040)     truncation < 2e-9 |x|
//   otherwise : exp2(x log2 e) - 1 with the SFU exponential          |error| < 2.5e-7 e^x  (<= 9e-7 relative)
// i.e. fp32-grade (one to a few ulps of the value) at a third of the instructions; the model goldens hold
// with the same bars as the exact path (tests/test_gpu_parity.py::test_model_vs_reference_golden[fp32tc-*]).
__device__ __forceinline__ float elu1_tc(float x) {
    const float p = x * fmaf(x, fmaf(x, fmaf(x, fmaf(x, fmaf(x, fmaf(x, 1.0f / 5040.0f, 1.0f / 720.0f),
                                                              1.0f / 120.0f), 1.0f / 24.0f), 1.0f / 6.0f), 0.5f), 1.0f);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 1.4426950408889634f));
    return x > 0.0f ? x : (x > -0.25f ? p : e - 1.0f);
}

// the pre-activation in front of every branch conv of PreActFixupResBlock
// (layers/conv_block.py:199-208):  conv(act(x + a) + b);  act optional (skip path has none)
struct PreOp {
    float a;
    float b;
    int use_elu;
    __device__ __forceinline__ float operator()(float x) const {
        float v = x + a;
        if (use_elu) v = elu1(v);
        return v + b;
    }
};

// The uint8 output of out_stem, the exact inverse of the input normalisation (vqae_normalize_u8):
// s_c = 255 std_c and o_c = 255 mean_c formed in fp32 on the host,
//     u8 = min(max(rint(fma(v, s_c, o_c)), 0), 255)      round half to even; NaN -> 0 (fmaxf drops it)
__device__ __forceinline__ uint8_t u8_store(float v, float s, float o) {
    return (uint8_t)fminf(fmaxf(rintf(fmaf(v, s, o)), 0.0f), 255.0f);
}

// Where the uint8 form of out_stem writes: image b of the call is patch q = first_patch + b of a
// canvas uint8 [canvas_rows, canvas_cols, 3] laid out as a grid of H x W patches with grid_cols
// patches per row, i.e. at canvas pixel ((q / grid_cols) H, (q % grid_cols) W) -- the addressing
// of codemap_place.  vec = 1: rows are 16-byte aligned (canvas_cols % 16 == 0, aligned base).
struct U8Canvas {
    uint8_t* canvas;
    int64_t canvas_cols, first_patch;
    int grid_cols, vec;
    float s[3], o[3];
};
// host: validates the placement (VQAE_OK or VQAE_ERR_BAD_ARG) and fills the canvas descriptor
int make_u8_canvas(uint8_t* canvas, int64_t canvas_rows, int64_t canvas_cols, int64_t first_patch,
                   int grid_cols, int64_t B, int H, int W, const float* mean, const float* stdv,
                   U8Canvas* cv);

// Per-device caches: function attributes, occupancy results and scratch allocations belong to ONE
// device; a process that drives several GPUs must not reuse them across devices.
constexpr int kMaxDevices = 64;
inline int current_device_index() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) return 0;
    return d;
}
template <typename T>
struct PerDevice {
    T v[kMaxDevices];
    T& cur() { return v[current_device_index()]; }
};

inline unsigned ceil_div_u(int64_t a, int64_t b) { return (unsigned)((a + b - 1) / b); }

}  // namespace vqae

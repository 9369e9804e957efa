// The rANS coder shared by the packed code maps (codemap_pack.cu, DESIGN.md section 4.13) and the residual
// layer (residual.cu, section 4.15): 32-bit state x in [L, 2^32), L = 2^16, 16-bit words, at most one word
// per symbol; and the fixed-order scan + compaction that turns worst-case slots into a payload.
#pragma once

#include "common.cuh"

namespace vqae {

constexpr uint32_t RANS_L = 1u << 16;           // lower end of the state interval

// encode one symbol of frequency f (0 < f <= 2^S) and start c: returns true and sets `word` when the state
// had to be renormalised first (the comparison is 64-bit: f = 2^S gives 2^32)
__device__ __forceinline__ bool rans_encode(uint32_t& x, uint32_t f, uint32_t c, int S, uint16_t& word) {
    bool emit = false;
    if ((uint64_t)x >= ((uint64_t)f << (32 - S))) {
        word = (uint16_t)(x & 0xffffu);
        x >>= 16;
        emit = true;
    }
    x = ((x / f) << S) + x % f + c;
    return emit;
}

// The P + 1 payload offsets of `sizes` (an exclusive scan in a fixed order, offsets[0] = 0), then every
// stream copied from its worst-case slot (slot p at slots + p * slot_bytes, sizes even) to its offset of
// the payload (codemap_pack.cu).
int rans_offsets_and_compact(const uint32_t* sizes, int64_t P, const uint8_t* slots, int64_t slot_bytes,
                             int64_t* offsets, uint8_t* payload, int64_t capacity, cudaStream_t stream);

}  // namespace vqae

// Entropy coding of stored code maps: packed code map, version 1 (DESIGN.md section 4.13;
// include/vqae_b200.h, vqae_codemap_histogram / vqae_codemap_pack / vqae_codemap_unpack).
//
// One chunk per code tile (patch), patches in row-major patch order, the n = th * tw codes of a tile in
// row-major order.  One static table per map: frequencies f[s] summing to M = 2^S (S <= 14), cumulative
// starts c[s] = f[0] + ... + f[s - 1].  Each patch is coded by rANS with one 32-bit state x in
// [L, 2^32), L = 2^16, and 16-bit renormalisation words:
//   encode s (codes taken last to first, x = L at the start):
//       if x >= f << (32 - S) (a 64-bit comparison: f = 2^S gives 2^32):  emit x & 0xffff, x >>= 16
//       x = ((x / f) << S) + x % f + c
//   decode (codes first to last, x = the stored state):
//       slot = x & (M - 1), s = the symbol with c[s] <= slot < c[s] + f[s],
//       x = f * (x >> S) + slot - c;  if x < L: x = (x << 16) | next word
// At most one word per code (x >> 16 < 2^16 <= f << (32 - S)), so a stream is at most 4 + 2 n bytes.
// A patch's stream: the final encoder state (4 bytes, little-endian), then the words in the order the
// decoder reads them (the reverse of the order they were emitted), 2 bytes each, little-endian.  A
// decoder that has decoded all n codes must be back at x = L with every word consumed.
//
// Kernels: one thread per patch.  The encoder stages its CTA's tiles in shared memory (uint16 per code,
// coalesced loads from the map), codes each tile in place -- the word emitted while coding code i goes
// to a position >= i of the tile's own buffer, which holds only codes that have been read -- and writes
// the streams, coalesced, into worst-case-sized slots of scratch with their sizes; a single-CTA scan turns
// the sizes into the P + 1 payload offsets and a compaction kernel copies each stream to its offset.  The
// decoder stages each stream into the tile buffer at positions [n - w, n) and decodes in place: after
// code i has been decoded, the first unread word sits at a position > i for a well-formed stream.
//
// Bounds by construction: every patch's reads are clamped to its own [offset, next offset) range of the
// payload (itself clamped to [0, payload bytes)), a stream's word count to [0, n]; a read past the end
// yields a zero word.  Symbols come from the slot table, which the validated frequencies fill with
// values below K.  Corrupt streams therefore give wrong codes and a raised flag, never an access outside
// the payload, the tables or the patch's own buffer.
#include "common.cuh"
#include "kernels.cuh"

namespace vqae {

namespace {

constexpr uint32_t PK_L = 1u << 16;           // lower end of the state interval
constexpr int PK_MAX_K = 1024;                // the quantiser's own codebook limit
constexpr int PK_MAX_S = 14;
constexpr int PK_MAX_CODES = 16384;           // th * tw
constexpr int PK_PPC = 32;                    // patches (= threads) per CTA of the coder kernels
constexpr size_t PK_SMEM_BUDGET = 200 * 1024;
constexpr int PK_HIST_THREADS = 256;
constexpr int PK_SCAN_THREADS = 1024;
constexpr uint16_t PK_BAD = 0xffff;           // staged code outside [0, K)

// f | c << 16 per symbol (f <= 2^14, c <= 2^14); symbols past K are never looked up
struct PackTable {
    uint32_t fc[PK_MAX_K];
};

// tile buffer stride in uint16: an odd number of 32-bit words, so the 32 threads of a warp reading
// position i of their own tiles hit 32 different banks
inline int tile_stride(int n) { return 2 * (((n + 1) / 2) | 1); }

template <typename MapT>
__device__ __forceinline__ uint32_t code_bin(MapT v, int K) {
    if constexpr (sizeof(MapT) == 1) return (int)v < K ? (uint32_t)v : (uint32_t)K;
    else return (v >= 0 && v < K) ? (uint32_t)v : (uint32_t)K;
}

// ---- histogram: privatised 64-bit shared bins, warp-aggregated, K + 1 bins (the last: codes outside
// [0, K)); integer sums, so the counts do not depend on the grid -------------------------------------
template <typename MapT>
__global__ void __launch_bounds__(PK_HIST_THREADS)
codemap_histogram_kernel(const MapT* __restrict__ map, int64_t map_cols, int64_t r0, int64_t c0, int64_t nr,
                         int64_t nc, int K, unsigned long long* __restrict__ counts) {
    __shared__ unsigned long long bins[PK_MAX_K + 1];
    for (int b = threadIdx.x; b <= K; b += blockDim.x) bins[b] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int64_t r = blockIdx.x; r < nr; r += gridDim.x) {
        const MapT* row = map + (r0 + r) * map_cols + c0;
        for (int64_t c = threadIdx.x; c < nc; c += blockDim.x) {
            const uint32_t b = code_bin(__ldg(row + c), K);
            const unsigned same = __match_any_sync(__activemask(), b);
            if (lane == __ffs(same) - 1) atomicAdd(&bins[b], (unsigned long long)__popc(same));
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b <= K; b += blockDim.x)
        if (bins[b]) atomicAdd(&counts[b], bins[b]);
}

// ---- encoder: one thread per patch, PK_PPC patches per CTA --------------------------------------------
template <typename MapT>
__global__ void __launch_bounds__(PK_PPC)
codemap_encode_kernel(const MapT* __restrict__ map, int64_t map_cols, int64_t grid_cols, int64_t P, int th,
                      int tw, int stride, int ppc, int K, int S, const __grid_constant__ PackTable tab,
                      uint8_t* __restrict__ slots, int64_t slot_bytes, uint32_t* __restrict__ sizes) {
    extern __shared__ uint32_t smem[];
    uint32_t* fc = smem;                                     // [K]
    uint16_t* buf = reinterpret_cast<uint16_t*>(fc + K);     // [ppc][stride]
    __shared__ uint32_t st_state[PK_PPC];
    __shared__ int st_words[PK_PPC];
    const int tid = threadIdx.x, n = th * tw;
    const int64_t p0 = (int64_t)blockIdx.x * ppc;
    const int np = (int)min((int64_t)ppc, P - p0);

    for (int s = tid; s < K; s += blockDim.x) fc[s] = tab.fc[s];

    for (int j = 0; j < np; ++j) {                          // stage: coalesced along tile rows
        const int64_t p = p0 + j, pr = p / grid_cols, pc = p - pr * grid_cols;
        const MapT* base = map + pr * th * map_cols + pc * tw;
        for (int e = tid; e < n; e += blockDim.x) {
            const int y = e / tw, x = e - y * tw;
            const uint32_t b = code_bin(__ldg(base + (int64_t)y * map_cols + x), K);
            buf[j * stride + e] = b < (uint32_t)K ? (uint16_t)b : PK_BAD;
        }
    }
    __syncthreads();

    if (tid < np) {
        uint16_t* t = buf + tid * stride;
        uint32_t x = PK_L;
        int w = 0;
        bool bad = false;
        for (int i = n - 1; i >= 0; --i) {
            const uint16_t s = t[i];
            uint32_t f = 0, c = 0;
            if (s != PK_BAD) {
                const uint32_t e = fc[s];
                f = e & 0xffffu;
                c = e >> 16;
            }
            if (f == 0) {                                   // not encodable: keep the state valid
                bad = true;
                f = 1u << S;
                c = 0;
            }
            if ((uint64_t)x >= ((uint64_t)f << (32 - S))) {
                t[n - 1 - w] = (uint16_t)(x & 0xffffu);     // position >= i: already read
                ++w;
                x >>= 16;
            }
            x = ((x / f) << S) + x % f + c;
        }
        st_state[tid] = x;
        st_words[tid] = w;
        sizes[p0 + tid] = bad ? 0u : 4u + 2u * (uint32_t)w;
    }
    __syncthreads();

    for (int j = 0; j < np; ++j) {                          // stream -> slot, coalesced
        uint16_t* slot = reinterpret_cast<uint16_t*>(slots + (p0 + j) * slot_bytes);
        const int w = st_words[j];
        const uint16_t* words = buf + j * stride + (n - w);
        for (int k = tid; k < w + 2; k += blockDim.x)
            slot[k] = k >= 2 ? words[k - 2] : (uint16_t)(k == 0 ? st_state[j] & 0xffffu : st_state[j] >> 16);
    }
}

// ---- exclusive scan of the stream sizes into the P + 1 payload offsets (one CTA, fixed order) ---------
__global__ void __launch_bounds__(PK_SCAN_THREADS)
codemap_offsets_kernel(const uint32_t* __restrict__ sizes, int64_t P, int64_t* __restrict__ offsets) {
    __shared__ int64_t warp_sum[PK_SCAN_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t per = (P + PK_SCAN_THREADS - 1) / PK_SCAN_THREADS;
    const int64_t lo = min(P, tid * per), hi = min(P, lo + per);
    int64_t mine = 0;
    for (int64_t i = lo; i < hi; ++i) mine += sizes[i];
    int64_t incl = mine;                                    // inclusive scan over the CTA
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int64_t v = warp_sum[lane], s = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t u = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += u;
        }
        warp_sum[lane] = s - v;                             // exclusive prefix of the warps
    }
    __syncthreads();
    int64_t run = warp_sum[warp] + incl - mine;
    if (tid == 0) offsets[0] = 0;
    for (int64_t i = lo; i < hi; ++i) {
        run += sizes[i];
        offsets[i + 1] = run;
    }
}

// ---- compaction: one warp per patch copies its stream from the slot to its offset ---------------------
__global__ void __launch_bounds__(256)
codemap_compact_kernel(const uint8_t* __restrict__ slots, int64_t slot_bytes, const int64_t* __restrict__ offsets,
                       int64_t P, uint8_t* __restrict__ payload, int64_t capacity) {
    const int64_t p = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (p >= P) return;
    const int lane = threadIdx.x & 31;
    const int64_t off = offsets[p], len = min(offsets[p + 1] - off, slot_bytes);
    if (off < 0 || (off & 1)) return;                       // sizes are even: never taken
    const uint16_t* src = reinterpret_cast<const uint16_t*>(slots + p * slot_bytes);
    uint16_t* dst = reinterpret_cast<uint16_t*>(payload + off);
    for (int64_t k = lane; 2 * k + 1 < len; k += 32)
        if (off + 2 * k + 1 < capacity) dst[k] = src[k];
}

// ---- decoder: one thread per patch of the region, PK_PPC patches per CTA ------------------------------
template <typename OutT>
__global__ void __launch_bounds__(PK_PPC)
codemap_decode_kernel(const uint8_t* __restrict__ payload, int64_t payload_bytes,
                      const int64_t* __restrict__ offsets, int64_t grid_cols, int th, int tw, int stride, int ppc,
                      int K, int S, const __grid_constant__ PackTable tab, int64_t r0, int64_t c0, int64_t nr,
                      int64_t nc, OutT* __restrict__ out, uint8_t* __restrict__ flags) {
    extern __shared__ uint32_t smem[];
    uint32_t* fc = smem;                                     // [K]
    uint16_t* sym = reinterpret_cast<uint16_t*>(fc + K);     // [2^S]
    uint16_t* buf = sym + (1 << S);                          // [ppc][stride]
    __shared__ int64_t st_start[PK_PPC];
    __shared__ int st_len[PK_PPC], st_words[PK_PPC];
    const int tid = threadIdx.x, n = th * tw;
    const int M = 1 << S;
    const int64_t t0 = (int64_t)blockIdx.x * ppc, total = nr * nc;
    const int np = (int)min((int64_t)ppc, total - t0);

    for (int s = tid; s < K; s += blockDim.x) fc[s] = tab.fc[s];
    if (tid < np) {                                          // this thread's stream, clamped
        const int64_t t = t0 + tid, pr = r0 + t / nc, pc = c0 + t % nc, p = pr * grid_cols + pc;
        int64_t a = offsets[p], b = offsets[p + 1];
        a = min(max(a, (int64_t)0), payload_bytes);
        b = min(max(b, a), payload_bytes);
        const int64_t len = min(b - a, (int64_t)(4 + 2 * n) + 2);
        st_start[tid] = a;
        st_len[tid] = (int)len;
        st_words[tid] = (int)min(max((len - 4) / 2, (int64_t)0), (int64_t)n);
    }
    __syncthreads();
    // slot -> symbol: thread i fills slots [i M / T, (i + 1) M / T), walking the symbols from the last
    // one whose start is <= its first slot (absent symbols have f = 0 and share their successor's start)
    {
        const int per = (M + blockDim.x - 1) / blockDim.x;
        const int lo = min(M, tid * per), hi = min(M, lo + per);
        if (lo < hi) {
            int a = 0, b = K - 1;                            // largest s with c[s] <= lo
            while (a < b) {
                const int m = (a + b + 1) >> 1;
                if ((int)(fc[m] >> 16) <= lo) a = m; else b = m - 1;
            }
            int s = a;
            for (int slot = lo; slot < hi; ++slot) {
                while (s + 1 < K && (int)(fc[s + 1] >> 16) <= slot) ++s;
                sym[slot] = (uint16_t)s;
            }
        }
    }
    for (int j = 0; j < np; ++j) {                           // stage the words at [n - w, n)
        const uint8_t* src = payload + st_start[j];
        const int w = st_words[j];
        uint16_t* dst = buf + j * stride + (n - w);
        for (int k = tid; k < w; k += blockDim.x) {
            const int i = 4 + 2 * k;                         // i + 1 < len: w <= (len - 4) / 2
            dst[k] = (uint16_t)(__ldg(src + i) | (__ldg(src + i + 1) << 8));
        }
    }
    __syncthreads();

    if (tid < np) {
        const uint8_t* src = payload + st_start[tid];
        const int len = st_len[tid], w = st_words[tid];
        uint32_t x = 0;
        for (int i = 0; i < 4; ++i) x |= (i < len ? (uint32_t)__ldg(src + i) : 0u) << (8 * i);
        uint16_t* t = buf + tid * stride;
        const uint16_t* words = t + (n - w);
        int k = 0;
        for (int i = 0; i < n; ++i) {
            const uint32_t slot = x & (uint32_t)(M - 1);
            const uint16_t s = sym[slot];
            const uint32_t e = fc[s];
            x = (e & 0xffffu) * (x >> S) + slot - (e >> 16);
            if (x < PK_L) {
                const uint32_t v = k < w ? words[k] : 0u;
                ++k;
                x = (x << 16) | v;
            }
            t[i] = s;                                        // position < the first unread word
        }
        const bool bad_len = len < 4 || (len & 1) || len > 4 + 2 * n;
        flags[t0 + tid] = (uint8_t)((x != PK_L ? 1 : 0) | (k != w ? 2 : 0) | (bad_len ? 4 : 0));
    }
    __syncthreads();

    const int64_t out_cols = nc * tw;
    for (int j = 0; j < np; ++j) {                           // tile -> [nr th, nc tw], coalesced
        const int64_t t = t0 + j, pr = t / nc, pc = t - pr * nc;
        OutT* base = out + pr * th * out_cols + pc * tw;
        const uint16_t* src = buf + j * stride;
        for (int e = tid; e < n; e += blockDim.x) {
            const int y = e / tw, x = e - y * tw;
            base[(int64_t)y * out_cols + x] = (OutT)src[e];
        }
    }
}

inline int64_t slot_bytes_of(int n) { return ((int64_t)4 + 2 * (int64_t)n + 3) & ~(int64_t)3; }
inline size_t align256p(size_t v) { return (v + 255) & ~(size_t)255; }

// host-side table checks (VQAE_OK or the error) and the f | c << 16 table
int make_table(const uint32_t* freq_host, int K, int S, PackTable* tab) {
    if (!freq_host) return VQAE_ERR_BAD_ARG;
    if (K < 1 || K > PK_MAX_K || S < 1 || S > PK_MAX_S) return VQAE_ERR_UNSUPPORTED;
    uint64_t c = 0;
    for (int s = 0; s < K; ++s) {
        if (freq_host[s] > (1u << S)) return VQAE_ERR_BAD_ARG;
        tab->fc[s] = freq_host[s] | (uint32_t)(c << 16);
        c += freq_host[s];
        if (c > (1u << S)) return VQAE_ERR_BAD_ARG;
    }
    for (int s = K; s < PK_MAX_K; ++s) tab->fc[s] = 0;
    return c == (1u << S) ? VQAE_OK : VQAE_ERR_BAD_ARG;
}

int check_grid(int64_t map_rows, int64_t map_cols, int th, int tw) {
    if (map_rows <= 0 || map_cols <= 0 || th <= 0 || tw <= 0) return VQAE_ERR_BAD_ARG;
    if (map_rows % th || map_cols % tw) return VQAE_ERR_BAD_ARG;
    if ((int64_t)th * tw > PK_MAX_CODES) return VQAE_ERR_UNSUPPORTED;
    if ((map_rows / th) * (map_cols / tw) > 0x7fffffff) return VQAE_ERR_UNSUPPORTED;
    return VQAE_OK;
}

int patches_per_cta(int n, size_t fixed) {
    const size_t per = (size_t)tile_stride(n) * sizeof(uint16_t);
    const size_t fit = (PK_SMEM_BUDGET - fixed) / per;
    return (int)(fit < (size_t)PK_PPC ? fit : PK_PPC);
}

template <typename K_>
int set_smem(K_ kern, size_t smem) {
    if (smem > 48 * 1024)
        VQAE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return VQAE_OK;
}

}  // namespace

int codemap_histogram(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int64_t r0,
                      int64_t c0, int64_t nr, int64_t nc, int K, int64_t* counts, cudaStream_t stream) {
    if (!map || !counts || map_rows <= 0 || map_cols <= 0 || nr <= 0 || nc <= 0 || r0 < 0 || c0 < 0)
        return VQAE_ERR_BAD_ARG;
    if (r0 + nr > map_rows || c0 + nc > map_cols) return VQAE_ERR_BAD_ARG;
    if (K < 1 || K > PK_MAX_K) return VQAE_ERR_UNSUPPORTED;
    int sm_count = 0;
    if (int rc = device_sm_count(&sm_count)) return rc;
    VQAE_CUDA_TRY(cudaMemsetAsync(counts, 0, (size_t)(K + 1) * sizeof(int64_t), stream));
    const int64_t cap = (int64_t)sm_count * 4;
    const unsigned grid = (unsigned)(nr < cap ? nr : cap);
    auto* cnt = reinterpret_cast<unsigned long long*>(counts);
    if (map_is_u8)
        codemap_histogram_kernel<uint8_t><<<grid, PK_HIST_THREADS, 0, stream>>>(
            static_cast<const uint8_t*>(map), map_cols, r0, c0, nr, nc, K, cnt);
    else
        codemap_histogram_kernel<int64_t><<<grid, PK_HIST_THREADS, 0, stream>>>(
            static_cast<const int64_t*>(map), map_cols, r0, c0, nr, nc, K, cnt);
    return check_launch();
}

size_t codemap_pack_scratch_bytes(int64_t n_patches, int th, int tw) {
    if (n_patches <= 0 || th <= 0 || tw <= 0 || (int64_t)th * tw > PK_MAX_CODES) return 0;
    return align256p((size_t)n_patches * slot_bytes_of(th * tw)) + align256p((size_t)n_patches * sizeof(uint32_t));
}

int64_t codemap_pack_worst_bytes(int64_t n_patches, int th, int tw) {
    if (n_patches <= 0 || th <= 0 || tw <= 0 || (int64_t)th * tw > PK_MAX_CODES) return 0;
    return n_patches * (4 + 2 * (int64_t)th * tw);
}

int codemap_pack(const void* map, int map_is_u8, int64_t map_rows, int64_t map_cols, int th, int tw,
                 const uint32_t* freq_host, int K, int S, int64_t* offsets, uint8_t* payload,
                 int64_t payload_capacity, void* scratch, size_t scratch_bytes, cudaStream_t stream) {
    if (!map || !offsets || !payload) return VQAE_ERR_BAD_ARG;
    if (int rc = check_grid(map_rows, map_cols, th, tw)) return rc;
    PackTable tab;
    if (int rc = make_table(freq_host, K, S, &tab)) return rc;
    const int64_t gc = map_cols / tw, P = (map_rows / th) * gc;
    if (payload_capacity < codemap_pack_worst_bytes(P, th, tw)) return VQAE_ERR_BAD_ARG;
    if (!scratch || scratch_bytes < codemap_pack_scratch_bytes(P, th, tw)) return VQAE_ERR_SCRATCH;

    const int n = th * tw, stride = tile_stride(n);
    const int64_t sb = slot_bytes_of(n);
    uint8_t* slots = static_cast<uint8_t*>(scratch);
    uint32_t* sizes = reinterpret_cast<uint32_t*>(slots + align256p((size_t)P * sb));
    const size_t fixed = (size_t)K * sizeof(uint32_t);
    const int ppc = patches_per_cta(n, fixed);
    const size_t smem = fixed + (size_t)ppc * stride * sizeof(uint16_t);
    const unsigned grid = ceil_div_u(P, ppc);
    if (map_is_u8) {
        if (int rc = set_smem(codemap_encode_kernel<uint8_t>, smem)) return rc;
        codemap_encode_kernel<uint8_t><<<grid, PK_PPC, smem, stream>>>(
            static_cast<const uint8_t*>(map), map_cols, gc, P, th, tw, stride, ppc, K, S, tab, slots, sb, sizes);
    } else {
        if (int rc = set_smem(codemap_encode_kernel<int64_t>, smem)) return rc;
        codemap_encode_kernel<int64_t><<<grid, PK_PPC, smem, stream>>>(
            static_cast<const int64_t*>(map), map_cols, gc, P, th, tw, stride, ppc, K, S, tab, slots, sb, sizes);
    }
    if (int rc = check_launch()) return rc;
    codemap_offsets_kernel<<<1, PK_SCAN_THREADS, 0, stream>>>(sizes, P, offsets);
    if (int rc = check_launch()) return rc;
    codemap_compact_kernel<<<ceil_div_u(P, 8), 256, 0, stream>>>(slots, sb, offsets, P, payload, payload_capacity);
    return check_launch();
}

int codemap_unpack(const uint8_t* payload, int64_t payload_bytes, const int64_t* offsets_host,
                   const int64_t* offsets, int64_t map_rows, int64_t map_cols, int th, int tw,
                   const uint32_t* freq_host, int K, int S, int64_t r0, int64_t c0, int64_t nr, int64_t nc,
                   void* out, int out_is_u8, uint8_t* flags, cudaStream_t stream) {
    if (!payload || !offsets_host || !offsets || !out || !flags) return VQAE_ERR_BAD_ARG;
    if (int rc = check_grid(map_rows, map_cols, th, tw)) return rc;
    const int64_t gr = map_rows / th, gc = map_cols / tw, P = gr * gc;
    if (r0 < 0 || c0 < 0 || nr <= 0 || nc <= 0 || r0 + nr > gr || c0 + nc > gc) return VQAE_ERR_BAD_ARG;
    PackTable tab;
    if (int rc = make_table(freq_host, K, S, &tab)) return rc;
    if (out_is_u8 && K > 256) return VQAE_ERR_UNSUPPORTED;
    const int n = th * tw;
    if (offsets_host[0] != 0 || offsets_host[P] != payload_bytes) return VQAE_ERR_BAD_ARG;
    for (int64_t p = 0; p < P; ++p) {
        const int64_t len = offsets_host[p + 1] - offsets_host[p];
        if (len < 4 || len > 4 + 2 * (int64_t)n || (len & 1)) return VQAE_ERR_BAD_ARG;
    }

    const int stride = tile_stride(n);
    const size_t fixed = (size_t)K * sizeof(uint32_t) + ((size_t)1 << S) * sizeof(uint16_t);
    const int ppc = patches_per_cta(n, fixed);
    const size_t smem = fixed + (size_t)ppc * stride * sizeof(uint16_t);
    const unsigned grid = ceil_div_u(nr * nc, ppc);
    if (out_is_u8) {
        if (int rc = set_smem(codemap_decode_kernel<uint8_t>, smem)) return rc;
        codemap_decode_kernel<uint8_t><<<grid, PK_PPC, smem, stream>>>(
            payload, payload_bytes, offsets, gc, th, tw, stride, ppc, K, S, tab, r0, c0, nr, nc,
            static_cast<uint8_t*>(out), flags);
    } else {
        if (int rc = set_smem(codemap_decode_kernel<int64_t>, smem)) return rc;
        codemap_decode_kernel<int64_t><<<grid, PK_PPC, smem, stream>>>(
            payload, payload_bytes, offsets, gc, th, tw, stride, ppc, K, S, tab, r0, c0, nr, nc,
            static_cast<int64_t*>(out), flags);
    }
    return check_launch();
}

}  // namespace vqae

// Device side of the deterministic synthetic-weight rule (see oracle/synth.py for the specification).
#pragma once
#include "common.cuh"
#include "row_map.cuh"

namespace fl {

constexpr uint64_t kGolden = 0x9E3779B97F4A7C15ULL;
constexpr uint32_t kSynthUnitBits = 0x37DDB3D7u;  // f32(1 / 37837.22719439421)

__host__ __device__ inline uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

inline uint64_t fnv1a64(const char* s) {
    uint64_t h = 0xCBF29CE484222325ULL;
    for (; *s; ++s) h = (h ^ (uint8_t)*s) * 0x100000001B3ULL;
    return h;
}

inline uint64_t tensor_seed(uint64_t seed, const char* name) { return mix64((seed * kGolden) ^ fnv1a64(name)); }

__device__ __forceinline__ uint16_t synth_bf16(uint64_t tseed, uint64_t i, float stdv) {
    uint64_t h = mix64(tseed + (i + 1) * kGolden);
    int s = (int)((h & 0xFFFF) + ((h >> 16) & 0xFFFF) + ((h >> 32) & 0xFFFF) + (h >> 48));
    float v = __fmul_rn(__fmul_rn((float)(s - 131070), __uint_as_float(kSynthUnitBits)), stdv);
    return f32_to_bf16_rne(v);
}

// The local [rows, cols] block is the window (src_row0.., src_col0..) of a full tensor with src_cols_full columns (tensor-
// parallel shards); element values depend only on the FULL-tensor index, so every shard layout sees the same weights.
struct SrcWin {
    int64_t row0, col0, cols_full;   // cols_full == 0: the block is the whole tensor
};
// Fills a [rows, cols] logical tensor into `dst`: logical row r lands at physical row map.map(r); element index = r * cols + c.
// `ld` = leading dimension of the destination matrix (== cols unless the local matrix carries zero-padded columns).
static __global__ void synth_fill_bf16_kernel(uint16_t* dst, int64_t rows, int64_t cols, int64_t ld, uint64_t tseed, float stdv, RowMap map,
                                              SrcWin win = SrcWin{0, 0, 0}) {
    int64_t n = rows * cols;
    const int64_t cf = win.cols_full ? win.cols_full : cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = i / cols, c = i - r * cols;
        dst[map.map(r) * ld + c] = synth_bf16(tseed, (uint64_t)((r + win.row0) * cf + c + win.col0), stdv);
    }
}

// f32 destination holding bf16-rounded values (biases, norm weights)
static __global__ void synth_fill_f32_kernel(float* dst, int64_t rows, uint64_t tseed, float stdv, RowMap map, int64_t src_row0 = 0) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x)
        dst[map.map(i)] = __uint_as_float((uint32_t)synth_bf16(tseed, (uint64_t)(i + src_row0), stdv) << 16);
}

static __global__ void fill_f32_kernel(float* dst, int64_t n, float v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = v;
}

}  // namespace fl

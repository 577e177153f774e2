// Where the rows of an uploaded or synthesised tensor land in its destination matrix (shared by the tensor table and the
// synthetic-weight kernels).
#pragma once
#include <cstdint>

namespace fl {

// Logical row r of a [rows, cols] tensor lands at physical row dst_row0 + perm(r) of the destination.
struct RowMap {
    int64_t dst_row0;   // first physical row
    int32_t mode;       // 0 identity, 1 rope-pair permutation within heads of `head_dim` rows, 2 interleave (phys = 2*r + lane)
    int32_t head_dim;
    int32_t lane;       // for mode 2: 0 = gate rows (even), 1 = up rows (odd)
    __host__ __device__ int64_t map(int64_t r) const {
        if (mode == 1) {
            int64_t h = r / head_dim, i = r % head_dim;
            int64_t half = head_dim / 2;
            int64_t j = (i < half) ? 2 * i : 2 * (i - half) + 1;
            return dst_row0 + h * head_dim + j;
        }
        if (mode == 2) return dst_row0 + 2 * r + lane;
        return dst_row0 + r;
    }
};

}  // namespace fl

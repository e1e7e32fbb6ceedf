// What the row copy kernels of env_rows.cu need to know about a packed env row.  api.cu decides the layout
// (env_row_layout) and describes it as pieces; the kernels copy pieces and know no section.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pcgrl {

constexpr int ROW_MAX_PIECES = 16;

// `count` items of `item` bytes, back to back from byte `off` of the row.  Item i of env e is at
// base + i * item_stride + e * item.  `unit` (1 .. 16, a power of two) divides off, item, item_stride and base: the
// widest access that is aligned everywhere in the piece.
struct RowPiece {
    void* base;
    int64_t item_stride;
    int32_t off, item, count, unit;
};

struct RowCopy {
    RowPiece piece[ROW_MAX_PIECES];   // in row order
    uint8_t* rows;                    // [n_rows, row_bytes]
    const int32_t* env_idx;           // NULL: row j is env j
    int32_t* status;
    int64_t n_rows, n_envs;
    int32_t n_pieces, row_bytes;
    uint32_t signature;
};

cudaError_t launch_save_envs(const RowCopy& r, cudaStream_t s);
cudaError_t launch_load_envs(const RowCopy& r, cudaStream_t s);

}  // namespace pcgrl

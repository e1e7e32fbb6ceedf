// Packed env rows (pcgrl_save_envs / pcgrl_load_envs): one thread per 16-byte chunk of a row, as k_la_gather.
// The layout arrives as a list of pieces (env_rows.cuh) built by api.cu.
//   k_save_envs  shard -> rows.  Chunk 0 is the header.  A chunk inside one 16-byte aligned piece (the grid, the frozen
//                mask, the per-env targets, a cache row whose stride is a multiple of 16) is one 16-byte load and store;
//                any other chunk is zeroed first (padding) and its pieces copied at their own width.  An index outside
//                the shard writes a zero row, header included, and sets status bit 512.
//   k_load_envs  rows -> shard.  Every thread of row j checks the row's header before it writes anything, so a row
//                that does not match loads nothing; the thread of chunk 0 sets the status bit (1024, or 512 for an
//                index outside the shard).
#include "env_rows.cuh"

namespace pcgrl {

// One block per SM is the stated minimum: with the thread count alone ptxas capped k_load_envs at 32 registers and
// spilled; it needs 34.
constexpr int ROW_THREADS = 256;

__device__ __forceinline__ void copy_unit(int unit, void* dst, const void* src) {
    switch (unit) {
        case 16: *(uint4*)dst = *(const uint4*)src; break;
        case 8: *(uint2*)dst = *(const uint2*)src; break;
        case 4: *(uint32_t*)dst = *(const uint32_t*)src; break;
        case 2: *(uint16_t*)dst = *(const uint16_t*)src; break;
        default: *(uint8_t*)dst = *(const uint8_t*)src; break;
    }
}

// byte o of piece q of env e in the shard
__device__ __forceinline__ uint8_t* shard_at(const RowPiece& q, int64_t e, int o) {
    const int i = q.count > 1 ? o / q.item : 0;
    return (uint8_t*)q.base + i * q.item_stride + e * q.item + (o - i * q.item);
}

// Copies the bytes [lo, lo + 16) of env e's row between `row` and the shard (SAVE: shard -> row, padding as zeros).
template <bool SAVE>
__device__ __forceinline__ void copy_chunk(const RowCopy& r, int64_t e, uint8_t* row, int lo) {
    const int hi = lo + 16;
    bool zeroed = !SAVE;
    for (int k = 0; k < r.n_pieces; ++k) {
        const RowPiece& q = r.piece[k];
        const int end = q.off + q.count * q.item;
        if (end <= lo) continue;
        if (q.off >= hi) break;
        if (q.unit == 16 && q.off <= lo && end >= hi) {   // the whole chunk, one 16-byte access each way
            uint8_t* s = shard_at(q, e, lo - q.off);
            if (SAVE) *(uint4*)(row + lo) = *(const uint4*)s;
            else *(uint4*)s = *(const uint4*)(row + lo);
            return;
        }
        if (!zeroed) {   // padding between the pieces of this chunk: zeros
            *(uint4*)(row + lo) = make_uint4(0, 0, 0, 0);
            zeroed = true;
        }
        const int a = lo > q.off ? lo : q.off, b = hi < end ? hi : end;
        for (int x = a; x < b; x += q.unit) {
            uint8_t* s = shard_at(q, e, x - q.off);
            if (SAVE) copy_unit(q.unit, row + x, s);
            else copy_unit(q.unit, s, row + x);
        }
    }
    if (!zeroed) *(uint4*)(row + lo) = make_uint4(0, 0, 0, 0);
}

__global__ void __launch_bounds__(ROW_THREADS, 1) k_save_envs(const RowCopy r) {
    const int chunks = r.row_bytes / 16;
    const int64_t i = (int64_t)blockIdx.x * ROW_THREADS + threadIdx.x;
    const int64_t j = i / chunks;
    const int c = (int)(i - j * chunks);
    if (j >= r.n_rows) return;
    const int64_t e = r.env_idx ? (int64_t)r.env_idx[j] : j;
    uint8_t* row = r.rows + j * r.row_bytes;
    if ((uint64_t)e >= (uint64_t)r.n_envs) {   // loads nothing; a zero header never matches
        ((uint4*)row)[c] = make_uint4(0, 0, 0, 0);
        if (c == 0 && r.status) atomicOr(r.status, 512);
        return;
    }
    if (c == 0) {
        ((uint4*)row)[0] = make_uint4(r.signature, (unsigned)r.row_bytes, 0, 0);
        return;
    }
    copy_chunk<true>(r, e, row, 16 * c);
}

__global__ void __launch_bounds__(ROW_THREADS, 1) k_load_envs(const RowCopy r) {
    const int chunks = r.row_bytes / 16;
    const int64_t i = (int64_t)blockIdx.x * ROW_THREADS + threadIdx.x;
    const int64_t j = i / chunks;
    const int c = (int)(i - j * chunks);
    if (j >= r.n_rows) return;
    const int64_t e = r.env_idx ? (int64_t)r.env_idx[j] : j;
    uint8_t* row = r.rows + j * r.row_bytes;
    const uint2 h = *(const uint2*)row;
    const int bad = ((uint64_t)e >= (uint64_t)r.n_envs ? 512 : 0) |
                    (h.x != r.signature || h.y != (unsigned)r.row_bytes ? 1024 : 0);
    if (bad) {
        if (c == 0 && r.status) atomicOr(r.status, bad);
        return;
    }
    if (c) copy_chunk<false>(r, e, row, 16 * c);
}

static unsigned row_blocks(const RowCopy& r) {
    return (unsigned)((r.n_rows * (r.row_bytes / 16) + ROW_THREADS - 1) / ROW_THREADS);
}

cudaError_t launch_save_envs(const RowCopy& r, cudaStream_t s) {
    k_save_envs<<<row_blocks(r), ROW_THREADS, 0, s>>>(r);
    return cudaGetLastError();
}

cudaError_t launch_load_envs(const RowCopy& r, cudaStream_t s) {
    k_load_envs<<<row_blocks(r), ROW_THREADS, 0, s>>>(r);
    return cudaGetLastError();
}

}  // namespace pcgrl

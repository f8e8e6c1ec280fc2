// kmap.cu -- coordinate hash table and kernel maps of the stride-1 K=5 submanifold conv.
//
// Replaces torchsparse 2.1.0's hash-map kernel-map build (selected by kmap_mode="hashmap",
// src/gs_compress/HAC/utils/pcc_utils.py:50-52) for spnn.Conv3d(32,32,5)
// (src/ai_pcc/GausPcgc/network_ue_4stage_conv.py:18-61).  The reference rebuilds the map for every
// fresh SparseTensor (pcc_utils.py:100,108,124,132,140); here it is built ONCE per coordinate set and
// shared by all convs on that set.
//
// Table: open addressing, linear probing, 16-byte slots {u64 block key, u32 base row, u32 mask} (one slot per x-block
// of 8 voxels) so a probe is one 128-bit load; capacity = power of two >= 2n (32 MB for a 1M-row level: L2 resident).
// Dense map is OFFSET-MAJOR [125][n] (coalesced over rows); offset index x-fastest
// k = ((dz+2)*5 + (dy+2))*5 + (dx+2).  The conv consumes per-tile pair lists grouped by offset.
#include "common.cuh"

// One slot describes an x-BLOCK of 8 voxels: key = voxel key >> 3 (= z, y, x>>3), `row` = row of the block's first
// voxel, `mask` = which of the 8 x positions are occupied.  Rows are sorted with x fastest, so a block's voxels are
// consecutive rows and row(x) = base + popcount(mask below x).  One 16-byte probe answers 8 positions: the 5 x-offsets
// of a (dz,dy) line fall into at most 2 blocks -> ~37 probes per row instead of 124.
struct __align__(16) HashSlot { u64 key; u32 row; u32 mask; };

__device__ __forceinline__ u32 hash_key(u64 k) {      // murmur3 fmix64
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return (u32)k;
}

extern "C" int64_t gpc_hash_capacity(int64_t n) {
    i64 cap = 1024;
    while (cap < 2 * n) cap <<= 1;
    return cap;
}

// keys sorted ascending, unique.  The first row of every x-block inserts the block.
__global__ void hash_insert_kernel(const u64 *__restrict__ keys, i64 n, HashSlot *table, u32 mask) {
    i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 key = keys[i];
    const u64 bk = key >> 3;
    if (i > 0 && (keys[i - 1] >> 3) == bk) return;
    u32 m = 1u << (u32)(key & 7);
    for (i64 j = i + 1; j < n && j < i + 8; ++j) {
        const u64 kj = keys[j];
        if ((kj >> 3) != bk) break;
        m |= 1u << (u32)(kj & 7);
    }
    u32 slot = hash_key(bk) & mask;
    while (true) {
        unsigned long long prev = atomicCAS((unsigned long long *)&table[slot].key, (unsigned long long)GPC_EMPTY_KEY,
                                            (unsigned long long)bk);
        if (prev == GPC_EMPTY_KEY || prev == bk) { table[slot].row = (u32)i; table[slot].mask = m; return; }
        slot = (slot + 1) & mask;
    }
}

// -> (base row, occupancy mask) of block bk, or mask 0 when absent
__device__ __forceinline__ uint2 hash_find_block(const HashSlot *__restrict__ table, u32 mask, u64 bk) {
    u32 slot = hash_key(bk) & mask;
    while (true) {
        const uint4 raw = __ldg((const uint4 *)&table[slot]);
        const u64 k = ((u64)raw.y << 32) | raw.x;
        if (k == bk) return make_uint2(raw.z, raw.w);
        if (k == GPC_EMPTY_KEY) return make_uint2(0u, 0u);
        slot = (slot + 1) & mask;
    }
}
__device__ __forceinline__ i32 block_row(uint2 b, u32 bit) {
    return ((b.y >> bit) & 1u) ? (i32)(b.x + __popc(b.y & ((1u << bit) - 1u))) : -1;
}
__device__ __forceinline__ i32 hash_find(const HashSlot *__restrict__ table, u32 mask, u64 key) {
    return block_row(hash_find_block(table, mask, key >> 3), (u32)(key & 7));
}

extern "C" int gpc_hash_build(const uint64_t *keys, int64_t n, void *table, int64_t capacity, void *stream) {
    cudaStream_t st = as_stream(stream);
    GPC_REQUIRE(capacity >= 2 * n && (capacity & (capacity - 1)) == 0, GPC_EINVAL, "capacity must be a power of two >= 2n");
    GPC_CUDA_CHECK(cudaMemsetAsync(table, 0xFF, (size_t)capacity * sizeof(HashSlot), st));
    if (n <= 0) return GPC_OK;
    hash_insert_kernel<<<cdiv(n, 256), 256, 0, st>>>(keys, n, (HashSlot *)table, (u32)(capacity - 1));
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

__global__ void hash_lookup_kernel(const HashSlot *__restrict__ table, u32 mask, const u64 *__restrict__ q, i64 n,
                                   i32 *__restrict__ rows) {
    i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rows[i] = hash_find(table, mask, q[i]);
}
extern "C" int gpc_hash_lookup(const void *table, int64_t capacity, const uint64_t *query, int64_t n, int32_t *rows,
                               void *stream) {
    if (n <= 0) return GPC_OK;
    hash_lookup_kernel<<<cdiv(n, 256), 256, 0, as_stream(stream)>>>((const HashSlot *)table, (u32)(capacity - 1), query, n, rows);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// one thread per (row o, line (dz,dy)); blockIdx.y = line, so every one of the 5 output planes is written coalesced.
// half = kernel_size / 2: offsets with a component beyond it are absent (-1) without a probe -- a K = 3 conv
// (compress_ue_4stage_conv.py:44) runs on the K = 5 machinery with its 27 offsets at their K = 5 indices.
// cell_counts (optional): number of present neighbours per (tile of tile_rows rows, offset), [tiles][126] -- the first pass of the
// tcgen05 conv's pair stream and the level's density fall out of the probes instead of a second read of the 500 B-per-row map.
__global__ void __launch_bounds__(256) kmap_dense_kernel(const HashSlot *__restrict__ table, u32 mask, const u64 *__restrict__ keys,
                                                        i64 n, i32 *__restrict__ map, int half, int tile_rows,
                                                        u32 *__restrict__ cell_counts) {
    __shared__ u32 cnt[2][5];                          // a block of 256 rows touches at most two tiles (tile_rows >= 256)
    const int line = blockIdx.y;                      // (dz+2)*5 + (dy+2)
    const i64 b0row = (i64)blockIdx.x * blockDim.x;
    const i64 o = b0row + threadIdx.x;
    if (cell_counts) {
        if (threadIdx.x < 10) cnt[threadIdx.x / 5][threadIdx.x % 5] = 0;
        __syncthreads();
    }
    const int dy = line % 5 - 2, dz = line / 5 - 2;
    i32 r[5] = {-1, -1, -1, -1, -1};
    if (o < n && abs(dy) <= half && abs(dz) <= half) {
        // fields never under/overflow: |c| <= 2^20 - 16
        const u64 k0 = (u64)((i64)keys[o] + ((i64)dy << 21) + ((i64)dz << 42) - 2);       // voxel at dx = -2
        const u64 b0 = k0 >> 3, b1 = (k0 + 4) >> 3;
        const uint2 e0 = hash_find_block(table, mask, b0);
        const uint2 e1 = b1 != b0 ? hash_find_block(table, mask, b1) : e0;
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) {
            const u64 kk = k0 + dx;
            const i32 v = block_row((kk >> 3) == b0 ? e0 : e1, (u32)(kk & 7));
            r[dx] = abs(dx - 2) > half ? -1 : v;
        }
    }
    if (o < n) {
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) map[(i64)(line * 5 + dx) * n + o] = r[dx];
    }
    if (cell_counts) {
        const i64 t0 = b0row / tile_rows;
        const int tw = (int)((b0row + (threadIdx.x & ~31)) / tile_rows - t0);              // the warp's 32 rows lie in one tile
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) {
            const u32 c = __popc(__ballot_sync(0xFFFFFFFFu, r[dx] >= 0));
            if ((threadIdx.x & 31) == 0 && c) atomicAdd(&cnt[tw][dx], c);
        }
        __syncthreads();
        if (threadIdx.x < 10) {
            const u32 c = cnt[threadIdx.x / 5][threadIdx.x % 5];
            if (c) atomicAdd(&cell_counts[(t0 + threadIdx.x / 5) * (GPC_K3 + 1) + line * 5 + threadIdx.x % 5], c);
        }
    }
}
extern "C" int gpc_kmap_dense(const void *table, int64_t capacity, const uint64_t *keys, int64_t n, int32_t *map,
                              int kernel_size, int tile_rows, uint32_t *cell_counts, void *stream) {
    if (n <= 0) return GPC_OK;
    GPC_REQUIRE(kernel_size == 3 || kernel_size == 5, GPC_EINVAL, "kernel_size must be 3 or 5");
    cudaStream_t st = as_stream(stream);
    if (cell_counts) {
        GPC_REQUIRE(tile_rows >= 256 && tile_rows % 32 == 0, GPC_EINVAL, "counting needs tile_rows >= 256, a multiple of 32");
        const i64 tiles = (n + tile_rows - 1) / tile_rows;
        GPC_CUDA_CHECK(cudaMemsetAsync(cell_counts, 0, (size_t)tiles * (GPC_K3 + 1) * 4, st));
    }
    dim3 grid(cdiv(n, 256), 25);
    kmap_dense_kernel<<<grid, 256, 0, st>>>((const HashSlot *)table, (u32)(capacity - 1), keys, n, map, kernel_size / 2,
                                            cell_counts ? tile_rows : 256, cell_counts);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// ---------------------------------------------------------------- per-tile pair lists grouped by offset
// counts[t*126 + k] = number of rows of tile t with a neighbour at offset k (k = 125 is a zero pad so
// that the exclusive scan leaves seg[t*126+125] == start of tile t+1).  pad > 1: every non-empty count is rounded up to a
// multiple of `pad` entries (8-pair MMA tiles of one offset).
__global__ void kmap_total_kernel(const u32 *__restrict__ seg, i64 m, u32 *__restrict__ n_pairs) { *n_pairs = seg[m]; }

// ---- warp-per-tile kernels (tile_rows = 32 * RPL, RPL = 1, 2, 4): no block barriers, each warp streams its tile's
// 125 x tile_rows slice of the dense map with coalesced loads and ballots.
template <int RPL>
__global__ void __launch_bounds__(128) kmap_pairs_count_warp_kernel(const i32 *__restrict__ map, i64 n, i64 ld, i64 tiles, int pad,
                                                                   u32 *__restrict__ counts, u32 *__restrict__ n_real) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const i64 t = blockIdx.x;                       // one CTA per tile, warp w takes offsets w, w + 4, ... ((tile, offset) cells are independent)
    const i64 r0 = t * (32 * RPL);
    u32 real = 0;
#pragma unroll 4
    for (int k = wid; k < GPC_K3; k += 4) {
        u32 c = 0;
#pragma unroll
        for (int i = 0; i < RPL; ++i) {
            const i64 r = r0 + i * 32 + lane;
            const bool v = r < n && map[(i64)k * ld + r] >= 0;
            c += __popc(__ballot_sync(0xFFFFFFFFu, v));
        }
        real += c;
        c = (c + pad - 1) / pad * pad;
        if (lane == 0) counts[t * (GPC_K3 + 1) + k] = c;
    }
    if (lane == 0) { if (wid == 0) counts[t * (GPC_K3 + 1) + GPC_K3] = 0; atomicAdd(n_real, real); }
}

template <int RPL>
__global__ void __launch_bounds__(128) kmap_pairs_fill_warp_kernel(const i32 *__restrict__ map, i64 n, i64 ld, i64 tiles,
                                                                  const u32 *__restrict__ seg, u32 *__restrict__ pair_nbr,
                                                                  u16 *__restrict__ pair_row, u64 *__restrict__ pairs) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const i64 t = blockIdx.x;
    const i64 r0 = t * (32 * RPL);
    const u32 lt = (1u << lane) - 1u;
    const i64 left = n - r0 - lane;                 // rows of this tile at or after this lane's first row
#pragma unroll 4
    for (int k = wid; k < GPC_K3; k += 4) {
        u32 p = seg[t * (GPC_K3 + 1) + k];
        const i32 *mk = map + (i64)k * ld + r0 + lane;
#pragma unroll
        for (int i = 0; i < RPL; ++i) {
            const i32 nb = i * 32 < left ? mk[i * 32] : -1;
            const u32 bal = __ballot_sync(0xFFFFFFFFu, nb >= 0);
            if (nb >= 0) {
                const u32 q = p + __popc(bal & lt);
                if (pair_nbr) { pair_nbr[q] = (u32)nb; pair_row[q] = (u16)(i * 32 + lane); }
                if (pairs) pairs[q] = (u64)(u32)nb | ((u64)(u32)(i * 32 + lane) << 32) | ((u64)(u32)k << 48);
            }
            p += __popc(bal);
        }
    }
}

// ---- sub-warp tiles (tile_rows = 8 or 16): one warp covers 32 / TW tiles, each group of TW lanes is one tile.
// Small tiles give the conv enough warps on the coarse octree levels (a few hundred to a few ten-thousand rows).
template <int TW>
__global__ void __launch_bounds__(128) kmap_pairs_count_sub_kernel(const i32 *__restrict__ map, i64 n, i64 ld, i64 tiles, int pad,
                                                                  u32 *__restrict__ counts, u32 *__restrict__ n_real) {
    constexpr int SUB = 32 / TW;
    const int lane = threadIdx.x & 31, sub = lane / TW, rl = lane % TW;
    const i64 t = ((i64)blockIdx.x * 4 + (threadIdx.x >> 5)) * SUB + sub;
    const i64 r = t * TW + rl;
    const bool live = t < tiles;
    u32 real = 0;
#pragma unroll 5
    for (int k = 0; k < GPC_K3; ++k) {
        const bool v = live && r < n && map[(i64)k * ld + r] >= 0;
        const u32 bits = (__ballot_sync(0xFFFFFFFFu, v) >> (TW * sub)) & ((1u << TW) - 1u);
        const u32 c = __popc(bits);
        real += c;
        if (live && rl == 0) counts[t * (GPC_K3 + 1) + k] = (c + pad - 1) / pad * pad;
    }
    if (live && rl == 0) { counts[t * (GPC_K3 + 1) + GPC_K3] = 0; atomicAdd(n_real, real); }
}
template <int TW>
__global__ void __launch_bounds__(128) kmap_pairs_fill_sub_kernel(const i32 *__restrict__ map, i64 n, i64 ld, i64 tiles,
                                                                 const u32 *__restrict__ seg, u32 *__restrict__ pair_nbr,
                                                                 u16 *__restrict__ pair_row, u64 *__restrict__ pairs) {
    constexpr int SUB = 32 / TW;
    const int lane = threadIdx.x & 31, sub = lane / TW, rl = lane % TW;
    const i64 t = ((i64)blockIdx.x * 4 + (threadIdx.x >> 5)) * SUB + sub;
    const i64 r = t * TW + rl;
    const bool live = t < tiles;
#pragma unroll 5
    for (int k = 0; k < GPC_K3; ++k) {
        const i32 nb = (live && r < n) ? map[(i64)k * ld + r] : -1;
        const u32 bits = (__ballot_sync(0xFFFFFFFFu, nb >= 0) >> (TW * sub)) & ((1u << TW) - 1u);
        if (nb >= 0) {
            const u32 q = seg[t * (GPC_K3 + 1) + k] + __popc(bits & ((1u << rl) - 1u));
            if (pair_nbr) { pair_nbr[q] = (u32)nb; pair_row[q] = (u16)rl; }
            if (pairs) pairs[q] = (u64)(u32)nb | ((u64)(u32)rl << 32) | ((u64)(u32)k << 48);
        }
    }
}

extern "C" size_t gpc_kmap_pairs_workspace_bytes(int64_t n, int tile_rows) {
    const i64 tiles = n > 0 ? (n + tile_rows - 1) / tile_rows : 1;
    const i64 m = tiles * (GPC_K3 + 1);
    return align_up((size_t)m * 4, 256) + align_up(scan_workspace_bytes<u32>(m), 256) + 1024;
}
// map: the rows [0, n) of a dense map whose offset planes are ld >= n ints apart (ld = n: a whole level; ld > n: a row range of a
// level, map already advanced to its first row -- gpc_kmap_pairs_count_range)
static int pairs_count(const int32_t *map, int64_t n, int64_t ld, int tile_rows, int pad, uint32_t *seg, uint32_t *n_pairs, void *ws,
                       size_t ws_bytes, void *stream) {
    cudaStream_t st = as_stream(stream);
    GPC_REQUIRE((tile_rows == 8 || tile_rows == 16 || tile_rows == 32 || tile_rows == 64 || tile_rows == 128) && pad >= 1, GPC_EINVAL,
                "tile_rows must be 8, 16, 32, 64 or 128, pad >= 1");
    if (n <= 0) { GPC_CUDA_CHECK(cudaMemsetAsync(n_pairs, 0, 8, st)); return GPC_OK; }
    GPC_REQUIRE(ws && ws_bytes >= gpc_kmap_pairs_workspace_bytes(n, tile_rows), GPC_ENOSPC, "workspace too small");
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    const i64 m = tiles * (GPC_K3 + 1);
    u32 *counts = (u32 *)ws;
    void *scan_ws = (char *)ws + align_up((size_t)m * 4, 256);
    GPC_CUDA_CHECK(cudaMemsetAsync(n_pairs, 0, 8, st));      // n_pairs[0] = stream entries (padded), n_pairs[1] = true pairs
    if (tile_rows == 8) kmap_pairs_count_sub_kernel<8><<<cdiv(tiles, 16), 128, 0, st>>>(map, n, ld, tiles, pad, counts, n_pairs + 1);
    else if (tile_rows == 16) kmap_pairs_count_sub_kernel<16><<<cdiv(tiles, 8), 128, 0, st>>>(map, n, ld, tiles, pad, counts, n_pairs + 1);
    else if (tile_rows == 32) kmap_pairs_count_warp_kernel<1><<<(unsigned)tiles, 128, 0, st>>>(map, n, ld, tiles, pad, counts, n_pairs + 1);
    else if (tile_rows == 64) kmap_pairs_count_warp_kernel<2><<<(unsigned)tiles, 128, 0, st>>>(map, n, ld, tiles, pad, counts, n_pairs + 1);
    else kmap_pairs_count_warp_kernel<4><<<(unsigned)tiles, 128, 0, st>>>(map, n, ld, tiles, pad, counts, n_pairs + 1);
    GPC_LAUNCH_CHECK();
    PtrLoad<u32> pl{counts};
    int rc = device_exclusive_scan<u32, PtrLoad<u32>>(pl, m, seg, scan_ws, st);      // seg has m+1 entries
    if (rc) return rc;
    kmap_total_kernel<<<1, 1, 0, st>>>(seg, m, n_pairs);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}
static int pairs_fill(const int32_t *map, int64_t n, int64_t ld, int tile_rows, const uint32_t *seg, uint32_t *pair_nbr,
                      uint16_t *pair_row, uint64_t *pairs, int64_t n_entries, void *stream) {
    if (n <= 0) return GPC_OK;
    GPC_REQUIRE(tile_rows == 8 || tile_rows == 16 || tile_rows == 32 || tile_rows == 64 || tile_rows == 128, GPC_EINVAL,
                "tile_rows must be 8, 16, 32, 64 or 128");
    // padded streams: entries not written below stay INVALID (all ones)
    if (pairs && n_entries > 0) GPC_CUDA_CHECK(cudaMemsetAsync(pairs, 0xFF, (size_t)n_entries * 8, as_stream(stream)));
    if (pair_nbr && n_entries > 0) {               // split arrays: padding = row 0xFFFFFFFF (out of bounds for the TMA gather: zero fill) / 0xFFFF
        GPC_CUDA_CHECK(cudaMemsetAsync(pair_nbr, 0xFF, (size_t)n_entries * 4, as_stream(stream)));
        GPC_CUDA_CHECK(cudaMemsetAsync(pair_row, 0xFF, (size_t)n_entries * 2, as_stream(stream)));
    }
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    cudaStream_t st = as_stream(stream);
    if (tile_rows == 8) kmap_pairs_fill_sub_kernel<8><<<cdiv(tiles, 16), 128, 0, st>>>(map, n, ld, tiles, seg, pair_nbr, pair_row, pairs);
    else if (tile_rows == 16) kmap_pairs_fill_sub_kernel<16><<<cdiv(tiles, 8), 128, 0, st>>>(map, n, ld, tiles, seg, pair_nbr, pair_row, pairs);
    else if (tile_rows == 32) kmap_pairs_fill_warp_kernel<1><<<(unsigned)tiles, 128, 0, st>>>(map, n, ld, tiles, seg, pair_nbr, pair_row, pairs);
    else if (tile_rows == 64) kmap_pairs_fill_warp_kernel<2><<<(unsigned)tiles, 128, 0, st>>>(map, n, ld, tiles, seg, pair_nbr, pair_row, pairs);
    else kmap_pairs_fill_warp_kernel<4><<<(unsigned)tiles, 128, 0, st>>>(map, n, ld, tiles, seg, pair_nbr, pair_row, pairs);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}
extern "C" int gpc_kmap_pairs_count(const int32_t *map, int64_t n, int tile_rows, int pad, uint32_t *seg, uint32_t *n_pairs,
                                    void *ws, size_t ws_bytes, void *stream) {
    return pairs_count(map, n, n, tile_rows, pad, seg, n_pairs, ws, ws_bytes, stream);
}
extern "C" int gpc_kmap_pairs_fill(const int32_t *map, int64_t n, int tile_rows, const uint32_t *seg, uint32_t *pair_nbr,
                                   uint16_t *pair_row, uint64_t *pairs, int64_t n_entries, void *stream) {
    return pairs_fill(map, n, n, tile_rows, seg, pair_nbr, pair_row, pairs, n_entries, stream);
}
// row ranges [row0, row1) of a level of n_level rows (a batch of scenes coded as one union level): tiles start at row0, neighbour
// indices stay the level's rows, and the totals are the range's own (entries, true pairs)
extern "C" int gpc_kmap_pairs_count_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows, int pad,
                                          uint32_t *seg, uint32_t *n_pairs, void *ws, size_t ws_bytes, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    return pairs_count(map + row0, row1 - row0, n_level, tile_rows, pad, seg, n_pairs, ws, ws_bytes, stream);
}
extern "C" int gpc_kmap_pairs_fill_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows,
                                         const uint32_t *seg, uint64_t *pairs, int64_t n_entries, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    return pairs_fill(map + row0, row1 - row0, n_level, tile_rows, seg, nullptr, nullptr, pairs, n_entries, stream);
}

// ---------------------------------------------------------------- pair stream of the tcgen05 conv (spconv_um.cu)
// Tiles of 256 .. 1024 output rows; one WARP per (tile, offset) cell: the cell's slice of the offset-major dense map is tile_rows
// consecutive ints, read with coalesced loads and ranked with ballots.  Every non-empty cell is padded to a multiple of 16 entries; the stream holds,
// per entry, the input row (padding: 0xFFFFFFFF = out of bounds for the gather) and the BYTE OFFSET of the pair's accumulator row
// inside the tile (row * 128; padding: the dummy row tile_rows * 128).
__global__ void __launch_bounds__(128) kmap_um_count_kernel(const i32 *__restrict__ map, i64 n, i64 ld, int tile_rows, i64 cells,
                                                           u32 *__restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const i64 cell = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);           // = tile * 126 + k; k == 125 is the zero pad of the scan
    if (cell >= cells) return;
    const i64 t = cell / (GPC_K3 + 1);
    const int k = (int)(cell - t * (GPC_K3 + 1));
    u32 c = 0;
    if (k < GPC_K3) {
        const i64 r0 = t * tile_rows;
        const int rows = (int)min((i64)tile_rows, n - r0);
        const i32 *m = map + (i64)k * ld + r0;
        for (int r = lane; r < rows; r += 32) c += m[r] >= 0;
        c = __reduce_add_sync(0xFFFFFFFFu, c);
    }
    if (lane == 0) counts[cell] = c;
}
// true pairs of the level = sum of the raw cell counts
__global__ void __launch_bounds__(256) kmap_um_total_kernel(const u32 *__restrict__ counts, i64 cells, unsigned long long *n_real) {
    __shared__ unsigned long long part[8];
    unsigned long long s = 0;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < cells; i += (i64)gridDim.x * 256) s += counts[i];
#pragma unroll
    for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, d);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) s += part[w];
        if (s) atomicAdd(n_real, s);
    }
}
struct Pad16Load {                                                       // every non-empty cell padded to a multiple of 16 entries
    const u32 *p;
    __device__ u32 operator()(i64 i) const { return (p[i] + 15u) & ~15u; }
};
__global__ void __launch_bounds__(128) kmap_um_fill_kernel(const i32 *__restrict__ map, i64 n, i64 ld, int tile_rows, i64 cells,
                                                          const u32 *__restrict__ seg, u32 *__restrict__ pair_nbr, u32 *__restrict__ pair_off) {
    const int lane = threadIdx.x & 31;
    const i64 cell = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (cell >= cells) return;
    const i64 t = cell / (GPC_K3 + 1);
    const int k = (int)(cell - t * (GPC_K3 + 1));
    if (k >= GPC_K3) return;
    u32 p = seg[cell];
    const u32 end = seg[cell + 1];
    if (p == end) return;
    const i64 r0 = t * tile_rows;
    const int rows = (int)min((i64)tile_rows, n - r0);
    const i32 *m = map + (i64)k * ld + r0;
    const u32 lt = (1u << lane) - 1u;
    for (int rb = 0; rb < rows; rb += 32) {                               // ascending row order inside a cell
        const int r = rb + lane;
        const i32 nb = r < rows ? m[r] : -1;
        const u32 bal = __ballot_sync(0xFFFFFFFFu, nb >= 0);
        if (nb >= 0) {
            const u32 q = p + __popc(bal & lt);
            pair_nbr[q] = (u32)nb;
            pair_off[q] = (u32)r * 128u;
        }
        p += __popc(bal);
    }
    for (u32 q = p + lane; q < end; q += 32) {                            // padding
        pair_nbr[q] = 0xFFFFFFFFu;
        pair_off[q] = (u32)tile_rows * 128u;
    }
}
extern "C" size_t gpc_kmap_um_workspace_bytes(int64_t n, int tile_rows) { return gpc_kmap_pairs_workspace_bytes(n, tile_rows); }
// totals: device u64[2] = {stream entries (padded), true pairs}.  cell_counts: what gpc_kmap_dense counted with the same tile_rows.
extern "C" int gpc_kmap_um_scan(const uint32_t *cell_counts, int64_t n, int tile_rows, uint32_t *seg, unsigned long long *totals,
                                void *ws, size_t ws_bytes, void *stream) {
    cudaStream_t st = as_stream(stream);
    GPC_REQUIRE(tile_rows >= 32 && tile_rows <= 1024, GPC_EINVAL, "tile_rows must be in 32..1024");
    GPC_CUDA_CHECK(cudaMemsetAsync(totals, 0, 16, st));
    if (n <= 0) return GPC_OK;
    GPC_REQUIRE(ws && ws_bytes >= gpc_kmap_um_workspace_bytes(n, tile_rows), GPC_ENOSPC, "workspace too small");
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    const i64 m = tiles * (GPC_K3 + 1);
    void *scan_ws = (char *)ws + align_up((size_t)m * 4, 256);
    kmap_um_total_kernel<<<(unsigned)min((i64)296, (m + 255) / 256), 256, 0, st>>>(cell_counts, m, totals + 1);
    GPC_LAUNCH_CHECK();
    Pad16Load pl{cell_counts};
    int rc = device_exclusive_scan<u32, Pad16Load>(pl, m, seg, scan_ws, st);         // seg has m + 1 entries
    if (rc) return rc;
    GPC_CUDA_CHECK(cudaMemcpyAsync(totals, seg + m, 4, cudaMemcpyDeviceToDevice, st));
    return GPC_OK;
}
// the same from a dense map that was built without counting (any tile_rows in 32..1024; tools, tests).  ld as in pairs_count.
static int um_count(const int32_t *map, int64_t n, int64_t ld, int tile_rows, uint32_t *seg, unsigned long long *totals, void *ws,
                    size_t ws_bytes, void *stream) {
    cudaStream_t st = as_stream(stream);
    GPC_REQUIRE(tile_rows >= 32 && tile_rows <= 1024, GPC_EINVAL, "tile_rows must be in 32..1024");
    if (n <= 0) { GPC_CUDA_CHECK(cudaMemsetAsync(totals, 0, 16, st)); return GPC_OK; }
    GPC_REQUIRE(ws && ws_bytes >= gpc_kmap_um_workspace_bytes(n, tile_rows), GPC_ENOSPC, "workspace too small");
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    const i64 m = tiles * (GPC_K3 + 1);
    u32 *counts = (u32 *)ws;
    kmap_um_count_kernel<<<cdiv(m, 4), 128, 0, st>>>(map, n, ld, tile_rows, m, counts);
    GPC_LAUNCH_CHECK();
    return gpc_kmap_um_scan(counts, n, tile_rows, seg, totals, ws, ws_bytes, stream);
}
static int um_fill(const int32_t *map, int64_t n, int64_t ld, int tile_rows, const uint32_t *seg, uint32_t *pair_nbr,
                   uint32_t *pair_off, void *stream) {
    if (n <= 0) return GPC_OK;
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    const i64 m = tiles * (GPC_K3 + 1);
    kmap_um_fill_kernel<<<cdiv(m, 4), 128, 0, as_stream(stream)>>>(map, n, ld, tile_rows, m, seg, pair_nbr, pair_off);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}
extern "C" int gpc_kmap_um_count(const int32_t *map, int64_t n, int tile_rows, uint32_t *seg, unsigned long long *totals, void *ws,
                                 size_t ws_bytes, void *stream) {
    return um_count(map, n, n, tile_rows, seg, totals, ws, ws_bytes, stream);
}
extern "C" int gpc_kmap_um_fill(const int32_t *map, int64_t n, int tile_rows, const uint32_t *seg, uint32_t *pair_nbr,
                                uint32_t *pair_off, void *stream) {
    return um_fill(map, n, n, tile_rows, seg, pair_nbr, pair_off, stream);
}
extern "C" int gpc_kmap_um_count_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows, uint32_t *seg,
                                       unsigned long long *totals, void *ws, size_t ws_bytes, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    return um_count(map + row0, row1 - row0, n_level, tile_rows, seg, totals, ws, ws_bytes, stream);
}
extern "C" int gpc_kmap_um_fill_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows,
                                      const uint32_t *seg, uint32_t *pair_nbr, uint32_t *pair_off, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    return um_fill(map + row0, row1 - row0, n_level, tile_rows, seg, pair_nbr, pair_off, stream);
}

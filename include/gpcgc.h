/*
 * gpcgc.h -- C ABI of libgpcgc.so: the B200 (sm_100a) implementation of the GausPcgc
 * anchor-geometry codec hot path of Wangkkklll/GausPcc.
 *
 * Boundary replaced (reference file:line, relative to /root/reference):
 *   src/gs_compress/HAC/utils/pcc_utils.py:12-22    calculate_morton_order
 *   src/gs_compress/HAC/utils/pcc_utils.py:24-217   compress_point_cloud
 *   src/gs_compress/HAC/utils/pcc_utils.py:230-400  decompress_point_cloud
 * and, underneath them, the third-party calls those functions make
 *   torchsparse 2.1.0: SparseTensor / spnn.Conv3d / hash kernel maps
 *                      (kit/nn.py:14-16,31; network_ue_4stage_conv.py:18-61)
 *   torch:             sort x4 (kit/op.py:17-30), embedding / linear / softmax / cumsum
 *   torchac 0.9.3:     encode/decode_int16_normalized_cdf (pcc_utils.py:174-177,322-366)
 *
 * Conventions
 *   - every entry point is extern "C", returns 0 on success or a negative GPC_E* code;
 *     gpc_last_error() gives a thread-local message.
 *   - pointers are DEVICE pointers unless the name ends in _h (host).  No allocation happens
 *     inside the library: the caller provides outputs and workspaces (sizes from the
 *     *_workspace_bytes queries).  `stream` is a cudaStream_t passed as void*.
 *   - a voxel key is u64: (z+2^20)<<42 | (y+2^20)<<21 | (x+2^20); ascending key order is the
 *     reference's row order: lexicographic (z,y,x) = op.sort_CF = calculate_morton_order.
 *     Valid coordinates: |c| <= GPC_COORD_MAX.
 *   - feature rows are fp32 [n, 32] row-major (128 B per row), GPC_C == 32, K == 5 (K^3 == 125)
 *     as in the reference call sites (pcc_utils.py:28-29).
 */
#ifndef GPCGC_H
#define GPCGC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPC_C 32
#define GPC_K 5
#define GPC_K3 125
#define GPC_COORD_BIAS (1 << 20)
#define GPC_COORD_MAX ((1 << 20) - 16)

#define GPC_OK 0
#define GPC_EINVAL (-1)     /* bad argument */
#define GPC_ECUDA (-2)      /* CUDA runtime error (see gpc_last_error) */
#define GPC_ERANGE (-3)     /* coordinate outside +-GPC_COORD_MAX or not integral */
#define GPC_ENOSPC (-4)     /* workspace / output too small */
#define GPC_EDATA (-5)      /* corrupt bitstream / symbol out of range */

const char *gpc_last_error(void);
int gpc_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t gpc_launch_count(void);
/* cudaMemcpyAsync(cudaMemcpyDefault) on `stream`: device or pinned host pointers on either side */
int gpc_copy_async(void *dst, const void *src, int64_t bytes, void *stream);

/* key transform for sorting: compact = ((z-minz)<<sz) | ((y-miny)<<sy) | (x-minx) on the biased
 * 21-bit fields; digits of `compact` are what the radix sort consumes (fewer passes than 63 bits) */
typedef struct { uint32_t minx, miny, minz, sy, sz, total_bits; } gpc_key_xform;

/* ---- a-1/a-2: voxel keys and ordering (pcc_utils.py:12-22; HAC/scene/gaussian_model.py:1107) ---- */
/* xyz [n,3] row-major -> keys[n]; *status (device int32, caller-zeroed) gets bit0 set on a
 * non-integral value, bit1 on out-of-range. */
int gpc_pack_keys_f32(const float *xyz, int64_t n, uint64_t *keys, int32_t *status, void *stream);
int gpc_pack_keys_i32(const int32_t *xyz, int64_t n, uint64_t *keys, int32_t *status, void *stream);
int gpc_unpack_keys_i32(const uint64_t *keys, int64_t n, int32_t *xyz, void *stream);
int gpc_unpack_keys_f32(const uint64_t *keys, int64_t n, float scale, float *xyz, void *stream);
/* min/max of the three biased fields -> minmax[6] = {minx,miny,minz,maxx,maxy,maxz} (device u32) */
int gpc_key_minmax(const uint64_t *keys, int64_t n, uint32_t *minmax, void *stream);
/* host helper: builds the transform from minmax read back by the caller */
int gpc_make_xform_h(const uint32_t *minmax_h, gpc_key_xform *out_h);

size_t gpc_sort_workspace_bytes(int64_t n);
/* stable LSD radix sort of (key, val) by compact(key); vals_in == NULL means val = row index.
 * keys_in/vals_in are clobbered; result in keys_out/vals_out (keys_out may be NULL). */
int gpc_sort_pairs(uint64_t *keys_in, uint32_t *vals_in, uint64_t *keys_out, uint32_t *vals_out,
                   int64_t n, gpc_key_xform xf, void *ws, size_t ws_bytes, void *stream);
/* calculate_morton_order: permutation (int64) that sorts rows by (z,y,x), stable.
 * is_f32 != 0: xyz is float32, else int32.  Synchronises the stream (it reads min/max back). */
size_t gpc_lexorder_workspace_bytes(int64_t n);
int gpc_lexorder_zyx(const void *xyz, int is_f32, int64_t n, int64_t *out_idx,
                     void *ws, size_t ws_bytes, void *stream);

/* ---- a-4: pyramid down (FOG, kit/nn.py:38-55) ---- */
size_t gpc_pyramid_workspace_bytes(int64_t n);
/* keys sorted ascending (duplicates allowed) -> unique keys; *n_out is a device u32 */
int gpc_unique_sorted(const uint64_t *keys, int64_t n, uint64_t *out_keys, uint32_t *n_out,
                      void *ws, size_t ws_bytes, void *stream);
/* child keys (sorted, unique) -> parent keys (sorted, unique) + occupancy byte; xf = transform
 * covering the PARENT level's extent; *n_parent device u32 */
int gpc_pyramid_down(const uint64_t *child_keys, int64_t n_child, gpc_key_xform parent_xf,
                     uint64_t *parent_keys, uint8_t *parent_occ, uint32_t *n_parent,
                     void *ws, size_t ws_bytes, void *stream);

/* ---- a-8: expand children (FCG, kit/nn.py:77-98 + sort_CF) ---- */
size_t gpc_expand_workspace_bytes(int64_t n_parent);
/* parents sorted -> children emitted directly in (z,y,x) order (no sort): child_keys[n_child],
 * child_parent[n_child] = parent row.  n_child must equal sum(popcount(occ)). */
int gpc_expand_children(const uint64_t *parent_keys, const uint8_t *parent_occ, int64_t n_parent,
                        int64_t n_child, uint64_t *child_keys, uint32_t *child_parent,
                        void *ws, size_t ws_bytes, void *stream);
/* decode epilogue (pcc_utils.py:375-379): children in PARENT-MAJOR order (octant ascending), as
 * float32 xyz * scale -- the row order the reference returns. */
int gpc_expand_leaves_f32(const uint64_t *parent_keys, const uint8_t *parent_occ, int64_t n_parent,
                          int64_t n_child, float scale, float *xyz, void *ws, size_t ws_bytes, void *stream);

/* ---- kernel maps (torchsparse hashmap kmap; pcc_utils.py:50-52) ---- */
int64_t gpc_hash_capacity(int64_t n);                      /* slots; table bytes = 16 * slots */
/* keys must be sorted ascending and unique (one slot per x-block of 8 voxels is inserted by the block's first row) */
int gpc_hash_build(const uint64_t *keys, int64_t n, void *table, int64_t capacity, void *stream);
int gpc_hash_lookup(const void *table, int64_t capacity, const uint64_t *query, int64_t n,
                    int32_t *rows, void *stream);
/* dense map, OFFSET-MAJOR: map[k*n + o] = row of (c_o + d_k) or -1; k = ((dz+2)*5+(dy+2))*5+(dx+2).  kernel_size = 5, or 3 (the
 * reference CLI's default, compress_ue_4stage_conv.py:44): offsets outside the inner 3^3 are then absent, and a K = 3 conv runs
 * on the K = 5 kernels with its 27 weight matrices placed at their K = 5 offset indices.
 * cell_counts (optional, may be NULL): u32[tiles * 126], tiles = ceil(n / tile_rows), tile_rows >= 256 and a multiple of 32:
 * the number of present neighbours per (tile, offset), counted from the probes themselves (zeroed by the call) -- the first
 * pass of gpc_kmap_um_scan and the level's density (true pairs per row) without a second read of the map. */
int gpc_kmap_dense(const void *table, int64_t capacity, const uint64_t *keys, int64_t n,
                   int32_t *map, int kernel_size, int tile_rows, uint32_t *cell_counts, void *stream);
/* tile pair lists for the mma.sync conv: tiles of `tile_rows` (8, 16, 32, 64 or 128) consecutive output rows; for tile t and offset
 * k the pairs are [seg[t*126+k], seg[t*126+k+1]) (seg[t*126+125] == next tile's start);
 * pair_nbr = input row, pair_row = output row - t*tile_rows.  Two calls: count (fills seg as an
 * exclusive scan, *n_pairs device u32), then fill. */
size_t gpc_kmap_pairs_workspace_bytes(int64_t n, int tile_rows);
/* pad >= 1: every non-empty (tile, offset) segment is rounded up to a multiple of `pad` entries; the
 * padding entries of the combined stream are all-ones (INVALID).  n_pairs is a device u32[2]:
 * [0] = stream entries (padded), [1] = true (row, neighbour) pairs. */
int gpc_kmap_pairs_count(const int32_t *map, int64_t n, int tile_rows, int pad, uint32_t *seg, uint32_t *n_pairs,
                         void *ws, size_t ws_bytes, void *stream);
/* fill writes the split arrays (pair_nbr/pair_row, may be NULL) and/or the combined stream
 * pairs[p] = nbr | row_in_tile << 32 | k << 48 (may be NULL) consumed by gpc_spconv_fwd_v6 */
int gpc_kmap_pairs_fill(const int32_t *map, int64_t n, int tile_rows, const uint32_t *seg,
                        uint32_t *pair_nbr, uint16_t *pair_row, uint64_t *pairs, int64_t n_entries, void *stream);
/* ---- row ranges of a level (a batch of scenes coded as one union level, pcc_utils.compress_point_clouds): the pair streams of the
 * output rows [row0, row1) of a level of n_level rows whose dense map has leading dimension n_level.  Tiles / blocks start at row0,
 * neighbour indices stay the level's rows, totals are the range's own; seg, rowptr and workspaces are sized for row1 - row0 rows.
 * The streams are exactly those of the range's rows coded as a level of their own, with neighbour indices + row0. */
int gpc_kmap_pairs_count_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows, int pad,
                               uint32_t *seg, uint32_t *n_pairs, void *ws, size_t ws_bytes, void *stream);
int gpc_kmap_pairs_fill_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows,
                              const uint32_t *seg, uint64_t *pairs, int64_t n_entries, void *stream);

/* ---- a-7/a-10/a-12: sparse conv (spnn.Conv3d(32,32,5), bias-less) ---- */
/* y[o,:] = act( sum_k x[nbr_k(o),:] . W[k] (+ residual[o,:]) ); W [125,32,32] fp32;
 * offsets accumulate in ascending k for every row (deterministic). flags: bit0 = ReLU. */
#define GPC_CONV_RELU 1
/* Wa [n_kernels*125][2][2][2][32] uint4: the mma.m16n8k16 A fragments of W[k]^T, bf16 hi and lo halves (one LDG.128 per lane) */
int gpc_spconv_pack_weights_frag(const float *W, int n_kernels, void *Wa, void *stream);

/* the mma.sync conv (spconv.cu): one warp per tile of tile_rows output rows over the combined pair stream padded to 8-entry MMA tiles
 * (pad = 8), W^T[k] as the MMA A operand, the gathered rows as the B operand (bf16 hi / lo split, three terms, fp32 accumulation).
 * variant 42 (tile_rows 64): cp.async gather ring; 46 (16, 32) / 47 (8): the offsets of a tile split over 8 / 16 warps (coarse
 * levels); 48 (32, 64, 128): rows loaded straight into the MMA fragments (v6d, big levels).  Other pairs: GPC_EINVAL. */
int gpc_spconv_fwd_v6(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs,
                      int64_t n, int tile_rows, const float *residual, int flags, float *y, int variant,
                      void *stream);

/* the v6d kernel (variant 48) for the output rows [row0, row1) of the level only (whole tiles; row1 may be n): the decoder codes a
 * level as a wavefront over row chunks, stage i+1 of a chunk as soon as stage i of its 5^3 halo is decoded (pcc_utils.py:319-366 has
 * the four stages strictly one after the other) */
int gpc_spconv_fwd_v6_rows(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs,
                           int64_t n, int tile_rows, const float *residual, int flags, float *y, int variant,
                           int64_t row0, int64_t row1, void *stream);
/* gpc_spconv_fwd_v6 for the output rows [row0, row1) of a level of n_level rows with the range's own pair stream
 * (gpc_kmap_pairs_count_range): x, y and residual are the level's arrays, the tiling starts at row0 */
int gpc_spconv_fwd_v6_range(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, int64_t n_level,
                            int64_t row0, int64_t row1, int tile_rows, const float *residual, int flags, float *y,
                            int variant, void *stream);

/* ---- training (spconv_grad.cu): weight gradient of gpc_spconv_fwd_v6 over the same pair stream (pad = 8) and tiling ----
 * dW[k][ci][co] = sum over the pairs (o, i) of offset k of x[i][ci] * dy[o][co]; x, dy fp32 [n,32], dW fp32 [125,32,32] (every offset
 * is written; offsets without pairs give exact zeros).  bf16 hi / lo split, three terms, fp32 accumulation as the forward; no atomics,
 * the summation order depends on (n, tile_rows) and the map only.  ws: gpc_spconv_wgrad_workspace_bytes(n, tile_rows) bytes.
 * The input gradient is gpc_spconv_fwd_v6 itself with W'[k] = W[124 - k]^T (a submanifold map is symmetric: nbr_k(o) = i <=>
 * nbr_{124-k}(i) = o). */
size_t gpc_spconv_wgrad_workspace_bytes(int64_t n, int tile_rows);
int gpc_spconv_wgrad_v6(const float *x, const float *dy, const uint32_t *seg, const uint64_t *pairs, int64_t n, int tile_rows,
                        float *dW, void *ws, size_t ws_bytes, void *stream);
/* The same dW over the same stream, with the work balanced by pairs rather than by tiles: every offset's 8-entry units are cut into
 * chunks of a compile-time number of units, one warp per chunk, and each offset's chunk partials are added in chunk order by a fixed
 * tree.  Same arithmetic and contract as gpc_spconv_wgrad_v6 (no atomics; the summation order depends on the map, tile_rows and the
 * chunk size only).  n_entries = the stream's entry count (KMap.n_pairs); the grid is sized from it, nothing is read back.
 * ws: gpc_spconv_wgrad_balanced_workspace_bytes(n, tile_rows, n_entries) bytes. */
size_t gpc_spconv_wgrad_balanced_workspace_bytes(int64_t n, int tile_rows, int64_t n_entries);
int gpc_spconv_wgrad_v6_balanced(const float *x, const float *dy, const uint32_t *seg, const uint64_t *pairs, int64_t n, int tile_rows,
                                 int64_t n_entries, float *dW, void *ws, size_t ws_bytes, void *stream);
/* The same dW, balanced the same way, over the pair stream of gpc_spconv_fwd_um (seg, pair_nbr, pair_off of gpc_kmap_um_fill with
 * tile_rows = 512; n_entries = the stream's entry count, a multiple of 16).  An entry's output row is tile * 512 + pair_off / 128;
 * padding entries (0xFFFFFFFF) add nothing.  ws: gpc_spconv_wgrad_um_workspace_bytes(n, tile_rows, n_entries) bytes.
 * The input gradient is gpc_spconv_fwd_um with the gpc_spconv_pack_weights_um pack of W'[k] = W[124 - k]^T. */
size_t gpc_spconv_wgrad_um_workspace_bytes(int64_t n, int tile_rows, int64_t n_entries);
int gpc_spconv_wgrad_um(const float *x, const float *dy, const uint32_t *seg, const uint32_t *pair_nbr, const uint32_t *pair_off,
                        int64_t n, int tile_rows, int64_t n_entries, float *dW, void *ws, size_t ws_bytes, void *stream);
/* The same dW over the sparse map of gpc_spconv_sparse_fwd (seg, pairs, rowptr of gpc_kmap_sparse_fill; n_entries = its entry count,
 * a multiple of 8).  The centre offset is x^T dy over all rows in 8-row units without a gather; the straggler segments are walked
 * like any other stream, each entry's output row read from a slot -> row array the call builds from rowptr in the workspace.
 * ws: gpc_spconv_wgrad_sparse_workspace_bytes(n, n_entries) bytes.  The input gradient is gpc_spconv_sparse_fwd with the
 * gpc_spconv_pack_weights_frag pack of W'[k] = W[124 - k]^T. */
size_t gpc_spconv_wgrad_sparse_workspace_bytes(int64_t n, int64_t n_entries);
int gpc_spconv_wgrad_sparse(const float *x, const float *dy, const uint32_t *seg, const uint64_t *pairs, const uint32_t *rowptr,
                            int64_t n, int64_t n_entries, float *dW, void *ws, size_t ws_bytes, void *stream);

/* ---- the conv of the SPARSE big levels (spconv_sparse.cu): dense centre product + offset-sorted "stragglers" ----
 * For levels with ~1-4 neighbours per row (the finest octree levels).  Sparse map: seg u32[gpc_kmap_sparse_segments(n) + 1]
 * (first entry of every (block of 8192 rows, offset != centre) segment, padded to 8 entries), pairs u64[entries] = nbr | dst << 32
 * (all ones = padding; dst = rowptr[row] + rank of the offset among the row's neighbours), rowptr u32[n + 1].
 * totals = device u32[2]: {entries, true stragglers}.  ws (gpc_kmap_sparse_workspace_bytes) is shared by count and fill. */
int64_t gpc_kmap_sparse_segments(int64_t n);
size_t gpc_kmap_sparse_workspace_bytes(int64_t n);
int gpc_kmap_sparse_count(const int32_t *map, int64_t n, uint32_t *seg, uint32_t *rowptr, uint32_t *totals, void *ws,
                          size_t ws_bytes, void *stream);
int gpc_kmap_sparse_fill(const int32_t *map, int64_t n, const uint32_t *seg, const uint32_t *rowptr, const void *ws,
                         uint64_t *pairs, int64_t n_entries, void *stream);
/* y[o,:] = act( W[centre]^T x[o,:] + sum of the row's stragglers in ascending offset order (+ residual[o,:]) ); fp32 rows in and
 * out; Wa = this conv's slice of gpc_spconv_pack_weights_frag; contrib = scratch of max(stragglers, 1) * 32 floats */
int gpc_spconv_sparse_fwd(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, const uint32_t *rowptr,
                          int64_t n, int64_t n_entries, float *contrib, const float *residual, int flags, float *y, void *stream);

/* the same for the output rows [row0, row1) only (whole 8192-row blocks; row1 may be n) */
int gpc_spconv_sparse_fwd_rows(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, const uint32_t *rowptr,
                               int64_t n, int64_t n_entries, float *contrib, const float *residual, int flags, float *y,
                               int64_t row0, int64_t row1, void *stream);
/* row ranges (see gpc_kmap_pairs_count_range): the sparse map of the rows [row0, row1), and the conv of those rows over the level's
 * arrays (stragglers gather the level's rows; the centre product and outputs are the range's rows) */
int gpc_kmap_sparse_count_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, uint32_t *seg, uint32_t *rowptr,
                                uint32_t *totals, void *ws, size_t ws_bytes, void *stream);
int gpc_kmap_sparse_fill_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, const uint32_t *seg,
                               const uint32_t *rowptr, const void *ws, uint64_t *pairs, int64_t n_entries, void *stream);
int gpc_spconv_sparse_fwd_range(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, const uint32_t *rowptr,
                                int64_t n_level, int64_t row0, int64_t row1, int64_t n_entries, float *contrib, const float *residual,
                                int flags, float *y, void *stream);

/* ---- split rows (spconv_fmt.cu): an activation row stored as 32 x bf16 hi | 32 x bf16 lo (128 B, x = hi + lo to 16 mantissa bits):
 * a gathered row is a tensor-core operand row as it stands */
int gpc_rows_split(const float *x, int64_t n, void *xs, void *stream);
int gpc_rows_join(const void *xs, int64_t n, float *x, void *stream);
#define GPC_CONV_RES_SPLIT 2   /* conv flags bit: residual points to split rows (else fp32 rows) */

/* ---- the tcgen05 sparse conv of the big levels (spconv_um.cu) ----
 * y[o,:] = act( sum_k W[k]^T xs[nbr_k(o),:] (+ residual[o,:]) ).  Transposed formulation: per (tile of tile_rows output rows, offset k)
 * the pairs are the N dimension of tcgen05.mma (chunks of 16..64 pairs), W[k]^T (bf16 hi | lo) is the A operand in tensor
 * memory, the gathered rows (TMA tile::gather4 into 128 B-swizzled tiles; TMA tile loads for the centre offset) are the B operand in shared
 * memory, D in tensor memory; the epilogue adds every pair to its output row's fp32 sum in shared memory, offsets ascending (one
 * fixed summation order per row).
 * xs = split rows; Wp = this conv's slice of gpc_spconv_pack_weights_um ([125][32 co][128 B]); seg / pair_nbr = the pair stream
 * and accumulator-row offsets built by gpc_kmap_um_count / _fill with tile_rows = 512 (the only tile height).  Outputs y (fp32
 * rows) and / or ys (split rows).  Only the output rows [row0, row1) are computed (whole tiles; row1 <= 0 or >= n: to the end):
 * the decoder wavefront.  flags: GPC_CONV_RELU, GPC_CONV_RES_SPLIT, GPC_CONV_PROFILE. */
#define GPC_CONV_PROFILE 256   /* flags bit: run the instrumented build (per-role cycle counters, gpc_debug_conv_um_profile) */
int gpc_debug_conv_um_profile(unsigned long long *out_h, int reset);
int gpc_spconv_pack_weights_um(const float *W, int n_kernels, void *Wp, void *stream);
/* pair stream of gpc_spconv_fwd_um, straight from the dense map (one warp per (tile, offset) cell): seg as gpc_kmap_pairs_count with
 * pad = 16; pair_nbr = input row (padding 0xFFFFFFFF), pair_off = byte offset of the accumulator row, row_in_tile * 128 (padding: the
 * dummy row tile_rows * 128).  totals = device u64[2]: {stream entries (padded), true pairs}. */
size_t gpc_kmap_um_workspace_bytes(int64_t n, int tile_rows);
int gpc_kmap_um_count(const int32_t *map, int64_t n, int tile_rows, uint32_t *seg, unsigned long long *totals, void *ws,
                      size_t ws_bytes, void *stream);
/* the same from the cell counts gpc_kmap_dense produced with this tile_rows (no pass over the map) */
int gpc_kmap_um_scan(const uint32_t *cell_counts, int64_t n, int tile_rows, uint32_t *seg, unsigned long long *totals, void *ws,
                     size_t ws_bytes, void *stream);
int gpc_kmap_um_fill(const int32_t *map, int64_t n, int tile_rows, const uint32_t *seg, uint32_t *pair_nbr, uint32_t *pair_off,
                     void *stream);
/* tile_order (optional, may be NULL): a permutation of the level's tile indices; CTA b of a FULL-level launch takes tile
 * tile_order[b] (heaviest tiles first shortens the tail of the launch; results do not depend on it).  Ignored for row ranges. */
int gpc_spconv_fwd_um(const void *xs, const void *Wp, const uint32_t *seg, const uint32_t *pair_nbr, const uint32_t *pair_off,
                      int64_t n, int tile_rows, const uint32_t *tile_order, const void *residual, int flags, float *y, void *ys,
                      int64_t row0, int64_t row1, void *stream);
/* row ranges (see gpc_kmap_pairs_count_range; tile_rows 512): the pair stream of the rows [row0, row1), and the conv of those rows
 * over the level's arrays.  The TMA descriptors span all n_level rows of xs; tile_order (may be NULL) permutes the range's tiles. */
int gpc_kmap_um_count_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows, uint32_t *seg,
                            unsigned long long *totals, void *ws, size_t ws_bytes, void *stream);
int gpc_kmap_um_fill_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, int tile_rows, const uint32_t *seg,
                           uint32_t *pair_nbr, uint32_t *pair_off, void *stream);
int gpc_spconv_fwd_um_range(const void *xs, const void *Wp, const uint32_t *seg, const uint32_t *pair_nbr, const uint32_t *pair_off,
                            int64_t n_level, int64_t row0, int64_t row1, const uint32_t *tile_order, const void *residual, int flags,
                            float *y, void *ys, void *stream);

/* ---- a-6/a-9/a-12: embeddings ---- */
/* Every producer of conv inputs writes fp32 rows (out), split rows (out_split: 32 x bf16 hi | 32 x bf16 lo, the operand format of
 * gpc_spconv_fwd_um) or both; either pointer may be NULL. */
/* out[o,:] = table[idx[o],:]  (prior_embedding, network_ue_4stage_conv.py:15) */
int gpc_embed_rows(const uint8_t *idx, int64_t n, const float *table, float *out, void *out_split, void *stream);
/* out[j,:] = feat[parent[j],:] + temb[octant(child_key[j]),:]  (FCG replicate + TargetEmbedding) */
int gpc_gather_parent_add_octant(const float *feat, const uint32_t *parent, const uint64_t *child_keys,
                                 int64_t n_child, const float *temb, float *out, void *out_split, void *stream);
/* out[o,:] = u[o,:] + emb[occ[o] >> shift, :]   (pred_head_s{1,2,3}_emb; shift = 7, 6, 4) */
int gpc_add_ctx_embed(const float *u, const uint8_t *occ, int shift, const float *emb, int64_t n,
                      float *out, void *out_split, void *stream);

/* ---- a-12/a-13: fused head: Linear-ReLU-Linear-softmax-cumsum-quantise ---- */
/* cdf [n, A+1] uint16 (int16 bit pattern of kit/op.py:67-79); prob [n, A] optional (may be NULL) */
int gpc_head_cdf(const float *f, int64_t n, const float *W1, const float *b1, const float *W2,
                 const float *b2, int A, uint16_t *cdf, float *prob, void *stream);
/* encoder variant: symbol split (a-11) fused; lohi[o] = c_low | c_high << 16 of THE symbol (c_high == 0 means 0x10000),
 * 4 bytes per row for the host coder instead of the whole CDF row; cdf / prob optional */
int gpc_head_cdf_sym(const float *f, int64_t n, const float *W1, const float *b1, const float *W2,
                     const float *b2, int A, const uint8_t *occ, int shift, uint32_t *lohi,
                     uint16_t *cdf, float *prob, void *stream);
/* a-11: symbol of stage i from the occupancy byte: sym = (occ >> shift) & mask */
int gpc_split_symbol(const uint8_t *occ, int64_t n, int shift, int mask, uint8_t *sym, void *stream);
/* decode: occ[o] |= sym[o] << shift */
int gpc_merge_symbol(uint8_t *occ, int64_t n, int shift, const uint8_t *sym, void *stream);

/* ---- a-14: host range coder (torchac-compatible) ---- */
int gpc_ac_encode_h(const uint16_t *cdf_h, const uint8_t *sym_h, int64_t n, int Lp,
                    uint8_t *out_h, int64_t cap, int64_t *out_len_h);
int gpc_ac_decode_h(const uint16_t *cdf_h, const uint8_t *in_h, int64_t in_len, int64_t n, int Lp,
                    uint8_t *sym_h);
/* gpc_ac_decode_h in pieces (one stream decoded chunk by chunk while later CDF rows are still being computed; the four stage
 * streams of a level then decode concurrently, pcc_utils.py:319-366 run as a wavefront).  `state_h`: caller-owned, state_bytes()
 * bytes; begin binds it to a stream that must outlive it; each `more` decodes the next n symbols from the next n CDF rows.
 * Any split yields the symbols of the one-shot call. */
int64_t gpc_ac_decode_state_bytes(void);
int gpc_ac_decode_begin_h(void *state_h, const uint8_t *in_h, int64_t in_len);
int gpc_ac_decode_more_h(void *state_h, const uint16_t *cdf_h, int64_t n, int Lp, uint8_t *sym_h);
/* same bitstream as gpc_ac_encode_h, fed with the (c_low, c_high) words of gpc_head_cdf_sym */
int gpc_ac_encode_lohi_h(const uint32_t *lohi_h, int64_t n, uint8_t *out_h, int64_t cap, int64_t *out_len_h);

/* ---- f-4: HAC's chunked attribute coder (HAC/submodules/arithmetic.zip!arithmetic/arithmetic_kernel.cu; binding
 * arithmetic.cpp:4-49; callers HAC/utils/encodings_cuda.py:317-432).  All pointers are DEVICE pointers.  A chunk of
 * `chunk_size` symbols (10 000 in encodings_cuda.py:6) is one serial 32-bit range coder, as in the reference. ---- */
/* arithmetic.calculate_cdf (arithmetic_kernel.cu:11-55): lower[n][Lp], Lp = max_value - min_value + 2 */
int gpc_attr_calculate_cdf(const float *mean, const float *scale, const float *Q, int64_t n, int min_value,
                           int max_value, float *lower, void *stream);
size_t gpc_attr_workspace_bytes(int64_t n, int chunk_size);
/* arithmetic.arithmetic_encode (:94-163, :186-232), first half: per-chunk streams into the workspace, cnt[chunks] = bytes per
 * chunk (the reference's out_cnt_all), offsets[chunks + 1] = their exclusive prefix sums (offsets[chunks] = total bytes).
 * Synchronises the stream once (status word).  Symbols outside [0, Lp - 2] are an error. */
int gpc_attr_encode_table(const int16_t *sym, const float *cdf, int64_t n, int Lp, int chunk_size, int32_t *cnt,
                          uint32_t *offsets, void *ws, size_t ws_bytes, void *stream);
/* the same with the Gaussian CDF evaluated for the two bin edges of each symbol instead of read from a table:
 * calculate_cdf + arithmetic_encode of encoder_gaussian (encodings_cuda.py:335-373) without lower[n][Lp] */
int gpc_attr_encode_gaussian(const int16_t *sym, const float *mean, const float *scale, const float *Q, int64_t n,
                             int min_value, int max_value, int chunk_size, int32_t *cnt, uint32_t *offsets, void *ws,
                             size_t ws_bytes, void *stream);
/* second half (merge_chunks_kernel, :166-183): out[offsets[chunks]] = the chunks' bytes back to back */
int gpc_attr_merge_chunks(const void *ws, int64_t n, int chunk_size, const uint32_t *offsets, uint8_t *out, void *stream);
/* arithmetic.arithmetic_decode (:290-356, :365-407) */
int gpc_attr_decode_table(const float *cdf, const uint8_t *in, const int32_t *cnt, int64_t n, int Lp, int chunk_size,
                          int16_t *sym, void *ws, size_t ws_bytes, void *stream);
/* calculate_cdf + arithmetic_decode of decoder_gaussian (encodings_cuda.py:394-432) without the table */
int gpc_attr_decode_gaussian(const float *mean, const float *scale, const float *Q, const uint8_t *in, const int32_t *cnt,
                             int64_t n, int min_value, int max_value, int chunk_size, int16_t *sym, void *ws,
                             size_t ws_bytes, void *stream);
/* HAC++'s mixture coder without the table: calculate_cdf per component, `* prob`, summed in list order and clamped to [0, 1]
 * (encoder_gaussian_mixed / decoder_gaussian_mixed, encodings_cuda.py:203-314), then arithmetic_encode / arithmetic_decode --
 * the same bytes and symbols, with each symbol's CDF entries evaluated on the fly.  mean / scale / prob: [k][n] float32,
 * Q: [n].  1 <= k <= 4, else GPC_EINVAL.  Workspace and merge: gpc_attr_workspace_bytes / gpc_attr_merge_chunks. */
int gpc_mixture_encode(const int16_t *sym, const float *mean, const float *scale, const float *prob, const float *Q,
                       int64_t n, int k, int min_value, int max_value, int chunk_size, int32_t *cnt, uint32_t *offsets,
                       void *ws, size_t ws_bytes, void *stream);
int gpc_mixture_decode(const float *mean, const float *scale, const float *prob, const float *Q, const uint8_t *in,
                       const int32_t *cnt, int64_t n, int k, int min_value, int max_value, int chunk_size, int16_t *sym,
                       void *ws, size_t ws_bytes, void *stream);
/* arithmetic_encode / arithmetic_decode of a table whose n rows are all the same float32 row[Lp]: the Bernoulli mask coder
 * (encoder / decoder, encodings_cuda.py:435-500, row [0, 1 - p, 1]) without the [n][3] table */
int gpc_row_encode(const int16_t *sym, const float *row, int64_t n, int Lp, int chunk_size, int32_t *cnt, uint32_t *offsets,
                   void *ws, size_t ws_bytes, void *stream);
int gpc_row_decode(const float *row, const uint8_t *in, const int32_t *cnt, int64_t n, int Lp, int chunk_size, int16_t *sym,
                   void *ws, size_t ws_bytes, void *stream);

/* ---- f-3: the chunked GPU coder on the geometry codec's own streams (container version 2; NOT the torchac bitstream: one coder
 * per chunk instead of one per stream).  Encode: lohi as gpc_head_cdf_sym writes it; no host synchronisation.  Decode: one stage
 * at a time (stage i + 1 needs stage i) -- one stream, or with _ranges the streams of many scenes whose rows are one after the
 * other in one level -- cdf rows as gpc_head_cdf writes them. ---- */
size_t gpc_chunk_workspace_bytes(int chunks, int max_chunk);
/* chunk w = symbols [starts[w], starts[w + 1]) of lohi (device u32[chunks + 1]; at most max_chunk symbols each): the streams of a
 * scene one after the other, every stream cut into chunks of its own length, all coded by ONE launch */
int gpc_chunk_encode_lohi(const uint32_t *lohi, const uint32_t *starts, int chunks, int max_chunk, int32_t *cnt,
                          uint32_t *offsets, void *ws, size_t ws_bytes, void *stream);
int gpc_chunk_merge(const void *ws, int chunks, int max_chunk, const uint32_t *offsets, uint8_t *out, void *stream);
/* offsets: device u32[chunks + 1], first byte of every chunk in `in` (prefix sums of the stream's u16 byte counts); Lp <= 32 */
int gpc_chunk_decode_u16(const uint16_t *cdf, const uint8_t *in, const uint32_t *offsets, int64_t n, int Lp, int chunk_size,
                         uint8_t *sym, void *stream);
/* chunk w decodes rows [rows[w], rows[w + 1]) of cdf / sym from bytes [offsets[w], offsets[w + 1]) of `in`;
 * rows, offsets: device u32[chunks + 1], non-decreasing; n = rows of cdf / sym; Lp <= 32.  Every chunk is clamped to rows [0, n)
 * (a malformed table decodes garbage, never outside the arrays' rows); bytes past a chunk's length read as zeros. */
int gpc_chunk_decode_u16_ranges(const uint16_t *cdf, int Lp, const uint8_t *in, const uint32_t *offsets, const uint32_t *rows,
                                int chunks, int64_t n, uint8_t *sym, void *stream);

/* ---- ASCII PLY text (textio.cu).  Formatter: row r of xyz (float32 [n][3]) becomes "x y z\n", every value widened to double and
 * written as Python's repr() writes it (shortest round-trip digits, positional for decimal exponents in [-4, 16), else d.ddde+XX),
 * rows back to back in row order; at most 75 bytes a row.  *out_len_h (host) = bytes of text; a buffer of fewer than that many
 * bytes (cap) gives GPC_EINVAL.  Synchronises `stream` (one read-back of the length).  n <= 2^32 / 75. ---- */
size_t gpc_ply_format_workspace_bytes(int64_t n);
int gpc_ply_format_f32(const float *xyz, int64_t n, char *out, uint64_t cap, uint64_t *out_len_h, void *ws, size_t ws_bytes,
                       void *stream);
/* Parser: the rows of cli.read_points' text branch.  Lines end at "\n", "\r\n" or a lone "\r"; a line of printable ASCII and
 * tabs gives a row when its first three space / tab separated tokens are all [+-]?(d+(.d*)?|.d+)([eE][+-]?d+)? (correctly rounded
 * to double, as float() does), no row when it has fewer than three tokens or one is not a float.  A line the GPU leaves to
 * float() itself (any other byte, a token [+-]?(inf|infinity|nan) in any case or holding "_", or a rounding the 128-bit product
 * cannot decide) is reported in host_lines as {first byte, end of its content (terminator excluded), rows before it}; its row, if
 * any, belongs before row `rows before it` of rows.  rows: double [(nbytes + 1) / 6][3]; host_lines: u32 [(nbytes + 1) / 2][3];
 * *n_rows_h, *n_host_h (host): counts.  nbytes < 2^32.  Synchronises `stream` (one read-back of the two counts). */
size_t gpc_text_parse_workspace_bytes(uint64_t nbytes);
int gpc_text_parse_xyz(const char *text, uint64_t nbytes, double *rows, uint32_t *n_rows_h, uint32_t *host_lines,
                       uint32_t *n_host_h, void *ws, size_t ws_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GPCGC_H */

// spconv_grad.cu -- weight gradient of the mma.sync sparse conv (training, gauspcc_b200/train.py).
//
// Forward (spconv.cu): y[o,:] = sum_k x[nbr_k(o),:] . W[k].  Its weight gradient is
//     dW[k][ci][co] = sum over the pairs (o, i = nbr_k(o)) of offset k of x[i][ci] * dy[o][co]
// over the same pair stream the forward consumes (gpc_kmap_pairs_count / _fill with pad = 8): per (tile, offset) segment, entries
// nbr | row_in_tile << 32 | k << 48, padded to whole 8-entry units with all-ones entries, which contribute nothing.
// (The input gradient needs no kernel of its own: on a submanifold map nbr_k(o) = i <=> nbr_{124-k}(i) = o, so dx is the forward
// conv with W'[k] = W[124 - k]^T -- see train.py.)
//
// One CTA per (offset k, group of consecutive tiles); warp w of the CTA walks the group's tiles w, w + 4, ... and, per 8-entry unit
// of the (tile, k) segment, runs mma.m16n8k8 with A = x^T (16 input channels x 8 pairs) and B = dy (8 pairs x 8 output channels):
// the 32 x 32 block of dW[k] is 2 x 4 fragments (32 fp32 registers per lane).  Operands are split into bf16 hi + lo and the three
// terms hi.lo + lo.hi + hi.hi are accumulated in fp32, as in the forward (DESIGN.md 5).  The four warps' sums are added in warp
// order, each group writes its partial to the workspace and a second kernel adds the groups in group order: no atomics, and the
// summation order depends on (n, tile_rows) and the map only, so two calls give the same bits.
//
// The balanced variant (gpc_spconv_wgrad_v6_balanced) splits the same work by pairs instead of by tiles.  On the sparse finest levels
// nearly every pair belongs to the centre offset, and 64 groups of tiles leave that offset as 256 serial chains of 8-pair units.
// Here a plan kernel counts every offset's units per tile (ucum[k][tiles + 1], running sums), every offset's units are cut into
// chunks of WGB_UNITS consecutive units (a chunk never spans two offsets), and one warp per chunk walks its units across tiles with
// the same MMA body.  The chunk partials of an offset are added in chunk order by a fixed tree of fan-in WGB_FANIN (the tree's
// shape depends on the chunk counts only).  No atomics, nothing is read back: the grid is sized from the entry count.
//
// The same machinery, templated on how a stream decodes (WgbUm, WgbSparse), gives the weight gradient of the two other conv
// families: gpc_spconv_wgrad_um over the tcgen05 conv's 512-row tiles, and gpc_spconv_wgrad_sparse over the sparse levels' map,
// whose centre offset is a dense x^T dy over consecutive rows.  The mma.sync kernels keep their own code (and SASS).
#include "common.cuh"

constexpr int WG_WARPS = 4;
constexpr int WG_MAX_GROUPS = 64;

// groups of tiles per offset: about 8 tiles per group (2 per warp), at most 64 groups (8000 CTAs on a 200 K-row level)
static inline i64 wgrad_groups(i64 n, int tile_rows) {
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    i64 g = (tiles + 7) / 8;
    return g < 1 ? 1 : (g > WG_MAX_GROUPS ? WG_MAX_GROUPS : g);
}

__device__ __forceinline__ void mma_bf16_k8(float (&d)[4], u32 a0, u32 a1, u32 b0) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(b0));
}

// acc += x^T dy for one unit of 8 pairs, given lane (g, t)'s x and dy values of pairs 2t (xa, da) and 2t + 1 (xb, db)
__device__ __forceinline__ void wgrad_mma(float (&acc)[2][4][4], const float (&xa)[4], const float (&xb)[4], const float (&da)[4],
                                          const float (&db)[4]) {
    u32 ah[4], al[4], bh[4], bl[4];                      // A: (ci g + 8 j, pairs 2t, 2t + 1); B: (pairs 2t, 2t + 1, co g + 8 j)
#pragma unroll
    for (int j = 0; j < 4; ++j) { split_bf16(xa[j], xb[j], ah[j], al[j]); split_bf16(da[j], db[j], bh[j], bl[j]); }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            mma_bf16_k8(acc[mt][nt], ah[2 * mt], ah[2 * mt + 1], bl[nt]);
            mma_bf16_k8(acc[mt][nt], al[2 * mt], al[2 * mt + 1], bh[nt]);
            mma_bf16_k8(acc[mt][nt], ah[2 * mt], ah[2 * mt + 1], bh[nt]);
        }
}

// one 8-entry unit of the pair stream at p (output rows of the unit's tile start at obase): acc += x^T dy over its pairs
__device__ __forceinline__ void wgrad_unit(float (&acc)[2][4][4], const float *__restrict__ x, const float *__restrict__ dy,
                                           const u64 *__restrict__ pairs, u32 p, i64 obase, int g, int t) {
    // lane (g, t) holds pairs 2t and 2t + 1 of the unit, channels g + 8 j of their x and dy rows
    const u64 ea = __ldg(pairs + p + 2 * t), eb = __ldg(pairs + p + 2 * t + 1);
    const u32 na = (u32)ea, nb = (u32)eb;
    float xa[4], xb[4], da[4], db[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) xa[j] = xb[j] = da[j] = db[j] = 0.f;
    if (na != 0xFFFFFFFFu) {
        const float *xr = x + (i64)na * GPC_C + g, *dr = dy + (obase + (i64)((ea >> 32) & 0xFFFFu)) * GPC_C + g;
#pragma unroll
        for (int j = 0; j < 4; ++j) { xa[j] = __ldg(xr + 8 * j); da[j] = __ldg(dr + 8 * j); }
    }
    if (nb != 0xFFFFFFFFu) {
        const float *xr = x + (i64)nb * GPC_C + g, *dr = dy + (obase + (i64)((eb >> 32) & 0xFFFFu)) * GPC_C + g;
#pragma unroll
        for (int j = 0; j < 4; ++j) { xb[j] = __ldg(xr + 8 * j); db[j] = __ldg(dr + 8 * j); }
    }
    wgrad_mma(acc, xa, xb, da, db);
}

// the same for a unit given as (input row, output row) of pairs 2t (na, oa) and 2t + 1 (nb, ob); an input row of 0xFFFFFFFF is
// padding and contributes nothing
__device__ __forceinline__ void wgrad_rows(float (&acc)[2][4][4], const float *__restrict__ x, const float *__restrict__ dy, u32 na,
                                           i64 oa, u32 nb, i64 ob, int g, int t) {
    float xa[4], xb[4], da[4], db[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) xa[j] = xb[j] = da[j] = db[j] = 0.f;
    if (na != 0xFFFFFFFFu) {
        const float *xr = x + (i64)na * GPC_C + g, *dr = dy + oa * GPC_C + g;
#pragma unroll
        for (int j = 0; j < 4; ++j) { xa[j] = __ldg(xr + 8 * j); da[j] = __ldg(dr + 8 * j); }
    }
    if (nb != 0xFFFFFFFFu) {
        const float *xr = x + (i64)nb * GPC_C + g, *dr = dy + ob * GPC_C + g;
#pragma unroll
        for (int j = 0; j < 4; ++j) { xb[j] = __ldg(xr + 8 * j); db[j] = __ldg(dr + 8 * j); }
    }
    wgrad_mma(acc, xa, xb, da, db);
}

// partial[grp][k][ci][co] of the tiles [grp * tiles / G, (grp + 1) * tiles / G)
__global__ void __launch_bounds__(32 * WG_WARPS) spconv_wgrad_partial_kernel(const float *__restrict__ x, const float *__restrict__ dy,
                                                                            const u32 *__restrict__ seg, const u64 *__restrict__ pairs,
                                                                            i64 tiles, int tile_rows, float *__restrict__ partial) {
    __shared__ float red[WG_WARPS][GPC_C * GPC_C];
    const int k = blockIdx.x, grp = blockIdx.y, G = gridDim.y;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const i64 t0 = tiles * grp / G, t1 = tiles * (grp + 1) / G;
    float acc[2][4][4];                                  // [mt: ci 16 mt..][nt: co 8 nt..][D fragment]
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;
    for (i64 tile = t0 + wid; tile < t1; tile += WG_WARPS) {
        const u32 p0 = __ldg(seg + tile * (GPC_K3 + 1) + k), p1 = __ldg(seg + tile * (GPC_K3 + 1) + k + 1);
        const i64 obase = tile * tile_rows;
#pragma unroll 2
        for (u32 p = p0; p < p1; p += 8) wgrad_unit(acc, x, dy, pairs, p, obase, g, t);
    }
    // D fragment: [0] = (ci 16mt + g, co 8nt + 2t), [1] = co + 1, [2] / [3] = ci + 8
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            float *r = &red[wid][(16 * mt + g) * GPC_C + 8 * nt + 2 * t];
            r[0] = acc[mt][nt][0]; r[1] = acc[mt][nt][1];
            r[8 * GPC_C] = acc[mt][nt][2]; r[8 * GPC_C + 1] = acc[mt][nt][3];
        }
    __syncthreads();
    float *out = partial + ((i64)grp * GPC_K3 + k) * (GPC_C * GPC_C);
    for (int e = threadIdx.x; e < GPC_C * GPC_C; e += 32 * WG_WARPS) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < WG_WARPS; ++w) v += red[w][e];          // warp order
        out[e] = v;
    }
}

// dW[k] = sum over the groups, in group order
__global__ void spconv_wgrad_reduce_kernel(const float *__restrict__ partial, int G, float *__restrict__ dW) {
    const i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (i64)GPC_K3 * GPC_C * GPC_C) return;
    float v = 0.f;
    for (int grp = 0; grp < G; ++grp) v += partial[(i64)grp * GPC_K3 * GPC_C * GPC_C + e];
    dW[e] = v;
}

extern "C" size_t gpc_spconv_wgrad_workspace_bytes(int64_t n, int tile_rows) {
    if (n <= 0 || tile_rows <= 0) return 0;
    return (size_t)wgrad_groups(n, tile_rows) * GPC_K3 * GPC_C * GPC_C * sizeof(float);
}

extern "C" int gpc_spconv_wgrad_v6(const float *x, const float *dy, const uint32_t *seg, const uint64_t *pairs, int64_t n,
                                   int tile_rows, float *dW, void *ws, size_t ws_bytes, void *stream) {
    GPC_REQUIRE(n >= 0, GPC_EINVAL, "n < 0");
    GPC_REQUIRE(tile_rows == 8 || tile_rows == 16 || tile_rows == 32 || tile_rows == 64 || tile_rows == 128, GPC_EINVAL,
                "tile_rows must be 8, 16, 32, 64 or 128 (the mma.sync conv's tile heights)");
    cudaStream_t st = as_stream(stream);
    if (n == 0) {
        GPC_CUDA_CHECK(cudaMemsetAsync(dW, 0, (size_t)GPC_K3 * GPC_C * GPC_C * sizeof(float), st));
        return GPC_OK;
    }
    GPC_REQUIRE(ws_bytes >= gpc_spconv_wgrad_workspace_bytes(n, tile_rows), GPC_ENOSPC, "wgrad workspace too small");
    const i64 tiles = (n + tile_rows - 1) / tile_rows;
    const int G = (int)wgrad_groups(n, tile_rows);
    spconv_wgrad_partial_kernel<<<dim3(GPC_K3, G), 32 * WG_WARPS, 0, st>>>(x, dy, seg, pairs, tiles, tile_rows, (float *)ws);
    GPC_LAUNCH_CHECK();
    spconv_wgrad_reduce_kernel<<<cdiv((i64)GPC_K3 * GPC_C * GPC_C, 256), 256, 0, st>>>((const float *)ws, G, dW);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// ---------------------------------------------------------------------------------------------------------------- balanced by pairs
#ifndef WGB_UNITS
#define WGB_UNITS 4                                      // 8-entry units per chunk (one warp), the fastest of 4..64 measured
#endif
constexpr int WGB_WARPS = 4;                             // independent warps (chunks) per CTA of the partial kernel
constexpr int WGB_FANIN = 32;                            // partials added per step of the reduction tree

// How a pair stream decodes, for the balanced machinery below.  A "tile" is the stream's unit of segmentation (a tile of the
// mma.sync or tcgen05 conv, an 8192-row block of the sparse conv) and k a slot of the weight gradient, equal to the offset it sums:
//   units(tile, k)        8-entry units of the (tile, k) segment
//   first(tile, k)        its first entry
//   unit(acc, .., p, ..)  acc += x^T dy over the 8 entries at p of the (tile, k) segment
// Segments of the mma.sync map (gpc_kmap_pairs_fill) and of the tcgen05 map: seg[tile * 126 + k].  (The mma.sync chunk kernel
// below decodes its entries itself.)
struct WgbSeg126 {
    const u32 *seg;
    __device__ __forceinline__ u32 first(i64 tile, int k) const { return __ldg(seg + tile * (GPC_K3 + 1) + k); }
    __device__ __forceinline__ u32 units(i64 tile, int k) const {
        return (__ldg(seg + tile * (GPC_K3 + 1) + k + 1) - __ldg(seg + tile * (GPC_K3 + 1) + k)) >> 3;
    }
};
// tcgen05 map (gpc_kmap_um_fill): 512-row tiles, cells padded to 16 entries; entry q has its input row pair_nbr[q] (0xFFFFFFFF =
// padding) and the byte offset pair_off[q] = row_in_tile * 128 of its accumulator row
struct WgbUm : WgbSeg126 {
    const u32 *nbr, *off;
    int tile_rows;
    __device__ __forceinline__ void unit(float (&acc)[2][4][4], const float *__restrict__ x, const float *__restrict__ dy, u32 p,
                                         i64 tile, int, int g, int t) const {
        const uint2 nb = __ldg(reinterpret_cast<const uint2 *>(nbr + p + 2 * t));    // p is a multiple of 8: 8-byte aligned
        const uint2 of = __ldg(reinterpret_cast<const uint2 *>(off + p + 2 * t));
        const i64 obase = tile * tile_rows;
        wgrad_rows(acc, x, dy, nb.x, obase + (of.x >> 7), nb.y, obase + (of.y >> 7), g, t);
    }
};
// sparse map (gpc_kmap_sparse_fill): tiles are 8192-row blocks b.  Slot 62 (the centre) has no segment: its units are the block's
// rows, 8 consecutive rows each (x[r]^T dy[r], no gather; the last block's rows past n are skipped).  Every other slot k is the
// straggler segment seg[b * 125 + kk], kk = k - (k > 62), of entries nbr | dst << 32 with dst a contribution slot (rowptr[row] +
// rank); slot_row[dst] is the output row (written by sp_slot_row_kernel).
constexpr int WGS_TB = 8192;
struct WgbSparse {
    const u32 *seg;
    const u64 *pairs;
    const u32 *slot_row;
    i64 n;
    __device__ __forceinline__ u32 first(i64 b, int k) const {
        return k == GPC_K3 / 2 ? 0u : __ldg(seg + b * GPC_K3 + k - (k > GPC_K3 / 2));
    }
    __device__ __forceinline__ u32 units(i64 b, int k) const {
        if (k == GPC_K3 / 2) return (u32)((min((i64)WGS_TB, n - b * WGS_TB) + 7) >> 3);
        const u32 *s = seg + b * GPC_K3 + k - (k > GPC_K3 / 2);
        return (__ldg(s + 1) - __ldg(s)) >> 3;
    }
    __device__ __forceinline__ void unit(float (&acc)[2][4][4], const float *__restrict__ x, const float *__restrict__ dy, u32 p,
                                         i64 b, int k, int g, int t) const {
        if (k == GPC_K3 / 2) {
            const i64 ra = b * WGS_TB + p + 2 * t, rb = ra + 1;
            wgrad_rows(acc, x, dy, ra < n ? (u32)ra : 0xFFFFFFFFu, ra, rb < n ? (u32)rb : 0xFFFFFFFFu, rb, g, t);
            return;
        }
        const u64 ea = __ldg(pairs + p + 2 * t), eb = __ldg(pairs + p + 2 * t + 1);
        const u32 na = (u32)ea, nb = (u32)eb;
        wgrad_rows(acc, x, dy, na, na != 0xFFFFFFFFu ? (i64)__ldg(slot_row + (ea >> 32)) : 0, nb,
                   nb != 0xFFFFFFFFu ? (i64)__ldg(slot_row + (eb >> 32)) : 0, g, t);
    }
};

// the balanced kernel's workspace: ucum u32[125][tiles + 1], plan i32[levels + 1][126] (per tree level the exclusive prefix of
// every offset's partial count; level 0 = the chunks), then per tree level its partials [count bound][32 * 32] fp32, then `extra`
// bytes of the layout's own (the sparse map's slot -> row array).
struct WgbLayout {
    i64 tiles = 0;
    int levels = 0;                                      // tree steps before the final one; then <= WGB_FANIN partials per offset
    size_t ucum = 0, plan = 0, part[8] = {}, extra = 0, bytes = 0;
    i64 bound[8] = {};                                   // partials of each level, at most
    int U = WGB_UNITS;                                   // units per chunk
};

static inline size_t wgb_align(size_t b) { return (b + 255) / 256 * 256; }

// tiles of the stream, units = 8-entry units of all its segments together (at most), U units per chunk
static WgbLayout wgb_layout_units(i64 tiles, i64 units, size_t extra, int U = WGB_UNITS) {
    WgbLayout L;
    L.tiles = tiles;
    L.U = U;
    L.bound[0] = GPC_K3 + (units + U - 1) / U;                     // sum over offsets of ceil(units_k / U)
    i64 per_offset = (units + U - 1) / U;                          // chunks of one offset, at most
    while (per_offset > WGB_FANIN) {
        per_offset = (per_offset + WGB_FANIN - 1) / WGB_FANIN;
        L.bound[L.levels + 1] = GPC_K3 + (L.bound[L.levels] + WGB_FANIN - 1) / WGB_FANIN;
        ++L.levels;
    }
    size_t off = 0;
    L.ucum = off; off = wgb_align(off + (size_t)GPC_K3 * (L.tiles + 1) * sizeof(u32));
    L.plan = off; off = wgb_align(off + (size_t)(L.levels + 1) * (GPC_K3 + 1) * sizeof(int));
    for (int l = 0; l <= L.levels; ++l) { L.part[l] = off; off = wgb_align(off + (size_t)L.bound[l] * GPC_C * GPC_C * sizeof(float)); }
    L.extra = off; off = wgb_align(off + extra);
    L.bytes = off;
    return L;
}

static WgbLayout wgb_layout(i64 n, int tile_rows, i64 n_entries) {
    return wgb_layout_units((n + tile_rows - 1) / tile_rows, (n_entries + 7) / 8, 0);
}

// units per chunk of the sparse and tcgen05 streams: WGB_UNITS, doubled while the level would have more than WGB_CHUNKS chunks.
// Every chunk writes a 4 KB partial; a dense level of 1.2 M rows has ~6 M units, whose partials at 4 units per chunk would be
// ~6 GB of traffic against a ~0.3 GB input.  WGB_CHUNKS warps are a few waves of the chunk kernel on 148 SMs.
constexpr i64 WGB_CHUNKS = 16384;
static int wgb_units_per_chunk(i64 units) {
    int U = WGB_UNITS;
    while (units > WGB_CHUNKS * U && U < 4096) U *= 2;
    return U;
}

// ucum[k][t] = units of offset k in the tiles before t; one CTA per offset, a block scan over the tiles
template <class L>
__device__ __forceinline__ void wgb_units_body(const L &lay, i64 tiles, u32 *__restrict__ ucum) {
    __shared__ u32 wsum[32];
    const int k = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    u32 *out = ucum + (i64)k * (tiles + 1);
    if (threadIdx.x == 0) out[0] = 0;
    u32 carry = 0;
    for (i64 base = 0; base < tiles; base += 1024) {
        const i64 tile = base + threadIdx.x;
        u32 v = tile < tiles ? lay.units(tile, k) : 0u;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 o = __shfl_up_sync(0xFFFFFFFFu, v, d);
            if (lane >= d) v += o;
        }
        if (lane == 31) wsum[wid] = v;
        __syncthreads();
        u32 before = carry;
        for (int w = 0; w < wid; ++w) before += wsum[w];
        if (tile < tiles) out[tile + 1] = before + v;
        u32 total = 0;
#pragma unroll
        for (int w = 0; w < 32; ++w) total += wsum[w];
        carry += total;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(1024) spconv_wgrad_units_kernel(const u32 *__restrict__ seg, i64 tiles, u32 *__restrict__ ucum) {
    wgb_units_body(WgbSeg126{seg}, tiles, ucum);
}
template <class L>
__global__ void __launch_bounds__(1024) wgrad_units_kernel(const L lay, i64 tiles, u32 *__restrict__ ucum) {
    wgb_units_body(lay, tiles, ucum);
}

// plan[0][k] = first chunk of offset k (chunks of WGB_UNITS units), plan[l][k] = first partial of offset k at tree level l.
// The counts are read in parallel; one thread scans them in shared memory.
__device__ __forceinline__ void wgb_plan_body(const u32 *__restrict__ ucum, i64 tiles, int levels, int *__restrict__ plan, u32 U) {
    __shared__ int cnt[GPC_K3], first[8][GPC_K3 + 1];
    const int k = threadIdx.x;
    if (k < GPC_K3) cnt[k] = (int)((__ldg(ucum + (i64)k * (tiles + 1) + tiles) + U - 1) / U);
    __syncthreads();
    if (k == 0) {
        for (int l = 0; l <= levels; ++l) {
            int c = 0;
            for (int j = 0; j < GPC_K3; ++j) {
                first[l][j] = c;
                c += l == 0 ? cnt[j] : (first[l - 1][j + 1] - first[l - 1][j] + WGB_FANIN - 1) / WGB_FANIN;
            }
            first[l][GPC_K3] = c;
        }
    }
    __syncthreads();
    for (int l = 0; l <= levels; ++l)
        if (k <= GPC_K3) plan[l * (GPC_K3 + 1) + k] = first[l][k];
}
__global__ void __launch_bounds__(128) spconv_wgrad_plan_kernel(const u32 *__restrict__ ucum, i64 tiles, int levels,
                                                                int *__restrict__ plan) {
    wgb_plan_body(ucum, tiles, levels, plan, WGB_UNITS);
}
__global__ void __launch_bounds__(128) wgrad_plan_kernel(const u32 *__restrict__ ucum, i64 tiles, int levels, int *__restrict__ plan,
                                                         int U) {
    wgb_plan_body(ucum, tiles, levels, plan, (u32)U);
}

// largest k in [0, 125) with first[k] <= i (first[] ascending): the offset whose partials hold index i
__device__ __forceinline__ int wgb_offset_of(const int *__restrict__ first, int i) {
    int lo = 0, hi = GPC_K3;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(first + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// one warp per chunk: units [j U, (j + 1) U) of offset k, walked across tiles -> partial[chunk][ci][co]
template <class L>
__device__ __forceinline__ void wgb_chunk_body(const float *__restrict__ x, const float *__restrict__ dy, const L &lay, i64 tiles,
                                               const u32 *__restrict__ ucum, const int *__restrict__ plan, float *__restrict__ partial,
                                               u32 U) {
    const int chunk = blockIdx.x * WGB_WARPS + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    if (chunk >= __ldg(plan + GPC_K3)) return;          // surplus warps of the host-sized grid
    const int k = wgb_offset_of(plan, chunk);
    const u32 *uc = ucum + (i64)k * (tiles + 1);
    u32 u = (u32)(chunk - __ldg(plan + k)) * U;
    const u32 uend = min(u + U, __ldg(uc + tiles));
    i64 lo = 0, hi = tiles;                              // the tile holding unit u: largest tile with uc[tile] <= u
    while (hi - lo > 1) {
        const i64 mid = (lo + hi) >> 1;
        if (__ldg(uc + mid) <= u) lo = mid; else hi = mid;
    }
    float acc[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;
    for (i64 tile = lo; u < uend; ++tile) {
        const u32 first = __ldg(uc + tile), stop = min(uend, __ldg(uc + tile + 1));
        u32 p = lay.first(tile, k) + 8 * (u - first);
#pragma unroll 2
        for (; u < stop; ++u, p += 8) lay.unit(acc, x, dy, p, tile, k, g, t);
    }
    float *out = partial + (i64)chunk * (GPC_C * GPC_C);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            float *r = out + (16 * mt + g) * GPC_C + 8 * nt + 2 * t;
            *reinterpret_cast<float2 *>(r) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
            *reinterpret_cast<float2 *>(r + 8 * GPC_C) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
        }
}
// (gpc_spconv_wgrad_v6_balanced keeps its own copy of the walk, written out for the mma.sync stream: its SASS stays what it was)
__global__ void __launch_bounds__(32 * WGB_WARPS) spconv_wgrad_chunk_kernel(const float *__restrict__ x, const float *__restrict__ dy,
                                                                           const u32 *__restrict__ seg, const u64 *__restrict__ pairs,
                                                                           i64 tiles, int tile_rows, const u32 *__restrict__ ucum,
                                                                           const int *__restrict__ plan, float *__restrict__ partial) {
    const int chunk = blockIdx.x * WGB_WARPS + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    if (chunk >= __ldg(plan + GPC_K3)) return;          // surplus warps of the host-sized grid
    const int k = wgb_offset_of(plan, chunk);
    const u32 *uc = ucum + (i64)k * (tiles + 1);
    u32 u = (u32)(chunk - __ldg(plan + k)) * WGB_UNITS;
    const u32 uend = min(u + (u32)WGB_UNITS, __ldg(uc + tiles));
    i64 lo = 0, hi = tiles;                              // the tile holding unit u: largest tile with uc[tile] <= u
    while (hi - lo > 1) {
        const i64 mid = (lo + hi) >> 1;
        if (__ldg(uc + mid) <= u) lo = mid; else hi = mid;
    }
    float acc[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;
    for (i64 tile = lo; u < uend; ++tile) {
        const u32 first = __ldg(uc + tile), stop = min(uend, __ldg(uc + tile + 1));
        u32 p = __ldg(seg + tile * (GPC_K3 + 1) + k) + 8 * (u - first);
        const i64 obase = tile * tile_rows;
#pragma unroll 2
        for (; u < stop; ++u, p += 8) wgrad_unit(acc, x, dy, pairs, p, obase, g, t);
    }
    float *out = partial + (i64)chunk * (GPC_C * GPC_C);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            float *r = out + (16 * mt + g) * GPC_C + 8 * nt + 2 * t;
            *reinterpret_cast<float2 *>(r) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
            *reinterpret_cast<float2 *>(r + 8 * GPC_C) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
        }
}
template <class L>
__global__ void __launch_bounds__(32 * WGB_WARPS) wgrad_chunk_kernel(const float *__restrict__ x, const float *__restrict__ dy, const L lay,
                                                                    i64 tiles, const u32 *__restrict__ ucum, const int *__restrict__ plan,
                                                                    float *__restrict__ partial, int U) {
    wgb_chunk_body(x, dy, lay, tiles, ucum, plan, partial, (u32)U);
}

// one step of the tree: output partial i of offset k = the sum, in order, of its inputs [j F, (j + 1) F) (j = i - first_out[k]).
// final: one CTA per offset writes dW[k] (+0 for an offset without partials)
__global__ void __launch_bounds__(256) spconv_wgrad_tree_kernel(const float *__restrict__ in, const int *__restrict__ first_in,
                                                               const int *__restrict__ first_out, float *__restrict__ out, int final_) {
    int k, i;
    if (final_) {
        k = blockIdx.x;
        i = k;
    } else {
        i = blockIdx.x;
        if (i >= __ldg(first_out + GPC_K3)) return;
        k = wgb_offset_of(first_out, i);
    }
    const int a0 = __ldg(first_in + k), a1 = __ldg(first_in + k + 1);
    const int j = final_ ? 0 : i - __ldg(first_out + k);
    const int b0 = a0 + j * WGB_FANIN, b1 = final_ ? a1 : min(a1, b0 + WGB_FANIN);
    float *o = out + (i64)i * (GPC_C * GPC_C);
    for (int e = threadIdx.x; e < GPC_C * GPC_C; e += 256) {
        float v = 0.f;
        for (int b = b0; b < b1; ++b) v += in[(i64)b * (GPC_C * GPC_C) + e];
        o[e] = v;
    }
}

// plan, chunks and the tree after the units kernel has written ucum
static int wgb_reduce_launch(const WgbLayout &L, char *w, float *dW, cudaStream_t st) {
    int *plan = (int *)(w + L.plan);
    for (int l = 1; l <= L.levels; ++l) {
        spconv_wgrad_tree_kernel<<<(unsigned)L.bound[l], 256, 0, st>>>((const float *)(w + L.part[l - 1]), plan + (l - 1) * (GPC_K3 + 1),
                                                                       plan + l * (GPC_K3 + 1), (float *)(w + L.part[l]), 0);
        GPC_LAUNCH_CHECK();
    }
    spconv_wgrad_tree_kernel<<<GPC_K3, 256, 0, st>>>((const float *)(w + L.part[L.levels]), plan + L.levels * (GPC_K3 + 1), nullptr, dW, 1);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// the whole balanced weight gradient over the stream of layout lay
template <class Lay>
static int wgb_run(const float *x, const float *dy, const Lay &lay, const WgbLayout &L, char *w, float *dW, cudaStream_t st) {
    u32 *ucum = (u32 *)(w + L.ucum);
    int *plan = (int *)(w + L.plan);
    wgrad_units_kernel<Lay><<<GPC_K3, 1024, 0, st>>>(lay, L.tiles, ucum);
    GPC_LAUNCH_CHECK();
    wgrad_plan_kernel<<<1, 128, 0, st>>>(ucum, L.tiles, L.levels, plan, L.U);
    GPC_LAUNCH_CHECK();
    wgrad_chunk_kernel<Lay><<<cdiv(L.bound[0], WGB_WARPS), 32 * WGB_WARPS, 0, st>>>(x, dy, lay, L.tiles, ucum, plan, (float *)(w + L.part[0]),
                                                                                    L.U);
    GPC_LAUNCH_CHECK();
    return wgb_reduce_launch(L, w, dW, st);
}

extern "C" size_t gpc_spconv_wgrad_balanced_workspace_bytes(int64_t n, int tile_rows, int64_t n_entries) {
    if (n <= 0 || tile_rows <= 0 || n_entries < 0) return 0;
    return wgb_layout(n, tile_rows, n_entries).bytes;
}

extern "C" int gpc_spconv_wgrad_v6_balanced(const float *x, const float *dy, const uint32_t *seg, const uint64_t *pairs, int64_t n,
                                            int tile_rows, int64_t n_entries, float *dW, void *ws, size_t ws_bytes, void *stream) {
    GPC_REQUIRE(n >= 0, GPC_EINVAL, "n < 0");
    GPC_REQUIRE(tile_rows == 8 || tile_rows == 16 || tile_rows == 32 || tile_rows == 64 || tile_rows == 128, GPC_EINVAL,
                "tile_rows must be 8, 16, 32, 64 or 128 (the mma.sync conv's tile heights)");
    GPC_REQUIRE(n_entries >= 0 && n_entries <= 0xFFFFFFFFll, GPC_EINVAL, "n_entries outside [0, 2^32)");
    cudaStream_t st = as_stream(stream);
    if (n == 0) {
        GPC_CUDA_CHECK(cudaMemsetAsync(dW, 0, (size_t)GPC_K3 * GPC_C * GPC_C * sizeof(float), st));
        return GPC_OK;
    }
    const WgbLayout L = wgb_layout(n, tile_rows, n_entries);
    GPC_REQUIRE(ws_bytes >= L.bytes, GPC_ENOSPC, "wgrad workspace too small");
    char *w = (char *)ws;
    u32 *ucum = (u32 *)(w + L.ucum);
    int *plan = (int *)(w + L.plan);
    spconv_wgrad_units_kernel<<<GPC_K3, 1024, 0, st>>>(seg, L.tiles, ucum);
    GPC_LAUNCH_CHECK();
    spconv_wgrad_plan_kernel<<<1, 128, 0, st>>>(ucum, L.tiles, L.levels, plan);
    GPC_LAUNCH_CHECK();
    spconv_wgrad_chunk_kernel<<<cdiv(L.bound[0], WGB_WARPS), 32 * WGB_WARPS, 0, st>>>(x, dy, seg, pairs, L.tiles, tile_rows, ucum, plan,
                                                                                     (float *)(w + L.part[0]));
    GPC_LAUNCH_CHECK();
    return wgb_reduce_launch(L, w, dW, st);
}

// ------------------------------------------------------------------------------------------------- tcgen05 map (spconv_um.cu)
// The same balanced machinery over the tcgen05 conv's stream: 512-row tiles, (tile, offset) cells padded to 16 entries (two
// units; padding entries gather nothing).  The centre offset's cells hold every row of the tile, like any other offset's.
static WgbLayout wgb_um_layout(i64 n, int tile_rows, i64 n_entries) {
    const i64 units = (n_entries + 7) / 8;
    return wgb_layout_units((n + tile_rows - 1) / tile_rows, units, 0, wgb_units_per_chunk(units));
}

extern "C" size_t gpc_spconv_wgrad_um_workspace_bytes(int64_t n, int tile_rows, int64_t n_entries) {
    if (n <= 0 || tile_rows <= 0 || n_entries < 0) return 0;
    return wgb_um_layout(n, tile_rows, n_entries).bytes;
}

extern "C" int gpc_spconv_wgrad_um(const float *x, const float *dy, const uint32_t *seg, const uint32_t *pair_nbr,
                                   const uint32_t *pair_off, int64_t n, int tile_rows, int64_t n_entries, float *dW, void *ws,
                                   size_t ws_bytes, void *stream) {
    GPC_REQUIRE(n >= 0, GPC_EINVAL, "n < 0");
    GPC_REQUIRE(tile_rows == 512, GPC_EINVAL, "tile_rows must be 512 (the tcgen05 conv's tile height)");
    GPC_REQUIRE(n_entries >= 0 && n_entries <= 0xFFFFFFFFll && n_entries % 16 == 0, GPC_EINVAL,
                "n_entries must be a multiple of 16 in [0, 2^32)");
    cudaStream_t st = as_stream(stream);
    if (n == 0) {
        GPC_CUDA_CHECK(cudaMemsetAsync(dW, 0, (size_t)GPC_K3 * GPC_C * GPC_C * sizeof(float), st));
        return GPC_OK;
    }
    const WgbLayout L = wgb_um_layout(n, tile_rows, n_entries);
    GPC_REQUIRE(ws_bytes >= L.bytes, GPC_ENOSPC, "wgrad workspace too small");
    return wgb_run(x, dy, WgbUm{{seg}, pair_nbr, pair_off, tile_rows}, L, (char *)ws, dW, st);
}

// ------------------------------------------------------------------------------------------------ sparse map (spconv_sparse.cu)
// The centre offset is a dense product over consecutive rows (slot 62 of WgbSparse: 8-row units, no gather), the stragglers are
// the map's (block, offset) segments.  A straggler entry names its contribution slot, not its row, so the output row of every slot
// is written first: slot_row[j] = r for j in [rowptr[r], rowptr[r + 1]).  That is one pass over rowptr (4 bytes per row) per call,
// a few microseconds, against a binary search of rowptr for every entry in the chunk loop; building it per call keeps the kernel
// map what the forward needs and nothing more.
__global__ void __launch_bounds__(256) sp_slot_row_kernel(const u32 *__restrict__ rowptr, i64 n, u32 *__restrict__ slot_row) {
    const i64 r = (i64)blockIdx.x * 256 + threadIdx.x;
    if (r >= n) return;
    const u32 a = __ldg(rowptr + r), b = __ldg(rowptr + r + 1);
    for (u32 j = a; j < b; ++j) slot_row[j] = (u32)r;
}

static WgbLayout wgb_sparse_layout(i64 n, i64 n_entries) {
    // units: the stragglers' (n_entries / 8, whole units per segment) and the centre's (8-row units; every block but the last
    // is a multiple of 8 rows); extra: slot_row, one word per straggler (at most one per entry)
    const i64 units = (n_entries + 7) / 8 + (n + 7) / 8;
    return wgb_layout_units((n + WGS_TB - 1) / WGS_TB, units, (size_t)n_entries * sizeof(u32), wgb_units_per_chunk(units));
}

extern "C" size_t gpc_spconv_wgrad_sparse_workspace_bytes(int64_t n, int64_t n_entries) {
    if (n <= 0 || n_entries < 0) return 0;
    return wgb_sparse_layout(n, n_entries).bytes;
}

extern "C" int gpc_spconv_wgrad_sparse(const float *x, const float *dy, const uint32_t *seg, const uint64_t *pairs,
                                       const uint32_t *rowptr, int64_t n, int64_t n_entries, float *dW, void *ws, size_t ws_bytes,
                                       void *stream) {
    GPC_REQUIRE(n >= 0 && n * (int64_t)(GPC_K3 - 1) < (1ll << 32), GPC_EINVAL, "n outside the sparse map's range (n * 124 < 2^32)");
    GPC_REQUIRE(n_entries >= 0 && n_entries % 8 == 0 && n_entries <= 0xFFFFFFFFll, GPC_EINVAL,
                "n_entries must be a multiple of 8 in [0, 2^32)");
    cudaStream_t st = as_stream(stream);
    if (n == 0) {
        GPC_CUDA_CHECK(cudaMemsetAsync(dW, 0, (size_t)GPC_K3 * GPC_C * GPC_C * sizeof(float), st));
        return GPC_OK;
    }
    const WgbLayout L = wgb_sparse_layout(n, n_entries);
    GPC_REQUIRE(ws_bytes >= L.bytes, GPC_ENOSPC, "wgrad workspace too small");
    char *w = (char *)ws;
    u32 *slot_row = (u32 *)(w + L.extra);
    if (n_entries > 0) {
        sp_slot_row_kernel<<<cdiv(n, 256), 256, 0, st>>>(rowptr, n, slot_row);
        GPC_LAUNCH_CHECK();
    }
    return wgb_run(x, dy, WgbSparse{seg, pairs, slot_row, n}, L, w, dW, st);
}

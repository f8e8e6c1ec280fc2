// spconv_sparse.cu -- the sparse convolution on the SPARSE big levels (the finest octree levels: ~1M rows, 1-3 neighbours per row).
//
// Reference: spnn.Conv3d(32, 32, 5) of src/ai_pcc/GausPcgc/network_ue_4stage_conv.py:17-62, semantics as in spconv.cu.
//
// Why a second formulation.  On these levels nearly every (64-row tile, offset) of the tiled kernel (spconv.cu v6) holds ONE
// neighbour pair: it still costs a whole 8-slot MMA tile and a 4 KB fetch of W[k]^T fragments, 38-42 clk per pair against 16 on
// the dense levels, and the three finest levels are 18 % of the step.  Here the conv is split by what is regular:
//   centre offset   every row is its own neighbour: a dense [n x 32] x [32 x 32] product over CONTIGUOUS rows, W[centre] held in
//                   registers for the whole kernel, no gather, no kernel map (kernel 2 below)
//   "stragglers"    the other pairs, sorted by (block of 8192 rows, offset, row): a segment of one offset holds ~10-140 pairs, so
//                   W[k] is fetched once per segment and the 8-pair MMA tiles are full (kernel 1).  A straggler's product is
//                   written to contrib[dst], dst = rowptr[row] + (rank of the offset among the row's neighbours): row-major,
//                   so that kernel 2 adds a row's contributions with contiguous reads, in ascending offset order -- one fixed
//                   summation order per row (encoder and decoder CDFs stay bit-identical), no atomics, no scatter-add.
// Kernel map of this mode ("sparse map"): seg[b * 125 + kk] = first entry of (block b, offset kk) (kk skips the centre; padded
// to 8 entries per segment; slot 124 of a block is an empty pad), pairs[q] = nbr | dst << 32 (all ones = padding), rowptr[n + 1].
#include "common.cuh"

namespace {

constexpr int SP_TB = 8192;                 // rows per block
constexpr int SP_ST = SP_TB / 32;           // 32-row sub-tiles (one warp each in the builders) per block
constexpr int SP_KK = GPC_K3 - 1;           // offsets without the centre
constexpr int SP_CENTRE = GPC_K3 / 2;       // 62: (0, 0, 0)

__device__ __forceinline__ int sp_offset(int kk) { return kk < SP_CENTRE ? kk : kk + 1; }

__device__ __forceinline__ void sp_cp_async16(void *smem_dst, const void *gmem_src) {
    const u32 d = (u32)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void sp_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void sp_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void sp_mma(float (&d)[4], const uint4 &a, u32 b0, u32 b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}

// ---------------------------------------------------------------- sparse map: count
// one warp per 32-row sub-tile: cnt2[(b * 124 + kk) * 256 + st] = rows of the sub-tile with a neighbour at offset kk; rowcnt[r]
__global__ void __launch_bounds__(128) sp_count_kernel(const i32 *__restrict__ map, i64 n, i64 ld, i64 n_sub, u32 *__restrict__ cnt2,
                                                       u32 *__restrict__ rowcnt) {
    const int lane = threadIdx.x & 31;
    const i64 sg = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (sg >= n_sub) return;
    const i64 r = sg * 32 + lane;
    const i64 b = sg / SP_ST;
    const int st = (int)(sg % SP_ST);
    u32 rc = 0;
#pragma unroll 4
    for (int kk = 0; kk < SP_KK; ++kk) {
        const bool v = r < n && map[(i64)sp_offset(kk) * ld + r] >= 0;
        const u32 c = __popc(__ballot_sync(0xFFFFFFFFu, v));
        rc += v ? 1u : 0u;
        if (lane == 0) cnt2[((size_t)b * SP_KK + kk) * SP_ST + st] = c;
    }
    if (r < n) rowcnt[r] = rc;
}
// one warp per (block, offset): exclusive scan of the 256 sub-tile counts in place; padded total -> tot8[b * 125 + kk]
__global__ void __launch_bounds__(128) sp_segment_kernel(u32 *__restrict__ cnt2, i64 n_seg, u32 *__restrict__ tot8) {
    const int lane = threadIdx.x & 31;
    const i64 i = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (i >= n_seg) return;
    u32 *c = cnt2 + (size_t)i * SP_ST + lane * 8;
    u32 v[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { v[j] = c[j]; sum += v[j]; }
    u32 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
    u32 run = incl - sum;
#pragma unroll
    for (int j = 0; j < 8; ++j) { c[j] = run; run += v[j]; }
    if (lane == 31) tot8[(i / SP_KK) * GPC_K3 + (i % SP_KK)] = (incl + 7u) & ~7u;
}
__global__ void sp_totals_kernel(const u32 *__restrict__ seg, i64 m, const u32 *__restrict__ rowptr, i64 n, u32 *__restrict__ totals) {
    totals[0] = seg[m];          // entries (padded)
    totals[1] = rowptr[n];       // true stragglers
}
// one warp per 32-row sub-tile: pairs[seg + pos2 + rank] = nbr | (rowptr[row] + rank of the offset within the row) << 32
__global__ void __launch_bounds__(128) sp_fill_kernel(const i32 *__restrict__ map, i64 n, i64 ld, i64 n_sub, const u32 *__restrict__ seg,
                                                      const u32 *__restrict__ pos2, const u32 *__restrict__ rowptr,
                                                      u64 *__restrict__ pairs) {
    const int lane = threadIdx.x & 31;
    const i64 sg = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (sg >= n_sub) return;
    const i64 r = sg * 32 + lane;
    const i64 b = sg / SP_ST;
    const int st = (int)(sg % SP_ST);
    const u32 lt = (1u << lane) - 1u;
    u32 dst = r < n ? rowptr[r] : 0u;
#pragma unroll 4
    for (int kk = 0; kk < SP_KK; ++kk) {
        const i32 nb = r < n ? map[(i64)sp_offset(kk) * ld + r] : -1;
        const u32 bal = __ballot_sync(0xFFFFFFFFu, nb >= 0);
        if (bal == 0) continue;
        if (nb >= 0) {
            const u32 q = seg[b * GPC_K3 + kk] + pos2[((size_t)b * SP_KK + kk) * SP_ST + st] + __popc(bal & lt);
            pairs[q] = (u64)(u32)nb | ((u64)dst << 32);
            ++dst;
        }
    }
}

// ---------------------------------------------------------------- kernel 1: stragglers, one warp per (block, offset) segment
// No shared memory: lane (g, t) of an 8-pair MMA tile needs exactly 32 contiguous bytes of pair g's row (channels 8t .. 8t+7 in the
// fragment order of gpc_spconv_pack_weights_frag), so the four lanes of a quad read one 128 B row straight into the B fragments
// (2 x LDG.128 per lane).  Entries are fetched 32 at a time (4 tiles, one coalesced 256 B load) and handed out by shuffles; the rows
// of tile T + 2 are requested before tile T is multiplied (four register slots, indexed statically by the unrolled loop).
__global__ void __launch_bounds__(128) sp_straggler_kernel(const float *__restrict__ x, const uint4 *__restrict__ Wa,
                                                           const u32 *__restrict__ seg, const u64 *__restrict__ pairs, i64 seg0, i64 n_seg,
                                                           int SP_SPLIT, float *__restrict__ contrib) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    // SP_SPLIT warps per segment (chosen by the host from the average segment length): the segments of the offsets next to the
    // centre are 10-50 x longer than the rest; a long one (>= 8 tiles per part) is cut into up to SP_SPLIT tile ranges so that the
    // tail of the launch is not a few warps deep.  Levels with short segments launch one warp per segment.
    const i64 wg = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);
    const i64 i = seg0 + wg / SP_SPLIT;                  // segments [seg0, n_seg) of this launch (a row range = a range of 8192-row blocks)
    const int part = (int)(wg % SP_SPLIT);
    if (i >= n_seg) return;
    const i64 b = i / SP_KK;
    const int kk = (int)(i % SP_KK);
    const u32 p00 = __ldg(seg + b * GPC_K3 + kk);
    const int ntiles_seg = (int)((__ldg(seg + b * GPC_K3 + kk + 1) - p00) >> 3);
    const int nparts = min(SP_SPLIT, (ntiles_seg + 7) / 8);
    if (part >= nparts) return;
    const int t_begin = (int)((i64)ntiles_seg * part / nparts), t_end = (int)((i64)ntiles_seg * (part + 1) / nparts);
    const int ntiles = t_end - t_begin;
    if (ntiles == 0) return;
    const u64 *tile_base = pairs + p00 + (size_t)t_begin * 8;
    auto load_bulk = [&](int k) -> u64 {                 // lane l: entry (tile 4k + l / 8, pair l % 8)
        const int e = k * 32 + lane;
        return e < ntiles * 8 ? __ldg(tile_base + e) : ~0ull;
    };
    u64 eb[2] = {load_bulk(0), load_bulk(1)};            // bulks 2j / 2j + 1, statically indexed (no register hand-over of a load in flight)
    uint4 w1[2][2], w2[2][2];                            // A fragments of W^T[k] (bf16 hi / lo), [mt][u]: once per segment
    {
        const uint4 *wsrc = Wa + (size_t)sp_offset(kk) * 256 + lane;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int u = 0; u < 2; ++u) { w1[mt][u] = __ldg(wsrc + (mt * 2 + u) * 32); w2[mt][u] = __ldg(wsrc + (4 + mt * 2 + u) * 32); }
    }
    float4 xa[4], xc[4];
    u32 dsa[4], dsb[4];
    // an entry is handed out in two steps one tile apart (as in spconv_fwd_v6d_kernel): pick = shuffles, fetch = row loads
    u32 p_nb = 0xFFFFFFFFu, p_da = 0xFFFFFFFFu, p_db = 0xFFFFFFFFu;
    auto pick = [&](u64 ebv, int tl) {                   // neighbour row + destinations of tile `tl` of the bulk in ebv
        p_nb = __shfl_sync(0xFFFFFFFFu, (u32)ebv, tl * 8 + g);
        const u32 hi = (u32)(ebv >> 32);
        p_da = __shfl_sync(0xFFFFFFFFu, hi, tl * 8 + 2 * t);
        p_db = __shfl_sync(0xFFFFFFFFu, hi, tl * 8 + 2 * t + 1);
    };
    auto fetch = [&](float4 &a, float4 &c, u32 &da, u32 &db) {
        da = p_da; db = p_db;
        a = make_float4(0.f, 0.f, 0.f, 0.f); c = a;
        if (p_nb != 0xFFFFFFFFu) {
            const float4 *src = reinterpret_cast<const float4 *>(x + (i64)p_nb * GPC_C + 8 * t);
            a = __ldg(src); c = __ldg(src + 1);
        }
    };
    pick(eb[0], 0); fetch(xa[0], xc[0], dsa[0], dsb[0]);
    if (ntiles > 1) { pick(eb[0], 1); fetch(xa[1], xc[1], dsa[1], dsb[1]); }
    if (ntiles > 2) { pick(eb[0], 2); fetch(xa[2], xc[2], dsa[2], dsb[2]); }
    pick(eb[0], 3);
#pragma unroll 1
    for (int k = 0; 8 * k < ntiles; ++k) {
#pragma unroll
        for (int u8 = 0; u8 < 8; ++u8) {
            const int u = u8 & 3, h = u8 >> 2;
            const int T = 8 * k + u8;
            if (T >= ntiles) break;
            if (T + 3 < ntiles) fetch(xa[(u + 3) & 3], xc[(u + 3) & 3], dsa[(u + 3) & 3], dsb[(u + 3) & 3]);
            if (u == 0) eb[h] = load_bulk(2 * k + h + 2);        // bulk eb[h] was picked completely during the previous four steps
            pick(eb[h ^ 1], u);                                  // tile T + 4
            u32 xf1[2][2], xf2[2][2];
            split_bf16(xa[u].x, xa[u].y, xf1[0][0], xf2[0][0]);
            split_bf16(xa[u].z, xa[u].w, xf1[0][1], xf2[0][1]);
            split_bf16(xc[u].x, xc[u].y, xf1[1][0], xf2[1][0]);
            split_bf16(xc[u].z, xc[u].w, xf1[1][1], xf2[1][1]);
            float d[2][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) { d[mt][0] = d[mt][1] = d[mt][2] = d[mt][3] = 0.f; }
#pragma unroll
            for (int uu = 0; uu < 2; ++uu)
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    sp_mma(d[mt], w1[mt][uu], xf2[uu][0], xf2[uu][1]);
                    sp_mma(d[mt], w2[mt][uu], xf1[uu][0], xf1[uu][1]);
                    sp_mma(d[mt], w1[mt][uu], xf1[uu][0], xf1[uu][1]);
                }
            // d[mt][0] = (co 16mt+g, pair 2t), [1] = (co, pair 2t+1), [2]/[3] = co+8.  A contribution row is stored PERMUTED: float4 g
            // = channels (g, g+8, g+16, g+24), i.e. exactly what lane g holds -> one 16-byte store per pair, 128 contiguous bytes per row
            if (dsa[u] != 0xFFFFFFFFu) reinterpret_cast<float4 *>(contrib)[(size_t)dsa[u] * 8 + g] = make_float4(d[0][0], d[0][2], d[1][0], d[1][2]);
            if (dsb[u] != 0xFFFFFFFFu) reinterpret_cast<float4 *>(contrib)[(size_t)dsb[u] * 8 + g] = make_float4(d[0][1], d[0][3], d[1][1], d[1][3]);
        }
    }
}

// ---------------------------------------------------------------- kernel 2: dense centre product + the rows' contributions
constexpr int SP_ROWS = 32;        // rows per warp (64 rows and 5 CTAs per SM: 0.329 / 0.176 / 0.144 ms on the three sparse levels; 32 rows and 8 CTAs: 0.295 / 0.147 / 0.115)
constexpr int SP_ACC = 36;

__global__ void __launch_bounds__(128, 8) sp_centre_kernel(const float *__restrict__ x, const uint4 *__restrict__ Wa,
                                                        const u32 *__restrict__ rowptr, const float *__restrict__ contrib, i64 row0, i64 n,
                                                        const float *__restrict__ residual, int flags, float *__restrict__ y) {
    __shared__ float acc_all[4][SP_ROWS][SP_ACC];
    float (*acc)[SP_ACC] = acc_all[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const i64 r0 = row0 + ((i64)blockIdx.x * 4 + (threadIdx.x >> 5)) * SP_ROWS;       // rows [row0, n) of this launch
    if (r0 >= n) return;
    uint4 w1[2][2], w2[2][2];
    {
        const uint4 *wsrc = Wa + (size_t)SP_CENTRE * 256 + lane;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int u = 0; u < 2; ++u) { w1[mt][u] = __ldg(wsrc + (mt * 2 + u) * 32); w2[mt][u] = __ldg(wsrc + (4 + mt * 2 + u) * 32); }
    }
    // all 16 row loads of the warp's 64 rows are issued before the first MMA (the tile loop is latency-, not bandwidth-bound otherwise)
    float4 xa[SP_ROWS / 8], xc[SP_ROWS / 8];
#pragma unroll
    for (int j = 0; j < SP_ROWS / 8; ++j) {
        const i64 row = r0 + 8 * j + g;                  // B column g of this 8-row tile: lanes t = 0..3 read its 4 x 32 bytes
        xa[j] = make_float4(0.f, 0.f, 0.f, 0.f); xc[j] = xa[j];
        if (row < n) {
            const float4 *src = reinterpret_cast<const float4 *>(x + row * GPC_C + 8 * t);
            xa[j] = __ldg(src); xc[j] = __ldg(src + 1);
        }
    }
    // first contribution of each of the 64 rows (+ the end of the last one): lane l holds rows l and 32 + l
    const u32 rp_a = __ldg(rowptr + min(r0 + lane, n)), rp_b = __ldg(rowptr + min(r0 + 32 + lane, n));
    const u32 rp_c = __ldg(rowptr + min(r0 + 64, n));
#pragma unroll
    for (int j = 0; j < SP_ROWS / 8; ++j) {
        u32 xf1[2][2], xf2[2][2];
        split_bf16(xa[j].x, xa[j].y, xf1[0][0], xf2[0][0]);
        split_bf16(xa[j].z, xa[j].w, xf1[0][1], xf2[0][1]);
        split_bf16(xc[j].x, xc[j].y, xf1[1][0], xf2[1][0]);
        split_bf16(xc[j].z, xc[j].w, xf1[1][1], xf2[1][1]);
        float d[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) { d[mt][0] = d[mt][1] = d[mt][2] = d[mt][3] = 0.f; }
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                sp_mma(d[mt], w1[mt][u], xf2[u][0], xf2[u][1]);
                sp_mma(d[mt], w2[mt][u], xf1[u][0], xf1[u][1]);
                sp_mma(d[mt], w1[mt][u], xf1[u][0], xf1[u][1]);
            }
        float *a = &acc[8 * j + 2 * t][g], *bq = &acc[8 * j + 2 * t + 1][g];
        a[0] = d[0][0]; a[8] = d[0][2]; a[16] = d[1][0]; a[24] = d[1][2];
        bq[0] = d[0][1]; bq[8] = d[0][3]; bq[16] = d[1][1]; bq[24] = d[1][3];
    }
    __syncwarp();
    // epilogue: eight lanes per row (16 bytes each), 4 rows per warp instruction, SP_H such instructions per step: 16 rows' contribution
    // loads are in flight together (one row at a time with lane = channel waited for rowptr, then for every contribution: 320 us on
    // the 981 K-row level; 8 rows in flight: 160 us)
    const bool relu = (flags & GPC_CONV_RELU) != 0;
    const int grp = lane >> 3, j4 = lane & 7;
    const float4 *c4 = reinterpret_cast<const float4 *>(contrib);
    constexpr int SP_H = 4;
#pragma unroll 1
    for (int it = 0; it < SP_ROWS / (4 * SP_H); ++it) {
        float4 v[SP_H];
        u32 p[SP_H], cnt[SP_H];
        i64 grow[SP_H];
        u32 cmax = 0;
#pragma unroll
        for (int h = 0; h < SP_H; ++h) {
            const int r = it * 4 * SP_H + h * 4 + grp;                   // row within the tile, 0..63
            const u32 pa = __shfl_sync(0xFFFFFFFFu, rp_a, r & 31), pb = __shfl_sync(0xFFFFFFFFu, rp_b, r & 31);
            const u32 qa = __shfl_sync(0xFFFFFFFFu, rp_a, (r + 1) & 31), qb = __shfl_sync(0xFFFFFFFFu, rp_b, (r + 1) & 31);
            p[h] = r < 32 ? pa : pb;
            const u32 pe = r + 1 < 32 ? qa : (r + 1 < 64 ? qb : rp_c);
            grow[h] = r0 + r;
            cnt[h] = grow[h] < n ? pe - p[h] : 0u;
            v[h] = make_float4(acc[r][j4], acc[r][j4 + 8], acc[r][j4 + 16], acc[r][j4 + 24]);     // the contribution rows' channel order
            cmax = max(cmax, cnt[h]);
        }
        for (u32 o = 0; o < cmax; ++o) {                                 // ascending offset per row: fixed summation order
#pragma unroll
            for (int h = 0; h < SP_H; ++h)
                if (o < cnt[h]) {
                    const float4 c = __ldg(c4 + (size_t)(p[h] + o) * 8 + j4);
                    v[h].x += c.x; v[h].y += c.y; v[h].z += c.z; v[h].w += c.w;
                }
        }
#pragma unroll
        for (int h = 0; h < SP_H; ++h) {
            if (grow[h] >= n) continue;
            float *yo = y + grow[h] * GPC_C + j4;                        // lane j4 owns channels j4, j4+8, j4+16, j4+24: 32-byte runs
            if (residual) {
                const float *rr = residual + grow[h] * GPC_C + j4;
                v[h].x += __ldg(rr); v[h].y += __ldg(rr + 8); v[h].z += __ldg(rr + 16); v[h].w += __ldg(rr + 24);
            }
            if (relu) { v[h].x = fmaxf(v[h].x, 0.f); v[h].y = fmaxf(v[h].y, 0.f); v[h].z = fmaxf(v[h].z, 0.f); v[h].w = fmaxf(v[h].w, 0.f); }
            yo[0] = v[h].x; yo[8] = v[h].y; yo[16] = v[h].z; yo[24] = v[h].w;
        }
    }
}

struct SpWs {
    u32 *cnt2, *tot8, *rowcnt;
    void *scan_ws;
    size_t total;
};
SpWs sp_ws_layout(void *ws, i64 n) {
    SpWs L;
    const i64 nb = n > 0 ? (n + SP_TB - 1) / SP_TB : 1;
    size_t off = 0;
    char *b = (char *)ws;
    L.cnt2 = (u32 *)(b + off); off += align_up((size_t)nb * SP_KK * SP_ST * 4, 256);
    L.tot8 = (u32 *)(b + off); off += align_up((size_t)nb * GPC_K3 * 4, 256);
    L.rowcnt = (u32 *)(b + off); off += align_up((size_t)(n > 0 ? n : 1) * 4, 256);
    const i64 big = n > nb * GPC_K3 ? n : nb * GPC_K3;
    L.scan_ws = b + off; off += align_up(scan_workspace_bytes<u32>(big), 256);
    L.total = off;
    return L;
}

}  // namespace

extern "C" int64_t gpc_kmap_sparse_segments(int64_t n) { return (n > 0 ? (n + SP_TB - 1) / SP_TB : 0) * GPC_K3; }
extern "C" size_t gpc_kmap_sparse_workspace_bytes(int64_t n) { return sp_ws_layout(nullptr, n).total; }

// map: dense offset-major map [125][n] (gpc_kmap_dense).  seg: u32[segments + 1], rowptr: u32[n + 1], totals: device u32[2] =
// {stream entries (padded to 8 per segment), true stragglers}.  ws is shared with gpc_kmap_sparse_fill (keep it alive).
// map: rows [0, n) of a dense map whose offset planes are ld ints apart (ld = n: a whole level; ld > n: a row range, map advanced
// to its first row)
static int sparse_count(const int32_t *map, int64_t n, int64_t ld, uint32_t *seg, uint32_t *rowptr, uint32_t *totals, void *ws,
                        size_t ws_bytes, void *stream) {
    cudaStream_t st = as_stream(stream);
    if (n <= 0) { GPC_CUDA_CHECK(cudaMemsetAsync(totals, 0, 8, st)); return GPC_OK; }
    SpWs L = sp_ws_layout(ws, n);
    GPC_REQUIRE(ws && ws_bytes >= L.total, GPC_ENOSPC, "workspace too small");
    GPC_REQUIRE(n * (int64_t)SP_KK < (1ll << 32), GPC_EINVAL, "level too large for 32-bit straggler indices");
    const i64 nb = (n + SP_TB - 1) / SP_TB, n_sub = (n + 31) / 32, n_seg = nb * SP_KK;
    GPC_CUDA_CHECK(cudaMemsetAsync(L.cnt2, 0, (size_t)nb * SP_KK * SP_ST * 4, st));        // sub-tiles past the end of the last block
    GPC_CUDA_CHECK(cudaMemsetAsync(L.tot8, 0, (size_t)nb * GPC_K3 * 4, st));
    sp_count_kernel<<<cdiv(n_sub, 4), 128, 0, st>>>(map, n, ld, n_sub, L.cnt2, L.rowcnt);
    GPC_LAUNCH_CHECK();
    sp_segment_kernel<<<cdiv(n_seg, 4), 128, 0, st>>>(L.cnt2, n_seg, L.tot8);
    GPC_LAUNCH_CHECK();
    PtrLoad<u32> p1{L.tot8};
    int rc = device_exclusive_scan<u32, PtrLoad<u32>>(p1, nb * GPC_K3, seg, L.scan_ws, st);
    if (rc) return rc;
    PtrLoad<u32> p2{L.rowcnt};
    rc = device_exclusive_scan<u32, PtrLoad<u32>>(p2, n, rowptr, L.scan_ws, st);
    if (rc) return rc;
    sp_totals_kernel<<<1, 1, 0, st>>>(seg, nb * GPC_K3, rowptr, n, totals);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}
static int sparse_fill(const int32_t *map, int64_t n, int64_t ld, const uint32_t *seg, const uint32_t *rowptr, const void *ws,
                       uint64_t *pairs, int64_t n_entries, void *stream) {
    if (n <= 0 || n_entries <= 0) return GPC_OK;
    cudaStream_t st = as_stream(stream);
    SpWs L = sp_ws_layout(const_cast<void *>(ws), n);
    GPC_CUDA_CHECK(cudaMemsetAsync(pairs, 0xFF, (size_t)n_entries * 8, st));
    const i64 n_sub = (n + 31) / 32;
    sp_fill_kernel<<<cdiv(n_sub, 4), 128, 0, st>>>(map, n, ld, n_sub, seg, L.cnt2, rowptr, pairs);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

extern "C" int gpc_kmap_sparse_count(const int32_t *map, int64_t n, uint32_t *seg, uint32_t *rowptr, uint32_t *totals, void *ws,
                                     size_t ws_bytes, void *stream) {
    return sparse_count(map, n, n, seg, rowptr, totals, ws, ws_bytes, stream);
}
extern "C" int gpc_kmap_sparse_fill(const int32_t *map, int64_t n, const uint32_t *seg, const uint32_t *rowptr, const void *ws,
                                    uint64_t *pairs, int64_t n_entries, void *stream) {
    return sparse_fill(map, n, n, seg, rowptr, ws, pairs, n_entries, stream);
}
// the sparse map of the rows [row0, row1) of a level of n_level rows: blocks start at row0, rowptr / dst are range-local, neighbour
// indices stay the level's rows; seg, rowptr and ws are sized for the range's row count (gpc_kmap_sparse_segments(row1 - row0), ...)
extern "C" int gpc_kmap_sparse_count_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, uint32_t *seg,
                                           uint32_t *rowptr, uint32_t *totals, void *ws, size_t ws_bytes, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    return sparse_count(map + row0, row1 - row0, n_level, seg, rowptr, totals, ws, ws_bytes, stream);
}
extern "C" int gpc_kmap_sparse_fill_range(const int32_t *map, int64_t n_level, int64_t row0, int64_t row1, const uint32_t *seg,
                                          const uint32_t *rowptr, const void *ws, uint64_t *pairs, int64_t n_entries, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    return sparse_fill(map + row0, row1 - row0, n_level, seg, rowptr, ws, pairs, n_entries, stream);
}

// y[o,:] = act( W[centre]^T x[o,:] + sum over the row's stragglers, ascending offset (+ residual[o,:]) ).  Wa = this conv's slice of
// gpc_spconv_pack_weights_frag; contrib = caller scratch of max(stragglers, 1) * 32 floats (fully rewritten by every call).
// xg: the rows the stragglers gather (x[nbr]); x: the centre rows, indexed like y (the same array but for a range of a union level).
static int sp_fwd_rows(const float *xg, const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, const uint32_t *rowptr, int64_t n,
                       int64_t n_entries, float *contrib, const float *residual, int flags, float *y, int64_t row0, int64_t row1,
                       void *stream) {
    if (n <= 0 || row1 <= row0) return GPC_OK;
    GPC_REQUIRE(x != y && xg != y, GPC_EINVAL, "conv is out of place (rows are gathered from x while y is written)");
    GPC_REQUIRE(row0 >= 0 && row1 <= n && row0 % SP_TB == 0 && (row1 % SP_TB == 0 || row1 == n), GPC_EINVAL,
                "row range must be made of whole 8192-row blocks");
    cudaStream_t st = as_stream(stream);
    const i64 nb = (n + SP_TB - 1) / SP_TB, n_seg = nb * SP_KK;
    const i64 seg0 = row0 / SP_TB * SP_KK, seg1 = (row1 + SP_TB - 1) / SP_TB * SP_KK;
    if (n_entries > 0) {
        const int split = n_entries >= 256 * n_seg ? 8 : (n_entries >= 64 * n_seg ? 4 : 1);      // by the level, not by the range
        sp_straggler_kernel<<<cdiv((seg1 - seg0) * split, 4), 128, 0, st>>>(xg, (const uint4 *)Wa, seg, pairs, seg0, seg1, split, contrib);
        GPC_LAUNCH_CHECK();
    }
    sp_centre_kernel<<<cdiv(row1 - row0, 4 * SP_ROWS), 128, 0, st>>>(x, (const uint4 *)Wa, rowptr, contrib, row0, row1, residual, flags, y);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}
extern "C" int gpc_spconv_sparse_fwd(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs,
                                     const uint32_t *rowptr, int64_t n, int64_t n_entries, float *contrib, const float *residual,
                                     int flags, float *y, void *stream) {
    return sp_fwd_rows(x, x, Wa, seg, pairs, rowptr, n, n_entries, contrib, residual, flags, y, 0, n, stream);
}
// The same conv for the output rows [row0, row1) only (whole 8192-row blocks; row1 may be n): x, y, residual, contrib and the map
// are the level's, rows outside the range are neither read as outputs nor written.  Used by the decoder's stage wavefront.
extern "C" int gpc_spconv_sparse_fwd_rows(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs,
                                          const uint32_t *rowptr, int64_t n, int64_t n_entries, float *contrib,
                                          const float *residual, int flags, float *y, int64_t row0, int64_t row1, void *stream) {
    return sp_fwd_rows(x, x, Wa, seg, pairs, rowptr, n, n_entries, contrib, residual, flags, y, row0, row1, stream);
}
// The conv of one scene of a batch union level: output rows [row0, row1) of a level of n_level rows with the sparse map of that range
// (gpc_kmap_sparse_count_range): the stragglers gather the level's rows x[nbr], the centre product and the outputs are the range's
// rows.  x, y and residual are the level's arrays.
extern "C" int gpc_spconv_sparse_fwd_range(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs,
                                           const uint32_t *rowptr, int64_t n_level, int64_t row0, int64_t row1, int64_t n_entries,
                                           float *contrib, const float *residual, int flags, float *y, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    GPC_REQUIRE(x != y, GPC_EINVAL, "conv is out of place (rows are gathered from x while y is written)");
    const int64_t n = row1 - row0;
    return sp_fwd_rows(x, x + row0 * GPC_C, Wa, seg, pairs, rowptr, n, n_entries, contrib, residual ? residual + row0 * GPC_C : nullptr,
                       flags, y + row0 * GPC_C, 0, n, stream);
}

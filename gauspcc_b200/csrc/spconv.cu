// spconv.cu -- submanifold sparse convolution forward, K=5, C=32 -> 32, bias-less (a-7, a-10, a-12).
//
// Replaces torchsparse's implicit-GEMM conv behind spnn.Conv3d(32,32,5)
// (src/ai_pcc/GausPcgc/kit/nn.py:14-16, network_ue_4stage_conv.py:18-61):
//     y[o,:] = act( sum_{k : nbr_k(o) exists} x[nbr_k(o),:] . W[k]  (+ residual[o,:]) )
//
// This file: the mma.sync kernels (v6: one warp per tile of 8..64 rows with a cp.async gather ring, optionally the 125 offsets
// split over the warps of a CTA; v6d: the gathered rows go straight into the MMA fragments).  They run the levels below 150 K rows
// and are the comparison point of the tcgen05 / TMA kernel (spconv_um.cu), which runs the big dense levels; the sparse big levels
// run spconv_sparse.cu.  All of them are output-stationary with fp32 accumulators and add a row's offsets in ascending order
// (one fixed accumulation order => the encoder and the decoder produce bit-identical features).
#include "common.cuh"

// (The FFMA / FFMA2 kernels v1-v3, the first mma.sync kernels v4 / v5 and the experiments v7 / v8 of round 1 are gone: the mma.sync
// conv below (v6 / v6d) superseded all of them; their measurements are kept in profiles/r01_*.md.)

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const u32 d = (u32)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }


// =====================================================================================================
// v5: as v4 but with the roles of the MMA operands swapped: W^T[k] (32 co x 32 ci) is the A operand (held
// in registers per offset, loaded with 8 x LDG.128 from a fragment-ordered pack), the gathered rows are the
// B operand (n = 8 pairs per MMA tile).  Padding granularity drops from 16 to 8 pairs per (sub-tile,
// offset) and the D fragment gives each lane (co, pair) scalars whose smem read-modify-write is one
// conflict-free wavefront for consecutive rows.  Leaner integer path: hardware cvt.rn.bf16x2 for the
// hi/lo split, a compacted list of non-empty offsets, L1 prefetch of the next offset's W.
// =====================================================================================================
// Wa [n_kernels*125][2 part][2 mt][2 u][32 lane] uint4 = (a0,a1,a2,a3) of mma.m16n8k16 for A = W^T:
//   lane (g,t): a0 = (co 16mt+g,   ch 8t+4u+{0,1}), a1 = (co 16mt+g+8, same ch),
//               a2 = (co 16mt+g,   ch 8t+4u+{2,3}), a3 = (co 16mt+g+8, same ch);  part 0 = bf16 hi, 1 = bf16 lo
__global__ void pack_weights_frag_kernel(const float *__restrict__ W, uint4 *__restrict__ Wa, int n_kernels) {
    i64 gi = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= (i64)n_kernels * GPC_K3 * 8 * 32) return;
    const int lane = (int)(gi & 31), u = (int)((gi >> 5) & 1), mt = (int)((gi >> 6) & 1), part = (int)((gi >> 7) & 1);
    const i64 k = gi >> 8;
    const int g = lane >> 2, t = lane & 3;
    const float *src = W + k * (GPC_C * GPC_C);
    u32 out[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int co = 16 * mt + g + 8 * (r & 1);
        const int ch = 8 * t + 4 * u + 2 * (r >> 1);
        u32 v = 0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const float w = src[(ch + e) * GPC_C + co];
            const float w1 = bf16_round(w);
            const float pv = part == 0 ? w1 : bf16_round(w - w1);
            v |= (__float_as_uint(pv) >> 16) << (16 * e);
        }
        out[r] = v;
    }
    Wa[gi] = make_uint4(out[0], out[1], out[2], out[3]);
}
extern "C" int gpc_spconv_pack_weights_frag(const float *W, int n_kernels, void *Wa, void *stream) {
    const i64 total = (i64)n_kernels * GPC_K3 * 8 * 32;
    pack_weights_frag_kernel<<<cdiv(total, 256), 256, 0, as_stream(stream)>>>(W, (uint4 *)Wa, n_kernels);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

__device__ __forceinline__ void mma_bf16_a4(float (&d)[4], const uint4 &a, u32 b0, u32 b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}


// =====================================================================================================
// v6: v5's contraction, re-plumbed for instruction count and latency.
//   * the pair stream is padded per (sub-tile, offset) to whole 8-entry MMA tiles (kmap pad = 8), so the
//     kernel walks a flat list of tiles: no offset iterators, no window bookkeeping; a tile's offset is the
//     k field of its first entry;
//   * explicit software pipeline inside the warp (in-order issue): while the 12 HMMAs of tile c run, the raw
//     inputs / row ids / W fragments of tile c+1 are already being loaded and are converted before the
//     read-modify-write of tile c -- no instruction waits on a load issued in the same iteration;
//   * tile c+D's rows are gathered by cp.async (2 x 16 B per lane), its entry was prefetched to a register
//     one iteration earlier.
// =====================================================================================================
constexpr int SC6_XS = 36;
constexpr int SC6_ACC = 36;

template <int TW, int D>
struct Sc6Smem {
    float acc[TW][SC6_ACC];
    float xs[D][8][SC6_XS];
    u32 rowk[D][12];              // [0..7] row of each pair in the tile (0xFFFF = padding), [8] = offset k
};

// G > 1 ("split offsets"): the CTA has G warps on the SAME TW rows; warp w contracts the offsets [125 w / G, 125 (w+1) / G) into its
// own accumulators and the partial sums are added in warp order at the end (still one fixed summation order per row).  The coarse
// octree levels have a few hundred to a few thousand rows with 35-70 neighbours each: one warp per 8 rows walked ~100 dependent
// 8-pair tiles and every such launch took ~70 us whatever its size (launch list, profiles/r01_step_breakdown.md).
template <int TW, int D, int G>
__global__ void __launch_bounds__(32 * G) spconv_fwd_v6_kernel(const float *__restrict__ x, const uint4 *__restrict__ Wa,
                                                               const u32 *__restrict__ seg_g, const u64 *__restrict__ pairs, i64 n,
                                                               const float *__restrict__ residual, int flags, float *__restrict__ y) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int wid = G > 1 ? (int)(threadIdx.x >> 5) : 0;
    Sc6Smem<TW, D> &s = reinterpret_cast<Sc6Smem<TW, D> *>(smem_raw)[wid];
    const int lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const i64 st = blockIdx.x;
    const i64 r0 = st * TW;
    const int rows = (int)min((i64)TW, n - r0);
    const int kb = GPC_K3 * wid / G, ke = GPC_K3 * (wid + 1) / G;
    const u32 p_begin = __ldg(seg_g + st * (GPC_K3 + 1) + kb);
    const int ntiles = (int)((__ldg(seg_g + st * (GPC_K3 + 1) + ke) - p_begin) >> 3);
    const u64 *tile_base = pairs + p_begin;

    for (int i = lane; i < TW * SC6_ACC / 4; i += 32) reinterpret_cast<float4 *>(&s.acc[0][0])[i] = make_float4(0.f, 0.f, 0.f, 0.f);

    const int er = lane & 7, epg = lane >> 3;          // this lane copies row `er` of a tile, 32-byte piece group `epg`
    auto load_entry = [&](int tile) -> u64 {
        return tile < ntiles ? __ldg(tile_base + (i64)tile * 8 + er) : 0xFFFFFFFFFFFFFFFFull;
    };
    auto issue_tile = [&](int tile, u64 e) {             // gather rows of `tile` into ring slot tile % D
        if (tile < ntiles) {
            const int slot = tile % D;
            const u32 nb = (u32)e;
            if (nb != 0xFFFFFFFFu) {
                const float *src = x + (i64)nb * GPC_C + epg * 8;
                cp_async16(&s.xs[slot][er][epg * 8], src);
                cp_async16(&s.xs[slot][er][epg * 8 + 4], src + 4);
            }
            if (lane < 8) s.rowk[slot][lane] = (u32)(e >> 32) & 0xFFFFu;
            if (lane == 0) s.rowk[slot][8] = (u32)(e >> 48);
        }
    };

    // prologue: tiles 0..D-1 in flight, entry of tile D in a register
    u64 e_next = load_entry(0);
#pragma unroll 1
    for (int i = 0; i < D; ++i) {
        const u64 e = e_next;
        e_next = load_entry(i + 1);
        issue_tile(i, e);
        cp_async_commit();
    }
    cp_async_wait<D - 1>();                              // tile 0 landed
    __syncwarp();

    uint4 w1[2][2], w2[2][2];                            // A fragments of W^T[k] (bf16 hi / lo), [mt][u]
    u32 xf1[2][2], xf2[2][2];                            // B fragments of the current tile (bf16 hi / lo), [u][b0/b1]
    u32 row_a = 0xFFFFu, row_b = 0xFFFFu;                // accumulator rows of pairs 2t, 2t+1 of the current tile
    u32 k_cur = 0xFFFFFFFFu;
    if (ntiles > 0) {
        const float4 xa = *reinterpret_cast<const float4 *>(&s.xs[0][g][8 * t]);
        const float4 xc = *reinterpret_cast<const float4 *>(&s.xs[0][g][8 * t + 4]);
        row_a = s.rowk[0][2 * t]; row_b = s.rowk[0][2 * t + 1];
        k_cur = s.rowk[0][8];
        const uint4 *wsrc = Wa + (size_t)k_cur * 256 + lane;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int u = 0; u < 2; ++u) { w1[mt][u] = __ldg(wsrc + (mt * 2 + u) * 32); w2[mt][u] = __ldg(wsrc + (4 + mt * 2 + u) * 32); }
        split_bf16(xa.x, xa.y, xf1[0][0], xf2[0][0]);
        split_bf16(xa.z, xa.w, xf1[0][1], xf2[0][1]);
        split_bf16(xc.x, xc.y, xf1[1][0], xf2[1][0]);
        split_bf16(xc.z, xc.w, xf1[1][1], xf2[1][1]);
    }

#pragma unroll 1
    for (int c = 0; c < ntiles; ++c) {
        // A. tiles <= c+1 have landed
        cp_async_wait<D - 2>();
        __syncwarp();
        // B. refill the ring slot tile c just vacated (its data lives in registers since the previous iteration)
        {
            const u64 e = e_next;
            e_next = load_entry(c + D + 1);
            issue_tile(c + D, e);
            cp_async_commit();
        }
        // C. loads for tile c+1 (raw rows, accumulator rows, offset, W if it changes)
        const bool more = c + 1 < ntiles;
        const int ns = (c + 1) % D;
        float4 xa = make_float4(0.f, 0.f, 0.f, 0.f), xc = xa;
        u32 nrow_a = 0xFFFFu, nrow_b = 0xFFFFu, k_next = k_cur;
        if (more) {
            xa = *reinterpret_cast<const float4 *>(&s.xs[ns][g][8 * t]);
            xc = *reinterpret_cast<const float4 *>(&s.xs[ns][g][8 * t + 4]);
            nrow_a = s.rowk[ns][2 * t]; nrow_b = s.rowk[ns][2 * t + 1];
            k_next = s.rowk[ns][8];
        }
        uint4 n1[2][2], n2[2][2];
        const bool newk = k_next != k_cur;               // warp-uniform
        if (newk) {
            const uint4 *wsrc = Wa + (size_t)k_next * 256 + lane;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int u = 0; u < 2; ++u) { n1[mt][u] = __ldg(wsrc + (mt * 2 + u) * 32); n2[mt][u] = __ldg(wsrc + (4 + mt * 2 + u) * 32); }
        }
        // D. contraction of tile c
        float d[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) { d[mt][0] = d[mt][1] = d[mt][2] = d[mt][3] = 0.f; }
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                mma_bf16_a4(d[mt], w1[mt][u], xf2[u][0], xf2[u][1]);
                mma_bf16_a4(d[mt], w2[mt][u], xf1[u][0], xf1[u][1]);
                mma_bf16_a4(d[mt], w1[mt][u], xf1[u][0], xf1[u][1]);
            }
        // E. convert tile c+1's inputs while the HMMAs drain
        u32 y1[2][2], y2[2][2];
        split_bf16(xa.x, xa.y, y1[0][0], y2[0][0]);
        split_bf16(xa.z, xa.w, y1[0][1], y2[0][1]);
        split_bf16(xc.x, xc.y, y1[1][0], y2[1][0]);
        split_bf16(xc.z, xc.w, y1[1][1], y2[1][1]);
        // F. scatter-add tile c: d[mt][0] = (co 16mt+g, pair 2t), [1] = (co, pair 2t+1), [2]/[3] = co+8.  The two pairs of a lane
        // belong to ONE offset, hence to different rows: all eight loads are issued before the first store (written as two
        // separate read-modify-writes the compiler has to assume they alias and serialises load - add - store - load - add - store)
        {
            const bool va = row_a != 0xFFFFu, vb = row_b != 0xFFFFu;
            float *pa = &s.acc[va ? row_a : 0u][g], *pb = &s.acc[vb ? row_b : 0u][g];
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
            if (va) { a0 = pa[0]; a1 = pa[8]; a2 = pa[16]; a3 = pa[24]; }
            if (vb) { b0 = pb[0]; b1 = pb[8]; b2 = pb[16]; b3 = pb[24]; }
            a0 += d[0][0]; a1 += d[0][2]; a2 += d[1][0]; a3 += d[1][2];
            b0 += d[0][1]; b1 += d[0][3]; b2 += d[1][1]; b3 += d[1][3];
            if (va) { pa[0] = a0; pa[8] = a1; pa[16] = a2; pa[24] = a3; }
            if (vb) { pb[0] = b0; pb[8] = b1; pb[16] = b2; pb[24] = b3; }
        }
        // G. rotate
#pragma unroll
        for (int u = 0; u < 2; ++u) { xf1[u][0] = y1[u][0]; xf1[u][1] = y1[u][1]; xf2[u][0] = y2[u][0]; xf2[u][1] = y2[u][1]; }
        row_a = nrow_a; row_b = nrow_b;
        if (newk) {
            k_cur = k_next;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int u = 0; u < 2; ++u) { w1[mt][u] = n1[mt][u]; w2[mt][u] = n2[mt][u]; }
        }
    }
    cp_async_wait<0>();
    __syncwarp();
    if (G > 1) __syncthreads();
    const bool relu = (flags & GPC_CONV_RELU) != 0;
    for (int r = wid; r < rows; r += G) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < G; ++w) v += reinterpret_cast<Sc6Smem<TW, D> *>(smem_raw)[w].acc[r][lane];      // warp order: offsets ascending
        if (residual) v += __ldg(residual + (r0 + r) * GPC_C + lane);
        if (relu) v = fmaxf(v, 0.f);
        y[(r0 + r) * GPC_C + lane] = v;
    }
}

// ---- v6d: v6 without the shared-memory gather ring.  Lane (g, t) of an 8-pair tile needs exactly the 32 contiguous bytes
// [8t, 8t+8) of pair g's row, so the four lanes of a quad read one 128 B row straight into the B fragments (2 x LDG.128 per lane):
// no cp.async, no staging, no LDS, no wait_group / syncwarp per tile.  Entries come 32 at a time (4 tiles, one coalesced 256 B load)
// and are handed out by shuffles; the rows of tile T + 3 are requested before tile T is multiplied (four register slots indexed
// statically by the unrolled loop), W^T[k] of tile T + 1 while tile T is multiplied.  Accumulators and their fixed order as in v6.
template <int TW>
__global__ void __launch_bounds__(32) spconv_fwd_v6d_kernel(const float *__restrict__ x, const uint4 *__restrict__ Wa,
                                                            const u32 *__restrict__ seg_g, const u64 *__restrict__ pairs, i64 n,
                                                            const float *__restrict__ residual, int flags, float *__restrict__ y,
                                                            i64 tile0) {
    __shared__ float acc[TW][SC6_ACC];
    const int lane = threadIdx.x;
    const int g = lane >> 2, t = lane & 3;
    const i64 st = tile0 + blockIdx.x;                   // tiles [tile0, tile0 + gridDim.x) of the level
    const i64 r0 = st * TW;
    const int rows = (int)min((i64)TW, n - r0);
    const u32 p_begin = __ldg(seg_g + st * (GPC_K3 + 1));
    const int ntiles = (int)((__ldg(seg_g + st * (GPC_K3 + 1) + GPC_K3) - p_begin) >> 3);
    const u64 *tile_base = pairs + p_begin;
    for (int i = lane; i < TW * SC6_ACC / 4; i += 32) reinterpret_cast<float4 *>(&acc[0][0])[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    auto load_bulk = [&](int k) -> u64 {                 // lane l: entry (tile 4k + l / 8, pair l % 8)
        const int e = k * 32 + lane;
        return e < ntiles * 8 ? __ldg(tile_base + e) : ~0ull;
    };
    u64 eb[2] = {load_bulk(0), load_bulk(1)};   // bulks 2j / 2j + 1: statically indexed (a register hand-over would wait for every load in flight)
    float4 xa[4], xc[4];
    u32 rwa[4], rwb[4], kof[4];
    // an entry is handed out in two steps one tile apart, so that nothing waits for a shuffle: pick (shuffles into p_*), then
    // fetch (row loads from the picked neighbour index, bookkeeping into the tile's slot)
    u32 p_nb = 0xFFFFFFFFu, p_ra = 0xFFFFu, p_rb = 0xFFFFu, p_kk = 0;
    auto pick = [&](u64 ebv, int tl) {
        p_nb = __shfl_sync(0xFFFFFFFFu, (u32)ebv, tl * 8 + g);
        const u32 hi = (u32)(ebv >> 32);
        p_ra = __shfl_sync(0xFFFFFFFFu, hi, tl * 8 + 2 * t) & 0xFFFFu;             // padding entries: 0xFFFF
        p_rb = __shfl_sync(0xFFFFFFFFu, hi, tl * 8 + 2 * t + 1) & 0xFFFFu;
        p_kk = __shfl_sync(0xFFFFFFFFu, hi, tl * 8) >> 16;                         // entry 0 of a tile is always a real pair
    };
    auto fetch = [&](float4 &a, float4 &c, u32 &ra, u32 &rb, u32 &kk) {
        ra = p_ra; rb = p_rb; kk = p_kk;
        a = make_float4(0.f, 0.f, 0.f, 0.f); c = a;
        if (p_nb != 0xFFFFFFFFu) {
            const float4 *src = reinterpret_cast<const float4 *>(x + (i64)p_nb * GPC_C + 8 * t);
            a = __ldg(src); c = __ldg(src + 1);
        }
    };
    auto load_w = [&](uint4 (&a1)[2][2], uint4 (&a2)[2][2], u32 k) {
        const uint4 *wsrc = Wa + (size_t)k * 256 + lane;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int u = 0; u < 2; ++u) { a1[mt][u] = __ldg(wsrc + (mt * 2 + u) * 32); a2[mt][u] = __ldg(wsrc + (4 + mt * 2 + u) * 32); }
    };
    uint4 w1[2][2], w2[2][2];
    u32 k_cur = 0xFFFFFFFFu;
    if (ntiles > 0) {
        pick(eb[0], 0); fetch(xa[0], xc[0], rwa[0], rwb[0], kof[0]);
        if (ntiles > 1) { pick(eb[0], 1); fetch(xa[1], xc[1], rwa[1], rwb[1], kof[1]); }
        if (ntiles > 2) { pick(eb[0], 2); fetch(xa[2], xc[2], rwa[2], rwb[2], kof[2]); }
        pick(eb[0], 3);
        k_cur = kof[0];
        load_w(w1, w2, k_cur);
    }
#pragma unroll 1
    for (int kb = 0; 8 * kb < ntiles; ++kb) {
#pragma unroll
        for (int u8 = 0; u8 < 8; ++u8) {
            const int u = u8 & 3, h = u8 >> 2;
            const int T = 8 * kb + u8;
            if (T >= ntiles) break;
            // tile T - 1's slot is free: its fragments were converted and its rows / offset consumed in the previous step
            if (T + 3 < ntiles) fetch(xa[(u + 3) & 3], xc[(u + 3) & 3], rwa[(u + 3) & 3], rwb[(u + 3) & 3], kof[(u + 3) & 3]);
            // bulk eb[h] (tiles T .. T + 3) was picked completely during the previous four steps: fetch the bulk after the next one
            if (u == 0) eb[h] = load_bulk(2 * kb + h + 2);
            pick(eb[h ^ 1], u);                          // tile T + 4
            // W of the next tile if its offset differs (warp-uniform): in flight during this tile's MMAs.  (Requesting it as soon as
            // the offset shows up in the 3-tile look-ahead window was measured 20 % SLOWER: the fragments then live across iterations.)
            const u32 k_next = T + 1 < ntiles ? kof[(u + 1) & 3] : k_cur;
            const bool newk = k_next != k_cur;
            uint4 n1[2][2], n2[2][2];
            if (newk) load_w(n1, n2, k_next);
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
                    mma_bf16_a4(d[mt], w1[mt][uu], xf2[uu][0], xf2[uu][1]);
                    mma_bf16_a4(d[mt], w2[mt][uu], xf1[uu][0], xf1[uu][1]);
                    mma_bf16_a4(d[mt], w1[mt][uu], xf1[uu][0], xf1[uu][1]);
                }
            {   // scatter-add: the two pairs of a lane are different rows; all loads before the first store
                const u32 row_a = rwa[u], row_b = rwb[u];
                const bool va = row_a != 0xFFFFu, vb = row_b != 0xFFFFu;
                float *pa = &acc[va ? row_a : 0u][g], *pb = &acc[vb ? row_b : 0u][g];
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
                if (va) { a0 = pa[0]; a1 = pa[8]; a2 = pa[16]; a3 = pa[24]; }
                if (vb) { b0 = pb[0]; b1 = pb[8]; b2 = pb[16]; b3 = pb[24]; }
                a0 += d[0][0]; a1 += d[0][2]; a2 += d[1][0]; a3 += d[1][2];
                b0 += d[0][1]; b1 += d[0][3]; b2 += d[1][1]; b3 += d[1][3];
                if (va) { pa[0] = a0; pa[8] = a1; pa[16] = a2; pa[24] = a3; }
                if (vb) { pb[0] = b0; pb[8] = b1; pb[16] = b2; pb[24] = b3; }
            }
            __syncwarp();                                // the next tile may touch the same accumulator rows from other lanes
            if (newk) {
                k_cur = k_next;
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int uu = 0; uu < 2; ++uu) { w1[mt][uu] = n1[mt][uu]; w2[mt][uu] = n2[mt][uu]; }
            }
        }
    }
    __syncwarp();
    const bool relu = (flags & GPC_CONV_RELU) != 0;
    for (int r = 0; r < rows; ++r) {
        float v = acc[r][lane];
        if (residual) v += __ldg(residual + (r0 + r) * GPC_C + lane);
        if (relu) v = fmaxf(v, 0.f);
        y[(r0 + r) * GPC_C + lane] = v;
    }
}

template <int TW, int D, int G = 1>
static int launch_spconv_v6(const float *x, const void *Wa, const u32 *seg, const u64 *pairs, i64 n, const float *residual,
                            int flags, float *y, cudaStream_t st) {
    static bool configured = false;
    const size_t smem = sizeof(Sc6Smem<TW, D>) * G;
    if (!configured) {
        GPC_CUDA_CHECK(cudaFuncSetAttribute(spconv_fwd_v6_kernel<TW, D, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    const i64 tiles = (n + TW - 1) / TW;
    spconv_fwd_v6_kernel<TW, D, G><<<(unsigned)tiles, 32 * G, smem, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// Wa from gpc_spconv_pack_weights_frag; pair stream built with pad = 8.  The (variant, tile_rows) pairs the codec runs
// (GausPcgcCodec._v6_config) plus 42 @ 64, the reference v6d is checked against; the other variants tried in round 1 are in git history.
extern "C" int gpc_spconv_fwd_v6(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, int64_t n,
                                 int tile_rows, const float *residual, int flags, float *y, int variant, void *stream) {
    if (n <= 0) return GPC_OK;
    GPC_REQUIRE(x != y, GPC_EINVAL, "conv is out of place (rows are gathered from x while y is written)");
    cudaStream_t st = as_stream(stream);
    if (variant == 42) {
        if (tile_rows == 64) return launch_spconv_v6<64, 4>(x, Wa, seg, pairs, n, residual, flags, y, st);
    } else if (variant == 46) {          // split offsets over 8 warps
        if (tile_rows == 16) return launch_spconv_v6<16, 4, 8>(x, Wa, seg, pairs, n, residual, flags, y, st);
        if (tile_rows == 32) return launch_spconv_v6<32, 4, 8>(x, Wa, seg, pairs, n, residual, flags, y, st);
    } else if (variant == 48) {          // v6d: rows straight into the MMA fragments (no shared-memory gather ring)
        const i64 tiles = (n + tile_rows - 1) / tile_rows;
        if (tile_rows == 64) { spconv_fwd_v6d_kernel<64><<<(unsigned)tiles, 32, 0, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y, 0); GPC_LAUNCH_CHECK(); return GPC_OK; }
        if (tile_rows == 32) { spconv_fwd_v6d_kernel<32><<<(unsigned)tiles, 32, 0, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y, 0); GPC_LAUNCH_CHECK(); return GPC_OK; }
        if (tile_rows == 128) { spconv_fwd_v6d_kernel<128><<<(unsigned)tiles, 32, 0, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y, 0); GPC_LAUNCH_CHECK(); return GPC_OK; }
    } else if (variant == 47) {          // split offsets over 16 warps
        if (tile_rows == 8) return launch_spconv_v6<8, 4, 16>(x, Wa, seg, pairs, n, residual, flags, y, st);
    }
    gpc_set_error("unsupported conv v6 variant %d / tile_rows %d", variant, tile_rows);
    return GPC_EINVAL;
}

// v6d (variant 48) for the output rows [row0, row1) only: row0 a multiple of tile_rows, row1 a multiple of tile_rows or n.  x, y,
// residual and the pair stream are the level's.  Used by the decoder's stage wavefront (codec.py).
extern "C" int gpc_spconv_fwd_v6_rows(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, int64_t n,
                                      int tile_rows, const float *residual, int flags, float *y, int variant, int64_t row0,
                                      int64_t row1, void *stream) {
    if (n <= 0 || row1 <= row0) return GPC_OK;
    GPC_REQUIRE(x != y, GPC_EINVAL, "conv is out of place (rows are gathered from x while y is written)");
    GPC_REQUIRE(variant == 48 && (tile_rows == 128 || tile_rows == 64 || tile_rows == 32), GPC_EINVAL, "row ranges: v6d (variant 48) only");
    GPC_REQUIRE(row0 >= 0 && row1 <= n && row0 % tile_rows == 0 && (row1 % tile_rows == 0 || row1 == n), GPC_EINVAL,
                "row range must be made of whole tiles");
    cudaStream_t st = as_stream(stream);
    const i64 tile0 = row0 / tile_rows, tiles = (row1 - row0 + tile_rows - 1) / tile_rows;
    if (tile_rows == 128) spconv_fwd_v6d_kernel<128><<<(unsigned)tiles, 32, 0, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y, tile0);
    else if (tile_rows == 64) spconv_fwd_v6d_kernel<64><<<(unsigned)tiles, 32, 0, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y, tile0);
    else spconv_fwd_v6d_kernel<32><<<(unsigned)tiles, 32, 0, st>>>(x, (const uint4 *)Wa, seg, pairs, n, residual, flags, y, tile0);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// The conv of one scene of a batch union level: output rows [row0, row1) of a level of n_level rows, with the pair stream of that
// range (gpc_kmap_pairs_count_range / _fill_range: tiles start at row0, neighbour indices are the level's rows).  x, y and residual
// are the level's arrays; every (variant, tile_rows) of gpc_spconv_fwd_v6.  The kernels gather x[nbr] and write tile-relative output
// rows, so the range is the whole-level launch on y + row0: its sums are the single scene's, bit for bit.
extern "C" int gpc_spconv_fwd_v6_range(const float *x, const void *Wa, const uint32_t *seg, const uint64_t *pairs, int64_t n_level,
                                       int64_t row0, int64_t row1, int tile_rows, const float *residual, int flags, float *y,
                                       int variant, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    GPC_REQUIRE(x != y, GPC_EINVAL, "conv is out of place (rows are gathered from x while y is written)");
    return gpc_spconv_fwd_v6(x, Wa, seg, pairs, row1 - row0, tile_rows, residual ? residual + row0 * GPC_C : nullptr, flags,
                             y + row0 * GPC_C, variant, stream);
}

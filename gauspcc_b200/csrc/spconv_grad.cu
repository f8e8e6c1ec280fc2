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
        for (u32 p = p0; p < p1; p += 8) {
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
            u32 ah[4], al[4], bh[4], bl[4];              // A: (ci g + 8 j, pairs 2t, 2t + 1); B: (pairs 2t, 2t + 1, co g + 8 j)
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

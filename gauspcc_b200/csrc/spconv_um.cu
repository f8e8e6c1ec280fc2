// spconv_um.cu -- the sparse convolution of the big octree levels on the 5th-generation tensor cores (tcgen05 / tensor memory).
//
// Reference: every spnn.Conv3d(C, C, 5) of src/ai_pcc/GausPcgc/network_ue_4stage_conv.py:17-62 (torchsparse 2.1.0 gather -
// implicit GEMM - scatter); semantics as restated in SURVEY.md 8(c):  y[o] = act( sum_k W[k]^T x[nbr_k(o)] (+ residual[o]) ).
//
// Formulation (TRANSPOSED: the pairs are the N dimension of the MMA, so a chunk is as long as the tile has pairs of one offset,
// in steps of 16, and nothing is padded to 128):
//     D^T[co][p] = sum_ci W[k]^T[co][ci] . x[nbr(p)][ci]          for the pairs p of ONE offset k inside one tile of TM output rows
//   A operand  W[k]^T, bf16 hi | lo, in TENSOR MEMORY (32 columns), the 32 output channels replicated into all four lane
//              quadrants (M = 128): every epilogue warp finds the whole product in the quadrant it may read
//   B operand  the gathered rows, K-major with 128 B swizzle, in shared memory.  The rows of a chunk are fetched by ONE producer
//              warp: for the non-centre offsets by TMA tile::gather4 (four arbitrary rows per instruction, issued by one elected
//              lane), for the centre offset, whose rows are consecutive, by one TMA tile load (cp.async.bulk.tensor, SWIZZLE_128B).
//              The rows land as transaction bytes on the chunk's mbarrier, with one asynchronous arrival per producer lane after
//              its cp.async of the chunk's row offsets (cp.async.mbarrier.arrive.noinc), so the producers never wait for data.
//              (A cp.async gather, eight lanes x 16 B per row, measured the same and was dropped -- profiles/r02_conv_um.md.)
//   D          fp32 in tensor memory, N columns; six MMAs per chunk (K = 2 x 16 for Whi.xhi, Whi.xlo, Wlo.xhi)
//   epilogue   tcgen05.ld gives lane = channel, register = pair.  Warp e takes 16 columns of every chunk and adds each to its
//              output row's fp32 sum in shared memory: one conflict-free 128 B read-modify-write per pair.  Within a chunk the
//              rows are distinct; one named barrier per chunk keeps the offsets of a row in ascending order: ONE fixed summation
//              order per row, whatever the launch geometry (encoder and decoder CDFs stay bit-identical).
// Activations are "split rows" (32 x bf16 hi | 32 x bf16 lo per row, spconv_fmt.cu): a gathered row is an operand row as it
// stands; x = hi + lo to 16 mantissa bits and the three-term product keeps the contraction within ~1.5e-4 of fp32 on the
// probabilities (DESIGN.md 5).
//
// Warp roles: 0 = MMA issue (+ TMEM allocation), 1-3 and 8 + NEW .. = producers (chunk c belongs to producer c % NPW), 4-7 =
// weights -> TMEM (one warp per lane quadrant), 8 .. 8 + NEW - 1 = epilogue.  All hand-offs are mbarriers; after the last chunk
// every warp helps to write the tile out.
#include <cuda.h>
#include "umma.cuh"

template <int TM, int NMAX, int GS, int DS, int WS, int NPW>
struct UmSmem {
    float acc[TM + 16][GPC_C];                         // rows TM ..: one dummy row per epilogue warp (target of padding pairs, never read)
    __align__(1024) unsigned char g[GS][NMAX * 128];   // gathered rows of a chunk (128 B swizzle atoms of 8 rows)
    __align__(16) u32 roff[GS + DS][NMAX];             // byte offset of every pair's accumulator row (row * 128; padding -> dummy row)
    __align__(16) u32 idx[NPW][4][NMAX];               // per producer: input rows of the pairs of its next chunks
    u32 seg[GPC_K3 + 3];
    u32 cstart[GPC_K3 + 3];
    u32 tab[GPC_K3 * ((TM + NMAX - 1) / NMAX) + 8];                 // chunk -> k | j << 8 | len << 12 | last chunk of its offset << 20 | offset ordinal << 24
    u32 wcnt[4];
    __align__(8) u64 full_g[GS];
    u64 empty_g[GS];
    u64 full_d[DS];
    u64 empty_d[DS];
    u64 full_w[WS];
    u64 empty_w[WS];
    u32 tmem_base;
};

__device__ __forceinline__ void um_tmem_st32(u32 taddr, const uint4 (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
                 "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
                 ::"r"(taddr), "r"(v[0].x), "r"(v[0].y), "r"(v[0].z), "r"(v[0].w), "r"(v[1].x), "r"(v[1].y), "r"(v[1].z), "r"(v[1].w),
                   "r"(v[2].x), "r"(v[2].y), "r"(v[2].z), "r"(v[2].w), "r"(v[3].x), "r"(v[3].y), "r"(v[3].z), "r"(v[3].w),
                   "r"(v[4].x), "r"(v[4].y), "r"(v[4].z), "r"(v[4].w), "r"(v[5].x), "r"(v[5].y), "r"(v[5].z), "r"(v[5].w),
                   "r"(v[6].x), "r"(v[6].y), "r"(v[6].z), "r"(v[6].w), "r"(v[7].x), "r"(v[7].y), "r"(v[7].z), "r"(v[7].w) : "memory");
}
// shared-memory accumulator accesses of the epilogue: volatile asm keeps the written order (all loads of a batch, then all stores)
// without a "memory" clobber that would serialise every read-modify-write behind the previous one
__device__ __forceinline__ float um_lds(u32 addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void um_sts(u32 addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v)); }
// D[tmem] (+)= A[tmem] . B[smem]^T with the descriptor given as two 32-bit halves (the high half is a constant)
__device__ __forceinline__ void um_mma(u32 tmem_d, u32 tmem_a, u32 desc_lo, u32 idesc, u32 accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 d;\n\tsetp.ne.b32 p, %4, 0;\n\tmov.b64 d, {%2, %5};\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], d, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "r"(tmem_a), "r"(desc_lo), "r"(idesc), "r"(accumulate), "r"(0x40004040u) : "memory");
}

// role profile (PROF instantiation only; tools/um_check.py): cycles summed over chunks, lane 0 of one warp per role
//  [0] producer: wait for its index words   [1] producer: wait empty_g   [2] producer: issue the chunk's copies
//  [3] mma: wait full_w   [4] mma: wait full_g   [5] mma: wait empty_d   [6] mma: issue + commit
//  [7] epilogue: wait full_d   [8] epilogue: column range + tcgen05.ld + read-modify-write
//  [11] chunks   [12] CTA total   [13] setup   [14] write-out   [15] CTAs
__device__ unsigned long long g_um_prof[16];
extern "C" int gpc_debug_conv_um_profile(unsigned long long *out_h, int reset) {
    GPC_CUDA_CHECK(cudaDeviceSynchronize());
    if (out_h) GPC_CUDA_CHECK(cudaMemcpyFromSymbol(out_h, g_um_prof, sizeof(unsigned long long) * 16));
    if (reset) { unsigned long long z[16] = {0}; GPC_CUDA_CHECK(cudaMemcpyToSymbol(g_um_prof, z, sizeof(z))); }
    return GPC_OK;
}
#define UM_T(var) do { if (PROF) var = clock64(); } while (0)
#define UM_ACC(i, a, b) do { if (PROF) pacc[i] += (b) - (a); } while (0)
#define UM_FLUSH(slot, i) do { if (PROF && lane == 0) atomicAdd(&g_um_prof[slot], (unsigned long long)pacc[i]); } while (0)

template <int TM, int NMAX, int GS, int DS, int WS, int NPW, int NEW, int TCOLS, int MINB, bool PROF>
__global__ void __launch_bounds__((8 + NEW + (NPW > 3 ? NPW - 3 : 0)) * 32, MINB)
spconv_um_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_g, const unsigned char *__restrict__ xs, const uint4 *__restrict__ Wp,
                 const u32 *__restrict__ seg_g, const u32 *__restrict__ pair_nbr, const u32 *__restrict__ pair_off, i64 n, i64 tile0,
                 const u32 *__restrict__ tile_order, int xrow0,
                 const void *__restrict__ residual, int flags, float *__restrict__ y, u32 *__restrict__ ys) {
    constexpr int NWARPS = 8 + NEW + (NPW > 3 ? NPW - 3 : 0), NTHREADS = NWARPS * 32;
    constexpr int RS = GS + DS;                  // row-offset ring: a chunk's entries live from its gather to the start of its epilogue
    constexpr u32 A_COL = DS * NMAX;             // first weight column of tensor memory
    static_assert(A_COL + WS * 32 <= TCOLS, "TMEM columns");
    static_assert(NMAX == 16 * NEW || NMAX == 8 * NEW, "an epilogue warp takes 8 or 16 columns of a chunk");
    static_assert(NPW >= 1 && (NMAX == 64 || NMAX == 96 || NMAX == 128), "shape");
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    typedef UmSmem<TM, NMAX, GS, DS, WS, NPW> Smem;
    Smem &s = *reinterpret_cast<Smem *>(smem_raw);
    if (((u32)__cvta_generic_to_shared(smem_raw) & 1023u) != 0u) __trap();      // 128 B swizzle atoms are 1024 B aligned
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // tile_order (full-level launches): heaviest tiles first, so that the last CTAs to start are the shortest (a level is only ~3
    // tiles per CTA slot: in index order the SMs idle up to one tile's duration at the end of the launch)
    const i64 t = tile0 + (tile_order ? (i64)tile_order[blockIdx.x] : (i64)blockIdx.x);
    long long pacc[4] = {0, 0, 0, 0}, t0 = 0, t1 = 0, t2 = 0, t3 = 0, t4 = 0, t_begin = 0, t_setup = 0;
    UM_T(t_begin);

    // ---- setup: segment table, chunk table, barriers, tensor memory, zeroed sums
    for (int i = tid; i <= GPC_K3; i += NTHREADS) s.seg[i] = seg_g[t * (GPC_K3 + 1) + i];
    for (int i = tid; i < TM * GPC_C / 4; i += NTHREADS) reinterpret_cast<float4 *>(&s.acc[0][0])[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid == 0) {
        for (int i = 0; i < GS; ++i) { mbar_init((u32)__cvta_generic_to_shared(&s.full_g[i]), 32); mbar_init((u32)__cvta_generic_to_shared(&s.empty_g[i]), 1); }
        for (int i = 0; i < DS; ++i) { mbar_init((u32)__cvta_generic_to_shared(&s.full_d[i]), 1); mbar_init((u32)__cvta_generic_to_shared(&s.empty_d[i]), NEW); }
        for (int i = 0; i < WS; ++i) { mbar_init((u32)__cvta_generic_to_shared(&s.full_w[i]), 4); mbar_init((u32)__cvta_generic_to_shared(&s.empty_w[i]), 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        const u32 dst = (u32)__cvta_generic_to_shared(&s.tmem_base);
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "n"(TCOLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    __syncthreads();
    if (tid < GPC_K3) s.cstart[tid] = (s.seg[tid + 1] - s.seg[tid] + NMAX - 1) / NMAX;
    __syncthreads();
    if (warp == 0) {                                             // exclusive scan of the 125 chunk counts
        u32 v[4], sum = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) { const int k = lane * 4 + i; v[i] = k < GPC_K3 ? s.cstart[k] : 0u; sum += v[i]; }
        u32 incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const u32 u = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += u; }
        u32 run = incl - sum;
#pragma unroll
        for (int i = 0; i < 4; ++i) { const int k = lane * 4 + i; if (k <= GPC_K3) s.cstart[k] = run; run += v[i]; }
    }
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();
    u32 live_ballot = 0;
    if (tid < 128) {                                             // offset ordinal among the non-empty offsets (weights ring)
        const bool live = tid < GPC_K3 && s.cstart[tid + 1] > s.cstart[tid];
        live_ballot = __ballot_sync(0xFFFFFFFFu, live);
        if (lane == 0) s.wcnt[warp] = __popc(live_ballot);
    }
    __syncthreads();
    if (tid < GPC_K3 && s.cstart[tid + 1] > s.cstart[tid]) {
        u32 ord = __popc(live_ballot & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) ord += s.wcnt[w];
        const u32 b = s.cstart[tid], e = s.cstart[tid + 1], tot = s.seg[tid + 1] - s.seg[tid];
        for (u32 c = b; c < e; ++c) {
            const u32 j = c - b, len = min((u32)NMAX, tot - j * NMAX);
            s.tab[c] = (u32)tid | (j << 8) | (len << 12) | ((c + 1 == e ? 1u : 0u) << 20) | (ord << 24);
        }
    }
    __syncthreads();
    const u32 n_chunks = s.cstart[GPC_K3];
    const u32 tmem = s.tmem_base;
    const u32 full_g0 = (u32)__cvta_generic_to_shared(&s.full_g[0]), empty_g0 = (u32)__cvta_generic_to_shared(&s.empty_g[0]);
    const u32 full_d0 = (u32)__cvta_generic_to_shared(&s.full_d[0]), empty_d0 = (u32)__cvta_generic_to_shared(&s.empty_d[0]);
    const u32 full_w0 = (u32)__cvta_generic_to_shared(&s.full_w[0]), empty_w0 = (u32)__cvta_generic_to_shared(&s.empty_w[0]);
    const u32 g0 = (u32)__cvta_generic_to_shared(&s.g[0][0]);
    UM_T(t_setup);

    const int prod = (warp >= 1 && warp < 4) ? warp - 1 : (warp >= 8 + NEW ? warp - (8 + NEW) + 3 : -1);
    if (warp == 0) {
        // =================================================================== MMA issue (whole warp loops, one elected lane issues)
        constexpr u32 IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);      // D f32, A = B = bf16 K-major, M = 128
        for (u32 c = 0; c < n_chunks; ++c) {
            const u32 e = s.tab[c], len = (e >> 12) & 0xFFu, wi = e >> 24, ws = wi % (u32)WS;
            const u32 gs = c % (u32)GS, ds = c % (u32)DS;
            UM_T(t0);
            if (((e >> 8) & 0xFu) == 0) mbar_wait_hint(full_w0 + ws * 8, (wi / (u32)WS) & 1u);     // first chunk of an offset: its weights
            UM_T(t1);
            mbar_wait_hint(full_g0 + gs * 8, (c / (u32)GS) & 1u);
            UM_T(t2);
            if (c >= (u32)DS) mbar_wait_hint(empty_d0 + ds * 8, ((c / (u32)DS) & 1u) ^ 1u);
            UM_T(t3);
            tmem_fence_after();
            if (elect_one()) {
                const u32 idesc = IDESC | ((len >> 3) << 17);
                const u32 d = tmem + ds * NMAX, a = tmem + A_COL + ws * 32;
                // K-major SWIZZLE_128B descriptor: start address >> 4 | LBO 1 << 16; high half = SBO 1024 B, version 1, layout type 2
                const u32 b = ((g0 + gs * (NMAX * 128)) >> 4) | (1u << 16);
                um_mma(d, a, b, idesc, 0u);                      // Whi . xhi   (K 0..15)
                um_mma(d, a + 8, b + 2, idesc, 1u);              //             (K 16..31: + 32 B)
                um_mma(d, a, b + 4, idesc, 1u);                  // Whi . xlo
                um_mma(d, a + 8, b + 6, idesc, 1u);
                um_mma(d, a + 16, b, idesc, 1u);                 // Wlo . xhi
                um_mma(d, a + 24, b + 2, idesc, 1u);
                umma_commit(empty_g0 + gs * 8);
                umma_commit(full_d0 + ds * 8);
                if ((e >> 20) & 1u) umma_commit(empty_w0 + ws * 8);              // last chunk of the offset
            }
            __syncwarp();
            UM_T(t4);
            UM_ACC(0, t0, t1); UM_ACC(1, t1, t2); UM_ACC(2, t2, t3); UM_ACC(3, t3, t4);
        }
        UM_FLUSH(3, 0); UM_FLUSH(4, 1); UM_FLUSH(5, 2); UM_FLUSH(6, 3);
        if (PROF && lane == 0) { atomicAdd(&g_um_prof[11], (unsigned long long)n_chunks); atomicAdd(&g_um_prof[15], 1ull); }
    } else if (prod >= 0) {
        // =================================================================== producers: chunk c belongs to producer c % NPW
        const u32 p = (u32)prod;
        const u32 roff0 = (u32)__cvta_generic_to_shared(&s.roff[0][0]);
        const u32 ring0 = (u32)__cvta_generic_to_shared(&s.idx[p][0][0]);
        auto start_of = [&](u32 e) { return s.seg[e & 0xFFu] + (u32)NMAX * ((e >> 8) & 0xFu); };
        auto prefetch = [&](u32 m) {                             // input rows of the pairs of my m-th chunk -> ring slot m % 4
            const u32 c = p + m * (u32)NPW;
            if (c < n_chunks) {
                const u32 e = s.tab[c], len = (e >> 12) & 0xFFu;
                if (4u * (u32)lane < len) cp_async16(ring0 + (m & 3u) * (NMAX * 4) + (u32)lane * 16u, pair_nbr + start_of(e) + 4u * (u32)lane);
            }
        };
        prefetch(0);
        cp_async_commit();
        prefetch(1);
        cp_async_commit();
        u32 m = 0;
        for (u32 c = p; c < n_chunks; c += (u32)NPW, ++m) {
            const u32 e = s.tab[c], k = e & 0xFFu, len = (e >> 12) & 0xFFu;
            const u32 start = start_of(e);
            const u32 gs = c % (u32)GS, f = c / (u32)GS;
            const u32 slot = g0 + gs * (NMAX * 128), bar = full_g0 + gs * 8;
            UM_T(t0);
            cp_async_wait<1>();                                  // my index words of this chunk (committed two of my chunks ago)
            __syncwarp();
            UM_T(t1);
            if (f) mbar_wait_hint(empty_g0 + gs * 8, (f & 1u) ^ 1u);  // the MMAs of chunk c - GS have read the slot
            UM_T(t2);
            if (k == 62u) {
                // centre offset: pair p is row (tile start + chunk start + p) itself: one TMA tile load of NMAX consecutive rows
                // (rows past the end of the level are zero-filled; columns past len are never read).  xrow0: the launch's first output
                // row is input row xrow0 (a scene of a union level; rows of the next scene may land in padding columns, whose products
                // go to the dummy rows)
                if (elect_one()) {
                    const u32 j = (e >> 8) & 0xFu;
                    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"((u32)NMAX * 128u) : "memory");
                    asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                                 ::"r"(slot), "l"(reinterpret_cast<u64>(&tmap)), "r"(bar), "r"(0), "r"(xrow0 + (int)(t * TM + j * NMAX)) : "memory");
                }
            } else {
                // TMA tile::gather4: four arbitrary rows per instruction, written with the 128 B swizzle; padding entries (row -1) are
                // out of bounds = zero fill.  Issued by ONE elected lane inside warp-uniform control flow (per-lane issue makes ptxas
                // emit an election loop with six R2UR.BROADCAST per instruction: ~50-100 clk each, profiles/r02_conv_um.md).
                const uint4 *ring = reinterpret_cast<const uint4 *>(&s.idx[p][m & 3u][0]);
                if (elect_one()) asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(len * 128u) : "memory");
#pragma unroll 4
                for (u32 q = 0; q < (len >> 2); ++q) {
                    const uint4 ix = ring[q];
                    if (elect_one())
                        asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                                     ::"r"(slot + q * 512u), "l"(reinterpret_cast<u64>(&tmap_g)), "r"(bar), "r"(0), "r"((int)ix.x), "r"((int)ix.y), "r"((int)ix.z), "r"((int)ix.w) : "memory");
                }
            }
            __syncwarp();
            if (4u * (u32)lane < len)                            // the chunk's accumulator-row offsets, for the epilogue
                cp_async16(roff0 + (c % (u32)RS) * (NMAX * 4) + (u32)lane * 16u, pair_off + start + 4u * (u32)lane);
            // asynchronous arrival: when every copy of this lane has landed (TMA rows arrive as transaction bytes)
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
            prefetch(m + 2);
            cp_async_commit();
            UM_T(t3);
            UM_ACC(0, t0, t1); UM_ACC(1, t1, t2); UM_ACC(2, t2, t3);
        }
        cp_async_wait<0>();
        if (warp == 1) { UM_FLUSH(1, 1); UM_FLUSH(2, 2); }
    } else if (warp < 8) {
        // =================================================================== weights: W[k]^T hi | lo -> this warp's lane quadrant
        const u32 q = (u32)warp & 3u;
        const u32 ta = tmem + ((q * 32u) << 16) + A_COL;
        int k = 0;
        while (k < GPC_K3 && s.seg[k + 1] == s.seg[k]) ++k;
        for (u32 wi = 0; k < GPC_K3; ++wi) {
            uint4 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __ldg(Wp + ((size_t)k * 8 + i) * 32 + lane);      // coalesced: chunk i of all 32 channels is contiguous
            ++k;
            while (k < GPC_K3 && s.seg[k + 1] == s.seg[k]) ++k;
            const u32 ws = wi % (u32)WS, f = wi / (u32)WS;
            if (f) mbar_wait_hint(empty_w0 + ws * 8, (f & 1u) ^ 1u);
            tmem_fence_after();
            um_tmem_st32(ta + ws * 32, v);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tmem_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(full_w0 + ws * 8);
        }
    } else {
        // =================================================================== epilogue: warp e adds the columns [CPW e, CPW e + CPW) of every
        // chunk to their rows.  Within a chunk the rows are distinct; a barrier between chunks keeps the offsets of a row in order.
        constexpr int CPW = NMAX / NEW;                          // 8 or 16 columns of a chunk per warp
        const u32 e = (u32)warp - 8u;
        const u32 acc0 = (u32)__cvta_generic_to_shared(&s.acc[0][0]) + (u32)lane * 4u;
        const u32 td = tmem + ((((u32)warp & 3u) * 32u) << 16) + e * CPW;       // my lane quadrant, my columns
        // load(c): my D columns (asynchronous) and the accumulator addresses of my pairs of chunk c -> registers; a padding entry
        // (offset of row TM) goes to this warp's own dummy row.  done(c): wait for the columns and hand the D buffer back -- the
        // row offsets have been consumed by then (the address arithmetic below), so their ring slot may be rewritten.
        const u32 pad_off = (u32)TM * 128u, my_dummy = acc0 + ((u32)TM + e) * 128u;
        auto load = [&](u32 c, u32 (&d)[CPW], u32 (&ra)[CPW], bool &on) {
            const u32 ds = c % (u32)DS;
            on = e * CPW < ((s.tab[c] >> 12) & 0xFFu);           // len is a multiple of 16: my columns are inside or outside
            mbar_wait_hint(full_d0 + ds * 8, (c / (u32)DS) & 1u);
            tmem_fence_after();
            if (on) {
                if (CPW == 16) tmem_ld16(td + ds * NMAX, *reinterpret_cast<u32(*)[16]>(&d[0]));
                else tmem_ld8(td + ds * NMAX, *reinterpret_cast<u32(*)[8]>(&d[0]));
                const uint4 *ro = reinterpret_cast<const uint4 *>(&s.roff[c % (u32)RS][e * CPW]);
#pragma unroll
                for (int i = 0; i < CPW / 4; ++i) {
                    const uint4 r = ro[i];
                    ra[4 * i] = r.x >= pad_off ? my_dummy : acc0 + r.x;
                    ra[4 * i + 1] = r.y >= pad_off ? my_dummy : acc0 + r.y;
                    ra[4 * i + 2] = r.z >= pad_off ? my_dummy : acc0 + r.z;
                    ra[4 * i + 3] = r.w >= pad_off ? my_dummy : acc0 + r.w;
                }
            }
        };
        auto done = [&](u32 c) {
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            tmem_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_d0 + (c % (u32)DS) * 8);     // values and addresses are in registers: hand the buffer back
        };
        auto rmw = [&](const u32 (&d)[CPW], const u32 (&ra)[CPW], bool on) {
            if (on) {
#pragma unroll
                for (int h = 0; h < CPW / 8; ++h) {
                    float a[8];
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) a[jj] = um_lds(ra[8 * h + jj]);
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) um_sts(ra[8 * h + jj], a[jj] + __uint_as_float(d[8 * h + jj]));
                }
            }
        };
        u32 dA[CPW], dB[CPW], rA[CPW], rB[CPW];
        bool onA = false, onB = false;
        UM_T(t0);
        if (n_chunks) { load(0, dA, rA, onA); done(0); }
        for (u32 c = 0; c < n_chunks; c += 2) {
            // chunk c (set A) is in registers; request chunk c + 1 (set B) before adding chunk c to its rows, and so on
            if (c + 1 < n_chunks) load(c + 1, dB, rB, onB);
            asm volatile("bar.sync 1, %0;" ::"n"(NEW * 32) : "memory");          // every epilogue warp is done with the previous chunk
            rmw(dA, rA, onA);
            if (c + 1 < n_chunks) {
                done(c + 1);
                if (c + 2 < n_chunks) load(c + 2, dA, rA, onA);
                asm volatile("bar.sync 1, %0;" ::"n"(NEW * 32) : "memory");
                rmw(dB, rB, onB);
                if (c + 2 < n_chunks) done(c + 2);
            }
        }
        asm volatile("" ::: "memory");
        UM_T(t1);
        UM_ACC(0, t0, t1);
        if (warp == 8) { UM_FLUSH(7, 0); UM_FLUSH(8, 1); UM_FLUSH(9, 2); UM_FLUSH(10, 3); }
        asm volatile("" ::: "memory");
    }
    tmem_fence_before();
    __syncthreads();
    UM_T(t0);
    if (warp == 0) {
        tmem_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TCOLS) : "memory");
    }
    // ---- write-out by all warps: (+ residual) (ReLU) -> fp32 rows and / or split rows, one 128 B store per row
    {
        const bool relu = (flags & GPC_CONV_RELU) != 0, res_split = (flags & GPC_CONV_RES_SPLIT) != 0;
        const i64 gbase = t * TM;
        const int rows = (int)max((i64)0, min((i64)TM, n - gbase));
        constexpr int UR = 4;
        for (int rb = warp; rb < rows; rb += NWARPS * UR) {
            float v[UR];
            u32 wh[UR], wl[UR];
#pragma unroll
            for (int u = 0; u < UR; ++u) {
                const int r = rb + u * NWARPS;
                v[u] = 0.f; wh[u] = 0u; wl[u] = 0u;
                if (r < rows) {
                    v[u] = s.acc[r][lane];
                    const i64 gr = gbase + r;
                    if (residual) {
                        if (res_split) {
                            const u32 *rs = reinterpret_cast<const u32 *>(residual) + gr * 32 + (lane >> 1);
                            wh[u] = __ldg(rs); wl[u] = __ldg(rs + 16);
                        } else {
                            wh[u] = __float_as_uint(__ldg(reinterpret_cast<const float *>(residual) + gr * 32 + lane));
                        }
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < UR; ++u) {
                const int r = rb + u * NWARPS;
                if (r < rows) {                                  // warp-uniform
                    const i64 gr = gbase + r;
                    float o = v[u];
                    if (residual) {
                        if (res_split) o += (lane & 1) ? __uint_as_float(wh[u] & 0xFFFF0000u) + __uint_as_float(wl[u] & 0xFFFF0000u)
                                                       : __uint_as_float(wh[u] << 16) + __uint_as_float(wl[u] << 16);
                        else o += __uint_as_float(wh[u]);
                    }
                    if (relu) o = fmaxf(o, 0.f);
                    if (y) y[gr * 32 + lane] = o;
                    if (ys) {
                        const float vh = bf16_round(o), vl = bf16_round(o - vh);
                        const u32 mine = (__float_as_uint(vh) >> 16) | (__float_as_uint(vl) & 0xFFFF0000u);      // hi in the low half, lo in the high half
                        const u32 other = __shfl_xor_sync(0xFFFFFFFFu, mine, 1);
                        // even lane 2j: hi word j = (hi[2j], hi[2j+1]); odd lane 2j+1: lo word 16 + j = (lo[2j], lo[2j+1])
                        const u32 word = (lane & 1) ? ((other >> 16) | (mine & 0xFFFF0000u)) : ((mine & 0xFFFFu) | (other << 16));
                        ys[gr * 32 + ((lane & 1) << 4) + (lane >> 1)] = word;
                    }
                }
            }
        }
    }
    if (PROF && tid == 0) {
        atomicAdd(&g_um_prof[14], (unsigned long long)(clock64() - t0));
        atomicAdd(&g_um_prof[12], (unsigned long long)(clock64() - t_begin));
        atomicAdd(&g_um_prof[13], (unsigned long long)(t_setup - t_begin));
    }
}

// ---- host side
typedef CUresult (*um_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                 const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static um_encode_fn um_encoder() {
    static um_encode_fn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (um_encode_fn)p;
    }
    return fn;
}

template <int TM, int NMAX, int GS, int DS, int WS, int NPW, int NEW, int TCOLS, int MINB, bool PROF = false>
static int launch_spconv_um(const CUtensorMap &tmap, const CUtensorMap &tmap_g, const void *xs, const void *Wp, const u32 *seg, const u32 *pair_nbr, const u32 *pair_off,
                            i64 n, i64 tile0, i64 tiles, const u32 *tile_order, int xrow0, const void *residual, int flags, float *y, void *ys,
                            cudaStream_t st) {
    static bool configured = false;
    typedef UmSmem<TM, NMAX, GS, DS, WS, NPW> Smem;
    constexpr size_t smem = sizeof(Smem);
    constexpr int NTHREADS = (8 + NEW + (NPW > 3 ? NPW - 3 : 0)) * 32;
    static_assert((smem + 1024) * MINB <= 233472, "shared memory per SM");
    if (!configured) {
        GPC_CUDA_CHECK(cudaFuncSetAttribute(spconv_um_kernel<TM, NMAX, GS, DS, WS, NPW, NEW, TCOLS, MINB, PROF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    spconv_um_kernel<TM, NMAX, GS, DS, WS, NPW, NEW, TCOLS, MINB, PROF><<<(unsigned)tiles, NTHREADS, smem, st>>>(
        tmap, tmap_g, (const unsigned char *)xs, (const uint4 *)Wp, seg, pair_nbr, pair_off, n, tile0, tile_order, xrow0, residual, flags, y, (u32 *)ys);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// xs = split rows [n][128 B]; Wp = this conv's slice of gpc_spconv_pack_weights_um; seg / pair_nbr = the pair stream built with
// tile_rows = 512 and pad = 16 (padding entries 0xFFFFFFFF), pair_off (gpc_kmap_um_count / _fill).  Output rows
// [row0, row1) (whole tiles; row1 <= 0 or >= n: to the end).  y (fp32 rows) and / or ys (split rows).
// n_in >= xrow0 + n: rows of xs (the TMA tensor); the launch's output row r reads the centre row xrow0 + r and writes y[r] / ys[r];
// neighbour indices address all n_in rows.  (n_in = n, xrow0 = 0: a whole level.)
static int um_fwd(const void *xs, int64_t n_in, int64_t xrow0, const void *Wp, const uint32_t *seg, const uint32_t *pair_nbr,
                  const uint32_t *pair_off, int64_t n, int tile_rows, const uint32_t *tile_order, const void *residual, int flags, float *y,
                  void *ys, int64_t row0, int64_t row1, void *stream) {
    const bool prof = (flags & GPC_CONV_PROFILE) != 0;
    flags &= ~GPC_CONV_PROFILE;
    if (n <= 0) return GPC_OK;
    GPC_REQUIRE(y || ys, GPC_EINVAL, "no output requested");
    GPC_REQUIRE(xs != ys && xs != (const void *)y, GPC_EINVAL, "conv is out of place (rows are gathered from xs while y is written)");
    GPC_REQUIRE(tile_rows == 512, GPC_EINVAL, "tile_rows must be 512");
    if (row1 <= 0 || row1 > n) row1 = n;
    GPC_REQUIRE(row0 >= 0 && row0 % tile_rows == 0 && (row1 % tile_rows == 0 || row1 == n), GPC_EINVAL, "row range must cover whole tiles");
    if (row0 >= row1) return GPC_OK;
    um_encode_fn enc = um_encoder();
    GPC_REQUIRE(enc != nullptr, GPC_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
    CUtensorMap tmap;                                            // [n_in rows][64 bf16], box = one chunk of consecutive rows (the centre offset)
    GPC_REQUIRE(n_in >= xrow0 + n && n_in < (1ll << 31), GPC_EINVAL, "input rows must cover the output rows and fit TMA coordinates");
    const cuuint64_t gdim[2] = {64, (cuuint64_t)n_in};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {64, 64};                          // 64 rows: NMAX of the launch below
    const cuuint32_t estr[2] = {1, 1};
    const CUresult rc = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(xs), gdim, gstride, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) { gpc_set_error("cuTensorMapEncodeTiled failed: %d", (int)rc); return GPC_ECUDA; }
    CUtensorMap tmap_g;                                          // the same tensor with a one-row box: tile::gather4
    const cuuint32_t box1[2] = {64, 1};
    const CUresult rc2 = enc(&tmap_g, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(xs), gdim, gstride, box1, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc2 != CUDA_SUCCESS) { gpc_set_error("cuTensorMapEncodeTiled (gather) failed: %d", (int)rc2); return GPC_ECUDA; }
    cudaStream_t st = as_stream(stream);
    const i64 tile0 = row0 / tile_rows, tiles = (row1 - row0 + tile_rows - 1) / tile_rows;
    const u32 *order = (row0 == 0 && row1 == n) ? tile_order : nullptr;            // a permutation of the level's tiles: full launches only
    const int xr0 = (int)xrow0;
    if (prof) return launch_spconv_um<512, 64, 4, 3, 2, 3, 8, 256, 2, true>(tmap, tmap_g, xs, Wp, seg, pair_nbr, pair_off, n, tile0, tiles, order, xr0, residual, flags, y, ys, st);
    return launch_spconv_um<512, 64, 4, 3, 2, 3, 8, 256, 2>(tmap, tmap_g, xs, Wp, seg, pair_nbr, pair_off, n, tile0, tiles, order, xr0, residual, flags, y, ys, st);
}
extern "C" int gpc_spconv_fwd_um(const void *xs, const void *Wp, const uint32_t *seg, const uint32_t *pair_nbr,
                                 const uint32_t *pair_off, int64_t n, int tile_rows, const uint32_t *tile_order, const void *residual,
                                 int flags, float *y, void *ys, int64_t row0, int64_t row1, void *stream) {
    return um_fwd(xs, n, 0, Wp, seg, pair_nbr, pair_off, n, tile_rows, tile_order, residual, flags, y, ys, row0, row1, stream);
}
// The conv of one scene of a batch union level: output rows [row0, row1) of a level of n_level rows, with the pair stream of that
// range (gpc_kmap_um_count_range / _fill_range).  The TMA descriptors span all n_level rows of xs (out-of-bounds padding entries,
// 0xFFFFFFFF, still read as zeros); the centre tiles start at row0.  xs, y, ys and residual are the level's arrays; tile_order (may be
// NULL) is a permutation of the RANGE's tiles.
extern "C" int gpc_spconv_fwd_um_range(const void *xs, const void *Wp, const uint32_t *seg, const uint32_t *pair_nbr,
                                       const uint32_t *pair_off, int64_t n_level, int64_t row0, int64_t row1, const uint32_t *tile_order,
                                       const void *residual, int flags, float *y, void *ys, void *stream) {
    GPC_RANGE_CHECK(n_level, row0, row1);
    GPC_REQUIRE(xs != ys && xs != (const void *)y, GPC_EINVAL, "conv is out of place (rows are gathered from xs while y is written)");
    const int64_t n = row1 - row0;
    return um_fwd(xs, n_level, row0, Wp, seg, pair_nbr, pair_off, n, 512, tile_order,
                  residual ? (const void *)((const uint32_t *)residual + row0 * GPC_C) : nullptr, flags, y ? y + row0 * GPC_C : nullptr,
                  ys ? (void *)((uint32_t *)ys + row0 * GPC_C) : nullptr, 0, n, stream);
}

// W [n_kernels*125][32 ci][32 co] fp32 -> Wp [n_kernels*125][8 chunks][32 co][4 words]: channel co's TMEM lane is 32 words = 8 chunks of
// 16 B (words 0..15 = bf16x2 (hi(W[2j][co]), hi(W[2j+1][co])), words 16..31 = the lo halves: K pairs packed as the A operand wants
// them); chunk i of all 32 channels is contiguous, so lane = channel reads its lane with eight COALESCED 16-byte loads (channel-major
// rows of 128 B cost 32 L1 wavefronts per load instruction: 110 M per conv, 70-80 % of the L1 data pipe -- profiles/r02_conv_um.md)
__global__ void pack_weights_um_kernel(const float *__restrict__ W, u32 *__restrict__ Wp, i64 total) {
    const i64 g = (i64)blockIdx.x * blockDim.x + threadIdx.x;      // one thread per (k, co, j)
    if (g >= total) return;
    const int j = (int)(g & 15), co = (int)((g >> 4) & 31);
    const i64 k = g >> 9;
    const float w0 = W[k * 1024 + (2 * j) * 32 + co], w1 = W[k * 1024 + (2 * j + 1) * 32 + co];
    const float h0 = bf16_round(w0), h1 = bf16_round(w1);
    const float l0 = bf16_round(w0 - h0), l1 = bf16_round(w1 - h1);
    auto at = [&](int w) { return Wp + ((k * 8 + (w >> 2)) * 32 + co) * 4 + (w & 3); };
    *at(j) = (__float_as_uint(h0) >> 16) | (__float_as_uint(h1) & 0xFFFF0000u);
    *at(16 + j) = (__float_as_uint(l0) >> 16) | (__float_as_uint(l1) & 0xFFFF0000u);
}
extern "C" int gpc_spconv_pack_weights_um(const float *W, int n_kernels, void *Wp, void *stream) {
    const i64 total = (i64)n_kernels * GPC_K3 * 32 * 16;
    pack_weights_um_kernel<<<cdiv(total, 256), 256, 0, as_stream(stream)>>>(W, (u32 *)Wp, total);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

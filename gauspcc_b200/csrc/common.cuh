// common.cuh -- shared helpers for libgpcgc (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/gpcgc.h"

typedef uint64_t u64;
typedef uint32_t u32;
typedef uint16_t u16;
typedef uint8_t u8;
typedef int64_t i64;
typedef int32_t i32;

void gpc_set_error(const char *fmt, ...);

#define GPC_CUDA_CHECK(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            gpc_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return GPC_ECUDA;                                                             \
        }                                                                                 \
    } while (0)

extern unsigned long long g_gpc_launches;     // kernels launched by this library (gpc_launch_count)
#define GPC_LAUNCH_CHECK()                                                                \
    do {                                                                                  \
        ++g_gpc_launches;                                                                 \
        GPC_CUDA_CHECK(cudaGetLastError());                                               \
    } while (0)

#define GPC_REQUIRE(cond, code, msg)                                                      \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            gpc_set_error("%s:%d: %s", __FILE__, __LINE__, msg);                          \
            return code;                                                                  \
        }                                                                                 \
    } while (0)
// [row0, row1) must be a row range of a level of n_level rows (the *_range entry points: one scene of a batch union level)
#define GPC_RANGE_CHECK(n_level, row0, row1) \
    GPC_REQUIRE((row0) >= 0 && (row0) <= (row1) && (row1) <= (n_level), GPC_EINVAL, "row range outside the level")

static inline cudaStream_t as_stream(void *s) { return (cudaStream_t)s; }
static inline unsigned cdiv(i64 a, i64 b) { return (unsigned)((a + b - 1) / b); }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------- voxel keys
#define GPC_FIELD_BITS 21
#define GPC_FIELD_MASK 0x1FFFFFull
#define GPC_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull

__host__ __device__ __forceinline__ u64 key_pack(i32 x, i32 y, i32 z) {
    return ((u64)(u32)(z + GPC_COORD_BIAS) << 42) | ((u64)(u32)(y + GPC_COORD_BIAS) << 21) |
           (u64)(u32)(x + GPC_COORD_BIAS);
}
__host__ __device__ __forceinline__ i32 key_x(u64 k) { return (i32)(k & GPC_FIELD_MASK) - GPC_COORD_BIAS; }
__host__ __device__ __forceinline__ i32 key_y(u64 k) { return (i32)((k >> 21) & GPC_FIELD_MASK) - GPC_COORD_BIAS; }
__host__ __device__ __forceinline__ i32 key_z(u64 k) { return (i32)((k >> 42) & GPC_FIELD_MASK) - GPC_COORD_BIAS; }

// parent voxel floor(c/2) per axis, on biased fields: f' = (f >> 1) + 2^19
__host__ __device__ __forceinline__ u64 key_parent(u64 k) {
    const u64 m20 = 0xFFFFFull | (0xFFFFFull << 21) | (0xFFFFFull << 42);
    const u64 b19 = (1ull << 19) | (1ull << 40) | (1ull << 61);
    return ((k >> 1) & m20) + b19;
}
// octant index of a voxel inside its parent: (x&1) + 2(y&1) + 4(z&1)  (kit/nn.py:43-45,114-116)
__host__ __device__ __forceinline__ u32 key_octant(u64 k) {
    return (u32)(k & 1) | ((u32)(k >> 21) & 1) << 1 | ((u32)(k >> 42) & 1) << 2;
}
// child 2c + (bx,by,bz) on biased fields: f' = 2f - 2^20 + b
__host__ __device__ __forceinline__ u64 key_child(u64 k, u32 oct) {
    const u64 b20 = (1ull << 20) | (1ull << 41) | (1ull << 62);
    return (k << 1) - b20 + ((u64)(oct & 1) | ((u64)((oct >> 1) & 1) << 21) | ((u64)((oct >> 2) & 1) << 42));
}
__host__ __device__ __forceinline__ u64 key_compact(u64 k, gpc_key_xform t) {
    u64 x = (k & GPC_FIELD_MASK) - t.minx;
    u64 y = ((k >> 21) & GPC_FIELD_MASK) - t.miny;
    u64 z = ((k >> 42) & GPC_FIELD_MASK) - t.minz;
    return (z << t.sz) | (y << t.sy) | x;
}

// ---------------------------------------------------------------- bf16 hi / lo split of fp32 (x = hi + lo + O(2^-17 x))
// round-to-nearest-even to bf16, as fp32.  NaN gives the canonical bf16 NaN, as cvt.rn.bf16x2 does: the integer rounding would carry
// the all-ones NaN mantissa into the sign bit (-0.0) and truncate a NaN whose payload lies in the low 16 bits to inf.
__device__ __forceinline__ float bf16_round(float v) {
    u32 u = __float_as_uint(v);
    if ((u & 0x7FFFFFFFu) > 0x7F800000u) return __uint_as_float(0x7FFF0000u);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return __uint_as_float(u & 0xFFFF0000u);
}
// (p0, p1) -> packed bf16x2 words: hi = bf16(p), lo = bf16(p - hi); p0 in the low half (lower address)
__device__ __forceinline__ void split_bf16(float p0, float p1, u32 &hi, u32 &lo) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(p1), "f"(p0));
    const float p0h = __uint_as_float(hi << 16), p1h = __uint_as_float(hi & 0xFFFF0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(p1 - p1h), "f"(p0 - p0h));
}
// the inverse for "split rows" (see spconv_umma.cu): two channels from one hi word and one lo word
__device__ __forceinline__ float2 join_bf16(u32 hi, u32 lo) {
    return make_float2(__uint_as_float(hi << 16) + __uint_as_float(lo << 16),
                       __uint_as_float(hi & 0xFFFF0000u) + __uint_as_float(lo & 0xFFFF0000u));
}

// ---------------------------------------------------------------- generic device-wide exclusive scan
// T needs operator+ and a zero(); LoadOp(i) produces element i.  Three phases per level:
//   scan_tiles: per-tile exclusive scan + tile total; (recursive) scan of tile totals; add_offsets.
// Output has n+1 entries (out[n] = grand total).
template <typename T> struct ScanZero { __device__ static T get() { return T(0); } };

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T *smem /* SCAN_THREADS/32 + 1 */, T &total) {
    // warp inclusive scan via shuffles on raw 32-bit words is type specific; do it through smem instead
    // (generic T, small blocks) -- two-level: warp serial over lanes is avoided with a Hillis-Steele pass.
    const int tid = threadIdx.x;
    __shared__ T buf[SCAN_THREADS];
    (void)smem;
    buf[tid] = v;
    __syncthreads();
#pragma unroll
    for (int off = 1; off < SCAN_THREADS; off <<= 1) {
        T add = ScanZero<T>::get();
        if (tid >= off) add = buf[tid - off];
        __syncthreads();
        if (tid >= off) buf[tid] = add + buf[tid];
        __syncthreads();
    }
    T incl = buf[tid];
    total = buf[SCAN_THREADS - 1];
    __syncthreads();
    T excl = (tid == 0) ? ScanZero<T>::get() : buf[tid - 1];
    (void)incl;
    __syncthreads();
    return excl;
}

template <typename T, typename LoadOp>
__global__ void __launch_bounds__(SCAN_THREADS) scan_tiles_kernel(LoadOp load, i64 n1 /* n+1 */, T *out, T *tile_totals) {
    const i64 base = (i64)blockIdx.x * SCAN_TILE + (i64)threadIdx.x * SCAN_ITEMS;
    T items[SCAN_ITEMS];
    T sum = ScanZero<T>::get();
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        i64 idx = base + i;
        items[i] = (idx < n1 - 1) ? load(idx) : ScanZero<T>::get();   // element n (the total slot) is zero
        sum = sum + items[i];
    }
    T total;
    T excl = block_exclusive_scan<T>(sum, nullptr, total);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        i64 idx = base + i;
        if (idx < n1) out[idx] = excl;
        excl = excl + items[i];
    }
    if (threadIdx.x == 0) tile_totals[blockIdx.x] = total;
}

template <typename T> struct PtrLoad {
    const T *p;
    __device__ T operator()(i64 i) const { return p[i]; }
};

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_add_offsets_kernel(T *out, i64 n1, const T *tile_offsets) {
    const i64 base = (i64)blockIdx.x * SCAN_TILE + (i64)threadIdx.x * SCAN_ITEMS;
    const T off = tile_offsets[blockIdx.x];
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        i64 idx = base + i;
        if (idx < n1) out[idx] = out[idx] + off;
    }
}

template <typename T> static inline size_t scan_workspace_bytes(i64 n) {
    size_t total = 0;
    i64 m = n + 1;
    while (true) {
        i64 tiles = (m + SCAN_TILE - 1) / SCAN_TILE;
        total += 2 * align_up((size_t)(tiles + 1) * sizeof(T), 256);   // tile totals + their scan
        if (tiles <= 1) break;
        m = tiles + 1;
    }
    return total + 256;
}

// out: n+1 entries.  ws: scan_workspace_bytes<T>(n).
template <typename T, typename LoadOp>
static int device_exclusive_scan(LoadOp load, i64 n, T *out, void *ws, cudaStream_t st) {
    const i64 n1 = n + 1;
    const i64 tiles = (n1 + SCAN_TILE - 1) / SCAN_TILE;
    T *totals = (T *)ws;
    scan_tiles_kernel<T, LoadOp><<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(load, n1, out, totals);
    GPC_LAUNCH_CHECK();
    if (tiles > 1) {
        // scan the tile totals in place-ish: totals_scanned has tiles+1 entries
        char *next_ws = (char *)ws + align_up((size_t)(tiles + 1) * sizeof(T), 256);
        T *scanned = (T *)next_ws;
        char *rec_ws = next_ws + align_up((size_t)(tiles + 1) * sizeof(T), 256);
        PtrLoad<T> pl{totals};
        int rc = device_exclusive_scan<T, PtrLoad<T>>(pl, tiles, scanned, rec_ws, st);
        if (rc) return rc;
        scan_add_offsets_kernel<T><<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(out, n1, scanned);
        GPC_LAUNCH_CHECK();
    }
    return GPC_OK;
}

// textio.cu -- ASCII PLY rows on the GPU: the writer's "x y z\n" rows with Python's float repr, and the text reader's rows with
// Python's float() (cli.read_points), so the file tools' text I/O runs at the codec's speed.  Per-value work: textio_core.cuh.
#include "common.cuh"
#include "textio_core.cuh"
#include "textio_tables.cuh"

__device__ const uint64_t g_ryu_pow5_inv[2 * GPC_RYU_POW5_INV_COUNT] = GPC_RYU_POW5_INV_DATA;
__device__ const uint64_t g_ryu_pow5[2 * GPC_RYU_POW5_COUNT] = GPC_RYU_POW5_DATA;
__device__ const uint64_t g_el_pow5[2 * (GPC_EL_POW5_MAX_Q - GPC_EL_POW5_MIN_Q + 1)] = GPC_EL_POW5_DATA;

constexpr int TIO_THREADS = 256;
constexpr int TIO_MAX_ROW = 3 * 24 + 3;      // three values of at most 24 bytes, two spaces and "\n"
constexpr int TIO_CHUNK = 32;                 // text bytes per parser thread: it takes the lines that START in its chunk

// ---------------------------------------------------------------- formatter
__device__ __forceinline__ int tio_row(const float *xyz, i64 r, char *out) {
    int len = 0;
#pragma unroll 1
    for (int c = 0; c < 3; ++c) {
        len += tio_format_double((double)xyz[3 * r + c], out ? out + len : nullptr, g_ryu_pow5_inv, g_ryu_pow5);
        if (out) out[len] = c < 2 ? ' ' : '\n';
        ++len;
    }
    return len;
}

__global__ void __launch_bounds__(TIO_THREADS) ply_row_len_kernel(const float *__restrict__ xyz, i64 n, u32 *__restrict__ len) {
    const i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) len[r] = (u32)tio_row(xyz, r, nullptr);
}

__global__ void __launch_bounds__(TIO_THREADS) ply_row_write_kernel(const float *__restrict__ xyz, i64 n, const u32 *__restrict__ off,
                                                                  char *__restrict__ out, u64 cap) {
    const i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n && off[r + 1] <= cap) tio_row(xyz, r, out + off[r]);    // a short buffer is refused after the read-back
}

static size_t ply_scan_bytes(i64 n) { return align_up((size_t)(n + 1) * sizeof(u32), 256); }

extern "C" size_t gpc_ply_format_workspace_bytes(int64_t n) {
    return 2 * ply_scan_bytes(n) + scan_workspace_bytes<u32>(n);
}

extern "C" int gpc_ply_format_f32(const float *xyz, int64_t n, char *out, uint64_t cap, uint64_t *out_len_h, void *ws,
                                  size_t ws_bytes, void *stream) {
    GPC_REQUIRE(n >= 0 && out_len_h, GPC_EINVAL, "bad argument");
    GPC_REQUIRE(n <= (int64_t)(0xFFFFFFFFull / TIO_MAX_ROW), GPC_EINVAL, "too many rows for u32 text offsets");
    GPC_REQUIRE(ws_bytes >= gpc_ply_format_workspace_bytes(n), GPC_ENOSPC, "workspace too small");
    *out_len_h = 0;
    if (n == 0) return GPC_OK;
    GPC_REQUIRE(xyz && out && ws, GPC_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    u32 *len = (u32 *)ws;
    u32 *off = (u32 *)((char *)ws + ply_scan_bytes(n));
    void *scan_ws = (char *)ws + 2 * ply_scan_bytes(n);
    ply_row_len_kernel<<<cdiv(n, TIO_THREADS), TIO_THREADS, 0, st>>>(xyz, n, len);
    GPC_LAUNCH_CHECK();
    int rc = device_exclusive_scan<u32>(PtrLoad<u32>{len}, n, off, scan_ws, st);
    if (rc) return rc;
    ply_row_write_kernel<<<cdiv(n, TIO_THREADS), TIO_THREADS, 0, st>>>(xyz, n, off, out, cap);
    GPC_LAUNCH_CHECK();
    u32 total = 0;
    GPC_CUDA_CHECK(cudaMemcpyAsync(&total, off + n, sizeof(u32), cudaMemcpyDeviceToHost, st));
    GPC_CUDA_CHECK(cudaStreamSynchronize(st));
    *out_len_h = total;
    if ((u64)total > cap) {
        gpc_set_error("%s:%d: the %u bytes of text do not fit in a %llu-byte buffer", __FILE__, __LINE__, total,
                      (unsigned long long)cap);
        return GPC_EINVAL;
    }
    return GPC_OK;
}

// ---------------------------------------------------------------- parser
// lines end at "\n", "\r\n" or a lone "\r" (universal newlines); line k's content runs from its first byte to its terminator

struct U32x2 {
    u32 rows, host;
    __device__ U32x2() = default;
    __device__ constexpr U32x2(u32 r, u32 h) : rows(r), host(h) {}
    __device__ U32x2 operator+(const U32x2 &o) const { return U32x2(rows + o.rows, host + o.host); }
};
template <> struct ScanZero<U32x2> { __device__ static U32x2 get() { return U32x2(0, 0); } };

__device__ __forceinline__ bool tio_starts_line(const char *t, u64 i) {
    if (i == 0) return true;
    const char p = t[i - 1];
    return p == '\n' || (p == '\r' && t[i] != '\n');
}

// every line starting in chunk c: its status, and with EMIT its row / host entry written at the chunk's offsets
template <bool EMIT>
__device__ __forceinline__ U32x2 tio_chunk_lines(const char *__restrict__ t, u64 nbytes, u64 c, U32x2 base, double *rows,
                                                 u32 *host) {
    const u64 b0 = c * TIO_CHUNK, b1 = min(nbytes, b0 + TIO_CHUNK);
    U32x2 cnt(0, 0);
#pragma unroll 1
    for (u64 i = b0; i < b1; ++i) {
        if (!tio_starts_line(t, i)) continue;
        u64 e = i;
        while (e < nbytes && t[e] != '\n' && t[e] != '\r') ++e;
        double xyz[3];
        const int st = tio_parse_line(t + i, (i64)(e - i), g_el_pow5, xyz);
        if (st == TIO_LINE_ROW) {
            if (EMIT) {
                double *o = rows + 3 * (u64)(base.rows + cnt.rows);
                o[0] = xyz[0]; o[1] = xyz[1]; o[2] = xyz[2];
            }
            ++cnt.rows;
        } else if (st == TIO_LINE_HOST) {
            if (EMIT) {
                u32 *h = host + 3 * (u64)(base.host + cnt.host);
                h[0] = (u32)i; h[1] = (u32)e; h[2] = base.rows + cnt.rows;
            }
            ++cnt.host;
        }
        i = e;      // past the content; the loop's ++i steps over the terminator's first byte
    }
    return cnt;
}

__global__ void __launch_bounds__(TIO_THREADS) text_parse_count_kernel(const char *__restrict__ t, u64 nbytes, i64 chunks,
                                                                     U32x2 *__restrict__ cnt) {
    const i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < chunks) cnt[c] = tio_chunk_lines<false>(t, nbytes, (u64)c, U32x2(0, 0), nullptr, nullptr);
}

__global__ void __launch_bounds__(TIO_THREADS) text_parse_emit_kernel(const char *__restrict__ t, u64 nbytes, i64 chunks,
                                                                    const U32x2 *__restrict__ off, double *__restrict__ rows,
                                                                    u32 *__restrict__ host) {
    const i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < chunks) tio_chunk_lines<true>(t, nbytes, (u64)c, off[c], rows, host);
}

static i64 text_chunks(u64 nbytes) { return (i64)((nbytes + TIO_CHUNK - 1) / TIO_CHUNK); }

extern "C" size_t gpc_text_parse_workspace_bytes(uint64_t nbytes) {
    const i64 chunks = text_chunks(nbytes);
    return 2 * align_up((size_t)(chunks + 1) * sizeof(U32x2), 256) + scan_workspace_bytes<U32x2>(chunks);
}

extern "C" int gpc_text_parse_xyz(const char *text, uint64_t nbytes, double *rows, uint32_t *n_rows_h, uint32_t *host_lines,
                                  uint32_t *n_host_h, void *ws, size_t ws_bytes, void *stream) {
    GPC_REQUIRE(n_rows_h && n_host_h, GPC_EINVAL, "null count pointer");
    GPC_REQUIRE(nbytes < (1ull << 32), GPC_EINVAL, "text of 2^32 bytes or more (u32 offsets)");
    GPC_REQUIRE(ws_bytes >= gpc_text_parse_workspace_bytes(nbytes), GPC_ENOSPC, "workspace too small");
    *n_rows_h = *n_host_h = 0;
    if (nbytes == 0) return GPC_OK;
    GPC_REQUIRE(text && rows && host_lines && ws, GPC_EINVAL, "null pointer");
    cudaStream_t st = as_stream(stream);
    const i64 chunks = text_chunks(nbytes);
    const size_t arr = align_up((size_t)(chunks + 1) * sizeof(U32x2), 256);
    U32x2 *cnt = (U32x2 *)ws, *off = (U32x2 *)((char *)ws + arr);
    void *scan_ws = (char *)ws + 2 * arr;
    // pass 1: rows and host lines of the lines starting in each chunk; scan; pass 2: the same lines again, written at the offsets.
    // Per 32-byte chunk rather than per line: no line-start array, so the workspace is 16 bytes per 32 bytes of text.
    text_parse_count_kernel<<<cdiv(chunks, TIO_THREADS), TIO_THREADS, 0, st>>>(text, nbytes, chunks, cnt);
    GPC_LAUNCH_CHECK();
    int rc = device_exclusive_scan<U32x2>(PtrLoad<U32x2>{cnt}, chunks, off, scan_ws, st);
    if (rc) return rc;
    text_parse_emit_kernel<<<cdiv(chunks, TIO_THREADS), TIO_THREADS, 0, st>>>(text, nbytes, chunks, off, rows, host_lines);
    GPC_LAUNCH_CHECK();
    U32x2 total;
    GPC_CUDA_CHECK(cudaMemcpyAsync(&total, off + chunks, sizeof(U32x2), cudaMemcpyDeviceToHost, st));
    GPC_CUDA_CHECK(cudaStreamSynchronize(st));
    *n_rows_h = total.rows;
    *n_host_h = total.host;
    return GPC_OK;
}

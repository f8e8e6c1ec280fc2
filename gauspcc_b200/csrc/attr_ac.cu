// attr_ac.cu -- HAC's chunked attribute coder (SURVEY.md 8f-4): the step right after the anchor geometry in
// conduct_encoding (HAC/scene/gaussian_model.py:1134-1206, decode :1239-1310).
//
// Replaces HAC/submodules/arithmetic.zip!arithmetic/arithmetic_kernel.cu:
//   calculate_cdf_kernel      :11-28    lower[n][Lp] = Gaussian CDF at the Lp = max - min + 2 quantisation bin edges
//   encode_arithmetic_kernel  :94-163   one 32-bit low/high range coder per chunk of 10 000 symbols, launched <<<chunks, 1>>>
//   merge_chunks_kernel       :166-183  one THREAD per chunk sums the lengths before it and copies its bytes
//   decode_arithmetic_kernel  :290-356  per chunk, binary search in the float CDF row (binsearch, :264-287)
// Same streams, same per-chunk byte counts, same decoded symbols (the format is the reference's: a chunk is one serial coder).
//
// B200 layout of the work:
//  * the table lower[n][Lp] (n * Lp * 4 bytes: 2.5 GB for 10 M symbols at Lp = 64, written once and read back with one
//    dependent, uncoalesced load per symbol) is never built on the Gaussian path: a fully parallel kernel evaluates the TWO
//    bin edges a symbol needs and writes 8 bytes per symbol (c_low, c_high); the decoder evaluates candidates on the fly;
//  * a chunk's coder is one WARP whose lanes all carry the coder state: the 32 lanes fetch 32 symbols' inputs with one
//    coalesced load and hand them round with shuffles; in the decoder the 32 lanes evaluate 32 candidate symbols at once
//    (window centred on the mean, else a 32-ary search), where the reference walks a binary search of dependent loads;
//  * bits leave through a 64-bit register, four bytes per store; chunks are merged by one CTA per chunk after a device scan;
//  * HAC++'s mixture of K <= 4 Gaussians (encodings_cuda.py:203-314 builds the table as clamp(sum_k cdf_k * prob_k, 0, 1)) goes
//    through the same two kernels with MixModel, which restates that float sum operation for operation; the Bernoulli mask
//    coder (:435-500, a table whose rows are all [0, 1 - p, 1]) reads its one shared row (SharedRowModel).
//
// Arithmetic restated exactly (float erfc, the double product for the bin edge, round-to-nearest-even to int, the `+ symbol`
// that keeps the integer CDF strictly increasing); `tests/test_attr_coder.py` checks the bytes against the C oracle and, on the
// GPU box, against the reference extension itself when oracle/_ref holds it.
#include "common.cuh"

namespace {

constexpr int ATTR_PRECISION = 16;

// arithmetic_kernel.cu:7-9 -- erfc on a float argument is the float erfc; the halving is exact in either width
__device__ __forceinline__ float attr_gauss_cdf(float x, float mean, float scale) {
    return 0.5f * erfcf(-(x - mean) / (scale * 1.41421356237309504880f));
}
// :22-26  sample_value = (min_value + i - 0.5) * Q  (evaluated in double, stored as float)
__device__ __forceinline__ float attr_edge(int min_value, int i, float q) {
    return (float)(((double)(min_value + i) - 0.5) * (double)q);
}
__device__ __forceinline__ float attr_clamp_scale(float s) { return (float)fmax((double)s, 1e-9); }           // :22

__global__ void attr_cdf_table_kernel(const float *__restrict__ mean, const float *__restrict__ scale, const float *__restrict__ Q,
                                      i64 n, int min_value, int Lp, float *__restrict__ lower) {
    const i64 t = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * Lp) return;
    const i64 row = t / Lp;
    const int i = (int)(t - row * Lp);
    lower[t] = attr_gauss_cdf(attr_edge(min_value, i, Q[row]), mean[row], attr_clamp_scale(scale[row]));
}

// ---- the models a symbol's integer CDF entries come from:  v(row, m) = rn(cdf(row, m) * (2^16 - (Lp - 1))) + m.
// A model's Row is what one symbol needs; shfl() hands lane src's row to the warp (the decoder fetches 32 rows with one coalesced
// load), and the centred models give centre(): the symbol the decoder's first window of 32 candidates is centred on.
struct TableModel {
    const float *cdf; int Lp; float scale16;
    struct Row { i64 base; };
    __device__ __forceinline__ Row row(i64 r) const { return Row{r * Lp}; }
    __device__ __forceinline__ Row shfl(const Row &rw, int src) const { return Row{__shfl_sync(0xFFFFFFFFu, rw.base, src)}; }
    __device__ __forceinline__ u32 v(const Row &rw, int m) const { return (u32)(__float2int_rn(cdf[rw.base + m] * scale16) + m); }
};
// integer CDF rows as the geometry codec's head kernel writes them (uint16 bit pattern of kit/op.py:67-79; the top of the last
// symbol is 0x10000 by rule): the chunked coder on the occupancy symbols themselves (container version 2, SURVEY 8f-3)
struct U16Model {
    const u16 *cdf; int Lp;
    struct Row { i64 base; };
    __device__ __forceinline__ Row row(i64 r) const { return Row{r * Lp}; }
    __device__ __forceinline__ u32 v(const Row &rw, int m) const { return (u32)cdf[rw.base + m]; }
};
// ONE float CDF row shared by every symbol: the Bernoulli mask coder (encodings_cuda.py:435-500), whose table is [0, 1 - p, 1]
// on every row.  The same v() as TableModel on that row.
struct SharedRowModel {
    const float *cdf; float scale16;
    struct Row {};
    __device__ __forceinline__ Row row(i64) const { return Row{}; }
    __device__ __forceinline__ Row shfl(const Row &rw, int) const { return rw; }
    __device__ __forceinline__ u32 v(const Row &, int m) const { return (u32)(__float2int_rn(cdf[m] * scale16) + m); }
};
struct GaussModel {
    const float *mean, *scale, *Q; int min_value; float scale16;
    struct Row { float mean, scale, q; };
    __device__ __forceinline__ Row row(i64 r) const { return Row{mean[r], attr_clamp_scale(scale[r]), Q[r]}; }
    __device__ __forceinline__ Row shfl(const Row &rw, int src) const {
        return Row{__shfl_sync(0xFFFFFFFFu, rw.mean, src), __shfl_sync(0xFFFFFFFFu, rw.scale, src), __shfl_sync(0xFFFFFFFFu, rw.q, src)};
    }
    __device__ __forceinline__ int centre(const Row &rw) const { return __float2int_rn(rw.mean / rw.q) - min_value; }
    __device__ __forceinline__ u32 v(const Row &rw, int m) const {
        return (u32)(__float2int_rn(attr_gauss_cdf(attr_edge(min_value, m, rw.q), rw.mean, rw.scale) * scale16) + m);
    }
};
// mixture of K Gaussians (HAC++'s encoder_gaussian_mixed, encodings_cuda.py:203-314): the table the reference builds is
//   lower = clamp(sum_k calculate_cdf(mean_k, scale_k) * prob_k, 0, 1)
// in float32, one rounding per product and per sum, in list order.  v() restates exactly that: __fmul_rn / __fadd_rn keep nvcc
// from contracting acc + c * p into an FMA, and the clamp is written with comparisons so that a NaN passes through as it does
// in torch.clamp.  mean / scale / prob are [K][n].
template <int K>
struct MixModel {
    const float *mean, *scale, *prob, *Q; i64 n; int min_value; float scale16;
    struct Row { float mean[K], scale[K], prob[K], q; };
    __device__ __forceinline__ Row row(i64 r) const {
        Row rw;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            rw.mean[k] = mean[k * n + r];
            rw.scale[k] = attr_clamp_scale(scale[k * n + r]);
            rw.prob[k] = prob[k * n + r];
        }
        rw.q = Q[r];
        return rw;
    }
    __device__ __forceinline__ Row shfl(const Row &rw, int src) const {
        Row o;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            o.mean[k] = __shfl_sync(0xFFFFFFFFu, rw.mean[k], src);
            o.scale[k] = __shfl_sync(0xFFFFFFFFu, rw.scale[k], src);
            o.prob[k] = __shfl_sync(0xFFFFFFFFu, rw.prob[k], src);
        }
        o.q = __shfl_sync(0xFFFFFFFFu, rw.q, src);
        return o;
    }
    // the mean of the most probable component (ties: the first): where most of the row's mass is when the components are apart
    __device__ __forceinline__ int centre(const Row &rw) const {
        float best = rw.prob[0], c = rw.mean[0];
#pragma unroll
        for (int k = 1; k < K; ++k)
            if (rw.prob[k] > best) { best = rw.prob[k]; c = rw.mean[k]; }
        return __float2int_rn(c / rw.q) - min_value;
    }
    __device__ __forceinline__ u32 v(const Row &rw, int m) const {
        const float edge = attr_edge(min_value, m, rw.q);
        float acc = __fmul_rn(attr_gauss_cdf(edge, rw.mean[0], rw.scale[0]), rw.prob[0]);
#pragma unroll
        for (int k = 1; k < K; ++k) acc = __fadd_rn(acc, __fmul_rn(attr_gauss_cdf(edge, rw.mean[k], rw.scale[k]), rw.prob[k]));
        acc = acc < 0.0f ? 0.0f : (acc > 1.0f ? 1.0f : acc);
        return (u32)(__float2int_rn(acc * scale16) + m);
    }
};

// c_low / c_high of every symbol (:121-122), fully parallel
template <typename Model>
__global__ void attr_bounds_kernel(Model md, const int16_t *__restrict__ sym, i64 n, int max_symbol, uint2 *__restrict__ bounds,
                                   int *__restrict__ status) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = sym[i];
    if (s < 0 || s > max_symbol) { atomicOr(status, 1); bounds[i] = make_uint2(0u, 1u); return; }
    const typename Model::Row rw = md.row(i);
    const u32 lo = md.v(rw, s);
    const u32 hi = s == max_symbol ? 0x10000u : md.v(rw, s + 1);
    bounds[i] = make_uint2(lo, hi);
}

// ---- bit output of one chunk: 64-bit register, big-endian words of four bytes, lane 0 stores
struct BitWriter {
    u8 *out; i64 cap; i64 pos; u64 acc; int nb; bool overflow;
    __device__ __forceinline__ void put(u32 v, int k, bool store) {                // k in 1..32, v < 2^k
        acc = (acc << k) | v;
        nb += k;
        if (nb >= 32) {
            const u32 w = (u32)(acc >> (nb - 32));
            if (pos + 4 <= cap) { if (store) *(u32 *)(out + pos) = __byte_perm(w, 0, 0x0123); }
            else overflow = true;
            pos += 4;
            nb -= 32;
        }
    }
    __device__ __forceinline__ void run(u32 bit, u64 count, bool store) {
        while (count) {
            const int k = count > 32 ? 32 : (int)count;
            put(bit ? (k == 32 ? 0xFFFFFFFFu : ((1u << k) - 1u)) : 0u, k, store);
            count -= k;
        }
    }
    __device__ __forceinline__ void finish(bool store) {                           // OutCacheString::flush, :76-83
        if (nb & 7) put(0u, 8 - (nb & 7), store);
        while (nb > 0) {
            const u32 b = (u32)(acc >> (nb - 8)) & 0xFFu;
            if (pos + 1 <= cap) { if (store) out[pos] = (u8)b; }
            else overflow = true;
            pos += 1;
            nb -= 8;
        }
    }
};

struct BoundsLoad {                                  // (c_low, c_high) as attr_bounds_kernel wrote them
    const uint2 *p;
    __device__ __forceinline__ uint2 operator()(i64 i) const { return p[i]; }
};
struct LohiLoad {                                    // c_low | c_high << 16, c_high == 0 meaning 0x10000 (gpc_head_cdf_sym)
    const u32 *p;
    __device__ __forceinline__ uint2 operator()(i64 i) const {
        const u32 e = p[i];
        return make_uint2(e & 0xFFFFu, (e >> 16) ? (e >> 16) : 0x10000u);
    }
};
// one warp per chunk (:94-163).  Every lane runs the coder on the same values; lane 0 writes.
template <typename Load>
__global__ void __launch_bounds__(128) attr_encode_chunks_kernel(Load bounds, i64 n, int chunk_size, int chunks,
                                                                u8 *__restrict__ cache, i64 cap, i32 *__restrict__ cnt,
                                                                int *__restrict__ status, const u32 *__restrict__ starts = nullptr) {
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (w >= chunks) return;
    // chunks of chunk_size symbols, or (starts given) chunk w = symbols [starts[w], starts[w + 1]) of at most chunk_size symbols
    const i64 base = starts ? (i64)starts[w] : (i64)w * chunk_size;
    const int len = starts ? (int)(starts[w + 1] - starts[w]) : (int)min((i64)chunk_size, n - base);
    BitWriter bw{cache + (i64)w * cap, cap, 0, 0ull, 0, false};
    const bool store = lane == 0;
    u32 low = 0u, high = 0xFFFFFFFFu;
    u64 pending = 0;
    uint2 nxt = lane < len ? bounds(base + lane) : make_uint2(0u, 0u);
    for (int j0 = 0; j0 < len; j0 += 32) {
        const uint2 cur = nxt;
        if (j0 + 32 + lane < len) nxt = bounds(base + j0 + 32 + lane);
        const int m = min(32, len - j0);
        for (int j = 0; j < m; ++j) {
            const u64 c_low = __shfl_sync(0xFFFFFFFFu, cur.x, j);
            const u64 c_high = __shfl_sync(0xFFFFFFFFu, cur.y, j);
            const u64 span = (u64)high - (u64)low + 1ull;
            high = (low - 1u) + (u32)((span * c_high) >> ATTR_PRECISION);
            low = low + (u32)((span * c_low) >> ATTR_PRECISION);
            for (;;) {                                                              // :127-148, the equal leading bits in one step
                const u32 diff = low ^ high;
                if (!(diff & 0x80000000u)) {
                    const int sh = diff ? __clz(diff) : 32;
                    const u32 first = low >> 31;
                    bw.put(first, 1, store);
                    if (pending) { bw.run(first ^ 1u, pending, store); pending = 0; }
                    if (sh > 1) bw.put(sh == 32 ? (low & 0x7FFFFFFFu) : ((low << 1) >> (32 - (sh - 1))), sh - 1, store);
                    if (sh == 32) { low = 0u; high = 0xFFFFFFFFu; }
                    else { low <<= sh; high = (high << sh) | ((1u << sh) - 1u); }
                } else if (low >= 0x40000000u && high < 0xC0000000u) {
                    ++pending;
                    low = (low << 1) & 0x7FFFFFFFu;
                    high = (high << 1) | 0x80000001u;
                } else {
                    break;
                }
            }
        }
    }
    ++pending;                                                                      // :151-160
    const u32 last = low < 0x40000000u ? 0u : 1u;
    bw.put(last, 1, store);
    bw.run(last ^ 1u, pending, store);
    bw.finish(store);
    if (store) {
        cnt[w] = (i32)bw.pos;
        if (bw.overflow) atomicOr(status, 2);
    }
}

// :166-183 with the prefix sums from a device scan; one CTA per chunk
__global__ void __launch_bounds__(256) attr_merge_kernel(const u8 *__restrict__ cache, i64 cap, const u32 *__restrict__ offsets,
                                                        u8 *__restrict__ out) {
    const int w = blockIdx.x;
    const u32 o = offsets[w], len = offsets[w + 1] - o;
    const u8 *src = cache + (i64)w * cap;
    for (u32 b = threadIdx.x; b < len; b += blockDim.x) out[o + b] = src[b];
}

// ---- bit input of one chunk (InCacheString, :237-262): zeros after the last byte.  The lanes hold 128 bytes of the stream
// (lane l: bytes 4l .. 4l+3 of the current segment, big-endian) and pass words round with shuffles.
struct BitReader {
    const u8 *in; i64 len; i64 seg; u32 mine; u64 buf; int nb; i64 word;
    __device__ __forceinline__ u32 load_lane(i64 s, int lane) const {
        const i64 b = (s * 32 + lane) * 4;
        u32 w = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) w = (w << 8) | (b + k < len ? (u32)in[b + k] : 0u);
        return w;
    }
    __device__ __forceinline__ void init(const u8 *p, i64 l, int lane) {
        in = p; len = l; seg = 0; mine = load_lane(0, lane); buf = 0; nb = 0; word = 0;
    }
    __device__ __forceinline__ u32 next_word(int lane) {
        const i64 s = word >> 5;
        if (s != seg) { seg = s; mine = load_lane(s, lane); }
        const u32 w = __shfl_sync(0xFFFFFFFFu, mine, (int)(word & 31));
        ++word;
        return w;
    }
    __device__ __forceinline__ u32 get(int k, int lane) {                           // k in 1..32
        if (nb < k) { buf = (buf << 32) | next_word(lane); nb += 32; }
        const u32 v = (u32)((buf >> (nb - k)) & (k == 32 ? 0xFFFFFFFFull : ((1ull << k) - 1ull)));
        nb -= k;
        return v;
    }
};

// largest m in [0, max_symbol] with v(m) <= count, 0 when there is none: what binsearch (:264-287) returns on a strictly
// increasing row.  Lanes test 32 candidates per round.
template <typename Model>
__device__ __forceinline__ int attr_search(const Model &md, const typename Model::Row &rw, u32 count, int max_symbol, int lo, int hi,
                                           int lane) {
    // invariant: the answer is in [lo, hi); v(lo) <= count or lo == 0
    while (hi - lo > 1) {
        const int step = (hi - lo - 1 + 31) / 32;
        const int m = lo + (lane + 1) * step;
        const bool le = m < hi && md.v(rw, m) <= count;
        const int k = __popc(__ballot_sync(0xFFFFFFFFu, le));
        const int nlo = lo + k * step;
        hi = min(hi, lo + (k + 1) * step);
        lo = nlo;
    }
    return lo;
}

template <typename Model, bool CENTRED, typename SymT>
__global__ void __launch_bounds__(128) attr_decode_chunks_kernel(Model md, const u8 *__restrict__ in, const u32 *__restrict__ offsets,
                                                                i64 n, int chunk_size, int chunks, int max_symbol,
                                                                SymT *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (w >= chunks) return;
    const i64 base = (i64)w * chunk_size;
    const int len = (int)min((i64)chunk_size, n - base);
    BitReader br;
    br.init(in + offsets[w], (i64)(offsets[w + 1] - offsets[w]), lane);
    u32 low = 0u, high = 0xFFFFFFFFu;
    u32 value = br.get(32, lane);                                                   // initialize, :258-262
    for (int j0 = 0; j0 < len; j0 += 32) {
        const int m = min(32, len - j0);
        typename Model::Row mine = md.row(base + j0 + min(lane, m - 1));            // one coalesced fetch for 32 symbols
        int my_sym = 0;
        for (int j = 0; j < m; ++j) {
            const typename Model::Row rw = md.shfl(mine, j);
            const u64 span = (u64)high - (u64)low + 1ull;
            // count = uint16(((value - low + 1) * 2^16 - 1) / span), :318-319 -- float estimate, exact correction
            const u64 X = (((u64)value - (u64)low + 1ull) << ATTR_PRECISION) - 1ull;
            u64 q = (u64)(__fdividef((float)(X >> 8), (float)(span >> 8)));
            if (q > 0) --q;
            u64 r = X - q * span;                                                   // wraps when the estimate overshoots
            if (r >= span) { r -= span; ++q; }
            if (r >= span) { r -= span; ++q; }
            if (r >= span) q = X / span;                                            // corrupt stream (value outside [low, high])
            const u32 count = (u32)(q & 0xFFFFu);
            int s;
            u32 c_low = 0, c_high = 0;
            bool have = false;
            if constexpr (CENTRED) {
                // window of 32 candidates around the model's centre: exact when the answer falls inside (the usual case)
                const int centre = md.centre(rw);
                const int w0 = max(0, min(centre - 15, max_symbol - 31));
                const int mm = w0 + lane;
                const u32 vv = mm <= max_symbol + 1 ? md.v(rw, min(mm, max_symbol + 1)) : 0u;
                const u32 bal = __ballot_sync(0xFFFFFFFFu, mm <= max_symbol && vv <= count);
                const int k = __popc(bal);
                const int top = min(31, max_symbol - w0);                          // last lane that holds a symbol
                if (k == 0 && w0 > 0) s = attr_search(md, rw, count, max_symbol, 0, w0, lane);
                else if (k == top + 1 && w0 + top < max_symbol) s = attr_search(md, rw, count, max_symbol, w0 + top, max_symbol + 1, lane);
                else {
                    s = w0 + max(k - 1, 0);
                    const int ls = s - w0;
                    c_low = __shfl_sync(0xFFFFFFFFu, vv, ls);
                    c_high = __shfl_sync(0xFFFFFFFFu, vv, min(ls + 1, 31));
                    have = ls + 1 <= 31;
                }
            } else {
                s = attr_search(md, rw, count, max_symbol, 0, max_symbol + 1, lane);
            }
            if (!have) { c_low = md.v(rw, s); c_high = s == max_symbol ? 0x10000u : md.v(rw, s + 1); }
            if (s == max_symbol) c_high = 0x10000u;
            if (lane == j) my_sym = s;
            high = (low - 1u) + (u32)((span * (u64)c_high) >> ATTR_PRECISION);
            low = low + (u32)((span * (u64)c_low) >> ATTR_PRECISION);
            for (;;) {                                                              // :333-353
                const u32 diff = low ^ high;
                if (!(diff & 0x80000000u)) {
                    const int sh = diff ? __clz(diff) : 32;
                    const u32 bits = br.get(sh, lane);
                    if (sh == 32) { low = 0u; high = 0xFFFFFFFFu; value = bits; }
                    else { low <<= sh; high = (high << sh) | ((1u << sh) - 1u); value = (value << sh) | bits; }
                } else if (low >= 0x40000000u && high < 0xC0000000u) {
                    low = (low << 1) & 0x7FFFFFFFu;
                    high = (high << 1) | 0x80000001u;
                    value -= 0x40000000u;
                    value = (value << 1) | br.get(1, lane);
                } else {
                    break;
                }
            }
        }
        if (lane < m) out[base + j0 + lane] = (SymT)my_sym;
    }
}

struct AttrWs { uint2 *bounds; u8 *cache; void *scan_ws; int *status; i64 cap; };

size_t attr_layout(i64 n, int chunk_size, void *ws, AttrWs *L) {
    const i64 chunks = (n + chunk_size - 1) / chunk_size;
    const i64 cap = (i64)chunk_size * 4;                                            // the reference's per-chunk cache, :197
    char *b = (char *)ws;
    size_t off = 0;
    auto take = [&](size_t bytes) { void *p = b ? b + off : nullptr; off += align_up(bytes, 256); return p; };
    L->status = (int *)take(256);
    L->bounds = (uint2 *)take((size_t)n * 8);
    L->cache = (u8 *)take((size_t)chunks * cap);
    L->scan_ws = take(scan_workspace_bytes<u32>(chunks + 1) + 1024);
    L->cap = cap;
    return off;
}

int attr_check(i64 n, int Lp, int chunk_size) {
    GPC_REQUIRE(n >= 0 && n < (1ll << 31), GPC_EINVAL, "n out of range");
    GPC_REQUIRE(Lp >= 2 && Lp <= 32768, GPC_EINVAL, "Lp out of range");
    GPC_REQUIRE(chunk_size >= 1 && chunk_size <= (1 << 24), GPC_EINVAL, "chunk_size out of range");
    return GPC_OK;
}

int attr_status(const AttrWs &L, cudaStream_t st, const char *what) {
    int h = 0;
    GPC_CUDA_CHECK(cudaMemcpyAsync(&h, L.status, 4, cudaMemcpyDeviceToHost, st));
    GPC_CUDA_CHECK(cudaStreamSynchronize(st));
    if (h & 1) { gpc_set_error("%s: a symbol is outside [0, Lp - 2]", what); return GPC_EINVAL; }
    if (h & 2) { gpc_set_error("%s: per-chunk output cache too small", what); return GPC_ENOSPC; }
    return GPC_OK;
}

template <typename Model>
int attr_encode(Model md, const int16_t *sym, i64 n, int Lp, int chunk_size, i32 *cnt, u32 *offsets, void *ws, size_t ws_bytes,
                cudaStream_t st) {
    AttrWs L;
    GPC_REQUIRE(ws && ws_bytes >= attr_layout(n, chunk_size, ws, &L), GPC_ENOSPC, "workspace too small");
    const int chunks = (int)((n + chunk_size - 1) / chunk_size);
    GPC_CUDA_CHECK(cudaMemsetAsync(L.status, 0, 4, st));
    if (n == 0) { GPC_CUDA_CHECK(cudaMemsetAsync(offsets, 0, 4, st)); return GPC_OK; }
    attr_bounds_kernel<Model><<<cdiv(n, 256), 256, 0, st>>>(md, sym, n, Lp - 2, L.bounds, L.status);
    GPC_LAUNCH_CHECK();
    attr_encode_chunks_kernel<BoundsLoad><<<cdiv(chunks, 4), 128, 0, st>>>(BoundsLoad{L.bounds}, n, chunk_size, chunks, L.cache, L.cap, cnt, L.status);
    GPC_LAUNCH_CHECK();
    PtrLoad<u32> pl{(const u32 *)cnt};
    int rc = device_exclusive_scan<u32, PtrLoad<u32>>(pl, chunks, offsets, L.scan_ws, st);
    if (rc) return rc;
    return attr_status(L, st, "attribute encoder");
}

template <typename Model, bool CENTRED, typename SymT>
int attr_decode(Model md, const u8 *in, const i32 *cnt, i64 n, int Lp, int chunk_size, SymT *sym, void *ws, size_t ws_bytes,
                cudaStream_t st) {
    AttrWs L;
    GPC_REQUIRE(ws && ws_bytes >= attr_layout(n, chunk_size, ws, &L), GPC_ENOSPC, "workspace too small");
    if (n == 0) return GPC_OK;
    const int chunks = (int)((n + chunk_size - 1) / chunk_size);
    u32 *offsets = (u32 *)L.bounds;                                                 // the bounds array is free on this side
    PtrLoad<u32> pl{(const u32 *)cnt};
    int rc = device_exclusive_scan<u32, PtrLoad<u32>>(pl, chunks, offsets, L.scan_ws, st);   // compute_cumsum, :358-363
    if (rc) return rc;
    attr_decode_chunks_kernel<Model, CENTRED, SymT><<<cdiv(chunks, 4), 128, 0, st>>>(md, in, offsets, n, chunk_size, chunks, Lp - 2, sym);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

}  // namespace

extern "C" int gpc_attr_calculate_cdf(const float *mean, const float *scale, const float *Q, int64_t n, int min_value, int max_value,
                                      float *lower, void *stream) {
    const int Lp = max_value - min_value + 2;
    GPC_REQUIRE(n >= 0 && Lp >= 2, GPC_EINVAL, "bad argument");
    if (n == 0) return GPC_OK;
    attr_cdf_table_kernel<<<cdiv(n * Lp, 256), 256, 0, as_stream(stream)>>>(mean, scale, Q, n, min_value, Lp, lower);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

extern "C" size_t gpc_attr_workspace_bytes(int64_t n, int chunk_size) {
    AttrWs L;
    if (n < 0 || chunk_size < 1) return 0;
    return attr_layout(n, chunk_size, nullptr, &L);
}

extern "C" int gpc_attr_encode_table(const int16_t *sym, const float *cdf, int64_t n, int Lp, int chunk_size, int32_t *cnt,
                                     uint32_t *offsets, void *ws, size_t ws_bytes, void *stream) {
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    TableModel md{cdf, Lp, (float)((1 << ATTR_PRECISION) - (Lp - 1))};
    return attr_encode(md, sym, n, Lp, chunk_size, cnt, offsets, ws, ws_bytes, as_stream(stream));
}

extern "C" int gpc_attr_encode_gaussian(const int16_t *sym, const float *mean, const float *scale, const float *Q, int64_t n,
                                        int min_value, int max_value, int chunk_size, int32_t *cnt, uint32_t *offsets, void *ws,
                                        size_t ws_bytes, void *stream) {
    const int Lp = max_value - min_value + 2;
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    GaussModel md{mean, scale, Q, min_value, (float)((1 << ATTR_PRECISION) - (Lp - 1))};
    return attr_encode(md, sym, n, Lp, chunk_size, cnt, offsets, ws, ws_bytes, as_stream(stream));
}

extern "C" int gpc_attr_merge_chunks(const void *ws, int64_t n, int chunk_size, const uint32_t *offsets, uint8_t *out, void *stream) {
    AttrWs L;
    attr_layout(n, chunk_size, (void *)ws, &L);
    if (n <= 0) return GPC_OK;
    const int chunks = (int)((n + chunk_size - 1) / chunk_size);
    attr_merge_kernel<<<chunks, 256, 0, as_stream(stream)>>>(L.cache, L.cap, offsets, out);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

extern "C" int gpc_attr_decode_table(const float *cdf, const uint8_t *in, const int32_t *cnt, int64_t n, int Lp, int chunk_size,
                                     int16_t *sym, void *ws, size_t ws_bytes, void *stream) {
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    TableModel md{cdf, Lp, (float)((1 << ATTR_PRECISION) - (Lp - 1))};
    return attr_decode<TableModel, false, int16_t>(md, in, cnt, n, Lp, chunk_size, sym, ws, ws_bytes, as_stream(stream));
}

extern "C" int gpc_attr_decode_gaussian(const float *mean, const float *scale, const float *Q, const uint8_t *in, const int32_t *cnt,
                                        int64_t n, int min_value, int max_value, int chunk_size, int16_t *sym, void *ws,
                                        size_t ws_bytes, void *stream) {
    const int Lp = max_value - min_value + 2;
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    GaussModel md{mean, scale, Q, min_value, (float)((1 << ATTR_PRECISION) - (Lp - 1))};
    return attr_decode<GaussModel, true, int16_t>(md, in, cnt, n, Lp, chunk_size, sym, ws, ws_bytes, as_stream(stream));
}

// ---- HAC++'s mixture coders and the Bernoulli mask coder without a per-symbol table: the same bytes as the table entry points fed
// with the table the reference builds, through the same workspace and gpc_attr_merge_chunks
// k = 1..4 components: calls run(MixModel<k>{...})
template <typename Run>
static int mixture_run(int k, const float *mean, const float *scale, const float *prob, const float *Q, i64 n, int min_value, int Lp,
                       Run run) {
    GPC_REQUIRE(k >= 1 && k <= 4, GPC_EINVAL, "mixture coder: 1 to 4 components are supported");
    const float s16 = (float)((1 << ATTR_PRECISION) - (Lp - 1));
    switch (k) {
    case 1: return run(MixModel<1>{mean, scale, prob, Q, n, min_value, s16});
    case 2: return run(MixModel<2>{mean, scale, prob, Q, n, min_value, s16});
    case 3: return run(MixModel<3>{mean, scale, prob, Q, n, min_value, s16});
    default: return run(MixModel<4>{mean, scale, prob, Q, n, min_value, s16});
    }
}

extern "C" int gpc_mixture_encode(const int16_t *sym, const float *mean, const float *scale, const float *prob, const float *Q,
                                  int64_t n, int k, int min_value, int max_value, int chunk_size, int32_t *cnt, uint32_t *offsets,
                                  void *ws, size_t ws_bytes, void *stream) {
    const int Lp = max_value - min_value + 2;
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    return mixture_run(k, mean, scale, prob, Q, n, min_value, Lp, [&](auto md) {
        return attr_encode(md, sym, n, Lp, chunk_size, cnt, offsets, ws, ws_bytes, as_stream(stream));
    });
}

extern "C" int gpc_mixture_decode(const float *mean, const float *scale, const float *prob, const float *Q, const uint8_t *in,
                                  const int32_t *cnt, int64_t n, int k, int min_value, int max_value, int chunk_size, int16_t *sym,
                                  void *ws, size_t ws_bytes, void *stream) {
    const int Lp = max_value - min_value + 2;
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    return mixture_run(k, mean, scale, prob, Q, n, min_value, Lp, [&](auto md) {
        return attr_decode<decltype(md), true, int16_t>(md, in, cnt, n, Lp, chunk_size, sym, ws, ws_bytes, as_stream(stream));
    });
}

extern "C" int gpc_row_encode(const int16_t *sym, const float *row, int64_t n, int Lp, int chunk_size, int32_t *cnt, uint32_t *offsets,
                              void *ws, size_t ws_bytes, void *stream) {
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    SharedRowModel md{row, (float)((1 << ATTR_PRECISION) - (Lp - 1))};
    return attr_encode(md, sym, n, Lp, chunk_size, cnt, offsets, ws, ws_bytes, as_stream(stream));
}

extern "C" int gpc_row_decode(const float *row, const uint8_t *in, const int32_t *cnt, int64_t n, int Lp, int chunk_size, int16_t *sym,
                              void *ws, size_t ws_bytes, void *stream) {
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    SharedRowModel md{row, (float)((1 << ATTR_PRECISION) - (Lp - 1))};
    return attr_decode<SharedRowModel, false, int16_t>(md, in, cnt, n, Lp, chunk_size, sym, ws, ws_bytes, as_stream(stream));
}

// ---- the same chunked coder on the geometry codec's own symbols (container version 2, SURVEY 8f-3): the occupancy streams of a
// level coded on the GPU in chunks instead of by one serial host coder per stream.  Not the reference's bitstream (torchac codes a
// stream as ONE coder): an opt-in container next to the drop-in one.
// chunks: chunk w = symbols [starts[w], starts[w + 1]) of lohi, at most max_chunk symbols each (the streams of a scene one after
// the other, every stream cut into chunks of its own length).  cnt[chunks], offsets[chunks + 1]; no host synchronisation.
static size_t chunk_var_layout(int chunks, int max_chunk, void *ws, AttrWs *L) {
    char *b = (char *)ws;
    size_t off = 0;
    auto take = [&](size_t bytes) { void *p = b ? b + off : nullptr; off += align_up(bytes, 256); return p; };
    L->status = (int *)take(256);
    L->bounds = nullptr;
    L->cap = (i64)max_chunk * 4;
    L->cache = (u8 *)take((size_t)chunks * L->cap);
    L->scan_ws = take(scan_workspace_bytes<u32>(chunks + 1) + 1024);
    return off;
}
extern "C" size_t gpc_chunk_workspace_bytes(int chunks, int max_chunk) {
    AttrWs L;
    if (chunks < 0 || max_chunk < 1) return 0;
    return chunk_var_layout(chunks, max_chunk, nullptr, &L);
}
extern "C" int gpc_chunk_encode_lohi(const uint32_t *lohi, const uint32_t *starts, int chunks, int max_chunk, int32_t *cnt,
                                     uint32_t *offsets, void *ws, size_t ws_bytes, void *stream) {
    GPC_REQUIRE(chunks >= 0 && max_chunk >= 1 && max_chunk <= (1 << 24), GPC_EINVAL, "bad argument");
    cudaStream_t st = as_stream(stream);
    AttrWs L;
    GPC_REQUIRE(ws && ws_bytes >= chunk_var_layout(chunks, max_chunk, ws, &L), GPC_ENOSPC, "workspace too small");
    GPC_CUDA_CHECK(cudaMemsetAsync(L.status, 0, 4, st));
    if (chunks == 0) { GPC_CUDA_CHECK(cudaMemsetAsync(offsets, 0, 4, st)); return GPC_OK; }
    attr_encode_chunks_kernel<LohiLoad><<<cdiv(chunks, 4), 128, 0, st>>>(LohiLoad{lohi}, 0, max_chunk, chunks, L.cache, L.cap, cnt, L.status, starts);
    GPC_LAUNCH_CHECK();
    PtrLoad<u32> pl{(const u32 *)cnt};
    return device_exclusive_scan<u32, PtrLoad<u32>>(pl, chunks, offsets, L.scan_ws, st);
}
extern "C" int gpc_chunk_merge(const void *ws, int chunks, int max_chunk, const uint32_t *offsets, uint8_t *out, void *stream) {
    AttrWs L;
    chunk_var_layout(chunks, max_chunk, (void *)ws, &L);
    if (chunks <= 0) return GPC_OK;
    attr_merge_kernel<<<chunks, 256, 0, as_stream(stream)>>>(L.cache, L.cap, offsets, out);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// Decoder of the geometry streams: alphabets of 2 / 2 / 4 / 16 symbols, so a whole CDF row (Lp <= 32 entries) is ONE coalesced load,
// lane m holding entry m, and the symbol is a ballot.  The rows do not depend on the decoded symbols: the row of symbol i + 1 is
// requested before symbol i is decoded, which takes the load latency off the serial chain.
// RANGES = false: chunk w is rows [w * chunk_size, min((w + 1) * chunk_size, n)) (one stream).  RANGES = true: chunk w is rows
// [rows[w], rows[w + 1]) (many streams of their own chunk lengths side by side), clamped to [0, n) and to a non-negative byte
// length whatever the table holds.
template <bool RANGES>
__global__ void __launch_bounds__(128) chunk_decode_u16_kernel(const u16 *__restrict__ cdf, int Lp, const u8 *__restrict__ in,
                                                              const u32 *__restrict__ offsets, const u32 *__restrict__ rows, i64 n,
                                                              int chunk_size, int chunks, u8 *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (w >= chunks) return;
    i64 base;
    int len;
    u32 o0 = offsets[w], o1 = offsets[w + 1];
    if constexpr (RANGES) {
        base = min((i64)rows[w], n);
        len = (int)(min(max((i64)rows[w + 1], base), n) - base);
        if (len == 0) return;                                                       // the whole warp: w is warp-uniform
        o1 = max(o1, o0);
    } else {
        base = (i64)w * chunk_size;
        len = (int)min((i64)chunk_size, n - base);
    }
    const int max_symbol = Lp - 2;
    BitReader br;
    br.init(in + o0, (i64)(o1 - o0), lane);
    u32 low = 0u, high = 0xFFFFFFFFu;
    u32 value = br.get(32, lane);
    const u16 *row = cdf + base * Lp;
    // lane m: entry m of the row; entries above the top symbol read as 0x10000 (the top of the last symbol, by rule)
    auto load_row = [&](int i) -> u32 { return lane <= max_symbol ? (u32)row[(i64)i * Lp + lane] : 0x10000u; };
    u32 vnext = load_row(0);
    int my_sym = 0;
    for (int i = 0; i < len; ++i) {
        const u32 v = vnext;
        if (i + 1 < len) vnext = load_row(i + 1);
        const u64 span = (u64)high - (u64)low + 1ull;
        const u64 X = (((u64)value - (u64)low + 1ull) << ATTR_PRECISION) - 1ull;
        // symbol = largest m <= max_symbol with v(m) <= floor(X / span) (0 when there is none): what the binary search returns.
        // v <= floor(X / span)  <=>  v * span <= X: every lane tests its own entry with one multiplication, no division on the chain
        const u32 bal = __ballot_sync(0xFFFFFFFFu, lane <= max_symbol && (u64)v * span <= X);
        const int s = max(__popc(bal) - 1, 0);
        const u32 c_low = __shfl_sync(0xFFFFFFFFu, v, s);
        const u32 c_high = __shfl_sync(0xFFFFFFFFu, v, s + 1);                  // lane max_symbol + 1 holds 0x10000
        if (lane == (i & 31)) my_sym = s;
        high = (low - 1u) + (u32)((span * (u64)c_high) >> ATTR_PRECISION);
        low = low + (u32)((span * (u64)c_low) >> ATTR_PRECISION);
        for (;;) {
            const u32 diff = low ^ high;
            if (!(diff & 0x80000000u)) {
                const int sh = diff ? __clz(diff) : 32;
                const u32 bits = br.get(sh, lane);
                if (sh == 32) { low = 0u; high = 0xFFFFFFFFu; value = bits; }
                else { low <<= sh; high = (high << sh) | ((1u << sh) - 1u); value = (value << sh) | bits; }
            } else if (low >= 0x40000000u && high < 0xC0000000u) {
                low = (low << 1) & 0x7FFFFFFFu;
                high = (high << 1) | 0x80000001u;
                value -= 0x40000000u;
                value = (value << 1) | br.get(1, lane);
            } else {
                break;
            }
        }
        if ((i & 31) == 31 || i + 1 == len) {
            const int i0 = i & ~31;
            if (i0 + lane <= i) out[base + i0 + lane] = (u8)my_sym;
        }
    }
}

// offsets: device u32[chunks + 1], first byte of every chunk in `in` (the caller's prefix sums of the chunks' byte counts)
extern "C" int gpc_chunk_decode_u16(const uint16_t *cdf, const uint8_t *in, const uint32_t *offsets, int64_t n, int Lp, int chunk_size,
                                    uint8_t *sym, void *stream) {
    int rc = attr_check(n, Lp, chunk_size);
    if (rc) return rc;
    GPC_REQUIRE(Lp <= 32, GPC_EINVAL, "a CDF row must fit one warp load (Lp <= 32)");
    if (n == 0) return GPC_OK;
    const int chunks = (int)((n + chunk_size - 1) / chunk_size);
    chunk_decode_u16_kernel<false><<<cdiv(chunks, 4), 128, 0, as_stream(stream)>>>(cdf, Lp, in, offsets, nullptr, n, chunk_size, chunks,
                                                                                  sym);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

// many streams in one launch (the member scenes of a union level, each stream cut by its own chunk length): chunk w decodes rows
// [rows[w], rows[w + 1]) of cdf / sym from bytes [offsets[w], offsets[w + 1]) of `in`
extern "C" int gpc_chunk_decode_u16_ranges(const uint16_t *cdf, int Lp, const uint8_t *in, const uint32_t *offsets, const uint32_t *rows,
                                           int chunks, int64_t n, uint8_t *sym, void *stream) {
    int rc = attr_check(n, Lp, 1);
    if (rc) return rc;
    GPC_REQUIRE(Lp <= 32, GPC_EINVAL, "a CDF row must fit one warp load (Lp <= 32)");
    GPC_REQUIRE(chunks >= 0, GPC_EINVAL, "chunks out of range");
    if (n == 0 || chunks == 0) return GPC_OK;
    GPC_REQUIRE(cdf && in && offsets && rows && sym, GPC_EINVAL, "null pointer");
    chunk_decode_u16_kernel<true><<<cdiv(chunks, 4), 128, 0, as_stream(stream)>>>(cdf, Lp, in, offsets, rows, n, 0, chunks, sym);
    GPC_LAUNCH_CHECK();
    return GPC_OK;
}

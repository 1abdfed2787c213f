// The modeler's input CSV parsed on the GPU: header-less "dim_id,timestamp,quantity" lines (reference
// src/jobs/prophet_modeler.py:12-17,102-116), e.g.
//   91,2021-03-06 00:15:00,20153
// The files of one read are concatenated into one device byte buffer (every file ending in '\n'); three passes turn
// it into columns:
//   1. count: newlines per TILE-byte tile, one warp per tile with 16-byte loads;
//   2. (an exclusive scan of the tile counts, done by the caller)
//   3. index: the end offset (one past the '\n') of every row;
//   4. parse: series_id (from a per-file table of byte ranges), dim_id, ds (int64 ns), quantity and its valid mask.
// The row parser is one __host__ __device__ function so that the CPU tests exercise the very code the kernel runs.
// It accepts a strict grammar and refuses everything else; the caller then reads the input with pyarrow instead:
//   dim_id    -?[0-9]{1,10} within int32
//   timestamp YYYY-MM-DD[ T]HH:MM:SS(.[0-9]{1,9})?, year 1900..2199, a valid calendar date, hh < 24, mm < 60, ss < 60
//   quantity  -?[0-9]{1,10} within int32, or empty (null)
//   line end  "\n" or "\r\n"
#pragma once
#include "csv_kernel.cuh"

namespace pb200 {
namespace csvin {

constexpr int TILE = 4096;           // bytes per tile of the count and index passes (8 iterations of 32 lanes x 16 B)
constexpr int ROW_STAGE = 64;        // staged bytes per row in the parse pass; the longest accepted row is 55 B
constexpr int STRIP = 32 * ROW_STAGE;

__host__ __device__ __forceinline__ bool is_digit(unsigned char c) { return (unsigned)(c - '0') < 10u; }

// -?[0-9]{1,10} within int32, the whole of [p, e)
__host__ __device__ __forceinline__ bool parse_i32(const unsigned char* p, const unsigned char* e, int32_t& out) {
    const bool neg = p < e && *p == '-';
    if (neg) ++p;
    const long long n = e - p;
    if (n < 1 || n > 10) return false;
    long long v = 0;
    for (; p < e; ++p) {
        if (!is_digit(*p)) return false;
        v = v * 10 + (*p - '0');
    }
    if (neg) v = -v;
    if (v < -2147483648LL || v > 2147483647LL) return false;
    out = (int32_t)v;
    return true;
}

__host__ __device__ __forceinline__ int two_digits(const unsigned char* p) { return (p[0] - '0') * 10 + (p[1] - '0'); }

// YYYY-MM-DD[ T]HH:MM:SS(.f{1,9})?, the whole of [p, e), as ns since the epoch
__host__ __device__ __forceinline__ bool parse_timestamp(const unsigned char* p, const unsigned char* e, int64_t& ns) {
    const long long n = e - p;
    if (n < 19 || n == 20 || n > 29) return false;
    constexpr uint32_t DIGIT_AT = 0x6DB6Fu;          // positions 0-3, 5-6, 8-9, 11-12, 14-15, 17-18
#pragma unroll
    for (int i = 0; i < 19; ++i)
        if (((DIGIT_AT >> i) & 1u) && !is_digit(p[i])) return false;
    if (p[4] != '-' || p[7] != '-' || (p[10] != ' ' && p[10] != 'T') || p[13] != ':' || p[16] != ':') return false;
    const int Y = two_digits(p) * 100 + two_digits(p + 2), M = two_digits(p + 5), D = two_digits(p + 8);
    const int h = two_digits(p + 11), mi = two_digits(p + 14), s = two_digits(p + 17);
    if (Y < 1900 || Y > 2199 || M < 1 || M > 12 || h > 23 || mi > 59 || s > 59) return false;
    const bool leap = (Y % 4 == 0 && Y % 100 != 0) || Y % 400 == 0;
    const int mdays = M == 2 ? 28 + leap : (M == 4 || M == 6 || M == 9 || M == 11) ? 30 : 31;
    if (D < 1 || D > mdays) return false;
    int64_t frac = 0;
    if (n > 19) {
        if (p[19] != '.') return false;
        for (const unsigned char* q = p + 20; q < e; ++q) {
            if (!is_digit(*q)) return false;
            frac = frac * 10 + (*q - '0');
        }
        for (long long k = n - 20; k < 9; ++k) frac *= 10;
    }
    ns = ((csv::days_from_civil(Y, M, D) * 86400 + h * 3600 + mi * 60 + s) * 1000000000LL) + frac;
    return true;
}

// One line [p, e), e one past its '\n'.  Returns false (refused) for anything outside the grammar above.
__host__ __device__ __forceinline__ bool parse_row(const unsigned char* p, const unsigned char* e, int32_t& dim,
                                                   int64_t& ds, int32_t& qty, bool& qty_valid) {
    if (e <= p || e[-1] != '\n') return false;
    --e;
    if (e > p && e[-1] == '\r') --e;
    const unsigned char* c1 = p;
    while (c1 < e && *c1 != ',') ++c1;
    if (c1 == e) return false;
    const unsigned char* c2 = c1 + 1;
    while (c2 < e && *c2 != ',') ++c2;
    if (c2 == e) return false;
    if (!parse_i32(p, c1, dim) || !parse_timestamp(c1 + 1, c2, ds)) return false;
    qty = 0;
    qty_valid = c2 + 1 < e;
    return !qty_valid || parse_i32(c2 + 1, e, qty);
}

struct InArgs {
    const unsigned char* text;       // 16-byte aligned, readable up to n_bytes rounded up to 16
    long long n_bytes;
    long long* tile_count;           // count pass: out
    const long long* tile_off;       // index pass: exclusive scan of tile_count
    long long* row_end;              // index pass: out; parse pass: in
    long long n_rows;
    const long long* file_start;     // [n_files] ascending byte offset of each file's first byte
    const int32_t* file_sid;         // [n_files] series_id of each file
    int n_files;
    int32_t* sid;
    int32_t* dim;
    long long* ds;
    int32_t* qty;
    unsigned char* qty_valid;
    unsigned long long* refused;     // [0] rows refused, [1] index of the first (ULLONG_MAX when none)
};

// bit b set when byte b of the 16 at pos is '\n' and pos + b < n
__device__ __forceinline__ unsigned newline_bits(const InArgs& a, long long pos) {
    if (pos >= a.n_bytes) return 0u;
    const uint4 v = *reinterpret_cast<const uint4*>(a.text + pos);
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
    unsigned bits = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned m = __vcmpeq4(w[k], 0x0A0A0A0Au);
        bits |= (((m >> 7) & 1u) | ((m >> 14) & 2u) | ((m >> 21) & 4u) | ((m >> 28) & 8u)) << (4 * k);
    }
    if (a.n_bytes - pos < 16) bits &= (1u << (a.n_bytes - pos)) - 1u;
    return bits;
}

// one warp per tile
__global__ void __launch_bounds__(256) input_count_kernel(const InArgs a) {
    const int lane = threadIdx.x & 31;
    const long long tiles = (a.n_bytes + TILE - 1) / TILE, nwarp = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long t = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); t < tiles; t += nwarp) {
        int c = 0;
#pragma unroll
        for (int it = 0; it < TILE / 512; ++it) c += __popc(newline_bits(a, t * TILE + it * 512 + lane * 16));
#pragma unroll
        for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) a.tile_count[t] = c;
    }
}

__global__ void __launch_bounds__(256) input_index_kernel(const InArgs a) {
    const int lane = threadIdx.x & 31;
    const long long tiles = (a.n_bytes + TILE - 1) / TILE, nwarp = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long t = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); t < tiles; t += nwarp) {
        long long row = a.tile_off[t];
        for (int it = 0; it < TILE / 512; ++it) {
            const long long pos = t * TILE + it * 512 + lane * 16;
            unsigned bits = newline_bits(a, pos);
            const int c = __popc(bits);
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            long long r = row + incl - c;
            while (bits) {
                const int b = __ffs(bits) - 1;
                a.row_end[r++] = pos + b + 1;
                bits &= bits - 1u;
            }
            row += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
}

// One warp per 32 consecutive rows: the warp stages the rows' bytes in its shared-memory strip with coalesced 4-byte
// loads (the writer's strip pattern in reverse), then every lane parses its row from there.  A span longer than the
// strip (only possible with a row the grammar refuses anyway) is parsed straight from global memory.
__global__ void __launch_bounds__(128) input_parse_kernel(const InArgs a) {
    __shared__ uint32_t strips[4][STRIP / 4 + 1];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t* strip = strips[w];
    const long long nwarp = (long long)gridDim.x * 4;
    for (long long base = ((long long)blockIdx.x * 4 + w) * 32; base < a.n_rows; base += nwarp * 32) {
        const long long i = base + lane;
        const long long s0 = base ? a.row_end[base - 1] : 0;
        const long long last = (base + 32 <= a.n_rows ? base + 32 : a.n_rows) - 1;
        const long long a0 = s0 & ~3LL, span = a.row_end[last] - a0;
        const bool staged = span <= STRIP;
        if (staged) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(a.text + a0);
            for (int k = lane; k < (int)((span + 3) >> 2); k += 32) strip[k] = src[k];
        }
        __syncwarp();
        if (i < a.n_rows) {
            const long long si = i ? a.row_end[i - 1] : 0, ei = a.row_end[i];
            const unsigned char* p = staged ? reinterpret_cast<const unsigned char*>(strip) + (si - a0) : a.text + si;
            int32_t d = 0, q = 0;
            int64_t t = 0;
            bool qv = false;
            const bool ok = parse_row(p, p + (ei - si), d, t, q, qv);
            int lo = 0, hi = a.n_files - 1;                 // the file holding the row: last file_start <= si
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (a.file_start[mid] <= si) lo = mid;
                else hi = mid - 1;
            }
            a.sid[i] = a.file_sid[lo];
            a.dim[i] = d;
            a.ds[i] = t;
            a.qty[i] = q;
            a.qty_valid[i] = ok && qv;
            if (!ok) {
                atomicAdd(&a.refused[0], 1ULL);
                atomicMin(&a.refused[1], (unsigned long long)i);
            }
        }
        __syncwarp();
    }
}

}  // namespace csvin
}  // namespace pb200

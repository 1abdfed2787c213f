// Forecast CSV rows formatted on the GPU.  Replaces the row formatting of convert_forecasts + write_forecasts
// (reference src/jobs/prophet_scorer.py:131-150: a per-row Python date UDF, then Spark's CSV writer) for the standard
// six-column forecast frame:
//   "created_timestamp",series_id,dim_id,"forecast_date","forecast_timestamp",forecast_quantity
//   "2026-09-23T04:10:26+00:00",0,17,"2021-03-06","2021-03-06T00:15:00.000Z",20153
// (strings quoted, integers bare, '\n' line ends: byte for byte what the host path's pyarrow writer emits, which is the
// parity target of tests/test_gpu_jobs.py).  Byte / integer work, HBM bound: 20 B in, ~75 B out per row.  Two passes
// over the rows -- lengths, then (after an exclusive scan of the lengths) the bytes -- each one thread per row; the row
// formatter is one __host__ __device__ function so that the CPU tests exercise the very code the kernel runs.
// Supported range: 1970-01-01 <= timestamp < 10000-01-01 (the callers check and otherwise keep the host writer).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pb200 {
namespace csv {

constexpr int FIXED_BYTES = 46;      // quotes, commas, the two formatted dates and the line end of one row

__host__ __device__ __forceinline__ int int_len(int32_t v) {
    // decimal digits of v, plus one for the sign
    uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
    int n = v < 0 ? 2 : 1;
    while (u >= 10u) { u /= 10u; ++n; }
    return n;
}

__host__ __device__ __forceinline__ char* put_int(char* p, int32_t v) {
    uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
    if (v < 0) *p++ = '-';
    char tmp[10];
    int n = 0;
    do { tmp[n++] = (char)('0' + u % 10u); u /= 10u; } while (u);
    while (n) *p++ = tmp[--n];
    return p;
}

__host__ __device__ __forceinline__ char* put_2(char* p, int v) {
    p[0] = (char)('0' + v / 10);
    p[1] = (char)('0' + v % 10);
    return p + 2;
}

// civil date of a day count since 1970-01-01 (proleptic Gregorian; days >= 0 here)
__host__ __device__ __forceinline__ void civil_from_days(int64_t z, int& y, int& m, int& d) {
    z += 719468;
    const int64_t era = z / 146097;
    const unsigned doe = (unsigned)(z - era * 146097);
    const unsigned yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    const unsigned doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    const unsigned mp = (5 * doy + 2) / 153;
    d = (int)(doy - (153 * mp + 2) / 5 + 1);
    m = (int)(mp < 10 ? mp + 3 : mp - 9);
    y = (int)(yoe + era * 400) + (m <= 2 ? 1 : 0);
}

// day count since 1970-01-01 of a civil date (proleptic Gregorian; the inverse of civil_from_days, any year >= 1 here)
__host__ __device__ __forceinline__ int64_t days_from_civil(int y, int m, int d) {
    y -= m <= 2;
    const int era = y / 400;                         // y >= 0: no floor correction needed
    const unsigned yoe = (unsigned)(y - era * 400);
    const unsigned doy = (153u * (unsigned)(m > 2 ? m - 3 : m + 9) + 2u) / 5u + (unsigned)d - 1u;
    const unsigned doe = yoe * 365u + yoe / 4u - yoe / 100u + doy;
    return (int64_t)era * 146097 + (int64_t)doe - 719468;
}

__host__ __device__ __forceinline__ int row_len(int32_t sid, int32_t did, int32_t qty, int created_len) {
    return created_len + int_len(sid) + int_len(did) + int_len(qty) + FIXED_BYTES;
}

// writes one row at p (row_len bytes), returns the end
__host__ __device__ __forceinline__ char* put_row(char* p, int32_t sid, int32_t did, int64_t ds_ns, int32_t qty,
                                                  const char* created, int created_len) {
    *p++ = '"';
    for (int i = 0; i < created_len; ++i) *p++ = created[i];
    *p++ = '"';
    *p++ = ',';
    p = put_int(p, sid);
    *p++ = ',';
    p = put_int(p, did);
    *p++ = ',';
    const int64_t ms_total = ds_ns / 1000000;                  // (the host path casts to timestamp[ms]: truncation)
    const int64_t sec_total = ms_total / 1000;
    const int ms = (int)(ms_total - sec_total * 1000);
    const int64_t days = sec_total / 86400;
    const int sod = (int)(sec_total - days * 86400);
    int Y, M, D;
    civil_from_days(days, Y, M, D);
    char date[10];
    date[0] = (char)('0' + Y / 1000); date[1] = (char)('0' + Y / 100 % 10); date[2] = (char)('0' + Y / 10 % 10); date[3] = (char)('0' + Y % 10);
    date[4] = '-'; put_2(date + 5, M); date[7] = '-'; put_2(date + 8, D);
    *p++ = '"';
    for (int i = 0; i < 10; ++i) *p++ = date[i];
    *p++ = '"';
    *p++ = ',';
    *p++ = '"';
    for (int i = 0; i < 10; ++i) *p++ = date[i];
    *p++ = 'T';
    p = put_2(p, sod / 3600); *p++ = ':';
    p = put_2(p, sod / 60 % 60); *p++ = ':';
    p = put_2(p, sod % 60); *p++ = '.';
    p[0] = (char)('0' + ms / 100); p[1] = (char)('0' + ms / 10 % 10); p[2] = (char)('0' + ms % 10);
    p += 3;
    *p++ = 'Z';
    *p++ = '"';
    *p++ = ',';
    p = put_int(p, qty);
    *p++ = '\n';
    return p;
}

constexpr int MAX_CREATED = 64;

struct CsvArgs {
    const int32_t* sid;
    const int32_t* did;
    const long long* ds_ns;
    const int32_t* qty;
    long long n;
    int created_len;
    char created[MAX_CREATED];
    long long* row_len;          // lengths pass: out
    const long long* row_off;    // bytes pass: exclusive scan of the lengths
    unsigned char* out;
};

__global__ void __launch_bounds__(256) csv_lengths_kernel(const CsvArgs a) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x)
        a.row_len[i] = row_len(a.sid[i], a.did[i], a.qty[i], a.created_len);
}

// One warp per 32 consecutive rows: every lane formats its row into the warp's shared-memory strip at the row's offset
// within the strip, then the warp copies the strip out with coalesced stores (rows are ~75 B: lane-private byte stores
// straight to global would touch every 32-byte sector of the output two or three times).
constexpr int ROW_MAX = FIXED_BYTES + MAX_CREATED + 33;     // three 11-character integers
constexpr int STRIP = 32 * ROW_MAX;

__global__ void __launch_bounds__(128) csv_rows_kernel(const CsvArgs a) {
    __shared__ unsigned char strips[4][STRIP];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned char* strip = strips[w];
    const long long nwarp = (long long)gridDim.x * 4;
    for (long long base = ((long long)blockIdx.x * 4 + w) * 32; base < a.n; base += nwarp * 32) {
        const long long i = base + lane;
        const long long off0 = a.row_off[base];
        if (i < a.n)
            put_row((char*)strip + (a.row_off[i] - off0), a.sid[i], a.did[i], a.ds_ns[i], a.qty[i], a.created, a.created_len);
        __syncwarp();
        const long long last = (base + 32 <= a.n ? base + 32 : a.n) - 1;
        const int bytes = (int)(a.row_off[last] - off0) +
                          row_len(a.sid[last], a.did[last], a.qty[last], a.created_len);
        for (int b = lane; b < bytes; b += 32) a.out[off0 + b] = strip[b];
        __syncwarp();
    }
}

}  // namespace csv
}  // namespace pb200

// naf_export.cuh -- the decoded fields of a job, from the arena into memory the caller owns on the device, as tokens
// (include/nafgpu.h: nafgpu_job_export).  Records are numbered across the job: archive 0's n_lengths records first, then
// archive 1's; an archive that failed contributes none.
//
//   k_export_flat     one field of every archive, concatenated in job order.  A thread produces 16 output bytes with one
//                     aligned 16-byte store; their source is read with load16u (unaligned whenever an archive's byte count
//                     is not a multiple of 16).  The archive of a piece is found by binary search over the output bases.
//   k_export_rows     a [n_rows, L] tile of (record, start) windows of the sequence or quality, padded.  Pieces of 16 output
//                     bytes again: inside one row and inside the record they are one unaligned load, else byte by byte.
//   k_export_offsets  job-global record offsets: the archive's record offset + its residue base.
// All are HBM-bound byte moves: algorithmic bytes = bytes read + bytes written.
//
// The kernels are compiled as part of nafgpu_api.cu, the C layer that launches them (internal linkage: include this header from
// that one translation unit only).
#pragma once
#include "cuda_compat.h"
#include "naf_load.cuh"
#include <stdint.h>

namespace nk {

constexpr uint64_t NO_FIELD = ~0ull;
constexpr uint32_t EXPORT_THREADS = 256;

// FLAT: the bytes of one field of one archive (at arena + src_off) go to out[out_base, next span's out_base).  Only archives
// with at least one byte of the field are listed, so the out_base are strictly increasing.
struct ExpSpan {
    uint64_t out_base, src_off;
};

// ROWS / OFFSETS: one per archive with at least one record (rec_base strictly increasing).
struct ExpRec {
    uint64_t rec_base;            // job record of the archive's first record
    uint64_t res_base;            // job residue of its first residue
    uint64_t rec_offsets_off;     // its record offsets (n_lengths + 1 entries) in the arena
    uint64_t field_off[2];        // its sequence ASCII / quality in the arena, NO_FIELD if not decoded
    uint64_t _pad;
};

struct ExpTable {
    uint8_t b[256];               // out byte = b[decoded byte]; passed by value with the launch
};

__device__ __forceinline__ uint32_t map4(uint32_t w, const uint8_t* t) {
    return (uint32_t)t[w & 0xFF] | ((uint32_t)t[(w >> 8) & 0xFF] << 8) | ((uint32_t)t[(w >> 16) & 0xFF] << 16) | ((uint32_t)t[w >> 24] << 24);
}

__device__ __forceinline__ uint4 map16(uint4 v, const uint8_t* t) { return make_uint4(map4(v.x, t), map4(v.y, t), map4(v.z, t), map4(v.w, t)); }

// last k in [0, n) with key(k) <= x (key(0) <= x holds for every caller)
__device__ __forceinline__ uint32_t last_span(const ExpSpan* s, uint32_t n, uint64_t x) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (s[mid].out_base <= x) lo = mid; else hi = mid; }
    return lo;
}

__device__ __forceinline__ uint32_t last_rec(const ExpRec* r, uint32_t n, uint64_t x) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (r[mid].rec_base <= x) lo = mid; else hi = mid; }
    return lo;
}

__device__ __forceinline__ void load_table(uint8_t* tab, const ExpTable& table) {
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = table.b[i];
    __syncthreads();
}

// Output pieces: piece u covers out[16u - a, 16u - a + 16) clipped to [0, total), where a = out & 15, so that every whole
// piece is one aligned store.
__device__ __forceinline__ void store_piece(uint8_t* out, int64_t p0, uint64_t total, const uint32_t o[4]) {
    if (p0 >= 0 && (uint64_t)p0 + 16 <= total) { *(uint4*)(out + p0) = make_uint4(o[0], o[1], o[2], o[3]); return; }
    for (uint32_t k = 0; k < 16; k++) {
        const int64_t p = p0 + k;
        if (p >= 0 && (uint64_t)p < total) out[p] = (uint8_t)(o[k >> 2] >> (8 * (k & 3)));
    }
}

static __global__ void __launch_bounds__(EXPORT_THREADS) k_export_flat(const uint8_t* __restrict__ arena, const ExpSpan* __restrict__ spans,
                                                                 uint32_t n_spans, uint64_t total, ExpTable table, uint32_t identity,
                                                                 uint8_t* __restrict__ out) {
    __shared__ uint8_t tab[256];
    load_table(tab, table);
    const uint32_t a = (uint32_t)((uintptr_t)out & 15);
    const uint64_t pieces = (total + a + 15) / 16;
    for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < pieces; u += (uint64_t)gridDim.x * blockDim.x) {
        const int64_t p0 = (int64_t)(u * 16) - a;
        const uint64_t first = p0 < 0 ? 0 : (uint64_t)p0;
        uint32_t k = last_span(spans, n_spans, first);
        uint64_t next = k + 1 < n_spans ? spans[k + 1].out_base : total;
        if (p0 >= 0 && (uint64_t)p0 + 16 <= next) {                    // inside one archive: one load, one store
            const uint4 v = load16u(arena + spans[k].src_off + ((uint64_t)p0 - spans[k].out_base));
            *(uint4*)(out + p0) = identity ? v : map16(v, tab);
            continue;
        }
        uint32_t o[4] = {0, 0, 0, 0};                                   // an archive boundary, or the first / last piece
        const uint64_t end = (uint64_t)(p0 + 16) < total ? (uint64_t)(p0 + 16) : total;
        for (uint64_t p = first; p < end; p++) {
            while (p >= next) { k++; next = k + 1 < n_spans ? spans[k + 1].out_base : total; }
            const uint32_t b = tab[arena[spans[k].src_off + (p - spans[k].out_base)]];
            o[(p - p0) >> 2] |= b << (8 * ((p - p0) & 3));
        }
        store_piece(out, p0, total, o);
    }
}

// The bytes row i draws from: src[0, avail) (avail = 0: the row is all pad).
struct RowSrc {
    const uint8_t* src;
    uint64_t avail;
};

__device__ __forceinline__ RowSrc row_src(const uint8_t* arena, const ExpRec* recs, uint32_t n_recs, uint64_t n_records, uint32_t field,
                                          const int64_t* rows, uint64_t i) {
    RowSrc R = {nullptr, 0};
    const int64_t r = rows[2 * i], s = rows[2 * i + 1];
    if (r < 0 || (uint64_t)r >= n_records || s < 0) return R;
    const ExpRec& E = recs[last_rec(recs, n_recs, (uint64_t)r)];
    const uint64_t off = E.field_off[field];
    if (off == NO_FIELD) return R;
    const uint64_t* o = (const uint64_t*)(arena + E.rec_offsets_off);
    const uint64_t local = (uint64_t)r - E.rec_base, o0 = o[local], len = o[local + 1] - o0;
    if ((uint64_t)s >= len) return R;
    R.src = arena + off + o0 + (uint64_t)s;
    R.avail = len - (uint64_t)s;
    return R;
}

static __global__ void __launch_bounds__(EXPORT_THREADS) k_export_rows(const uint8_t* __restrict__ arena, const ExpRec* __restrict__ recs,
                                                                 uint32_t n_recs, uint64_t n_records, uint32_t field,
                                                                 const int64_t* __restrict__ rows, uint64_t row_length, uint64_t total,
                                                                 ExpTable table, uint32_t identity, uint32_t pad, uint8_t* __restrict__ out) {
    __shared__ uint8_t tab[256];
    load_table(tab, table);
    const uint32_t a = (uint32_t)((uintptr_t)out & 15);
    const uint64_t pieces = (total + a + 15) / 16;
    const uint32_t pad4 = pad * 0x01010101u;
    for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < pieces; u += (uint64_t)gridDim.x * blockDim.x) {
        const int64_t p0 = (int64_t)(u * 16) - a;
        const uint64_t first = p0 < 0 ? 0 : (uint64_t)p0;
        uint64_t row = first / row_length, col = first - row * row_length;
        RowSrc R = row_src(arena, recs, n_recs, n_records, field, rows, row);
        if (p0 >= 0 && (uint64_t)p0 + 16 <= total && col + 16 <= row_length) {      // inside one row
            if (col + 16 <= R.avail) {
                const uint4 v = load16u(R.src + col);
                *(uint4*)(out + p0) = identity ? v : map16(v, tab);
                continue;
            }
            if (col >= R.avail) { *(uint4*)(out + p0) = make_uint4(pad4, pad4, pad4, pad4); continue; }
        }
        uint32_t o[4] = {0, 0, 0, 0};                                   // the record's end, a row boundary, the first / last piece
        const uint64_t end = (uint64_t)(p0 + 16) < total ? (uint64_t)(p0 + 16) : total;
        for (uint64_t p = first; p < end; p++) {
            if (col == row_length) { row++; col = 0; R = row_src(arena, recs, n_recs, n_records, field, rows, row); }
            const uint32_t b = col < R.avail ? (uint32_t)tab[R.src[col]] : pad;
            o[(p - p0) >> 2] |= b << (8 * ((p - p0) & 3));
            col++;
        }
        store_piece(out, p0, total, o);
    }
}

static __global__ void __launch_bounds__(EXPORT_THREADS) k_export_offsets(const uint8_t* __restrict__ arena, const ExpRec* __restrict__ recs,
                                                                    uint32_t n_recs, uint64_t n_records, uint64_t total_residues,
                                                                    int64_t* __restrict__ out) {
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n_records; j += (uint64_t)gridDim.x * blockDim.x) {
        if (j == n_records) { out[j] = (int64_t)total_residues; continue; }
        const ExpRec& E = recs[last_rec(recs, n_recs, j)];
        const uint64_t* o = (const uint64_t*)(arena + E.rec_offsets_off);
        out[j] = (int64_t)(E.res_base + o[j - E.rec_base]);
    }
}

// enough CTAs to fill the `sms` multiprocessors several times over; the kernels loop over whatever is left
static uint32_t export_ctas(uint64_t items, uint32_t sms) {
    const uint64_t ctas = (items + EXPORT_THREADS - 1) / EXPORT_THREADS;
    return (uint32_t)(ctas < sms * 16u ? (ctas ? ctas : 1) : sms * 16u);
}

// out[0, total) <- table[field bytes of spans[0, n_spans)] (16-byte aligned stores; out may have any alignment).
static void launch_export_flat(const uint8_t* arena, const ExpSpan* spans, uint32_t n_spans, uint64_t total, const ExpTable& table,
                        bool identity, uint8_t* out, uint32_t sms, cudaStream_t st) {
    if (!total) return;
    NAF_LAUNCH(k_export_flat, export_ctas(total / 16 + 2, sms), EXPORT_THREADS, 0, st, arena, spans, n_spans, total, table, identity ? 1u : 0u, out);
}

// out[i * L + c] <- table[field byte `start + c` of record `record`] for (record, start) = rows[2i], rows[2i + 1]; pad past the
// record's end, and the whole row for a record out of [0, n_records), a start outside [0, length) or a field not decoded.
static void launch_export_rows(const uint8_t* arena, const ExpRec* recs, uint32_t n_recs, uint64_t n_records, uint32_t field,
                        const int64_t* rows, uint64_t n_rows, uint64_t row_length, const ExpTable& table, bool identity,
                        uint8_t pad, uint8_t* out, uint32_t sms, cudaStream_t st) {
    const uint64_t total = n_rows * row_length;
    if (!total) return;
    NAF_LAUNCH(k_export_rows, export_ctas(total / 16 + 2, sms), EXPORT_THREADS, 0, st, arena, recs, n_recs, n_records, field, rows,
               row_length, total, table, identity ? 1u : 0u, (uint32_t)pad, out);
}

// out[j] <- job-global exclusive offset of record j, j in [0, n_records]; out[n_records] = total_residues.
static void launch_export_offsets(const uint8_t* arena, const ExpRec* recs, uint32_t n_recs, uint64_t n_records, uint64_t total_residues,
                           int64_t* out, uint32_t sms, cudaStream_t st) {
    NAF_LAUNCH(k_export_offsets, export_ctas(n_records + 1, sms), EXPORT_THREADS, 0, st, arena, recs, n_recs, n_records, total_residues, out);
}

}  // namespace nk

// naf_text.cu -- FASTA / FASTQ formatter kernels (sm_100a); see naf_text.cuh for the text being produced.
//
//   k_text_layout   one CTA per archive: text size of every record, exclusive scan -> offs[n+1], total -> sizes[a]
//   k_text_write    one CTA per 8 KB of OUTPUT text: finds the records that intersect its chunk (binary search over
//                   offs + a shared-memory table of the record starts inside the chunk), then every thread produces 16
//                   output bytes with one 16-byte store.  Interior stretches of sequence / quality are moved with two
//                   aligned 16-byte loads and a funnel shift; headers, line ends and record boundaries go byte by byte.
// Both are HBM-bound byte shuffling: algorithmic bytes = text out + the ASCII / quality / ids / comments read once.
#include "naf_text.cuh"

#include "naf_load.cuh"
#include "zstd_core.cuh"

namespace nk {

#define FULL 0xFFFFFFFFu

// Exclusive scan of one u64 per thread over the CTA; *total gets the sum.  All threads must call.
__device__ __forceinline__ uint64_t block_excl_scan64(uint64_t v, uint64_t* total) {
    __shared__ uint64_t ws[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    uint64_t inc = v;
    for (int d = 1; d < 32; d <<= 1) { const uint64_t t = __shfl_up_sync(FULL, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint64_t x = lane < nwarps ? ws[lane] : 0;
        uint64_t xi = x;
        for (int d = 1; d < 32; d <<= 1) { const uint64_t t = __shfl_up_sync(FULL, xi, d); if (lane >= d) xi += t; }
        ws[lane] = xi - x;
        if (lane == 31) ws[32] = xi;
    }
    __syncthreads();
    const uint64_t r = inc - v + ws[warp];
    *total = ws[32];
    __syncthreads();
    return r;
}

// What record r contributes, as the reference's iterator would yield it (include/nafgpu.h, nafgpu_result): fields past
// the end of their stream are absent (empty here).
struct RecView {
    uint64_t id0, idlen, com0, comlen, seq0, L;
    uint64_t hdr;
};

struct ArchView {
    const uint8_t *ids, *com, *seq, *qual;
    const uint64_t *id_offs, *com_offs, *rec_offs;
    uint64_t n, n_ids, n_com, n_len, W, cap;
    uint32_t fastq, sep;
};

__device__ __forceinline__ ArchView arch_view(const uint8_t* arena, const NafDev& A, const TextDev& T) {
    const NafCounts* C = (const NafCounts*)(arena + A.counts_off);
    ArchView V;
    V.ids = arena + A.ids_off; V.com = arena + A.com_off; V.seq = arena + A.ascii_off; V.qual = arena + A.qual_off;
    V.id_offs = (const uint64_t*)(arena + A.id_offsets_off);
    V.com_offs = (const uint64_t*)(arena + A.com_offsets_off);
    V.rec_offs = (const uint64_t*)(arena + A.rec_offsets_off);
    V.n = A.n_records;
    V.n_ids = (A.has & HAS_IDS) ? (C->n_ids < V.n ? C->n_ids : V.n) : 0;
    V.n_com = (A.has & HAS_COMMENTS) ? (C->n_comments < V.n ? C->n_comments : V.n) : 0;
    V.n_len = (A.has & HAS_SEQUENCE) ? C->n_lengths : 0;
    V.W = T.line_length; V.fastq = T.fastq; V.sep = T.sep;
    // lengths that overrun their streams flag the archive (E_LENGTHS); the formatter must still stay inside the buffers
    V.cap = A.seq_residues;
    if (T.fastq && A.qual_size < V.cap) V.cap = A.qual_size;
    return V;
}

__device__ __forceinline__ RecView rec_view(const ArchView& V, uint64_t r) {
    RecView R;
    R.id0 = 0; R.idlen = 0; R.com0 = 0; R.comlen = 0; R.seq0 = 0; R.L = 0;
    if (r < V.n_ids) { R.id0 = V.id_offs[r]; R.idlen = V.id_offs[r + 1] - R.id0 - 1; }
    if (r < V.n_com) { R.com0 = V.com_offs[r]; R.comlen = V.com_offs[r + 1] - R.com0 - 1; }
    if (r < V.n_len) {
        R.seq0 = V.rec_offs[r]; R.L = V.rec_offs[r + 1] - R.seq0;
        if (R.seq0 > V.cap) { R.seq0 = V.cap; R.L = 0; } else if (R.L > V.cap - R.seq0) R.L = V.cap - R.seq0;
    }
    R.hdr = 1 + R.idlen + (R.comlen ? 1 + R.comlen : 0) + 1;
    return R;
}

// bytes of text of the record (a 64-bit division: only where it is needed)
__device__ __forceinline__ uint64_t rec_total(const ArchView& V, const RecView& R) {
    if (V.fastq) return R.hdr + 2 * R.L + 4;
    return R.hdr + (V.W ? R.L + (R.L + V.W - 1) / V.W : R.L + 1);
}

__global__ void __launch_bounds__(1024) k_text_layout(const uint8_t* arena, const NafDev* archives, uint8_t* text,
                                                       const TextDev* texts, uint32_t* status) {
    const NafDev& A = archives[blockIdx.x];
    const TextDev& T = texts[blockIdx.x];
    const ArchView V = arch_view(arena, A, T);
    uint64_t* offs = (uint64_t*)(text + T.offs_off);
    uint64_t carry = 0;
    for (uint64_t base = 0; base < V.n; base += 1024) {
        const uint64_t r = base + threadIdx.x;
        const uint64_t sz = r < V.n ? rec_total(V, rec_view(V, r)) : 0;
        uint64_t tot;
        const uint64_t ex = block_excl_scan64(sz, &tot);
        if (r < V.n) offs[r] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) {
        offs[V.n] = carry;
        if (carry > T.cap) { atomicOr(status, zc::E_INTERNAL); carry = 0; }      // (the host's bound is exact arithmetic: cannot happen)
        ((uint64_t*)text)[blockIdx.x] = carry;
    }
}

__global__ void __launch_bounds__(TEXT_THREADS) k_text_write(const uint8_t* arena, const NafDev* archives, uint8_t* text,
                                                              const TextDev* texts) {
    __shared__ uint32_t starts[TEXT_CHUNK / 2 + 2];     // starts[t] = text offset of record r0 + t, relative to the chunk (t >= 1)
    __shared__ uint64_t s_r0;
    const NafDev& A = archives[blockIdx.y];
    const TextDev& T = texts[blockIdx.y];
    const uint64_t total = ((const uint64_t*)text)[blockIdx.y];
    const uint64_t p0 = (uint64_t)blockIdx.x * TEXT_CHUNK;
    if (p0 >= total) return;
    const uint64_t p1 = p0 + TEXT_CHUNK < total ? p0 + TEXT_CHUNK : total;
    const ArchView V = arch_view(arena, A, T);
    const uint64_t* offs = (const uint64_t*)(text + T.offs_off);
    const uint32_t tid = threadIdx.x;
    // the record that holds the first byte of the chunk: last r with offs[r] <= p0
    if (tid == 0) {
        uint64_t lo = 0, hi = V.n;                       // offs[0] = 0 <= p0 < total = offs[n]
        while (hi - lo > 1) { const uint64_t mid = lo + (hi - lo) / 2; if (offs[mid] <= p0) lo = mid; else hi = mid; }
        s_r0 = lo;
    }
    __syncthreads();
    const uint64_t r0 = s_r0;
    // starts of the following records, as long as they lie inside the chunk (a record has at least 2 bytes of text)
    uint32_t n_tab = 1;
    for (uint32_t b = 1; b <= TEXT_CHUNK / 2; b += TEXT_THREADS) {
        const uint32_t t = b + tid;
        const uint64_t r = r0 + t;
        uint32_t v = TEXT_CHUNK;
        if (t <= TEXT_CHUNK / 2 && r < V.n) { const uint64_t o = offs[r]; if (o < p1) v = (uint32_t)(o - p0); }
        if (t <= TEXT_CHUNK / 2 + 1) starts[t] = v;
        const uint32_t inside = (uint32_t)__syncthreads_count(v < TEXT_CHUNK);
        n_tab += inside;                                                // entries [1, n_tab) start inside the chunk (sorted)
        if (inside < TEXT_THREADS) break;
    }
    for (uint32_t piece = tid; piece < TEXT_CHUNK / 16; piece += TEXT_THREADS) {
        const uint64_t p = p0 + (uint64_t)piece * 16;
        if (p >= p1) return;
        // my record: last t with starts[t] <= piece * 16 (t = 0: the record that began before the chunk)
        uint32_t lo = 0, hi = n_tab;
        while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (starts[mid] <= piece * 16) lo = mid; else hi = mid; }
        uint64_t r = r0 + lo;
        RecView R = rec_view(V, r);
        uint64_t q = lo == 0 ? p - offs[r0] : (uint64_t)(piece * 16 - starts[lo]);
        // position inside the sequence for the FASTA body
        uint64_t idx = 0, col = 0;
        if (!V.fastq && q > R.hdr) {
            const uint64_t qp = q - R.hdr;
            if (V.W == 0) idx = qp;
            else if (((qp | V.W) >> 31) == 0) {                                // the usual case: 32-bit division
                const uint32_t line = (uint32_t)qp / ((uint32_t)V.W + 1u);
                col = (uint32_t)qp - line * ((uint32_t)V.W + 1u); idx = (uint64_t)line * V.W + col;
            } else { const uint64_t line = qp / (V.W + 1); col = qp - line * (V.W + 1); idx = line * V.W + col; }
        }
        const uint32_t nout = p1 - p >= 16 ? 16u : (uint32_t)(p1 - p);
        uint8_t* dst = text + T.text_off + p;
        // fast paths: 16 bytes from the inside of one line of sequence (or quality)
        if (nout == 16 && q >= R.hdr) {
            const uint8_t* src = nullptr;
            if (!V.fastq) {
                if (idx + 16 <= R.L && (V.W == 0 || col + 16 <= V.W)) src = V.seq + R.seq0 + idx;
                else if (V.W >= 16 && V.W - col < 16 && idx + 15 <= R.L) {
                    // exactly one line end inside the 16 bytes (a line and its '\n' are at least 17 bytes): 15 residues, with
                    // '\n' inserted after the first j of them
                    const uint32_t j = (uint32_t)(V.W - col);                   // 0..15
                    const uint4 a = load16u(V.seq + R.seq0 + idx);
                    const uint32_t A[4] = {a.x, a.y, a.z, a.w};
                    const uint32_t B[4] = {a.x << 8, __funnelshift_l(a.x, a.y, 8), __funnelshift_l(a.y, a.z, 8), __funnelshift_l(a.z, a.w, 8)};   // bytes moved up by one
                    uint32_t o4[4];
#pragma unroll
                    for (uint32_t i = 0; i < 4; i++) {
                        if (4 * i + 3 < j) o4[i] = A[i];
                        else if (4 * i > j) o4[i] = B[i];
                        else {
                            const uint32_t sh = 8 * (j - 4 * i), low = (1u << sh) - 1u;      // bytes below j from A, byte j = '\n', above from B
                            o4[i] = (A[i] & low) | (0x0Au << sh) | (B[i] & ~((low << 8) | 0xFFu));
                        }
                    }
                    *(uint4*)dst = make_uint4(o4[0], o4[1], o4[2], o4[3]);
                    continue;
                }
            } else {
                const uint64_t qp = q - R.hdr;
                if (qp + 16 <= R.L) src = V.seq + R.seq0 + qp;
                else if (qp >= R.L + 3 && qp + 16 <= 2 * R.L + 3) src = V.qual + R.seq0 + (qp - R.L - 3);
            }
            if (src) { *(uint4*)dst = load16u(src); continue; }
        }
        uint32_t o[4] = {0, 0, 0, 0};
        uint64_t rtotal = rec_total(V, R);
        for (uint32_t k = 0; k < nout; k++) {
            if (q == rtotal) { r++; R = rec_view(V, r); rtotal = rec_total(V, R); q = 0; idx = 0; col = 0; }
            uint32_t b;
            if (q < R.hdr) {
                if (q == 0) b = V.fastq ? '@' : '>';
                else if (q - 1 < R.idlen) b = V.ids[R.id0 + q - 1];
                else if (q == R.hdr - 1) b = '\n';
                else if (q == 1 + R.idlen) b = V.sep;                         // only reached when there is a comment
                else b = V.com[R.com0 + (q - 2 - R.idlen)];
            } else if (!V.fastq) {
                if (idx == R.L || (V.W && col == V.W)) { b = '\n'; col = 0; }
                else { b = V.seq[R.seq0 + idx]; idx++; col++; }
            } else {
                const uint64_t qp = q - R.hdr;
                if (qp < R.L) b = V.seq[R.seq0 + qp];
                else if (qp == R.L || qp == R.L + 2) b = '\n';
                else if (qp == R.L + 1) b = '+';
                else if (qp < 2 * R.L + 3) b = V.qual[R.seq0 + (qp - R.L - 3)];
                else b = '\n';
            }
            o[k >> 2] |= b << (8 * (k & 3));
            q++;
        }
        if (nout == 16) *(uint4*)dst = make_uint4(o[0], o[1], o[2], o[3]);
        else for (uint32_t k = 0; k < nout; k++) dst[k] = (uint8_t)(o[k >> 2] >> (8 * (k & 3)));
    }
}

int launch_text_stage(uint8_t* arena, const NafDev* archives, uint8_t* text, const TextDev* texts, uint32_t n_archives,
                      uint64_t max_cap, uint32_t* status, cudaStream_t st) {
    if (n_archives == 0) return 0;
    NAF_LAUNCH(k_text_layout, n_archives, 1024, 0, st, arena, archives, text, texts, status);
    const uint32_t chunks = (uint32_t)((max_cap + TEXT_CHUNK - 1) / TEXT_CHUNK);
    if (chunks == 0) return 1;
    NAF_LAUNCH(k_text_write, dim3(chunks, n_archives), TEXT_THREADS, 0, st, arena, archives, text, texts);
    return 2;
}

}  // namespace nk

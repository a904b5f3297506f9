// naf_kernels.cu -- NAF layer kernels (sm_100a).  Reference semantics restated here:
//   CStringReader::next   reader.rs:20-31    -> k_naf_scan task 0/1 (NUL positions -> string offsets)
//   LengthReader::next    reader.rs:46-68    -> k_naf_scan task 2   (u32 words, 0xFFFFFFFF continues a length)
//   MaskReader::next      reader.rs:196-231  -> k_naf_scan task 3   (byte RLE, 0xFF continues a run)
//   Decoder::mask_sequence mod.rs:402-441    -> toggle bitmap (+ per-chunk parity) + k_mask_fix (the record-tail quirk) + k_unpack
//   SequenceReader::read_nucleotide / decode reader.rs:121-172 -> k_unpack (4-bit -> IUPAC, low nibble first)
//   String::from_utf8     reader.rs:108-109  -> k_ascii_check + k_utf8_validate
#include "naf_kernels.cuh"

#include <algorithm>

#include "zstd_core.cuh"

namespace nk {

#define FULL 0xFFFFFFFFu

// An error of one archive: its own status word (archives of a batch fail independently) and the job-wide OR.
__device__ __forceinline__ void flag_archive(NafCounts* counts, uint32_t* status, uint32_t bits) {
    atomicOr((unsigned long long*)&counts->status, (unsigned long long)bits);
    atomicOr(status, bits);
}

struct CS { uint32_t c; uint64_t s; };

// Exclusive scan of (count, sum) over a 1024-thread CTA; *total gets the CTA totals.  All threads must call.
__device__ __forceinline__ CS block_excl_scan(uint32_t c, uint64_t s, CS* total) {
    __shared__ uint32_t wc[33];
    __shared__ uint64_t ws[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    uint32_t ic = c;
    uint64_t is = s;
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t tc = __shfl_up_sync(FULL, ic, d);
        uint64_t ts = __shfl_up_sync(FULL, is, d);
        if (lane >= d) { ic += tc; is += ts; }
    }
    if (lane == 31) { wc[warp] = ic; ws[warp] = is; }
    __syncthreads();
    if (warp == 0) {
        uint32_t xc = lane < nwarps ? wc[lane] : 0, oc = xc;
        uint64_t xs = lane < nwarps ? ws[lane] : 0, os = xs;
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t tc = __shfl_up_sync(FULL, xc, d);
            uint64_t ts = __shfl_up_sync(FULL, xs, d);
            if (lane >= d) { xc += tc; xs += ts; }
        }
        wc[lane] = xc - oc; ws[lane] = xs - os;
        if (lane == 31) { wc[32] = xc; ws[32] = xs; }
    }
    __syncthreads();
    CS r;
    r.c = ic - c + wc[warp];
    r.s = is - s + ws[warp];
    total->c = wc[32];
    total->s = ws[32];
    __syncthreads();
    return r;
}

// Flips the mask state from residue `pos` on; the parity of the toggles of every CHUNK_RESIDUES chunk is kept beside the
// bitmap (two toggles on the same bit cancel in both), so k_unpack gets its carry-in without a separate parity pass.
__device__ __forceinline__ void toggle_bit(uint32_t* bits, uint32_t* chunk_par, uint64_t pos) {
    atomicXor(&bits[pos >> 5], 1u << (pos & 31));
    atomicXor(&chunk_par[pos / CHUNK_RESIDUES], 1u);
}

// --------------------------------------------------------------------------------------------------------------
// k_naf_scan: the four streaming scans of the NAF layer -- ids and comments (k-th NUL -> string offsets), lengths (u32 words,
// 0xFFFFFFFF continues a length -> record offsets), mask (byte RLE, 0xFF continues a run -> run bounds + toggle bitmap).
// Every section is cut into NAF_SLICE-byte slices, one CTA of 1024 threads each: grid (4 tasks x n_slices, n_archives).
// What a slice needs from everything before it is a pair (count of terminators, sum): with more than one slice, k_naf_agg
// computes every slice's pair first and a slice adds up the pairs of the slices before it (a 10^6-read FASTQ archive has
// 17 MB of ids: one CTA streaming them took 3.5 ms); with one slice per section there is nothing to add and no extra launch.
struct SliceView { const uint8_t* src; uint64_t size, begin, end; bool present, last; };

__device__ __forceinline__ SliceView slice_view(const uint8_t* arena, const NafDev& A, int task, uint32_t slice) {
    SliceView V;
    V.present = task == 0 ? (A.has & HAS_IDS) != 0 : task == 1 ? (A.has & HAS_COMMENTS) != 0 : task == 2 ? (A.has & HAS_LENGTHS) != 0
                                                                                                          : (A.has & HAS_MASK) && (A.has & HAS_SEQUENCE);
    V.src = arena + (task == 0 ? A.ids_off : task == 1 ? A.com_off : task == 2 ? A.len_off : A.mask_off);
    V.size = !V.present ? 0 : task == 0 ? A.ids_size : task == 1 ? A.com_size : task == 2 ? (A.len_size & ~3ull) : A.mask_size;
    V.begin = (uint64_t)slice * NAF_SLICE;
    V.end = V.begin + NAF_SLICE < V.size ? V.begin + NAF_SLICE : V.size;
    V.last = V.begin < V.size ? V.end == V.size : (slice == 0);          // an empty section is "finished" by its slice 0
    return V;
}

// (terminators, sum) of 16 bytes of a section: ids / comments: NULs; lengths: words != FFFFFFFF and the sum of all words;
// mask: bytes != FF and the sum of all bytes.  `nvalid` bytes of v count.
__device__ __forceinline__ void pair_of16(int task, const uint4& v, uint32_t nvalid, uint32_t& c, uint64_t& s) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    if (task == 2) { for (uint32_t j = 0; j < nvalid / 4; j++) { c += (w[j] != FULL); s += w[j]; } return; }
    const uint32_t term = task == 3 ? 0xFFu : 0u;
    for (uint32_t j = 0; j < nvalid; j++) {
        const uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFF;
        c += task == 3 ? (b != term) : (b == term);
        if (task == 3) s += b;
    }
}

__global__ void __launch_bounds__(1024) k_naf_agg(const uint8_t* arena, const NafDev* archives, CS* agg, uint32_t n_slices) {
    const NafDev& A = archives[blockIdx.y];
    const int task = blockIdx.x / n_slices;
    const uint32_t slice = blockIdx.x % n_slices;
    const SliceView V = slice_view(arena, A, task, slice);
    uint32_t c = 0;
    uint64_t s = 0;
    for (uint64_t p0 = V.begin + (uint64_t)threadIdx.x * 16; p0 < V.end; p0 += 1024 * 16) {
        const uint4 v = *(const uint4*)(V.src + p0);
        pair_of16(task, v, V.end - p0 >= 16 ? 16u : (uint32_t)(V.end - p0), c, s);
    }
    CS tot;
    block_excl_scan(c, s, &tot);
    if (threadIdx.x == 0) agg[((size_t)blockIdx.y * 4 + task) * n_slices + slice] = tot;
}

__global__ void __launch_bounds__(1024) k_naf_scan(uint8_t* arena, const NafDev* archives, uint32_t* status, const CS* agg, uint32_t n_slices) {
    const NafDev& A = archives[blockIdx.y];
    const int task = blockIdx.x / n_slices;
    const uint32_t slice = blockIdx.x % n_slices;
    const int tid = threadIdx.x;
    NafCounts* counts = (NafCounts*)(arena + A.counts_off);
    const SliceView V = slice_view(arena, A, task, slice);
    if (V.begin >= V.size && slice != 0) return;                          // (uniform) nothing of the section in this slice
    // what the slices before this one hold
    uint64_t carry_c = 0, carry_s = 0;
    if (slice) {
        const CS* ag = agg + ((size_t)blockIdx.y * 4 + task) * n_slices;
        uint32_t c = 0;
        uint64_t s = 0;
        for (uint32_t j = tid; j < slice; j += 1024) { c += ag[j].c; s += ag[j].s; }
        CS tot;
        block_excl_scan(c, s, &tot);
        carry_c = tot.c; carry_s = tot.s;
    }
    if (task <= 1) {
        // ---- ids / comments: string k ends at the k-th NUL; offsets[k+1] = position after it -----------------
        if (!V.present) { if (tid == 0) { if (task == 0) counts->n_ids = 0; else counts->n_comments = 0; } return; }
        uint64_t* offs = (uint64_t*)(arena + (task == 0 ? A.id_offsets_off : A.com_offsets_off));
        if (tid == 0 && slice == 0) offs[0] = 0;
        uint64_t carry = carry_c;
        uint32_t hi = 0;
        for (uint64_t base = V.begin; base < V.end; base += 1024 * 16) {
            uint64_t p0 = base + (uint64_t)tid * 16;
            uint4 v = make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
            if (p0 < V.end) v = *(const uint4*)(V.src + p0);
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
            uint32_t nvalid = p0 >= V.end ? 0 : (V.end - p0 >= 16 ? 16 : (uint32_t)(V.end - p0));
            uint32_t c = 0;
            for (uint32_t j = 0; j < nvalid; j++) {
                uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFF;
                c += (b == 0);
                hi |= b;
            }
            CS tot;
            CS ex = block_excl_scan(c, 0, &tot);
            uint64_t k = carry + ex.c;
            if (c) {
                for (uint32_t j = 0; j < nvalid; j++) {
                    uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFF;
                    if (b == 0) { k++; if (k <= A.n_records) offs[k] = p0 + j + 1; }
                }
            }
            carry += tot.c;
        }
        if (__any_sync(FULL, hi & 0x80)) { if ((tid & 31) == 0) atomicOr((unsigned long long*)&counts->nonascii, 1ull << task); }
        if (tid == 0 && V.last) {
            if (task == 0) counts->n_ids = carry; else counts->n_comments = carry;
            if (carry < A.n_records && V.size > 0 && V.src[V.size - 1] != 0) flag_archive(counts, status, zc::E_NUL);
        }
    } else if (task == 2) {
        // ---- lengths: rec_offsets[k+1] = sum of all words up to and including the k-th terminating word -----
        uint64_t* rec = (uint64_t*)(arena + A.rec_offsets_off);
        uint64_t* lens = (uint64_t*)(arena + A.lengths_off);
        if (tid == 0 && slice == 0) rec[0] = 0;
        const uint64_t w_begin = V.begin / 4, w_end = V.end / 4;
        for (uint64_t base = w_begin; base < w_end; base += 1024 * 4) {
            uint64_t i0 = base + (uint64_t)tid * 4;
            uint4 v = make_uint4(FULL, FULL, FULL, FULL);
            if (i0 < w_end) v = *(const uint4*)(V.src + i0 * 4);
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
            uint32_t nvalid = i0 >= w_end ? 0 : (w_end - i0 >= 4 ? 4 : (uint32_t)(w_end - i0));
            uint32_t c = 0;
            uint64_t s = 0;
            for (uint32_t j = 0; j < nvalid; j++) { c += (w[j] != FULL); s += w[j]; }
            CS tot;
            CS ex = block_excl_scan(c, s, &tot);
            uint64_t k = carry_c + ex.c, S = carry_s + ex.s;
            for (uint32_t j = 0; j < nvalid; j++) {
                S += w[j];
                if (w[j] != FULL) { k++; if (k <= A.n_records) rec[k] = S; }
            }
            carry_c += tot.c; carry_s += tot.s;
        }
        if (n_slices > 1) {                                  // other slices are still writing rec[]: k_naf_lengths finishes the job
            if (tid == 0 && V.last) counts->n_lengths = carry_c;
            return;
        }
        __syncthreads();
        uint64_t n_len = carry_c < A.n_records ? carry_c : A.n_records;
        uint64_t total = rec[n_len];
        if (tid == 0) {
            counts->n_lengths = n_len;
            counts->total_residues = total;
            counts->first_bad_record = NO_RECORD;
            if ((A.has & HAS_SEQUENCE) && total > A.seq_residues) flag_archive(counts, status, zc::E_LENGTHS);
            if ((A.has & HAS_QUALITY) && total > A.qual_size) flag_archive(counts, status, zc::E_LENGTHS);
        }
        for (uint64_t k = tid; k < n_len; k += blockDim.x) lens[k] = rec[k + 1] - rec[k];
    } else {
        // ---- mask: run k ends at the inclusive byte sum at the k-th byte != 0xFF; toggle the bitmap there --------
        if (!V.present) { if (tid == 0 && slice == 0) { counts->n_mask_runs = 0; counts->mask_sum = 0; } return; }
        uint64_t* bounds = (uint64_t*)(arena + A.mask_bounds_off);
        uint32_t* bits = (uint32_t*)(arena + A.mask_bits_off);
        uint32_t* cpar = (uint32_t*)(arena + A.chunk_par_off);
        for (uint64_t base = V.begin; base < V.end; base += 1024 * 16) {
            uint64_t p0 = base + (uint64_t)tid * 16;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (p0 < V.end) v = *(const uint4*)(V.src + p0);
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
            uint32_t nvalid = p0 >= V.end ? 0 : (V.end - p0 >= 16 ? 16 : (uint32_t)(V.end - p0));
            uint32_t c = 0;
            uint64_t s = 0;
            for (uint32_t j = 0; j < nvalid; j++) {
                uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFF;
                c += (b != 0xFF); s += b;
            }
            CS tot;
            CS ex = block_excl_scan(c, s, &tot);
            uint64_t k = carry_c + ex.c, S = carry_s + ex.s;
            for (uint32_t j = 0; j < nvalid; j++) {
                uint32_t b = (w[j >> 2] >> (8 * (j & 3))) & 0xFF;
                S += b;
                if (b != 0xFF) { bounds[k++] = S; if (S <= A.seq_residues) toggle_bit(bits, cpar, S); }
            }
            carry_c += tot.c; carry_s += tot.s;
        }
        if (tid == 0 && V.last) {
            if (V.size > 0 && V.src[V.size - 1] == 0xFF) {        // trailing 0xFF bytes at EOF still form a unit (reader.rs:206-209)
                bounds[carry_c++] = carry_s;
                if (carry_s <= A.seq_residues) toggle_bit(bits, cpar, carry_s);
            }
            counts->n_mask_runs = carry_c;
            counts->mask_sum = carry_s;
        }
    }
}

// k_naf_lengths: after a SLICED lengths scan (every slice has written its part of rec_offsets): the record count, the total,
// the checks, and lengths[k] = rec_offsets[k + 1] - rec_offsets[k].  Thread per record.
__global__ void __launch_bounds__(256) k_naf_lengths(uint8_t* arena, const NafDev* archives, uint32_t* status) {
    const NafDev& A = archives[blockIdx.y];
    NafCounts* counts = (NafCounts*)(arena + A.counts_off);
    const uint64_t* rec = (const uint64_t*)(arena + A.rec_offsets_off);
    uint64_t* lens = (uint64_t*)(arena + A.lengths_off);
    const uint64_t raw = (A.has & HAS_LENGTHS) ? counts->n_lengths : 0;   // (written by the last slice; clamping it below is idempotent)
    const uint64_t n_len = raw < A.n_records ? raw : A.n_records;
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_len) lens[r] = rec[r + 1] - rec[r];
    if (r == 0) {
        const uint64_t total = rec[n_len];
        counts->n_lengths = n_len;
        counts->total_residues = total;
        counts->first_bad_record = NO_RECORD;
        if ((A.has & HAS_SEQUENCE) && total > A.seq_residues) flag_archive(counts, status, zc::E_LENGTHS);
        if ((A.has & HAS_QUALITY) && total > A.qual_size) flag_archive(counts, status, zc::E_LENGTHS);
    }
}

// --------------------------------------------------------------------------------------------------------------
// k_mask_fix: the reference quirk (decoder/mod.rs:413-416): a Masked unit that reaches the end of a record is
// carried over WITHOUT lower-casing the record's tail.  Residue i in masked run [a,b) is lower-cased iff
// b < end_of_record(i).  Per record: if its last residue lies in a masked run, un-toggle [max(a,start), end).
__global__ void __launch_bounds__(256) k_mask_fix(uint8_t* arena, const NafDev* archives, uint32_t* status) {
    const NafDev& A = archives[blockIdx.y];
    if (!(A.has & HAS_MASK) || !(A.has & HAS_SEQUENCE)) return;
    NafCounts* counts = (NafCounts*)(arena + A.counts_off);
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= counts->n_lengths) return;
    const uint64_t* rec = (const uint64_t*)(arena + A.rec_offsets_off);
    const uint64_t* bounds = (const uint64_t*)(arena + A.mask_bounds_off);
    uint32_t* bits = (uint32_t*)(arena + A.mask_bits_off);
    const uint64_t S = rec[r], E = rec[r + 1];
    if (E == S || E > A.seq_residues) return;
    const uint64_t pos = E - 1, n_runs = counts->n_mask_runs;
    uint64_t lo = 0, hi = n_runs;                       // first k with bounds[k] > pos
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (bounds[mid] > pos) hi = mid; else lo = mid + 1;
    }
    if (lo == n_runs) { flag_archive(counts, status, zc::E_MASK); return; }      // "failed to get mask unit" (mod.rs:429-434)
    if (lo & 1) {
        uint64_t a = lo ? bounds[lo - 1] : 0;
        uint32_t* cpar = (uint32_t*)(arena + A.chunk_par_off);
        toggle_bit(bits, cpar, a > S ? a : S);
        toggle_bit(bits, cpar, E);
    }
}

// --------------------------------------------------------------------------------------------------------------
// k_unpack: fused 4-bit -> IUPAC unpack + soft mask.  Thread = 16 packed bytes = 32 residues = one toggle word.
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t s) {
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(s));
    return d;
#else
    return __byte_perm(a, b, s);
#endif
}

// 4 nibbles (16 bits, residue order) -> 4 ASCII bytes.  LUT "-TGKCYSBAWRDMHVN" (reader.rs:151-172) as four words.
__device__ __forceinline__ uint32_t iupac4(uint32_t x16, uint32_t l0) {
    const uint32_t sel = x16 & 0x7777u;
    const uint32_t lo = prmt(l0, 0x42535943u, sel);                 // entries 0..7  : - T/U G K C Y S B
    const uint32_t hi = prmt(0x44525741u, 0x4E56484Du, sel);        // entries 8..15 : A W R D M H V N
    const uint32_t m = prmt(0x80808080u, 0u, x16 & 0x8888u);        // 0xFF where nibble >= 8, else 0x80 (ASCII < 0x80)
    return (lo & ~m) | (hi & m);
}

__device__ __forceinline__ uint32_t spread4_x20(uint32_t q) {        // 4 mask bits -> 0x20 in the matching bytes
    return ((q * 0x00204081u) & 0x01010101u) << 5;
}

__global__ void __launch_bounds__(UNPACK_T) k_unpack(uint8_t* arena, const NafDev* archives) {
    const NafDev& A = archives[blockIdx.y];
    if (!(A.has & HAS_SEQUENCE) || A.seq_type > 1 || blockIdx.x >= A.n_chunks) return;
    __shared__ uint32_t wp[32], wp2[32];
    __shared__ uint32_t wball, cball;
    const NafCounts* counts = (const NafCounts*)(arena + A.counts_off);
    // lengths that sum to more than the section holds are an error of the archive (E_LENGTHS): never unpack past the section
    const uint64_t total = counts->total_residues < A.seq_residues ? counts->total_residues : A.seq_residues;
    const uint64_t wi = (uint64_t)blockIdx.x * CHUNK_WORDS + UNPACK_W * threadIdx.x;   // UNPACK_W adjacent toggle words per thread
    const uint64_t r0 = wi * 32;
    uint32_t mask[UNPACK_W];
#pragma unroll
    for (uint32_t k = 0; k < UNPACK_W; k++) mask[k] = 0;
    if (A.has & HAS_MASK) {                                           // uniform per CTA
        const uint32_t* bits = (const uint32_t*)(arena + A.mask_bits_off);
        const uint64_t n_words = (A.seq_residues + 32) / 32;
        uint32_t par = 0;                                             // parity of the toggles of the words before word k of this thread
#pragma unroll
        for (uint32_t k = 0; k < UNPACK_W; k++) {
            const uint32_t w = wi + k < n_words ? bits[wi + k] : 0;
            uint32_t m = w;
            m ^= m << 1; m ^= m << 2; m ^= m << 4; m ^= m << 8; m ^= m << 16;   // in-word prefix XOR
            mask[k] = par ? ~m : m;
            par ^= __popc(w) & 1;
        }
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        uint32_t b = __ballot_sync(FULL, par);
        if (lane == 0) wp[warp] = __popc(b) & 1;
        __syncthreads();
        if (warp == 0) { uint32_t bb = __ballot_sync(FULL, lane < (int)(UNPACK_T / 32) ? wp[lane] : 0u); if (lane == 0) wball = bb; }
        __syncthreads();
        // carry into this chunk = parity of all toggles in the chunks before it
        const uint32_t* cpar = (const uint32_t*)(arena + A.chunk_par_off);
        uint32_t cp = 0;
        for (uint32_t c = threadIdx.x; c < blockIdx.x; c += blockDim.x) cp ^= cpar[c];
        const uint32_t cb = __ballot_sync(FULL, cp & 1);
        if (lane == 0) wp2[warp] = __popc(cb) & 1;
        __syncthreads();
        if (warp == 0) { uint32_t bb = __ballot_sync(FULL, lane < (int)(UNPACK_T / 32) ? wp2[lane] : 0u); if (lane == 0) cball = bb; }
        __syncthreads();
        const uint32_t carry = (__popc(cball) & 1) ^ (__popc(wball & ((1u << warp) - 1u)) & 1) ^ (__popc(b & ((1u << lane) - 1u)) & 1);
        if (carry) {
#pragma unroll
            for (uint32_t k = 0; k < UNPACK_W; k++) mask[k] = ~mask[k];
        }
    }
    if (r0 >= total) return;
    const uint32_t l0 = A.seq_type == 1 ? 0x4B47552Du : 0x4B47542Du;       // RNA: 'U' at code 1
    const uint4* src = (const uint4*)(arena + A.seq_off + r0 / 2);
    uint4 pk[UNPACK_W];
#pragma unroll
    for (uint32_t k = 0; k < UNPACK_W; k++) {                              // every load is issued before the first is used
        pk[k] = make_uint4(0, 0, 0, 0);
        if (r0 + 32 * k < total) pk[k] = src[k];
    }
    uint4* dst = (uint4*)(arena + A.ascii_off + r0);
#pragma unroll
    for (uint32_t k = 0; k < UNPACK_W; k++) {
        if (r0 + 32 * k >= total) break;
        const uint32_t x[4] = {pk[k].x, pk[k].y, pk[k].z, pk[k].w};
        uint32_t o[8];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            o[2 * j] = iupac4(x[j] & 0xFFFFu, l0) | spread4_x20((mask[k] >> (8 * j)) & 0xFu);
            o[2 * j + 1] = iupac4(x[j] >> 16, l0) | spread4_x20((mask[k] >> (8 * j + 4)) & 0xFu);
        }
        dst[2 * k] = make_uint4(o[0], o[1], o[2], o[3]);
        dst[2 * k + 1] = make_uint4(o[4], o[5], o[6], o[7]);
    }
}

// k_text_mask: protein / text archives with a mask section: mask_sequence lower-cases A-Z in place (no type check
// in the reference).  Thread = 32 bytes.
__global__ void __launch_bounds__(CHUNK_WORDS) k_text_mask(uint8_t* arena, const NafDev* archives) {
    const NafDev& A = archives[blockIdx.y];
    if (!(A.has & HAS_SEQUENCE) || !(A.has & HAS_MASK) || A.seq_type <= 1 || blockIdx.x >= A.n_chunks) return;
    const NafCounts* counts = (const NafCounts*)(arena + A.counts_off);
    const uint64_t total = counts->total_residues < A.seq_residues ? counts->total_residues : A.seq_residues;
    const uint64_t wi = (uint64_t)blockIdx.x * CHUNK_WORDS + threadIdx.x;
    const uint32_t* bits = (const uint32_t*)(arena + A.mask_bits_off);
    const uint32_t* par = (const uint32_t*)(arena + A.chunk_par_off);
    const uint64_t n_words = (A.seq_residues + 32) / 32;
    if (wi >= n_words) return;
    // carry: chunk carry ^ parity of the words of this chunk before wi (serial: this path is rare)
    uint32_t carry = 0;
    for (uint32_t c = 0; c < blockIdx.x; c++) carry ^= par[c] & 1;
    for (uint64_t j = (uint64_t)blockIdx.x * CHUNK_WORDS; j < wi; j++) carry ^= __popc(bits[j]) & 1;
    uint32_t m = bits[wi];
    m ^= m << 1; m ^= m << 2; m ^= m << 4; m ^= m << 8; m ^= m << 16;
    if (carry) m = ~m;
    uint8_t* s = arena + A.seq_off;
    for (int j = 0; j < 32; j++) {
        uint64_t i = wi * 32 + j;
        if (i >= total) break;
        uint8_t c = s[i];
        if (((m >> j) & 1) && c >= 'A' && c <= 'Z') s[i] = c | 0x20;
    }
}

// --------------------------------------------------------------------------------------------------------------
// UTF-8: String::from_utf8 per record (reader.rs:108-109).  k_ascii_check flags fields that contain bytes >= 0x80;
// only those run the per-record DFA.
__global__ void __launch_bounds__(256) k_ascii_check(uint8_t* arena, const NafDev* archives) {
    const NafDev& A = archives[blockIdx.y];
    const int field = blockIdx.z;                                  // 0: text sequence, 1: quality
    const uint8_t* src;
    uint64_t size;
    if (field == 0) { if (!(A.has & HAS_SEQUENCE) || A.seq_type <= 1) return; src = arena + A.seq_off; size = A.seq_size; }
    else { if (!(A.has & HAS_QUALITY)) return; src = arena + A.qual_off; size = A.qual_size; }
    NafCounts* counts = (NafCounts*)(arena + A.counts_off);
    uint32_t acc = 0;
    const uint64_t n16 = (size + 15) / 16;                         // section buffers are padded to 16 B with readable bytes
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) {
        uint4 v = *(const uint4*)(src + i * 16);
        if (i * 16 + 16 > size) {                                   // mask the bytes past the end
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
            for (int j = 0; j < 16; j++) if (i * 16 + j < size) acc |= (w[j >> 2] >> (8 * (j & 3))) & 0xFF;
        } else acc |= v.x | v.y | v.z | v.w;
    }
    if (__any_sync(FULL, acc & 0x80808080u)) { if ((threadIdx.x & 31) == 0) atomicOr((unsigned long long*)&counts->nonascii, 1ull << (2 + field)); }
}

__device__ __forceinline__ bool utf8_ok(const uint8_t* s, uint64_t n) {
    uint64_t i = 0;
    while (i < n) {
        uint32_t b = s[i];
        if (b < 0x80) { i++; continue; }
        uint32_t need, cp;
        if (b >= 0xC2 && b <= 0xDF) { need = 1; cp = b & 0x1F; }
        else if (b >= 0xE0 && b <= 0xEF) { need = 2; cp = b & 0x0F; }
        else if (b >= 0xF0 && b <= 0xF4) { need = 3; cp = b & 0x07; }
        else return false;
        if (n - i <= need) return false;
        for (uint32_t k = 1; k <= need; k++) {
            uint32_t c = s[i + k];
            if ((c & 0xC0) != 0x80) return false;
            cp = (cp << 6) | (c & 0x3F);
        }
        if (need == 2 && (cp < 0x800 || (cp >= 0xD800 && cp <= 0xDFFF))) return false;
        if (need == 3 && (cp < 0x10000 || cp > 0x10FFFF)) return false;
        i += need + 1;
    }
    return true;
}

// grid (ceil(max_records/256), n_archives, 4 fields: ids, comments, text sequence, quality)
__global__ void __launch_bounds__(256) k_utf8_validate(uint8_t* arena, const NafDev* archives, uint32_t* status) {
    const NafDev& A = archives[blockIdx.y];
    const int field = blockIdx.z;
    NafCounts* counts = (NafCounts*)(arena + A.counts_off);
    if (!((counts->nonascii >> field) & 1)) return;
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint8_t* s;
    uint64_t b, e;
    if (field <= 1) {
        uint64_t n = field == 0 ? counts->n_ids : counts->n_comments;
        if (n > A.n_records) n = A.n_records;
        if (r >= n) return;
        const uint64_t* offs = (const uint64_t*)(arena + (field == 0 ? A.id_offsets_off : A.com_offsets_off));
        s = arena + (field == 0 ? A.ids_off : A.com_off);
        b = offs[r]; e = offs[r + 1] - 1;
    } else {
        if (r >= counts->n_lengths) return;
        const uint64_t* rec = (const uint64_t*)(arena + A.rec_offsets_off);
        s = arena + (field == 2 ? A.seq_off : A.qual_off);
        b = rec[r]; e = rec[r + 1];
        if (e > (field == 2 ? A.seq_size : A.qual_size)) return;
    }
    if (!utf8_ok(s + b, e - b)) {
        flag_archive(counts, status, zc::E_UTF8);
        atomicMin((unsigned long long*)&counts->first_bad_record, (unsigned long long)r);
    }
}

// --------------------------------------------------------------------------------------------------------------
int launch_naf_stage(uint8_t* arena, const NafDev* archives, uint32_t n_archives, uint64_t max_records, uint64_t max_scan_bytes, void* scan_agg,
                     uint32_t max_chunks, uint64_t max_text_bytes, bool any_mask, bool any_text_mask, uint32_t* status, uint32_t sms,
                     cudaStream_t st, StageEvents* ev) {
    StageEvents none;
    if (!ev) ev = &none;
    int launches = 0;
    if (n_archives == 0) { for (int i = 0; i < NAF_STAGES; i++) ev->mark(); return 0; }
    const uint32_t n_slices = (uint32_t)std::max<uint64_t>(1, (max_scan_bytes + NAF_SLICE - 1) / NAF_SLICE);
    uint32_t rec_grid = (uint32_t)((max_records + 255) / 256);
    if (n_slices > 1) { NAF_LAUNCH(k_naf_agg, dim3(4 * n_slices, n_archives), 1024, 0, st, arena, archives, (CS*)scan_agg, n_slices); launches++; }
    NAF_LAUNCH(k_naf_scan, dim3(4 * n_slices, n_archives), 1024, 0, st, arena, archives, status, (const CS*)scan_agg, n_slices); launches++;
    if (n_slices > 1) { NAF_LAUNCH(k_naf_lengths, dim3(rec_grid ? rec_grid : 1, n_archives), 256, 0, st, arena, archives, status); launches++; }
    ev->mark();
    if (max_chunks > 0 && any_mask) {
        if (rec_grid) { NAF_LAUNCH(k_mask_fix, dim3(rec_grid, n_archives), 256, 0, st, arena, archives, status); launches++; }
        ev->mark();
        ev->mark();
    } else { ev->mark(); ev->mark(); }
    if (max_chunks > 0) {
        NAF_LAUNCH(k_unpack, dim3(max_chunks, n_archives), UNPACK_T, 0, st, arena, archives); launches++;
        if (any_text_mask) { NAF_LAUNCH(k_text_mask, dim3(max_chunks, n_archives), CHUNK_WORDS, 0, st, arena, archives); launches++; }
    }
    ev->mark();
    if (max_text_bytes > 0) {
        uint32_t g = (uint32_t)((max_text_bytes / 16 + 255) / 256);
        if (g > sms * 8) g = sms * 8;
        if (g == 0) g = 1;
        NAF_LAUNCH(k_ascii_check, dim3(g, n_archives, 2), 256, 0, st, arena, archives); launches++;
    }
    if (rec_grid) { NAF_LAUNCH(k_utf8_validate, dim3(rec_grid, n_archives, 4), 256, 0, st, arena, archives, status); launches++; }
    ev->mark();
    return launches;
}

}  // namespace nk

// zstd_kernels.cu -- hand-written sm_100a kernels that replace libzstd's ZSTD_decompressStream on the
// nafcodec decode path (the reference reaches it through zstd::stream::read::Decoder,
// nafcodec/src/decoder/mod.rs:32,221-223).  No library decompressor, no CPU fallback.
//
// One job = any number of frames (NAF sections, possibly of many archives).  Two branches run on two streams and join
// before the LZ stage (a third stream carries a kernel of either branch beside its sibling where a job has both kinds of work):
//   FSE branch      k_build_tables<0>        per block: parse the FSE table descriptions, build LL/OF/ML decode tables (whole warp)
//                   k_decode_sequences       per block: tANS decode of (ll, ml, offset): three-lane producer / consumer warp, symbolic repeat offsets
//                   k_decode_sequences_tiny  blocks of at most 32 sequences, one warp each (jobs with thousands of them: FASTQ flushed per record)
//                   k_frame_scan (+ k_fs_reduce / k_fs_prefix / k_fs_apply for frames of 10^4+ blocks)
//                                            per frame: block output offsets (prefix sum) + repeat-offset carry across blocks
//   Huffman branch  k_build_tables<1>        per block: Huffman tree description -> 256 weights, once per tree
//                   k_huf_scout              per big block: the exact start and output offset of every range of its four streams
//                   k_huf_decode_block       per big block: intra-stream parallel decode of its four streams into the literal staging buffer
//                   k_huf_decode_big         the same per stream, four CTAs of a block as a cluster (DSMEM): a job of a few blocks
//                   k_huf_decode_small       short streams
//   LZ stage        k_lz_literals (+ _tiny)  per block: raw / RLE blocks, literal runs -> their output positions
//                   k_lz_small               a job of at most 2048 matches: the whole match stage in one CTA
//                   k_lz_index, k_lz_first   per match: position index; round 1 of the dependency-resolving match execution (+ redirect through copies)
//                   k_lz_resolve             persistent cooperative kernel: further rounds over a worklist, one grid barrier per round
//                   k_lz_flow                chains of a few dozen generations: matches in order by ticket, each waiting for the ones it needs
//                   k_lz_finish, k_lz_finish2  endless chains (text-like sections): byte-level pointer jumping inside 64 KB chunks on all SMs,
//                                            then across chunks over the chunks' roots
//                   k_frame_checksum         frames that carry a content checksum (XXH64)
#include "frame_walk.h"          // (first: the emulator's cuda_compat.h defines __noinline__, which <string> uses)
#include "zstd_kernels.cuh"

#include <algorithm>

namespace zk {

using namespace zf;
using zc::BackBits;
using zc::SeqCell;

__device__ __forceinline__ void flag_error(const JobDev& J, uint32_t frame, uint32_t bits) {
    atomicOr(J.status, bits);
    atomicOr(&J.frame_bad[frame], bits);              // per frame (= per section of one archive): archives of a batch fail independently
}

// --------------------------------------------------------------------------------------------------------------
// Backward bit reader over a shared-memory image of the bitstream (32-bit words; >= 16 zero bytes below bit 0).
// 64-bit register window, refilled 32 bits at a time; read(k) for k <= 32.
struct SmemBits {
    const uint32_t* sw;
    uint64_t w;          // stream bits [32*qi, 32*qi + 64)
    int qi, rr;          // rr = x - 32*qi, position of the next unread bit inside the window (kept in [32, 64] before a read)
    int x_zero;          // smem bit position of stream bit 0
    __device__ __forceinline__ void init(const uint32_t* words, int x, int xz) {
        sw = words; x_zero = xz;
        qi = (x >> 5) - 1;
        rr = x - (qi << 5);
        w = ((uint64_t)sw[qi + 1] << 32) | sw[qi];
    }
    __device__ __forceinline__ uint32_t read(int k) {
        if (rr < k) { w = (w << 32) | sw[--qi]; rr += 32; }
        rr -= k;
        return k ? (uint32_t)(w >> rr) & (k >= 32 ? 0xFFFFFFFFu : ((1u << k) - 1u)) : 0u;
    }
    __device__ __forceinline__ int remaining() const { return (qi << 5) + rr - x_zero; }   // unread payload bits (negative: over-read)
};

// ---- shared-memory access by explicit shared-space address ---------------------------------------------------------
// The hot loops below address shared memory through 32-bit shared-space addresses and ld.shared PTX: with generic
// pointers nvcc re-derives the shared window base inside the loops (S2R SR_CgaCtaId + LEA per access, seen in SASS).
#if defined(__CUDA_ARCH__)
typedef uint32_t saddr_t;
__device__ __forceinline__ saddr_t to_saddr(const void* p) { return (saddr_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds32(saddr_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint2 lds64(saddr_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds16(saddr_t a) { uint16_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds8(saddr_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts8(saddr_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(a), "r"(v)); }
__device__ __forceinline__ void sts32(saddr_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v)); }
#else
typedef uintptr_t saddr_t;
static inline saddr_t to_saddr(const void* p) { return (saddr_t)p; }
static inline uint32_t lds32(saddr_t a) { return *(const uint32_t*)a; }
static inline uint2 lds64(saddr_t a) { return *(const uint2*)a; }
static inline uint32_t lds16(saddr_t a) { return *(const uint16_t*)a; }
static inline uint32_t lds8(saddr_t a) { return *(const uint8_t*)a; }
static inline void sts8(saddr_t a, uint32_t v) { *(uint8_t*)a = (uint8_t)v; }
static inline void sts32(saddr_t a, uint32_t v) { *(uint32_t*)a = v; }
#endif

// bits [o, o + k) of a shared-memory image of a bitstream (32-bit words), k <= 32: no reader state
__device__ __forceinline__ uint32_t smem_bits(const uint32_t* sw, int o, uint32_t k) {         // bits [o, o + k) of the image, k <= 32
    const uint32_t lo = sw[o >> 5], hi = sw[(o >> 5) + 1];
    const uint32_t v = __funnelshift_r(lo, hi, (uint32_t)o);          // (shift taken modulo 32)
    return k >= 32 ? v : (v & ((1u << k) - 1u));
}

// FSE decode table by a whole warp (RFC 8878 4.1.1; the serial restatement is zc::fse_build in zstd_core.cuh).
//   A  low-probability symbols (-1) take the top cells in symbol order; counts and cumulative counts of the others
//   B  the serial "spread" visits positions (j * step) & mask, j = 0, 1, ..., skipping those >= high: the t-th placement
//      is the t-th position of that sequence below `high` (ballot ranks), and it belongs to the symbol whose cumulative
//      count range holds t (binary search)
//   C  cell i continues its symbol's state counter: start count + the number of lower cells with the same symbol
//      (__match_any_sync ranks inside 32 consecutive cells, running per-symbol counters across them)
template <class Emit>
__device__ __forceinline__ bool fse_build_warp(const int16_t* norm, int max_symbol, int al, uint8_t* cell_sym, uint16_t* cnt, uint16_t* cum,
                                               int lane, Emit emit) {
    const int size = 1 << al, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
    const uint32_t lt = (1u << lane) - 1u;
    int n_low = 0, reg_total = 0;
    for (int s0 = 0; s0 <= max_symbol; s0 += 32) {
        const int s = s0 + lane;
        const int nv = s <= max_symbol ? (int)norm[s] : 0;
        const bool low = nv == -1;
        const uint32_t lb = __ballot_sync(0xFFFFFFFFu, low);
        if (low) cell_sym[size - 1 - (n_low + __popc(lb & lt))] = (uint8_t)s;
        const int c = nv > 0 ? nv : 0;
        int inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
        if (s <= max_symbol) { cnt[s] = (uint16_t)(low ? 1 : c); cum[s] = (uint16_t)(reg_total + inc - c); }
        reg_total += __shfl_sync(0xFFFFFFFFu, inc, 31);
        n_low += __popc(lb);
    }
    if (lane == 0) cum[max_symbol + 1] = (uint16_t)reg_total;
    __syncwarp();
    if (reg_total + n_low != size) return false;           // (the serial spread would not come back to position 0)
    const int high = size - n_low;
    int placed = 0;
    for (int j0 = 0; j0 < size; j0 += 32) {
        const int p = ((j0 + lane) * step) & mask;
        const bool valid = p < high;
        const uint32_t vb = __ballot_sync(0xFFFFFFFFu, valid);
        if (valid) {
            const int t = placed + __popc(vb & lt);
            int lo = 0, hi = max_symbol + 1;                 // cum[lo] <= t < cum[hi]
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if ((int)cum[mid] <= t) lo = mid; else hi = mid; }
            cell_sym[p] = (uint8_t)lo;
        }
        placed += __popc(vb);
    }
    __syncwarp();
    for (int i0 = 0; i0 < size; i0 += 32) {
        const int i = i0 + lane;
        const int s = cell_sym[i];
        const uint32_t same = __match_any_sync(0xFFFFFFFFu, s);
        const int r = __popc(same & lt);
        const uint32_t nx = (uint32_t)cnt[s] + (uint32_t)r;
        __syncwarp();
        if (r == 0) cnt[s] = (uint16_t)(cnt[s] + __popc(same));
        __syncwarp();
        const int nb = al - zc::highbit32(nx);
        emit(i, s, nb, (int)((nx << nb) - (uint32_t)size));
    }
    return true;
}

// zc::fse_read_ncount over the staged (word-aligned, zero-padded) copy of the table descriptions, for the one lane that parses
// them: fields cut out of the image with a funnel shift, the two cases of a field as selects (the restatement's byte reader and
// branches cost ~240 cycles per symbol on a lone lane: 15 us for the three tables of a block, on the critical path of a single
// archive).  `norm` must be zeroed by the caller.  Returns bytes consumed, or 0 on error, like the restatement.
__device__ __forceinline__ uint32_t fse_read_ncount_staged(const uint32_t* dw, uint32_t byte0, uint32_t src_len, int max_symbol, int max_al,
                                                           int16_t* norm, int* al_out) {
    uint32_t pos = byte0 * 8u;
    const uint32_t limit = pos + src_len * 8u;
    auto peek = [&](uint32_t k) { const uint32_t i = pos >> 5; return __funnelshift_r(dw[i], dw[i + 1], pos) & ((1u << k) - 1u); };
    const int al = (int)peek(4) + 5;
    pos += 4;
    if (al > max_al) return 0;
    int rem = 1 << al, sym = 0;
    while (rem > 0 && sym <= max_symbol) {
        const uint32_t bits = 32u - (uint32_t)__clz(rem + 1);
        uint32_t v = peek(bits);
        const uint32_t low = (1u << (bits - 1)) - 1u, thr = (1u << bits) - 1u - (uint32_t)(rem + 1);
        const bool small = (v & low) < thr;
        pos += bits - (small ? 1u : 0u);
        v = small ? (v & low) : (v > low ? v - thr : v);
        const int pr = (int)v - 1;
        rem -= pr < 0 ? -pr : pr;
        norm[sym++] = (int16_t)pr;
        if (pr == 0) {
            for (;;) {
                const uint32_t r = peek(2);
                pos += 2;
                sym += (int)r;                      // r extra zero-probability symbols
                if (r != 3) break;
                if (pos > limit) return 0;
            }
            if (sym > max_symbol + 1) return 0;
        }
        if (pos > limit) return 0;
    }
    if (rem != 0 || sym > max_symbol + 1) return 0;
    *al_out = al;
    return ((pos + 7u) >> 3) - byte0;
}

// k_build_tables: one warp per block (+ one extra CTA that builds the three predefined tables into slots 0..2).
// part 0: FSE tables (32 threads, grid n_blocks + 1); part 1: Huffman weights (32 threads, grid n_blocks).  Two launches so
// that the Huffman branch and the FSE branch of the zstd stage can run on different streams.
// part 0 runs three warps: the three table descriptions are parsed one after the other by one lane (each starts where the one
// before ends), then every warp builds one table (a single small archive waits for this kernel: 21 -> see profiles).
template <int PART>
__global__ void __launch_bounds__(PART == 0 ? 96 : 32) k_build_tables(JobDev J) {
    if (PART == 1) {
        // warp 1: the block's Huffman tree description -> 256 weights, decoded ONCE per tree (streams and treeless
        // blocks that reuse the tree read the weights back and build their decode table in parallel).
        if (blockIdx.x >= J.n_blocks) return;
        const BlockDesc& B = J.blocks[blockIdx.x];
        if (B.btype != BT_COMPRESSED || B.lit_type != LT_HUF) return;
        // The weight decode is a serial chain (FSE with two interleaved states): everything it touches sits in shared memory
        // (tree description, packed table cells, weights) and it reads bits through a register window; what is not a
        // chain (staging, zeroing, validation sums, the write-back) is done by the whole warp.  (A thread-local version
        // -- zstd_core.cuh's huf_read_weights, still the host/test restatement -- took 67 us per tree, this one ~12.)
        __shared__ __align__(16) uint8_t tree[192];         // the tree description (<= 129 bytes), zero padded
        __shared__ __align__(16) uint32_t sb[48];           // the FSE bitstream of the weights behind 16 zero bytes
        __shared__ uint32_t cells[64];                      // symbol | bits << 8 | base << 16
        __shared__ uint8_t cell_sym[64];
        __shared__ __align__(4) uint8_t w[256];
        __shared__ int s_n, s_mode, s_start, s_nbytes, s_al;
        __shared__ int16_t hnorm[16];
        __shared__ uint16_t hcnt[16], hcum[16];
        const int l1 = threadIdx.x;
        const uint32_t tsize = B.lit_csize < 130u ? B.lit_csize : 130u;
        for (uint32_t i = l1; i < 192; i += 32) tree[i] = i < tsize ? J.comp[B.src_off + B.lit_src + i] : 0;
        for (uint32_t i = l1; i < 64; i += 32) ((uint32_t*)w)[i] = 0;
        for (uint32_t i = l1; i < 48; i += 32) sb[i] = 0;
        if (l1 == 0) { s_n = 0; s_mode = -1; }
        __syncwarp();
        const uint32_t h = tsize ? tree[0] : 0u;
        if (l1 == 0 && tsize) {
            if (h >= 128) { if (1u + (h - 127u + 1u) / 2u <= tsize) { s_mode = 0; s_n = (int)h - 127; } }
            else if (h >= 2 && 1u + h <= tsize) {
                int al = 0;
                // weights are 0..11: at most 13 symbols, at most 64 cells
                const uint32_t used = zc::fse_read_ncount(tree + 1, h, 12, zc::MAX_AL_HUF, hnorm, &al);
                if (used != 0 && used < h) { s_mode = 2; s_start = 1 + (int)used; s_nbytes = (int)(h - used); s_al = al; }
            }
        }
        __syncwarp();
        if (s_mode == 2) {                                   // (uniform) the table of the weights' FSE code, by the whole warp
            const bool good = fse_build_warp(hnorm, 12, s_al, cell_sym, hcnt, hcum, l1,
                                             [&](int i, int sy, int nb, int base) { cells[i] = (uint32_t)sy | ((uint32_t)nb << 8) | ((uint32_t)base << 16); });
            __syncwarp();
            if (l1 == 0) s_mode = good ? 1 : -1;
            __syncwarp();
        }
        int n = 0;
        bool good = s_mode >= 0;
        if (s_mode == 0) {
            n = s_n;
            for (int i = l1; i < n; i += 32) { const uint8_t b = tree[1 + (i >> 1)]; w[i] = (i & 1) ? (b & 15) : (b >> 4); }
        } else if (s_mode == 1) {
            for (int i = l1; i < s_nbytes; i += 32) ((uint8_t*)sb)[16 + i] = tree[s_start + i];
            __syncwarp();
            if (l1 == 0) {
                const uint8_t last = ((const uint8_t*)sb)[16 + s_nbytes - 1];
                bool ok = last != 0;
                if (ok) {
                    // Two interleaved states over one backward bitstream.  `pos` = unread bits; a field is cut straight out of
                    // the image (16 zero bytes below bit 0: an over-read yields zeros and a negative pos, which ends the walk
                    // exactly where the serial reader does).  Both cells of a pair are fetched before either state moves, so the
                    // two table look-ups overlap: ~40 cycles per weight instead of ~130 with a refilling reader and a test
                    // after every read (a single small archive waits for this chain: 25 trees x 255 weights).
                    const int al = s_al;
                    int pos = 8 * (s_nbytes - 1) + zc::highbit32(last);
                    pos -= al; uint32_t s1 = smem_bits(sb, 128 + pos, (uint32_t)al);
                    pos -= al; uint32_t s2 = smem_bits(sb, 128 + pos, (uint32_t)al);
                    ok = pos >= 0;
                    int k = 0;
                    bool ended = false;
                    // (one test per pair of weights: at most 254 weights before the last one = 127 pairs; both weights of a pair are
                    //  stored whatever happens -- when the stream ends inside the pair they are exactly what the serial reader emits)
                    if (ok) for (int it = 0; it < 127; it++) {
                        const uint32_t c1 = cells[s1], c2 = cells[s2];
                        const int n1 = (int)((c1 >> 8) & 0xFF), n2 = (int)((c2 >> 8) & 0xFF);
                        const int p1 = pos - n1, p2 = p1 - n2;
                        const uint32_t b1 = smem_bits(sb, 128 + p1, (uint32_t)n1);
                        const uint32_t b2 = smem_bits(sb, 128 + (p2 < -96 ? -96 : p2), (uint32_t)n2);
                        w[k] = (uint8_t)c1; w[k + 1] = (uint8_t)c2;
                        s1 = (c1 >> 16) + b1;
                        s2 = (c2 >> 16) + b2;
                        if (p2 < 0) {
                            if (p1 < 0) k += 2;                                            // the stream ended with the first of the pair
                            else { w[k + 2] = (uint8_t)cells[s1]; k += 3; }                // ... with the second
                            ended = true;
                            break;
                        }
                        k += 2; pos = p2;
                    }
                    ok = ok && ended;
                    s_n = ok ? k : 0;
                }
                if (!ok) s_n = 0;
            }
            __syncwarp();
            n = s_n;
            good = n > 0;
        }
        __syncwarp();
        // validation: weights <= 11, the sum of 2^(w-1) is short of a power of two by a power of two (the implied last weight),
        // and at least two symbols of weight 1, the implied one included (libzstd's HUF_readStats: the longest codes come in
        // pairs; a tree without them, e.g. weights 2, 2, has no code of Max_Number_of_Bits)
        uint32_t tot = 0, bad = 0, ones = 0;
        for (int i = l1; i < n; i += 32) { const uint32_t x = w[i]; if (x > (uint32_t)zc::HUF_MAX_BITS) bad = 1; else if (x) tot += 1u << (x - 1); ones += x == 1; }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            tot += __shfl_xor_sync(0xFFFFFFFFu, tot, d); bad |= __shfl_xor_sync(0xFFFFFFFFu, bad, d); ones += __shfl_xor_sync(0xFFFFFFFFu, ones, d);
        }
        int ns = 0, mb = 0;
        if (good && !bad && tot != 0) {
            mb = zc::highbit32(tot) + 1;
            const uint32_t left = (1u << mb) - tot;
            if (mb <= zc::HUF_MAX_BITS && (left & (left - 1)) == 0 && ones + (left == 1u) >= 2) {
                if (l1 == 0) w[n] = (uint8_t)(zc::highbit32(left) + 1);
                ns = n + 1;
            }
        }
        __syncwarp();
        uint32_t* gw = (uint32_t*)(J.huf_weights + (size_t)B.huf_slot * 256);
        for (int i = l1; i < 64; i += 32) gw[i] = ((const uint32_t*)w)[i];
        if (l1 != 0) return;
        J.huf_meta[(size_t)B.huf_slot * 2] = (uint8_t)(ns ? ns - 1 : 0);
        J.huf_meta[(size_t)B.huf_slot * 2 + 1] = (uint8_t)(ns ? mb : 0);
        if (ns == 0) flag_error(J, B.frame, zc::E_HUF_TREE);
        return;
    }
    __shared__ int16_t norm[3][56];
    __shared__ uint8_t cell_sym[3][512];
    __shared__ uint16_t cnt[3][56];
    __shared__ int al[3];
    __shared__ int mode[3];
    __shared__ int rle_sym[3];
    __shared__ int ok;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t bi = blockIdx.x;
    uint32_t slot[3];
    uint32_t frame = 0;
    if (bi == J.n_blocks) {                 // predefined tables
        if (threadIdx.x < 3) {
            int k = (int)threadIdx.x;
            for (int s = 0; s <= zc::kind_max_symbol(k); s++) norm[k][s] = zc::predef_norm(k, s);
            al[k] = zc::predef_al(k);
            mode[k] = SM_FSE;
        }
        if (threadIdx.x == 0) ok = 1;
        slot[0] = 0; slot[1] = 1; slot[2] = 2;
    } else {
        const BlockDesc& B = J.blocks[bi];
        if (B.btype != BT_COMPRESSED || B.n_seq == 0) return;
        frame = B.frame;
        slot[0] = B.tbl[0]; slot[1] = B.tbl[1]; slot[2] = B.tbl[2];
        // stage the table descriptions (at most ~3 x 64 bytes) in shared memory for the serial bit parser
        __shared__ __align__(16) uint8_t desc[272];
        const uint32_t dsize = (B.src_size - B.seq_src) < 240u ? (B.src_size - B.seq_src) : 240u;
        for (uint32_t i = threadIdx.x; i < 272; i += blockDim.x) desc[i] = i < dsize ? J.comp[B.src_off + B.seq_src + i] : 0;
        for (uint32_t i = threadIdx.x; i < 3 * 56; i += blockDim.x) (&norm[0][0])[i] = 0;
        __syncthreads();
        if (threadIdx.x == 0) {
            ok = 1;
            const uint8_t* src = desc - B.seq_src;      // so that src[p] addresses the staged copy for p >= seq_src
            uint32_t p = B.seq_src;
            for (int k = 0; k < 3; k++) {
                int m = (B.modes >> (6 - 2 * k)) & 3;
                mode[k] = (B.defines >> k) & 1 ? m : -1;
                if (p - B.seq_src + 80 > 256 && (m == SM_RLE || m == SM_FSE)) src = J.comp + B.src_off;   // oversized: read global memory
                if (m == SM_RLE) {
                    if (p >= B.src_size) { ok = 0; break; }
                    rle_sym[k] = src[p++];
                    if (rle_sym[k] > zc::kind_max_symbol(k)) { ok = 0; break; }
                } else if (m == SM_FSE) {
                    int a = 0;
                    const bool in_stage = src != J.comp + B.src_off;         // (else: oversized descriptions, read from global memory)
                    uint32_t used = in_stage ? fse_read_ncount_staged((const uint32_t*)desc, p - B.seq_src, B.src_size - p, zc::kind_max_symbol(k), zc::kind_max_al(k), norm[k], &a)
                                             : zc::fse_read_ncount(src + p, B.src_size - p, zc::kind_max_symbol(k), zc::kind_max_al(k), norm[k], &a);
                    if (used == 0 || p + used > B.src_size) { ok = 0; break; }
                    al[k] = a;
                    p += used;
                }
            }
            if (p >= B.src_size) ok = 0;      // the bitstream needs at least one byte
            J.bstate[bi].seq_bits_off = p;
        }
    }
    __syncthreads();
    if (!ok) {
        if (threadIdx.x == 0) flag_error(J, frame, zc::E_FSE_TABLE);
        return;
    }
    __shared__ uint16_t cum3[3][60];
    for (int k = warp; k < 3; k += (int)(blockDim.x >> 5)) {            // (mode, al, norm are uniform: shared memory) one table per warp
        uint16_t* cum = cum3[k];
        if (mode[k] < 0) continue;
        SeqCell* T = J.tables + (size_t)slot[k] * FSE_SLOT_CELLS;
        if (mode[k] == SM_RLE) {
            if (lane == 0) { T[0] = zc::make_seq_cell(k, rle_sym[k], 0, 0); J.table_al[slot[k]] = 0; }
        } else {
            const bool good = fse_build_warp(norm[k], zc::kind_max_symbol(k), al[k], cell_sym[k], cnt[k], cum, lane,
                                             [&](int i, int s, int nb, int base) { T[i] = zc::make_seq_cell(k, s, nb, base); });
            if (lane == 0) { J.table_al[slot[k]] = (uint8_t)al[k]; if (!good) flag_error(J, frame, zc::E_FSE_TABLE); }
        }
        __syncwarp();
    }
}

// --------------------------------------------------------------------------------------------------------------
// k_decode_sequences: the serial FSE stage.  One warp per block, lane 0 walks the three interleaved tANS states.
// The repeat-offset state is tracked symbolically (each slot = constant, or incoming slot minus a delta) so blocks
// decode independently; k_frame_scan composes the per-block transfer functions.
struct RepSym { int32_t src; uint32_t val; };   // src < 0: constant val; else rep_in[src] - val

__device__ __forceinline__ uint32_t encode_off(RepSym r) {
    return r.src < 0 ? r.val : (OFF_SYMBOLIC | ((uint32_t)r.src << 29) | (r.val & 0x1FFFFFFFu));
}



// A transfer function of the three repeat offsets: slot k = constant v[k] (s[k] < 0), or incoming slot s[k] minus v[k].  One
// sequence is such a map, so is a block, so is any run of either: they compose associatively (scans below and in k_frame_scan).
struct RepMap { int32_t s[3]; uint32_t v[3]; };

__device__ __forceinline__ void rep_identity(RepMap& m) { m.s[0] = 0; m.s[1] = 1; m.s[2] = 2; m.v[0] = m.v[1] = m.v[2] = 0; }

// m <- (m after f).  Branch-free: the consumer warp of k_decode_sequences runs this inside a shuffle scan, and a lone warp pays
// for every divergent branch (the same rewrite of the producer's loop took it from 284 to 189 cycles per sequence).
__device__ __forceinline__ void rep_compose(RepMap& m, const RepMap& f, bool& bad) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const int sk = m.s[k];
        const bool has = sk >= 0;
        const int32_t es = sk == 0 ? f.s[0] : (sk == 1 ? f.s[1] : f.s[2]);
        const uint32_t ev = sk == 0 ? f.v[0] : (sk == 1 ? f.v[1] : f.v[2]);
        const bool cst = es < 0;
        const bool badk = has && cst && ev <= m.v[k];
        const uint32_t nv = cst ? ev - m.v[k] : ev + m.v[k];
        m.v[k] = has ? (badk ? 1u : nv) : m.v[k];
        m.s[k] = has ? (cst ? -1 : es) : sk;
        bad = bad || badk;
    }
}

// m <- (m after f) where `take` holds, m otherwise (no branch)
__device__ __forceinline__ void rep_compose_if(RepMap& m, const RepMap& f, bool take, bool& bad) {
    RepMap t = m;
    bool b = false;
    rep_compose(t, f, b);
#pragma unroll
    for (int k = 0; k < 3; k++) { m.s[k] = take ? t.s[k] : m.s[k]; m.v[k] = take ? t.v[k] : m.v[k]; }
    bad = bad || (take && b);
}

// out <- m(in); returns false if an offset would not be positive
__device__ __forceinline__ bool rep_apply(const RepMap& m, const uint32_t in[3], uint32_t out[3]) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        if (m.s[k] < 0) out[k] = m.v[k];
        else {
            const uint32_t x = m.s[k] == 0 ? in[0] : (m.s[k] == 1 ? in[1] : in[2]);
            if (x <= m.v[k]) { ok = false; out[k] = 1; } else out[k] = x - m.v[k];
        }
    }
    return ok;
}

// inclusive scan of maps over the lanes of a warp (lane i ends up with map_i after ... after map_0)
__device__ __forceinline__ void rep_warp_scan(RepMap& m, int lane, bool& bad) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        RepMap f;
#pragma unroll
        for (int k = 0; k < 3; k++) { f.s[k] = __shfl_up_sync(0xFFFFFFFFu, m.s[k], d); f.v[k] = __shfl_up_sync(0xFFFFFFFFu, m.v[k], d); }
        rep_compose_if(m, f, lane >= d, bad);
    }
}

__device__ __forceinline__ void rep_shfl(RepMap& out, const RepMap& m, int src) {
#pragma unroll
    for (int k = 0; k < 3; k++) { out.s[k] = __shfl_sync(0xFFFFFFFFu, m.s[k], src); out.v[k] = __shfl_sync(0xFFFFFFFFu, m.v[k], src); }
}

// The tANS walk, written once over a reader type: shared-memory window (common) or global memory (huge sections).
// PRODUCER side of k_decode_sequences: decodes `cnt` sequences into raw (offset value, match length, literal length)
// triples in shared memory; the three states live in the caller's registers across batches.
template <class RD>
__device__ __forceinline__ void seq_produce(RD& rd, const SeqCell* TLL, const SeqCell* TOF, const SeqCell* TML, uint32_t& sLL, uint32_t& sOF,
                                            uint32_t& sML, uint32_t cnt, bool last_batch, uint32_t* r_ov, uint32_t* r_ml, uint32_t* r_ll) {
    for (uint32_t j = 0; j < cnt; j++) {
        const SeqCell cOF = TOF[sOF], cML = TML[sML], cLL = TLL[sLL];
        r_ov[j] = cOF.base_value + rd.read(cOF.add_bits);
        const uint32_t xb = rd.read(cML.add_bits + cLL.add_bits);        // ML then LL extra bits, one read
        r_ml[j] = cML.base_value + (xb >> cLL.add_bits);
        r_ll[j] = cLL.base_value + (xb & ((1u << cLL.add_bits) - 1u));
        if (!(last_batch && j + 1 == cnt)) {                             // LL, ML, OF state bits (<= 27) in one read
            const uint32_t sb = rd.read(cLL.nb + cML.nb + cOF.nb);
            sOF = cOF.next_base + (sb & ((1u << cOF.nb) - 1u));
            sML = cML.next_base + ((sb >> cOF.nb) & ((1u << cML.nb) - 1u));
            sLL = cLL.next_base + (sb >> (cOF.nb + cML.nb));
        }
    }
}

// The same walk over the shared-memory image by THREE LANES, one per state (lane 0: offset, 1: match length, 2: literal
// length).  Measured (ncu, round 1; and two rewrites of the one-lane reader this round): a lone lane retires one instruction
// per ~5 cycles whether or not the instructions depend on each other, so what counts is the NUMBER of warp instructions
// per sequence -- 133 in the one-lane walk.  Here every lane loads its own cell, the field widths of the three cells are
// exchanged with three shuffles (packed: extra bits | state bits << 8), and every lane cuts its own two fields (extra bits,
// next-state bits) straight out of the shared-memory image at the bit address that the prefix sums of those widths give:
//   extra bits, consumed OF, ML, LL from position P down:   field k = [P - pre_a(k) - a_k, P - pre_a(k))
//   state bits, consumed LL, ML, OF after them:             field k = [Pend + pre_n(k), Pend + pre_n(k) + n_k),  Pend = P - sum a - sum n
// ~40 warp instructions per sequence, no reader state but P.

// All 32 lanes of the producer warp call this; lanes 0..2 work.  Decodes `cnt` sequences from smem bit position P (counting
// down); returns false once the stream is over-read (P below x_zero: corrupt) -- uniform, P is the same in every lane.
// bits [o, o + k) for k <= 31 (field widths of the sequence codes: at most 31 extra bits, 9 state bits): one instruction less than
// the general form, and no select
__device__ __forceinline__ uint32_t smem_bits31(const uint32_t* sw, int o, uint32_t k) {
    const uint32_t lo = sw[o >> 5], hi = sw[(o >> 5) + 1];
    return __funnelshift_r(lo, hi, (uint32_t)o) & ~(0xFFFFFFFFu << k);
}

__device__ __forceinline__ bool seq_produce3(const uint32_t* sw, int& P, int x_zero, const SeqCell* T, uint32_t& state, int lane, uint32_t cnt,
                                             bool last_batch, uint32_t* r_mine) {
    // the widths travel as  nb | add_bits << 8  = the top half of the cell's second word, as it is
    const uint32_t j_last = last_batch ? cnt - 1u : 0xFFFFFFFFu;       // no state update after the last sequence of the block
    const bool mine = lane < 3;
    for (uint32_t j = 0; j < cnt; j++) {
        if (P < x_zero) return false;
        const uint2 q = *(const uint2*)&T[state];                       // base_value | next_base (16) | nb (8) | add_bits (8)
        uint32_t pk = mine ? q.y >> 16 : 0u;
        if (j == j_last) pk &= 0xFF00u;
        const uint32_t p0 = __shfl_sync(0xFFFFFFFFu, pk, 0), p1 = __shfl_sync(0xFFFFFFFFu, pk, 1), p2 = __shfl_sync(0xFFFFFFFFu, pk, 2);
        const uint32_t tot = p0 + p1 + p2;                              // sums stay inside their bytes (3 x 9, 3 x 31)
        const uint32_t pre = (lane > 0 ? p0 : 0u) + (lane > 1 ? p1 : 0u);
        const int Pend = P - (int)(tot & 0xFFu) - (int)(tot >> 8);
        // (no branch around the three working lanes -- a lone warp pays dearly for divergence: the others cut empty fields at
        //  valid addresses and keep state 0)
        const uint32_t a = pk >> 8, n = pk & 0xFFu;
        const uint32_t v = q.x + smem_bits31(sw, P - (int)(pre >> 8) - (int)a, a);
        const uint32_t ns = (q.y & 0xFFFFu) + smem_bits31(sw, Pend + (int)(pre & 0xFFu), n);
        if (mine) r_mine[j] = v;
        state = mine ? ns : 0u;
        P = Pend;
    }
    return true;
}

// The same loop with everything it touches (bit image, the lane's table, the lane's output array) addressed by 32-bit
// shared-space addresses: with generic pointers nvcc re-derived the shared window base inside the loop (S2R SR_CgaCtaId + LEA in
// front of every load -- on the dependent chain of every sequence).  k_decode_sequences' producer; the tiny-block kernel, whose
// tables stay in global memory, keeps the generic form above.
__device__ __forceinline__ uint32_t sbits31(saddr_t sw, int o, uint32_t k) {
    o = o < 0 ? 0 : o;                                 // (a corrupt stream over-reads: it is caught after the batch, P below the zero padding)
    const saddr_t a = sw + (saddr_t)(4 * (o >> 5));
    return __funnelshift_r(lds32(a), lds32(a + 4), (uint32_t)o) & ~(0xFFFFFFFFu << k);
}

__device__ __forceinline__ bool seq_produce3s(saddr_t sw, int& P, int x_zero, saddr_t T, uint32_t& state, int lane, uint32_t cnt,
                                              bool last_batch, saddr_t r_mine) {
    const uint32_t j_last = last_batch ? cnt - 1u : 0xFFFFFFFFu;
    const bool mine = lane < 3;
    (void)x_zero;
    for (uint32_t j = 0; j < cnt; j++) {
        const uint2 q = lds64(T + 8u * state);
        uint32_t pk = mine ? q.y >> 16 : 0u;
        if (j == j_last) pk &= 0xFF00u;
        const uint32_t p0 = __shfl_sync(0xFFFFFFFFu, pk, 0), p1 = __shfl_sync(0xFFFFFFFFu, pk, 1), p2 = __shfl_sync(0xFFFFFFFFu, pk, 2);
        const uint32_t tot = p0 + p1 + p2;
        const uint32_t pre = (lane > 0 ? p0 : 0u) + (lane > 1 ? p1 : 0u);
        const int Pend = P - (int)(tot & 0xFFu) - (int)(tot >> 8);
        // (no branch around the three working lanes: the others cut empty fields at valid addresses and keep state 0)
        const uint32_t a = pk >> 8, n = pk & 0xFFu;
        const uint32_t v = q.x + sbits31(sw, P - (int)(pre >> 8) - (int)a, a);
        const uint32_t ns = (q.y & 0xFFFFu) + sbits31(sw, Pend + (int)(pre & 0xFFu), n);
        if (mine) sts32(r_mine + 4u * j, v);
        state = mine ? ns : 0u;
        P = Pend;
    }
    return true;
}

// CONSUMER side, one batch of at most 32 sequences held by a warp (lane j: sequence j): repeat offsets, positions, records.
struct SeqTotals {
    RepMap carry;                    // the block's repeat-offset map up to the current batch (uniform over the warp)
    uint32_t litpos, outpos;         // running totals, uniform over the warp
    bool bad;
    __device__ __forceinline__ void init() { rep_identity(carry); litpos = outpos = 0; bad = false; }
};

__device__ __forceinline__ void seq_consume_batch(uint32_t* b_ov, const uint32_t* b_ml, const uint32_t* b_ll, uint32_t cnt, int lane, uint4* rec,
                                                  uint32_t bi, SeqTotals& t) {
    const uint32_t ll = (uint32_t)lane < cnt ? b_ll[lane] : 0u, ml = (uint32_t)lane < cnt ? b_ml[lane] : 0u;
    {
        // repeat offsets (RFC 8878 3.1.1.5): what a sequence does to the three slots is a map; the offset it uses is slot 0
        // AFTER its own map.  An inclusive scan over the batch (on top of the carry) gives every sequence its offset,
        // symbolically in the block's incoming slots -- 5 shuffle steps instead of a 32-step chain in one lane (which had
        // become as slow as the tANS walk: 319 cycles per sequence, measured).
        RepMap m; rep_identity(m);
        if ((uint32_t)lane < cnt) {
            const uint32_t ov = b_ov[lane];
            if (ov > 3) { m.s[0] = -1; m.v[0] = ov - 3; m.s[1] = 0; m.s[2] = 1; }
            else {
                const uint32_t idx = ov - 1 + (ll == 0 ? 1u : 0u);
                if (idx == 1) { m.s[0] = 1; m.s[1] = 0; }
                else if (idx == 2) { m.s[0] = 2; m.s[1] = 0; m.s[2] = 1; }
                else if (idx == 3) { m.v[0] = 1; m.s[1] = 0; m.s[2] = 1; }
            }
        }
        rep_compose_if(m, t.carry, lane == 0, t.bad);
        if (cnt <= 8) {
            // a handful of sequences (the tiny blocks of a FASTQ section flushed per record): a short chain of shuffles is
            // cheaper than the five-step scan
            for (uint32_t j = 1; j < cnt; j++) {
                RepMap f;
                rep_shfl(f, m, (int)j - 1);
                rep_compose_if(m, f, (uint32_t)lane == j, t.bad);
            }
            RepMap last;
            rep_shfl(last, m, (int)cnt - 1);
            if ((uint32_t)lane >= cnt) m = last;                     // (lane 31 carries the batch's total below)
        } else rep_warp_scan(m, lane, t.bad);
        RepSym off; off.src = m.s[0]; off.val = m.v[0];
        if (off.src >= 0 ? off.val > 0x1FFFFFFFu : off.val > 0x7FFFFFFFu) t.bad = true;    // (raw offsets with bit 31 set: OF codes 31+, corrupt)
        if ((uint32_t)lane < cnt) b_ov[lane] = encode_off(off);
        rep_shfl(t.carry, m, 31);                        // (lanes past the batch hold the identity: lane 31 has the batch's total)
    }
    __syncwarp();
    // positions: exclusive scans of ll and ll + ml over the batch, on top of the running totals
    uint32_t il = ll, io = ll + ml;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t tl = __shfl_up_sync(0xFFFFFFFFu, il, d), to = __shfl_up_sync(0xFFFFFFFFu, io, d);
        if (lane >= d) { il += tl; io += to; }
    }
    if ((uint32_t)lane < cnt) {
        const uint32_t lp = t.litpos + il - ll, op = t.outpos + io - (ll + ml);
        rec[2 * lane] = make_uint4(ll, ml, b_ov[lane], lp);
        rec[2 * lane + 1] = make_uint4(op, bi, 0u, 0u);
    }
    t.litpos += __shfl_sync(0xFFFFFFFFu, il, 31);
    const uint32_t otot = __shfl_sync(0xFFFFFFFFu, io, 31);
    if (otot > BLOCK_MAX || t.outpos + otot > BLOCK_MAX) t.bad = true;      // (match lengths are < 2^17 each: no wrap within a batch)
    t.outpos += otot;
}

// what a block's sequences leave behind (one lane): regenerated size, the block's repeat-offset map
__device__ __forceinline__ void seq_finish_block(const JobDev& J, const BlockDesc& B, BlockState& S, const SeqTotals& t, int left) {
    if (t.bad || left != 0) { flag_error(J, B.frame, zc::E_SEQ_STREAM); return; }
    if (t.litpos > B.lit_regen) { flag_error(J, B.frame, zc::E_LITERALS); return; }
    const uint32_t regen = t.outpos + (B.lit_regen - t.litpos);
    if (regen > BLOCK_MAX) { flag_error(J, B.frame, zc::E_SIZE); return; }
    S.regen = regen;
    for (int k = 0; k < 3; k++) { S.rep_src[k] = t.carry.s[k]; S.rep_val[k] = t.carry.v[k]; }
}

// k_decode_sequences: one CTA of two warps per block.  Warp 0, lane 0 is the PRODUCER: the serial chain of the three
// interleaved tANS states and nothing else (every instruction on it costs ~6 cycles of a lone dependent warp: ncu shows
// `wait` as the top stall, profiles/r1_fse_stage_k_decode_sequences.txt).  Warp 1 is the CONSUMER, one batch of 32
// sequences behind through a double buffer in shared memory: repeat-offset bookkeeping (symbolic, so blocks decode
// independently), literal / output positions by a shuffle scan, and the 32-byte sequence records with coalesced stores.
constexpr uint32_t SEQ_BATCH = 32;

// optional cycle accounting of the two sides (NAFGPU_DEBUG_HUF=1): work vs waiting at the hand-over barrier
#if defined(__CUDA_ARCH__)
#define SEQ_CLK(t) do { if (J.debug_seq) t = clock64(); } while (0)
#define SEQ_LAP(acc, t) do { if (J.debug_seq) { const long long _n = clock64(); acc += _n - t; t = _n; } } while (0)
#define SEQ_REPORT(slot, a, b, nseq) do { if (J.debug_seq && lane == 0) { atomicAdd(&J.debug_seq[slot], (unsigned long long)(a)); atomicAdd(&J.debug_seq[(slot) + 1], (unsigned long long)(b)); \
                                         if (nseq) atomicAdd(&J.debug_seq[4], (unsigned long long)(nseq)); } } while (0)
#else
#define SEQ_CLK(t) ((void)t)
#define SEQ_LAP(acc, t) ((void)acc)
#define SEQ_REPORT(slot, a, b, nseq) ((void)0)
#endif

// A block whose sequences are not decoded (its frame failed before, or its own stream is corrupt) still owns its records:
// the LZ stages find the frame of sequence i through J.seq[i].block before they look at the frame's status, and a record
// left as the previous job wrote it would send them to another frame's block, or past the end of the tables.
__device__ __forceinline__ void seq_claim_records(const JobDev& J, const BlockDesc& B, uint32_t bi, uint32_t t, uint32_t nt) {
    for (uint32_t j = t; j < B.n_seq; j += nt) J.seq[B.seq_base + j].block = bi;
}

__global__ void __launch_bounds__(64) k_decode_sequences(JobDev J) {
    NAF_DYN_SMEM(uint32_t, sbits);                       // staged bitstream: J.seq_stage_bytes (job maximum, capped)
    __shared__ __align__(8) SeqCell stab[3][FSE_SLOT_CELLS];
    __shared__ uint32_t r_ov[2][SEQ_BATCH], r_ml[2][SEQ_BATCH], r_ll[2][SEQ_BATCH];
    __shared__ int s_left;
    const uint32_t bi = J.tiny_blocks ? J.seq_big_list[blockIdx.x] : blockIdx.x;      // (with tiny_blocks: a list of the blocks that are not
    const BlockDesc& B = J.blocks[bi];                                                  //  k_decode_sequences_tiny's -- 2 x 10^6 CTAs that exit at once cost 2.9 ms)
    if (B.btype != BT_COMPRESSED || B.n_seq == 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (J.frame_bad[B.frame]) { seq_claim_records(J, B, bi, tid, 64); return; }
    BlockState& S = J.bstate[bi];
    const uint8_t* src = J.comp + B.src_off;
    if (S.seq_bits_off >= B.src_size) { if (tid == 0) flag_error(J, B.frame, zc::E_SEQ_STREAM); seq_claim_records(J, B, bi, tid, 64); return; }
    const uint32_t nbytes = B.src_size - S.seq_bits_off;
    const uint8_t* g = src + S.seq_bits_off;
    const bool staged = nbytes + 48 <= J.seq_stage_bytes;
    const uint32_t a = (uint32_t)((uintptr_t)g & 15);
    int al[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        al[k] = J.table_al[B.tbl[k]];
        const uint2* T = (const uint2*)(J.tables + (size_t)B.tbl[k] * FSE_SLOT_CELLS);
        for (int i = tid; i < (1 << al[k]); i += 64) ((uint2*)stab[k])[i] = T[i];
    }
    if (staged) {
        const uint4* gbase = (const uint4*)(g - a);
        const uint32_t nchunks = (a + nbytes + 15) >> 4;
        for (uint32_t c = tid; c < nchunks; c += 64) ((uint4*)sbits)[1 + c] = gbase[c];
    }
    const uint8_t last = g[nbytes - 1];
    if (last == 0) { if (tid == 0) flag_error(J, B.frame, zc::E_SEQ_STREAM); seq_claim_records(J, B, bi, tid, 64); return; }     // (uniform)
    __syncthreads();
    if (staged && (uint32_t)tid < 16 + a) ((uint8_t*)sbits)[tid] = 0;
    if (tid == 0) s_left = 0;
    __syncthreads();
    const int P0 = 8 * (int)(nbytes - 1) + zc::highbit32(last);
    const uint32_t n = B.n_seq, base = B.seq_base;
    const uint32_t nbatch = (n + SEQ_BATCH - 1) / SEQ_BATCH;
    if (warp == 0) {
        // ---- producer ---------------------------------------------------------------------------------------------
        BackBits rg{};
        const int xz = (int)(16 + a) * 8;                // smem bit position of stream bit 0
        int P = xz + P0;                                 // staged: the smem bit position of the next unread bit (the same in every lane)
        uint32_t sLL = 0, sOF = 0, sML = 0;              // global-memory reader (lane 0)
        uint32_t state = 0;                              // staged reader: this lane's state (lane 0: OF, 1: ML, 2: LL)
        const int kind = lane == 0 ? 1 : (lane == 1 ? 2 : 0);                               // stab / al / r_* index of the lane's state
        uint32_t* const r_base = lane == 0 ? &r_ov[0][0] : (lane == 1 ? &r_ml[0][0] : &r_ll[0][0]);
        bool dead = false;
        saddr_t s_bits_a = to_saddr(sbits), s_tab_a = to_saddr(stab[kind]), s_out_a = to_saddr(r_base);
#if defined(__CUDA_ARCH__)
        // (opaque to the compiler, or it rematerialises the three addresses from SR_CgaCtaId inside the loop)
        asm volatile("" : "+r"(s_bits_a), "+r"(s_tab_a), "+r"(s_out_a));
#endif
        if (staged) {
            // the three initial states: AL_ll, AL_of, AL_ml bits from the top, in that order
            const int before = lane == 2 ? 0 : (lane == 0 ? al[0] : al[0] + al[1]);
            if (lane < 3) state = smem_bits(sbits, P - before - al[kind], (uint32_t)al[kind]);
            P -= al[0] + al[1] + al[2];
        } else if (lane == 0) { rg.init(g, nbytes); sLL = rg.read(al[0]); sOF = rg.read(al[1]); sML = rg.read(al[2]); }
        long long t_work = 0, t_wait = 0, t0 = 0;
        for (uint32_t k = 0; k < nbatch; k++) {
            const uint32_t cnt = (k + 1 < nbatch) ? SEQ_BATCH : n - k * SEQ_BATCH;
            SEQ_CLK(t0);
            if (staged) {
                if (!dead) {
                    const bool ok = seq_produce3s(s_bits_a, P, xz, s_tab_a, state, lane, cnt, k + 1 == nbatch, s_out_a + (saddr_t)((k & 1) * SEQ_BATCH * 4));
                    // a corrupt stream over-reads: bit addresses are clamped to the image (no test inside the chain), P ends below
                    // bit 0, the block is flagged and the batches after this one are not decoded
                    const int left = ok ? P - xz : -1;
                    if (left < 0) { dead = true; if (lane == 0) s_left = left; }
                    else if (k + 1 == nbatch && lane == 0) s_left = left;
                }
            } else if (lane == 0 && !dead) {
                seq_produce(rg, stab[0], stab[1], stab[2], sLL, sOF, sML, cnt, k + 1 == nbatch, r_ov[k & 1], r_ml[k & 1], r_ll[k & 1]);
                const int left = (int)rg.P;
                if (left < 0) { dead = true; s_left = left; }
                else if (k + 1 == nbatch) s_left = left;
            }
            SEQ_LAP(t_work, t0);
            __syncthreads();                             // batch k is ready; the consumer has finished batch k - 1
            SEQ_LAP(t_wait, t0);
        }
        SEQ_REPORT(0, t_work, t_wait, n);
        return;
    }
    // ---- consumer -------------------------------------------------------------------------------------------------
    SeqTotals tot; tot.init();
    uint4* rec = (uint4*)(J.seq + base);
    long long c_work = 0, c_wait = 0, c0 = 0;
    SEQ_CLK(c0);
    for (uint32_t k = 0; k < nbatch; k++) {
        SEQ_LAP(c_work, c0);
        __syncthreads();
        SEQ_LAP(c_wait, c0);
        const uint32_t cnt = (k + 1 < nbatch) ? SEQ_BATCH : n - k * SEQ_BATCH;
        seq_consume_batch(r_ov[k & 1], r_ml[k & 1], r_ll[k & 1], cnt, lane, rec + 2 * (size_t)k * SEQ_BATCH, bi, tot);
    }
    tot.bad = __any_sync(0xFFFFFFFFu, tot.bad);
    if (lane != 0) return;
    SEQ_LAP(c_work, c0);
    SEQ_REPORT(2, c_work, c_wait, 0);
    seq_finish_block(J, B, S, tot, s_left);
}

// The same decode for TINY blocks (at most one batch of sequences): one WARP per block, eight blocks per CTA.  A FASTQ
// archive in the reference encoder's framing (one flush per record) is 2 x 10^6 blocks of 3-20 sequences per 10^6 reads; a
// two-warp CTA each, with the shared memory of the job's largest block, kept an SM at 5-7 blocks in flight (11 ms for 10^6
// reads).  Here the bitstream (at most 361 bytes: 32 sequences of at most 89 bits, 26 bits of initial states, the end mark)
// is staged per warp, the table cells are read where k_build_tables left them (a tiny block uses predefined or repeated
// tables: hot in L1), lanes 0..2 walk the three states, and the same warp then does the consumer's batch.
constexpr int SEQ_TINY_WARPS = 8;
constexpr uint32_t SEQ_TINY_BYTES = 368;
constexpr uint32_t SEQ_TINY_WORDS = (16 + 16 + SEQ_TINY_BYTES + 16 + 16) / 4;

__global__ void __launch_bounds__(SEQ_TINY_WARPS * 32) k_decode_sequences_tiny(JobDev J) {
    __shared__ __align__(16) uint32_t sb_all[SEQ_TINY_WARPS][SEQ_TINY_WORDS];
    __shared__ uint32_t r_all[SEQ_TINY_WARPS][3][SEQ_BATCH];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t bi = blockIdx.x * SEQ_TINY_WARPS + warp;
    if (bi >= J.n_blocks) return;
    const BlockDesc& B = J.blocks[bi];
    if (!tiny_seq_block(B)) return;
    if (J.frame_bad[B.frame]) { seq_claim_records(J, B, bi, lane, 32); return; }
    BlockState& S = J.bstate[bi];
    if (S.seq_bits_off >= B.src_size) { if (lane == 0) flag_error(J, B.frame, zc::E_SEQ_STREAM); seq_claim_records(J, B, bi, lane, 32); return; }
    const uint32_t nbytes = B.src_size - S.seq_bits_off;
    const uint8_t* g = J.comp + B.src_off + S.seq_bits_off;
    // (more bytes than 32 sequences can consume: the stream cannot end exactly at bit 0)
    if (nbytes > SEQ_TINY_BYTES || g[nbytes - 1] == 0) { if (lane == 0) flag_error(J, B.frame, zc::E_SEQ_STREAM); seq_claim_records(J, B, bi, lane, 32); return; }
    uint32_t* sbits = sb_all[warp];
    const uint32_t a = (uint32_t)((uintptr_t)g & 15);
    const uint32_t nchunks = (a + nbytes + 15) >> 4;                       // <= 25
    if ((uint32_t)lane < nchunks) ((uint4*)sbits)[1 + lane] = ((const uint4*)(g - a))[lane];
    const uint8_t last = g[nbytes - 1];
    __syncwarp();
    if ((uint32_t)lane < 16 + a) ((uint8_t*)sbits)[lane] = 0;
    __syncwarp();
    const int kind = lane == 0 ? 1 : (lane == 1 ? 2 : 0);                  // lane 0: OF, 1: ML, 2: LL (as in k_decode_sequences)
    const int al0 = J.table_al[B.tbl[0]], al1 = J.table_al[B.tbl[1]], al2 = J.table_al[B.tbl[2]];
    const int alk = kind == 0 ? al0 : (kind == 1 ? al1 : al2);
    const SeqCell* T = (const SeqCell*)(J.tables + (size_t)B.tbl[kind] * FSE_SLOT_CELLS);
    const int xz = (int)(16 + a) * 8;
    int P = xz + 8 * (int)(nbytes - 1) + zc::highbit32(last);
    uint32_t state = 0;
    {
        const int before = lane == 2 ? 0 : (lane == 0 ? al0 : al0 + al1);
        if (lane < 3) state = smem_bits(sbits, P - before - alk, (uint32_t)alk);
        P -= al0 + al1 + al2;
    }
    const uint32_t n = B.n_seq;
    uint32_t* r_mine = r_all[warp][kind];
    const bool ok = P >= xz && seq_produce3(sbits, P, xz, T, state, lane, n, true, r_mine);
    const int left = ok ? P - xz : -1;
    __syncwarp();
    SeqTotals tot; tot.init();
    if (left == 0) seq_consume_batch(r_all[warp][1], r_all[warp][2], r_all[warp][0], n, lane, (uint4*)(J.seq + B.seq_base), bi, tot);
    else seq_claim_records(J, B, bi, lane, 32);                             // (the block is flagged below)
    tot.bad = __any_sync(0xFFFFFFFFu, tot.bad);
    if (lane != 0) return;
    seq_finish_block(J, B, S, tot, left);
}

// --------------------------------------------------------------------------------------------------------------
// k_frame_scan: one CTA per frame.  Exclusive prefix sum of regenerated block sizes -> out_off; composes the
// repeat-offset transfer functions -> rep_in per block; checks the total against the size the container states.
//
// A block's effect on the three repeat offsets is a map: slot k = constant v, or incoming slot s minus v (blocks
// without sequences are the identity).  Maps compose associatively, so the chain across the blocks of a frame is a
// scan: shuffles inside a warp, the warps' aggregates scanned once more by every warp; FSCAN_T blocks per step.
// A genome frame has a handful of blocks; a FASTQ section flushed per record has 10^5 of them.
constexpr int FSCAN_T = 512, FSCAN_W = FSCAN_T / 32;

// Blocks [b_begin, b_end) of frame f, FSCAN_T per step.  REDUCE: only what the range does as a whole (regenerated bytes, the
// composed repeat-offset map) -- the first pass over a tile of a long frame.  Otherwise: from the state at b_begin (`off`,
// `rep`), write every block's output offset and incoming repeat offsets; the state after b_end is left in `off` / `rep`.
template <bool REDUCE>
__device__ __forceinline__ void fs_range(const JobDev& J, uint32_t b_begin, uint32_t b_end, uint64_t& off, uint32_t rep[3], RepMap& total, bool& bad) {
    __shared__ RepMap agg_map[2][FSCAN_W];
    __shared__ uint32_t agg_regen[2][FSCAN_W];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int buf = 0;
    for (uint32_t b0 = b_begin; b0 < b_end; b0 += FSCAN_T, buf ^= 1) {
        const uint32_t b = b0 + threadIdx.x;
        const bool valid = b < b_end;
        uint32_t regen = 0;
        bool has_seq = false;
        RepMap m; rep_identity(m);
        if (valid) {
            const BlockDesc& B = J.blocks[b];
            has_seq = B.btype == BT_COMPRESSED && B.n_seq > 0;
            if (has_seq) {
                const BlockState& S = J.bstate[b];
                regen = S.regen;
#pragma unroll
                for (int k = 0; k < 3; k++) { m.s[k] = S.rep_src[k]; m.v[k] = S.rep_val[k]; }
            } else regen = B.known_regen;
        }
        uint32_t inc = regen;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
        rep_warp_scan(m, lane, bad);
        if (lane == 31) { agg_map[buf][w] = m; agg_regen[buf][w] = inc; }
        __syncthreads();                                   // (aggregates are double-buffered: one barrier per step)
        // the warps' aggregates, scanned by every warp for itself
        RepMap a; rep_identity(a);
        uint32_t ar = 0;
        if (lane < FSCAN_W) { a = agg_map[buf][lane]; ar = agg_regen[buf][lane]; }
        uint32_t ainc = ar;
#pragma unroll
        for (int d = 1; d < FSCAN_W; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, ainc, d); if (lane >= d) ainc += t; }
        rep_warp_scan(a, lane, bad);
        RepMap tot;
        rep_shfl(tot, a, FSCAN_W - 1);
        if (REDUCE) {
            rep_compose(tot, total, bad);                  // tot <- (tot after everything so far)
            total = tot;
        } else {
            // everything before this thread's block: the warps before mine, then the lanes before mine
            RepMap wp, x;
            rep_shfl(wp, a, w ? w - 1 : 0);
            uint32_t wregen = __shfl_sync(0xFFFFFFFFu, ainc, w ? w - 1 : 0);
            if (w == 0) { rep_identity(wp); wregen = 0; }
            rep_shfl(x, m, lane ? lane - 1 : 0);
            if (lane == 0) rep_identity(x);
            bool xbad = false;
            rep_compose(x, wp, xbad);
            uint32_t in[3];
            const bool ok = rep_apply(x, rep, in);
            if (valid) {
                BlockState& S = J.bstate[b];
                S.regen = regen; S.out_off = off + wregen + (inc - regen);
                if (has_seq) { S.rep_in[0] = in[0]; S.rep_in[1] = in[1]; S.rep_in[2] = in[2]; if (!ok || xbad) bad = true; }
            }
            // what leaves this group of blocks
            uint32_t out[3];
            if (!rep_apply(tot, rep, out)) bad = true;
            rep[0] = out[0]; rep[1] = out[1]; rep[2] = out[2];
        }
        off += __shfl_sync(0xFFFFFFFFu, ainc, FSCAN_W - 1);
    }
}

__global__ void __launch_bounds__(FSCAN_T) k_frame_scan(JobDev J) {
    const uint32_t f = blockIdx.x;
    if (J.frame_bad[f]) return;
    const FrameDesc& F = J.frames[f];
    if (F.n_blocks > J.fs_big_frame) return;               // long frames: k_fs_reduce / k_fs_prefix / k_fs_apply, a CTA per tile
    uint64_t off = F.dst_off;
    uint32_t rep[3] = {1, 4, 8};
    bool bad = false;
    RepMap unused; rep_identity(unused);
    fs_range<false>(J, F.first_block, F.first_block + F.n_blocks, off, rep, unused, bad);
    if (off - F.dst_off != F.dst_size) bad = true;
    if (__syncthreads_or(bad) && threadIdx.x == 0) flag_error(J, f, zc::E_SIZE);
}

// Frames of more than FS_BIG_FRAME blocks (a FASTQ section flushed per record has 10^6 of them: one CTA took 10 ms for it)
// are cut into tiles of FS_TILE blocks: (1) every tile's aggregate, (2) one thread per frame walks its tiles' aggregates
// -- a few hundred -- and leaves every tile its starting state, (3) every tile scans its blocks from there.
__global__ void __launch_bounds__(FSCAN_T) k_fs_reduce(JobDev J) {
    const FsTile T = J.fs_tiles[blockIdx.x];
    if (J.frame_bad[T.frame]) return;
    uint64_t sum = 0;
    uint32_t rep[3] = {0, 0, 0};
    bool bad = false;
    RepMap total; rep_identity(total);
    fs_range<true>(J, T.first_block, T.first_block + T.n_blocks, sum, rep, total, bad);
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) {
        FsTileState& S = J.fs_state[blockIdx.x];
        S.regen = sum; S.bad = bad ? 1u : 0u;
#pragma unroll
        for (int k = 0; k < 3; k++) { S.ms[k] = total.s[k]; S.mv[k] = total.v[k]; }
    }
}

__global__ void __launch_bounds__(32) k_fs_prefix(JobDev J) {
    if (threadIdx.x != 0) return;
    const FsBigFrame G = J.fs_big[blockIdx.x];
    if (J.frame_bad[G.frame]) return;
    const FrameDesc& F = J.frames[G.frame];
    uint64_t off = F.dst_off;
    uint32_t rep[3] = {1, 4, 8};
    bool bad = false;
    for (uint32_t t = G.first_tile; t < G.first_tile + G.n_tiles; t++) {
        FsTileState& S = J.fs_state[t];
        S.off_in = off; S.rep_in[0] = rep[0]; S.rep_in[1] = rep[1]; S.rep_in[2] = rep[2];
        RepMap m;
#pragma unroll
        for (int k = 0; k < 3; k++) { m.s[k] = S.ms[k]; m.v[k] = S.mv[k]; }
        uint32_t out[3];
        if (!rep_apply(m, rep, out) || S.bad) bad = true;
        rep[0] = out[0]; rep[1] = out[1]; rep[2] = out[2];
        off += S.regen;
    }
    if (off - F.dst_off != F.dst_size) bad = true;
    if (bad) flag_error(J, G.frame, zc::E_SIZE);
}

__global__ void __launch_bounds__(FSCAN_T) k_fs_apply(JobDev J) {
    const FsTile T = J.fs_tiles[blockIdx.x];
    if (J.frame_bad[T.frame]) return;
    const FsTileState& S = J.fs_state[blockIdx.x];
    uint64_t off = S.off_in;
    uint32_t rep[3] = {S.rep_in[0], S.rep_in[1], S.rep_in[2]};
    bool bad = false;
    RepMap unused; rep_identity(unused);
    fs_range<false>(J, T.first_block, T.first_block + T.n_blocks, off, rep, unused, bad);
    if (__syncthreads_or(bad) && threadIdx.x == 0) flag_error(J, T.frame, zc::E_SIZE);
}

// --------------------------------------------------------------------------------------------------------------
// k_huf_decode_small: one CTA per short Huffman bitstream, intra-stream parallel.
//
// A zstd Huffman stream is one serial bitstream of up to 32 Ki symbols, read backwards; with one thread per stream a
// 5 Mbp genome keeps ~80 lanes busy.  Here the stream is cut into HUF_T_SMALL equal bit ranges, one per thread.  A thread
// does not know where the first codeword of its range starts, but it must be one of the `max_bits` positions at the
// top of the range.  So it follows ALL candidates ("tracks") through its range: tracks that reach the same bit
// position merge (prefix codes usually resynchronise within a few symbols, so one track survives; near-fixed-length
// codes such as 4-bit packed uniform DNA never resynchronise and keep one track per phase, 4 of them).  The result is
// a transition map candidate -> (candidate of the next range, symbols decoded).  Composing the maps along the stream
// (a scan over function composition, maps packed as 4-bit fields of a u64) gives every thread its true start, exactly:
// thread 0 starts on the stream's first codeword.  Then: block-scan the symbol counts, decode once more from the true
// start into a shared-memory image of the output, flush with 16-byte stores.
//
// Shared memory: the common prefix (HufSmem) | output image (same 16 B phase as the destination) | compressed stream
// (16 B-aligned image of global memory, preceded by >= 16 zero bytes so reads below bit 0 see zeros).
constexpr int HUF_T_SMALL = 128;                  // four warps for short streams (1-stream blocks, tiny flushed blocks)
constexpr int HUF_SEG = 96;                       // tracks are compared for merging every HUF_SEG bits
constexpr int MAXC = zc::HUF_MAX_BITS;            // candidates per range

// The common prefix of the shared memory of every Huffman kernel; each kernel's own space follows it.
struct HufSmem {
    uint16_t t1[2048];                            // base table: index = next max_bits bits -> symbol << 8 | length
    uint8_t weights[256];
    uint16_t wcnt[128];                           // [8 symbol groups][16 weights]; after the table build: composed map of each warp
    uint32_t misc[64];                            // scan buffers, warp start candidates; [56..57] the mbarrier of the bulk copies
};
static_assert(sizeof(HufSmem) == 4864, "HufSmem: t1 4096 | weights 256 | wcnt 256 | misc 256");
// k_huf_decode_small: output image (phase 2) / boundary masks 8 KB + track queue 32 B per thread (phase 1)
constexpr uint32_t HUF_SMALL_SOUT = 8192u + 32u * HUF_T_SMALL + 64u;
constexpr uint32_t HUF_SMALL_FIXED = sizeof(HufSmem) + HUF_SMALL_SOUT;

constexpr int HUF_W = 12;                          // index width of the multi-symbol tables

// 64-bit register window over the stream image: {hi:lo} = stream bits [Q, Q+64), Q 32-aligned; rr = x - Q in [14, 46).
// (14, not 12: the byte offset of a 4-byte table entry, 4 * the next 12 bits, is then ONE funnel shift by rr - 14 and a mask.)
constexpr int WIN_MIN = HUF_W + 2;
struct Win {
    saddr_t waddr;      // shared address of the `lo` word
    uint32_t lo, hi;
    int rr;
};
__device__ __forceinline__ void win_init(Win& w, saddr_t comp, int x) {
    const int qi = (x - WIN_MIN) >> 5;
    w.waddr = comp + 4 * qi;
    w.lo = lds32(w.waddr);
    w.hi = lds32(w.waddr + 4);
    w.rr = x - (qi << 5);
}
// (rr - 14 is in [0, 32): a funnel shift takes its amount modulo 32, so the 12-bit and x2 forms are derived from this one)
__device__ __forceinline__ uint32_t win_peek_x4(const Win& w) { return __funnelshift_r(w.lo, w.hi, w.rr - WIN_MIN) & 0x3FFCu; }     // 4 * (next 12 bits)
__device__ __forceinline__ uint32_t win_peek_x2(const Win& w) { return win_peek_x4(w) >> 1; }
__device__ __forceinline__ uint32_t win_peek(const Win& w) { return win_peek_x4(w) >> 2; }
// The refill is PREDICATED, not branched: per lookup a lane needs it with p = 0.3, so some lane of a warp always does, and
// a branch costs the whole warp the body plus the divergence bookkeeping (ncu, round 1: 14 % of the kernel's instructions
// at 0.64 thread efficiency on this line).
__device__ __forceinline__ void win_consume(Win& w, int len) {
    w.rr -= len;
#if defined(__CUDA_ARCH__)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.s32 p, %3, 14;\n\t@p mov.b32 %1, %0;\n\t@p sub.u32 %2, %2, 4;\n\t@p ld.shared.u32 %0, [%2];\n\t@p add.s32 %3, %3, 32;\n\t}"
                 : "+r"(w.lo), "+r"(w.hi), "+r"(w.waddr), "+r"(w.rr));
#else
    if (w.rr < WIN_MIN) { w.hi = w.lo; w.waddr -= 4; w.lo = lds32(w.waddr); w.rr += 32; }
#endif
}

// Follows one track from q (bits below the top of the stream) to the FIRST codeword boundary >= lim, counting symbols.
// bm: boundary-mask table, index = next 12 bits, bit j set <=> j+1 bits is a cumulative length of whole codewords.
__device__ __forceinline__ int msb_index(uint32_t m) {            // position of the highest set bit (m != 0): one BFIND
#if defined(__CUDA_ARCH__)
    int r; asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(m)); return r;
#else
    return 31 - __clz((int)m);
#endif
}

__device__ __forceinline__ void track_advance(saddr_t comp, saddr_t bm, int xtop, int& q, int& cnt, int lim) {
    int rem = lim - q;
    if (rem <= 0) return;
    Win w;
    win_init(w, comp, xtop - q);
    // steady state: whole windows, no test against the limit (every window holds >= 1 whole codeword: max_bits <= 11)
    while (rem > HUF_W) {
        const uint32_t m = lds16(bm + win_peek_x2(w));
        const int used = msb_index(m) + 1;
        cnt += __popc(m);
        rem -= used;
        win_consume(w, used);
    }
    // the last windows: stop at the first boundary at or past the limit
    while (rem > 0) {
        const uint32_t m = lds16(bm + win_peek_x2(w));
        const uint32_t t = m >> (rem - 1);
        if (t) {
            const int j = __ffs((int)t) - 1 + rem - 1;
            cnt += __popc(m & ((2u << j) - 1u));
            rem -= j + 1;
            break;
        }
        const int used = msb_index(m) + 1;
        cnt += __popc(m);
        rem -= used;
        win_consume(w, used);
    }
    q = lim - rem;
}

// Write pass of k_huf_decode_small: decodes from q to the first boundary >= lim, storing symbols at out.. (shared address).
// Returns the count.  t1: index = next max_bits bits, entry = symbol << 8 | length
__device__ __forceinline__ int track_write(saddr_t comp, saddr_t t1, int maxbits, int xtop, int q, int lim, saddr_t out) {
    int rem = lim - q;
    if (rem <= 0) return 0;
    Win w;
    win_init(w, comp, xtop - q);
    int cnt = 0;
    const int sh1 = HUF_W - maxbits;
    while (rem > 0) {
        const uint32_t e = lds16(t1 + 2 * (win_peek(w) >> sh1));
        const int len = (int)(e & 0xFFu);
        sts8(out + cnt, e >> 8);
        cnt++;
        rem -= len;
        win_consume(w, len);
    }
    return cnt;
}

// Warp-cooperative copy of n bytes from shared memory (any alignment) to global memory: destination-aligned 16-byte
// stores, each assembled from five shared-memory words with funnel shifts; ragged ends go byte-wise.
// The shared buffer must be readable 20 bytes past the last source byte.
__device__ __forceinline__ void warp_copy_s2g(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, int lane) {
    if (n < 48) { for (uint32_t k = lane; k < n; k += 32) dst[k] = src[k]; return; }
    const uint32_t h = (uint32_t)(-(intptr_t)dst) & 15u;
    if ((uint32_t)lane < h) dst[lane] = src[lane];
    const uint32_t body = (n - h) >> 4;
    const uintptr_t sa = (uintptr_t)(src + h);
    const uint32_t* sw = (const uint32_t*)(sa & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(sa & 3) * 8;
    uint4* d4 = (uint4*)(dst + h);
    for (uint32_t c = lane; c < body; c += 32) {
        const uint32_t* p = sw + 4 * c;
        const uint32_t w0 = p[0], w1 = p[1], w2 = p[2], w3 = p[3], w4 = p[4];
        d4[c] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
    }
    const uint32_t done = h + (body << 4);
    for (uint32_t k = done + lane; k < n; k += 32) dst[k] = src[k];
}

// maps over candidate indices 0..15 packed as 4-bit fields; compose(g, f)(k) = g(f(k))
__device__ __forceinline__ uint64_t map_compose(uint64_t g, uint64_t f) {
    uint64_t r = 0;
#pragma unroll
    for (int k = 0; k < MAXC; k++) {
        uint32_t fk = (uint32_t)(f >> (4 * k)) & 15u;
        r |= ((g >> (4 * fk)) & 15ull) << (4 * k);
    }
    return r;
}
constexpr uint64_t MAP_IDENTITY = 0xFEDCBA9876543210ull;

// Entries [lo, hi) of the tables over 12-bit windows, from the finished base table: decode the window while whole
// codewords fit (no barrier inside; the caller separates it from the base-table build and from the first use).
//   bm (optional): boundary masks, bit j set <=> j+1 bits is a cumulative length of whole codewords
//   t3 (MULTI): 3-symbol write table, entry = sym1 | sym2 << 8 | sym3 << 16 | total length << 24 | n << 28
//   tc (optional): count table, entry = bits of all whole codewords | their number << 4 (both <= 12)
template <int HUF_T, bool MULTI>
__device__ __forceinline__ void huf_build_wide(const uint16_t* table, int maxbits, uint16_t* bm, uint32_t* t3, uint32_t lo, uint32_t hi,
                                               uint8_t* tc = nullptr) {
    const int sh1 = HUF_W - maxbits;
    for (uint32_t i = lo + threadIdx.x; i < hi; i += HUF_T) {
        uint32_t used = 0, n = 0, syms = 0, used3 = 0, mask = 0;
        for (;;) {
            const uint32_t e = table[((i << used) & 0xFFFu) >> sh1];
            const uint32_t len = e & 0xFFu;
            if (used + len > (uint32_t)HUF_W) break;
            if (n < 3) { syms |= (e >> 8) << (8 * n); used3 = used + len; n++; }
            used += len;
            mask |= 1u << (used - 1);
            if (used == (uint32_t)HUF_W) break;
        }
        if (bm) bm[i] = (uint16_t)mask;
        if (MULTI) t3[i] = syms | (used3 << 24) | (n << 28);
        if (tc) tc[i] = (uint8_t)(used | ((uint32_t)__popc(mask) << 4));
    }
}

// Builds the base table of one Huffman tree in shared memory (all HUF_T threads of the CTA must call):
//   table: index = next max_bits bits -> symbol << 8 | length (RFC 8878 4.2.1: ascending weight, then symbol)
template <int HUF_T>
__device__ __forceinline__ void huf_build_t1(const uint8_t* weights, int nsym, int maxbits, uint16_t* table, uint16_t* wcnt) {
    const int tid = threadIdx.x, lane = tid & 31;
    // symbols are handled in 8 groups of 32 (group g = symbols 32g..32g+31); wcnt[g][w] = symbols of weight w in group g
    constexpr int GROUPS_PER_PASS = HUF_T >= 256 ? 8 : HUF_T / 32;
    int wreg[8 / GROUPS_PER_PASS], rankreg[8 / GROUPS_PER_PASS];
#pragma unroll
    for (int p = 0; p < 8 / GROUPS_PER_PASS; p++) {
        wreg[p] = 0; rankreg[p] = 0;
        if (tid < 32 * GROUPS_PER_PASS) {
            const int sym = p * 32 * GROUPS_PER_PASS + tid, grp = sym >> 5;
            const int w = sym < nsym ? weights[sym] : 0;
            wreg[p] = w;
            for (int wv = 1; wv <= zc::HUF_MAX_BITS; wv++) {
                uint32_t bal = __ballot_sync(0xFFFFFFFFu, w == wv);
                if (lane == 0) wcnt[grp * 16 + wv] = (uint16_t)__popc(bal);
                if (w == wv) rankreg[p] = __popc(bal & ((1u << lane) - 1u));
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 8 / GROUPS_PER_PASS; p++) {
        const int w = wreg[p];
        if (tid < 32 * GROUPS_PER_PASS && w > 0) {
            const int sym = p * 32 * GROUPS_PER_PASS + tid, grp = sym >> 5;
            uint32_t start = 0;
            for (int wv = 1; wv < w; wv++) {
                uint32_t c = 0;
                for (int k = 0; k < 8; k++) c += wcnt[k * 16 + wv];
                start += c << (wv - 1);
            }
            int rank = rankreg[p];
            for (int k = 0; k < grp; k++) rank += wcnt[k * 16 + w];
            uint32_t pos = start + ((uint32_t)rank << (w - 1)), n = 1u << (w - 1);
            uint16_t e = (uint16_t)((sym << 8) | (maxbits + 1 - w));
            if (n >= 8) {                                        // groups start on multiples of their size: 16-byte stores
                const uint32_t e2 = (uint32_t)e | ((uint32_t)e << 16);
                const uint4 v = make_uint4(e2, e2, e2, e2);
                for (uint32_t i = 0; i < n; i += 8) *(uint4*)(table + pos + i) = v;
            } else {
                for (uint32_t i = 0; i < n; i++) table[pos + i] = e;
            }
        }
    }
    __syncthreads();
}

// The tree of a block: its 256 weights to shared memory (NT threads), and its symbol count and max_bits (0: a bad tree, already
// flagged by k_build_tables)
struct HufTree { int nsym, maxbits; };
template <int NT>
__device__ __forceinline__ HufTree huf_tree(const JobDev& J, const BlockDesc& B, uint8_t* weights) {
    for (int i = threadIdx.x; i < 64; i += NT) ((uint32_t*)weights)[i] = ((const uint32_t*)(J.huf_weights + (size_t)B.huf_slot * 256))[i];
    return {(int)J.huf_meta[(size_t)B.huf_slot * 2] + 1, (int)J.huf_meta[(size_t)B.huf_slot * 2 + 1]};
}

// Geometry of a staged stream.  `img`: 16 zero bytes, then the 16 B-aligned image of global memory (the stream at 16 + a).
// q = distance (in bits) from the top of the stream; smem bit position x = XTOP - q.  The stream is cut into `nranges` ranges
// of S bits; k_huf_scout finds the starts of k_huf_decode_block's ranges, so the two must take S from here.
struct HufShape { uint32_t last; int P0, XTOP, S; };
__device__ __forceinline__ HufShape huf_stream_shape(const uint8_t* img, uint32_t a, uint32_t src_size, int nranges) {
    const uint32_t last = img[16 + a + src_size - 1];                   // (0: the caller refuses the stream before using the rest)
    const int P0 = 8 * (int)(src_size - 1) + zc::highbit32(last);
    int S = (P0 + nranges - 1) / nranges;
    if (S < 2 * MAXC) S = 2 * MAXC;
    return {last, P0, (int)(16 + a) * 8 + P0, S};
}

// Flush of the output image by NT threads: sout[a2 + k] -> dst[k] for k < n, where a2 = dst & 15; aligned 16 B chunks in the
// middle, bytes at the ragged ends
template <int NT>
__device__ __forceinline__ void flush_image(uint8_t* dst, const uint8_t* sout, uint32_t a2, uint32_t n) {
    const int tid = threadIdx.x;
    const uint32_t endb = a2 + n;
    uint8_t* dal = dst - a2;
    const uint32_t first_full = a2 ? 1u : 0u, last_full = endb >> 4;     // chunks [first_full, last_full) are complete
    for (uint32_t c = first_full + tid; c < last_full; c += NT) ((uint4*)dal)[c] = ((const uint4*)sout)[c];
    if (a2) { uint32_t hend = endb < 16 ? endb : 16; for (uint32_t k = a2 + tid; k < hend; k += NT) dal[k] = sout[k]; }
    if (last_full >= first_full && (last_full << 4) < endb && !(a2 && last_full == 0))
        for (uint32_t k = (last_full << 4) + tid; k < endb; k += NT) dal[k] = sout[k];
}

__global__ void __launch_bounds__(HUF_T_SMALL, 4) k_huf_decode_small(JobDev J, const HufItem* items) {
    NAF_DYN_SMEM(unsigned char, smem);
    constexpr int NWARPS = HUF_T_SMALL / 32;
    HufSmem& sm = *(HufSmem*)smem;
    uint16_t* table = sm.t1;
    uint16_t* wcnt = sm.wcnt;
    uint32_t* misc = sm.misc;                                           // [0..32] count scan, [34..49] warp start candidates
    uint64_t* wmap = (uint64_t*)sm.wcnt;                                // [NWARPS] composed map of each warp
    uint8_t* sout = smem + sizeof(HufSmem);                             // output image (phase 2, flush)
    uint16_t* bm = (uint16_t*)sout;                                     // boundary masks of 12-bit windows (phase 1): same space
    uint32_t* scomp = (uint32_t*)(smem + HUF_SMALL_FIXED);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const HufItem it = items[blockIdx.x];
    const BlockDesc& B = J.blocks[it.block];
    if (J.frame_bad[B.frame]) return;
    // ---- stage the compressed stream (coalesced 16 B loads of the aligned image) and the weights -------------------
    const uint8_t* g = J.comp + B.src_off + it.src_off;
    const uint32_t a = (uint32_t)((uintptr_t)g & 15);
    const uint4* gbase = (const uint4*)(g - a);
    const uint32_t nchunks = (a + it.src_size + 15) >> 4;
    for (uint32_t c = tid; c < nchunks; c += HUF_T_SMALL) ((uint4*)scomp)[1 + c] = gbase[c];
    const HufTree tree = huf_tree<HUF_T_SMALL>(J, B, sm.weights);
    const int maxbits = tree.maxbits;
    if (maxbits == 0) return;                                           // bad tree: already flagged by k_build_tables
    __syncthreads();
    if ((uint32_t)tid < 16 + a) ((uint8_t*)scomp)[tid] = 0;              // bits below the stream start read as zero
    huf_build_t1<HUF_T_SMALL>(sm.weights, tree.nsym, maxbits, table, wcnt);
    huf_build_wide<HUF_T_SMALL, false>(table, maxbits, bm, nullptr, 0u, 1u << HUF_W);
    __syncthreads();

    // ---- phase 1: transition map of every range -------------------------------------------------------------------------
    const HufShape shape = huf_stream_shape((const uint8_t*)scomp, a, it.src_size, HUF_T_SMALL);
    if (shape.last == 0) { if (tid == 0) flag_error(J, B.frame, zc::E_HUF_STREAM); return; }
    const int P0 = shape.P0, XTOP = shape.XTOP, S = shape.S;
    const int q0 = tid * S;                                             // top of this thread's range
    const int qe = (q0 + S < P0) ? q0 + S : P0;                         // end of the range (exclusive)
    const bool active = q0 < P0;
    // track k: pc[k] = (q - q0) | (symbols << 16); merged tracks: mg[k] = (count offset & 0xFFFF) | (representative << 16)
    uint32_t pc[MAXC], mg[MAXC];
    uint32_t live = active ? ((1u << maxbits) - 1u) : 0u;
#pragma unroll
    for (int k = 0; k < MAXC; k++) { pc[k] = (uint32_t)k; mg[k] = 0; }
    const saddr_t s_comp = to_saddr(scomp), s_bm = to_saddr(bm);
    // Merge of tracks that reached the same position (the representative always has the lower index).
    auto dedupe = [&]() {
        if (!(live & (live - 1))) return;
#pragma unroll
        for (int k = 1; k < MAXC; k++) {
            if (live & (1u << k)) {
#pragma unroll
                for (int j = 0; j < k; j++) {
                    if ((live & (1u << j)) && (live & (1u << k)) && ((pc[j] ^ pc[k]) & 0xFFFFu) == 0) {
                        live &= ~(1u << k);
                        mg[k] = (((pc[k] >> 16) - (pc[j] >> 16)) & 0xFFFFu) | ((uint32_t)j << 16);
                    }
                }
            }
        }
    };
    // (1) first stop right below the candidate window: one boundary-mask lookup per candidate lands every track on its
    //     first codeword boundary >= q0 + 12; candidates on the same codeword chain coincide there and merge.
    if (active) {
        const int l = (q0 + HUF_W < qe) ? q0 + HUF_W : qe;
#pragma unroll
        for (int k = 0; k < MAXC; k++) {
            if (live & (1u << k)) {
                int q = q0 + k, c = 0;
                track_advance(s_comp, s_bm, XTOP, q, c, l);
                pc[k] = (uint32_t)(q - q0) | ((uint32_t)c << 16);
            }
        }
        dedupe();
    }
    // (2) the surviving tracks of ALL ranges (1 per range for codes that resynchronise, up to one per phase otherwise)
    //     become work items in a shared-memory queue and are spread evenly over the CTA: following tracks thread-by-
    //     thread leaves lanes with fewer survivors idle (45 % thread efficiency measured); the queue keeps every lane on
    //     one track of equal length.  Two legs: to 96 bits past the first stop (twins merge), then to the range end.
    constexpr int HUF_QCAP = 4 * HUF_T_SMALL;
    uint32_t* q_owner = (uint32_t*)(sout + 8192);                        // [HUF_QCAP] owner thread | track << 16 (after the boundary masks)
    uint32_t* q_pc = q_owner + HUF_QCAP;                                 // [HUF_QCAP] position | symbols << 16
    for (int leg = 0; leg < 2; leg++) {
        uint32_t l4 = 0;                                                 // up to four lowest live tracks go to the queue
        { uint32_t t = live; for (int i = 0; i < 4 && t; i++) { l4 |= t & (0u - t); t &= t - 1; } }
        const uint32_t n_mine = (uint32_t)__popc(l4);
        uint32_t inc = n_mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
        if (lane == 31) misc[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint32_t x = lane < NWARPS ? misc[lane] : 0, o = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, d); if (lane >= d) x += t; }
            misc[lane] = x - o;
            if (lane == 31) misc[32] = x;
        }
        __syncthreads();
        const uint32_t qbase = inc - n_mine + misc[warp], qtotal = misc[32];
        {
            uint32_t idx = qbase;
#pragma unroll
            for (int k = 0; k < MAXC; k++) if (l4 & (1u << k)) { q_owner[idx] = (uint32_t)tid | ((uint32_t)k << 16); q_pc[idx] = pc[k]; idx++; }
        }
        __syncthreads();
        for (uint32_t i = tid; i < qtotal; i += HUF_T_SMALL) {
            const int ot = (int)(q_owner[i] & 0xFFFFu);
            const int oq0 = ot * S, oqe = (oq0 + S < P0) ? oq0 + S : P0;
            const int mid = oq0 + HUF_W + HUF_SEG;
            const int lim = (leg == 0 && mid < oqe) ? mid : oqe;
            const uint32_t p = q_pc[i];
            int q = oq0 + (int)(p & 0xFFFFu), c = (int)(p >> 16);
            track_advance(s_comp, s_bm, XTOP, q, c, lim);
            q_pc[i] = (uint32_t)(q - oq0) | ((uint32_t)c << 16);
        }
        __syncthreads();
        {
            uint32_t idx = qbase;
#pragma unroll
            for (int k = 0; k < MAXC; k++) if (l4 & (1u << k)) { pc[k] = q_pc[idx]; idx++; }
        }
        {
            const int mid = q0 + HUF_W + HUF_SEG;
            const int lim = (leg == 0 && mid < qe) ? mid : qe;
            for (uint32_t m = live & ~l4; m; m &= m - 1) {               // more than four survivors (rare): the owner follows them
                const int kk = __ffs((int)m) - 1;
                int q = 0, c = 0;
#pragma unroll
                for (int k = 0; k < MAXC; k++) if (k == kk) { q = q0 + (int)(pc[k] & 0xFFFFu); c = (int)(pc[k] >> 16); }
                track_advance(s_comp, s_bm, XTOP, q, c, lim);
#pragma unroll
                for (int k = 0; k < MAXC; k++) if (k == kk) pc[k] = (uint32_t)(q - q0) | ((uint32_t)c << 16);
            }
        }
        dedupe();
        __syncthreads();                                                 // the queue is rewritten by the next leg
    }
    // resolve merged tracks (representatives always have a lower index): landing position and symbol count per candidate
    uint64_t fmap = MAP_IDENTITY;
    if (active) {
        fmap = 0;
#pragma unroll
        for (int k = 0; k < MAXC; k++) {
            if (!(live & (1u << k)) && k < maxbits) {
                const uint32_t j = mg[k] >> 16;
                uint32_t pj = 0;
#pragma unroll
                for (int t = 0; t < k; t++) if ((uint32_t)t == j) pj = pc[t];
                pc[k] = (pj & 0xFFFFu) | ((((pj >> 16) + mg[k]) & 0xFFFFu) << 16);
            }
            int land = (int)(pc[k] & 0xFFFFu) - S;                      // candidate index in the next range
            if (land < 0 || land > 15) land = 15;                       // only garbage tracks or the last range get here
            fmap |= (uint64_t)land << (4 * k);
        }
    }
    // ---- compose the maps along the stream: inclusive scan in the warp, then warp totals serially ------------------------
    uint64_t inc_map = fmap;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t o = __shfl_up_sync(0xFFFFFFFFu, inc_map, d);
        if (lane >= d) inc_map = map_compose(inc_map, o);
    }
    uint64_t exc_map = __shfl_up_sync(0xFFFFFFFFu, inc_map, 1);
    if (lane == 0) exc_map = MAP_IDENTITY;
    if (lane == 31) wmap[warp] = inc_map;
    __syncthreads();
    if (tid == 0) {
        uint32_t k = 0;
        for (int w = 0; w < NWARPS; w++) { misc[34 + w] = k; k = (uint32_t)(wmap[w] >> (4 * k)) & 15u; }
    }
    __syncthreads();
    const uint32_t kw = misc[34 + warp];
    const uint32_t ktrue = (uint32_t)(exc_map >> (4 * kw)) & 15u;      // this thread's true candidate
    uint32_t mypc = 0;
#pragma unroll
    for (int k = 0; k < MAXC; k++) if ((uint32_t)k == ktrue) mypc = pc[k];
    const uint32_t mycnt = active && ktrue < (uint32_t)maxbits ? (mypc >> 16) : 0u;
    const int myland = q0 + (int)(mypc & 0xFFFFu);
    // the stream must end exactly on its first bit: the last active range's true track lands on P0
    const bool bad_end = active && qe == P0 && (ktrue >= (uint32_t)maxbits || myland != P0);
    // ---- count, scan, write ------------------------------------------------------------------------------------------
    uint32_t inc = mycnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) misc[warp] = inc;
    const int any_bad = __syncthreads_or(bad_end);
    if (warp == 0) {
        uint32_t x = lane < NWARPS ? misc[lane] : 0, o = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, d); if (lane >= d) x += t; }
        misc[lane] = x - o;
        if (lane == 31) misc[32] = x;
    }
    __syncthreads();
    const uint32_t off = inc - mycnt + misc[warp];
    const uint32_t total = misc[32];
    if (any_bad || total != it.n_sym) { if (tid == 0) flag_error(J, B.frame, zc::E_HUF_STREAM); return; }
    // destination: the block's slot in the literal staging buffer (k_lz_literals places the runs; the Huffman branch of
    // the stage does not depend on the FSE branch, so the two run on different streams)
    uint8_t* dst = J.lit + B.lit_base + it.dst_off;
    const uint32_t a2 = (uint32_t)((uintptr_t)dst & 15);
    if (mycnt) track_write(s_comp, to_saddr(table), maxbits, XTOP, q0 + (int)ktrue, qe, to_saddr(sout) + a2 + off);
    __syncthreads();
    flush_image<HUF_T_SMALL>(dst, sout, a2, it.n_sym);
}

// --------------------------------------------------------------------------------------------------------------
// k_huf_decode_big: the streams of 4-stream blocks (up to 32 Ki symbols each), one CTA of 256 threads per stream, the four
// CTAs of a block launched as ONE THREAD-BLOCK CLUSTER.
//
//   * The compressed stream is staged with ONE bulk asynchronous copy (cp.async.bulk global -> shared, completion on an
//     mbarrier) issued by a single thread; the other threads build the decode tables meanwhile.
//   * The four streams of a block share a Huffman tree: every CTA builds the small base table itself and ONE QUARTER of the
//     two tables over 12-bit windows (boundary masks, 3-symbol write table), then fetches the other three quarters from its
//     cluster peers through distributed shared memory.  Round 1 built them once per tree in a separate kernel and every stream
//     CTA copied 28 KB back from global memory (+ 175 MB of DRAM reads per 256-archive step, + one launch).
//   * Intra-stream parallelism as in k_huf_decode (candidate tracks, transition maps, composition), restructured around what
//     ncu showed (profiles/r1_huf_decode512_batch256.txt: 40 thread-instructions per table lookup, most of them bookkeeping):
//       - 256 ranges per stream instead of 512: the price of not knowing where a range starts is ~1000 bit-steps of
//         speculation PER RANGE whatever its length (measured on cfg2: 3.7 tracks alive 12 bits into a range, 2.0 at 108,
//         1.4 at 256, 1.2 at 512), and every per-range fixed cost halves;
//       - the live tracks of a range at a checkpoint are a BITMASK of landing offsets (a track lands on the first codeword
//         boundary at or past the checkpoint, at most max_bits - 1 further): merging tracks is an OR, not 55 compares;
//       - what a track did on a leg (landing offset, symbols) goes to a small shared-memory table indexed by (leg, range,
//         offset); the per-candidate results are recovered by walking three entries, only for what is needed;
//       - all tracks of all ranges on a leg are work items dealt out evenly over the CTA (as before);
//       - composing the transition maps: a map that sends every candidate to the same offset (all tracks merged: nearly every
//         range) absorbs whatever comes before it, so the shuffle scan skips the 11-nibble gather when no lane needs it;
//       - the window refill is predicated; the write pass assembles 4-byte words in registers (one store per four symbols
//         instead of four byte stores: the pass was bound by shared-memory bank conflicts, not by issue slots).
constexpr int HB_T = 256;
constexpr int HB_NW = HB_T / 32;
#if defined(NAFGPU_EMULATE)
constexpr int HB_CL = 1;                            // the emulator runs one CTA at a time: every CTA builds whole tables
#define HB_CLUSTER_ATTR
#else
constexpr int HB_CL = 4;
#define HB_CLUSTER_ATTR __cluster_dims__(4, 1, 1)
#endif
constexpr int HB_NLEG = 3;
constexpr int HB_CK0 = 12, HB_CK1 = 108, HB_CK2 = 320;      // checkpoints (bits below the top of a range) where tracks are compared
constexpr uint32_t HB_SOUT = 32768u + 64u;                  // output image (phase 2); phase 1: boundary masks | leg tables | work queue
constexpr uint32_t HB_BM_BYTES = 8192u, HB_LEG_BYTES = HB_NLEG * HB_T * MAXC * 2u, HB_Q_BYTES = HB_T * MAXC * 2u;
static_assert(HB_BM_BYTES + HB_LEG_BYTES + HB_Q_BYTES <= HB_SOUT, "phase-1 scratch must fit the output image");
// shared memory of k_huf_decode_big and k_huf_decode_block: HufSmem | t3 | output image | compressed stream image
constexpr uint32_t HB_T3_AT = sizeof(HufSmem), HB_SOUT_AT = HB_T3_AT + 4u * (1u << HUF_W), HB_FIXED = HB_SOUT_AT + HB_SOUT;
__host__ __device__ constexpr uint32_t hb_smem_bytes(uint32_t max_stream) { return HB_FIXED + ((max_stream + 15u + 16u + 16u + 15u) & ~15u); }

// Exclusive prefix sum of one small value per thread over the CTA (HB_T threads); *total gets the sum.  One barrier; `buf`
// (HB_NW words) must not be reused before another barrier.
__device__ __forceinline__ uint32_t hb_scan(uint32_t v, uint32_t* buf, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) buf[warp] = inc;
    __syncthreads();
    uint32_t before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < HB_NW; w++) { const uint32_t x = buf[w]; all += x; if (w < warp) before += x; }
    *total = all;
    return before + inc - v;
}

__device__ __forceinline__ bool map_is_const(uint64_t m, int maxbits) {        // every candidate < maxbits goes to the same offset
    const uint64_t lowmask = maxbits >= 16 ? ~0ull : ((1ull << (4 * maxbits)) - 1ull);
    const uint64_t rep = (m & 15ull) * 0x1111111111111111ull;
    return ((m ^ rep) & lowmask) == 0;
}

// Staging of the compressed streams: bulk asynchronous copies (cp.async.bulk global -> shared) that complete on an mbarrier.
// The emulator has no asynchronous copy: stage_stream copies synchronously, and the mbarrier calls do nothing.
__device__ __forceinline__ void mbar_init(saddr_t mbar, uint32_t count) {     // one thread, before anyone arrives
#if defined(__CUDA_ARCH__)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(mbar), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
}
// One thread: `bytes` (a multiple of 16) from src (16 B aligned) to dst, in one copy
__device__ __forceinline__ void stage_stream(void* dst, const uint8_t* src, uint32_t bytes, saddr_t mbar) {
#if defined(__CUDA_ARCH__)
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(to_saddr(dst)), "l"(src), "r"(bytes), "r"(mbar) : "memory");
#else
    for (uint32_t c = 0; c < (bytes >> 4); c++) ((uint4*)dst)[c] = ((const uint4*)src)[c];
#endif
}
// Waits for phase `parity` of the mbarrier.  Every thread waits, also before an early exit: the shared memory must not be handed
// to another CTA under a copy.
__device__ __forceinline__ void mbar_wait(saddr_t mbar, uint32_t parity) {
#if defined(__CUDA_ARCH__)
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
    } while (!done);
#endif
}

// A tree whose codes all have the same length (e.g. 16 equiprobable byte values) never lets tracks merge -- and does not need
// to: the codeword boundaries are the multiples of that length.  One barrier: the whole CTA calls.
__device__ __forceinline__ bool huf_fixed_length(const uint16_t* wcnt) {
    const int tid = threadIdx.x;
    return !__syncthreads_or(tid < 128 && (tid & 15) >= 2 && (tid & 15) <= zc::HUF_MAX_BITS && wcnt[tid] != 0);
}

// First stop of phase 1: every candidate start q0 + k (k < max_bits) lands on its first codeword boundary at or past l0, so
// candidates of the same codeword chain land together.  `count(q, c, lim)` follows one track.  Out: first / fcnt = candidate ->
// landing offset (q - l0) / symbols so far (4 bits each; candidates that cannot occur: dead, 15); live |= landing offsets.
template <class Count>
__device__ __forceinline__ void hb_first_stop(int q0, int l0, int maxbits, bool fixed_len, Count count, uint64_t& first, uint64_t& fcnt,
                                              uint32_t& live) {
    first = 0;
    if (fixed_len) {
        int q = q0 + (maxbits - q0 % maxbits) % maxbits, c = 0;         // the one candidate that is a boundary; the others follow it
        count(q, c, l0);
        first = (uint64_t)(uint32_t)(q - l0) * 0x1111111111111111ull;
        fcnt = (uint64_t)(uint32_t)c * 0x1111111111111111ull;
        live = 1u << (q - l0);
    } else {
        for (int k = 0; k < maxbits; k++) {
            int q = q0 + k, c = 0;
            count(q, c, l0);
            const uint32_t o = (uint32_t)(q - l0);
            first |= (uint64_t)o << (4 * k);
            fcnt |= (uint64_t)c << (4 * k);
            live |= 1u << o;
        }
    }
    if (maxbits < 16) first |= ~0ull << (4 * maxbits);
}

// Composes the transition maps along each stream of WPS consecutive warps: inclusive scan in the warp, then the stream's warp
// totals serially; returns this thread's true candidate.  inc_map(lane) = f_lane o ... o f_(lane - 2^d + 1); a constant map
// absorbs everything before it, and after the first step nearly every lane holds one: the gather runs only when some lane of
// the warp still needs it.  wmap, kw: one entry per warp.  Two barriers: all HB_T threads call.
template <int WPS>
__device__ __forceinline__ uint32_t hb_compose(uint64_t fmap, int maxbits, uint64_t* wmap, uint32_t* kw) {
    static_assert(HB_NW % WPS == 0, "hb_compose: whole streams");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint64_t inc_map = fmap;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t o = __shfl_up_sync(0xFFFFFFFFu, inc_map, d);
        const bool need = lane >= d && !map_is_const(inc_map, maxbits);
        if (__any_sync(0xFFFFFFFFu, need)) { if (need) inc_map = map_compose(inc_map, o); }
    }
    uint64_t exc_map = __shfl_up_sync(0xFFFFFFFFu, inc_map, 1);
    if (lane == 0) exc_map = MAP_IDENTITY;
    if (lane == 31) wmap[warp] = inc_map;
    __syncthreads();
    if (tid < HB_NW / WPS) {
        uint32_t k = 0;
        for (int w = tid * WPS; w < (tid + 1) * WPS; w++) { kw[w] = k; k = (uint32_t)(wmap[w] >> (4 * k)) & 15u; }
    }
    __syncthreads();
    return (uint32_t)(exc_map >> (4 * kw[warp])) & 15u;
}

// Write pass of one range: from q (bits below the top of the stream) to the first boundary at or past qe, the symbols to `out`
// on (shared address).  Bytes go out as aligned 4-byte words assembled in a register pair; the ragged head and tail (words
// shared with the neighbouring ranges) as bytes.
__device__ __forceinline__ void hb_write_range(saddr_t comp, saddr_t t3, saddr_t t1, int maxbits, int xtop, int q, int qe, saddr_t out) {
    int rem = qe - q;
    Win w;
    win_init(w, comp, xtop - q);
    const int sh1 = HUF_W - maxbits;
    while ((out & 3u) && rem > 0) {                                     // head: single symbols up to a word boundary
        const uint32_t e = lds16(t1 + 2 * (win_peek(w) >> sh1));
        sts8(out, e >> 8); out++;
        rem -= (int)(e & 0xFFu);
        win_consume(w, (int)(e & 0xFFu));
    }
    uint32_t acc_lo = 0, acc_hi = 0;
    int pc = 0;                                                         // bytes waiting in acc
    while (rem > HUF_W) {
        const uint32_t e = lds32(t3 + win_peek_x4(w));
        const int n = (int)(e >> 28), len = (int)(e >> 24) & 15;
        const uint32_t sy = e & 0xFFFFFFu;
        acc_lo |= sy << (8 * pc);
        acc_hi |= __funnelshift_l(sy, 0u, 8 * pc);                      // the bits that fall off the top of acc_lo
        pc += n;
        if (pc >= 4) { sts32(out, acc_lo); out += 4; acc_lo = acc_hi; acc_hi = 0; pc -= 4; }
        rem -= len;
        win_consume(w, len);
    }
    while (rem > 0) {                                                   // the last symbols, one at a time
        const uint32_t e = lds16(t1 + 2 * (win_peek(w) >> sh1));
        acc_lo |= (e >> 8) << (8 * pc);
        pc++;
        if (pc == 4) { sts32(out, acc_lo); out += 4; acc_lo = 0; pc = 0; }
        rem -= (int)(e & 0xFFu);
        win_consume(w, (int)(e & 0xFFu));
    }
    for (int k = 0; k < pc; k++) sts8(out + k, acc_lo >> (8 * k));
}

__global__ void HB_CLUSTER_ATTR __launch_bounds__(HB_T, 3) k_huf_decode_big(JobDev J) {
    NAF_DYN_SMEM(unsigned char, smem);
    HufSmem& sm = *(HufSmem*)smem;
    uint16_t* t1 = sm.t1;
    uint32_t* misc = sm.misc;                                           // [0..15] two scan buffers, [16..23] warp start candidates, [56..57] mbarrier
    uint32_t* t3 = (uint32_t*)(smem + HB_T3_AT);
    uint8_t* sout = smem + HB_SOUT_AT;
    uint16_t* bm = (uint16_t*)sout;
    uint16_t* legtab = (uint16_t*)(sout + HB_BM_BYTES);                 // [leg][range][offset] = landing offset | symbols << 4
    uint16_t* qitems = (uint16_t*)(sout + HB_BM_BYTES + HB_LEG_BYTES);  // range | offset << 8
    uint32_t* scomp = (uint32_t*)(smem + HB_FIXED);
    const int tid = threadIdx.x;

    const HufItem it = J.huf_items[blockIdx.x];
    const BlockDesc& B = J.blocks[it.block];
    // ---- stage the stream: the 16 B-aligned image of global memory, behind 16 bytes that stay zero --------------------------
    const uint8_t* g = J.comp + B.src_off + it.src_off;
    const uint32_t a = (uint32_t)((uintptr_t)g & 15);
    const saddr_t mbar = to_saddr(&misc[56]);
    if (tid == 0) { mbar_init(mbar, 1); stage_stream(scomp + 4, g - a, ((a + it.src_size + 15u) >> 4) << 4, mbar); }
    const HufTree tree = huf_tree<HB_T>(J, B, sm.weights);
    const int maxbits = tree.maxbits;
    __syncthreads();
    // a bad tree (flagged by k_build_tables) is the same for the whole cluster: nobody builds, nobody waits for a peer
    if (maxbits != 0) {
        huf_build_t1<HB_T>(sm.weights, tree.nsym, maxbits, t1, sm.wcnt);
#if defined(__CUDA_ARCH__)
        namespace cg = cooperative_groups;
        cg::cluster_group cluster = cg::this_cluster();
        const uint32_t rank = cluster.block_rank();
        constexpr uint32_t QUARTER = (1u << HUF_W) / HB_CL;
        huf_build_wide<HB_T, true>(t1, maxbits, bm, t3, rank * QUARTER, (rank + 1) * QUARTER);
        cluster.sync();
        // the other quarters, from the peers' shared memory (DSMEM): 2 KB of boundary masks + 4 KB of write table each
        constexpr uint32_t BM16 = QUARTER * 2 / 16, T316 = QUARTER * 4 / 16;
        for (uint32_t i = tid; i < (HB_CL - 1) * (BM16 + T316); i += HB_T) {
            const uint32_t r = (rank + 1 + i / (BM16 + T316)) % HB_CL, j = i % (BM16 + T316);
            if (j < BM16) ((uint4*)bm)[r * BM16 + j] = ((const uint4*)cluster.map_shared_rank(bm, r))[r * BM16 + j];
            else ((uint4*)t3)[r * T316 + (j - BM16)] = ((const uint4*)cluster.map_shared_rank(t3, r))[r * T316 + (j - BM16)];
        }
        cluster.sync();                                                 // (nobody overwrites its boundary masks or exits while a peer still reads)
#else
        huf_build_wide<HB_T, true>(t1, maxbits, bm, t3, 0u, 1u << HUF_W);
        __syncthreads();
#endif
    }
    mbar_wait(mbar, 0);
    // (one thread reads the flag: another stream's kernel may set it at any moment, and the decision must be the CTA's)
    if (__syncthreads_or(maxbits == 0 || (tid == 0 && J.frame_bad[B.frame] != 0))) return;
    if ((uint32_t)tid < 16 + a) ((uint8_t*)scomp)[tid] = 0;              // bits below the stream start read as zero
    const bool fixed_len = huf_fixed_length(sm.wcnt);

    // ---- phase 1: transition map of every range -------------------------------------------------------------------------
    const HufShape shape = huf_stream_shape((const uint8_t*)scomp, a, it.src_size, HB_T);
    if (shape.last == 0) { if (tid == 0) flag_error(J, B.frame, zc::E_HUF_STREAM); return; }
    const int P0 = shape.P0, XTOP = shape.XTOP, S = shape.S;
    const int ck[HB_NLEG + 1] = {S < HB_CK0 ? S : HB_CK0, S < HB_CK1 ? S : HB_CK1, S < HB_CK2 ? S : HB_CK2, S};
    const int q0 = tid * S;
    const int qe = (q0 + S < P0) ? q0 + S : P0;
    const bool active = q0 < P0;
    const saddr_t s_comp = to_saddr(scomp), s_bm = to_saddr(bm);
    auto cp_at = [&](int rq0, int rqe, int j) { const int x = rq0 + ck[j]; return x < rqe ? x : rqe; };      // checkpoint j of a range

    // (1) first stop at checkpoint 0 (one lookup per candidate, out of one 64-bit window)
    uint64_t first = ~0ull, fcnt = 0;                                   // candidate -> landing offset / symbols so far (4 bits each)
    uint32_t live = 0;                                                  // landing offsets in use at the current checkpoint
    if (active) {
        const auto advance = [&](int& q, int& c, int lim) { track_advance(s_comp, s_bm, XTOP, q, c, lim); };
        hb_first_stop(q0, cp_at(q0, qe, 0), maxbits, fixed_len, advance, first, fcnt, live);
    }
    // (2) legs between checkpoints: the live tracks of ALL ranges are work items dealt out evenly over the CTA
    uint32_t leg_done = 0;
    for (int leg = 0; leg < HB_NLEG; leg++) {
        if (ck[leg + 1] == ck[leg]) continue;                           // (uniform) short ranges: nothing between these checkpoints
        leg_done |= 1u << leg;
        const uint32_t n_mine = (uint32_t)__popc(live);
        uint32_t qtotal;
        uint32_t idx = hb_scan(n_mine, misc + 8 * (leg & 1), &qtotal);
        for (uint32_t m = live; m; m &= m - 1) qitems[idx++] = (uint16_t)((uint32_t)tid | ((uint32_t)(__ffs((int)m) - 1) << 8));
        __syncthreads();
        for (uint32_t i = tid; i < qtotal; i += HB_T) {
            const uint32_t item = qitems[i];
            const int owner = (int)(item & 0xFFu), o = (int)(item >> 8);
            const int oq0 = owner * S, oqe = (oq0 + S < P0) ? oq0 + S : P0;
            const int lim = cp_at(oq0, oqe, leg + 1);
            int q = cp_at(oq0, oqe, leg) + o, c = 0;
            track_advance(s_comp, s_bm, XTOP, q, c, lim);
            legtab[(leg * HB_T + owner) * MAXC + o] = (uint16_t)((uint32_t)(q - lim) | ((uint32_t)c << 4));
        }
        __syncthreads();
        uint32_t nl = 0;
        for (uint32_t m = live; m; m &= m - 1) nl |= 1u << (legtab[(leg * HB_T + tid) * MAXC + (__ffs((int)m) - 1)] & 15u);
        live = nl;
    }
    // (3) the map candidate -> candidate of the next range: exit offset of every landing offset in use after the first stop
    uint64_t fmap = MAP_IDENTITY;
    if (active) {
        uint64_t exit_of = 0;
        uint32_t starts = 0;
        for (int k = 0; k < maxbits; k++) starts |= 1u << ((uint32_t)(first >> (4 * k)) & 15u);
        for (uint32_t m = starts; m; m &= m - 1) {
            const int o0 = __ffs((int)m) - 1;
            uint32_t o = (uint32_t)o0;
#pragma unroll
            for (int leg = 0; leg < HB_NLEG; leg++) if (leg_done & (1u << leg)) o = legtab[(leg * HB_T + tid) * MAXC + o] & 15u;
            exit_of |= (uint64_t)o << (4 * o0);
        }
        fmap = 0;
        for (int k = 0; k < maxbits; k++) fmap |= ((exit_of >> (4 * ((uint32_t)(first >> (4 * k)) & 15u))) & 15ull) << (4 * k);
        if (maxbits < 16) fmap |= ~0ull << (4 * maxbits);
    }
    // ---- compose the maps along the stream ----------------------------------------------------------------------------------
    const uint32_t ktrue = hb_compose<HB_NW>(fmap, maxbits, (uint64_t*)sm.wcnt, misc + 16);      // this thread's true candidate
    // symbols of the true track, and where it lands
    uint32_t mycnt = 0;
    int myland = -1;
    if (active && ktrue < (uint32_t)maxbits) {
        uint32_t o = (uint32_t)(first >> (4 * ktrue)) & 15u;
        mycnt = (uint32_t)(fcnt >> (4 * ktrue)) & 15u;
#pragma unroll
        for (int leg = 0; leg < HB_NLEG; leg++) {
            if (leg_done & (1u << leg)) { const uint32_t e = legtab[(leg * HB_T + tid) * MAXC + o]; o = e & 15u; mycnt += e >> 4; }
        }
        myland = qe + (int)o;
    }
    // the stream must end exactly on its first bit: the last active range's true track lands on P0
    const bool bad_end = active && qe == P0 && myland != P0;
    // ---- count, scan, write ------------------------------------------------------------------------------------------
    const int any_bad = __syncthreads_or(bad_end);                      // (also: every read of the leg tables is done before phase 2 overwrites them)
    uint32_t total;
    const uint32_t off = hb_scan(mycnt, misc, &total);
    if (any_bad || total != it.n_sym) { if (tid == 0) flag_error(J, B.frame, zc::E_HUF_STREAM); return; }
    uint8_t* dst = J.lit + B.lit_base + it.dst_off;
    const uint32_t a2 = (uint32_t)((uintptr_t)dst & 15);
    // write pass: from the true start to the first boundary at or past the end of the range
    if (mycnt) hb_write_range(s_comp, to_saddr(t3), to_saddr(t1), maxbits, XTOP, q0 + (int)ktrue, qe, to_saddr(sout) + a2 + off);
    __syncthreads();
    flush_image<HB_T>(dst, sout, a2, it.n_sym);
}

// The counting legs of k_huf_scout: like track_advance, but the steady state reads the count table (bits and number of all
// whole codewords of the next 12 bits: one byte, no bit tricks) and the exact stop at `lim` walks single symbols with the
// base table.
__device__ __forceinline__ void track_count(saddr_t comp, saddr_t tc, saddr_t t1, int maxbits, int xtop, int& q, int& cnt, int lim) {
    int rem = lim - q;
    if (rem <= 0) return;
    Win w;
    win_init(w, comp, xtop - q);
    while (rem > HUF_W) {
        const uint32_t e = lds8(tc + win_peek(w));
        const int used = (int)(e & 15u);
        cnt += (int)(e >> 4);
        rem -= used;
        win_consume(w, used);
    }
    const int sh1 = HUF_W - maxbits;
    while (rem > 0) {
        const uint32_t e = lds16(t1 + 2 * (win_peek(w) >> sh1));
        cnt++;
        rem -= (int)(e & 0xFFu);
        win_consume(w, (int)(e & 0xFFu));
    }
    q = lim - rem;
}

// k_huf_scout: where every range of k_huf_decode_block starts, for the block's four streams at once (one CTA per block, one
// thread per COARSE range of HS_F consecutive fine ranges; the fine ranges are k_huf_decode_block's 256 ranges of S bits).
// The speculation of the cluster kernel's phase 1 -- all max_bits candidates at the top of a range, tracks merging at
// checkpoints 12, 108 and 320 bits in -- is paid once per coarse range instead of once per fine range; from the end of the
// first fine range on, the (nearly always single) surviving track is followed to the next fine boundary, and so on.  Every
// leg between checkpoints is dealt out as work items over the whole CTA (all four streams), as in k_huf_decode_big.
// Leg tables, one slot per fine range: [slot][range][landing offset at the top] = landing offset at the end | symbols << 4;
// slot 0 holds the first fine range composed (indexed by the offset where the first stop landed), slots 1..3 serve the legs
// inside the first fine range until it is composed, then the further fine ranges.  The coarse maps are composed along each
// stream (64 entries: two warps), the true candidate of every coarse range resolves the chain of its fine ranges, and a
// scan of the symbol counts gives their output offsets.  Output: J.huf_bounds, 256 words per stream (fine range order):
// output offset << 4 | start offset (bits below the top of the range).
// The four compressed streams are staged side by side (bulk asynchronous copies): the counting reads them about 1.3 times.
// Shared memory: 36.3 KB + 4 stream images (cfg2: 101 KB, 2 CTAs per SM); ptxas (sm_100a): 55 registers, no spills.
constexpr int HS_C = 64;                                    // coarse ranges per stream
constexpr int HS_T = 4 * HS_C;                              // threads: the coarse ranges of the block's four streams
constexpr int HS_F = HB_T / HS_C;                           // fine ranges per coarse range
constexpr int HS_NLEG = HB_NLEG + HS_F - 1;                 // legs after the first stop
static_assert(HS_T == HB_T && HS_F > HB_NLEG, "k_huf_scout: one scan shape with k_huf_decode_block; slots 1..3 for the first fine range's legs");
constexpr uint32_t HS_LEG_BYTES = HS_F * HS_T * MAXC * 2u, HS_Q_BYTES = HS_T * MAXC * 2u;
constexpr uint32_t HS_TC_AT = sizeof(HufSmem), HS_LEG_AT = HS_TC_AT + 4096u, HS_Q_AT = HS_LEG_AT + HS_LEG_BYTES;
constexpr uint32_t HS_FIXED = HS_Q_AT + HS_Q_BYTES;                // HufSmem | count table | leg tables | queue
__host__ __device__ constexpr uint32_t hs_image_bytes(uint32_t max_stream) { return (max_stream + 15u + 16u + 16u + 15u) & ~15u; }
__host__ __device__ constexpr uint32_t hs_smem_bytes(uint32_t max_stream) { return HS_FIXED + 4u * hs_image_bytes(max_stream); }

// checkpoint j of a coarse range (bits below the top of the stream): the first stop's limit, two more inside the first fine
// range, then the fine boundaries; never past the end of the stream
__device__ __forceinline__ int hs_checkpoint(int ctop, int S, int P0, int j) {
    const int ck = j == 0 ? HB_CK0 : j == 1 ? HB_CK1 : HB_CK2;
    const int rel = j < HB_NLEG ? (S < ck ? S : ck) : (j - HB_NLEG + 1) * S;
    return ctop + rel < P0 ? ctop + rel : P0;
}

__global__ void __launch_bounds__(HS_T, 2) k_huf_scout(JobDev J) {
    NAF_DYN_SMEM(unsigned char, smem);
    HufSmem& sm = *(HufSmem*)smem;
    uint16_t* t1 = sm.t1;
    uint32_t* misc = sm.misc;                                           // [0..15] scan buffers, [16..23] warp start candidates,
                                                                        // [24..39] per stream: XTOP, P0, S; [56..57] mbarrier
    uint8_t* tc = smem + HS_TC_AT;
    uint16_t* legtab = (uint16_t*)(smem + HS_LEG_AT);
    uint16_t* qitems = (uint16_t*)(smem + HS_Q_AT);                     // range | offset << 8
    uint8_t* images = smem + HS_FIXED;
    const uint32_t stride = hs_image_bytes(J.max_huf_stream);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = tid / HS_C, c = tid % HS_C;                            // stream, coarse range

    const uint32_t item0 = blockIdx.x * 4u;
    const BlockDesc& B = J.blocks[J.huf_items[item0].block];
    const HufItem it = J.huf_items[item0 + s];
    const uint8_t* g = J.comp + B.src_off + it.src_off;
    const uint32_t a = (uint32_t)((uintptr_t)g & 15);
    uint8_t* img = images + s * stride;                                 // 16 zero bytes, then the 16 B-aligned image of global memory
    const saddr_t mbar = to_saddr(&misc[56]);
    if (tid == 0) mbar_init(mbar, 4);
    __syncthreads();
    if (c == 0) stage_stream(img + 16, g - a, ((a + it.src_size + 15u) >> 4) << 4, mbar);
    const HufTree tree = huf_tree<HS_T>(J, B, sm.weights);
    const int maxbits = tree.maxbits;
    __syncthreads();
    if (maxbits != 0) {                                                 // (a bad tree was flagged by k_build_tables)
        huf_build_t1<HS_T>(sm.weights, tree.nsym, maxbits, t1, sm.wcnt);
        huf_build_wide<HS_T, false>(t1, maxbits, nullptr, nullptr, 0u, 1u << HUF_W, tc);
    }
    const bool fixed_len = huf_fixed_length(sm.wcnt);
    // (one thread reads the flag: another stream's kernel may set it at any moment, and the decision must be the CTA's)
    const bool skip = __syncthreads_or(maxbits == 0 || (tid == 0 && J.frame_bad[B.frame] != 0));
    mbar_wait(mbar, 0);
    if (skip) return;
    if ((uint32_t)c < 16 + a) img[c] = 0;                                // bits below the stream start read as zero
    const HufShape shape = huf_stream_shape(img, a, it.src_size, HB_T); // (the fine ranges are k_huf_decode_block's)
    if (__syncthreads_or(shape.last == 0)) { if (tid == 0) flag_error(J, B.frame, zc::E_HUF_STREAM); return; }
    const int P0 = shape.P0, XTOP = shape.XTOP, S = shape.S;
    if (c == 0) { misc[24 + 4 * s] = (uint32_t)XTOP; misc[25 + 4 * s] = (uint32_t)P0; misc[26 + 4 * s] = (uint32_t)S; }
    const int ctop = c * HS_F * S;
    const bool active = ctop < P0;
    const saddr_t s_images = to_saddr(images), s_tc = to_saddr(tc), s_t1 = to_saddr(t1);
    const saddr_t s_comp = s_images + s * stride;

    // (1) first stop at checkpoint 0
    uint64_t first = ~0ull, fcnt = 0;                                   // candidate -> landing offset / symbols so far (4 bits each)
    uint32_t live = 0;                                                  // landing offsets in use at the current checkpoint
    if (active) {
        const auto count = [&](int& q, int& n, int lim) { track_count(s_comp, s_tc, s_t1, maxbits, XTOP, q, n, lim); };
        hb_first_stop(ctop, hs_checkpoint(ctop, S, P0, 0), maxbits, fixed_len, count, first, fcnt, live);
    }
    // (2) legs between checkpoints: the live tracks of ALL coarse ranges are work items dealt out evenly over the CTA
    auto slot_of = [](int leg) { return leg <= HB_NLEG ? leg : leg - HB_NLEG; };
    auto tab = [&](int slot, int range, uint32_t o) { return to_saddr(legtab) + 2u * (((uint32_t)slot * HS_T + (uint32_t)range) * MAXC + o); };
    uint32_t leg_done = 0, live1 = 0;
    uint64_t land1 = 0;                                                 // first-stop landing -> landing at the end of fine range 0
    for (int leg = 1; leg <= HS_NLEG; leg++) {
        if (leg == HB_NLEG + 1) {                                       // the first fine range is complete: compose it into slot 0
            if (active) {
                uint32_t starts = 0;
                for (int k = 0; k < maxbits; k++) starts |= 1u << ((uint32_t)(first >> (4 * k)) & 15u);
                for (uint32_t m = starts; m; m &= m - 1) {
                    const uint32_t o0 = (uint32_t)(__ffs((int)m) - 1);
                    uint32_t o = o0, n = 0;
                    for (int l = 1; l <= HB_NLEG; l++)
                        if (leg_done & (1u << l)) { const uint32_t e = lds16(tab(l, tid, o)); o = e & 15u; n += e >> 4; }
                    legtab[(uint32_t)tid * MAXC + o0] = (uint16_t)(o | (n << 4));
                    land1 |= (uint64_t)o << (4 * o0);
                }
            }
            live1 = live;
        }
        const int slot = slot_of(leg);
        const uint32_t mine = (active && hs_checkpoint(ctop, S, P0, leg - 1) < hs_checkpoint(ctop, S, P0, leg)) ? live : 0u;
        if (mine) leg_done |= 1u << leg;
        uint32_t qtotal;
        uint32_t idx = hb_scan((uint32_t)__popc(mine), misc + 8 * (leg & 1), &qtotal);
        for (uint32_t m = mine; m; m &= m - 1) qitems[idx++] = (uint16_t)((uint32_t)tid | ((uint32_t)(__ffs((int)m) - 1) << 8));
        __syncthreads();
        for (uint32_t i = tid; i < qtotal; i += HS_T) {
            const uint32_t item = qitems[i];
            const int owner = (int)(item & 0xFFu), o = (int)(item >> 8);
            const int os = owner / HS_C;
            const int oxtop = (int)misc[24 + 4 * os], op0 = (int)misc[25 + 4 * os], oS = (int)misc[26 + 4 * os];
            const int octop = (owner % HS_C) * HS_F * oS;
            const int lim = hs_checkpoint(octop, oS, op0, leg);
            int q = hs_checkpoint(octop, oS, op0, leg - 1) + o, n = 0;
            track_count(s_images + os * stride, s_tc, s_t1, maxbits, oxtop, q, n, lim);
            legtab[((uint32_t)slot * HS_T + (uint32_t)owner) * MAXC + (uint32_t)o] = (uint16_t)((uint32_t)(q - lim) | ((uint32_t)n << 4));
        }
        __syncthreads();
        if (mine) {
            uint32_t nl = 0;
            for (uint32_t m = mine; m; m &= m - 1) nl |= 1u << (lds16(tab(slot, tid, (uint32_t)(__ffs((int)m) - 1))) & 15u);
            live = nl;
        }
    }
    // (3) the map candidate -> candidate of the next coarse range
    uint64_t fmap = MAP_IDENTITY;
    if (active) {
        uint64_t exit_of = 0;                                           // landing at the end of fine range 0 -> at the end of the coarse range
        for (uint32_t m = live1; m; m &= m - 1) {
            const uint32_t o1 = (uint32_t)(__ffs((int)m) - 1);
            uint32_t o = o1;
#pragma unroll
            for (int j = 1; j < HS_F; j++) if (leg_done & (1u << (HB_NLEG + j))) o = lds16(tab(j, tid, o)) & 15u;
            exit_of |= (uint64_t)o << (4 * o1);
        }
        fmap = 0;
        for (int k = 0; k < maxbits; k++) {
            const uint32_t o1 = (uint32_t)(land1 >> (4 * ((uint32_t)(first >> (4 * k)) & 15u))) & 15u;
            fmap |= ((exit_of >> (4 * o1)) & 15ull) << (4 * k);
        }
        if (maxbits < 16) fmap |= ~0ull << (4 * maxbits);
    }
    // ---- compose the maps along each stream ----------------------------------------------------------------------------------
    constexpr int WPS = HS_C / 32;                                      // warps per stream
    const uint32_t ktrue = hb_compose<WPS>(fmap, maxbits, (uint64_t*)sm.wcnt, misc + 16);       // this coarse range's true candidate
    // ---- the chain of the true track through the fine ranges: start offsets and symbols ------------------------------------
    uint32_t start[HS_F], cnt[HS_F];
#pragma unroll
    for (int j = 0; j < HS_F; j++) { start[j] = 0; cnt[j] = 0; }
    bool bad_end = false;
    if (active) {
        const bool at_end = ctop + HS_F * S >= P0;                      // the stream ends in this coarse range: the true track must land on P0
        if (ktrue < (uint32_t)maxbits) {
            const uint32_t o0 = (uint32_t)(first >> (4 * ktrue)) & 15u;
            const uint32_t e0 = lds16(tab(0, tid, o0));
            start[0] = ktrue;
            cnt[0] = ((uint32_t)(fcnt >> (4 * ktrue)) & 15u) + (e0 >> 4);
            uint32_t o = e0 & 15u;
#pragma unroll
            for (int j = 1; j < HS_F; j++) {
                start[j] = o;
                if (leg_done & (1u << (HB_NLEG + j))) { const uint32_t e = lds16(tab(j, tid, o)); o = e & 15u; cnt[j] = e >> 4; }
            }
            bad_end = at_end && o != 0;
        } else {
            bad_end = at_end;
        }
    }
    uint32_t mine = 0;
#pragma unroll
    for (int j = 0; j < HS_F; j++) mine += cnt[j];
    // ---- output offsets: exclusive scan of the symbols over each stream ------------------------------------------------
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) misc[warp] = inc;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < WPS; w++) { const uint32_t x = misc[s * WPS + w]; total += x; if (s * WPS + w < warp) before += x; }
    if (__syncthreads_or(bad_end || total != it.n_sym)) { if (tid == 0) flag_error(J, B.frame, zc::E_HUF_STREAM); return; }
    uint32_t off = before + inc - mine;
    uint32_t* dst = J.huf_bounds + (size_t)(item0 + s) * HB_T + (uint32_t)c * HS_F;
#pragma unroll
    for (int j = 0; j < HS_F; j += 4) {
        uint32_t v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) { v[u] = (off << 4) | start[j + u]; off += cnt[j + u]; }
        *(uint4*)(dst + j) = make_uint4(v[0], v[1], v[2], v[3]);
    }
}

// k_huf_decode_block: the write pass, ONE CTA PER BLOCK working through the block's four streams one after the other, every
// thread from the exact start and output offset k_huf_scout found for its range.  The tables (base table, 3-symbol table) are
// built once per block by the CTA itself -- no cluster, no exchange -- and stay in shared memory for all four streams.  The
// next stream's bytes are fetched (bulk asynchronous copy) while the current stream's output is flushed.
__global__ void __launch_bounds__(HB_T, 3) k_huf_decode_block(JobDev J) {
    NAF_DYN_SMEM(unsigned char, smem);
    HufSmem& sm = *(HufSmem*)smem;
    uint32_t* t3 = (uint32_t*)(smem + HB_T3_AT);
    uint8_t* sout = smem + HB_SOUT_AT;
    uint32_t* scomp = (uint32_t*)(smem + HB_FIXED);
    const int tid = threadIdx.x;

    const uint32_t item0 = blockIdx.x * 4u;                              // the block's four streams are four consecutive items
    const BlockDesc& B = J.blocks[J.huf_items[item0].block];
    const saddr_t mbar = to_saddr(&sm.misc[56]);
    // stages stream `sidx`: the 16 B-aligned image of global memory, behind 16 bytes that stay zero
    auto stage = [&](uint32_t sidx) {
        const HufItem si = J.huf_items[item0 + sidx];
        const uint8_t* sg = J.comp + B.src_off + si.src_off;
        const uint32_t sa = (uint32_t)((uintptr_t)sg & 15);
        if (tid == 0) stage_stream(scomp + 4, sg - sa, ((sa + si.src_size + 15u) >> 4) << 4, mbar);
    };
    if (tid == 0) mbar_init(mbar, 1);
    __syncthreads();
    stage(0);
    const HufTree tree = huf_tree<HB_T>(J, B, sm.weights);
    const int maxbits = tree.maxbits;
    __syncthreads();
    if (maxbits != 0) {                                                 // (a bad tree was flagged by k_build_tables)
        huf_build_t1<HB_T>(sm.weights, tree.nsym, maxbits, sm.t1, sm.wcnt);
        huf_build_wide<HB_T, true>(sm.t1, maxbits, nullptr, t3, 0u, 1u << HUF_W);
    }
    // (one thread reads the flag: k_huf_scout flags every stream it refuses, and another stream's kernel may set it at any
    // moment -- the decision must be the CTA's)
    const bool skip = __syncthreads_or(maxbits == 0 || (tid == 0 && J.frame_bad[B.frame] != 0));
    for (uint32_t sidx = 0; sidx < 4u; sidx++) {
        const HufItem it = J.huf_items[item0 + sidx];
        const uint32_t bound = skip ? 0u : J.huf_bounds[(size_t)(item0 + sidx) * HB_T + tid];     // output offset << 4 | start offset
        const uint8_t* g = J.comp + B.src_off + it.src_off;
        const uint32_t a = (uint32_t)((uintptr_t)g & 15);
        mbar_wait(mbar, sidx & 1u);                                     // the bulk copy of this stream has landed
        if (skip) break;
        if ((uint32_t)tid < 16 + a) ((uint8_t*)scomp)[tid] = 0;          // bits below the stream start read as zero
        __syncthreads();

        const HufShape shape = huf_stream_shape((const uint8_t*)scomp, a, it.src_size, HB_T);     // (k_huf_scout refused a zero last byte)
        const int P0 = shape.P0, S = shape.S;
        const int q0 = tid * S;
        const int qe = (q0 + S < P0) ? q0 + S : P0;
        uint8_t* dst = J.lit + B.lit_base + it.dst_off;
        const uint32_t a2 = (uint32_t)((uintptr_t)dst & 15);
        // write pass: from the exact start k_huf_scout found to the first boundary at or past the end of the range
        if (q0 < P0)
            hb_write_range(to_saddr(scomp), to_saddr(t3), to_saddr(sm.t1), maxbits, shape.XTOP, q0 + (int)(bound & 15u), qe,
                           to_saddr(sout) + a2 + (bound >> 4));
        __syncthreads();
        if (sidx + 1 < 4u) stage(sidx + 1);                             // the next stream's bytes travel while this one's output is flushed
        flush_image<HB_T>(dst, sout, a2, it.n_sym);
        __syncthreads();                                                // the output image is overwritten by the next stream
    }
}

// --------------------------------------------------------------------------------------------------------------
// k_lz_literals: one CTA per block.  Raw / RLE blocks and literal-only blocks are plain copies or fills; for
// blocks with sequences every literal run goes to its final position and match destinations are published.
// Cooperative global -> global copy of n bytes with arbitrary alignments by `nlanes` threads (a warp or a CTA):
// destination-aligned 16-byte stores; each is assembled from the two aligned 16-byte source words that span it.
// The source must be readable up to 31 bytes past its end (staging buffers are padded).
__device__ __forceinline__ void copy_g2g_plain(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, int lane, int nlanes) {
    if (n < 64) { for (uint32_t k = lane; k < n; k += nlanes) dst[k] = src[k]; return; }
    const uint32_t h = (uint32_t)(-(intptr_t)dst) & 15u;
    for (uint32_t k = lane; k < h; k += nlanes) dst[k] = src[k];
    const uint32_t body = (n - h) >> 4;
    const uintptr_t sa = (uintptr_t)(src + h);
    const uint4* sw = (const uint4*)(sa & ~(uintptr_t)15);
    const uint32_t mis = (uint32_t)(sa & 15), q = mis >> 2, sh = (mis & 3) * 8;
    uint4* d4 = (uint4*)(dst + h);
    for (uint32_t c = lane; c < body; c += nlanes) {
        const uint4 A = sw[c], B = sw[c + 1];
        uint32_t w0, w1, w2, w3, w4;                   // the five words starting at word q of {A, B}
        if (q == 0) { w0 = A.x; w1 = A.y; w2 = A.z; w3 = A.w; w4 = B.x; }
        else if (q == 1) { w0 = A.y; w1 = A.z; w2 = A.w; w3 = B.x; w4 = B.y; }
        else if (q == 2) { w0 = A.z; w1 = A.w; w2 = B.x; w3 = B.y; w4 = B.z; }
        else { w0 = A.w; w1 = B.x; w2 = B.y; w3 = B.z; w4 = B.w; }
        d4[c] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
    }
    const uint32_t done = h + (body << 4);
    for (uint32_t k = done + lane; k < n; k += nlanes) dst[k] = src[k];
}

// U: chunks per lane in flight.  1 (the loop above) for the short runs of a batch -- registers: k_lz_literals lost 40 % with 4.
// 4 where a lone CTA or warp copies kilobytes and would otherwise pay a round trip to memory per chunk (a single small
// archive): every load of a pass is issued before its first store -- head and tail bytes (fewer than 16 each: one per lane)
// and up to U chunks per lane: one round trip for a match of up to U x nlanes x 16 bytes.  nlanes >= 32.
template <int U>
__device__ __forceinline__ void copy_g2g_1rt(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, int lane, int nlanes);
template <int U = 1>
__device__ __forceinline__ void copy_g2g(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, int lane, int nlanes) {
    if (U == 1) copy_g2g_plain(dst, src, n, lane, nlanes);
    else copy_g2g_1rt<U>(dst, src, n, lane, nlanes);
}
template <int U>
__device__ __forceinline__ void copy_g2g_1rt(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, int lane, int nlanes) {
    if (n < 64) {                                      // both bytes of a lane loaded before either is stored
        const uint32_t k0 = lane, k1 = lane + nlanes;
        uint8_t v0 = 0, v1 = 0;
        if (k0 < n) v0 = src[k0];
        if (k1 < n) v1 = src[k1];
        if (k0 < n) dst[k0] = v0;
        if (k1 < n) dst[k1] = v1;
        return;
    }
    const uint32_t h = (uint32_t)(-(intptr_t)dst) & 15u;
    const uint32_t body = (n - h) >> 4;
    const uintptr_t sa = (uintptr_t)(src + h);
    const uint4* sw = (const uint4*)(sa & ~(uintptr_t)15);
    const uint32_t mis = (uint32_t)(sa & 15), q = mis >> 2, sh = (mis & 3) * 8;
    uint4* d4 = (uint4*)(dst + h);
    const uint32_t tk = h + (body << 4) + (uint32_t)lane;
    uint8_t hb = 0, tb = 0;
    if ((uint32_t)lane < h) hb = src[lane];
    if (tk < n) tb = src[tk];
    for (uint32_t c = lane; c < body; c += (uint32_t)U * (uint32_t)nlanes) {
        uint4 A[U], B[U];
#pragma unroll
        for (int u = 0; u < U; u++) { const uint32_t x = c + (uint32_t)u * nlanes; if (x < body) { A[u] = sw[x]; B[u] = sw[x + 1]; } }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint32_t x = c + (uint32_t)u * nlanes;
            if (x < body) {
                const uint4 a = A[u], b = B[u];
                uint32_t w0, w1, w2, w3, w4;
                if (q == 0) { w0 = a.x; w1 = a.y; w2 = a.z; w3 = a.w; w4 = b.x; }
                else if (q == 1) { w0 = a.y; w1 = a.z; w2 = a.w; w3 = b.x; w4 = b.y; }
                else if (q == 2) { w0 = a.z; w1 = a.w; w2 = b.x; w3 = b.y; w4 = b.z; }
                else { w0 = a.w; w1 = b.x; w2 = b.y; w3 = b.z; w4 = b.w; }
                d4[x] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
            }
        }
    }
    if ((uint32_t)lane < h) dst[lane] = hb;
    if (tk < n) dst[tk] = tb;
}

constexpr int LZLIT_G = 32;                        // lanes per literal run (8-lane groups, four runs in flight per warp, measured no faster)
constexpr int LZLIT_SPLIT = 4;                     // CTAs that share the runs of one block
constexpr uint32_t LZLIT_LONG = 4096;              // longer runs are copied by the whole CTA (at most 32 per block)

// U: see copy_g2g (4 for a job of a few blocks, where the long runs of a block are what the kernel waits for)
// (the batch variant is held to 6 CTAs per SM: at 45 registers instead of 40 -- one more select for the block index -- it lost
//  an eighth of its rate, 0.52 -> 0.60 ms on the 256-archive job)
template <int U>
__global__ void __launch_bounds__(256, U == 1 ? 6 : 1) k_lz_literals(JobDev J) {
    __shared__ uint32_t lq_n, lq_lp[40], lq_op[40], lq_ll[40];
    const uint32_t bi = J.tiny_blocks ? J.lit_big_list[blockIdx.x] : blockIdx.x;       // (with tiny_blocks: the blocks that are not k_lz_literals_tiny's)
    const BlockDesc& B = J.blocks[bi];
    if (J.frame_bad[B.frame]) return;
    const BlockState& S = J.bstate[bi];
    uint8_t* out = J.out + S.out_off;
    // gridDim.y CTAs share a block: the time of this kernel is the time of the block with the most sequences (one literal
    // run per warp and step, two dependent latencies each), so the runs of a block are dealt out to several CTAs
    const int tid = threadIdx.x + blockIdx.y * blockDim.x, nt = blockDim.x * gridDim.y;
    if (B.btype == BT_RAW) { copy_g2g(out, J.comp + B.src_off, B.src_size, tid, nt); return; }   // (COMP_PAD covers the over-read)
    if (B.btype == BT_RLE) {
        uint8_t v = J.comp[B.src_off];
        for (uint32_t i = tid; i < B.src_size; i += nt) out[i] = v;
        return;
    }
    const uint8_t* lsrc = nullptr;                   // raw literals sit in the compressed block, Huffman literals in the staging buffer
    uint8_t rle = 0;
    if (B.lit_type == LT_RAW) lsrc = J.comp + B.src_off + B.lit_src;
    else if (B.lit_type == LT_RLE) rle = J.comp[B.src_off + B.lit_src];
    else lsrc = J.lit + B.lit_base;
    if (B.n_seq == 0) {
        if (B.lit_type == LT_RLE) for (uint32_t i = tid; i < B.lit_regen; i += nt) out[i] = rle;
        else copy_g2g(out, lsrc, B.lit_regen, tid, nt);
        return;
    }
    // one literal run (a few hundred bytes) per group of LZLIT_G lanes
    // (consecutive runs go to different CTAs: a block of a real genome has a handful of runs of tens of kilobytes, each copied
    //  by the whole CTA that owns it)
    //  (U == 1, a batch: the runs of a block stay with neighbouring warps -- dealt across CTAs k_lz_literals took 0.63 ms
    //  instead of 0.52 on the 256-archive job)
    const int lane = tid % LZLIT_G, ng = nt / LZLIT_G, grp = U > 1 ? (int)(threadIdx.x / LZLIT_G) * (int)gridDim.y + (int)blockIdx.y : tid / LZLIT_G;
    const uint32_t n = B.n_seq, base = B.seq_base;
    if (threadIdx.x == 0) lq_n = 0;
    __syncthreads();
    // the record of the NEXT run is loaded before the copy of this one: a run costs two dependent latencies (record, then
    // literals), and the copy hides the first of them
    auto fetch = [&](uint32_t i, uint32_t& lp, uint32_t& op, uint32_t& ll, uint32_t& ml) {
        if (i > n) return;
        const uint32_t j = i < n ? i : n - 1;
        const uint4 r = *(const uint4*)&J.seq[base + j];                 // ll, ml, off, litpos
        ll = r.x; ml = r.y; lp = r.w; op = J.seq[base + j].outpos;
    };
    uint32_t lp = 0, op = 0, ll = 0, ml = 0;
    fetch((uint32_t)grp, lp, op, ll, ml);
    for (uint32_t i = grp; i <= n; i += ng) {
        uint32_t nlp = 0, nop = 0, nll = 0, nml = 0;
        fetch(i + ng, nlp, nop, nll, nml);
        if (i < n) {
            if (lane == 0) J.seq[base + i].match_pos = S.out_off + op + ll;     // absolute destination of the match
        } else {                                       // literals after the last sequence (the record is that of sequence n - 1)
            lp += ll; op += ll + ml; ll = B.lit_regen - lp;
        }
        if (ll > LZLIT_LONG && B.lit_type != LT_RLE) {                    // a long run (often the literals after the last sequence of a block
            if (lane == 0) { const uint32_t q = atomicAdd(&lq_n, 1u); lq_lp[q] = lp; lq_op[q] = op; lq_ll[q] = ll; }   // with few sequences): whole CTA
        } else if (B.lit_type == LT_RLE) for (uint32_t k = lane; k < ll; k += LZLIT_G) out[op + k] = rle;
        else copy_g2g(out + op, lsrc + lp, ll, lane, LZLIT_G);            // (head, body and tail loaded together, copy_g2g_1rt<1>: measured the same 0.52 ms on the 256-archive job)
        lp = nlp; op = nop; ll = nll; ml = nml;
    }
    __syncthreads();
    for (uint32_t q = 0; q < lq_n; q++) copy_g2g<U>(out + lq_op[q], lsrc + lq_lp[q], lq_ll[q], (int)threadIdx.x, (int)blockDim.x);
}

// One warp per tiny block, eight blocks per CTA: a CTA per block spent its time being launched (5.5 ms for the 2 x 10^6
// blocks of a 10^6-read archive).  Lane j holds the record of sequence j; the runs are copied one after the other by the
// whole warp (they are a few dozen bytes each).
__global__ void __launch_bounds__(256) k_lz_literals_tiny(JobDev J) {
    const int lane = threadIdx.x & 31;
    const uint32_t bi = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (bi >= J.n_blocks) return;
    const BlockDesc& B = J.blocks[bi];
    if (!tiny_lit_block(B)) return;
    if (J.frame_bad[B.frame]) return;
    const BlockState& S = J.bstate[bi];
    uint8_t* out = J.out + S.out_off;
    if (B.btype == BT_RAW) { copy_g2g(out, J.comp + B.src_off, B.src_size, lane, 32); return; }
    if (B.btype == BT_RLE) {
        const uint8_t v = J.comp[B.src_off];
        for (uint32_t i = lane; i < B.src_size; i += 32) out[i] = v;
        return;
    }
    const uint8_t* lsrc = nullptr;
    uint8_t rle = 0;
    if (B.lit_type == LT_RAW) lsrc = J.comp + B.src_off + B.lit_src;
    else if (B.lit_type == LT_RLE) rle = J.comp[B.src_off + B.lit_src];
    else lsrc = J.lit + B.lit_base;
    const uint32_t n = B.n_seq, base = B.seq_base;
    uint32_t lp = 0, op = 0, ll = 0, ml = 0;
    if ((uint32_t)lane < n) {
        const uint4 r = *(const uint4*)&J.seq[base + lane];                  // ll, ml, off, litpos
        ll = r.x; ml = r.y; lp = r.w; op = J.seq[base + lane].outpos;
        J.seq[base + lane].match_pos = S.out_off + op + ll;                  // absolute destination of the match
    }
    // the literals after the last sequence: lane n (n <= 32; lane 32 does not exist, so lane 31's record is extended in place)
    uint32_t t_lp = 0, t_op = 0;
    if (n) {
        const uint32_t e_lp = __shfl_sync(0xFFFFFFFFu, lp + ll, (int)n - 1), e_op = __shfl_sync(0xFFFFFFFFu, op + ll + ml, (int)n - 1);
        t_lp = e_lp; t_op = e_op;
    }
    for (uint32_t i = 0; i <= n; i++) {
        uint32_t rl, rp, ro;
        if (i < n) { rl = __shfl_sync(0xFFFFFFFFu, ll, (int)i); rp = __shfl_sync(0xFFFFFFFFu, lp, (int)i); ro = __shfl_sync(0xFFFFFFFFu, op, (int)i); }
        else { rp = t_lp; ro = t_op; rl = B.lit_regen > t_lp ? B.lit_regen - t_lp : 0u; }
        if (rl == 0) continue;
        if (rp + rl > B.lit_regen) break;                // (inconsistent records: the block was flagged by the sequence decode)
        if (B.lit_type == LT_RLE) for (uint32_t k = lane; k < rl; k += 32) out[ro + k] = rle;
        else copy_g2g(out + ro, lsrc + rp, rl, lane, 32);
    }
}

// --------------------------------------------------------------------------------------------------------------
// Match execution.
__device__ __forceinline__ uint32_t resolve_offset(const JobDev& J, uint32_t v, uint32_t block) {
    if (!(v & OFF_SYMBOLIC)) return v;
    uint32_t in = J.bstate[block].rep_in[(v >> 29) & 3];
    uint32_t d = v & 0x1FFFFFFFu;
    return in > d ? in - d : 0;
}

// bytes [d, d+ml) <- periodic extension of [d-off, d): byte k comes from d-off + (k mod off); all sources lie
// strictly below d, so the copy has no intra-match hazard even when off < ml.
//
// Loads and stores go to the same buffer, so the compiler keeps them in program order; a plain byte loop then has ONE
// load in flight (every store waits for its load, every load for the store before it): ~0.5 us per byte, 30 us for a
// 64-byte match, and a round lasts as long as its slowest copy.  The copies below issue 8 independent loads before the
// first store.
__device__ __forceinline__ void copy_match(uint8_t* out, uint64_t d, uint32_t off, uint32_t ml, int lane, int nlanes) {
    const uint8_t* s = out + d - off;
    uint8_t* o = out + d;
    const bool periodic = off < ml;
    for (uint32_t k0 = 0; k0 < ml; k0 += 8u * (uint32_t)nlanes) {
        uint8_t t[8];
#pragma unroll
        for (uint32_t j = 0; j < 8; j++) {
            const uint32_t k = k0 + j * (uint32_t)nlanes + (uint32_t)lane;
            if (k < ml) t[j] = s[periodic ? k % off : k];
        }
#pragma unroll
        for (uint32_t j = 0; j < 8; j++) {
            const uint32_t k = k0 + j * (uint32_t)nlanes + (uint32_t)lane;
            if (k < ml) o[k] = t[j];
        }
    }
}

// A run of one byte value (offset 1: N stretches, zero padding), n >= 1 bytes at dst, by `nlanes` threads: 16-byte stores.
__device__ __forceinline__ void fill_run(uint8_t* dst, uint32_t v, uint32_t n, int lane, int nlanes) {
    const uint32_t h = (uint32_t)(-(intptr_t)dst) & 15u;
    if (n < 32u + h) { for (uint32_t k = lane; k < n; k += nlanes) dst[k] = (uint8_t)v; return; }
    if ((uint32_t)lane < h) dst[lane] = (uint8_t)v;
    const uint32_t body = (n - h) >> 4, w = v * 0x01010101u;
    uint4* d4 = (uint4*)(dst + h);
    for (uint32_t c = lane; c < body; c += nlanes) d4[c] = make_uint4(w, w, w, w);
    for (uint32_t k = h + (body << 4) + lane; k < n; k += nlanes) dst[k] = (uint8_t)v;
}

// A long match by `nlanes` threads (a warp, or the CTA for the very long ones).
__device__ __forceinline__ void copy_long_match(uint8_t* out, uint64_t d, uint32_t off, uint32_t ml, int lane, int nlanes) {
    if (off >= ml) copy_g2g(out + d, out + d - off, ml, lane, nlanes);        // disjoint: 16-byte loads and stores
    else if (off == 1) fill_run(out + d, out[d - 1], ml, lane, nlanes);
    else copy_match(out, d, off, ml, lane, nlanes);
}

// k_lz_index: for every 4 KB cell of every frame's output, the first match of the frame that ends after the start of the cell
// (the frame's match count if none does).  Matches are ordered and disjoint, so match i owns the cells whose start lies in
// [end of match i - 1, end of match i).  One thread per match; the last match of a frame also fills the cells behind it.
constexpr uint32_t LZ_IDX_SHIFT = 12, LZ_IDX_PER_CHUNK = 65536u >> LZ_IDX_SHIFT;          // index cells per 64 KB chunk of the chunk table

__global__ void __launch_bounds__(256) k_lz_index(JobDev J) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= J.n_seq) return;
    const SeqRec& R = J.seq[i];
    const BlockDesc& B = J.blocks[R.block];
    const FrameDesc& F = J.frames[B.frame];
    if (J.frame_bad[B.frame]) return;
    uint32_t* ix = J.lz_idx + (size_t)J.fin_chunk_first[B.frame] * LZ_IDX_PER_CHUNK + B.frame;      // (one extra cell per frame: the cell past its end)
    const uint64_t n_cells = (uint64_t)(J.fin_chunk_first[B.frame + 1] - J.fin_chunk_first[B.frame]) * LZ_IDX_PER_CHUNK + 1;     // (+1: the cell past the end)
    const uint64_t e_prev = i == F.first_seq ? 0 : (J.seq[i - 1].match_pos + J.seq[i - 1].ml - F.dst_off);
    const uint64_t e = R.match_pos + R.ml - F.dst_off;
    // cells k with e_prev <= k * 4096 < e  (the first match: every cell from 0 on)
    uint64_t k0 = i == F.first_seq ? 0 : (e_prev + (1u << LZ_IDX_SHIFT) - 1) >> LZ_IDX_SHIFT;
    uint64_t k1 = (e + (1u << LZ_IDX_SHIFT) - 1) >> LZ_IDX_SHIFT;      // first cell that starts at or after e
    if (k1 > n_cells) k1 = n_cells;
    for (uint64_t k = k0; k < k1; k++) ix[k] = (uint32_t)i;
    if (i + 1 == (uint64_t)F.first_seq + F.n_seq) for (uint64_t k = k1; k < n_cells; k++) ix[k] = (uint32_t)(i + 1);
}

// Match resolution.
//
// A match may run once every earlier match whose destination intersects its source range has finished in an EARLIER
// round (all literals are final before round 1).  Two mechanisms keep the number of rounds small:
//   * redirect ("pointer jumping"): if the whole source range lies inside the destination of ONE unfinished match j,
//     the bytes wanted are by definition equal to those `off_j` further back (out[p] == out[p - off_j] for every p in
//     j's destination, also for overlapping j).  So the match rewrites its own offset, off += off_j, and looks again:
//     chains of copies-of-copies (repeat families, reads sampled from one genome) collapse in a few hops.
//   * rounds are driven by a persistent cooperative kernel over a compacted worklist of the matches still pending,
//     with a grid-wide barrier between rounds: deep chains (text-like sections) cost one barrier per level instead of
//     one kernel launch, and there is no serial fallback.
// Short matches (the common case: a few tens of bytes) are copied by their own thread; long ones (N stretches:
// offset 1, ~100 KB) are queued in shared memory and copied by the whole CTA.
constexpr uint32_t LZ_SHORT = 64;
constexpr uint32_t LZ_WARP_MAX = 4096;             // longer matches are copied by the whole CTA
constexpr int LZ_CTA = 256;
constexpr int LZ_HOPS = 8;
constexpr uint32_t LZ_MIN_ROUNDS = 3, LZ_MIN_PENDING = 192;        // no hand-over before round 3 or for a handful of matches

// Returns 1 when match i may be copied now (d/off/ml filled), 0 when it has to wait, 2 when it was rejected.
__device__ __forceinline__ int lz_try(const JobDev& J, uint32_t i, uint32_t round, uint64_t& d, uint32_t& off, uint32_t& ml) {
    // What blocked this match last time is remembered: while that match is still unfinished there is nothing to look for
    // (one load instead of a binary search and a dozen dependent probes).  Sections whose matches descend from one another
    // through tens of generations -- a diverged repeat family, cfg3: 78 rounds with ~2 % of the pending matches becoming ready
    // in each -- spent their time re-examining matches that could not have become ready.
    // (lz_round does that check before calling here)
    SeqRec& R = J.seq[i];
    const uint32_t bi = R.block;
    const BlockDesc& B = J.blocks[bi];
    if (J.frame_bad[B.frame]) { J.seq_done[i] = round; return 2; }
    const FrameDesc& F = J.frames[B.frame];
    ml = R.ml;
    const uint32_t off0 = resolve_offset(J, R.off, bi);
    off = off0;
    d = R.match_pos;
    int verdict = 0;
    for (int hop = 0; hop <= LZ_HOPS; hop++) {
        if (off == 0 || (uint64_t)off > d - F.dst_off) {
            flag_error(J, B.frame, zc::E_OFFSET);
            J.seq_done[i] = round;
            return 2;
        }
        const uint64_t s = d - off;
        const uint64_t e = (off < ml) ? d : s + ml;                   // external source range [s, e)
        // first earlier match (same frame) ending after s: between the index entries of the 4 KB cell that holds s and of the
        // next one (k_lz_index), so the bisection has ~5 steps instead of ~20 over a frame of 10^6 matches
        uint32_t lo = F.first_seq, hi = i;
        {
            const uint32_t* ix = J.lz_idx + (size_t)J.fin_chunk_first[B.frame] * LZ_IDX_PER_CHUNK + B.frame + ((s - F.dst_off) >> LZ_IDX_SHIFT);
            const uint32_t a = ix[0], b = ix[1];
            if (a > lo) lo = a;
            if (b < hi) hi = b;
            if (lo > hi) lo = hi;
        }
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (J.seq[mid].match_pos + J.seq[mid].ml > s) hi = mid; else lo = mid + 1;
        }
        uint32_t blocker = 0xFFFFFFFFu;
        for (uint32_t j = lo; j < i && J.seq[j].match_pos < e; j++) {
            const uint32_t dn = J.seq_done[j];
            if (dn == 0 || dn >= round) { blocker = j; break; }
        }
        if (blocker == 0xFFFFFFFFu) { verdict = 1; break; }
        const SeqRec& Q = J.seq[blocker];
        if (hop == LZ_HOPS || off < ml || Q.match_pos > s || e > Q.match_pos + Q.ml) { J.lz_blocker[i] = blocker; break; }      // cannot redirect: wait
        const uint32_t add = resolve_offset(J, Q.off, Q.block);
        if (add > 0x7FFFFFFFu - off) { J.lz_blocker[i] = blocker; break; }     // (the sum is stored in R.off: bit 31 would read as OFF_SYMBOLIC)
        off += add;
    }
    if (off != off0) R.off = off;                                      // keep the shortcut for later rounds (and for others)
    return verdict;
}

// One round over a list of matches: items [0, n) of `list` (or the identity when list == nullptr).  Matches that still
// have to wait are appended to `next` (count in *next_n).
constexpr int LZ_U = 4;                             // list entries per thread and step: their "still blocked?" loads are in flight together

__device__ __forceinline__ void lz_round(const JobDev& J, const uint32_t* list, uint32_t n, uint32_t round, uint32_t* next, uint32_t* next_n,
                                         uint32_t first, uint32_t stride,
                                         uint32_t* q_n, uint64_t* q_d, uint32_t* q_off, uint32_t* q_ml, uint32_t* q_i) {
    const int tid = threadIdx.x, lane = tid & 31;
    for (uint32_t base = first; base < n; base += stride * LZ_U) {   // `base` is CTA-uniform
        if (tid == 0) *q_n = 0;
        __syncthreads();
        // (a) which of this thread's entries are worth a look: not executed yet, and not waiting for a match that is still
        //     unfinished.  LZ_U independent chains of two loads; in deep rounds ~98 % of the entries stop here.
        uint32_t idx[LZ_U];
        bool look[LZ_U], pend[LZ_U];
#pragma unroll
        for (int u = 0; u < LZ_U; u++) {
            const uint32_t k = base + (uint32_t)u * stride + (uint32_t)tid;
            look[u] = false; pend[u] = false; idx[u] = 0;
            if (k < n) {
                const uint32_t i = list ? list[k] : k;
                idx[u] = i;
                if (J.seq_done[i] == 0) {
                    look[u] = true;
                    if (round > 1u + J.lz_flow_early) {
                        const uint32_t b = J.lz_blocker[i];
                        if (b != 0xFFFFFFFFu) { const uint32_t dn = J.seq_done[b]; if (dn == 0 || dn >= round) { look[u] = false; pend[u] = true; } }
                    }
                }
            }
        }
        // (b) the full readiness probe, and the copy if the match may run
#pragma unroll
        for (int u = 0; u < LZ_U; u++) {
            if (look[u]) {
                uint64_t d; uint32_t off, ml;
                const int v = lz_try(J, idx[u], round, d, off, ml);
                if (v == 0) pend[u] = true;
                else if (v == 1) {
                    if (ml <= LZ_SHORT) { copy_match(J.out, d, off, ml, 0, 1); J.seq_done[idx[u]] = round; }
                    else {
                        const uint32_t slot = atomicAdd(q_n, 1u);
                        if (slot < (uint32_t)LZ_CTA) { q_d[slot] = d; q_off[slot] = off; q_ml[slot] = ml; q_i[slot] = idx[u]; }
                        else pend[u] = true;                         // (queue full: next round)
                    }
                }
            }
        }
        // (c) entries that stay pending go to the next round's list
#pragma unroll
        for (int u = 0; u < LZ_U; u++) {
            const uint32_t pb = __ballot_sync(0xFFFFFFFFu, pend[u]);
            uint32_t wbase = 0;
            if (lane == 0 && pb) wbase = atomicAdd(next_n, (uint32_t)__popc(pb));
            wbase = __shfl_sync(0xFFFFFFFFu, wbase, 0);
            if (pend[u]) next[wbase + __popc(pb & ((1u << lane) - 1u))] = idx[u];
        }
        __syncthreads();
        uint32_t nq = *q_n;
        if (nq > (uint32_t)LZ_CTA) nq = LZ_CTA;
        // long matches: one warp each; the very long ones (N stretches: offset 1, ~100 KB) by the whole CTA
        for (uint32_t t = (uint32_t)tid >> 5; t < nq; t += LZ_CTA / 32)
            if (q_ml[t] <= LZ_WARP_MAX) copy_long_match(J.out, q_d[t], q_off[t], q_ml[t], lane, 32);
        for (uint32_t t = 0; t < nq; t++)
            if (q_ml[t] > LZ_WARP_MAX) copy_long_match(J.out, q_d[t], q_off[t], q_ml[t], tid, LZ_CTA);
        if ((uint32_t)tid < nq) J.seq_done[q_i[tid]] = round;
        __syncthreads();
    }
}

#define LZ_SHARED_QUEUE \
    __shared__ uint32_t q_n; __shared__ uint64_t q_d[LZ_CTA]; __shared__ uint32_t q_off[LZ_CTA], q_ml[LZ_CTA], q_i[LZ_CTA]

// Round 1: every match of the job, one thread each.
__global__ void __launch_bounds__(LZ_CTA, 4) k_lz_first(JobDev J) {
    LZ_SHARED_QUEUE;
    lz_round(J, nullptr, (uint32_t)J.n_seq, 1u + J.lz_flow_early, J.lz_list[0], &J.lz_count[0], blockIdx.x * LZ_CTA, gridDim.x * LZ_CTA,
             &q_n, q_d, q_off, q_ml, q_i);
}

// Rounds 2..: persistent cooperative kernel over the worklist.  Three lists rotate (read / append / being cleared), so a
// round needs a single grid barrier.
__global__ void __launch_bounds__(LZ_CTA) k_lz_resolve(JobDev J) {
    LZ_SHARED_QUEUE;
    uint32_t cur = 0;
    const uint32_t r0 = J.lz_flow_early;                             // (round numbers are one higher after an early k_lz_flow, whose matches carry 1)
    for (uint32_t round = 2 + r0;; round++) {
        const uint32_t nxt = cur == 2 ? 0 : cur + 1, clr = nxt == 2 ? 0 : nxt + 1;
        const uint32_t n = J.lz_count[cur];                          // stable: written before the last grid barrier
        if (blockIdx.x == 0 && threadIdx.x == 0) { *J.lz_rounds = round - 1 - r0; if (round - 2 - r0 < 24) J.lz_pending[round - 2 - r0] = n; }
        if (n == 0) break;
        if (blockIdx.x == 0 && threadIdx.x == 0) J.lz_count[clr] = 0; // append target of the NEXT round; idle in this one
        lz_round(J, J.lz_list[cur], n, round, J.lz_list[nxt], &J.lz_count[nxt], blockIdx.x * LZ_CTA, gridDim.x * LZ_CTA,
                 &q_n, q_d, q_off, q_ml, q_i);
        NAF_GRID_SYNC();                                             // copies, list appends and the cleared counter are visible
        const uint32_t n_next = J.lz_count[nxt];
        cur = nxt;
        // A round costs a grid barrier (~3 us) plus a pass over the worklist, whatever it resolves.  At the current rate
        // the rest would take n_next / progress more rounds; when that costs more than k_lz_finish (whose cost depends on
        // the bytes of the frame, not on the depth of the chain), the section is text-like: hand it over.
        const uint32_t progress = n - n_next;
        const uint64_t round_ns = 5000 + n_next / 25;                      // measured: ~30 us per round at 600 K entries (most of them one load: still blocked)
        // chains of a few dozen generations (at this rate the rest needs 8..256 more rounds): k_lz_flow, where a generation
        // costs a visibility latency instead of a round.  Endless chains (text-like sections: thousands of rounds) go to the finisher.
        if (round >= LZ_MIN_ROUNDS + r0 && n_next > LZ_MIN_PENDING && J.lz_flow_on) {
            const uint64_t est = (uint64_t)n_next / (progress ? progress : 1u);
            if ((est >= 8 && est <= 256) || J.lz_flow_on == 2u) {       // (2: tests force the kernel on small inputs)
                if (blockIdx.x == 0 && threadIdx.x == 0) *J.lz_flow = 1;
                break;
            }
        }
        if (round >= LZ_MIN_ROUNDS + r0 && n_next > LZ_MIN_PENDING &&
            (uint64_t)n_next * round_ns > (uint64_t)(progress ? progress : 1u) * J.fin_cost_us * 1000u) {
            if (blockIdx.x == 0 && threadIdx.x == 0) *J.lz_handover = round - r0;
            break;
        }
    }
}

// k_lz_flow: the matches that k_lz_resolve's rounds leave when the dependency chains are DEEP BUT NOT ENDLESS -- a diverged repeat
// family in a chromosome (cfg3): 78 generations of matches, ~2 % of the pending ones becoming ready per round, every round a
// grid barrier and a pass over the worklist (25 us each, 1.9 ms).  Here the matches are taken IN ORDER, 32 per warp by a ticket,
// and a match simply waits for the matches its source range needs (they have smaller indices: finished, or held by a warp
// that took an earlier ticket and is therefore running -- no deadlock, no co-residency requirement beyond "a warp that holds
// a ticket runs").  A generation then costs one visibility latency (~1-2 us) instead of a round.  The waiting is a CONVERGENT
// loop of the warp (every lane polls once per iteration; no lane ever spins inside a divergent branch that a peer lane would
// have to leave first), bounded by a deadline: a section whose chain is as long as the section (quality strings) would
// serialise here, so k_lz_resolve only chooses this kernel when the remaining depth looks small, and when the deadline
// passes anyway the kernel gives up and hands what is left to the byte-level finisher.
__device__ __forceinline__ unsigned long long flow_now_ns() {
#if defined(__CUDA_ARCH__)
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t;
#else
    return 0ull;
#endif
}

constexpr int LZF_T = 256;

// `early`: the kernel runs BEFORE the rounds, over every match, for jobs of a few thousand to a few ten thousand matches (one
// genome alone): their three or four generations then cost a launch, a probe and a few visibility latencies instead of a launch
// plus a grid barrier and a dozen dependent loads per round (one cfg2 archive: 78 -> see profiles).  Its deadline is short; what it
// leaves (a text-like section) goes through k_lz_first / k_lz_resolve as before, which skip what is done.
constexpr unsigned long long LZF_EARLY_NS = 60000ull;

__global__ void __launch_bounds__(LZF_T) k_lz_flow(JobDev J, int early) {
    if (!early && *J.lz_flow == 0) return;
    volatile uint32_t* done = J.seq_done;
    volatile uint32_t* abort_flag = J.lz_flow + (early ? 4 : 2);
    uint32_t* const ticket = J.lz_flow + (early ? 3 : 1);
    const int lane = threadIdx.x & 31;
    const uint32_t n = (uint32_t)J.n_seq;
    // "done" value of the matches executed here: to the rounds that may follow the early run, a match is finished when its value is
    // below their round number (they start at 2 then, k_lz_first); nothing runs after the late one
    const uint32_t stamp = early ? 1u : 0x7FFFFFFFu;
    const unsigned long long deadline = flow_now_ns() + (early ? LZF_EARLY_NS : (unsigned long long)J.fin_cost_us * 1000ull);
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(ticket, 32u);
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base >= n) return;
        const uint32_t i = base + (uint32_t)lane;
        bool active = i < n && done[i] == 0;
        uint64_t d = 0, e = 0;
        uint32_t off = 0, ml = 0, j = 0, frame = 0;
        if (active) {
            const SeqRec& R = J.seq[i];
            const BlockDesc& B = J.blocks[R.block];
            frame = B.frame;
            const FrameDesc& F = J.frames[frame];
            if (J.frame_bad[frame]) { done[i] = stamp; active = false; }
            else {
                ml = R.ml; d = R.match_pos; off = resolve_offset(J, R.off, R.block);       // (possibly redirected by the rounds: any value it had is valid)
                if (off == 0 || (uint64_t)off > d - F.dst_off) { flag_error(J, frame, zc::E_OFFSET); done[i] = stamp; active = false; }
                else {
                    const uint64_t sp = d - off;
                    e = off < ml ? d : sp + ml;                                            // external source range [sp, e)
                    uint32_t lo = F.first_seq, hi = i;
                    const uint32_t* ix = J.lz_idx + (size_t)J.fin_chunk_first[frame] * LZ_IDX_PER_CHUNK + frame + ((sp - F.dst_off) >> LZ_IDX_SHIFT);
                    const uint32_t a = ix[0], b = ix[1];
                    if (a > lo) lo = a;
                    if (b < hi) hi = b;
                    if (lo > hi) lo = hi;
                    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (J.seq[mid].match_pos + J.seq[mid].ml > sp) hi = mid; else lo = mid + 1; }
                    j = lo;                                                                // first match that ends after the start of my source
                }
            }
        }
        uint32_t idle = 0;
        while (__any_sync(0xFFFFFFFFu, active)) {
            bool ready = false;
            if (active) {
                // the cursor moves over the finished matches of my source range; it stops at the first unfinished one
                while (j < i && J.seq[j].match_pos < e && done[j] != 0) j++;
                ready = !(j < i && J.seq[j].match_pos < e);
            }
            const uint32_t rb = __ballot_sync(0xFFFFFFFFu, ready);
            if (rb) {
                // the ready matches one after the other, each copied by the WHOLE warp with its loads issued before its stores
                // (a lane copying its own 150 bytes pays a round trip to memory per 8 of them, and the next generation waits for it)
                __threadfence();                                                           // their bytes before mine
                for (uint32_t m = rb; m; m &= m - 1) {
                    const int src = __ffs((int)m) - 1;
                    const uint64_t dd = ((uint64_t)__shfl_sync(0xFFFFFFFFu, (uint32_t)(d >> 32), src) << 32) | __shfl_sync(0xFFFFFFFFu, (uint32_t)d, src);
                    const uint32_t oo = __shfl_sync(0xFFFFFFFFu, off, src), mm = __shfl_sync(0xFFFFFFFFu, ml, src);
                    if (oo >= mm) copy_g2g_1rt<4>(J.out + dd, J.out + dd - oo, mm, lane, 32);
                    else copy_long_match(J.out, dd, oo, mm, lane, 32);
                }
                __threadfence();
                if (ready) { done[i] = stamp; active = false; }
                idle = 0;
                continue;
            }
            // nobody moved: the warp waits for matches of other warps.  Check the clock now and then.
            if ((++idle & 63u) == 0) {
                uint32_t stop = 0;
                if (lane == 0) { stop = *abort_flag; if (!stop && flow_now_ns() > deadline) { *abort_flag = 1; stop = 1; } }
                if (__shfl_sync(0xFFFFFFFFu, stop, 0)) {
                    if (lane == 0 && !early) atomicMax(J.lz_handover, *J.lz_rounds + 1u);  // what is left goes to k_lz_finish (early: to the rounds)
                    return;
                }
            }
#if defined(__CUDA_ARCH__)
            __nanosleep(100);
#endif
        }
        uint32_t stop = 0;
        if (lane == 0) stop = *abort_flag;
        if (__shfl_sync(0xFFFFFFFFu, stop, 0)) { if (lane == 0 && !early) atomicMax(J.lz_handover, *J.lz_rounds + 1u); return; }     // (uniform)
    }
}

// k_lz_small: the whole match stage of a SMALL job (one bacterial genome: a few hundred to a few thousand matches) in one CTA.
// The rounds above cost a kernel launch (round 1) or a grid barrier (the others) plus a dozen dependent global loads each --
// list entry, record, blocker's flag, index cells, bisection steps: ~8 us per round whatever the number of matches, 85 us for
// the 107 matches and 7 rounds of the cfg1 fixture.  Here the records (position, length, resolved offset, done round, frame)
// sit in shared memory, a round is a pass of the CTA over its pending matches and a __syncthreads, and only the copies touch
// global memory.  Same readiness rule, same redirects, same hand-over to the finisher as lz_try / k_lz_resolve.
constexpr uint32_t LZS_MAX = 8192;               // matches (the host sets J.lz_small when the job has no more, and an arena below 4 GB)
constexpr int LZS_T = 1024;
__host__ __device__ constexpr uint32_t lzs_smem_bytes(uint32_t n) { return ((n + 3u) & ~3u) * 24u; }

__global__ void __launch_bounds__(LZS_T) k_lz_small(JobDev J) {
    NAF_DYN_SMEM(uint32_t, lzs);
    const uint32_t n = (uint32_t)J.n_seq, np = (n + 3u) & ~3u;
    uint32_t* pos = lzs;                          // destination, relative to J.out
    uint32_t* mlen = pos + np;
    uint32_t* moff = mlen + np;                   // resolved offset (redirects add to it)
    uint16_t* done = (uint16_t*)(moff + np);      // 0: pending, else the round that copied (or rejected) it
    uint16_t* frm = done + np;
    uint32_t* q_i = (uint32_t*)(frm + np);        // the matches a round may copy: index, then the offset to copy with
    uint32_t* q_off = q_i + np;
    __shared__ uint32_t q_n, q_big, s_pending[3];      // (three counters rotate: the one a round adds to is cleared two rounds earlier, while nobody reads it)
    const int tid = threadIdx.x, lane = tid & 31;
    for (uint32_t i = tid; i < n; i += LZS_T) {
        const SeqRec& R = J.seq[i];
        const BlockDesc& B = J.blocks[R.block];
        pos[i] = (uint32_t)R.match_pos; mlen[i] = R.ml; frm[i] = (uint16_t)B.frame;
        moff[i] = resolve_offset(J, R.off, R.block);
        done[i] = J.frame_bad[B.frame] ? 1 : 0;
    }
    if (tid == 0) { s_pending[0] = s_pending[1] = s_pending[2] = 0; }
    __shared__ uint32_t fr_first[64], fr_off[64];            // a single archive has a handful of frames: their first match and offset
    const bool fr_cached = J.n_frames <= 64u;
    if (fr_cached && (uint32_t)tid < J.n_frames) { fr_first[tid] = J.frames[tid].first_seq; fr_off[tid] = (uint32_t)J.frames[tid].dst_off; }
    __syncthreads();
    long long t_probe = 0, t_copy = 0, t0 = 0, t_begin = 0;      // (cycle accounting with NAFGPU_DEBUG_HUF=1)
    SEQ_CLK(t_begin);
    uint32_t prev_pending = n, handover = 0, round = 1;
    for (;; round++) {
        if (tid == 0) { q_n = 0; q_big = 0; s_pending[(round + 1) % 3] = 0; }
        __syncthreads();
        SEQ_CLK(t0);
        uint32_t mine = 0;
        for (uint32_t i = tid; i < n; i += LZS_T) {
            if (done[i]) continue;
            const uint32_t f = frm[i];
            const uint32_t f_first = fr_cached ? fr_first[f] : J.frames[f].first_seq, f_off = fr_cached ? fr_off[f] : (uint32_t)J.frames[f].dst_off;
            const uint32_t d = pos[i], ml = mlen[i];
            uint32_t off = moff[i];
            int verdict = 0;
            for (int hop = 0; hop <= LZ_HOPS; hop++) {
                if (off == 0 || off > d - f_off) { flag_error(J, f, zc::E_OFFSET); verdict = 2; break; }
                const uint32_t sp = d - off, e = off < ml ? d : sp + ml;      // external source range [sp, e)
                uint32_t lo = f_first, hi = i;
                while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (pos[mid] + mlen[mid] > sp) hi = mid; else lo = mid + 1; }
                uint32_t blocker = 0xFFFFFFFFu;
                for (uint32_t j = lo; j < i && pos[j] < e; j++) {
                    const uint32_t dn = done[j];
                    if (dn == 0 || dn >= round) { blocker = j; break; }
                }
                if (blocker == 0xFFFFFFFFu) { verdict = 1; break; }
                if (hop == LZ_HOPS || off < ml || pos[blocker] > sp || e > pos[blocker] + mlen[blocker]) break;      // cannot redirect: wait
                off += moff[blocker];
            }
            moff[i] = off;                              // (only this thread writes it; others read it for their redirects: any
                                                        //  value it ever had is a valid offset of this match)
            if (verdict == 2) done[i] = (uint16_t)round;
            else if (verdict == 1) {
                // two queues in one array: matches a warp copies whole from the front, long disjoint ones (copied in pieces by all
                // warps) from the back
                const bool big = ml > 2048u && off >= ml;
                const uint32_t slot = big ? np - 1u - atomicAdd(&q_big, 1u) : atomicAdd(&q_n, 1u);
                q_i[slot] = i; q_off[slot] = off;
            }
            else mine++;
        }
        if (mine) atomicAdd(&s_pending[round % 3], mine);
        __syncthreads();
        SEQ_LAP(t_probe, t0);
        // the copies of the round, a warp per match (a thread copying its own 40 bytes pays a round trip to memory per 8 of
        // them, and the round lasts as long as its slowest copy); the long disjoint ones in 2 KB pieces dealt to all warps.
        // No barrier in between: every piece is one round trip, all in flight together.
        const uint32_t nq = q_n, nbig = q_big;
        {
            const uint32_t warp = (uint32_t)tid >> 5, NW = LZS_T / 32;
            for (uint32_t t = warp; t < nq; t += NW) {
                const uint32_t i = q_i[t], ml = mlen[i], off = q_off[t];
                if (off >= ml) copy_g2g<4>(J.out + pos[i], J.out + pos[i] - off, ml, lane, 32);
                else copy_long_match(J.out, pos[i], off, ml, lane, 32);
            }
            for (uint32_t t = 0; t < nbig; t++) {
                const uint32_t i = q_i[np - 1u - t], ml = mlen[i], off = q_off[np - 1u - t], d = pos[i];
                for (uint32_t pc = (warp + NW - (t & (NW - 1))) & (NW - 1); pc * 2048u < ml; pc += NW) {
                    const uint32_t b = pc * 2048u, len = ml - b < 2048u ? ml - b : 2048u;
                    copy_g2g<4>(J.out + d + b, J.out + d - off + b, len, lane, 32);
                }
            }
        }
        __syncthreads();                                // (the done flags are written after every copy of the round)
        SEQ_LAP(t_copy, t0);
        for (uint32_t t = tid; t < nq; t += LZS_T) done[q_i[t]] = (uint16_t)round;
        for (uint32_t t = tid; t < nbig; t += LZS_T) done[q_i[np - 1u - t]] = (uint16_t)round;
        __syncthreads();
        const uint32_t pending = s_pending[round % 3];
        if (tid == 0 && round - 1 < 24) J.lz_pending[round - 1] = pending;             // (matches still waiting after round 1, 2, ...)
        if (pending == 0) break;
        // the hand-over rule of k_lz_resolve, with this kernel's cost of a round
        const uint32_t progress = prev_pending - pending;
        if (round >= LZ_MIN_ROUNDS && pending > LZ_MIN_PENDING && round < 60000u &&
            (uint64_t)pending * (1500u + pending / 2u) > (uint64_t)(progress ? progress : 1u) * J.fin_cost_us * 1000u) { handover = round; break; }
        if (round >= 60000u) { handover = round; break; }             // (16-bit round numbers; unreachable with 8192 matches)
        prev_pending = pending;
    }
    // what the finisher and the statistics read
    for (uint32_t i = tid; i < n; i += LZS_T) J.seq_done[i] = done[i];
    if (tid == 0) { *J.lz_rounds = round; if (handover) *J.lz_handover = handover; }
    long long t_end = 0;
    SEQ_CLK(t_end);
    if (J.debug_seq && tid == 0) { J.debug_seq[5] = (unsigned long long)t_probe; J.debug_seq[6] = (unsigned long long)t_copy; J.debug_seq[7] = (unsigned long long)(t_end - t_begin); }
}

// k_lz_finish / k_lz_finish2: what k_lz_resolve leaves behind when its rounds stop paying (text-like sections -- quality
// strings, ids -- where nearly every match feeds the next one: a dependency chain as long as the section has matches).
// Walking such a chain in order costs hundreds of cycles per match on a GPU; instead the chain is cut at BYTE level, where
// an LZ77 stream is a forest: every byte of a pending match points at the byte `off` behind it (the periodic extension
// for an overlapping match), every other byte is a root.
//
// Level 1 (k_lz_finish): the frames are cut into 64 KB chunks, ALL chunks processed in parallel, one at a time per CTA in
// shared memory: 16-bit chunk-relative parents, in-place pointer jumping (ptr[e] = ptr[ptr[e]]) to the roots in
// log2(depth) steps.  A root is either final (literal, finished match): its bytes are written now; or it is a byte whose
// source lies BELOW the chunk, which may itself still be unresolved: for every byte hanging off such a root the distance
// back to that source goes to fin_g (u32 per byte of the chunk; 0 = final).
// Level 2 (k_lz_finish2, cooperative): pointer jumping over fin_g across chunks.  A byte whose source is final takes its
// value; otherwise it adopts its source's source (dist += dist[source]).  Sources always lie in an earlier chunk, so the
// depth is at most the number of chunks of the frame: <= log2 of that many rounds, one grid barrier each.
constexpr uint32_t FIN_C = 65536;        // chunk bytes (16-bit pointers); frame_walk.h uses the same value for the chunk table
constexpr uint32_t FIN_T = 1024;         // threads
constexpr uint32_t FIN_U = 4;            // matches per thread and scan step (independent loads in flight)
constexpr uint32_t FIN_INLINE = 64;      // longer pieces are set up by the whole CTA
constexpr uint32_t FIN_SMEM = FIN_C + FIN_C * 2 + FIN_C / 8 + FIN_T * 20;
constexpr int FIN2_T = 256;

// One byte of a pending match: chunk-relative e, parent at chunk-relative (signed) s.  Parents below the chunk: the byte
// becomes an external root, its distance to the source goes to g[e].
__device__ __forceinline__ void fin_byte(uint16_t* ptr, uint32_t* extbit, uint32_t* g, uint32_t e, int32_t s) {
    if (s >= 0) ptr[e] = (uint16_t)s;
    else { g[e] = (uint32_t)((int32_t)e - s); atomicOr(&extbit[e >> 5], 1u << (e & 31)); }
}

// frame that owns chunk c: last f with chunk_first[f] <= c < chunk_first[f + 1]
__device__ __forceinline__ uint32_t fin_frame_of(const JobDev& J, uint32_t c) {
    uint32_t lo = 0, hi = J.n_frames;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (J.fin_chunk_first[mid] <= c) lo = mid; else hi = mid; }
    return lo;
}

__global__ void __launch_bounds__(FIN_T) k_lz_finish(JobDev J) {
    if (*J.lz_handover == 0) return;                // the rounds finished everything (the normal case)
    NAF_DYN_SMEM(unsigned char, fin_smem);
    uint8_t* val = fin_smem;                                   // [FIN_C] chunk bytes
    uint16_t* ptr = (uint16_t*)(fin_smem + FIN_C);             // [FIN_C] chunk-relative parent; self = root
    uint32_t* extbit = (uint32_t*)(fin_smem + FIN_C * 3);      // [FIN_C / 32] roots whose source lies below the chunk
    uint32_t* q_rel = extbit + FIN_C / 32;                     // [FIN_T] long pieces: first chunk-relative byte,
    uint32_t* q_len = q_rel + FIN_T;                           //         length,
    uint32_t* q_off = q_len + FIN_T;                           //         match offset,
    uint32_t* q_m0 = q_off + FIN_T;                            //         first byte of the piece within the match,
    uint32_t* q_ml = q_m0 + FIN_T;                             //         match length
    __shared__ uint32_t s_f, s_mi, s_q, s_bad, s_unres;
    const uint32_t tid = threadIdx.x;

    for (uint32_t c = blockIdx.x; c < J.fin_total_chunks; c += gridDim.x) {
        __syncthreads();
        if (tid == 0) {
            const uint32_t f = fin_frame_of(J, c);
            s_f = f; s_bad = 0; s_unres = 0;
            // first match of the frame that ends after the start of the chunk: k_lz_index's cell for the chunk's first 4 KB
            // (a bisection over the frame's matches here cost 24 dependent loads with the CTA waiting)
            if (!J.lz_small) s_mi = J.frames[f].n_seq ? J.lz_idx[(size_t)c * LZ_IDX_PER_CHUNK + f] : J.frames[f].first_seq;
            else {                                   // (a small job's rounds ran in k_lz_small: no index)
                const uint64_t cs = J.frames[f].dst_off + (uint64_t)(c - J.fin_chunk_first[f]) * FIN_C;
                uint32_t lo = J.frames[f].first_seq, hi = lo + J.frames[f].n_seq;
                while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (J.seq[mid].match_pos + J.seq[mid].ml > cs) hi = mid; else lo = mid + 1; }
                s_mi = lo;
            }
        }
        __syncthreads();
        const uint32_t f = s_f, mi = s_mi;
        if (J.frame_bad[f]) continue;
        const uint64_t f0 = J.frames[f].dst_off, fend = f0 + J.frames[f].dst_size;
        const uint32_t end = J.frames[f].first_seq + J.frames[f].n_seq;
        const uint64_t c0 = f0 + (uint64_t)(c - J.fin_chunk_first[f]) * FIN_C;
        const uint64_t c1 = (c0 + FIN_C < fend) ? c0 + FIN_C : fend;
        const uint32_t cn = (uint32_t)(c1 - c0);
        uint8_t* out_c0 = J.out + c0;
        uint32_t* g = J.fin_g + J.fin_g_base[f] + (size_t)(c - J.fin_chunk_first[f]) * FIN_C;
        // any pending match in this chunk?  (most chunks of a job have none)
        bool mine = false;
        for (uint32_t base = mi;; base += FIN_T) {
            const uint32_t i = base + tid;
            bool stop = i >= end;
            if (!stop) {
                const SeqRec& R = J.seq[i];
                if (R.match_pos >= c1) stop = true;
                else if (J.seq_done[i] == 0) mine = true;
            }
            if (__syncthreads_or(stop || mine)) break;
        }
        if (!__syncthreads_or(mine)) continue;
        // chunk bytes as they stand (literals and finished matches are final, pending bytes are garbage), self pointers,
        // no external roots, all distances zero
        for (uint32_t e = tid * 16; e < FIN_C; e += FIN_T * 16) {
            uint32_t* p2 = (uint32_t*)(ptr + e);
#pragma unroll
            for (uint32_t k = 0; k < 8; k++) p2[k] = (e + 2 * k) | ((e + 2 * k + 1) << 16);
            if (e < cn) {                                                    // (frames are 16-entry aligned in fin_g; the arena is padded)
                *(uint4*)(val + e) = __ldcg((const uint4*)(out_c0 + e));
#pragma unroll
                for (uint32_t k = 0; k < 4; k++) ((uint4*)(g + e))[k] = make_uint4(0, 0, 0, 0);
            }
        }
        for (uint32_t e = tid; e < FIN_C / 32; e += FIN_T) extbit[e] = 0;
        __syncthreads();
        // pending matches that intersect the chunk
        for (uint32_t base = mi;; base += FIN_T * FIN_U) {
            if (tid == 0) s_q = 0;
            __syncthreads();
            uint64_t pos[FIN_U];
            uint32_t ml[FIN_U], ov[FIN_U], blk[FIN_U];
            bool pend[FIN_U];
#pragma unroll
            for (uint32_t j = 0; j < FIN_U; j++) {
                const uint32_t i = base + j * FIN_T + tid;
                pos[j] = ~0ull; ml[j] = 0; ov[j] = 0; blk[j] = 0; pend[j] = false;
                if (i < end) {
                    const SeqRec& R = J.seq[i];
                    pos[j] = R.match_pos; ml[j] = R.ml; ov[j] = R.off; blk[j] = R.block; pend[j] = J.seq_done[i] == 0;
                }
            }
            bool stop = false;
#pragma unroll
            for (uint32_t j = 0; j < FIN_U; j++) {
                const uint32_t i = base + j * FIN_T + tid;
                if (i >= end || pos[j] >= c1) stop = true;
                else if (pend[j] && pos[j] + ml[j] > c0) {
                    const uint32_t off = resolve_offset(J, ov[j], blk[j]);
                    if (off == 0 || (uint64_t)off > pos[j] - f0 || off > 0x7F000000u) { flag_error(J, f, zc::E_OFFSET); s_bad = 1; }
                    else {
                        const uint64_t b0 = pos[j] > c0 ? pos[j] : c0, b1 = pos[j] + ml[j] < c1 ? pos[j] + ml[j] : c1;
                        const uint32_t rel = (uint32_t)(b0 - c0), len = (uint32_t)(b1 - b0), m0 = (uint32_t)(b0 - pos[j]);
                        const int32_t srel = (int32_t)((int64_t)(pos[j] - off) - (int64_t)c0);   // |srel| < 2^31: offsets are capped above
                        if (len > FIN_INLINE) {
                            const uint32_t slot = atomicAdd(&s_q, 1u);
                            q_rel[slot] = rel; q_len[slot] = len; q_off[slot] = off; q_m0[slot] = m0; q_ml[slot] = ml[j];
                        } else if (off >= ml[j]) {
                            int32_t sp = srel + (int32_t)m0;
                            for (uint32_t k = 0; k < len; k++, sp++) fin_byte(ptr, extbit, g, rel + k, sp);
                        } else {
                            uint32_t r = m0 % off;
                            for (uint32_t k = 0; k < len; k++) { fin_byte(ptr, extbit, g, rel + k, srel + (int32_t)r); if (++r == off) r = 0; }
                        }
                    }
                }
            }
            const int all_stop = __syncthreads_or(stop);
            const uint32_t nq = s_q;
            for (uint32_t t = 0; t < nq; t++) {
                const uint32_t rel = q_rel[t], len = q_len[t], off = q_off[t], m0 = q_m0[t], mlen = q_ml[t];
                const int32_t srel = (int32_t)rel - (int32_t)m0 - (int32_t)off;
                for (uint32_t k = tid; k < len; k += FIN_T)
                    fin_byte(ptr, extbit, g, rel + k, srel + (int32_t)(off < mlen ? (m0 + k) % off : m0 + k));
            }
            if (all_stop) break;
            __syncthreads();                                                // queue drained before it is refilled
        }
        __syncthreads();
        if (s_bad) continue;                                                // (uniform; the frame is flagged)
        // pointer jumping, in place: a pointer only ever moves to an ancestor, roots never move
        for (;;) {
            bool changed = false;
            for (uint32_t e = tid; e < cn; e += FIN_T) {
                const uint32_t p = ptr[e];
                if (p != e) { const uint32_t pp = ptr[p]; if (pp != p) { ptr[e] = (uint16_t)pp; changed = true; } }
            }
            if (!__syncthreads_or(changed)) break;
        }
        // bytes under a final root take its value now; bytes under an external root get the distance to its source
        uint32_t unres = 0;
        for (uint32_t e = tid; e < cn; e += FIN_T) {
            const uint32_t p = ptr[e];
            const bool ext = (extbit[p >> 5] >> (p & 31)) & 1u;
            if (p != e) {
                if (ext) { g[e] = e - p; unres++; }                         // same value as its root p, which level 2 resolves
                else out_c0[e] = val[p];                                    // roots are not written here: no hazard
            } else if (ext) unres++;
        }
        if (unres) atomicAdd(&s_unres, unres);
        __syncthreads();
        if (s_unres) {                                                      // (uniform) the chunk's external roots, for level 2
            uint32_t* xb = J.fin_ext + (size_t)c * (FIN_C / 32);
            for (uint32_t e = tid; e < FIN_C / 32; e += FIN_T) xb[e] = extbit[e];
        }
        if (tid == 0 && s_unres) { J.fin_chunk_flag[c] = 1; atomicAdd(J.fin_unresolved, s_unres); }
    }
}

// Level 2: see above.  Cooperative.  Only the ROOTS take part in the rounds (the chunk's bitmap of external roots, compacted
// per 8 KB tile): in a text-like section the offsets are a few hundred bytes, so a chunk has a few hundred roots at its
// start and 60 000 bytes hanging off them -- jumping every byte (round 1 of this kernel's life) moved 205 M distances per
// round for a 10^6-read archive, 15 ms; the roots are 1.5 M.  A last pass gives every other byte the value of its root.
constexpr uint32_t FIN2_U = 8;                   // roots per thread between two fences
constexpr uint32_t FIN2_TILE = FIN2_T * 32;      // bytes of a chunk whose roots are compacted at a time (one bitmap word per thread)

__global__ void __launch_bounds__(FIN2_T) k_lz_finish2(JobDev J) {
    if (*J.lz_handover == 0 || *J.fin_unresolved == 0) return;
    __shared__ uint32_t s_left, s_wsum[FIN2_T / 32];
    __shared__ uint16_t s_root[FIN2_TILE];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    volatile uint32_t* G = J.fin_g;
    volatile uint32_t* flag = J.fin_chunk_flag;       // 1: unresolved roots; 2: roots final, the bytes under them not yet written; 0: final
    for (uint32_t round = 0;; round++) {
        // three counters rotate: this round adds to `cur` and reads it after the barrier (a slow CTA as late as during the next
        // round); the NEXT round's counter is cleared now, while nobody reads it or adds to it
        const uint32_t cur = round % 3, clr = (round + 1) % 3;
        if (blockIdx.x == 0 && tid == 0) J.fin_count[clr] = 0;
        uint32_t left_total = 0;
        for (uint32_t c = blockIdx.x; c < J.fin_total_chunks; c += gridDim.x) {
            if (flag[c] != 1) continue;                                     // (uniform)
            __syncthreads();
            if (tid == 0) s_left = 0;
            const uint32_t f = fin_frame_of(J, c);
            const uint32_t cf = J.fin_chunk_first[f];
            const size_t gb = (size_t)J.fin_g_base[f];                       // the frame's entries in fin_g
            const uint64_t f0 = J.frames[f].dst_off;
            const uint64_t crel = (uint64_t)(c - cf) * FIN_C;               // chunk start relative to the frame
            const uint32_t* xb = J.fin_ext + (size_t)c * (FIN_C / 32);
            uint32_t left = 0;
            for (uint32_t t0 = 0; t0 < FIN_C; t0 += FIN2_TILE) {
                const uint32_t word = xb[(t0 >> 5) + tid];
                if (!__syncthreads_or(word != 0)) continue;                  // (roots sit at the start of a chunk: most tiles have none)
                // compact the tile's roots: exclusive scan of the words' bit counts
                const uint32_t cnt = __popc(word);
                uint32_t inc = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, inc, d); if ((int)lane >= d) inc += v; }
                if (lane == 31) s_wsum[warp] = inc;
                __syncthreads();
                uint32_t before = inc - cnt, total = 0;
                for (uint32_t w = 0; w < FIN2_T / 32; w++) { const uint32_t v = s_wsum[w]; if (w < warp) before += v; total += v; }
                for (uint32_t m = word, k = before; m; m &= m - 1, k++) s_root[k] = (uint16_t)(t0 + tid * 32 + (uint32_t)(__ffs(m) - 1));
                __syncthreads();
                // FIN2_U roots per thread at a time, so that the two fences (sources seen final -> their bytes; my bytes -> my
                // zeroed distances) are paid once per batch instead of once per root (10.4 ms -> see profiles for a 10^6-read archive)
                for (uint32_t k0 = tid; k0 < total; k0 += FIN2_T * FIN2_U) {
                    uint32_t re[FIN2_U], rd[FIN2_U], rs[FIN2_U];            // root, its distance, what to do: 0 nothing, 1 take the source's byte, 2 adopt
                    uint8_t rv[FIN2_U];
#pragma unroll
                    for (uint32_t u = 0; u < FIN2_U; u++) {
                        const uint32_t k = k0 + u * FIN2_T;
                        rs[u] = 0; re[u] = 0; rd[u] = 0; rv[u] = 0;
                        if (k >= total) continue;
                        const uint32_t e = s_root[k];
                        const uint32_t dist = G[gb + crel + e];
                        if (dist == 0) continue;                            // final since an earlier round
                        const uint64_t prel = crel + e;                     // my position and my source, relative to the frame
                        if (dist > prel) { flag_error(J, f, zc::E_OFFSET); G[gb + crel + e] = 0; continue; }
                        const uint64_t srel = prel - dist;
                        const uint32_t sc = cf + (uint32_t)(srel >> 16);
                        uint32_t gs = 0;
                        if (flag[sc] != 0) gs = G[gb + srel];
                        re[u] = e;
                        if (gs == 0) { rs[u] = 1; rd[u] = dist; }
                        else {                                              // adopt the source's source (a root's, or the root of a byte under one)
                            const uint64_t nd = (uint64_t)dist + gs;
                            if (nd > 0xFFFFFFFFull) { flag_error(J, f, zc::E_SIZE); G[gb + crel + e] = 0; continue; }
                            rs[u] = 2; rd[u] = (uint32_t)nd;
                        }
                    }
                    __threadfence();                                        // a source seen final has its byte written
#pragma unroll
                    for (uint32_t u = 0; u < FIN2_U; u++)
                        if (rs[u] == 1) rv[u] = *(volatile const uint8_t*)(J.out + f0 + crel + re[u] - rd[u]);
#pragma unroll
                    for (uint32_t u = 0; u < FIN2_U; u++)
                        if (rs[u] == 1) J.out[f0 + crel + re[u]] = rv[u];
                    __threadfence();                                        // my bytes before my zeroed distances
#pragma unroll
                    for (uint32_t u = 0; u < FIN2_U; u++) {
                        if (rs[u] == 1) G[gb + crel + re[u]] = 0;
                        else if (rs[u] == 2) { G[gb + crel + re[u]] = rd[u]; left++; }
                    }
                }
                __syncthreads();                                            // the list is reused by the next tile
            }
            if (left) atomicAdd(&s_left, left);
            __syncthreads();
            if (tid == 0) {
                if (s_left == 0) { __threadfence(); flag[c] = 2; }          // every root of the chunk is final now
                left_total += s_left;
            }
        }
        if (tid == 0 && left_total) atomicAdd(&J.fin_count[cur], left_total);
        NAF_GRID_SYNC();
        if (J.fin_count[cur] == 0) break;
    }
    // every root is final and written (the barrier above): the bytes under a root take its value
    for (uint32_t c = blockIdx.x; c < J.fin_total_chunks; c += gridDim.x) {
        if (flag[c] == 0) continue;
        const uint32_t f = fin_frame_of(J, c);
        const uint64_t f0 = J.frames[f].dst_off, fend = f0 + J.frames[f].dst_size;
        const uint64_t crel = (uint64_t)(c - J.fin_chunk_first[f]) * FIN_C;
        const uint32_t cn = (uint32_t)((crel + FIN_C < fend - f0) ? FIN_C : fend - f0 - crel);
        const uint32_t* g = J.fin_g + J.fin_g_base[f] + crel;
        uint8_t* o = J.out + f0 + crel;
        for (uint32_t e0 = tid * 4; e0 < cn; e0 += FIN2_T * 4) {           // (cn may end inside the last group: fin_g is padded per frame)
            const uint4 d = __ldcg((const uint4*)(g + e0));
            const uint32_t dd[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
            for (uint32_t k = 0; k < 4; k++)
                if (dd[k] != 0 && e0 + k < cn && dd[k] <= e0 + k) o[e0 + k] = __ldcg(o + e0 + k - dd[k]);
        }
    }
}

// --------------------------------------------------------------------------------------------------------------
// k_frame_checksum: frames whose header sets Content_Checksum_flag end with the low 32 bits of XXH64(content, 0), which
// libzstd -- reached from decoder/mod.rs:221 -- verifies.  NAF writers never set the flag, third-party zstd frames may.
// XXH64 is four multiplicative chains over 32-byte stripes: one warp per frame, lanes 0..3 own one accumulator each
// (a serial chain by construction: ~10 ns per stripe; it runs only for frames that ask for it).
__device__ __forceinline__ uint64_t xxh_rotl(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
constexpr uint64_t XXP1 = 0x9E3779B185EBCA87ull, XXP2 = 0xC2B2AE3D27D4EB4Full, XXP3 = 0x165667B19E3779F9ull, XXP4 = 0x85EBCA77C2B2AE63ull,
                   XXP5 = 0x27D4EB2F165667C5ull;
__device__ __forceinline__ uint64_t xxh_round(uint64_t acc, uint64_t in) { return xxh_rotl(acc + in * XXP2, 31) * XXP1; }
__device__ __forceinline__ uint64_t xxh_merge(uint64_t h, uint64_t v) { return (h ^ xxh_round(0, v)) * XXP1 + XXP4; }

__global__ void __launch_bounds__(32) k_frame_checksum(JobDev J) {
    const uint32_t f = blockIdx.x;
    const FrameDesc& F = J.frames[f];
    if (!F.has_checksum || J.frame_bad[f]) return;
    const int lane = threadIdx.x;
    const uint8_t* p = J.out + F.dst_off;                       // (frames regenerate at 16 B-aligned arena offsets)
    const uint64_t len = F.dst_size, stripes = len >> 5;
    uint64_t h;
    if (stripes) {
        uint64_t v = lane == 0 ? XXP1 + XXP2 : (lane == 1 ? XXP2 : (lane == 2 ? 0ull : 0ull - XXP1));
        if (lane < 4) {
            const uint64_t* q = (const uint64_t*)p + lane;
            uint64_t s = 0;
            for (; s + 8 <= stripes; s += 8) {                  // eight independent loads in flight per chain step
                uint64_t in[8];
#pragma unroll
                for (int k = 0; k < 8; k++) in[k] = q[4 * (s + k)];
#pragma unroll
                for (int k = 0; k < 8; k++) v = xxh_round(v, in[k]);
            }
            for (; s < stripes; s++) v = xxh_round(v, q[4 * s]);
        }
        const uint64_t v1 = __shfl_sync(0xFFFFFFFFu, v, 0), v2 = __shfl_sync(0xFFFFFFFFu, v, 1), v3 = __shfl_sync(0xFFFFFFFFu, v, 2),
                       v4 = __shfl_sync(0xFFFFFFFFu, v, 3);
        h = xxh_rotl(v1, 1) + xxh_rotl(v2, 7) + xxh_rotl(v3, 12) + xxh_rotl(v4, 18);
        h = xxh_merge(h, v1); h = xxh_merge(h, v2); h = xxh_merge(h, v3); h = xxh_merge(h, v4);
    } else h = XXP5;
    if (lane != 0) return;
    h += len;
    uint64_t i = stripes << 5;
    for (; i + 8 <= len; i += 8) { h ^= xxh_round(0, *(const uint64_t*)(p + i)); h = xxh_rotl(h, 27) * XXP1 + XXP4; }
    if (i + 4 <= len) { h ^= (uint64_t)(*(const uint32_t*)(p + i)) * XXP1; h = xxh_rotl(h, 23) * XXP2 + XXP3; i += 4; }
    for (; i < len; i++) { h ^= (uint64_t)p[i] * XXP5; h = xxh_rotl(h, 11) * XXP1; }
    h ^= h >> 33; h *= XXP2; h ^= h >> 29; h *= XXP3; h ^= h >> 32;
    if ((uint32_t)h != F.checksum) flag_error(J, f, zc::E_CHECKSUM);
}

uint32_t lz_resolve_max_ctas(int device) {
#if defined(NAFGPU_EMULATE)
    (void)device;
    return 1;
#else
    int sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lz_resolve, LZ_CTA, 0);
    if (per_sm > 4) per_sm = 4;
    return (uint32_t)(sms > 0 && per_sm > 0 ? sms * per_sm : 1);
#endif
}

// CTAs for the two finisher kernels: level 1 is one 212 KB CTA per SM, level 2 is cooperative (co-resident CTAs).
void lz_finish_ctas(int device, uint32_t* level1, uint32_t* level2) {
#if defined(NAFGPU_EMULATE)
    (void)device;
    *level1 = 2; *level2 = 1;
#else
    int sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lz_finish2, FIN2_T, 0);
    if (per_sm > 4) per_sm = 4;
    *level1 = (uint32_t)(sms > 0 ? sms : 1);
    *level2 = (uint32_t)(sms > 0 && per_sm > 0 ? sms * per_sm : 1);
#endif
}

bool Streams::create() {
    for (cudaStream_t* s : {&st, &st2, &st3}) if (cudaStreamCreateWithFlags(s, cudaStreamNonBlocking) != cudaSuccess) return false;
    for (cudaEvent_t* e : {fork, fork + 1, fork + 2, join, join + 1, join + 2}) if (cudaEventCreateWithFlags(e, cudaEventDisableTiming) != cudaSuccess) return false;
    return true;
}

void Streams::destroy() {
    for (cudaEvent_t* e : {fork, fork + 1, fork + 2, join, join + 1, join + 2}) { if (*e) cudaEventDestroy(*e); *e = nullptr; }
    for (cudaStream_t* s : {&st, &st2, &st3}) { if (*s) cudaStreamDestroy(*s); *s = 0; }
}

// A cooperative grid for `want` CTAs of work: at least 8, at most the co-resident `max` (a barrier over 27 CTAs returns sooner
// than one over 592, and a cooperative grid costs microseconds to launch even when it has nothing to do).
static uint32_t coop_grid(uint64_t want, uint32_t max) {
    const uint32_t cap = max ? max : 1u;
    return want < 8 ? std::min(8u, cap) : (uint32_t)std::min<uint64_t>(want, cap);
}

Launch choose_paths(JobDev& J, const fw::JobPlan& pl, const Overrides& ov, uint32_t sms, uint64_t arena_size) {
    const uint64_t nseq = J.n_seq;
    // thousands of tiny blocks (a FASTQ section flushed per record): warp-per-block kernels for them, and the two-warp CTAs of
    // the others do not carry the shared memory of ... the others
    J.tiny_blocks = ov.tiny_blocks ? *ov.tiny_blocks : (pl.n_tiny_seq_blocks >= 4096u ? 1u : 0u);
    J.seq_stage_bytes = std::min<uint32_t>((((J.tiny_blocks ? pl.max_seq_section_big : pl.max_seq_section) + 15u) & ~15u) + 64u, 16u * 1024u);
    // one CTA for the matches of a small job (k_lz_small holds up to 8192; beyond ~2000 the general rounds are faster)
    const uint64_t small_max = ov.lz_small ? *ov.lz_small : 2048;
    J.lz_small = (nseq <= small_max && J.n_frames <= 65535 && arena_size < (1ull << 32)) ? 1u : 0u;
    J.lz_flow_on = ov.lz_flow ? *ov.lz_flow : (nseq > 8192 ? 1u : 0u);
    J.flow_ctas = (uint32_t)std::min<uint64_t>((nseq + 255) / 256, sms * 8u);
    J.lz_flow_early = ov.lz_flow_early ? *ov.lz_flow_early : ((nseq > 2048 && nseq <= 65536 && !ov.lz_small) ? 1u : 0u);
    // the finisher's first level handles a 64 KB chunk in ~90 us on one SM, all SMs at once; its second level (barrier rounds over
    // the unresolved bytes) costs about twice that again when the chains cross many chunks (cfg3: 13 M bytes)
    const uint64_t waves = ((uint64_t)J.fin_total_chunks + J.fin_ctas - 1) / std::max<uint32_t>(J.fin_ctas, 1u);
    J.fin_cost_us = ov.fin_cost_us ? *ov.fin_cost_us : (uint32_t)std::min<uint64_t>(300 + waves * 270, 0x7FFFFFFFu);   // (both levels: 3.6 ms for the 1907 chunks of a 250 Mbp frame)
    J.huf_block_min = ov.huf_block_min ? *ov.huf_block_min : 0;

    Launch L;
    // a job with both kinds of Huffman streams (one archive: the big blocks of the sequence, the short ids / lengths / last
    // block): the two decodes side by side -- for a single small archive this branch is the critical path (25 us each)
    L.huf_side = J.n_huf_big && J.n_huf_items > J.n_huf_big;
    // Two shapes of the same decode of the big streams.  Enough blocks to fill the device several times over (a batch, a
    // chromosome): one CTA per BLOCK, its four streams in turn, tables built once, the range starts found beforehand by
    // k_huf_scout (the pair: 1.17 ms on the 256-archive job; 1.63 ms for the cluster kernel).  A handful of blocks (one small
    // archive): one CTA per STREAM, the four of a block as a thread-block cluster that shares the table construction through
    // DSMEM -- four times the CTAs in flight and no second launch, which is what latency wants (k_huf_decode_big).
    L.huf_per_block = J.n_huf_big / 4 >= (J.huf_block_min ? J.huf_block_min : 296u);
    L.huf_small_smem = HUF_SMALL_FIXED + ((J.max_huf_small + 15 + 16 + 16 + 15) & ~15u);
    L.huf_big_smem = hb_smem_bytes(J.max_huf_stream);
    L.huf_scout_smem = hs_smem_bytes(J.max_huf_stream);
    // a job with both kinds of blocks (a FASTQ archive: 2 x 10^6 tiny blocks and the ~130 big blocks of the ids, each one chain of
    // ~10^4 sequences, 2.9 ms): the general kernel beside the tiny blocks' (2.0 ms)
    L.seq_side = J.tiny_blocks && J.n_seq_big;
    // (jobs of 10^5+ tiny blocks -- FASTQ flushed per record -- have a handful of runs per block: no split, fewer CTAs)
    L.lit_blocks = J.tiny_blocks ? J.n_lit_big : J.n_blocks;
    L.lit_few = L.lit_blocks <= 64u;
    L.lit_split = L.lit_few ? 4 * LZLIT_SPLIT : (L.lit_blocks > 16384u ? 1 : LZLIT_SPLIT);
    L.lz_small_smem = lzs_smem_bytes((uint32_t)nseq);
    // (small jobs: one entry per thread, as many CTAs as entries need -- latency; big jobs: LZ_U entries per thread)
    L.first_ctas = (uint32_t)((nseq + LZ_CTA - 1) / LZ_CTA);
    if (L.first_ctas > sms * 8u) L.first_ctas = std::max<uint32_t>(sms * 8u, (uint32_t)((nseq + LZ_CTA * LZ_U - 1) / (LZ_CTA * LZ_U)));
    if (L.first_ctas > sms * 64u) L.first_ctas = sms * 64u;
    // a small job takes no more CTAs than its matches can use: a single archive pays one barrier per dependency round
    L.resolve_ctas = coop_grid((nseq + LZ_CTA * 2 - 1) / (LZ_CTA * 2), J.coop_ctas);
    L.finish_ctas = J.fin_total_chunks < J.fin_ctas ? J.fin_total_chunks : J.fin_ctas;
    L.finish = L.finish_ctas && nseq > LZ_MIN_PENDING;       // (k_lz_resolve never hands over fewer than LZ_MIN_PENDING matches)
    L.finish2_ctas = coop_grid(J.fin_total_chunks * 2u, J.fin2_ctas);
    return L;
}

int launch_zstd_stage(const JobDev& J, const Launch& L, const Streams& S, StageEvents* ev) {
    StageEvents none;
    if (!ev) ev = &none;
    int launches = 0, stage = 0;
    // the one place that marks stage ends: a stage a job skips gets an empty interval, so that there are always ZSTD_STAGES
    const auto end_stage = [&](int s) { for (; stage < s; stage++) ev->mark(); };
    if (J.n_blocks == 0) { end_stage(ZSTD_STAGES); return 0; }
    // Two independent branches: (A) FSE tables -> sequences -> frame scan on `st`; (B) Huffman weights -> Huffman decode into
    // the literal staging buffer on `st2` (not in a profiled run).  They join before k_lz_literals.
    const cudaStream_t st = S.st, st2 = ev != &none ? (cudaStream_t)0 : S.st2, st3 = S.st3;
    const cudaStream_t sb = st2 ? st2 : st;
    (void)sb; (void)st3;                               // (the emulator's launch macro ignores the stream)
    if (st2) { cudaEventRecord(S.fork[0], st); cudaStreamWaitEvent(st2, S.fork[0], 0); }
    if (J.n_huf_items) {
        NAF_LAUNCH(k_build_tables<1>, J.n_blocks, 32, 0, sb, J); launches++;
        const bool side = st2 && st3 && L.huf_side;
        if (side) {
            cudaEventRecord(S.fork[1], sb); cudaStreamWaitEvent(st3, S.fork[1], 0);
            NAF_LAUNCH(k_huf_decode_small, J.n_huf_items - J.n_huf_big, HUF_T_SMALL, L.huf_small_smem, st3, J, J.huf_items + J.n_huf_big); launches++;
            cudaEventRecord(S.join[1], st3);
        }
        if (J.n_huf_big) {   // items [0, n_huf_big): the streams of 4-stream blocks, four consecutive items (= one cluster) per block
            if (!st2) ev->kernel_begin();
            if (L.huf_per_block) {
                // (the scout and its write pass are one decode of the big streams: counted as one launch, like the cluster kernel)
                NAF_SET_MAX_SMEM(k_huf_scout, L.huf_scout_smem);
                NAF_LAUNCH(k_huf_scout, J.n_huf_big / 4, HS_T, L.huf_scout_smem, sb, J);
                NAF_SET_MAX_SMEM(k_huf_decode_block, L.huf_big_smem);
                NAF_LAUNCH(k_huf_decode_block, J.n_huf_big / 4, HB_T, L.huf_big_smem, sb, J); launches++;
            } else {
                NAF_SET_MAX_SMEM(k_huf_decode_big, L.huf_big_smem);
                NAF_LAUNCH(k_huf_decode_big, J.n_huf_big, HB_T, L.huf_big_smem, sb, J); launches++;
            }
            if (!st2) ev->kernel_end();
        }
        if (side) cudaStreamWaitEvent(sb, S.join[1], 0);
        else if (J.n_huf_items > J.n_huf_big) {
            NAF_LAUNCH(k_huf_decode_small, J.n_huf_items - J.n_huf_big, HUF_T_SMALL, L.huf_small_smem, sb, J, J.huf_items + J.n_huf_big); launches++;
        }
    }
    if (st2) cudaEventRecord(S.join[0], st2);
    end_stage(1);                                      // (serial: the Huffman branch first)
    NAF_LAUNCH(k_build_tables<0>, J.n_blocks + 1, 96, 0, st, J); launches++;
    end_stage(2);
    const bool seq_side = st2 && st3 && L.seq_side;
    if (seq_side) {
        cudaEventRecord(S.fork[2], st); cudaStreamWaitEvent(st3, S.fork[2], 0);
        NAF_LAUNCH(k_decode_sequences, J.n_seq_big, 64, J.seq_stage_bytes, st3, J); launches++;
        cudaEventRecord(S.join[2], st3);
    }
    if (J.tiny_blocks) { NAF_LAUNCH(k_decode_sequences_tiny, (J.n_blocks + SEQ_TINY_WARPS - 1) / SEQ_TINY_WARPS, SEQ_TINY_WARPS * 32, 0, st, J); launches++; }
    if (seq_side) cudaStreamWaitEvent(st, S.join[2], 0);
    else if (!J.tiny_blocks || J.n_seq_big) { NAF_LAUNCH(k_decode_sequences, J.tiny_blocks ? J.n_seq_big : J.n_blocks, 64, J.seq_stage_bytes, st, J); launches++; }
    end_stage(3);
    NAF_LAUNCH(k_frame_scan, J.n_frames, FSCAN_T, 0, st, J); launches++;
    if (J.n_fs_tiles) {
        NAF_LAUNCH(k_fs_reduce, J.n_fs_tiles, FSCAN_T, 0, st, J);
        NAF_LAUNCH(k_fs_prefix, J.n_fs_big, 32, 0, st, J);
        NAF_LAUNCH(k_fs_apply, J.n_fs_tiles, FSCAN_T, 0, st, J);
        launches += 3;
    }
    end_stage(4);
    if (st2) cudaStreamWaitEvent(st, S.join[0], 0);
    if (J.tiny_blocks) { NAF_LAUNCH(k_lz_literals_tiny, (J.n_blocks + 7) / 8, 256, 0, st, J); launches++; }
    if (L.lit_blocks && L.lit_few) { NAF_LAUNCH(k_lz_literals<4>, dim3(L.lit_blocks, L.lit_split), 256, 0, st, J); launches++; }
    else if (L.lit_blocks) { NAF_LAUNCH(k_lz_literals<1>, dim3(L.lit_blocks, L.lit_split), 256, 0, st, J); launches++; }
    end_stage(5);
    if (J.n_seq > 0) {
        if (J.lz_small) {
            NAF_SET_MAX_SMEM(k_lz_small, L.lz_small_smem);
            NAF_LAUNCH(k_lz_small, 1, LZS_T, L.lz_small_smem, st, J); launches++;
            end_stage(7);
        } else {
            NAF_LAUNCH(k_lz_index, (uint32_t)((J.n_seq + 255) / 256), 256, 0, st, J); launches++;
            if (J.lz_flow_early) { NAF_LAUNCH(k_lz_flow, J.flow_ctas, LZF_T, 0, st, J, 1); launches++; }
            NAF_LAUNCH(k_lz_first, L.first_ctas, LZ_CTA, 0, st, J); launches++;
            end_stage(6);
            JobDev Jc = J;
            NAF_LAUNCH_COOP(k_lz_resolve, L.resolve_ctas, LZ_CTA, st, Jc); launches++;
            if (J.lz_flow_on) { NAF_LAUNCH(k_lz_flow, J.flow_ctas, LZF_T, 0, st, J, 0); launches++; }
            end_stage(7);
        }
        JobDev Jc = J;
        if (L.finish) {
            NAF_SET_MAX_SMEM(k_lz_finish, FIN_SMEM);
            NAF_LAUNCH(k_lz_finish, L.finish_ctas, FIN_T, FIN_SMEM, st, J); launches++;
            NAF_LAUNCH_COOP(k_lz_finish2, L.finish2_ctas, FIN2_T, st, Jc); launches++;
        }
    }
    end_stage(ZSTD_STAGES);
    if (J.n_checksums) { NAF_LAUNCH(k_frame_checksum, J.n_frames, 32, 0, st, J); launches++; }      // (profiled runs count it with the next stage)
    return launches;
}

}  // namespace zk

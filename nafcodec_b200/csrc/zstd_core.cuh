// zstd_core.cuh -- bit-level zstd primitives shared by the sm_100a kernels and the host-side frame walker.
//
// Everything here is __host__ __device__ so the same code that runs inside the kernels can be driven
// serially by tests/emul (a CPU harness that checks the bit-level logic against libzstd before any GPU
// time is spent).  The format rules follow RFC 8878 (the zstd arithmetic is NOT in the reference tree: it
// lives in crate zstd ^0.13.1 -> zstd-sys -> libzstd, reached from nafcodec/src/decoder/mod.rs:221-223).
#pragma once
#include <stdint.h>
#include <stddef.h>

#if defined(__CUDACC__)
#define ZHD __host__ __device__ __forceinline__
#else
#define ZHD inline
#endif

namespace zc {

// ---- error bits (OR-ed into a per-job status word; 0 = ok) -------------------------------------------------
enum : uint32_t {
    E_OK = 0,
    E_FSE_TABLE = 1u << 0,       // bad FSE table description
    E_HUF_TREE = 1u << 1,        // bad Huffman tree description
    E_HUF_STREAM = 1u << 2,      // Huffman bitstream did not end on its first bit / bad jump table
    E_SEQ_STREAM = 1u << 3,      // sequence bitstream over/under-run
    E_LITERALS = 1u << 4,        // literal lengths exceed the literals of the block
    E_OFFSET = 1u << 5,          // match offset reaches before the frame start / is zero
    E_SIZE = 1u << 6,            // regenerated size differs from the size the NAF header states
    E_NO_TABLE = 1u << 7,        // repeat/treeless mode without a previous table
    E_LENGTHS = 1u << 8,         // NAF: lengths exceed the sequence stream
    E_MASK = 1u << 9,            // NAF: mask runs end before the sequences do
    E_UTF8 = 1u << 10,           // NAF: text field is not valid UTF-8
    E_NUL = 1u << 11,            // NAF: id/comment stream does not end with NUL
    E_CHECKSUM = 1u << 12,       // frame content checksum (XXH64) does not match
    E_INTERNAL = 1u << 30
};

ZHD int highbit32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return 31 - __clz((int)v);
#else
    return v ? 31 - __builtin_clz(v) : -1;          // (the device's value for 0; __builtin_clz(0) is undefined)
#endif
}

// ---- bit access ---------------------------------------------------------------------------------------------
// 64 stream bits starting at absolute bit offset `bit` from byte pointer `p` (LSB-first within bytes, i.e.
// stream bit i is bit (i&7) of byte i>>3).  Built from two ALIGNED 8-byte loads so it is legal on the device
// for any alignment; the buffer must be readable up to 15 bytes past the last byte touched (all compressed
// buffers are padded) and `p` rounded down to 8 must be inside the allocation (allocations are >= 8-aligned).
ZHD uint64_t load_bits64(const uint8_t* p, uint64_t bit) {
    uintptr_t a = (uintptr_t)p + (bit >> 3);
    const uint64_t* w = (const uint64_t*)(a & ~(uintptr_t)7);
    uint32_t sh = (uint32_t)((a & 7) * 8 + (bit & 7));
    uint64_t lo = w[0];
    if (sh == 0) return lo;
    uint64_t hi = w[1];
    return (lo >> sh) | (hi << (64 - sh));
}

// Backward bitstream (RFC 8878 4.1): the last byte carries a final 1-bit marker above the payload; bits are
// consumed from the marker downwards.  P = number of unread payload bits.
struct BackBits {
    const uint8_t* base;
    int64_t P;
    ZHD bool init(const uint8_t* b, uint32_t nbytes) {
        base = b;
        P = 0;
        if (nbytes == 0) return false;
        uint8_t last = b[nbytes - 1];
        if (last == 0) return false;
        P = 8 * (int64_t)(nbytes - 1) + highbit32(last);
        return true;
    }
    // next k (<= 32) bits without consuming; bits below the start of the stream read as zero
    ZHD uint32_t peek(int k) const {
        if (k == 0) return 0;
        uint32_t m = (k >= 32) ? 0xFFFFFFFFu : ((1u << k) - 1u);
        if (P >= k) return (uint32_t)load_bits64(base, (uint64_t)(P - k)) & m;
        if (P <= 0) return 0;
        uint32_t avail = (uint32_t)load_bits64(base, 0) & ((1u << (int)P) - 1u);
        return (avail << (k - (int)P)) & m;
    }
    ZHD uint32_t read(int k) {
        uint32_t v = peek(k);
        P -= k;
        return v;
    }
};

// Forward LSB-first reader with bounds (FSE table descriptions).
struct FwdBits {
    const uint8_t* p;
    uint32_t nbytes;
    uint32_t pos;     // bit position
    ZHD uint32_t byte_at(uint32_t i) const { return i < nbytes ? p[i] : 0u; }
    ZHD uint32_t peek(int k) const {   // k <= 16
        uint32_t b = pos >> 3, s = pos & 7;
        uint32_t v = byte_at(b) | (byte_at(b + 1) << 8) | (byte_at(b + 2) << 16);
        return (v >> s) & ((1u << k) - 1u);
    }
    ZHD void skip(int k) { pos += (uint32_t)k; }
    ZHD uint32_t read(int k) { uint32_t v = peek(k); pos += (uint32_t)k; return v; }
    ZHD bool overrun() const { return pos > nbytes * 8u; }
    ZHD uint32_t bytes_used() const { return (pos + 7) >> 3; }
};

// ---- FSE ----------------------------------------------------------------------------------------------------
constexpr int MAX_LL = 35, MAX_OF = 31, MAX_ML = 52, MAX_HUF_W = 255;
constexpr int MAX_AL_LL = 9, MAX_AL_OF = 8, MAX_AL_ML = 9, MAX_AL_HUF = 6;

// Reads a normalized-count table description.  norm[] gets max_symbol+1 entries (unused = 0).
// Returns bytes consumed, or 0 on error.  *al_out = accuracy log.
ZHD uint32_t fse_read_ncount(const uint8_t* src, uint32_t src_len, int max_symbol, int max_al, int16_t* norm, int* al_out) {
    FwdBits fb{src, src_len, 0};
    int al = (int)fb.read(4) + 5;
    if (al > max_al) return 0;
    int rem = 1 << al;
    int sym = 0;
    for (int i = 0; i <= max_symbol; i++) norm[i] = 0;
    while (rem > 0 && sym <= max_symbol) {
        int bits = highbit32((uint32_t)(rem + 1)) + 1;
        uint32_t v = fb.peek(bits);
        uint32_t low = (1u << (bits - 1)) - 1u;
        uint32_t thr = (1u << bits) - 1u - (uint32_t)(rem + 1);
        if ((v & low) < thr) {
            fb.skip(bits - 1);
            v &= low;
        } else {
            fb.skip(bits);
            if (v > low) v -= thr;
        }
        int pr = (int)v - 1;
        rem -= (pr < 0) ? -pr : pr;
        norm[sym++] = (int16_t)pr;
        if (pr == 0) {
            for (;;) {
                uint32_t r = fb.read(2);
                sym += (int)r;                      // r extra zero-probability symbols
                if (r != 3) break;
                if (fb.overrun()) return 0;
            }
            if (sym > max_symbol + 1) return 0;
        }
        if (fb.overrun()) return 0;
    }
    if (rem != 0 || sym > max_symbol + 1) return 0;
    *al_out = al;
    return fb.bytes_used();
}

// Generic FSE decode cell (Huffman-weight tables): symbol, nbBits, newState base.
struct FseCell { uint16_t base; uint8_t nb; uint8_t sym; };

// Sequence decode cell: one 8-byte lookup gives everything a sequence symbol needs.
struct SeqCell { uint32_t base_value; uint16_t next_base; uint8_t nb; uint8_t add_bits; };

// Serial table build (RFC 8878 4.1.1).  cell_sym: scratch of `size` bytes; cnt: scratch of max_symbol+1 u16.
// Emit(i, sym, nb, base) is called for every cell in index order.
template <class Emit>
ZHD bool fse_build(const int16_t* norm, int max_symbol, int al, uint8_t* cell_sym, uint16_t* cnt, Emit emit) {
    int size = 1 << al;
    int high = size;
    for (int s = 0; s <= max_symbol; s++) {
        if (norm[s] == -1) { cell_sym[--high] = (uint8_t)s; cnt[s] = 1; }
        else cnt[s] = (uint16_t)(norm[s] > 0 ? norm[s] : 0);
    }
    int step = (size >> 1) + (size >> 3) + 3, pos = 0, mask = size - 1;
    for (int s = 0; s <= max_symbol; s++) {
        for (int i = 0; i < norm[s]; i++) {
            cell_sym[pos] = (uint8_t)s;
            do { pos = (pos + step) & mask; } while (pos >= high);
        }
    }
    if (pos != 0) return false;
    for (int i = 0; i < size; i++) {
        int s = cell_sym[i];
        uint32_t nx = cnt[s]++;
        int nb = al - highbit32(nx);
        emit(i, s, nb, (int)((nx << nb) - (uint32_t)size));
    }
    return true;
}

// Code -> (baseline, extra bits) tables (RFC 8878 3.1.1.3.2.1.1).  In device code they live in constant memory
// (a function-local array would be rebuilt on the thread's stack at every call).
#define ZC_LL_BASE {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536}
#define ZC_LL_BITS {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16}
#define ZC_ML_BASE {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, \
                    35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539}
#define ZC_ML_BITS {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, \
                    1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16}
#define ZC_PRE_LL {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1}
#define ZC_PRE_OF {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1}
#define ZC_PRE_ML {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, \
                   1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1}
#if defined(__CUDACC__)
__device__ __constant__ uint32_t d_ll_base[36] = ZC_LL_BASE;
__device__ __constant__ uint8_t d_ll_bits[36] = ZC_LL_BITS;
__device__ __constant__ uint32_t d_ml_base[53] = ZC_ML_BASE;
__device__ __constant__ uint8_t d_ml_bits[53] = ZC_ML_BITS;
__device__ __constant__ int8_t d_pre_ll[36] = ZC_PRE_LL;
__device__ __constant__ int8_t d_pre_of[29] = ZC_PRE_OF;
__device__ __constant__ int8_t d_pre_ml[53] = ZC_PRE_ML;
#endif
static const uint32_t h_ll_base[36] = ZC_LL_BASE;
static const uint8_t h_ll_bits[36] = ZC_LL_BITS;
static const uint32_t h_ml_base[53] = ZC_ML_BASE;
static const uint8_t h_ml_bits[53] = ZC_ML_BITS;
static const int8_t h_pre_ll[36] = ZC_PRE_LL;
static const int8_t h_pre_of[29] = ZC_PRE_OF;
static const int8_t h_pre_ml[53] = ZC_PRE_ML;
#if defined(__CUDA_ARCH__)
#define ZC_TAB(name) d_##name
#else
#define ZC_TAB(name) h_##name
#endif
ZHD uint32_t ll_base(int c) { return ZC_TAB(ll_base)[c]; }
ZHD int ll_bits(int c) { return ZC_TAB(ll_bits)[c]; }
ZHD uint32_t ml_base(int c) { return ZC_TAB(ml_base)[c]; }
ZHD int ml_bits(int c) { return ZC_TAB(ml_bits)[c]; }

enum { KIND_LL = 0, KIND_OF = 1, KIND_ML = 2 };
ZHD int kind_max_symbol(int k) { return k == KIND_LL ? MAX_LL : (k == KIND_OF ? MAX_OF : MAX_ML); }
ZHD int kind_max_al(int k) { return k == KIND_LL ? MAX_AL_LL : (k == KIND_OF ? MAX_AL_OF : MAX_AL_ML); }
ZHD SeqCell make_seq_cell(int kind, int sym, int nb, int base) {
    SeqCell c;
    c.nb = (uint8_t)nb;
    c.next_base = (uint16_t)base;
    if (kind == KIND_LL) { c.base_value = ll_base(sym); c.add_bits = (uint8_t)ll_bits(sym); }
    else if (kind == KIND_ML) { c.base_value = ml_base(sym); c.add_bits = (uint8_t)ml_bits(sym); }
    else { c.base_value = 1u << sym; c.add_bits = (uint8_t)sym; }
    return c;
}

// Predefined distributions (RFC 8878 3.1.1.3.2.2)
ZHD int16_t predef_norm(int kind, int s) {
    if (kind == KIND_LL) return ZC_TAB(pre_ll)[s];
    if (kind == KIND_OF) return s < 29 ? ZC_TAB(pre_of)[s] : 0;
    return ZC_TAB(pre_ml)[s];
}
ZHD int predef_al(int kind) { return kind == KIND_OF ? 5 : 6; }

// ---- Huffman ------------------------------------------------------------------------------------------------
constexpr int HUF_MAX_BITS = 11;

// Size in bytes of a Huffman tree description starting at header byte h (including the header byte).
ZHD uint32_t huf_tree_desc_size(uint8_t h) { return h < 128 ? 1u + h : 1u + ((uint32_t)(h - 127) + 1u) / 2u; }

// Decodes the weights of a tree description.  weights[256] (zero padded).  Returns number of symbols
// (including the implied last one) and *max_bits, or 0 on error.  scratch: >= 64 FseCell + 64 bytes + 256 u16.
ZHD int huf_read_weights(const uint8_t* src, uint32_t src_len, uint8_t* weights, int* max_bits_out) {
    if (src_len == 0) return 0;
    uint8_t h = src[0];
    int n = 0;
    for (int i = 0; i < 256; i++) weights[i] = 0;
    if (h >= 128) {
        n = h - 127;
        if (1u + (uint32_t)(n + 1) / 2u > src_len) return 0;
        for (int i = 0; i < n; i++) {
            uint8_t b = src[1 + (i >> 1)];
            weights[i] = (i & 1) ? (b & 15) : (b >> 4);
        }
    } else {
        if (1u + h > src_len || h < 2) return 0;
        int16_t norm[MAX_HUF_W + 1];
        int al = 0;
        // weights are 0..11, so the alphabet of the FSE-compressed weight stream is tiny; zstd caps it at 255 but
        // the table has at most 64 cells, hence at most 64 distinct symbols.
        uint32_t used = fse_read_ncount(src + 1, h, 12, MAX_AL_HUF, norm, &al);
        if (used == 0 || used >= h) return 0;
        FseCell cells[64];
        uint8_t cell_sym[64];
        uint16_t cnt[16];
        bool ok = fse_build(norm, 12, al, cell_sym, cnt, [&](int i, int s, int nb, int base) {
            cells[i].sym = (uint8_t)s; cells[i].nb = (uint8_t)nb; cells[i].base = (uint16_t)base;
        });
        if (!ok) return 0;
        BackBits bb;
        if (!bb.init(src + 1 + used, h - used)) return 0;
        uint32_t s1 = bb.read(al), s2 = bb.read(al);
        if (bb.P < 0) return 0;
        for (;;) {
            if (n > 253) return 0;
            weights[n++] = cells[s1].sym;
            s1 = cells[s1].base + bb.read(cells[s1].nb);
            if (bb.P < 0) { weights[n++] = cells[s2].sym; break; }
            if (n > 253) return 0;
            weights[n++] = cells[s2].sym;
            s2 = cells[s2].base + bb.read(cells[s2].nb);
            if (bb.P < 0) { weights[n++] = cells[s1].sym; break; }
        }
    }
    uint32_t tot = 0, ones = 0;
    for (int i = 0; i < n; i++) {
        if (weights[i] > HUF_MAX_BITS) return 0;
        if (weights[i]) tot += 1u << (weights[i] - 1);
        ones += weights[i] == 1;
    }
    if (tot == 0) return 0;
    int max_bits = highbit32(tot) + 1;
    if (max_bits > HUF_MAX_BITS) return 0;
    uint32_t left = (1u << max_bits) - tot;
    if (left & (left - 1)) return 0;           // must be a power of two
    if (ones + (left == 1u) < 2) return 0;     // at least two codes of max_bits (libzstd's HUF_readStats)
    weights[n++] = (uint8_t)(highbit32(left) + 1);
    *max_bits_out = max_bits;
    return n;
}

// Huffman decode table entry: low byte = code length, high byte = symbol.
// Serial build: start offsets per weight then fill (RFC 8878 4.2.1: ascending weight, then ascending symbol).
ZHD void huf_build_table_serial(const uint8_t* weights, int nsym, int max_bits, uint16_t* table) {
    uint32_t count[HUF_MAX_BITS + 2];
    for (int w = 0; w <= HUF_MAX_BITS + 1; w++) count[w] = 0;
    for (int s = 0; s < nsym; s++) count[weights[s]]++;
    uint32_t start[HUF_MAX_BITS + 2];
    uint32_t acc = 0;
    for (int w = 1; w <= max_bits + 0 && w <= HUF_MAX_BITS + 1; w++) { start[w] = acc; acc += count[w] << (w - 1); }
    for (int s = 0; s < nsym; s++) {
        int w = weights[s];
        if (!w) continue;
        uint32_t len = (uint32_t)(max_bits + 1 - w), n = 1u << (w - 1);
        uint16_t e = (uint16_t)((s << 8) | len);
        for (uint32_t i = 0; i < n; i++) table[start[w] + i] = e;
        start[w] += n;
    }
}

}  // namespace zc

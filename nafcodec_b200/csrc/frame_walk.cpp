// frame_walk.cpp -- see frame_walk.h.  Format: RFC 8878 3.1.1 (frame header, block header, literals section
// header, sequences section header).  Only byte-aligned header fields are read here.
#include "frame_walk.h"

#include <stdio.h>
#include <string.h>

#include <algorithm>

namespace fw {

static const int ERR_INVALID = -2;   // NAFGPU_ERR_INVALID_DATA
static const int ERR_EOF = -1;       // NAFGPU_ERR_UNEXPECTED_EOF
static const int ERR_UNSUPPORTED = -9;

#define FAIL(code, ...) do { char _b[160]; snprintf(_b, sizeof _b, __VA_ARGS__); err = _b; return (code); } while (0)

// Frame header: returns its size through p, the window through `window`, whether a content checksum follows the blocks.
static int frame_header(const uint8_t* s, uint64_t n, uint64_t dst_size, uint64_t& p, uint64_t& window, int& checksum, std::string& err) {
    p = 0;
    if (n < 1) FAIL(ERR_EOF, "zstd frame: empty");
    uint8_t fhd = s[p++];
    int fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, dict_flag = fhd & 3;
    checksum = (fhd >> 2) & 1;
    if (fhd & 0x08) FAIL(ERR_INVALID, "zstd frame: reserved bit set");
    window = 0;
    if (!single) {
        if (p >= n) FAIL(ERR_EOF, "zstd frame: truncated header");
        uint8_t wd = s[p++];
        uint64_t base = 1ull << (10 + (wd >> 3));
        window = base + (base >> 3) * (wd & 7);
    }
    // match offsets travel through the kernels as 31-bit values: bit 31 marks the symbolic repeat-offset encoding
    // (zstd_format.h, OFF_SYMBOLIC; a decoded raw offset with bit 31 set flags the block, and the LZ rounds never redirect a
    // match to a sum of 2^31 or more).  A window descriptor above 512 MiB (zstd --long=30/31) is refused, not mis-decoded;
    // a single-segment frame's window is its content size, checked below.
    if (window > (1ull << 29)) FAIL(ERR_UNSUPPORTED, "zstd frame: window of %llu bytes exceeds the supported 512 MiB", (unsigned long long)window);
    static const int dict_sz[4] = {0, 1, 2, 4};
    uint32_t dict_id = 0;
    if (p + dict_sz[dict_flag] > n) FAIL(ERR_EOF, "zstd frame: truncated header");
    for (int i = 0; i < dict_sz[dict_flag]; i++) dict_id |= (uint32_t)s[p++] << (8 * i);
    if (dict_id != 0) FAIL(ERR_UNSUPPORTED, "zstd frame: dictionaries are not supported");
    int fcs_sz = fcs_flag == 0 ? (single ? 1 : 0) : (fcs_flag == 1 ? 2 : (fcs_flag == 2 ? 4 : 8));
    if (p + fcs_sz > n) FAIL(ERR_EOF, "zstd frame: truncated header");
    uint64_t fcs = 0;
    for (int i = 0; i < fcs_sz; i++) fcs |= (uint64_t)s[p++] << (8 * i);
    if (fcs_sz == 2) fcs += 256;
    if (single) window = fcs;
    // (offsets of a single-segment frame are below its content size; up to 1 GiB they stay clear of bit 31 and of the
    //  finisher's bound on chunk-relative distances, 0x7F000000)
    if (single && window > (1ull << 30)) FAIL(ERR_UNSUPPORTED, "zstd frame: single-segment window of %llu bytes exceeds the supported 1 GiB", (unsigned long long)window);
    if (fcs_sz && fcs != dst_size) FAIL(ERR_INVALID, "zstd frame: content size %llu differs from the section size %llu",
                                        (unsigned long long)fcs, (unsigned long long)dst_size);

    return 0;
}

int chain_blocks(const uint8_t* s, uint64_t n, uint64_t dst_size, uint32_t every, std::vector<uint64_t>& cuts, uint64_t& n_blocks, std::string& err) {
    uint64_t p, window;
    int checksum;
    if (int rc = frame_header(s, n, dst_size, p, window, checksum, err)) return rc;
    cuts.clear();
    n_blocks = 0;
    // the serial dependency of the whole walk: position -> header -> next position.  Nothing else is looked at here (reserved
    // block types, sizes beyond the maximum and truncated contents are reported by the parts).
    while (p + 4 <= n) {
        uint32_t left = every;
        uint32_t bh = 0;
        do {
            memcpy(&bh, s + p, 4);                               // (little-endian host; the fourth byte is masked off)
            bh &= 0xFFFFFF;
            p += 3 + (((bh >> 1) & 3) == zf::BT_RLE ? 1u : (bh >> 3));
            n_blocks++;
        } while (!(bh & 1) && --left && p + 4 <= n);
        if (bh & 1) return 0;
        if (!left) cuts.push_back(p);
    }
    // fewer than 4 bytes left: the last header of a frame without content after it, or a truncated frame
    for (;;) {
        if (p + 3 > n) FAIL(ERR_EOF, "zstd frame: truncated block header");
        const uint32_t bh = s[p] | (s[p + 1] << 8) | (s[p + 2] << 16);
        p += 3 + (((bh >> 1) & 3) == zf::BT_RLE ? 1u : (bh >> 3));
        n_blocks++;
        if (bh & 1) break;
    }
    return 0;
}

int walk_frame_part(const uint8_t* frame, uint64_t src_off, uint64_t src_size, uint64_t dst_off, uint64_t dst_size,
                    uint64_t p_begin, uint64_t p_end, bool first, bool last_part, RangeState& st, JobPlan& plan, std::string& err) {
    const uint8_t* s = frame;
    uint64_t n = src_size, p = p_begin;
    int checksum = 0;
    uint32_t frame_idx = 0;                                    // (a continuation part has no frame of its own: the merge points its blocks at the first part's)
    size_t fd_at = (size_t)-1;
    st = RangeState();
    if (first) {
        uint64_t window;
        if (int rc = frame_header(s, n, dst_size, p, window, checksum, err)) return rc;
        zf::FrameDesc fd{};
        fd.src_off = src_off; fd.src_size = src_size; fd.dst_off = dst_off; fd.dst_size = dst_size;
        fd.first_block = (uint32_t)plan.blocks.size(); fd.first_seq = (uint32_t)plan.seq_total; fd.window = window;
        frame_idx = (uint32_t)plan.frames.size();
        fd_at = plan.frames.size();
        plan.frames.push_back(fd);
    } else {
        checksum = (s[0] >> 2) & 1;
        st.last_huf = PREV_BLOCK;
        st.cur_tbl[0] = st.cur_tbl[1] = st.cur_tbl[2] = PREV_SLOT;
    }
    const size_t first_block = plan.blocks.size();
    const uint64_t first_seq = plan.seq_total;
    uint32_t& last_huf = st.last_huf;
    uint32_t& last_huf_slot = st.last_huf_slot;
    uint32_t* cur_tbl = st.cur_tbl;
    uint64_t& known_total = st.known_total;
    for (;;) {
        if (!last_part && p == p_end) break;
        if (!last_part && p > p_end) FAIL(ERR_INVALID, "zstd frame: block chain changed between the passes");
        if (p + 3 > n) FAIL(ERR_EOF, "zstd frame: truncated block header");
        uint32_t bh = s[p] | (s[p + 1] << 8) | (s[p + 2] << 16);
        p += 3;
        int last = bh & 1, bt = (bh >> 1) & 3;
        uint32_t bsize = bh >> 3;
        if (bt == 3) FAIL(ERR_INVALID, "zstd block: reserved block type");
        if (bsize > zf::BLOCK_MAX) FAIL(ERR_INVALID, "zstd block: size %u exceeds the block maximum", bsize);
        zf::BlockDesc b{};
        b.src_off = src_off + p; b.src_size = bsize; b.frame = frame_idx; b.btype = (uint8_t)bt;
        b.huf_block = zf::NO_BLOCK; b.tbl[0] = b.tbl[1] = b.tbl[2] = zf::NO_SLOT;
        uint32_t self = (uint32_t)plan.blocks.size();
        uint64_t content = (bt == zf::BT_RLE) ? 1 : bsize;
        if (p + content > n) FAIL(ERR_EOF, "zstd block: truncated content");
        if (bt != zf::BT_COMPRESSED) {
            b.known_regen = bsize;
        } else {
            const uint8_t* c = s + p;
            if (bsize < 2) FAIL(ERR_INVALID, "zstd block: compressed block too small");
            uint8_t b0 = c[0];
            int lt = b0 & 3, sf = (b0 >> 2) & 3;
            uint32_t hdr, regen, csize;
            int streams = 1;
            if (lt == zf::LT_RAW || lt == zf::LT_RLE) {
                if (sf == 0 || sf == 2) { hdr = 1; regen = b0 >> 3; }
                else if (sf == 1) { hdr = 2; if (bsize < 2) FAIL(ERR_INVALID, "zstd literals: truncated"); regen = (b0 >> 4) | ((uint32_t)c[1] << 4); }
                else { hdr = 3; if (bsize < 3) FAIL(ERR_INVALID, "zstd literals: truncated"); regen = (b0 >> 4) | ((uint32_t)c[1] << 4) | ((uint32_t)c[2] << 12); }
                csize = (lt == zf::LT_RAW) ? regen : 1;
            } else {
                if (sf <= 1) {
                    hdr = 3; if (bsize < 3) FAIL(ERR_INVALID, "zstd literals: truncated");
                    uint32_t v = c[0] | (c[1] << 8) | (c[2] << 16);
                    regen = (v >> 4) & 0x3FF; csize = (v >> 14) & 0x3FF; streams = sf == 0 ? 1 : 4;
                } else if (sf == 2) {
                    hdr = 4; if (bsize < 4) FAIL(ERR_INVALID, "zstd literals: truncated");
                    uint32_t v = c[0] | (c[1] << 8) | (c[2] << 16) | ((uint32_t)c[3] << 24);
                    regen = (v >> 4) & 0x3FFF; csize = v >> 18; streams = 4;
                } else {
                    hdr = 5; if (bsize < 5) FAIL(ERR_INVALID, "zstd literals: truncated");
                    uint64_t v = c[0] | (c[1] << 8) | (c[2] << 16) | ((uint64_t)c[3] << 24) | ((uint64_t)c[4] << 32);
                    regen = (uint32_t)((v >> 4) & 0x3FFFF); csize = (uint32_t)((v >> 22) & 0x3FFFF); streams = 4;
                }
            }
            if (regen > zf::BLOCK_MAX) FAIL(ERR_INVALID, "zstd literals: regenerated size %u too large", regen);
            if ((uint64_t)hdr + csize > bsize) FAIL(ERR_INVALID, "zstd literals: section exceeds the block");
            b.lit_type = (uint8_t)lt; b.n_streams = (uint8_t)streams; b.lit_regen = regen; b.lit_csize = csize; b.lit_src = hdr;
            if (lt == zf::LT_HUF) { last_huf = self; b.huf_block = self; last_huf_slot = plan.n_huf_slots++; b.huf_slot = last_huf_slot; }
            else if (lt == zf::LT_TREELESS) {
                if (last_huf == zf::NO_BLOCK) FAIL(ERR_INVALID, "zstd literals: treeless block without a previous tree");
                if (last_huf == PREV_BLOCK) st.used_prev_huf = true;     // (a tree from before this part: the merge fills it in)
                b.huf_block = last_huf; b.huf_slot = last_huf_slot;
            }
            if (lt >= zf::LT_HUF) {
                plan.n_huf_blocks++;
                b.lit_base = plan.lit_total;              // every Huffman block decodes into the literal staging buffer
                plan.lit_total += (regen + 15u + 16u) & ~15u;
                // locate the bitstreams: [tree description][jump table (4 streams)] streams...
                uint32_t pay = hdr, pay_size = csize;
                if (lt == zf::LT_HUF) {
                    if (pay_size < 1) FAIL(ERR_INVALID, "zstd literals: missing Huffman tree");
                    uint8_t hb = c[pay];
                    uint32_t t = hb < 128 ? 1u + hb : 1u + ((uint32_t)(hb - 127) + 1u) / 2u;
                    if (t > pay_size) FAIL(ERR_INVALID, "zstd literals: Huffman tree exceeds the literals section");
                    pay += t; pay_size -= t;
                }
                if (regen == 0) FAIL(ERR_INVALID, "zstd literals: empty Huffman literals");
                uint32_t so[4], ss[4], dn[4], dof[4];
                if (streams == 1) { so[0] = pay; ss[0] = pay_size; dn[0] = regen; dof[0] = 0; }
                else {
                    if (pay_size < 6) FAIL(ERR_INVALID, "zstd literals: missing jump table");
                    uint32_t z1 = c[pay] | (c[pay + 1] << 8), z2 = c[pay + 2] | (c[pay + 3] << 8), z3 = c[pay + 4] | (c[pay + 5] << 8);
                    uint32_t seg = (regen + 3) / 4;
                    if (6ull + z1 + z2 + z3 >= pay_size) FAIL(ERR_INVALID, "zstd literals: bad jump table");
                    // libzstd's MIN_LITERALS_FOR_4_STREAMS.  From 6 on, 3 * seg <= regen: the fourth stream regenerates
                    // regen - 3 * seg >= 0 symbols (0 at 6 and 9: a stream of one byte, the end marker alone)
                    if (regen < 6) FAIL(ERR_INVALID, "zstd literals: fewer than 6 literals in 4-stream mode");
                    so[0] = pay + 6; so[1] = so[0] + z1; so[2] = so[1] + z2; so[3] = so[2] + z3;
                    ss[0] = z1; ss[1] = z2; ss[2] = z3; ss[3] = pay_size - 6 - z1 - z2 - z3;
                    for (int k = 0; k < 4; k++) { dof[k] = seg * k; dn[k] = k < 3 ? seg : regen - 3 * seg; }
                }
                for (int k = 0; k < streams; k++) {
                    if (ss[k] == 0) FAIL(ERR_INVALID, "zstd literals: empty Huffman stream");
                    // codes are at most 11 bits: a longer stream cannot be consumed exactly (libzstd: corruption_detected); it also
                    // bounds the shared memory a stream is staged in
                    if ((uint64_t)ss[k] * 8 > (uint64_t)dn[k] * 11 + 16) FAIL(ERR_INVALID, "zstd literals: Huffman stream longer than its symbols allow");
                    zf::HufItem it{self, so[k], ss[k], dof[k], dn[k], streams == 4 ? (regen + 3) / 4 : 0u};
                    plan.huf_items.push_back(it);
                }
            }
            // sequences section header
            uint32_t q = hdr + csize;
            if (q >= bsize) FAIL(ERR_INVALID, "zstd sequences: missing section");
            uint32_t nseq = c[q++];
            if (nseq >= 128) {
                if (nseq == 255) {
                    if (q + 2 > bsize) FAIL(ERR_INVALID, "zstd sequences: truncated header");
                    nseq = c[q] + (c[q + 1] << 8) + 0x7F00; q += 2;
                } else {
                    if (q + 1 > bsize) FAIL(ERR_INVALID, "zstd sequences: truncated header");
                    nseq = ((nseq - 128) << 8) + c[q]; q += 1;
                }
            }
            b.n_seq = nseq;
            if (nseq == 0) {
                if (q != bsize) FAIL(ERR_INVALID, "zstd sequences: trailing bytes after an empty section");
                b.known_regen = regen;
            } else {
                if (q >= bsize) FAIL(ERR_INVALID, "zstd sequences: truncated header");
                uint8_t modes = c[q++];
                if (modes & 3) FAIL(ERR_INVALID, "zstd sequences: reserved mode bits set");
                b.modes = modes;
                for (int k = 0; k < 3; k++) {
                    int m = (modes >> (6 - 2 * k)) & 3;
                    if (m == zf::SM_PREDEF) { b.tbl[k] = (uint32_t)k; cur_tbl[k] = (uint32_t)k; }
                    else if (m == zf::SM_REPEAT) {
                        if (cur_tbl[k] == zf::NO_SLOT) FAIL(ERR_INVALID, "zstd sequences: repeat mode without a previous table");
                        if (cur_tbl[k] == PREV_SLOT) st.used_prev_tbl[k] = true;
                        b.tbl[k] = cur_tbl[k];
                    } else { b.tbl[k] = plan.n_slots++; b.defines |= (uint8_t)(1 << k); cur_tbl[k] = b.tbl[k]; }
                }
                b.seq_base = (uint32_t)plan.seq_total;
                plan.seq_total += nseq;
                if (plan.seq_total > 0xFFFFFFF0ull) FAIL(ERR_UNSUPPORTED, "job has too many sequences");
                plan.n_seq_blocks++;
                if (bsize - q > plan.max_seq_section) plan.max_seq_section = bsize - q;
                if (nseq <= 32) plan.n_tiny_seq_blocks++;
                else if (bsize - q > plan.max_seq_section_big) plan.max_seq_section_big = bsize - q;
            }
            b.seq_src = q;
        }
        known_total += b.known_regen;
        if (zf::needs_seq_kernel(b)) plan.big_seq.push_back((uint32_t)plan.blocks.size());
        if (!zf::tiny_lit_block(b)) plan.big_lit.push_back((uint32_t)plan.blocks.size());
        plan.blocks.push_back(b);
        p += content;
        if (last) { if (!last_part) FAIL(ERR_INVALID, "zstd frame: block chain changed between the passes"); break; }
    }
    if (last_part && checksum) {
        if (p + 4 > n) FAIL(ERR_EOF, "zstd frame: truncated checksum");
        st.has_checksum = 1; st.checksum = (uint32_t)s[p] | ((uint32_t)s[p + 1] << 8) | ((uint32_t)s[p + 2] << 16) | ((uint32_t)s[p + 3] << 24);
        p += 4;
        plan.n_checksums++;
    }
    st.n_blocks = (uint32_t)(plan.blocks.size() - first_block);
    st.n_seq = (uint32_t)(plan.seq_total - first_seq);
    if (first) {
        zf::FrameDesc& fd = plan.frames[fd_at];
        fd.n_blocks = st.n_blocks; fd.n_seq = st.n_seq;
        fd.has_checksum = st.has_checksum; fd.checksum = st.checksum;
    }
    return 0;
}

int check_frame_total(uint64_t n_seq, uint64_t known_total, uint64_t dst_size, std::string& err) {
    if (n_seq == 0 && known_total != dst_size)
        FAIL(ERR_INVALID, "zstd frame regenerates %llu bytes but the section header says %llu",
             (unsigned long long)known_total, (unsigned long long)dst_size);
    return 0;
}

int walk_frame(const uint8_t* frame, uint64_t src_off, uint64_t src_size, uint64_t dst_off, uint64_t dst_size,
               JobPlan& plan, std::string& err) {
    RangeState st;
    if (int rc = walk_frame_part(frame, src_off, src_size, dst_off, dst_size, 0, 0, true, true, st, plan, err)) return rc;
    return check_frame_total(st.n_seq, st.known_total, dst_size, err);
}

void JobPlan::finalize(uint32_t small_max_symbols) {
    // big = the streams of a 4-stream block whose streams regenerate more than small_max symbols: classified per BLOCK, so the
    // four streams of a block stay together and in order (k_huf_decode_big runs them as one thread-block cluster)
    auto is_big = [&](const zf::HufItem& it) { return it.seg_symbols > small_max_symbols; };
    auto mid = std::stable_partition(huf_items.begin(), huf_items.end(), is_big);
    n_huf_big = (uint32_t)(mid - huf_items.begin());
    max_huf_stream = max_huf_small = 0;
    for (size_t i = 0; i < huf_items.size(); i++) {
        uint32_t& m = i < n_huf_big ? max_huf_stream : max_huf_small;
        m = std::max(m, huf_items[i].src_size);
    }
}

}  // namespace fw

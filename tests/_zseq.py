"""zstd frames built to order from an explicit list of sequences (libzstd's ZSTD_compressSequences), a plain LZ77 replay as
the reference, and a small pure-Python reader of sequence sections that reports which codes and modes a frame really holds.

libzstd's own match finder decides what a frame made from data contains; here the test decides: far offsets at every offset
code, the repeat-offset special cases (RFC 8878 3.1.1.5), literal and match lengths at the code boundaries, block shapes.
libzstd still chooses how each offset is coded (ZSTD_finalizeOffBase: an offset equal to rep1 or rep2, or with ll == 0 to
rep0 - 1, becomes a repeat code), so every case reads its frame back with `frame_codes` to prove that its edge is there.

There is no zstd.h on the machines that run the suite: the parameter ids below are libzstd 1.5.5's (experimental ones
included), so the module refuses any other version."""
import ctypes as C
import ctypes.util

import pytest

ZSTD_VERSION = 10505

# ZSTD_cParameter / ZSTD_dParameter ids of libzstd 1.5.5
C_FORMAT, C_WINDOW_LOG, C_MIN_MATCH = 10, 101, 105
C_CONTENT_SIZE, C_CHECKSUM = 200, 201
C_LITERAL_MODE, C_BLOCK_DELIMITERS, C_VALIDATE = 1002, 1008, 1009
C_REPCODE_SEARCH = 1016                 # ZSTD_c_searchForExternalRepcodes: left at auto, levels below 10 never emit repeat codes
D_WINDOW_LOG_MAX, D_FORMAT = 100, 1000
LIT_HUFFMAN, LIT_RAW = 1, 2
BLOCK = 128 * 1024                      # Block_Maximum_Size

_lib = None


class ZSeq(C.Structure):
    _fields_ = [("offset", C.c_uint32), ("litLength", C.c_uint32), ("matchLength", C.c_uint32), ("rep", C.c_uint32)]


def lib():
    """libzstd, or a skip when it is missing or not the version whose parameter ids are written down here."""
    global _lib
    if _lib is None:
        try:
            L = C.CDLL(ctypes.util.find_library("zstd") or "libzstd.so.1")
        except OSError as e:
            pytest.skip(f"libzstd not loadable: {e}")
        if L.ZSTD_versionNumber() != ZSTD_VERSION:
            pytest.skip(f"libzstd {L.ZSTD_versionNumber()}: the parameter ids of tests/_zseq.py are those of {ZSTD_VERSION}")
        L.ZSTD_createCCtx.restype = C.c_void_p
        L.ZSTD_createDCtx.restype = C.c_void_p
        L.ZSTD_freeCCtx.argtypes = [C.c_void_p]
        L.ZSTD_freeDCtx.argtypes = [C.c_void_p]
        L.ZSTD_CCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.ZSTD_CCtx_setParameter.restype = C.c_size_t
        L.ZSTD_DCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.ZSTD_DCtx_setParameter.restype = C.c_size_t
        L.ZSTD_isError.argtypes = [C.c_size_t]
        L.ZSTD_getErrorName.argtypes = [C.c_size_t]
        L.ZSTD_getErrorName.restype = C.c_char_p
        L.ZSTD_compressBound.argtypes = [C.c_size_t]
        L.ZSTD_compressBound.restype = C.c_size_t
        L.ZSTD_compressSequences.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]
        L.ZSTD_compressSequences.restype = C.c_size_t
        L.ZSTD_decompressDCtx.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t]
        L.ZSTD_decompressDCtx.restype = C.c_size_t
        _lib = L
    return _lib


def _ok(rc, what):
    L = lib()
    if L.ZSTD_isError(rc):
        raise RuntimeError(f"{what}: {L.ZSTD_getErrorName(rc).decode()}")
    return rc


# ---- the reference -------------------------------------------------------------------------------------------------
def replay(seqs, literals: bytes) -> bytes:
    """LZ77 replay of (literal length, match length, offset) triples over `literals`; the literals left over after the last
    sequence end the output.  Offsets are raw byte distances (no repeat codes).  Overlapping copies go byte by byte; a long
    overlapping copy (the offset-1 runs that fill the space in front of a far match) is the periodic extension of its source,
    which is what the byte loop computes, written as one slice so that a few hundred MB replay in seconds."""
    out = bytearray()
    lp = 0
    for ll, ml, off in seqs:
        out += literals[lp:lp + ll]
        lp += ll
        if ml == 0:
            continue
        d = len(out)
        assert 1 <= off <= d, (off, d)
        if off >= ml:
            out += out[d - off:d - off + ml]
        elif ml <= 4096:
            for k in range(ml):
                out.append(out[d - off + k])
        else:
            src = bytes(out[d - off:d])
            out += (src * (ml // off + 1))[:ml]
    out += literals[lp:]
    return bytes(out)


# ---- the builder ---------------------------------------------------------------------------------------------------
def build(blocks, window_log=20, single_segment=True, checksum=False, literal_mode=0):
    """A magicless frame of explicit blocks.  `blocks` is a list of blocks; a block is a list of (literals, match length,
    offset) with raw offsets, ended by its trailing literals (a bytes object, possibly empty).  Returns (payload, frame) where
    payload is `replay` of the whole list.  `single_segment`=False clears the content-size flag, so the header carries a
    window descriptor of 2^window_log instead of the content size; `literal_mode` 1 forces Huffman literals, 2 raw."""
    L = lib()
    seqs, flat, lits = [], [], bytearray()
    for blk in blocks:
        *body, tail = blk
        for lit, ml, off in body:
            seqs.append((0 if ml == 0 else off, len(lit), ml))
            flat.append((len(lit), ml, off))
            lits += lit
        seqs.append((0, len(tail), 0))                      # block delimiter: offset 0, match length 0, the trailing literals
        flat.append((len(tail), 0, 0))
        lits += tail
    payload = replay(flat, bytes(lits))
    cc = L.ZSTD_createCCtx()
    try:
        params = [(C_FORMAT, 1), (C_WINDOW_LOG, window_log), (C_MIN_MATCH, 3), (C_CONTENT_SIZE, int(single_segment)),
                  (C_CHECKSUM, int(checksum)), (C_BLOCK_DELIMITERS, 1), (C_VALIDATE, 1), (C_LITERAL_MODE, literal_mode), (C_REPCODE_SEARCH, 1)]
        for p, v in params:
            _ok(L.ZSTD_CCtx_setParameter(cc, p, v), f"parameter {p}")
        arr = (ZSeq * len(seqs))(*[ZSeq(o, ll, ml, 0) for o, ll, ml in seqs])
        cap = L.ZSTD_compressBound(len(payload)) + 4 * len(blocks) + 1024
        out = C.create_string_buffer(cap)
        n = _ok(L.ZSTD_compressSequences(cc, out, cap, arr, len(seqs), payload, len(payload)), "ZSTD_compressSequences")
        return payload, out.raw[:n]
    finally:
        L.ZSTD_freeCCtx(cc)


def libzstd_decompress(frame: bytes, size: int, window_log_max=30) -> bytes:
    """libzstd's decoder with its window limit raised (its default refuses windows above 2^27)."""
    L = lib()
    dc = L.ZSTD_createDCtx()
    try:
        _ok(L.ZSTD_DCtx_setParameter(dc, D_FORMAT, 1), "format")
        _ok(L.ZSTD_DCtx_setParameter(dc, D_WINDOW_LOG_MAX, window_log_max), "windowLogMax")
        buf = C.create_string_buffer(size + 1)
        n = _ok(L.ZSTD_decompressDCtx(dc, buf, size + 1, frame, len(frame)), "ZSTD_decompressDCtx")
        return buf.raw[:n]
    finally:
        L.ZSTD_freeDCtx(dc)


# ---- reading a frame back ------------------------------------------------------------------------------------------
LL_BASE = list(range(16)) + [16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536]
LL_BITS = [0] * 16 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]
ML_BASE = list(range(3, 35)) + [35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539]
ML_BITS = [0] * 32 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]
_PREDEF = {  # RFC 8878 3.1.1.3.2.2: (accuracy log, distribution)
    "ll": (6, [4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1]),
    "of": (5, [1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1]),
    "ml": (6, [1, 4, 3, 2, 2, 2, 2, 2, 2] + [1] * 37 + [-1] * 7),
}
_MAX_SYM = {"ll": 35, "of": 31, "ml": 52}
MODE_NAMES = ("predefined", "rle", "fse", "repeat")


def _fse_table(al, norm):
    """Decoding table of an FSE distribution (RFC 8878 4.1.1): a list of (symbol, bits, baseline)."""
    size = 1 << al
    sym = [0] * size
    high = size - 1
    nxt = []
    for s, p in enumerate(norm):
        if p == -1:
            sym[high] = s
            high -= 1
        nxt.append(1 if p == -1 else p)
    step, pos = (size >> 1) + (size >> 3) + 3, 0
    for s, p in enumerate(norm):
        for _ in range(max(p, 0)):
            sym[pos] = s
            pos = (pos + step) & (size - 1)
            while pos > high:
                pos = (pos + step) & (size - 1)
    table = []
    for u in range(size):
        s = sym[u]
        x = nxt[s]
        nxt[s] += 1
        nb = al - (x.bit_length() - 1)
        table.append((s, nb, (x << nb) - size))
    return table


def _read_ncount(buf, pos, max_sym):
    """FSE table description (RFC 8878 4.1.1) at buf[pos]: (accuracy log, distribution, bytes used)."""
    bit = 0

    def peek(n):
        return (int.from_bytes(buf[pos + (bit >> 3):pos + (bit >> 3) + 5], "little") >> (bit & 7)) & ((1 << n) - 1)

    al = peek(4) + 5
    bit += 4
    remaining, threshold, nb = (1 << al) + 1, 1 << al, al + 1
    norm, prev0 = [], False
    while remaining > 1:
        if prev0:
            while True:
                r = peek(2)
                bit += 2
                norm += [0] * r
                if r != 3:
                    break
        mx = 2 * threshold - 1 - remaining
        v = peek(nb)
        if (v & (threshold - 1)) < mx:
            count = v & (threshold - 1)
            bit += nb - 1
        else:
            count = v & (2 * threshold - 1)
            if count >= threshold:
                count -= mx
            bit += nb
        count -= 1
        remaining -= abs(count)
        norm.append(count)
        prev0 = count == 0
        while remaining < threshold:
            nb -= 1
            threshold >>= 1
    assert remaining == 1 and len(norm) <= max_sym + 1, "bad FSE table description"
    return al, norm, (bit + 7) >> 3


class _Back:
    """Backward bit reader (RFC 8878 4.1): reads from the top of a stream whose last byte holds the end marker; bits below the
    start read as zero."""

    def __init__(self, data: bytes):
        self.v = int.from_bytes(data, "little")
        self.p = 8 * (len(data) - 1) + data[-1].bit_length() - 1

    def read(self, n):
        self.p -= n
        if n == 0:
            return 0
        if self.p >= 0:
            return (self.v >> self.p) & ((1 << n) - 1)
        return (self.v << -self.p) & ((1 << n) - 1)


class Block:
    """One block of a frame as `frame_codes` reads it: type, size; for compressed blocks the literals section (type, streams,
    sizes, Huffman depth when a tree is described) and the sequences (codes, values, resolved offsets)."""

    def __init__(self, btype, size):
        self.btype, self.size = btype, size            # "raw", "rle", "compressed"
        self.lit_type = self.lit_streams = self.lit_regen = self.huf_depth = None
        self.modes = None                                # the Symbol_Compression_Modes byte
        self.ll_mode = self.of_mode = self.ml_mode = None
        self.al = {}                                     # accuracy log of each table this block describes (FSE mode)
        self.seq_bytes = 0                               # size of the sequence bitstream
        self.seqs = []                                   # (ll_code, ml_code, of_code, offset_value, ll, ml, offset)

    @property
    def regen(self):
        if self.btype != "compressed":
            return self.size
        return self.lit_regen + sum(s[5] for s in self.seqs)


def frame_codes(frame: bytes):
    """Blocks of a magicless zstd frame (valid frames only), with every sequence's codes and resolved offset.
    Returns (header, blocks): header = dict(single_segment, window, content_size, checksum)."""
    f = bytes(frame)
    fhd = f[0]
    fcs_flag, single, checksum, dict_flag = fhd >> 6, (fhd >> 5) & 1, (fhd >> 2) & 1, fhd & 3
    p, window = 1, None
    if not single:
        wd = f[p]; p += 1
        base = 1 << (10 + (wd >> 3))
        window = base + (base >> 3) * (wd & 7)
    p += (0, 1, 2, 4)[dict_flag]
    fcs_size = (1 if single else 0, 2, 4, 8)[fcs_flag]
    fcs = int.from_bytes(f[p:p + fcs_size], "little") + (256 if fcs_size == 2 else 0) if fcs_size else None
    p += fcs_size
    hdr = dict(single_segment=bool(single), window=fcs if single else window, content_size=fcs, checksum=bool(checksum))
    blocks = []
    reps = [1, 4, 8]
    prev = {"ll": None, "of": None, "ml": None}
    while True:
        bh = int.from_bytes(f[p:p + 3], "little"); p += 3
        last, bt, bsize = bh & 1, (bh >> 1) & 3, bh >> 3
        b = Block(("raw", "rle", "compressed")[bt], bsize)
        blocks.append(b)
        if bt == 2:
            _read_block(f[p:p + bsize], b, reps, prev)
        p += 1 if bt == 1 else bsize
        if last:
            break
    return hdr, blocks


def _read_block(c, b, reps, prev):
    b0 = c[0]
    lt, sf = b0 & 3, (b0 >> 2) & 3
    b.lit_type = ("raw", "rle", "huffman", "treeless")[lt]
    if lt < 2:
        hsz = (1, 2, 1, 3)[sf]
        regen = b0 >> 3 if hsz == 1 else (b0 >> 4) | (c[1] << 4) | ((c[2] << 12) if hsz == 3 else 0)
        csize = regen if lt == 0 else 1
        b.lit_streams = 0
    else:
        hsz = (3, 3, 4, 5)[sf]
        v = int.from_bytes(c[:hsz], "little") >> 4
        bits = (10, 10, 14, 18)[sf]
        regen, csize = v & ((1 << bits) - 1), v >> bits
        b.lit_streams = 1 if sf == 0 else 4
        if lt == 2:
            from _zhuf import read_tree                  # (tests/_zhuf.py reads Huffman sections; it builds on this module)
            w, _ = read_tree(c[hsz:hsz + csize])
            b.huf_depth = sum(1 << (x - 1) for x in w if x).bit_length() - 1
    b.lit_regen = regen
    q = hsz + csize
    n = c[q]
    if n == 0:
        return
    if n < 128:
        q += 1
    elif n < 255:
        n = ((n - 128) << 8) + c[q + 1]; q += 2
    else:
        n = c[q + 1] + (c[q + 2] << 8) + 0x7F00; q += 3
    b.modes = c[q]; q += 1
    tables = {}
    for kind, shift in (("ll", 6), ("of", 4), ("ml", 2)):
        mode = (b.modes >> shift) & 3
        setattr(b, kind + "_mode", MODE_NAMES[mode])
        if mode == 0:
            al, norm = _PREDEF[kind]
            tables[kind] = (al, _fse_table(al, norm))
        elif mode == 1:
            tables[kind] = (0, [(c[q], 0, 0)]); q += 1
        elif mode == 2:
            al, norm, used = _read_ncount(c, q, _MAX_SYM[kind]); q += used
            tables[kind] = (al, _fse_table(al, norm))
            b.al[kind] = al
        else:
            tables[kind] = prev[kind]
        prev[kind] = tables[kind]
    (all_, tll), (aof, tof), (aml, tml) = tables["ll"], tables["of"], tables["ml"]
    b.seq_bytes = len(c) - q
    rd = _Back(bytes(c[q:]))
    sll, sof, sml = rd.read(all_), rd.read(aof), rd.read(aml)
    for i in range(n):
        llc, ofc, mlc = tll[sll][0], tof[sof][0], tml[sml][0]
        ov = (1 << ofc) + rd.read(ofc)
        ml = ML_BASE[mlc] + rd.read(ML_BITS[mlc])
        ll = LL_BASE[llc] + rd.read(LL_BITS[llc])
        if ov > 3:
            off = ov - 3
            reps[:] = [off, reps[0], reps[1]]
        else:
            idx = ov - 1 + (ll == 0)
            if idx == 0:
                off = reps[0]
            elif idx == 1:
                off = reps[1]; reps[:] = [off, reps[0], reps[2]]
            elif idx == 2:
                off = reps[2]; reps[:] = [off, reps[0], reps[1]]
            else:
                off = reps[0] - 1; reps[:] = [off, reps[0], reps[1]]
        b.seqs.append((llc, mlc, ofc, ov, ll, ml, off))
        if i + 1 < n:
            for t, kind in ((tll, "ll"), (tml, "ml"), (tof, "of")):
                _, nb, base = t[{"ll": sll, "ml": sml, "of": sof}[kind]]
                nv = base + rd.read(nb)
                if kind == "ll": sll = nv
                elif kind == "ml": sml = nv
                else: sof = nv
    assert rd.p == 0, f"sequence bitstream not consumed exactly ({rd.p} bits left)"


def all_seqs(blocks):
    return [s for b in blocks for s in b.seqs]


def regenerate(frame: bytes, content: bytes) -> bytes:
    """The frame regenerated from `frame_codes`' sequences with the literals taken out of `content` (the frame's known
    content) at the positions those sequences give them: equal to `content` only if every length and offset was read right."""
    _, blocks = frame_codes(frame)
    flat, lits, pos = [], bytearray(), 0
    for b in blocks:
        if b.btype != "compressed":
            flat.append((b.size, 0, 0)); lits += content[pos:pos + b.size]; pos += b.size
            continue
        start = len(lits)
        for *_, ll, ml, off in b.seqs:
            flat.append((ll, ml, off)); lits += content[pos:pos + ll]; pos += ll + ml
        tail = b.lit_regen - (len(lits) - start)
        flat.append((tail, 0, 0)); lits += content[pos:pos + tail]; pos += tail
    return replay(flat, bytes(lits))

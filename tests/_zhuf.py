"""Huffman literals sections (RFC 8878 3.1.1.3.1, 4.2) built to order, blocks and frames around them, and a plain reader.

libzstd's encoder picks the tree, its depth, the weight form and the stream split by itself; here the test does: every
depth from 1 to 11, fixed-length trees, direct and FSE-compressed weight descriptions of any count, FSE weight streams that
end on either state, streams of any length down to the end marker alone, and treeless sections that reuse a tree.

`read_literals` decodes a section one bit at a time by walking the canonical code (per-length first codes and counts, no
decode tables) and reports what the section holds, so that every case can prove that the edge it is named after is there.
The FSE pieces (`_fse_table`, `_read_ncount`, `_Back`) and libzstd come from tests/_zseq.py."""
import _zseq as Z

MAX_BITS = 11                           # RFC 8878 4.2.1: Max_Number_of_Bits


# ---- trees ---------------------------------------------------------------------------------------------------------
def weights_of_lengths(lengths):
    """Full weight vector (index = symbol, up to the last symbol with a code) of a complete prefix code given as
    {symbol: code length}."""
    depth = max(lengths.values())
    assert sum(1 << (depth - n) for n in lengths.values()) == 1 << depth, "code lengths do not fill the code space"
    w = [0] * (max(lengths) + 1)
    for s, n in lengths.items():
        w[s] = depth + 1 - n
    return w


def depth_of(weights):
    """Max_Number_of_Bits of a full weight vector; asserts that it describes a complete code."""
    total = sum(1 << (x - 1) for x in weights if x)
    depth = total.bit_length() - 1
    assert total == 1 << depth, f"weights sum to {total}, not a power of two"
    return depth


def canonical_code(weights):
    """{symbol: (code, length)}: codes in order of ascending weight, then symbol, counting up from 0 (RFC 8878 4.2.1.4)."""
    depth = depth_of(weights)
    out, pos = {}, 0
    for w in range(1, depth + 1):
        for s, x in enumerate(weights):
            if x == w:
                out[s] = (pos >> (w - 1), depth + 1 - w)
                pos += 1 << (w - 1)
    assert pos == 1 << depth
    return out


# ---- the writer ----------------------------------------------------------------------------------------------------
def huffman_stream(data: bytes, code, pad_bits="") -> bytes:
    """One Huffman bitstream of `data`: read backwards, its first symbol right below the end marker.  `pad_bits` (a string of
    0/1) goes below the last symbol: such a stream does not end on its first bit (a corrupt stream)."""
    parts = ["1"]
    for b in data:
        c, n = code[b]
        parts.append(format(c, f"0{n}b"))
    bits = "".join(parts) + pad_bits
    return int(bits, 2).to_bytes((len(bits) + 7) // 8, "little")


def write_ncount(al, norm):
    """FSE table description (RFC 8878 4.1.1) of `norm` (counts, -1 for less than one), the inverse of _zseq._read_ncount."""
    assert sum(abs(c) for c in norm) == 1 << al, norm
    acc, nbit = al - 5, 4
    remaining, threshold, nb = (1 << al) + 1, 1 << al, al + 1
    i = 0
    while remaining > 1:
        if i and norm[i - 1] == 0:                                  # after a zero: the run of zeros that follows, 2 bits at a time
            z = 0
            while norm[i + z] == 0:
                z += 1
            i += z
            while z >= 3:
                acc |= 3 << nbit; nbit += 2; z -= 3
            acc |= z << nbit; nbit += 2
        c = norm[i]
        v, mx = c + 1, 2 * threshold - 1 - remaining
        if v < mx:
            acc |= v << nbit; nbit += nb - 1
        else:
            acc |= (v + mx if v >= threshold else v) << nbit; nbit += nb
        remaining -= abs(c)
        i += 1
        while remaining < threshold:
            nb -= 1
            threshold >>= 1
    assert remaining == 1 and all(c == 0 for c in norm[i:])
    return acc.to_bytes((nbit + 7) // 8, "little")


def normalize(values, al, low=()):
    """An FSE distribution over the symbols of `values` (weights here) at accuracy log `al`: counts proportional to the
    occurrences, at least 1 each; the symbols in `low` get -1 (less than one), whether they occur or not (a weight stream of
    one value needs a second symbol: with one, no state reads a bit and the stream cannot end)."""
    occ = {}
    for v in values:
        occ[v] = occ.get(v, 0) + 1
    norm = [0] * (max(list(occ) + list(low)) + 1)
    for s in low:
        norm[s] = -1
    free = (1 << al) - len(low)
    rest = [s for s in occ if s not in low]
    assert len(rest) <= free, "too many symbols for this accuracy log"
    tot = sum(occ[s] for s in rest)
    for s in rest:
        norm[s] = max(1, occ[s] * free // tot)
    while sum(norm[s] for s in rest) > free:
        norm[max(rest, key=lambda s: norm[s])] -= 1
    norm[max(rest, key=lambda s: occ[s])] += free - sum(norm[s] for s in rest)
    return norm


def fse_weights(ws, al=6, low=(), norm=None, slack=""):
    """FSE-compressed weight description (header byte < 128): `ws` (the explicit weights) coded with two interleaved states
    over one backward bitstream.  A stream of n weights ends on state 1 when n is even (its update after weight n - 2 reads
    past the start), on state 2 when n is odd.  `slack` (bits, at most the width of that last read minus one) is placed
    below everything: the final read is then partly inside the stream."""
    norm = norm or normalize(ws, al, low)
    table = Z._fse_table(al, norm)
    enc = {}                                                     # symbol -> next state -> (state, bits, width)
    for u, (s, nb, base) in enumerate(table):
        for v in range(1 << nb):
            enc.setdefault(s, {})[base + v] = (u, v, nb)
    first = {}
    for u, (s, nb, base) in enumerate(table):                   # start states: the widest read of the symbol
        if s not in first or nb > table[first[s]][1]:
            first[s] = u
    n = len(ws)
    assert n >= 2
    st = [None] * n
    st[n - 1], st[n - 2] = first[ws[n - 1]], first[ws[n - 2]]
    assert len(slack) < table[st[n - 2]][1]
    chunks = []                                                  # written bottom up
    for i in range(n - 3, -1, -1):
        u, v, nb = enc[ws[i]][st[i + 2]]
        st[i] = u
        if nb:
            chunks.append(format(v, f"0{nb}b"))
    bits = "1" + format(st[0], f"0{al}b") + format(st[1], f"0{al}b") + "".join(reversed(chunks)) + slack
    body = int(bits, 2).to_bytes((len(bits) + 7) // 8, "little")
    desc = write_ncount(al, norm) + body
    assert len(desc) < 128, len(desc)
    return bytes([len(desc)]) + desc


def direct_weights(ws):
    """Direct weight description (header byte 127 + n): n <= 128 explicit weights as 4-bit fields, the first in the high half."""
    n = len(ws)
    assert 1 <= n <= 128 and all(0 <= w < 16 for w in ws)
    padded = list(ws) + [0] * (n & 1)
    return bytes([127 + n]) + bytes((padded[i] << 4) | padded[i + 1] for i in range(0, n + (n & 1), 2))


def tree_description(weights, form="direct", **kw):
    """The description of a full weight vector: every weight but the last symbol's, which is implied."""
    depth_of(weights)
    assert weights[-1] != 0
    ws = weights[:-1]
    return direct_weights(ws) if form == "direct" else fse_weights(ws, **kw)


def literals_header(lt, sf, regen, csize):
    """Literals section header of a Huffman (lt 2) or treeless (lt 3) section in size format sf."""
    bits = (10, 10, 14, 18)[sf]
    assert regen < 1 << bits and csize < 1 << bits, (sf, regen, csize)
    v = lt | (sf << 2) | (regen << 4) | (csize << (4 + bits))
    return v.to_bytes((3, 3, 4, 5)[sf], "little")


def literals_section(data: bytes, weights, streams=4, form="direct", treeless=False, sf=None, stream_bytes=None, desc=None, **kw):
    """A Huffman (or treeless) literals section of `data` under the tree `weights`.  Four streams split at
    segment = (regen + 3) // 4 behind a jump table; `stream_bytes` replaces the encoded streams and `desc` the tree
    description (corrupt sections); sf: the smallest size format that fits unless given."""
    code = canonical_code(weights)
    regen = len(data)
    if stream_bytes is None:
        if streams == 1:
            stream_bytes = [huffman_stream(data, code)]
        else:
            seg = (regen + 3) // 4
            stream_bytes = [huffman_stream(data[k * seg:(k + 1) * seg], code) for k in range(4)]
    body = b"" if treeless else desc if desc is not None else tree_description(weights, form, **kw)
    if streams == 4:
        body += b"".join(len(s).to_bytes(2, "little") for s in stream_bytes[:3])
    body += b"".join(stream_bytes)
    if sf is None:
        sf = 0 if streams == 1 else next(f for f in (1, 2, 3) if max(regen, len(body)) < 1 << (10, 10, 14, 18)[f])
    return literals_header(3 if treeless else 2, sf, regen, len(body)) + body


def block(content: bytes, last=False, btype=2) -> bytes:
    return ((btype << 1) | int(last) | (len(content) << 3)).to_bytes(3, "little") + content


def frame(blocks, content_size, fcs_bytes=None) -> bytes:
    """A magicless single-segment frame of `blocks` (each a block header and its content) that regenerates content_size
    bytes; the content size field takes 1, 2 or 4 bytes (smallest that fits unless given)."""
    if fcs_bytes is None:
        fcs_bytes = 1 if content_size < 256 else 2 if content_size < 65536 + 256 else 4
    flag = {1: 0, 2: 1, 4: 2}[fcs_bytes]
    v = content_size - 256 if fcs_bytes == 2 else content_size
    assert 0 <= v < 1 << (8 * fcs_bytes)
    return bytes([(flag << 6) | 0x20]) + v.to_bytes(fcs_bytes, "little") + b"".join(blocks)


def literals_only(sections, fcs_bytes=None):
    """A frame of literals-only compressed blocks (Number_of_Sequences = 0), one per (section, regenerated size)."""
    bl = [block(s + b"\0", last=i == len(sections) - 1) for i, (s, _) in enumerate(sections)]
    return frame(bl, sum(n for _, n in sections), fcs_bytes)


def splice(frame_bytes: bytes, make_section):
    """Replaces the raw literals section of every compressed block of a magicless frame (Z.build(..., literal_mode=LIT_RAW))
    by make_section(index of the block among the compressed ones, literal bytes) and fixes the block size up."""
    f = bytes(frame_bytes)
    fhd = f[0]
    assert fhd & 0x20 and not fhd & 3 and not fhd & 4, "single segment, no dictionary, no checksum"
    p = 1 + (1, 2, 4, 8)[fhd >> 6]
    out, k = bytearray(f[:p]), 0
    while True:
        bh = int.from_bytes(f[p:p + 3], "little")
        last, bt, size = bh & 1, (bh >> 1) & 3, bh >> 3
        c = f[p + 3:p + 3 + (1 if bt == 1 else size)]
        if bt == 2:
            b0 = c[0]
            assert b0 & 3 == 0, "raw literals expected"
            sf = (b0 >> 2) & 3
            hsz = (1, 2, 1, 3)[sf]
            regen = b0 >> 3 if hsz == 1 else (b0 >> 4) | (c[1] << 4) | ((c[2] << 12) if hsz == 3 else 0)
            c = make_section(k, c[hsz:hsz + regen]) + c[hsz + regen:]
            k += 1
        out += block(c, last, bt)
        p += 3 + (1 if bt == 1 else size)
        if last:
            return bytes(out + f[p:])


# ---- the reader ----------------------------------------------------------------------------------------------------
class Literals:
    """What a literals section holds, as `read_literals` found it."""

    def __init__(self):
        self.lit_type = self.sf = self.regen = self.csize = self.hsize = None
        self.weights = None          # full weight vector (the implied last weight included)
        self.form = None             # "direct" or "fse" (a described tree), None (treeless: the previous tree)
        self.n_explicit = None       # weights written in the description
        self.al = self.norm = None   # FSE weight descriptions: accuracy log and distribution
        self.end_state = None        # FSE: the state whose read went past the start of the weight stream (1 or 2)
        self.depth = None
        self.stream_sizes = []       # bytes
        self.counts = []             # symbols per stream
        self.marker_bits = []        # bit of the end marker in each stream's last byte
        self.data = None


def read_tree(c, lit=None):
    """The Huffman tree description at c[0] (RFC 8878 4.2.1): (full weights, bytes used).  Fills form, counts, al, end state
    of `lit` when given.  Raises ValueError where a decoder must refuse."""
    lit = lit or Literals()
    hb = c[0]
    if hb >= 128:
        n = hb - 127
        used = 1 + (n + 1) // 2
        if used > len(c):
            raise ValueError("direct weights past the section")
        w = [(c[1 + i // 2] >> (0 if i % 2 else 4)) & 15 for i in range(n)]
        lit.form = "direct"
    else:
        if hb + 1 > len(c) or hb < 2:
            raise ValueError("FSE weights past the section")
        al, norm, nused = Z._read_ncount(c, 1, 12)
        if al > 6:
            raise ValueError("accuracy log of the weights above 6")
        if nused >= hb:
            raise ValueError("no weight bitstream")
        t = Z._fse_table(al, norm)
        stream = bytes(c[1 + nused:1 + hb])
        if stream[-1] == 0:
            raise ValueError("weight bitstream without end marker")
        rd = Z._Back(stream)
        s1, s2 = rd.read(al), rd.read(al)
        if rd.p < 0:
            raise ValueError("weight bitstream shorter than its states")
        w = []
        while True:
            if len(w) > 253:
                raise ValueError("more than 255 weights")
            sym, nb, base = t[s1]; w.append(sym); s1 = base + rd.read(nb)
            if rd.p < 0:
                w.append(t[s2][0]); lit.end_state = 1; break
            sym, nb, base = t[s2]; w.append(sym); s2 = base + rd.read(nb)
            if rd.p < 0:
                w.append(t[s1][0]); lit.end_state = 2; break
        lit.form, lit.al, lit.norm = "fse", al, norm
        used = 1 + hb
    lit.n_explicit = len(w)
    if any(x > MAX_BITS for x in w):
        raise ValueError("weight above 11")
    total = sum(1 << (x - 1) for x in w if x)
    if total == 0:
        raise ValueError("no weights")
    depth = total.bit_length()
    left = (1 << depth) - total
    if left & (left - 1):
        raise ValueError("weights do not leave a power of two")
    w.append(left.bit_length())
    if w.count(1) < 2:
        raise ValueError("fewer than two weight-1 symbols")          # (libzstd's HUF_readStats; the count is even by construction)
    return w, used


def _decode_stream(s: bytes, weights, depth):
    """Symbols of one stream, one bit at a time down the canonical code: (bytes, end marker bit)."""
    if not s or s[-1] == 0:
        raise ValueError("stream without end marker")
    count, first, syms = [0] * (depth + 1), [0] * (depth + 2), [[] for _ in range(depth + 1)]
    for sym, x in enumerate(weights):
        if x:
            count[depth + 1 - x] += 1
            syms[depth + 1 - x].append(sym)
    for n in range(depth - 1, 0, -1):                            # the longest codes start at 0
        first[n] = (first[n + 1] + count[n + 1]) >> 1
    bits = bin(int.from_bytes(s, "little"))[3:]                  # below the end marker, top bit first
    out, i = bytearray(), 0
    while i < len(bits):
        code = 0
        for n in range(1, depth + 1):
            if i >= len(bits):
                raise ValueError("stream ends inside a code")
            code = 2 * code + (bits[i] == "1")
            i += 1
            if 0 <= code - first[n] < count[n]:
                out.append(syms[n][code - first[n]])
                break
    return bytes(out), s[-1].bit_length() - 1


def read_literals(c, prev_weights=None) -> Literals:
    """A Huffman or treeless literals section at c[0], decoded; raises ValueError where a decoder must refuse (libzstd's and
    the RFC's rules, and the 11-bit depth limit)."""
    lit = Literals()
    b0 = c[0]
    lt, sf = b0 & 3, (b0 >> 2) & 3
    assert lt >= 2, "not a Huffman literals section"
    hsz = (3, 3, 4, 5)[sf]
    bits = (10, 10, 14, 18)[sf]
    v = int.from_bytes(c[:hsz], "little") >> 4
    lit.lit_type, lit.sf, lit.hsize = ("huffman", "treeless")[lt - 2], sf, hsz
    lit.regen, lit.csize = v & ((1 << bits) - 1), v >> bits
    streams = 1 if sf == 0 else 4
    if streams == 4 and lit.regen < 6:
        raise ValueError("fewer than 6 literals in 4-stream mode")
    sec = bytes(c[hsz:hsz + lit.csize])
    if len(sec) < lit.csize:
        raise ValueError("section past the block")
    if lt == 2:
        lit.weights, used = read_tree(sec, lit)
    else:
        if prev_weights is None:
            raise ValueError("treeless section without a previous tree")
        lit.weights, used = list(prev_weights), 0
    lit.depth = sum(1 << (x - 1) for x in lit.weights if x).bit_length() - 1
    if lit.depth > MAX_BITS:
        raise ValueError("Huffman tree deeper than 11 bits")
    pay = sec[used:]
    if streams == 1:
        parts, want = [pay], [lit.regen]
    else:
        if len(pay) < 10:
            raise ValueError("jump table and four streams need 10 bytes")
        z = [int.from_bytes(pay[2 * k:2 * k + 2], "little") for k in range(3)]
        if 6 + sum(z) >= len(pay):
            raise ValueError("jump table past the section")
        o = [6, 6 + z[0], 6 + z[0] + z[1], 6 + sum(z), len(pay)]
        parts = [pay[o[k]:o[k + 1]] for k in range(4)]
        seg = (lit.regen + 3) // 4
        want = [seg, seg, seg, lit.regen - 3 * seg]
    out = bytearray()
    for s, n in zip(parts, want):
        d, m = _decode_stream(s, lit.weights, lit.depth)
        lit.stream_sizes.append(len(s)); lit.counts.append(len(d)); lit.marker_bits.append(m)
        if len(d) != n:
            raise ValueError(f"stream decodes {len(d)} symbols, not {n}")
        out += d
    lit.data = bytes(out)
    return lit


def frame_literals(frame_bytes: bytes):
    """`read_literals` of every Huffman and treeless section of a magicless frame, in order (a treeless section reads with
    the tree of the last described one), with the frame's block kinds: a list of (block type, Literals or None)."""
    _, blocks = Z.frame_codes(frame_bytes)
    f = bytes(frame_bytes)
    fhd = f[0]
    p = 1 + (0 if fhd & 0x20 else 1) + (0, 1, 2, 4)[fhd & 3] + ((1 if fhd & 0x20 else 0), 2, 4, 8)[fhd >> 6]
    out, prev = [], None
    for b in blocks:
        b.start = p + 3                                          # (where the block's content starts in the frame)
        c = f[p + 3:p + 3 + b.size]
        lit = None
        if b.btype == "compressed" and b.lit_type in ("huffman", "treeless"):
            lit = read_literals(c, prev)
            prev = lit.weights
        out.append((b, lit))
        p += 3 + (1 if b.btype == "rle" else b.size)
    return out


def regenerate(frame_bytes: bytes) -> bytes:
    """A magicless frame regenerated with every literals section read by this module (raw, RLE, or decoded by
    `read_literals`) and the sequences read by _zseq.frame_codes: equal to libzstd's output only if each Huffman section was
    read right."""
    f = bytes(frame_bytes)
    flat, lits = [], bytearray()
    for b, lit in frame_literals(f):
        if b.btype != "compressed":
            flat.append((b.size, 0, 0))
            lits += f[b.start:b.start + b.size] if b.btype == "raw" else f[b.start:b.start + 1] * b.size
            continue
        if lit is not None:
            data = lit.data
        else:
            c = f[b.start:]
            hsz = (1, 2, 1, 3)[(c[0] >> 2) & 3]
            data = c[hsz:hsz + b.lit_regen] if b.lit_type == "raw" else c[hsz:hsz + 1] * b.lit_regen
        start = len(lits)
        lits += data
        for *_, ll, ml, off in b.seqs:
            flat.append((ll, ml, off))
        flat.append((b.lit_regen - sum(s[4] for s in b.seqs), 0, 0))
        assert len(lits) - start == b.lit_regen
    return Z.replay(flat, bytes(lits))

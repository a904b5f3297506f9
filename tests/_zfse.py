"""zstd sequences sections (RFC 8878 3.1.1.3.2) built to order: FSE table descriptions, the tables they describe and the
interleaved tANS bitstream, written here rather than by libzstd.

libzstd's encoder normalises every distribution itself and writes only what its normaliser produces; here the test decides:
each kind's accuracy log from 5 to its maximum, -1 (low-probability) symbols anywhere and as many as fit, one symbol holding
every cell, long zero runs, descriptions that end early, RLE at each kind's largest symbol, repeat mode across blocks, every
Number_of_Sequences form (canonical or not), which cell each state ends on and where the end marker falls.  Corrupt sections
take description or bitstream bytes verbatim.

Every description written is read back by `_zseq._read_ncount`, every frame by `_zseq.frame_codes` (the same codes and
values, the bitstream consumed to bit 0), so a case cannot quietly hold something easier than it asks for."""
import numpy as np

import _zhuf as H
import _zseq as Z

KINDS = ("ll", "of", "ml")
MAX_SYM = Z._MAX_SYM                                   # ll 35, of 31, ml 52
MAX_AL = Z._MAX_AL                                     # ll 9, of 8, ml 9
ASCII = np.frombuffer(bytes(range(48, 112)), np.uint8)


def ll_code(v):
    return max(c for c in range(36) if Z.LL_BASE[c] <= v)


def ml_code(v):
    return max(c for c in range(53) if Z.ML_BASE[c] <= v)


def of_code(ov):
    return ov.bit_length() - 1


def codes(seq):
    """(ll code, of code, ml code) of a (literal length, match length, offset value) triple."""
    ll, ml, ov = seq
    return ll_code(ll), of_code(ov), ml_code(ml)


# ---- distributions and their descriptions ---------------------------------------------------------------------------
def distribution(al, weights, low=(), zeros=(), length=None):
    """A normalised distribution summing to 2^al: symbols in `low` get -1, those in `zeros` 0, the others of `weights`
    ({symbol: weight}) counts proportional to their weights, at least 1 each.  `length`: the description covers symbols
    0..length-1 (its last symbol must be nonzero)."""
    low, zeros = set(low), set(zeros)
    pos = [s for s in weights if s not in low and s not in zeros]
    n = length if length is not None else max(list(weights) + list(low)) + 1
    norm = [0] * n
    for s in low:
        norm[s] = -1
    free = (1 << al) - len(low)
    assert len(pos) <= free, "too many symbols for this accuracy log"
    if pos:
        tot = sum(weights[s] for s in pos)
        for s in pos:
            norm[s] = max(1, weights[s] * free // tot)
        while sum(norm[s] for s in pos) > free:
            norm[max(pos, key=lambda s: norm[s])] -= 1
        norm[max(pos, key=lambda s: weights[s])] += free - sum(norm[s] for s in pos)
    assert sum(abs(c) for c in norm) == 1 << al and norm[-1] != 0, norm
    return norm


def ncount(al_field, norm, tail_flags=None, runs=None):
    """The FSE table description of `norm` (RFC 8878 4.1.1), field by field as a decoder reads it, with no check of the sum:
    the fields stop where the decoder would stop (nothing left to distribute).  After a zero, the 2-bit repeat flags code the
    zeros that follow; `tail_flags` replaces the flags after a final zero (runs that end at or past the last symbol).
    `runs` gives, for each zero field in order, how many of the zeros behind it its flags code (default: all of them; fewer
    leaves the next zero to a field of its own, a longer but legal form).  `al_field` is written as is (al_field - 5 in 4 bits)."""
    runs = list(runs) if runs is not None else None
    acc, nbit = al_field - 5, 4
    remaining, threshold, nb = (1 << al_field) + 1, 1 << al_field, al_field + 1
    i = 0
    while i < len(norm) and remaining > 1:
        c = norm[i]
        v, mx = c + 1, 2 * threshold - 1 - remaining
        if v < mx:
            acc |= v << nbit; nbit += nb - 1
        else:
            acc |= (v + mx if v >= threshold else v) << nbit; nbit += nb
        remaining -= abs(c)
        i += 1
        while remaining < threshold and threshold > 1:
            nb -= 1
            threshold >>= 1
        if c == 0:
            z = 0
            while i + z < len(norm) and norm[i + z] == 0:
                z += 1
            if runs is not None:
                z = min(z, runs.pop(0))
            if i + z == len(norm) and tail_flags is not None:
                flags = list(tail_flags)
            else:
                flags = [3] * (z // 3) + [z % 3]
            for f in flags:
                acc |= f << nbit; nbit += 2
            i += z
    return acc.to_bytes((nbit + 7) // 8, "little")


def description(al, norm, runs=None):
    """A legal description, checked: it reads back through _zseq._read_ncount to the same (al, norm)."""
    d = ncount(al, norm, runs=runs)
    assert sum(abs(c) for c in norm) == 1 << al
    ral, rnorm, used = Z._read_ncount(d + bytes(8), 0, 63)
    assert (ral, rnorm, used) == (al, list(norm), len(d)), (al, norm, ral, rnorm, used, len(d))
    return d


def _field_cost(rem):
    """(field width, values below `thr` take one bit less) when `rem` is left to distribute."""
    bits = (rem + 1).bit_length()
    return bits, (1 << bits) - 2 - rem


def longest_description(kind):
    """The longest legal FSE table description of a kind: (bytes, al, norm, runs), by an exact search over (next symbol, what is
    left) of the bits each choice costs -- a nonzero count (-1 included), or a zero and the run of zeros behind it."""
    ms, best = MAX_SYM[kind], None
    for al in range(5, MAX_AL[kind] + 1):
        size = 1 << al
        NEG = -10 ** 9
        F = np.full((ms + 3, size + 1), NEG, np.int64)      # F[s, rem]: most bits to finish from symbol s with rem left
        F[:, 0] = 0
        choice = {}
        for s in range(ms, -1, -1):
            for rem in range(1, size + 1):
                bits, thr = _field_cost(rem)
                # nonzero counts: pr = -1 (v = 0) and pr = 1..rem (v = 2..rem + 1); cost bits - 1 when v < thr
                v = np.arange(rem + 2)
                nrem = np.where(v == 0, rem - 1, rem - (v - 1))
                cost = np.where(v < thr, bits - 1, bits)
                tot = cost + F[s + 1, np.clip(nrem, 0, size)]
                tot[1] = NEG                                  # v = 1 is a zero, below
                k = int(np.argmax(tot))
                cand = (int(tot[k]), ("count", k - 1))
                # a zero (v = 1) and r more zeros behind it: 2 bits of flags per started group of three
                r = np.arange(ms - s)
                t = (bits - 1 if 1 < thr else bits) + 2 * (r // 3 + 1) + F[s + 1 + r, rem]
                if len(r) and int(t.max()) > cand[0]:
                    cand = (int(t.max()), ("zeros", int(np.argmax(t))))
                F[s, rem] = cand[0]
                choice[s, rem] = cand[1]
        if F[0, size] <= 0:
            continue
        norm, runs, s, rem = [], [], 0, size
        while rem:
            what, x = choice[s, rem]
            if what == "count":
                norm.append(x); rem -= abs(x); s += 1
            else:
                norm += [0] * (1 + x); runs.append(x); s += 1 + x
        d = description(al, norm, runs)
        assert 8 * len(d) - 8 < 4 + int(F[0, size]) <= 8 * len(d)
        if best is None or len(d) > len(best[0]):
            best = (d, al, norm, runs)
    return best


# ---- tables and the tANS encoder --------------------------------------------------------------------------------------
def table_of(spec, kind, prev=None):
    """(al, decoding table) of a table spec: ("predefined",), ("rle", symbol), ("fse", al, norm) or ("repeat",) (`prev`)."""
    if spec[0] == "predefined":
        al, norm = Z._PREDEF[kind]
        return al, Z._fse_table(al, norm)
    if spec[0] == "rle":
        return 0, [(spec[1], 0, 0)]
    if spec[0] == "fse":
        return spec[1], Z._fse_table(spec[1], spec[2])
    assert prev is not None, "repeat mode without an earlier table"
    return prev


def cells_of(table, sym):
    return [u for u, (s, _, _) in enumerate(table) if s == sym]


def encode(seqs, tables, last=None, pad="", drop=0):
    """The interleaved tANS bitstream of `seqs` ((ll, ml, ov) triples) under tables {kind: (al, table)}, in the decoder's
    order (RFC 8878 3.1.1.3.2.2, _zseq._read_block): initial states LL, OF, ML; per sequence the extra bits of OF, ML, LL;
    then, except after the last sequence, the state updates LL, ML, OF.  The encoder runs backwards from the last sequence,
    whose cell per kind is `last[kind]`: "wide" (most state bits, default), "narrow" (fewest) or a cell index.
    `pad` (bits) goes below everything (left over: corrupt); `drop` bits are cut off the bottom (missing: corrupt).
    Returns (bytes, end-marker bit, bits written)."""
    last = last or {}
    n = len(seqs)
    cs = [codes(s) for s in seqs]
    st = {}
    for ki, kind in enumerate(KINDS):
        al, t = tables[kind]
        enc = {}
        for u, (s, nb, base) in enumerate(t):
            for v in range(1 << nb):
                enc[s, base + v] = (u, v, nb)
        cand = cells_of(t, cs[-1][ki])
        assert cand, f"{kind} code {cs[-1][ki]} has no cell"
        how = last.get(kind, "wide")
        if how == "wide":
            u = max(cand, key=lambda c: (t[c][1], -c))
        elif how == "narrow":
            u = min(cand, key=lambda c: (t[c][1], c))
        else:
            u = how
            assert u in cand
        states = [u]
        ups = []                                            # ups[i]: (bits value, width) of the update after sequence i
        for i in range(n - 2, -1, -1):
            assert (cs[i][ki], states[0]) in enc, f"{kind} code {cs[i][ki]} has no cell"
            u2, v, nb = enc[cs[i][ki], states[0]]
            states.insert(0, u2)
            ups.insert(0, (v, nb))
        st[kind] = (al, states, ups)
    parts = ["1"]
    for kind in KINDS:                                      # initial states LL, OF, ML
        al, states, _ = st[kind]
        if al:
            parts.append(format(states[0], f"0{al}b"))
    for i, (ll, ml, ov) in enumerate(seqs):
        llc, ofc, mlc = cs[i]
        for val, w in ((ov - (1 << ofc), ofc), (ml - Z.ML_BASE[mlc], Z.ML_BITS[mlc]), (ll - Z.LL_BASE[llc], Z.LL_BITS[llc])):
            assert 0 <= val < 1 << w or (w == 0 and val == 0), (seqs[i], w, val)
            if w:
                parts.append(format(val, f"0{w}b"))
        if i + 1 < n:
            for kind in ("ll", "ml", "of"):
                v, nb = st[kind][2][i]
                if nb:
                    parts.append(format(v, f"0{nb}b"))
    bits = "".join(parts) + pad
    if drop:
        bits = bits[:-drop]
    return int(bits, 2).to_bytes((len(bits) + 7) // 8, "little"), (len(bits) - 1) % 8, len(bits)


def nseq_header(n, form=None):
    """Number_of_Sequences in 1, 2 or 3 bytes (the smallest that fits unless `form` is given: a 2-byte form of a count below
    128 is non-canonical; the 3-byte form holds 0x7F00 and up only)."""
    form = form or (1 if n < 128 else 2 if n < 0x7F00 else 3)
    if form == 1:
        assert n < 128
        return bytes([n])
    if form == 2:
        assert n < 0x7F00
        return bytes([128 + (n >> 8), n & 255])
    assert 0x7F00 <= n < 0x7F00 + 65536
    return bytes([255]) + (n - 0x7F00).to_bytes(2, "little")


def raw_literals(lits):
    n = len(lits)
    if n < 32:
        return bytes([n << 3]) + lits
    if n < 4096:
        return bytes([((n & 15) << 4) | 0b0100, n >> 4]) + lits
    return bytes([((n & 15) << 4) | 0b1100, (n >> 4) & 255, n >> 12]) + lits


# ---- frames -------------------------------------------------------------------------------------------------------------
class Section:
    """What the writer put in one sequences section (for the cases to assert on)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


class Writer:
    """A magicless single-segment frame of raw blocks and compressed blocks whose sequences sections are written here.
    Keeps the output (`payload`), the repeat offsets and each kind's last table, as a decoder does."""

    def __init__(self, rng):
        self.rng = rng
        self.blocks, self.out = [], bytearray()
        self.reps = [1, 4, 8]
        self.prev = {k: None for k in KINDS}
        self.sections = []

    def text(self, n):
        return bytes(self.rng.choice(ASCII, size=n))

    def raw(self, data):
        self.blocks.append((data, 0))
        self.out += data

    def resolve(self, ll, ov):
        """The offset an offset value gives after a literal length (RFC 8878 3.1.1.5), updating the repeat offsets."""
        r = self.reps
        if ov > 3:
            off = ov - 3
            self.reps = [off, r[0], r[1]]
            return off
        idx = ov - 1 + (ll == 0)
        if idx == 0:
            return r[0]
        if idx == 1:
            self.reps = [r[1], r[0], r[2]]
        elif idx == 2:
            self.reps = [r[2], r[0], r[1]]
        else:
            self.reps = [r[0] - 1, r[0], r[1]]
        return self.reps[0]

    def seq_block(self, seqs, ll=("predefined",), of=("predefined",), ml=("predefined",), tail=0, form=None, last=None,
                  pad="", drop=0, reserved=0, desc=None, bitstream=None, tamper=None, lits=None, bad_offsets=False):
        """A compressed block of raw literals and `seqs` ((literal length, match length, offset value) triples) under the
        three table specs, `tail` trailing literals.  Corrupt blocks: `reserved` (mode bits 0..1), `desc` (the description
        bytes, verbatim), `bitstream` (verbatim), `tamper` (a function of the encoded bitstream), `pad` / `drop` (see encode), `bad_offsets` (offsets past the output
        are replayed as zeros).  Returns the Section."""
        specs = {"ll": ll, "of": of, "ml": ml}
        tables, dsc = {}, b""
        for kind in KINDS:
            sp = specs[kind]
            tables[kind] = table_of(sp, kind, self.prev[kind])
            if sp[0] == "rle":
                assert 0 <= sp[1] <= 255
                dsc += bytes([sp[1]])
            elif sp[0] == "fse":
                dsc += description(sp[1], sp[2]) if sum(abs(c) for c in sp[2]) == 1 << sp[1] else ncount(sp[1], sp[2])
        modes = sum(("predefined", "rle", "fse", "repeat").index(specs[k][0]) << s for k, s in (("ll", 6), ("of", 4), ("ml", 2))) | reserved
        marker = nbits = None
        if bitstream is None:
            bitstream, marker, nbits = encode(seqs, tables, last, pad, drop)
            if tamper:
                bitstream = tamper(bitstream)
        nlit = sum(s[0] for s in seqs) + tail
        lits = self.text(nlit) if lits is None else lits
        body = nseq_header(len(seqs), form) + bytes([modes]) + (dsc if desc is None else desc) + bitstream
        content = raw_literals(lits) + body
        assert len(content) <= Z.BLOCK, len(content)
        lp, start = 0, len(self.out)
        for l, m, ov in seqs:
            self.out += lits[lp:lp + l]; lp += l
            off = self.resolve(l, ov)
            d = len(self.out)
            if bad_offsets and not 1 <= off <= d:
                self.out += bytes(m)
                continue
            assert 1 <= off <= d, (off, d)
            for k in range(m) if off < m else ():
                self.out.append(self.out[d - off + k])
            if off >= m:
                self.out += self.out[d - off:d - off + m]
        self.out += lits[lp:]
        assert len(self.out) - start <= Z.BLOCK, len(self.out) - start
        for kind in KINDS:
            self.prev[kind] = tables[kind]
        sec = Section(seqs=list(seqs), specs=specs, tables=tables, modes=modes, desc=dsc, bitstream=bitstream, marker=marker,
                      nbits=nbits, header=nseq_header(len(seqs), form), index=len(self.blocks))
        self.sections.append(sec)
        self.blocks.append((content, 2))
        return sec

    def frame(self, check=True):
        """(payload, frame).  With `check`, frame_codes reads every written block back: the same modes, accuracy logs, codes
        and values, each bitstream consumed to bit 0."""
        bl = [H.block(c, i == len(self.blocks) - 1, bt) for i, (c, bt) in enumerate(self.blocks)]
        f = H.frame(bl, len(self.out))
        payload = bytes(self.out)
        if check:
            self.check(f)
        return payload, f

    def check(self, f):
        _, blocks = Z.frame_codes(f)
        assert len(blocks) == len(self.blocks)
        for sec in self.sections:
            b = blocks[sec.index]
            assert b.btype == "compressed" and b.modes == sec.modes
            for kind in KINDS:
                sp = sec.specs[kind]
                assert getattr(b, kind + "_mode") == sp[0], (kind, sp[0])
                if sp[0] == "fse":
                    assert b.al[kind] == sp[1]
            got = [(s[4], s[5], s[3]) for s in b.seqs]
            assert got == sec.seqs, "frame_codes reads other sequences than were written"
            assert [(s[0], s[2], s[1]) for s in b.seqs] == [codes(s) for s in sec.seqs]
            assert b.seq_bytes == len(sec.bitstream)


def seqs_for(rng, want, pos, ll_small=False):
    """(ll, ml, ov) triples with the wanted (ll code, of code, ml code) each, random extra bits; offsets reach at most `pos`
    back (the output before the block) and never resolve to rep0 - 1 (ov 3 with ll 0)."""
    out = []
    for llc, ofc, mlc in want:
        ll = Z.LL_BASE[llc] + int(rng.integers(0, min(1 << Z.LL_BITS[llc], 4096)))      # (LL 35 and ML 52 both fit one
        ml = Z.ML_BASE[mlc] + int(rng.integers(0, min(1 << Z.ML_BITS[mlc], 4096)))      #  block with small other lengths)
        if ofc == 0:
            ov = 1
        elif ofc == 1:
            ov = 2 if ll == 0 else int(rng.integers(2, 4))
        else:
            hi = min((1 << (ofc + 1)) - 1, pos + 3)
            assert hi >= 1 << ofc, f"offset code {ofc} needs {1 << ofc} bytes of history"
            ov = int(rng.integers(1 << ofc, hi + 1))
        out.append((ll, ml, ov))
    return out


def pack(rng, want, pos, limit=Z.BLOCK - 64):
    """`want` (code triples) cut into blocks whose regenerated size stays under `limit`: a list of lists of (ll, ml, ov)."""
    blocks, cur, size = [], [], 0
    for s in seqs_for(rng, want, pos):
        n = s[0] + s[1]
        if cur and size + n > limit:
            blocks.append(cur); cur, size = [], 0
        cur.append(s); size += n
    if cur:
        blocks.append(cur)
    return blocks

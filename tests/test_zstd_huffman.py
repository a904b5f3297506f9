"""The Huffman literal decoders (k_build_tables<1>, k_huf_decode<128>, k_huf_decode_block, k_huf_decode_big) on literals
sections built to order (tests/_zhuf.py): trees of every depth, fixed-length trees, both weight forms at their count limits,
stream lengths around the kernels' range and size boundaries, treeless reuse, and the sections a decoder must refuse.
Each case reads its section back with the plain reader to prove that its edge is there, then checks that the reader,
libzstd and the device agree on every byte, under both big-stream kernels (NAFGPU_HUF_BLOCK_MIN=1: one CTA per block;
1000000: four clustered CTAs).  Streams of at most 2048 symbols go to k_huf_decode<128> whatever the setting."""
import numpy as np
import pytest

import _cases as K
import _oracle as O
import _zhuf as H
import _zseq as Z
import nafcodec_b200 as N
from _harness import BACKENDS, assert_same_as_oracle, library
from conftest import read_golden

SMALL_MAX = 2048                           # symbols per stream up to which a 4-stream block is decoded by k_huf_decode<128>
RANGE_MIN_BITS = 256 * 2 * H.MAX_BITS      # big-stream kernels: 256 ranges of at least 2 * 11 bits
ASCII0 = 48                                # trees over printable symbols 48.. (up to 64 of them) make valid TEXT payloads


def _ctx(backend):
    return N.shared_context(0, library(backend))


def _agree(backend, frame, payload, label=""):
    """The reader (through a full regeneration), libzstd and the device give `payload`."""
    assert H.regenerate(frame) == payload, label
    assert Z.libzstd_decompress(frame, len(payload)) == payload, label
    got = _ctx(backend).zstd_decompress(frame, len(payload))
    if got != payload:
        x, y = np.frombuffer(got, np.uint8), np.frombuffer(payload, np.uint8)
        k = int(np.nonzero(x != y)[0][0])
        pytest.fail(f"{label}: device differs from byte {k} on ({int((x != y).sum())} bytes differ)")


def _lits(backend, sections, label, fcs_bytes=None):
    """A frame of literals-only blocks, one per (data, section); checked by _agree.  Returns what the reader found."""
    payload = b"".join(d for d, _ in sections)
    frame = H.literals_only([(s, len(d)) for d, s in sections], fcs_bytes)
    _agree(backend, frame, payload, label)
    return [lit for _, lit in H.frame_literals(frame)]


def _balanced(m, symbols=None):
    """Weights of a complete code over m symbols with lengths d - 1 and d (d = ceil(log2 m)): fixed-length when m is a power
    of two.  `symbols`: which symbol values get the codes (default 0..m-1)."""
    d = max(1, (m - 1).bit_length())
    a = (1 << d) - m                                             # symbols one bit shorter
    symbols = list(range(m)) if symbols is None else symbols
    return H.weights_of_lengths({s: d - 1 if i < a else d for i, s in enumerate(symbols)})


def _skewed(depth, base=0):
    """Weights of a depth-`depth` code over depth + 1 symbols: lengths 1, 2, ..., depth - 1, depth, depth."""
    if depth == 1:
        return H.weights_of_lengths({base: 1, base + 1: 1})
    lens = {base + i: i + 1 for i in range(depth)}
    lens[base + depth] = depth
    return H.weights_of_lengths(lens)


def _stair(depth, m, base=ASCII0):
    """Weights of a depth-`depth` code over m symbols: lengths 1, 2, ..., k for the first k, the other m - k sharing the last
    2^-k of the code space as a two-length subtree."""
    for k in range(m - 1):
        r = m - k
        b = max(1, (r - 1).bit_length())
        if k + b == depth:
            a = (1 << b) - r
            lens = {base + i: i + 1 for i in range(k)}
            lens.update({base + k + i: k + (b - 1 if i < a else b) for i in range(r)})
            return H.weights_of_lengths(lens)
    raise ValueError(f"no staircase of depth {depth} over {m} symbols")


def _symbols(weights):
    return [s for s, w in enumerate(weights) if w]


def _data(rng, weights, n, deep_share=None):
    """n symbols of the tree, uniform over its symbols (deep codes dominate), or with `deep_share` of them the longest code."""
    syms = np.array(_symbols(weights), np.uint8)
    out = rng.choice(syms, size=n)
    if deep_share is not None:
        deep = np.array([s for s in _symbols(weights) if weights[s] == min(weights[x] for x in _symbols(weights))], np.uint8)
        m = rng.random(n) < deep_share
        out[m] = rng.choice(deep, size=int(m.sum()))
    return bytes(out)


HUF_KERNELS = pytest.mark.parametrize("huf_block_min", ["1", "1000000"], ids=["block", "cluster"])


@pytest.fixture
def huf_env(monkeypatch, huf_block_min):
    monkeypatch.setenv("NAFGPU_HUF_BLOCK_MIN", huf_block_min)
    return huf_block_min


# ---- the writer and the reader against libzstd ----------------------------------------------------------------------
def test_reader_reads_libzstd_frames():
    """The reader regenerates every frame of the fixtures and of libzstd's own encoder (Huffman and treeless sections of one
    and four streams) exactly as libzstd does."""
    seen = set()
    for name in ["masked.naf", "LuxC.naf", "phix.naf", "CP040672.naf", "NZ_AAEN01000029.naf"]:
        data = read_golden(name)
        L = O.parse(data)
        for i in range(6):
            s = L.sec[i]
            if s.present:
                frame = data[s.offset:s.offset + s.compressed_size]
                assert H.regenerate(frame) == O.zstd_decompress(frame), (name, O.SEC_NAMES[i])
                seen |= {(lit.lit_type, len(lit.counts), lit.form) for _, lit in H.frame_literals(frame) if lit}
    rng = np.random.default_rng(4)
    p = b"".join(b"read/%d %s\n" % (i, K.random_dna(rng, 60, b"ACGTN")) for i in range(5000))
    for level in (1, 19):
        frame = K.zstd_frame(p, level)
        assert H.regenerate(frame) == p
        seen |= {(lit.lit_type, len(lit.counts), lit.form) for _, lit in H.frame_literals(frame) if lit}
    assert {("huffman", 4, "fse"), ("treeless", 4, None)} <= seen, seen


def test_writer_sections_decode_under_libzstd():
    """Every form the writer makes (both weight forms at their count limits, -1 probabilities, zero runs, slack bits below
    the last FSE state read, each literals header size format, each content-size field) decodes under libzstd to what the
    reader reads."""
    rng = np.random.default_rng(1)
    cases = []
    for n in (1, 2, 127, 128):
        cases.append((_balanced(n + 1), dict(form="direct")))
    for n in (2, 3, 254, 255):
        for al in (5, 6):
            cases.append((_balanced(n + 1), dict(form="fse", al=al, low=(0,))))
    gaps = H.weights_of_lengths({**{s: 6 for s in range(100, 132)}, 255: 1})
    cases.append((gaps, dict(form="fse", al=6)))
    cases.append((_skewed(9), dict(form="fse", al=5, slack="1")))
    for w, kw in cases:
        data = _data(rng, w, 3000)
        for streams in (1, 4):
            for sf in ((0,) if streams == 1 else (1, 2, 3)):
                d = data[:900] if sf <= 1 else data
                sec = H.literals_section(d, w, streams=streams, sf=sf, **kw)
                frame = H.literals_only([(sec, len(d))], fcs_bytes=4)
                assert Z.libzstd_decompress(frame, len(d)) == d == H.read_literals(sec).data, (kw, streams, sf)
    for fcs in (1, 2, 4):
        d = bytes(_data(rng, _skewed(3), 200 if fcs == 1 else 3000))
        frame = H.literals_only([(H.literals_section(d, _skewed(3)), len(d))], fcs_bytes=fcs)
        assert frame[0] >> 6 == {1: 0, 2: 1, 4: 2}[fcs] and Z.libzstd_decompress(frame, len(d)) == d


# ---- depths and fixed-length trees ----------------------------------------------------------------------------------
def _depth_sections(rng, w, **kw):
    """One tree in three sections: a 1-stream section (k_huf_decode<128>), a 4-stream section of short streams (also
    k_huf_decode<128>) and one of 6000 symbols per stream (a big-stream kernel)."""
    out = []
    for n, streams in ((700, 1), (4000, 4), (24_000, 4)):
        d = _data(rng, w, n)
        out.append((d, H.literals_section(d, w, streams=streams, **kw)))
    return out


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_fixed_length_trees(backend, huf_env):
    """2^k symbols of k bits, k = 1..8 (256 symbols need the FSE weight form: direct weights stop at 128)."""
    rng = np.random.default_rng(10)
    for k in range(1, 9):
        w = _balanced(1 << k)
        kw = dict(form="fse", low=(0,)) if k == 8 else {}
        lits = _lits(backend, _depth_sections(rng, w, **kw), f"fixed {k} bits")
        assert all(l.depth == k and set(l.weights) == {1} and len(l.weights) == 1 << k for l in lits)
        assert lits[-1].counts[0] > SMALL_MAX >= lits[1].counts[0]


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_every_depth(backend, huf_env):
    """Skewed trees (lengths 1, 2, ..., d, d) and two-length trees of every depth from 1 to 11, direct and FSE weights."""
    rng = np.random.default_rng(11)
    for d in range(1, 12):
        shapes = [(f"skewed {d}", _skewed(d))]
        if 3 <= d <= 8:
            shapes.append((f"two lengths {d}", _balanced((1 << (d - 1)) + 3)))
        if d >= 7:
            shapes.append((f"staircase {d}", _stair(d, 40)))
        for label, w in shapes:
            form = "fse" if (d % 2 and len(w) > 2) or len(w) > 129 else "direct"
            lits = _lits(backend, _depth_sections(rng, w, form=form), label)
            assert all(l.depth == d and l.form == form for l in lits), label


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_largest_stream(backend, huf_env):
    """The largest stream a block can hold: 32 Ki symbols, nearly all of them 11-bit codes (about 45 KB, the shared-memory
    worst case of the big-stream kernels), in a 128 KiB block whose other three streams are 1-bit codes."""
    rng = np.random.default_rng(12)
    lens = {ASCII0 + i: i + 1 for i in range(7)}
    lens.update({ASCII0 + 7 + i: 11 for i in range(16)})           # 1/2 + ... + 1/128 + 16/2048
    w = H.weights_of_lengths(lens)
    seg = 32 * 1024
    first = _data(rng, w, seg, deep_share=0.97)
    rest = bytes([ASCII0]) * (3 * seg)
    d = first + rest
    sec = H.literals_section(d, w, sf=3)
    (lit,) = _lits(backend, [(d, sec)], "largest stream")
    assert lit.regen == Z.BLOCK and lit.depth == 11 and lit.counts == [seg] * 4
    assert lit.stream_sizes[0] > 44_000, lit.stream_sizes


# ---- weight descriptions ----------------------------------------------------------------------------------------------
def _weight_cases():
    """(label, weights, description keywords, what the reader must find)"""
    out = []
    for n in (1, 2, 127, 128):
        out.append((f"direct {n}", _balanced(n + 1), dict(form="direct"), dict(form="direct", n_explicit=n)))
    for n in (2, 3, 254, 255):
        for al in (5, 6):
            out.append((f"fse {n} al {al}", _balanced(n + 1), dict(form="fse", al=al, low=(0,)),
                        dict(form="fse", n_explicit=n, al=al, end_state=1 if n % 2 == 0 else 2)))
    # zero-weight gaps, symbol 255 carrying the implied weight; weights {0, 1, 6}: a zero run in the FSE description
    gaps = H.weights_of_lengths({**{s: 6 for s in range(100, 132)}, 255: 1})
    out.append(("gaps, implied 255", gaps, dict(form="fse", al=6), dict(form="fse", n_explicit=255)))
    out.append(("gaps, direct", H.weights_of_lengths({3: 2, 9: 2, 40: 3, 41: 3, 77: 2}), dict(form="direct"), dict(form="direct", n_explicit=77)))
    # explicit weights that already sum to a power of two: the implied weight doubles the total
    out.append(("implied completes a power of two", [1, 1, 2], dict(form="direct"), dict(form="direct", n_explicit=2, depth=2)))
    return out


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_weight_descriptions(backend, huf_env):
    rng = np.random.default_rng(13)
    for label, w, kw, want in _weight_cases():
        lits = _lits(backend, _depth_sections(rng, w, **kw), label)
        for l in lits:
            assert l.weights == w, label
            for k, v in want.items():
                assert getattr(l, k) == v, (label, k, getattr(l, k))
    # FSE weight streams whose last read is partly inside the stream (slack bits below the last state read)
    w = _skewed(9)
    for slack in ("", "1", "01"):
        lits = _lits(backend, _depth_sections(rng, w, form="fse", al=6, slack=slack), f"slack {slack!r}")
        assert lits[0].form == "fse"


# ---- stream geometry ------------------------------------------------------------------------------------------------
GEO_TREE = H.weights_of_lengths({ASCII0: 1, ASCII0 + 1: 2, ASCII0 + 2: 3, ASCII0 + 3: 3})


def _bits_stream(seg, target_bits):
    """seg symbols of GEO_TREE whose codes take exactly target_bits."""
    three, two = divmod(target_bits - seg, 2)
    assert three + two <= seg
    return bytes([ASCII0 + 2]) * three + bytes([ASCII0 + 1]) * two + bytes([ASCII0]) * (seg - three - two)


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_stream_geometry(backend, huf_env):
    rng = np.random.default_rng(14)
    w = GEO_TREE
    # symbols per stream at the small/big classification: 2047, 2048 (k_huf_decode<128>), 2049 (big); regen 8193 is big too
    for regen in (4 * 2047, 4 * 2048, 4 * 2048 + 1, 4 * 2049):
        d = _data(rng, w, regen)
        (lit,) = _lits(backend, [(d, H.literals_section(d, w))], f"regen {regen}")
        assert lit.counts[0] == (regen + 3) // 4
    # stream bit lengths around 256 ranges of 22 bits (the range minimum of the big-stream kernels), and a stream just past
    # the 108-bit checkpoint of every range; each of the four streams one bit apart
    for bits in (RANGE_MIN_BITS - 2, RANGE_MIN_BITS, RANGE_MIN_BITS + 2, 256 * 108 + 1):
        seg = 2049 if bits < 4098 * 2 else bits * 2 // 3
        streams = [_bits_stream(seg, bits - 1 + k) for k in range(4)]
        d = b"".join(streams)
        (lit,) = _lits(backend, [(d, H.literals_section(d, GEO_TREE))], f"stream of {bits} bits")
        assert [8 * n - 8 + m for n, m in zip(lit.stream_sizes, lit.marker_bits)] == [bits - 1 + k for k in range(4)]
    # ranges shorter than the 12- and 108-bit checkpoints: streams of a few bits to a few hundred (short ranges of the big
    # kernels need more than 2048 symbols: 1-bit codes, 2049 of them, leave 8 bits per range)
    for n in (1, 2, 5, 11, 12, 13, 107, 108, 109, 700):
        d = bytes([ASCII0]) * n
        _lits(backend, [(d, H.literals_section(d, w, streams=1))], f"1-stream of {n} bits")
    # the end marker at every bit of the last byte, in 1-stream and big 4-stream sections
    for j in range(8):
        d1 = bytes([ASCII0]) * (800 + j)
        seg = 2056 + j
        d4 = bytes([ASCII0]) * (4 * seg)
        lits = _lits(backend, [(d1, H.literals_section(d1, w, streams=1)), (d4, H.literals_section(d4, w))], f"marker bit {j}")
        assert lits[0].marker_bits == [j] and lits[1].marker_bits == [j] * 4
    # four-stream blocks whose fourth stream is 0..3 symbols short, small and big
    for seg in (100, 2100):
        for short in range(4):
            d = _data(rng, w, 4 * seg - short)
            (lit,) = _lits(backend, [(d, H.literals_section(d, w))], f"fourth stream {short} short")
            assert lit.counts == [seg, seg, seg, seg - short]


@pytest.mark.parametrize("backend", BACKENDS)
def test_four_stream_minimum(backend):
    """regen 1..12 in 4-stream mode: libzstd refuses fewer than 6 literals (MIN_LITERALS_FOR_4_STREAMS) and decodes 6 and 9,
    whose fourth stream regenerates no symbol (one byte: the end marker alone)."""
    rng = np.random.default_rng(15)
    for regen in range(1, 13):
        d = _data(rng, GEO_TREE, regen)
        sec = H.literals_section(d, GEO_TREE, sf=1)
        frame = H.literals_only([(sec, regen)])
        if regen < 6:
            with pytest.raises(RuntimeError, match="Literals"):
                Z.libzstd_decompress(frame, regen)
            with pytest.raises(ValueError):
                H.read_literals(sec)
            with pytest.raises(N.NafIoError, match="4-stream"):
                _ctx(backend).zstd_decompress(frame, regen)
        else:
            _agree(backend, frame, d, f"regen {regen}")
            lit = H.read_literals(sec)
            assert lit.counts[3] == regen - 3 * ((regen + 3) // 4)
            if regen in (6, 9):
                assert lit.counts[3] == 0 and lit.stream_sizes[3] == 1 and lit.marker_bits[3] == 0


# ---- tree reuse -----------------------------------------------------------------------------------------------------
def _raw_section(d):
    return bytes([((len(d) & 15) << 4) | 0b0100, len(d) >> 4]) + d if len(d) >= 32 else bytes([len(d) << 3]) + d


def _rle_section(byte, n):
    return bytes([((n & 15) << 4) | 0b0101, n >> 4]) + bytes([byte])


def _reuse_frame(rng):
    """Literals-only blocks: for every depth 1..11 a tree, then treeless runs (one and four streams, small and big), with raw
    and RLE literals sections and raw and RLE blocks between them.  All symbols printable."""
    parts, payload = [], b""

    def add(content, d, btype=2):
        nonlocal payload
        parts.append((content, btype))
        payload += d

    for depth in range(1, 12):
        w = _skewed(depth, ASCII0)
        d = _data(rng, w, 600)
        add(H.literals_section(d, w, streams=1, form="fse" if depth > 2 else "direct") + b"\0", d)
        for n, streams in ((300, 1), (3000, 4), (9000, 4)):
            d = _data(rng, w, n)
            add(H.literals_section(d, w, streams=streams, treeless=True) + b"\0", d)
        raw = bytes(rng.choice(np.arange(ASCII0, ASCII0 + 60, dtype=np.uint8), size=40))
        add(_raw_section(raw) + b"\0", raw)
        add(_rle_section(ASCII0 + 5, 50) + b"\0", bytes([ASCII0 + 5]) * 50)
        add(raw[:17], raw[:17], btype=0)
        add(bytes([ASCII0 + 2]), bytes([ASCII0 + 2]) * 33, btype=1)
        d = _data(rng, w, 5000)
        add(H.literals_section(d, w, treeless=True) + b"\0", d)
    blocks = []
    for i, (c, bt) in enumerate(parts):
        last = i == len(parts) - 1
        if bt == 1:
            blocks.append(((1 << 1) | int(last) | (33 << 3)).to_bytes(3, "little") + c)
        else:
            blocks.append(H.block(c, last, bt))
    return payload, H.frame(blocks, len(payload))


def _as_text_archive(payload, frame):
    """A TEXT archive of one record whose sequence section is `frame` (regenerating `payload`)."""
    arc = O.encode(sequence_type=O.TEXT, ids=[b"crafted"], sequences=[b"A" * len(payload)], level=1)
    s = O.parse(arc).sec[4]
    k = len(O.write_variable_length(s.compressed_size))
    return arc[:s.offset - k] + O.write_variable_length(len(frame)) + frame + arc[s.offset + s.compressed_size:]


def _batch(backend, crafted, strict=True):
    """Crafted archives in one decode_batch between ordinary ones; with strict=False, the results."""
    arcs = [read_golden("phix.naf")] + [a for c in crafted for a in (c, K.multi_record_dna(5, 12, 900, level=19))]
    lib = library(backend)
    res = _ctx(backend).decode([N.parse_archive(a, lib) for a in arcs], strict=strict)
    return arcs, res


def _batch_parity(backend, crafted):
    arcs, res = _batch(backend, crafted)
    for i, (r, a) in enumerate(zip(res, arcs)):
        assert_same_as_oracle(r, O.decode(a), f"archive {i}")


def _spliced(rng):
    """Frames of matches and literals (Z.build with raw literals) whose literals sections are replaced by Huffman sections of
    trees of changing depth and by treeless sections: custom-tree literals placed between matches."""
    text = np.arange(ASCII0, ASCII0 + 12, dtype=np.uint8)
    blocks = [[bytes(rng.choice(text, size=3000))]]
    for b in range(24):
        n = int(rng.integers(1, 40))
        body = [(bytes(rng.choice(text, size=int(rng.integers(0, 900)))), int(rng.integers(3, 200)), int(rng.integers(1, 2900)))
                for _ in range(n)]
        blocks.append(body + [bytes(rng.choice(text, size=int(rng.integers(0, 30))))])
    payload, raw = Z.build(blocks, literal_mode=Z.LIT_RAW)
    trees = {}

    def section(k, lits):
        depth = 4 + (k // 3) % 8                                  # a new tree every third block, depth 4..11
        if len(lits) < 6:
            return _raw_section(lits)
        if k % 3 == 0 or depth not in trees:
            trees[depth] = _stair(depth, 12)
            return H.literals_section(lits, trees[depth], streams=1 if len(lits) < 1000 else 4, form="fse" if k % 2 else "direct")
        return H.literals_section(lits, trees[depth], streams=1 if len(lits) < 1000 else 4, treeless=True)
    return payload, H.splice(raw, section)


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_tree_reuse(backend, huf_env, monkeypatch):
    rng = np.random.default_rng(16)
    payload, frame = _reuse_frame(rng)
    _agree(backend, frame, payload, "treeless runs")
    found = H.frame_literals(frame)
    kinds = [(b.btype, lit.lit_type if lit else b.lit_type) for b, lit in found]
    assert ("compressed", "treeless") in kinds and ("raw", None) in kinds and ("rle", None) in kinds
    assert {lit.depth for _, lit in found if lit and lit.lit_type == "treeless"} == set(range(1, 12))
    sp_payload, sp_frame = _spliced(rng)
    _agree(backend, sp_frame, sp_payload, "spliced")
    sp = [(b, lit) for b, lit in H.frame_literals(sp_frame) if lit]
    assert {lit.lit_type for _, lit in sp} == {"huffman", "treeless"} and all(b.seqs for b, _ in sp)
    # the same frames in archives, every block a walk part of its own: each tree crosses a cut
    monkeypatch.setenv("NAFGPU_WALK_SPLIT", "1")
    _batch_parity(backend, [_as_text_archive(payload, frame), _as_text_archive(sp_payload, sp_frame)])


@pytest.mark.parametrize("backend", BACKENDS)
@HUF_KERNELS
def test_mixed_job(backend, huf_env):
    """One batch with archives of short streams, big streams and fixed-length trees: every Huffman kernel in one job."""
    rng = np.random.default_rng(17)
    crafted = []
    for w, n, streams in ((_skewed(11, ASCII0), 700, 1), (_balanced(64, list(range(ASCII0, ASCII0 + 64))), 30_000, 4),
                          (_skewed(7, ASCII0), 5000, 4), (_balanced(37, list(range(ASCII0, ASCII0 + 37))), 40_000, 4)):
        d = _data(rng, w, n)
        frame = H.literals_only([(H.literals_section(d, w, streams=streams), n)])
        _agree(backend, frame, d, f"{n} symbols")
        crafted.append(_as_text_archive(d, frame))
    _batch_parity(backend, crafted)


# ---- refusals -------------------------------------------------------------------------------------------------------
def _refusals(rng):
    """(label, frame, regenerated size the header claims, whether libzstd 1.5.5 refuses it too).  libzstd's four-stream
    decoder does not check that a stream ends on its first bit (its fast loop stops at the output end), and its FSE weight
    decoder reads the two start states below the stream start without complaint; the device and the reader refuse both, as
    its one-stream decoder does."""
    w = _skewed(5, ASCII0)
    d = _data(rng, w, 3000)
    code = H.canonical_code(w)
    out = []

    def add(label, sec, n=len(d), libzstd=True):
        out.append((label, H.literals_only([(sec, n)]), n, libzstd))

    add("remainder not a power of two", H.literals_section(d, w, desc=H.direct_weights([3, 0, 0, 1])))      # 4 + 1: 3 short of 8
    for streams, n in ((1, 1000), (4, 3000)):
        seg = (n + 3) // 4 if streams == 4 else n
        good = [H.huffman_stream(d[k * seg:(k + 1) * seg], code) for k in range(streams)]
        last = d[(streams - 1) * seg:n]
        bad = {"last byte 0": good[-1] + b"\0", "one symbol short": H.huffman_stream(last[:-1], code),
               "one symbol long": H.huffman_stream(last + last[:1], code), "a stray bit": H.huffman_stream(last, code, "0")}
        for what, s_ in bad.items():
            add(f"{streams}-stream, {what}", H.literals_section(d[:n], w, streams=streams, stream_bytes=good[:-1] + [s_]), n, streams == 1)
    sec = bytearray(H.literals_section(d, w))
    at = (3, 3, 4, 5)[(sec[0] >> 2) & 3] + len(H.tree_description(w))
    sec[at:at + 2] = (60000).to_bytes(2, "little")
    add("jump table past the section", bytes(sec))
    add("more than 255 FSE weights", H.literals_section(d, w, desc=H.fse_weights(_balanced(257)[:256], al=6, low=(0,))))
    nc = H.write_ncount(6, H.normalize([1, 2], 6))
    add("FSE weight stream shorter than its two states", H.literals_section(d, w, desc=bytes([len(nc) + 1]) + nc + b"\x01"), libzstd=False)
    add("treeless first block", H.literals_section(d, w, treeless=True))
    for n in (4, 5):
        add(f"4-stream regen {n}", H.literals_section(d[:n], w, sf=1), n)
    add("no two weight-1 symbols", H.literals_section(bytes([ASCII0, ASCII0 + 1]) * 300, [0] * ASCII0 + [2, 2], streams=1), 600)
    return out


@pytest.mark.parametrize("backend", BACKENDS)
def test_refusals(backend):
    """Corrupt sections: the device refuses each with a clean NafIoError, as the reader does (and libzstd, except where its
    checks are laxer, see _refusals), and inside a batch the other archives still decode."""
    rng = np.random.default_rng(18)
    cases = _refusals(rng)
    for label, frame, n, libzstd_refuses in cases:
        if libzstd_refuses:
            with pytest.raises(RuntimeError):
                Z.libzstd_decompress(frame, n)
        with pytest.raises((ValueError, AssertionError)):
            H.regenerate(frame)
        with pytest.raises(N.NafIoError):
            _ctx(backend).zstd_decompress(frame, n)
    arcs, res = _batch(backend, [_as_text_archive(b"0" * n, f) for _, f, n, _ in cases], strict=False)
    for i, (r, a) in enumerate(zip(res, arcs)):
        if i % 2:
            assert r.status != 0, cases[i // 2][0]
        else:
            assert r.status == 0
            assert_same_as_oracle(r, O.decode(a), f"archive {i}")


@pytest.mark.parametrize("backend", BACKENDS)
def test_twelve_bit_tree_is_refused(backend):
    """A 12-bit tree: libzstd 1.5.5 decodes it, RFC 8878 caps Max_Number_of_Bits at 11, and the device refuses it (status
    E_HUF_TREE) by design."""
    lens = {ASCII0 + i: i + 1 for i in range(12)}
    lens[ASCII0 + 12] = 12
    w = H.weights_of_lengths(lens)
    d = bytes(np.random.default_rng(19).choice(np.array(_symbols(w), np.uint8), size=3000))
    frame = H.literals_only([(H.literals_section(d, w), len(d))])
    assert Z.libzstd_decompress(frame, len(d)) == d
    with pytest.raises(ValueError, match="11"):
        H.regenerate(frame)
    with pytest.raises(N.NafIoError, match=r"device status 0x2\)"):
        _ctx(backend).zstd_decompress(frame, len(d))

"""k_huf_scout, the pass that finds where every range of k_huf_decode_block starts (NAFGPU_HUF_BLOCK_MIN=1), on streams built
to order (tests/_zhuf.py).  The scout cuts each stream into 64 coarse ranges of four of the write kernel's 256 fine ranges of
S = max(ceil(P0 / 256), 22) bits; these cases sit on the edges that split creates: a short last coarse range, one with a
single fine range, coarse ranges with none, S at its minimum, a stream that ends on a coarse boundary, tracks that never
merge (a non-constant map at every fine boundary), and single flipped bits, which must be refused with E_HUF_STREAM while
the other archives of the job decode."""
import numpy as np
import pytest

import _oracle as O
import _zhuf as H
import nafcodec_b200 as N
from _harness import BACKENDS, assert_same_as_oracle, library
from test_zstd_huffman import ASCII0, GEO_TREE, _agree, _as_text_archive, _batch, _bits_stream, _data, _skewed

FINE = 256                                 # ranges of k_huf_decode_block per stream
COARSE = 64                                # coarse ranges of k_huf_scout per stream
PER = FINE // COARSE                       # fine ranges per coarse range
S_MIN = 2 * H.MAX_BITS


@pytest.fixture(autouse=True)
def block_path(monkeypatch):
    monkeypatch.setenv("NAFGPU_HUF_BLOCK_MIN", "1")


def geometry(p0):
    """(S, fine ranges that hold stream bits, fine ranges in the last coarse range that holds any)"""
    s = max(-(-p0 // FINE), S_MIN)
    nf = -(-p0 // s)
    return s, nf, nf - PER * ((nf - 1) // PER)


def _payload_bits(stream):
    """The stream's payload bits from the top (below the end marker), as a string of 0/1."""
    return bin(int.from_bytes(stream, "little"))[3:]


def _sections(backend, seg, bits, label):
    """One 4-stream block of GEO_TREE whose streams carry exactly bits[k] payload bits each, the codes in random order (so
    that range tops fall inside codewords)."""
    rng = np.random.default_rng(sum(bits))
    d = b"".join(bytes(rng.permutation(np.frombuffer(_bits_stream(seg, b), np.uint8))) for b in bits)
    sec = H.literals_section(d, GEO_TREE)
    lit = H.read_literals(sec)
    assert [8 * n - 8 + m for n, m in zip(lit.stream_sizes, lit.marker_bits)] == list(bits), label
    _agree(backend, H.literals_only([(sec, len(d))]), d, label)


@pytest.mark.parametrize("backend", BACKENDS)
def test_last_coarse_range(backend):
    """Streams whose last coarse range is short (a partial fine range), holds a single fine range, holds none (the stream
    ends one coarse range early), or ends exactly on a coarse boundary (coarse and fine boundary coincide with the end)."""
    cases = {7675: "short", 7570: "one fine range", 7440: "no fine range", 7560: "ends on a coarse boundary"}
    s, nf, last = geometry(7675)
    assert (s, nf, last) == (30, 256, 4) and 7675 % s != 0
    assert geometry(7570)[1:] == (253, 1)
    assert geometry(7440)[1] == 248 and 248 // PER < COARSE
    assert geometry(7560)[0] * FINE // COARSE * (COARSE - 1) == 7560
    _sections(backend, 2600, list(cases), "last coarse range")


@pytest.mark.parametrize("backend", BACKENDS)
def test_minimum_range(backend):
    """Just above the small-stream limit (2049 symbols per stream): S clamped at 22 bits, only 94 fine ranges, 24 coarse ranges
    with bits; a stream of 1-bit codes only (every bit a codeword boundary: every range starts on its top); S = 22 exactly
    with all 256 fine ranges; and 3000 bits."""
    bits = [2050, 2049, 256 * S_MIN, 3000]
    assert [geometry(b)[0] for b in bits] == [S_MIN, S_MIN, S_MIN, S_MIN]
    assert geometry(2050)[1:] == (94, 2) and geometry(256 * S_MIN)[1:] == (256, 4)
    _sections(backend, 2049, bits, "minimum range")


def _boundaries(bits, code, start, lim):
    """Walks the code from `start` (bits below the top) to the first codeword boundary at or past `lim`."""
    p = start
    while p < lim:
        n = 1
        while bits[p:p + n] not in code:
            n += 1
            assert n <= H.MAX_BITS
        p += n
    return p


@pytest.mark.parametrize("backend", BACKENDS)
def test_tracks_that_never_merge(backend):
    """A deep skewed tree whose all-zero codeword (the longest) fills the streams: a track started at any bit reads the same
    zeros and never meets the true one, so every fine boundary of a coarse range records a map that is not constant, and the
    true candidate must be carried through all of them."""
    for depth in (11, 7):
        w = _skewed(depth, ASCII0)
        code = {format(c, f"0{n}b"): s for s, (c, n) in H.canonical_code(w).items()}
        deep = [s for s, (c, n) in H.canonical_code(w).items() if c == 0 and n == depth]
        assert len(deep) == 1
        seg = 6000
        rng = np.random.default_rng(depth)
        d = bytes(deep) * (4 * seg - 300) + _data(rng, w, 300)
        sec = H.literals_section(d, w)
        lit = H.read_literals(sec)
        assert lit.depth == depth and lit.counts == [seg] * 4
        # the edge: in stream 0, the tracks started at the top of coarse range 1 land on `depth` different offsets at its
        # first inner fine boundary, and the same holds one coarse range further
        stream0 = H.huffman_stream(d[:seg], H.canonical_code(w))
        bits = _payload_bits(stream0)
        s = geometry(len(bits))[0]
        for ctop in (PER * s, 2 * PER * s):
            lands = {_boundaries(bits, code, ctop + k, ctop + s) for k in range(depth)}
            assert len(lands) == depth, (depth, ctop, lands)
        frame = H.literals_only([(sec, len(d))])
        _agree(backend, frame, d, f"never merging, depth {depth}")


def _flip(stream, bit):
    """The stream with payload bit `bit` (counted from the top) inverted."""
    p0 = len(_payload_bits(stream))
    v = int.from_bytes(stream, "little") ^ (1 << (p0 - 1 - bit))
    return v.to_bytes(len(stream), "little")


@pytest.mark.parametrize("backend", BACKENDS)
def test_flipped_bit_is_refused(backend):
    """One bit flipped in the middle of a coarse range, and one in the first fine range of a coarse range, of a big stream:
    the reader refuses each, the device refuses each with E_HUF_STREAM, and in a job with good archives around it only the
    corrupt archive fails."""
    w = _skewed(5, ASCII0)
    code = H.canonical_code(w)
    rng = np.random.default_rng(21)
    seg = 8000
    d = _data(rng, w, 4 * seg)
    good = [H.huffman_stream(d[k * seg:(k + 1) * seg], code) for k in range(4)]
    s = geometry(len(_payload_bits(good[2])))[0]
    frames = []
    for label, lo, hi in (("middle of a coarse range", 10 * PER * s + s + s // 2, 10 * PER * s + 3 * s),
                          ("first fine range", 20 * PER * s + s // 4, 20 * PER * s + s)):
        # the first bit from `lo` whose flip the reader refuses (a flip may also turn one codeword into others and still fit)
        for bit in range(lo, hi):
            bad = good[:2] + [_flip(good[2], bit)] + good[3:]
            sec = H.literals_section(d, w, stream_bytes=bad)
            try:
                H.read_literals(sec)
            except (ValueError, AssertionError):
                break
        else:
            pytest.fail(f"{label}: no refused flip in bits [{lo}, {hi})")
        frame = H.literals_only([(sec, len(d))])
        with pytest.raises(N.NafIoError, match=r"device status 0x4\)"):
            N.shared_context(0, library(backend)).zstd_decompress(frame, len(d))
        frames.append(frame)
    # the corrupt archives between archives of the same big streams intact, and ordinary ones
    good_arc = _as_text_archive(d, H.literals_only([(H.literals_section(d, w, stream_bytes=good), len(d))]))
    crafted = [a for f in frames for a in (_as_text_archive(b"0" * len(d), f), good_arc)]
    arcs, res = _batch(backend, crafted, strict=False)
    for i, (r, a) in enumerate(zip(res, arcs)):
        if i in (1, 5):
            assert r.status != 0, i
        else:
            assert r.status == 0
            assert_same_as_oracle(r, O.decode(a), f"archive {i}")

"""Archives that lie about their sizes, batches with one bad member, and zstd frame shapes NAF writers never emit
(content checksums, very long windows).  The reference rejects such files lazily and never corrupts memory
(SURVEY 5); the device path sizes its arenas from header fields, so every one of them is validated on the host first.
Both backends; the emulator build is what an AddressSanitizer run (tests/emul/Makefile: `make asan`) checks."""
import numpy as np
import pytest

import _cases as K
import _oracle as O
import nafcodec_b200 as N
from _harness import BACKENDS, assert_same_as_oracle, library
from nafcodec_b200 import _ffi

pytestmark = pytest.mark.parametrize("backend", BACKENDS)


def _varint(n):
    return O.write_variable_length(n)


def _section(payload: bytes, claimed=None):
    frame = O.zstd_compress(payload, 3)
    return _varint(len(payload) if claimed is None else claimed) + _varint(len(frame)) + frame


def _header(flags, nrec, line=60):
    return bytes([0x01, 0xF9, 0xEC, 0x01, flags, 0x20]) + _varint(line) + _varint(nrec)


@pytest.mark.parametrize("nrec", [2 ** 61, 2 ** 64 - 1])
def test_absurd_record_count_is_harmless(backend, nrec):
    # number_of_sequences is any varint the file likes; the streams hold 200 000 ids.  The offset tables are sized by
    # what the streams can hold, so nothing is written out of bounds and the ids that exist are still returned.
    lib = library(backend)
    ids = b"\0" * 200_000
    data = _header(0x20 | 0x08, nrec) + _section(ids) + _section(b"")
    r = N.shared_context(0, lib).decode([N.parse_archive(data, lib)])[0]
    assert r.n_records == nrec and r.n_ids == 200_000 and r.n_lengths == 0
    assert r.id_bytes(0) == b"" and r.id_bytes(199_999) == b"" and r.id_bytes(200_000) is None
    assert len(r.id_offsets) == 200_001 and int(r.id_offsets[-1]) == 200_000


@pytest.mark.parametrize("claimed", [2 ** 64 - 16, 2 ** 40, 10 ** 9])
def test_absurd_original_size_is_rejected(backend, claimed):
    # a frame of c bytes regenerates at most (c / 3 + 1) * 128 KiB: anything beyond is refused before the arena is laid out
    lib = library(backend)
    data = _header(0x20 | 0x08, 3) + _section(b"a\0b\0c\0", claimed) + _section(b"")
    with pytest.raises(N.NafIoError):
        N.shared_context(0, lib).decode([N.parse_archive(data, lib)])


def test_lengths_longer_than_the_sequence_do_not_overrun(backend):
    # ADVICE r1: 2 residues stored, one length word of 16000 -> k_unpack used to write 16 KB past the arena
    lib = library(backend)
    good = O.encode(ids=[b"x"], sequences=[b"AC"])
    L = O.parse(good)
    words = np.array([16000], dtype="<u4").tobytes()
    frame = O.zstd_compress(words, 3)
    s_len, s_seq = L.sec[2], L.sec[4]
    data = (good[:s_len.offset - 2] + _varint(4) + _varint(len(frame)) + frame +
            good[s_len.offset + s_len.compressed_size:])
    assert O.parse(data).sec[4].original_size == 2
    with pytest.raises(N.NafIoError):                      # E_LENGTHS -> UnexpectedEof, as the reference's read_exact would
        N.shared_context(0, lib).decode([N.parse_archive(data, lib)])
    # and the formatter stays inside its buffers too
    with pytest.raises(N.NafIoError):
        N.to_text(data, "fasta", _library=lib)
    del s_seq


def test_one_bad_archive_does_not_fail_the_batch(backend):
    # the reference decodes archives with independent Decoders; a batch call reports per archive
    lib = library(backend)
    arcs = [K.genome(700 + i, 20_000 + 777 * i, level=3) for i in range(4)]
    want = [O.decode(a) for a in arcs]
    corrupt = bytearray(arcs[1])
    L = O.parse(arcs[1])
    s = L.sec[4]
    corrupt[s.offset + s.compressed_size // 2] ^= 0x5A               # damages the sequence frame (device-side detection)
    truncated_frame = bytearray(arcs[2])
    s2 = O.parse(arcs[2]).sec[4]
    truncated_frame[s2.offset + 2] = 0xFF                            # first block header: reserved type / absurd size (host walk)
    batch = [arcs[0], bytes(corrupt), bytes(truncated_frame), arcs[3]]
    parsed = [N.parse_archive(a, lib) for a in batch]
    ctx = N.shared_context(0, lib)
    res = ctx.decode(parsed, strict=False)
    assert res[0].status == 0 and res[3].status == 0
    assert_same_as_oracle(res[0], want[0], "good archive 0")
    assert_same_as_oracle(res[3], want[3], "good archive 3")
    assert res[2].status in (_ffi.ERR_INVALID_DATA, _ffi.ERR_UNEXPECTED_EOF) and res[2].sequence is None
    try:
        d1 = O.decode(bytes(corrupt))
    except O.OracleError:
        assert res[1].status in (_ffi.ERR_INVALID_DATA, _ffi.ERR_UNEXPECTED_EOF)
    else:                                                            # the flip landed where both decoders accept it
        assert res[1].status == 0
        assert_same_as_oracle(res[1], d1, "mutated archive")
    with pytest.raises(N.NafIoError, match="archive"):               # strict (default): the first bad archive raises, named
        ctx.decode(parsed)
    # text of the same batch: the good archives are formatted, the bad ones carry their status
    n = len(parsed)
    arr = (_ffi.Archive * n)(*parsed)
    texts = (_ffi.Text * n)()
    rc = lib.dll.nafgpu_format_batch(ctx._ctx, arr, n, _ffi.WANT_ALL, _ffi.TEXT_FASTA, _ffi.LINE_LENGTH_FROM_HEADER, texts)
    assert rc == 0
    assert texts[0].status == 0 and texts[0].size == len(O.format_text(arcs[0], "fasta"))
    assert texts[2].status != 0 and not texts[2].data


def test_frame_content_checksum_is_verified(backend):
    # libzstd (reached from decoder/mod.rs:221) verifies XXH64 when the frame carries one; so does k_frame_checksum
    ctx = N.shared_context(0, library(backend))
    rng = np.random.default_rng(5)
    for n in (0, 1, 3, 4, 7, 8, 31, 32, 33, 63, 64, 100, 4099, 300_001):
        p = bytes(rng.integers(0, 4, size=n, dtype=np.uint8) + 65)
        frame = O.zstd_compress(p, 3, checksum=True)
        assert frame[0] & 0x04, "Content_Checksum_flag"
        assert O.zstd_decompress(frame) == p
        assert ctx.zstd_decompress(frame, n) == p, n
        bad = bytearray(frame)
        bad[-1] ^= 0x80
        with pytest.raises(O.OracleError):
            O.zstd_decompress(bytes(bad))
        with pytest.raises(N.NafIoError, match="checksum"):
            ctx.zstd_decompress(bytes(bad), n)


def test_window_beyond_the_offset_encoding_is_refused(backend):
    # a frame that declares a 1 GiB window (zstd --long=30) is refused on the host instead of being mis-decoded
    # (tests/test_zstd_sequences.py: offsets up to 2^29, single-segment frames)
    ctx = N.shared_context(0, library(backend))
    p = b"ACGT" * 1000
    frame = bytearray(O.zstd_compress(p, 3))
    assert not (frame[0] & 0x20), "window descriptor present"
    assert ctx.zstd_decompress(bytes(frame), len(p)) == p
    frame[1] = (20 << 3)                                              # 2^30
    with pytest.raises(N.NafIoError, match="window"):
        ctx.zstd_decompress(bytes(frame), len(p))
    frame[1] = (19 << 3)                                              # 2^29: still representable
    assert ctx.zstd_decompress(bytes(frame), len(p)) == p


@pytest.mark.parametrize("max_bytes", [0, 1, 4096])
def test_windows_over_an_absurd_record_count(backend, max_bytes):
    # nafgpu_job_fetch_window: windows are clamped by what the streams hold, not by number_of_sequences (2^61 here); a window
    # far past the stored ids is empty-handed (id None), not out of bounds
    lib = library(backend)
    ids = b"".join(b"id%d\0" % k for k in range(5000))
    data = _header(0x20 | 0x08, 2 ** 61) + _section(ids) + _section(b"")
    ctx = N.Context(0, lib)
    ctx.prepare([N.parse_archive(data, lib)])
    ctx.run()
    w = ctx.fetch_window(0, 4990, 2 ** 61 - 4990, max_bytes)
    assert w.n_records >= 1 and w.id_bytes(0) == b"id4990"
    if max_bytes == 0:
        assert w.n_records == 2 ** 61 - 4990 and w.n_ids == 10 and w.id_bytes(9) == b"id4999" and w.id_bytes(10) is None
    w = ctx.fetch_window(0, 2 ** 60, 1000, max_bytes)
    assert w.n_ids == 0 and w.id_bytes(0) is None and w.n_records >= 1
    w = ctx.fetch_window(0, 2 ** 64 - 1, 2 ** 64 - 1, max_bytes)        # first past the end: empty window
    assert w.n_records == 0
    ctx.close()


def test_window_of_a_corrupt_archive_reports_its_status(backend):
    lib = library(backend)
    good = O.encode(ids=[b"a", b"b"], sequences=[b"ACGT" * 300, b"GGCC" * 200], level=3)
    L = O.parse(good)
    bad = bytearray(good)
    s = L.sec[4]
    for k in range(s.offset + 6, s.offset + s.compressed_size - 2):
        bad[k] ^= 0xA5
    dec = N.Decoder(__import__("io").BytesIO(bytes(bad)), buffer_size=64, _library=lib)
    with pytest.raises(N.NafIoError):
        next(dec)
    # and a header-level lie is refused by prepare, before any window
    data = _header(0x20 | 0x08, 3) + _section(b"a\0b\0c\0", 2 ** 40) + _section(b"")
    with pytest.raises(N.NafIoError):
        next(N.Decoder(__import__("io").BytesIO(data), buffer_size=64, _library=lib))


def test_windows_when_the_header_overstates_the_records(backend):
    # test_edge_cases.py::test_header_says_more_records_than_the_streams_hold, through windows of one record
    data = bytearray(O.encode(ids=[b"r1", b"r2"], comments=[b"c1", b"c2"], sequences=[b"ACGT", b"GG"]))
    L = O.parse(bytes(data))
    data[L.header_size - 1] = 5
    recs = list(N.Decoder(__import__("io").BytesIO(bytes(data)), buffer_size=1, _library=library(backend)))
    assert len(recs) == 5 and recs[2].id is None and recs[2].sequence is None and recs[1].sequence == "GG"
    assert [r.length for r in recs] == [4, 2, None, None, None]

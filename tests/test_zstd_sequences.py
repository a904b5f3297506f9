"""The zstd kernels on frames built to order (tests/_zseq.py): every offset code up to 2^29, the repeat-offset special cases,
literal and match lengths at the code boundaries, every table mode and literals header form.  Frames made by libzstd's match
finder (the rest of the suite) contain only what that finder happens to emit; each case here asserts through `frame_codes`
that the code, mode or boundary it is named after is really in its frame, then that the plain replay, libzstd and the
device agree on every byte."""
import numpy as np
import pytest

import _cases as K
import _oracle as O
import _zseq as Z
import nafcodec_b200 as N
from _harness import BACKENDS, assert_same_as_oracle, library
from conftest import read_golden

ASCII = np.frombuffer(bytes(range(48, 112)), np.uint8)       # 64 printable symbols: payloads that are valid TEXT records


def _text(rng, n):
    return bytes(rng.choice(ASCII, size=n))


def _ctx(backend):
    return N.shared_context(0, library(backend))


def _decodes(backend, payload, frame, label=""):
    """libzstd and the device regenerate `payload` (the replay of the frame's sequence list) from `frame`, and frame_codes
    reads every length and offset of the frame right: its sequences replayed over the payload's literals give the payload."""
    assert Z.libzstd_decompress(frame, len(payload)) == payload, label
    assert Z.regenerate(frame, payload) == payload, label
    got = _ctx(backend).zstd_decompress(frame, len(payload))
    if got != payload:
        x, y = np.frombuffer(got, np.uint8), np.frombuffer(payload, np.uint8)
        k = int(np.nonzero(x != y)[0][0])
        pytest.fail(f"{label}: device differs from byte {k} on ({int((x != y).sum())} bytes differ)")
    return Z.frame_codes(frame)


def _as_text_archive(payload, frame):
    """A TEXT archive of one record whose sequence section is `frame` (regenerating `payload`)."""
    arc = O.encode(sequence_type=O.TEXT, ids=[b"crafted"], sequences=[b"A" * len(payload)], level=1)
    s = O.parse(arc).sec[4]
    k = len(O.write_variable_length(s.compressed_size))
    return arc[:s.offset - k] + O.write_variable_length(len(frame)) + frame + arc[s.offset + s.compressed_size:]


def _batch_parity(backend, crafted):
    """Crafted archives in one decode_batch between ordinary ones (job-global sequence indices, table slots, seq_base shifted).
    Archives are walked by nafgpu_job_prepare, the only path that cuts long sections into parts (NAFGPU_WALK_SPLIT)."""
    arcs = [read_golden("phix.naf")] + [a for c in crafted for a in (c, K.multi_record_dna(5, 12, 900, level=19))]
    res = N.decode_batch(arcs, _library=library(backend))
    for i, (r, a) in enumerate(zip(res, arcs)):
        assert_same_as_oracle(r, O.decode(a), f"archive {i}")


def test_frame_codes_reads_libzstd_frames():
    """The reader the other cases rely on: on the fixtures and on frames of libzstd's own parsers (every table mode, repeat
    codes, treeless literals), its sequences replayed with the section's literals regenerate the section."""
    for name in ["masked.naf", "LuxC.naf", "phix.naf", "CP040672.naf", "NZ_AAEN01000029.naf"]:
        data = read_golden(name)
        L = O.parse(data)
        for i in range(6):
            s = L.sec[i]
            if s.present:
                frame = data[s.offset:s.offset + s.compressed_size]
                want = O.zstd_decompress(frame)
                assert Z.regenerate(frame, want) == want, (name, O.SEC_NAMES[i])
    rng = np.random.default_rng(5)
    p = b"".join(b"read/%d length=%d %s\n" % (i, i * 7 % 300, K.random_dna(rng, 40, b"ACGTN")) for i in range(6000))
    seen = set()
    for level, flush in ((1, 0), (19, 0), (3, 300), (19, 4001)):
        frame = K.zstd_frame(p, level, flush_every=flush)
        assert Z.regenerate(frame, p) == p, (level, flush)
        _, blocks = Z.frame_codes(frame)
        seen |= {b.lit_type for b in blocks} | {m for b in blocks for m in (b.ll_mode, b.of_mode, b.ml_mode)}
        seen |= {("ov", s[3]) for s in Z.all_seqs(blocks) if s[3] <= 3}
    assert {"huffman", "treeless", "fse", "repeat", "predefined", ("ov", 1), ("ov", 2), ("ov", 3)} <= seen, seen


# ---- offsets, one far match at every offset code ----------------------------------------------------------------------
def _far_blocks(rng, window_log, single):
    """Blocks that reach just past 2^window_log (window descriptor) or stay inside it (single segment, whose window is the
    content size), then a block of matches at distances 2^k - 3, 2^k - 2, 2^k + 2^(k-1) and 2^(k+1) - 4 for every offset
    code k that fits.  The space in between is filled with blocks of exactly 128 KiB: 251 new random bytes, repeated by an
    offset-251 match, so that a match read from a wrong distance lands on other bytes."""
    W = 1 << window_log
    head = 64 * 1024
    fill_to = W + 2 * head if not single else W - head - 8192
    blocks, pos = [], 0
    while pos < fill_to:
        m = min(Z.BLOCK, fill_to - pos) - 251
        blocks.append([(_text(rng, 251), m, 251), b""] if m >= 3 else [_text(rng, m + 251)])
        pos += m + 251
    blocks.append([_text(rng, head)])                              # recent random text: the sources of the short distances
    pos += head
    far, dists = [], []
    for k in range(2, window_log + 1):
        for d in sorted({(1 << k) - 3, (1 << k) - 2, (1 << k) + (1 << (k - 1)) - 3, (1 << (k + 1)) - 4}):
            here = pos + sum(1 + 20 for _ in far) + 1
            if d <= min(W, here) and d not in dists:
                far.append((_text(rng, 1), 20, d))
                dists.append(d)
    if not single and W not in dists:
        far.append((_text(rng, 1), 20, W))                         # an offset equal to the declared window
    blocks.append(far + [_text(rng, 7)])
    return blocks


# (2^26 on the emulator too: seconds there, and the first window that holds offsets with more than 24 extra bits, the top one set)
WINDOWS = [pytest.param("emul", w, id=f"emul-{w}") for w in (18, 22, 26)] + \
          [pytest.param("cuda", w, id=f"cuda-{w}", marks=[pytest.mark.gpu] + ([pytest.mark.slow] if w >= 28 else [])) for w in (22, 25, 27, 28, 29)]


@pytest.mark.parametrize("backend,window_log", WINDOWS)
@pytest.mark.parametrize("single", [True, False], ids=["single_segment", "window_descriptor"])
def test_offsets_by_code(backend, window_log, single):
    rng = np.random.default_rng(window_log)
    payload, frame = Z.build(_far_blocks(rng, window_log, single), window_log=window_log, single_segment=single)
    hdr, blocks = _decodes(backend, payload, frame, f"window 2^{window_log}")
    assert hdr["single_segment"] == single
    codes = {s[2] for s in Z.all_seqs(blocks)}
    top = window_log if not single else window_log - 1
    assert set(range(2, top + 1)) <= codes, sorted(codes)
    assert blocks[0].btype == "compressed" and blocks[0].regen == Z.BLOCK     # filler blocks of exactly Block_Maximum_Size
    if not single:
        assert hdr["window"] == 1 << window_log
        assert max(s[6] for s in Z.all_seqs(blocks)) == 1 << window_log       # a match as far back as the window
    if window_log <= 27:                                                       # (the reference decoder's default limit)
        _batch_parity(backend, [_as_text_archive(payload, frame)])


@pytest.mark.parametrize("backend", BACKENDS)
def test_level_22_parser(backend):
    """libzstd's own ultra parser (level 22, window 2^27) on data with repeats far apart."""
    n = 1 << 20 if backend == "emul" else 24 << 20
    rng = np.random.default_rng(22)
    unit = _text(rng, 50_000)
    dna = K.random_dna(rng, n, b"ACGT")
    p = unit + dna[:n // 2] + unit[:30_000] + dna[n // 2:] + unit[10_000:]
    frame = O.zstd_compress(p, 22, window_log=27)
    _decodes(backend, p, frame, "level 22")
    assert max(s[6] for s in Z.all_seqs(Z.frame_codes(frame)[1])) > n // 2


# ---- repeat offsets -------------------------------------------------------------------------------------------------
def _rep_step(reps, off, ll):
    """The repeat offsets after a sequence, as libzstd codes it (ZSTD_finalizeOffBase) and the decoder updates them."""
    if ll and off == reps[0]:
        return reps
    if off == reps[1]:
        return [off, reps[0], reps[2]]
    return [off, reps[0], reps[1]]


def _rep_program(rng, n_blocks, seqs_per_block):
    """Blocks whose sequences pick, at random, one of the six repeat cases (ll > 0: rep0, rep1, rep2; ll == 0: rep1, rep2,
    rep0 - 1), a run of ll == 0 rep0 - 1, or a new offset."""
    reps = [1, 4, 8]
    blocks = [[_text(rng, 3000)]]
    pos = 3000
    for b in range(n_blocks):
        body = []
        n = seqs_per_block[b % len(seqs_per_block)]
        while len(body) < n:
            case = int(rng.integers(0, 8))
            run = int(rng.integers(2, 40)) if case == 6 else 1
            for _ in range(min(run, n - len(body))):
                ll = 0 if case >= 3 and case != 7 else int(rng.integers(1, 4))
                if case < 7:
                    off = [reps[0], reps[1], reps[2], reps[1], reps[2], reps[0] - 1, reps[0] - 1][case]
                else:
                    off = int(rng.integers(1, min(pos, 2900)))
                if not 1 <= off <= pos + ll:
                    break
                ml = int(rng.integers(20, 80))                      # (long enough that libzstd keeps the block compressed)
                body.append((_text(rng, ll), ml, off))
                pos += ll + ml
                reps = _rep_step(reps, off, ll)
        tail = _text(rng, int(rng.integers(0, 4)))
        pos += len(tail)
        blocks.append(body + [tail])
    return blocks


def _rep_kinds(blocks):
    """(ll == 0, Offset_Value) of every repeat-coded sequence."""
    return {(s[4] == 0, s[3]) for s in Z.all_seqs(blocks) if s[3] <= 3}


ALL_SIX = {(False, 1), (False, 2), (False, 3), (True, 1), (True, 2), (True, 3)}


def _rep_frames(rng, n_blocks):
    """(label, payload, frame, what frame_codes must find) of the repeat-offset cases."""
    out = []
    blocks = _rep_program(rng, n_blocks, [1, 5, 32, 33, 2, 90])
    p, f = Z.build(blocks)
    out.append(("six cases", p, f, lambda bl: ALL_SIX <= _rep_kinds(bl)))
    # the first sequence of a frame against the initial repeat offsets 1, 4, 8 (ll > 0: Offset_Value 1, 2, 3)
    for off, ov in ((1, 1), (4, 2), (8, 3)):
        p, f = Z.build([[(_text(rng, 9), 300, off), b"z"]])
        out.append((f"first sequence, offset {off}", p, f, lambda bl, ov=ov: bl[0].seqs[0][3] == ov))
    # the first sequence of a block after a raw, an RLE and a literals-only block, with ll == 0 (4 = rep1, 8 = rep2)
    for kind, lead in (("raw", [[bytes(range(256)) * 8]]), ("rle", [[_text(rng, 40)], [(b"q", 4999, 1), b""]]), ("literals-only", [[b"ACGT" * 600]])):
        for off, ov in ((4, 1), (8, 2)):
            p, f = Z.build(lead + [[(b"", 300, off), (b"k", 50, 17), b""]], literal_mode=Z.LIT_RAW if kind == "raw" else 0)
            want = {"raw": "raw", "rle": "rle", "literals-only": "compressed"}[kind]

            def ok(bl, want=want, ov=ov, kind=kind):
                prev = bl[-2]
                return prev.btype == want and (kind != "literals-only" or not prev.seqs) and bl[-1].seqs[0][3] == ov and bl[-1].seqs[0][4] == 0
            out.append((f"first sequence after a {kind} block, offset {off}", p, f, ok))
    # a repeat offset set 10^4 blocks earlier: three offsets, then 10^4 blocks without sequences, then rep0, rep1, rep2
    far = [[_text(rng, 500)], [(b"a", 110, 100), (b"b", 120, 200), (b"c", 130, 300), b""]]
    far += [[_text(rng, 2)] for _ in range(10_000)]
    far += [[(b"d", 140, 300), (b"e", 150, 200), (b"f", 160, 100), b"g"]]
    p, f = Z.build(far)
    out.append(("repeat offsets 10^4 blocks back", p, f, lambda bl: [s[3] for s in bl[-1].seqs] == [1, 2, 3] and len(bl) > 10_000))
    return out


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("env", [{}, {"NAFGPU_FS_TILE": "37"}, {"NAFGPU_WALK_SPLIT": "1"}, {"NAFGPU_WALK_SPLIT": "5"},
                                 {"NAFGPU_TINY_BLOCKS": "0"}, {"NAFGPU_TINY_BLOCKS": "1"}],
                         ids=["default", "fs_tile_37", "walk_split_1", "walk_split_5", "tiny_0", "tiny_1"])
def test_repeat_codes(backend, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(8)
    frames = _rep_frames(rng, 150 if backend == "emul" else 3000)
    for label, p, f, present in frames:
        _, blocks = _decodes(backend, p, f, label)
        assert present(blocks), label
        if len(blocks) > 2 * 37:
            # (a frame of more than two tiles of 37 blocks: the tiled scan ran on it)
            assert _ctx(backend).stats().n_blocks == len(blocks), label
    # the walk in parts happens for archives only: every frame with a text payload, spliced into one, in one batch
    _batch_parity(backend, [_as_text_archive(p, f) for _, p, f, _ in frames if p.isascii()])


# ---- lengths -------------------------------------------------------------------------------------------------------
def _length_blocks(rng):
    """Match lengths at every ML code boundary and 131072 - ll; literal lengths at every LL code boundary up to 65536 and
    above, paired so that the ML and LL extra bits are 31 wide together; overlapping copies at distances around the 16- and
    32-byte copy widths; matches that end a block; blocks without and with many trailing literals."""
    blocks = [[_text(rng, Z.BLOCK)]]                                 # random text to copy from
    pos = Z.BLOCK
    cur, size = [], 0

    def add(ll, ml, off, new_block=False):
        nonlocal cur, size, pos
        if new_block or size + ll + ml > Z.BLOCK - 16:
            if cur:
                blocks.append(cur + [b""])
            cur, size = [], 0
        cur.append((_text(rng, ll), ml, off)); size += ll + ml; pos += ll + ml

    for c in range(len(Z.ML_BASE)):
        for ml in (Z.ML_BASE[c], Z.ML_BASE[c] + (1 << Z.ML_BITS[c]) - 1):
            ml = min(ml, Z.BLOCK - 1)
            add(1, ml, int(rng.integers(1, min(pos, 100_000))))
    for c in range(len(Z.LL_BASE)):
        for ll in (Z.LL_BASE[c], Z.LL_BASE[c] + (1 << Z.LL_BITS[c]) - 1):
            add(min(ll, Z.BLOCK - 3 - c), 3 + c, int(rng.integers(1, 5000)))
    for ll, ml in ((65536 + 12345, 32771 + 16000), (32768 + 5000, 65539 + 20000), (65536, 65536 - 16), (1, Z.BLOCK - 1)):
        add(ll, ml, int(rng.integers(1, 90_000)), new_block=True)
    for d in (1, 2, 3, 4, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65):
        for ml in sorted({3, 4, 5, d - 1, d, d + 1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 100, 1000} - {0, 1, 2}):
            add(int(rng.integers(0, 3)), ml, d)
    blocks.append(cur + [b""])                                     # the last match ends the block
    # LL code 35 (16 extra bits) beside ML code 51 (15): a 31-bit ML+LL read, inside a sequence bitstream too long to be
    # staged in shared memory (more than 16 KiB: k_decode_sequences' global-memory reader, seq_produce)
    body = [(b"", int(rng.integers(3, 6)), (1 << int(rng.integers(14, 21))) + int(rng.integers(0, 999))) for _ in range(7000)]
    body.insert(3000, (_text(rng, 65536), 32771 + 29, 33_000))
    blocks.append(body + [b""])
    blocks.append([(_text(rng, 40), 5000, 33), _text(rng, 9000)])   # many trailing literals
    return blocks


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("lz_small", ["0", "8192"])
def test_lengths(backend, monkeypatch, lz_small):
    monkeypatch.setenv("NAFGPU_LZ_SMALL", lz_small)
    rng = np.random.default_rng(3)
    p, f = Z.build(_length_blocks(rng), window_log=22)
    _, blocks = _decodes(backend, p, f, "lengths")
    seqs = Z.all_seqs(blocks)
    assert set(range(53)) <= {s[1] for s in seqs} and set(range(36)) <= {s[0] for s in seqs}
    assert any(Z.LL_BITS[s[0]] + Z.ML_BITS[s[1]] == 31 for s in seqs), "ML+LL extra bits 31 wide"
    assert any(s[4] + s[5] == Z.BLOCK for s in seqs)
    assert any(b.seq_bytes > 16384 and any(s[0] == 35 and s[1] == 51 for s in b.seqs) for b in blocks)
    assert {(d, m) for d in (1, 16, 32, 64) for m in (15, 16, 17, 31, 32, 33, 63, 64, 65)} <= {(s[6], s[5]) for s in seqs}
    assert any(b.btype == "compressed" and b.regen == Z.BLOCK and b.seqs and b.lit_regen == sum(s[4] for s in b.seqs) for b in blocks), \
        "a block of 128 KiB that ends with a match"
    _batch_parity(backend, [_as_text_archive(p, f)])


# ---- table modes and literals --------------------------------------------------------------------------------------
def _mode_blocks(rng):
    """A block of 3000 sequences whose codes spread over every LL, ML and OF code (FSE at the largest accuracy logs), a block
    where every match length is the same (RLE) and the literal lengths few (predefined), behind 2 MiB of text."""
    blocks, pos = [], 0
    for _ in range(16):
        blocks.append([_text(rng, Z.BLOCK)]); pos += Z.BLOCK
    body, size = [], 0
    while len(body) < 3000:
        llc, mlc = int(rng.integers(0, 26)), int(rng.integers(0, 43))
        ll = Z.LL_BASE[llc] + int(rng.integers(0, 1 << Z.LL_BITS[llc]))
        ml = Z.ML_BASE[mlc] + int(rng.integers(0, 1 << Z.ML_BITS[mlc]))
        if size + ll + ml > Z.BLOCK - 8:
            ll, ml = int(rng.integers(0, 3)), 3
        if size + ll + ml > Z.BLOCK - 8:
            break
        off = (1 << int(rng.integers(2, 21))) + int(rng.integers(0, 4))
        body.append((_text(rng, ll), ml, off)); size += ll + ml
    blocks.append(body + [b""])
    blocks.append([(_text(rng, 1 + i % 3), 20, 1000 + 7 * i) for i in range(200)] + [b"x"])
    blocks.append([(_text(rng, 5), 7 + i, 3000 + 100 * i) for i in range(4)] + [b"y"])
    return blocks


def _fib_symbols(rng):
    """All 256 symbols, 20 of them with Fibonacci counts (a Huffman tree deeper than 11 without the depth limit), shuffled."""
    fib = [1, 1]
    while len(fib) < 20:
        fib.append(fib[-1] + fib[-2])
    counts = fib + [1] * 236
    syms = np.repeat(np.arange(256, dtype=np.uint8), counts)
    return bytes(rng.permutation(syms))


def _literal_frames(rng):
    """(label, payload, frame, literals kind, size): literals sections at the boundaries of their header forms (raw: 31/32,
    4095/4096; Huffman: 1023/1024, 16383/16384), one and four Huffman streams, up to nearly 128 KiB; a match in each block
    saves enough that libzstd keeps the block compressed."""
    out = []
    for mode, name, sizes in ((Z.LIT_RAW, "raw", (31, 32, 4095, 4096, 126_976)), (Z.LIT_HUFFMAN, "huffman", (200, 1023, 1024, 16383, 16384, 126_976))):
        for n in sizes:
            text = K.random_dna(rng, n, b"ACGT")
            ml = min(Z.BLOCK - n, max(64, n // 16))
            blocks = [[_text(rng, 4096)], [(text, ml, 4000), b""]]
            out.append((f"{name} literals of {n}", *Z.build(blocks, literal_mode=mode), name, n))
    fib = _fib_symbols(rng)
    out.append(("fibonacci", *Z.build([[fib], [(fib[::-1], 30, 20_001), b""]], literal_mode=Z.LIT_HUFFMAN), "huffman", 11))
    # many blocks of one distribution: the tree is described once and reused (treeless) across every walk-part cut
    acgt = K.random_dna(rng, 400 * 300, b"ACGTACGTN")
    out.append(("treeless", *Z.build([[(acgt[i:i + 300], 8, 150), b""] for i in range(0, len(acgt), 300)]), "treeless", 0))
    return out


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("huf_block_min", ["1", "1000000"])
def test_table_modes_and_literals(backend, monkeypatch, huf_block_min):
    monkeypatch.setenv("NAFGPU_HUF_BLOCK_MIN", huf_block_min)
    rng = np.random.default_rng(12)
    p, f = Z.build(_mode_blocks(rng), window_log=22)
    _, blocks = _decodes(backend, p, f, "table modes")
    dense, rle, few = blocks[-3:]
    assert (dense.ll_mode, dense.of_mode, dense.ml_mode) == ("fse", "fse", "fse") and dense.al == {"ll": 9, "of": 8, "ml": 9}, (dense.modes, dense.al)
    assert rle.ml_mode == "rle", rle.modes
    assert "predefined" in (few.ll_mode, few.of_mode, few.ml_mode), few.modes
    streams = set()
    for label, p, f, kind, n in _literal_frames(rng):
        _, blocks = _decodes(backend, p, f, label)
        lit = [b for b in blocks if b.btype == "compressed"]
        if kind == "raw":
            assert any(b.lit_type == "raw" and b.lit_regen == n for b in lit), label
        elif kind == "huffman" and label != "fibonacci":
            assert any(b.lit_type in ("huffman", "treeless") and b.lit_regen == n for b in lit), label
            streams |= {b.lit_streams for b in lit if b.lit_regen == n}
        elif label == "fibonacci":
            assert max(b.huf_depth or 0 for b in lit) == 11, label
        else:
            assert sum(b.lit_type == "treeless" for b in lit) > 300, label
            monkeypatch.setenv("NAFGPU_WALK_SPLIT", "1")                   # (every block a part of its own: the tree crosses each cut)
            _batch_parity(backend, [_as_text_archive(p, f)])
            monkeypatch.delenv("NAFGPU_WALK_SPLIT")
    assert streams == {1, 4}


# ---- single-segment frames above 512 MiB -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.slow
def test_single_segment_frame_above_512_mib():
    """A single-segment header declares no window: its window is the content size.  2^29 + 2^20 bytes, one match more than
    2^29 back."""
    rng = np.random.default_rng(30)
    size = (1 << 29) + (1 << 20)
    head = _text(rng, 4096)
    blocks, pos = [[head]], 4096
    while pos < size - 8192:
        m = min(Z.BLOCK, size - 8192 - pos) - 251
        blocks.append([(_text(rng, 251), m, 251), b""] if m >= 3 else [_text(rng, m + 251)])
        pos += m + 251
    tail = size - pos - 200
    blocks.append([(_text(rng, tail), 100, pos + tail - 1000), (b"!", 99, (1 << 29) + 17), b""])
    payload, frame = Z.build(blocks, window_log=30, single_segment=True)
    assert len(payload) == size
    hdr, bl = _decodes("cuda", payload, frame, "single segment above 512 MiB")
    assert hdr["single_segment"] and hdr["window"] == size
    assert max(s[6] for s in Z.all_seqs(bl)) > 1 << 29


@pytest.mark.parametrize("backend", BACKENDS)
def test_windows_beyond_the_offset_encoding_are_refused(backend):
    """A window descriptor above 2^29 and a single-segment header claiming more than 2^30 bytes are refused by the host walk,
    before anything of that size is allocated; a single-segment header of 2^29 + 2^20 bytes is not refused for its window
    (here it only disagrees with the size the caller expects; test_single_segment_frame_above_512_mib decodes one)."""
    ctx = _ctx(backend)
    rng = np.random.default_rng(31)
    blocks = [[_text(rng, 3000)], [(b"x", 500, 2999), b"y"]]
    p, f = Z.build(blocks, window_log=20, single_segment=False)
    assert not Z.frame_codes(f)[0]["single_segment"] and ctx.zstd_decompress(f, len(p)) == p
    bad = bytearray(f)
    bad[1] = 20 << 3                                                   # window descriptor: 2^30
    assert Z.libzstd_decompress(bytes(bad), len(p)) == p
    with pytest.raises(N.NafIoError, match="window"):
        ctx.zstd_decompress(bytes(bad), len(p))
    p, f = Z.build(blocks, window_log=20, single_segment=True)
    hdr, _ = Z.frame_codes(f)
    assert hdr["single_segment"] and f[0] >> 6 == 1                    # 2-byte content size
    body = f[3:]
    for claim, refused in (((1 << 30) + 1, True), ((1 << 29) + (1 << 20), False)):
        edited = bytes([0xE0 | (f[0] & 0x04)]) + claim.to_bytes(8, "little") + body      # 8-byte content size, single segment
        assert Z.frame_codes(edited)[0]["window"] == claim
        with pytest.raises(N.NafIoError) as e:
            ctx.zstd_decompress(edited, len(p))
        assert ("window" in str(e.value)) == refused, str(e.value)

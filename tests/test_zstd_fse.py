"""The FSE sequence decoders (k_build_tables<0>: fse_read_ncount_staged and fse_build_warp; k_decode_sequences: seq_produce3s
and the global-memory seq_produce; k_decode_sequences_tiny: seq_produce3) on sequences sections written to order by
tests/_zfse.py: every accuracy log, -1 symbols that really occur, single-symbol tables, wide symbols, zero runs, the longest
descriptions, RLE and repeat modes, every Number_of_Sequences form, each end-marker bit, and the sections a decoder must
refuse.  Each case checks that the plain replay, libzstd and the device agree and that frame_codes finds the case's edge
(mode, accuracy log, distribution, codes, bitstream size, header form) in the frame."""
import numpy as np
import pytest

import _cases as K
import _oracle as O
import _zfse as F
import _zseq as Z
import nafcodec_b200 as N
from _harness import BACKENDS, assert_same_as_oracle, library
from conftest import read_golden

HISTORY = 1 << 17                       # raw text in front of the sequence blocks: offset codes up to 16 have a source
OF_TOP = 16
READERS = pytest.mark.parametrize("tiny", ["0", "1"], ids=["tiny_0", "tiny_1"])


def _ctx(backend):
    return N.shared_context(0, library(backend))


def _writer(seed, history=HISTORY):
    w = F.Writer(np.random.default_rng(seed))
    for k in range(0, history, 1 << 16):
        w.raw(w.text(min(1 << 16, history - k)))
    return w


def _decodes(backend, w, label=""):
    """The writer's frame: its replay (the payload), libzstd, frame_codes' regeneration and the device agree.  Returns
    frame_codes' blocks."""
    payload, frame = w.frame()
    assert Z.regenerate(frame, payload) == payload, label
    assert Z.libzstd_decompress(frame, len(payload)) == payload, label
    got = _ctx(backend).zstd_decompress(frame, len(payload))
    if got != payload:
        x, y = np.frombuffer(got, np.uint8), np.frombuffer(payload, np.uint8)
        k = int(np.nonzero(x != y)[0][0])
        pytest.fail(f"{label}: device differs from byte {k} on ({int((x != y).sum())} bytes differ)")
    return Z.frame_codes(frame)[1]


def _used(blocks, kind, index=None):
    """Codes of `kind` found in the bitstreams of `blocks` (or of blocks[index])."""
    col = {"ll": 0, "ml": 1, "of": 2}[kind]
    bl = blocks if index is None else [blocks[index]]
    return {s[col] for b in bl for s in b.seqs}


def _filler(kind, rng):
    """A code of `kind` for the kinds not under test: small, in the predefined tables."""
    return {"ll": int(rng.integers(0, 16)), "of": int(rng.integers(2, 11)), "ml": int(rng.integers(0, 24))}[kind]


def _want(rng, kind, symbols, n):
    """n code triples: `kind` cycles through `symbols`, the other kinds small codes."""
    out = []
    for i in range(n):
        t = {k: _filler(k, rng) for k in F.KINDS}
        t[kind] = symbols[i % len(symbols)]
        out.append((t["ll"], t["of"], t["ml"]))
    return out


def _usable(kind, syms):
    """Symbols a block can use: offset codes up to OF_TOP, LL and ML codes below the ones a 128 KiB block cannot hold twice."""
    return [s for s in syms if kind != "of" or s <= OF_TOP]


def _table_program(w, kind, al, norm, rng, use=None, tiny=False, others=None):
    """Blocks that describe (al, norm) for `kind` once and repeat it, until every symbol of `use` (default: every usable
    symbol with nonzero probability) has occurred in a bitstream.  The other kinds: predefined, or `others` specs."""
    use = use if use is not None else _usable(kind, [s for s, c in enumerate(norm) if c])
    # each symbol once per block at most where its lengths are long; a tiny block (<= 32 sequences) when asked
    want = _want(rng, kind, sorted(use, key=lambda s: rng.random()) * 2, len(use) * 2)
    groups = F.pack(rng, want, len(w.out))
    if tiny:
        groups = [g[i:i + 32] for g in groups for i in range(0, len(g), 32)]
    secs = []
    for i, g in enumerate(groups):
        spec = {"ll": ("predefined",), "of": ("predefined",), "ml": ("predefined",)}
        spec.update(others or {})
        spec[kind] = ("fse", al, norm) if i == 0 else ("repeat",)
        secs.append(w.seq_block(g, **spec, tail=int(rng.integers(0, 5))))
    return secs


def _shapes(kind, al, top):
    """(label, norm): flat and skewed distributions over symbols 0..top."""
    syms = list(range(min(top + 1, 1 << al)))
    return [("flat", F.distribution(al, {s: 1 for s in syms})),
            ("skewed", F.distribution(al, {s: 1 + (1 << max(0, 12 - s)) for s in syms}))]


TOPS = {"ll": 24, "of": OF_TOP, "ml": 40}


# ---- 1. accuracy logs -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_accuracy_logs(backend, monkeypatch, tiny):
    """Every accuracy log from 5 to the kind's maximum, flat and skewed, each described once and then repeated until every
    symbol of the table has been decoded."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(1)
    w = _writer(1)
    cases = []
    for kind in F.KINDS:
        for al in range(5, F.MAX_AL[kind] + 1):
            for label, norm in _shapes(kind, al, TOPS[kind]):
                first = len(w.blocks)
                _table_program(w, kind, al, norm, rng, tiny=al % 2 == 0)
                cases.append((kind, al, norm, first, len(w.blocks)))
    blocks = _decodes(backend, w, "accuracy logs")
    for kind, al, norm, a, b in cases:
        assert blocks[a].al[kind] == al and getattr(blocks[a], kind + "_mode") == "fse"
        assert all(getattr(x, kind + "_mode") == "repeat" for x in blocks[a + 1:b])
        assert _used(blocks[a:b], kind) == set(_usable(kind, [s for s, c in enumerate(norm) if c])), (kind, al)
    assert any(x.btype == "compressed" and len(x.seqs) <= 32 for x in blocks) and any(len(x.seqs) > 32 for x in blocks)


# ---- 2-4. low-probability, full-probability and wide symbols -------------------------------------------------------------
def _low_tables():
    """(label, kind, al, norm, symbols the bitstream must use)."""
    out = []
    for kind in F.KINDS:
        ms = F.MAX_SYM[kind]
        top = OF_TOP if kind == "of" else ms
        out.append((f"{kind} -1 at 0", kind, 6, F.distribution(6, {s: 1 + s % 3 for s in range(top + 1)}, low=(0,)), None))
        out.append((f"{kind} -1 at {ms}", kind, 6, F.distribution(6, {s: 1 for s in range(min(top, 20))}, low=(ms,)), None))
        # several -1 symbols: they take the top cells in symbol order
        lows = (1, 5, 6, 11, top)
        out.append((f"{kind} -1 among the top cells", kind, 7, F.distribution(7, {s: 1 + s for s in range(top + 1)}, low=lows), None))
    # the most -1 symbols a table can hold: LL 35 of 36 and ML 52 of 53 (one symbol takes the rest of 64 cells), OF all 32 of 32
    out.append(("ll 35 symbols at -1", "ll", 6, F.distribution(6, {3: 1}, low=[s for s in range(36) if s != 3]), None))
    out.append(("ml 52 symbols at -1", "ml", 6, F.distribution(6, {0: 1}, low=range(1, 53)), None))
    out.append(("of 32 symbols at -1", "of", 5, [-1] * 32, None))
    return out


@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_low_probability_symbols(backend, monkeypatch, tiny):
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(2)
    w = _writer(2)
    cases = []
    for label, kind, al, norm, use in _low_tables():
        a = len(w.blocks)
        _table_program(w, kind, al, norm, rng, use=use, tiny=len(cases) % 2 == 0)
        cases.append((label, kind, al, norm, a, len(w.blocks)))
    blocks = _decodes(backend, w, "low-probability symbols")
    for label, kind, al, norm, a, b in cases:
        low = {s for s, c in enumerate(norm) if c == -1}
        assert blocks[a].al[kind] == al and low
        used = _used(blocks[a:b], kind)
        assert set(_usable(kind, low)) <= used, (label, sorted(set(_usable(kind, low)) - used))
        t = Z._fse_table(al, norm)
        top = [s for s, _, _ in t[len(t) - len(low):]]
        assert top == sorted(low, reverse=True), label                     # -1 symbols in the top cells, in symbol order


@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_full_probability_tables(backend, monkeypatch, tiny):
    """One symbol holds all 2^AL cells: every state update reads 0 bits.  Each kind alone, then all three at once."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(3)
    w = _writer(3)
    full = {"ll": (9, 20), "of": (8, 14), "ml": (9, 40)}
    marks = []
    for kind, (al, s) in full.items():
        norm = [0] * s + [1 << al]
        _table_program(w, kind, al, norm, rng, tiny=kind != "ll")
        marks.append((len(w.blocks) - 1, {kind: (al, s)}))
    for al in (5, 7):
        specs = {"ll": ("fse", al, [0] * 7 + [1 << al]), "of": ("fse", min(al, 8), [0] * 9 + [1 << min(al, 8)]), "ml": ("fse", al, [0] * 30 + [1 << al])}
        seqs = F.seqs_for(rng, [(7, 9, 30)] * (20 if al == 5 else 300), len(w.out))
        w.seq_block(seqs, **specs, tail=3)
        marks.append((len(w.blocks) - 1, {"ll": (al, 7), "of": (al, 9), "ml": (al, 30)}))
    blocks = _decodes(backend, w, "full-probability tables")
    for i, want in marks:
        for kind, (al, s) in want.items():
            assert _used(blocks, kind, i) == {s}
    for sec in w.sections:
        for kind in F.KINDS:
            if sec.specs[kind][0] == "fse" and sec.specs[kind][2][-1] == 1 << sec.specs[kind][1]:
                assert all(nb == 0 for _, nb, _ in sec.tables[kind][1])


@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_wide_symbols(backend, monkeypatch, tiny):
    """Symbols of 33, 64 and 2^AL - k cells (state counters across 32-cell groups), every LL and every ML symbol in one
    table, and OF 30 and 31 described with nonzero probability but never used."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(4)
    w = _writer(4)
    cases = []
    for kind, al in (("ll", 9), ("ml", 9), ("of", 8)):
        size = 1 << al
        norm = [33, 64, 1, 2] + [0] * 3 + [size - 33 - 64 - 3 - 5 - 1, 5, -1]
        cases.append((kind, al, norm))
        for k in (1, 2, 3):
            cases.append((kind, al, [size - k] + [1] * k))
    cases.append(("ll", 9, F.distribution(9, {s: 1 + (s * 7) % 13 for s in range(36)})))
    cases.append(("ml", 9, F.distribution(9, {s: 1 + (s * 5) % 11 for s in range(53)})))
    cases.append(("of", 8, F.distribution(8, {s: 3 for s in range(OF_TOP + 1)} | {30: 1, 31: 1})))
    spans = []
    for kind, al, norm in cases:
        a = len(w.blocks)
        _table_program(w, kind, al, norm, rng, tiny=len(spans) % 2 == 0)
        spans.append((kind, al, norm, a, len(w.blocks)))
    blocks = _decodes(backend, w, "wide symbols")
    for kind, al, norm, a, b in spans:
        assert blocks[a].al[kind] == al
        assert _used(blocks[a:b], kind) == set(_usable(kind, [s for s, c in enumerate(norm) if c])), (kind, norm[:8])
    assert {s for s in range(36)} <= _used(blocks, "ll") and {s for s in range(53)} <= _used(blocks, "ml")
    assert not {30, 31} & _used(blocks, "of")
    assert max(max(n) for _, _, n in cases) == 511 and 33 in cases[0][2] and 64 in cases[0][2]


# ---- 5. zero runs ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_zero_runs(backend, monkeypatch, tiny):
    """Gaps of 1 to 7 zero-probability symbols (repeat flag 3 once, twice: 6 and 7 zeros), descriptions that stop before the
    kind's last symbol, and runs whose next symbol is the kind's last one."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(5)
    w = _writer(5)
    cases = []
    gaps = [0]
    for g in range(1, 8):
        gaps.append(gaps[-1] + g + 1)                                   # symbols 0, 2, 5, 9, 14, 20, 27, 35
    cases.append(("ll", 7, F.distribution(7, {s: 1 + s % 4 for s in gaps})))
    cases.append(("ml", 8, F.distribution(8, {s: 2 for s in gaps + [43, 52]})))
    cases.append(("of", 6, F.distribution(6, {s: 2 for s in gaps[:5]} | {16: 3})))
    for kind in F.KINDS:
        top = OF_TOP if kind == "of" else F.MAX_SYM[kind]
        cases.append((kind, 6, F.distribution(6, {0: 5, 3: 7}, length=4)))                 # stops long before the last symbol
        cases.append((kind, 5, [20] + [0] * (top - 1) + [12]))                               # one run up to the last symbol
        if kind == "of":
            cases.append((kind, 5, [31] + [0] * 30 + [-1]))                                  # ... of OF (31, never used)
    spans = []
    for kind, al, norm in cases:
        a = len(w.blocks)
        _table_program(w, kind, al, norm, rng, tiny=len(spans) % 2 == 0)
        spans.append((kind, al, norm, a, len(w.blocks)))
    blocks = _decodes(backend, w, "zero runs")
    for kind, al, norm, a, b in spans:
        assert _used(blocks[a:b], kind) == set(_usable(kind, [s for s, c in enumerate(norm) if c])), (kind, norm)
    assert cases[0][2].count(0) == sum(range(1, 8))


# ---- 6. the longest descriptions -----------------------------------------------------------------------------------------
def test_longest_descriptions_are_exact():
    """The longest legal description of each kind (an exact search): LL 50, OF 41, ML 74 bytes.  The ML description starts
    at most 91 bytes into the section (after the longest LL and OF ones), inside the 240 bytes k_build_tables stages, and
    k_build_tables only switches to global memory for a description that starts more than 176 bytes in: that branch cannot
    be reached by a section whose earlier descriptions are legal (an illegal one is refused before the next is read)."""
    sizes = {}
    for kind in F.KINDS:
        d, al, norm, runs = F.longest_description(kind)
        assert al == F.MAX_AL[kind] and Z._read_ncount(d + bytes(8), 0, F.MAX_SYM[kind])[2] == len(d)
        sizes[kind] = len(d)
    assert sizes == {"ll": 50, "of": 41, "ml": 74}
    assert sizes["ll"] + sizes["of"] + 80 <= 256 and sizes["ll"] + sizes["of"] + sizes["ml"] <= 240


def _longest_variants():
    """Legal descriptions as long as the longest ones whose symbols a block can use: LL (50 bytes) with LL 34 in use,
    ML (74 bytes, every cell ML 52); every OF description of 41 bytes gives all its cells to codes 29-31, beyond any window
    here (the longest, every cell to 31)."""
    ll = [0] * 34 + [1, 511]
    d_ll = F.description(9, ll, runs=[0] * 34)
    d_ml, al_ml, ml, runs_ml = F.longest_description("ml")
    d_of, al_of, of, runs_of = F.longest_description("of")
    return (ll, [0] * 34, d_ll), (ml, runs_ml, d_ml), (of, runs_of, d_of)


@pytest.mark.parametrize("backend", BACKENDS)
def test_longest_descriptions_back_to_back(backend):
    """The three longest descriptions in one block: 165 bytes of descriptions, the ML one 91 bytes in.  With OF's longest
    every sequence has offset code 31 (an offset of 2^31 or more): libzstd and the device refuse the block for its offsets, the device
    with a sequence status, not a table status (the descriptions were read and the tables built).  A decodable block puts
    the longest LL and ML descriptions around an OF description of every usable offset code."""
    (ll, rll, d_ll), (ml, rml, d_ml), (of, rof, d_of) = _longest_variants()
    assert (len(d_ll), len(d_of), len(d_ml)) == (50, 41, 74)
    rng = np.random.default_rng(6)
    # decodable: LL 34 and ML 52 (98 KiB per sequence pair), offsets 1..16
    w = _writer(6)
    of_ok = F.distribution(8, {s: 1 for s in range(OF_TOP + 1)})
    seqs = F.seqs_for(rng, [(34, 16, 52)], len(w.out))
    d_of_ok = F.description(8, of_ok)
    w.seq_block(seqs, ll=("fse", 9, ll), of=("fse", 8, of_ok), ml=("fse", 9, ml), desc=d_ll + d_of_ok + d_ml)
    blocks = _decodes(backend, w, "longest LL and ML")
    b = blocks[-1]
    assert b.al == {"ll": 9, "of": 8, "ml": 9} and (b.seqs[0][0], b.seqs[0][1]) == (34, 52)
    assert len(b.seqs) == 1 and b.size > 50 + len(d_of_ok) + 74
    # refused for its offsets: the three longest back to back
    w = _writer(7, history=1 << 16)
    seqs = [(32768, 65539, (1 << 31) + 5)]
    sec = w.seq_block(seqs, ll=("fse", 9, ll), of=("fse", 8, of), ml=("fse", 9, ml),
                      desc=d_ll + d_of + d_ml, bad_offsets=True)
    payload, frame = w.frame(check=False)
    _, bl = Z.frame_codes(frame)
    assert bl[-1].al == {"ll": 9, "of": 8, "ml": 9} and bl[-1].seqs[0][2] == 31
    assert len(sec.header) + 1 + len(d_ll) + len(d_of) == 1 + 1 + 91
    with pytest.raises(RuntimeError):
        Z.libzstd_decompress(frame, len(payload))
    with pytest.raises(N.NafIoError) as e:
        _ctx(backend).zstd_decompress(frame, len(payload))
    assert "device status 0x1)" not in str(e.value), str(e.value)


# ---- 7. RLE mode ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_rle_mode(backend, monkeypatch, tiny):
    """RLE at symbol 0 and at each kind's largest usable symbol (LL 35: literal lengths of 65536 and more, ML 52: match
    lengths of 65539 and more, OF 16 here), and repeat mode after an RLE table."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(7)
    w = _writer(8)
    marks = []
    for kind, syms in (("ll", (0, 35)), ("ml", (0, 52)), ("of", (0, 2, OF_TOP))):
        for s in syms:
            n = 1 if (kind, s) in (("ll", 35), ("ml", 52)) else (12 if s == 0 else 70)
            want = _want(rng, kind, [s], n)
            for i in range(2):
                seqs = F.seqs_for(rng, want, len(w.out))
                spec = {kind: ("rle", s) if i == 0 else ("repeat",)}
                w.seq_block(seqs, **spec, tail=2)
                marks.append((len(w.blocks) - 1, kind, s, spec[kind][0]))
    blocks = _decodes(backend, w, "RLE")
    for i, kind, s, mode in marks:
        assert getattr(blocks[i], kind + "_mode") == mode and _used(blocks, kind, i) == {s}
    assert max(s[4] for s in Z.all_seqs(blocks)) >= 65536 and max(s[5] for s in Z.all_seqs(blocks)) >= 65539


# ---- 8. repeat mode across blocks, walk parts and archives -------------------------------------------------------------
def _as_text_archive(payload, frame):
    """A TEXT archive of one record whose sequence section is `frame` (regenerating `payload`)."""
    arc = O.encode(sequence_type=O.TEXT, ids=[b"crafted"], sequences=[b"A" * len(payload)], level=1)
    s = O.parse(arc).sec[4]
    k = len(O.write_variable_length(s.compressed_size))
    return arc[:s.offset - k] + O.write_variable_length(len(frame)) + frame + arc[s.offset + s.compressed_size:]


def _batch(backend, crafted, strict=True):
    arcs = [read_golden("phix.naf")] + [a for c in crafted for a in (c, K.multi_record_dna(5, 12, 900, level=19))]
    res = _ctx(backend).decode([N.parse_archive(a, library(backend)) for a in arcs], strict=strict)
    return arcs, res


def _repeat_frame(seed, n_blocks):
    """A hand-built table for each kind described once, then repeated over n_blocks blocks, mixed with predefined and RLE
    blocks for the other kinds (which then repeat those)."""
    rng = np.random.default_rng(seed)
    w = _writer(seed, history=1 << 14)
    tables = {"ll": ("fse", 7, F.distribution(7, {s: 1 + s % 5 for s in range(20)}, low=(3, 17))),
              "of": ("fse", 6, F.distribution(6, {s: 2 for s in range(2, 14)}, low=(0,))),
              "ml": ("fse", 8, F.distribution(8, {s: 1 + s % 3 for s in range(30)}, low=(29,)))}
    for b in range(n_blocks):
        kind = F.KINDS[b % 3]
        spec = {k: ("repeat",) for k in F.KINDS}
        if b < 3:
            spec = dict(tables)
        elif b % 7 == 3:
            spec[kind] = ("predefined",)
        elif b % 7 == 5:
            spec[kind] = ("rle", 2 if kind != "of" else 5)
        elif b % 7 == 6:
            spec[kind] = tables[kind]
        use = {}
        for k in F.KINDS:
            sp = spec[k] if spec[k][0] != "repeat" else None
            cur = sp or w.sections[-1].specs_resolved[k]
            use[k] = cur
        n = [1, 5, 31, 33, 90][b % 5]
        want = []
        for _ in range(n):
            t = []
            for k in F.KINDS:
                sp = use[k]
                if sp[0] == "rle":
                    t.append(sp[1])
                elif sp[0] == "predefined":
                    t.append(_filler(k, rng))
                else:
                    t.append(int(rng.choice([s for s, c in enumerate(sp[2]) if c])))
            want.append((t[0], t[1], t[2]))
        sec = w.seq_block(F.seqs_for(rng, want, len(w.out)), **spec, tail=1)
        sec.specs_resolved = use
    return w


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("split", ["0", "1", "5"], ids=["default", "walk_split_1", "walk_split_5"])
def test_repeat_mode(backend, monkeypatch, split):
    if split != "0":
        monkeypatch.setenv("NAFGPU_WALK_SPLIT", split)
    w = _repeat_frame(9, 60 if backend == "emul" else 400)
    blocks = _decodes(backend, w, "repeat mode")
    modes = {(k, getattr(b, k + "_mode")) for b in blocks if b.btype == "compressed" for k in F.KINDS}
    assert {(k, m) for k in F.KINDS for m in ("fse", "repeat", "predefined", "rle")} <= modes
    assert sum(1 for b in blocks if b.btype == "compressed" and b.ll_mode == "repeat") > 20
    # the same frame, and a second one, as archives of a batch between ordinary archives: every table slot and walk part
    w2 = _repeat_frame(10, 40)
    crafted = [_as_text_archive(*x.frame()) for x in (w, w2)]
    arcs, res = _batch(backend, crafted)
    for i, (r, a) in enumerate(zip(res, arcs)):
        assert_same_as_oracle(r, O.decode(a), f"archive {i}")


# ---- 9. sequence counts -----------------------------------------------------------------------------------------------
COUNTS = [1, 8, 9, 31, 32, 33, 64, 65, 127, 128, 0x7EFF, 0x7F00, 43690]


@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_sequence_counts(backend, monkeypatch, tiny):
    """Number_of_Sequences in every form at its boundaries (127/128, 0x7EFF/0x7F00), 2-byte forms of counts below 128
    (non-canonical), and a block of 43690 three-byte matches (131070 bytes, near the 128 KiB limit).  The consumer's short
    shuffle chain ends at 8, the warp scan starts at 9, a batch is 32 and a tiny block at most 32."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(10)
    w = _writer(11, history=1 << 12)
    marks = []
    for n in COUNTS:
        for form in ([None, 2] if n < 128 else [None]):
            seqs = [(0 if i % 3 else 1, 3 + (i % 2), 1 if i % 3 else 2) for i in range(n)]      # repeat offsets, 3-4 bytes
            if n == 43690:
                seqs = [(0, 3, 1)] * n
            w.seq_block(seqs, form=form, tail=0 if n == 43690 else 2)
            marks.append((len(w.blocks) - 1, n, w.sections[-1].header))
    blocks = _decodes(backend, w, "sequence counts")
    for i, n, hdr in marks:
        assert len(blocks[i].seqs) == n
    forms = {(n, len(h)) for _, n, h in marks}
    assert {(127, 1), (128, 2), (0x7EFF, 2), (0x7F00, 3), (1, 2), (127, 2)} <= forms
    assert max(b.regen for b in blocks) == 131070


# ---- 10. the global-memory reader ---------------------------------------------------------------------------------------
N_READ = 6000

@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_readers_agree(backend, monkeypatch, tiny):
    """The same sequences under hand-built tables (-1 symbols in use, accuracy logs 9, 8, 9) through the
    global-memory reader (one block whose bitstream is more than 16 KiB: seq_produce), the staged reader (blocks of 33 and
    more) and the tiny-block reader (blocks of at most 32): the same bytes."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(12)
    ll = F.distribution(9, {s: 1 + s % 4 for s in range(10)} | {22: 1}, low=(19,))
    ml = F.distribution(9, {s: 1 + s % 5 for s in range(13)} | {43: 1}, low=(40,))
    of = F.distribution(8, {s: 1 + s for s in range(11, OF_TOP + 1)}, low=(0,))
    want = []
    pick = [(np.arange(len(t)), np.abs(t) / np.abs(t).sum()) for t in (np.array(ll), np.array(of), np.array(ml))]
    for i in range(N_READ):
        want.append(tuple(int(rng.choice(a, p=p)) for a, p in pick))
    want[1000] = (19, 16, 40)
    base = _writer(13)
    seqs = F.seqs_for(rng, want, len(base.out))
    lits = base.text(sum(s[0] for s in seqs) + 4)
    assert sum(s[0] + s[1] for s in seqs) < Z.BLOCK
    outs = []
    for cut in (N_READ, 33, 32):
        w = _writer(13)
        lp = 0
        for k in range(0, N_READ, cut):
            g = seqs[k:k + cut]
            n = sum(s[0] for s in g) + (4 if k + cut >= N_READ else 0)
            spec = dict(ll=("fse", 9, ll), of=("fse", 8, of), ml=("fse", 9, ml)) if k == 0 else dict(ll=("repeat",), of=("repeat",), ml=("repeat",))
            w.seq_block(g, **spec, lits=lits[lp:lp + n]); lp += n
        blocks = _decodes(backend, w, f"blocks of {cut}")
        if cut == N_READ:
            assert blocks[-1].seq_bytes > 16 * 1024 and any(s[0] == 19 for s in blocks[-1].seqs)
        outs.append(w.frame(check=False)[0])
    assert outs[0] == outs[1] == outs[2]


# ---- 11. the end of the bitstream ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_end_marker(backend, monkeypatch, tiny):
    """The end marker at each bit of the last byte: all three kinds RLE, one sequence whose offset code k has k extra bits
    (k = 0: a one-byte bitstream, the marker alone), and under FSE tables where the last cells choose it."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    rng = np.random.default_rng(13)
    w = _writer(14, history=1 << 12)
    for k in range(8):
        seqs = F.seqs_for(rng, [(5, k, 7)] * (1 if k % 2 else 9), len(w.out))       # 1 + 9k bits: the marker at bit k
        w.seq_block(seqs, ll=("rle", 5), of=("rle", k), ml=("rle", 7), tail=1)
    seen = {}
    tabs = dict(ll=("fse", 6, F.distribution(6, {s: 1 + s for s in range(10)}, low=(4,))),
                of=("fse", 5, F.distribution(5, {s: 1 for s in range(2, 9)})), ml=("fse", 6, F.distribution(6, {s: 1 for s in range(20)})))
    for t in range(64):
        if len(seen) == 8:
            break
        seqs = F.seqs_for(rng, [(int(rng.integers(0, 10)), int(rng.integers(2, 9)), int(rng.integers(0, 20))) for _ in range(int(rng.integers(1, 40)))], len(w.out))
        last = {k: ("wide", "narrow")[(t >> i) & 1] for i, k in enumerate(F.KINDS)}
        sec = w.seq_block(seqs, **tabs, last=last)
        seen.setdefault(sec.marker, len(w.blocks) - 1)
    blocks = _decodes(backend, w, "end marker")
    rle = [s for s in w.sections if s.specs["ll"][0] == "rle"]
    assert [s.marker for s in rle] == list(range(8)) and len(rle[0].bitstream) == 1 and rle[0].bitstream == b"\x01"
    assert sorted(seen) == list(range(8))
    assert blocks[rle[0].index].seq_bytes == 1


# ---- 11-12. refusals ---------------------------------------------------------------------------------------------------
def _refusals():
    """(label, frame, size, libzstd refuses).  Refusals the device makes and libzstd 1.5.5 does not: reserved bits set in
    the modes byte, and a sequence bitstream that does not end exactly on its first bit (one bit left over, or one bit read
    past the start): libzstd 1.5.5 checks neither.  A sum of probabilities above 2^AL cannot be written: the largest value
    a field can hold is what is left to distribute."""
    out = []
    ok_seqs = [(3, 5, 9), (1, 4, 2), (0, 6, 12)]
    tab = ("fse", 6, F.distribution(6, {s: 1 + s % 3 for s in range(16)}))

    good = _writer(20, history=1 << 10)
    good_bits = good.seq_block(ok_seqs).bitstream                  # (predefined tables: the stream of refused tables)

    def add(label, libzstd=True, pre=None, **kw):
        w = _writer(20, history=1 << 10)
        if pre:
            pre(w)
        if "ll" not in kw:
            kw["ll"] = tab
        elif "bitstream" not in kw:
            kw["bitstream"] = good_bits
        w.seq_block(ok_seqs, **kw)
        p, f = w.frame(check=False)
        out.append((label, f, len(p), libzstd))

    for kind in F.KINDS:
        kw = {"ll": ("predefined",), kind: ("fse", F.MAX_AL[kind] + 1, [1 << (F.MAX_AL[kind] + 1)])}
        add(f"{kind} accuracy log {F.MAX_AL[kind] + 1}", **kw)
        add(f"{kind} RLE symbol {F.MAX_SYM[kind] + 1}", **{"ll": ("predefined",), kind: ("rle", F.MAX_SYM[kind] + 1)})
        ms = F.MAX_SYM[kind]
        # probabilities summing to 2^AL - 1 over every symbol: the description runs out of symbols
        short = [1] * ms + [(1 << 6) - ms - 1] if ms < 63 else None
        add(f"{kind} sum one below", **{"ll": ("predefined",), kind: ("fse", 6, short)})
        # a zero run that reaches the symbol after the last one, and one past it
        for over in (0, 1, 4):
            z = ms - 1 + over                     # zeros after symbol 0's count and the zero field of symbol 1
            flags = [3] * (z // 3) + [z % 3]
            d = F.ncount(6, [32, 0], tail_flags=flags)
            add(f"{kind} zero run to {ms + 1 + over}", desc=d, **{"ll": ("predefined",), kind: ("fse", 6, [32, 0])})
    # a description cut off by the end of the block
    d = F.description(6, F.distribution(6, {s: 1 for s in range(30)}))
    add("description cut by the block end", ll=("predefined",), desc=d[:-3], bitstream=b"")
    for r in (1, 2, 3):
        add(f"reserved mode bits {r}", reserved=r, libzstd=False)
    add("repeat mode without an earlier table", ll=("repeat",), bitstream=good_bits, pre=lambda w: setattr(w, "prev", {"ll": (0, [(3, 0, 0)]), "of": None, "ml": None}))
    # the end of the bitstream
    add("last byte 0", tamper=lambda b: b + b"\0")
    add("one bit left over", pad="0", libzstd=False)
    add("one bit missing", drop=1, libzstd=False)
    add("tiny block of 369 bytes", pad="0" * (8 * 369))
    add("no byte after the descriptions", bitstream=b"")
    return out


@pytest.mark.parametrize("backend", BACKENDS)
@READERS
def test_refusals(backend, monkeypatch, tiny):
    """Each corrupt section is refused with a clean NafIoError by the device, by the reader (frame_codes) and, unless noted
    in _refusals, by libzstd; inside a batch the other archives still decode."""
    monkeypatch.setenv("NAFGPU_TINY_BLOCKS", tiny)
    cases = _refusals()
    for label, frame, n, libzstd_refuses in cases:
        if libzstd_refuses:
            with pytest.raises(RuntimeError):
                Z.libzstd_decompress(frame, n)
        with pytest.raises((AssertionError, IndexError, KeyError, TypeError)):
            Z.frame_codes(frame)
        with pytest.raises(N.NafIoError):
            _ctx(backend).zstd_decompress(frame, n)
    arcs, res = _batch(backend, [_as_text_archive(b"0" * n, f) for _, f, n, _ in cases], strict=False)
    for i, (r, a) in enumerate(zip(res, arcs)):
        if i % 2:
            assert r.status != 0, cases[i // 2][0]
        else:
            assert r.status == 0
            assert_same_as_oracle(r, O.decode(a), f"archive {i}")

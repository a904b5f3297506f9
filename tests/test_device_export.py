"""Device-resident export (nafgpu_job_counts / nafgpu_job_export, nafcodec_b200.decode_to_device): every export is compared
with the host path (decode_batch / ArchiveResult) mapped through the same table in numpy.  Under the emulator the "device"
is host memory, so the emul backend uses device="cpu"."""
import ctypes as C

import numpy as np
import pytest

import _cases as K
import _oracle as O
import nafcodec_b200 as N
from nafcodec_b200 import _ffi
from _harness import BACKENDS, library
from conftest import read_golden

torch = pytest.importorskip("torch")

GOLDEN = ["masked.naf", "phix.naf", "CP040672.naf", "LuxC.naf", "NZ_AAEN01000029.naf"]


def device_of(backend):
    return "cuda:0" if backend == "cuda" else "cpu"


@pytest.fixture(scope="module")
def job_files():
    return [read_golden(n) for n in GOLDEN] + [K.multi_record_dna(3, 300, 900, level=3, empty_every=7), K.fastq_reads(5, 1500)]


def host_job(files, lib, **fields):
    """Records of the job in job order as the host path sees them: [(sequence bytes | None, quality bytes | None)]."""
    res = N.decode_batch(files, _library=lib, **fields) if files else []
    recs = []
    for r in res:
        for i in range(r.n_lengths):
            recs.append((r.sequence_bytes(i), r.quality_bytes(i)))
    return res, recs


def mapped(data: bytes, table) -> np.ndarray:
    t = np.frombuffer(N.device._table(table), np.uint8)
    return t[np.frombuffer(data, np.uint8)]


def ref_rows(recs, rows, length, field, table, pad):
    t = np.frombuffer(N.device._table(table), np.uint8)
    out = np.full((len(rows), length), pad, np.uint8)
    for i, (r, s) in enumerate(rows):
        if r < 0 or r >= len(recs) or s < 0:
            continue
        b = recs[r][field]
        if b is None or s >= len(b):
            continue
        piece = np.frombuffer(b[s:s + length], np.uint8)
        out[i, :len(piece)] = t[piece]
    return out


def cpu(x):
    return x.cpu().numpy()


@pytest.mark.parametrize("backend", BACKENDS)
def test_flat_exports_and_offsets_for_every_table(backend, job_files):
    lib = library(backend)
    res, recs = host_job(job_files, lib)
    with N.decode_to_device(job_files, device=device_of(backend), _library=lib) as d:
        lens = [len(s) for s, _ in recs]
        assert d.n_records == len(recs)
        assert d.archive_records == list(np.concatenate([[0], np.cumsum([r.n_lengths for r in res])]))
        assert np.array_equal(cpu(d.offsets), np.concatenate([[0], np.cumsum(lens)]))
        assert np.array_equal(cpu(d.lengths), lens)
        seq = b"".join(r.sequence for r in res)
        qual = b"".join(r.quality or b"" for r in res)          # an archive without qualities contributes none
        custom = np.random.default_rng(1).integers(0, 256, 256).astype(np.uint8)
        for table in [None, "dna5", "iupac", "mask", "phred33", custom, torch.from_numpy(custom.astype(np.int64)), bytes(custom)]:
            assert np.array_equal(cpu(d.sequence(table)), mapped(seq, table)), table if isinstance(table, str) else type(table)
            assert np.array_equal(cpu(d.quality(table)), mapped(qual, table))
        assert np.array_equal(cpu(d.quality()), mapped(qual, "phred33"))


def test_preset_tables():
    t = {k: np.frombuffer(v, np.uint8) for k, v in N.TABLES.items()}
    assert [t["dna5"][c] for c in b"ACGTUacgtuNn-"] == [0, 1, 2, 3, 3, 0, 1, 2, 3, 3, 4, 4, 4]
    assert [t["iupac"][c] for c in b"-TGKCYSBAWRDMHVNtn"] == list(range(16)) + [1, 15]
    assert [t["mask"][c] for c in b"aAzZn-"] == [1, 0, 1, 0, 1, 0]
    assert [t["phred33"][c] for c in b"!+I"] == [0, 10, 40]
    with pytest.raises(ValueError):
        N.device._table("dna4")
    with pytest.raises(ValueError):
        N.device._table(bytes(255))
    with pytest.raises(ValueError):
        N.device._table(np.arange(256) + 1)
    with pytest.raises(TypeError):
        N.device._table(list(range(256)))


@pytest.mark.parametrize("backend", BACKENDS)
def test_ids_and_comments(backend, job_files):
    lib = library(backend)
    res = N.decode_batch(job_files, _library=lib)
    with N.decode_to_device(job_files, id=True, comment=True, device=device_of(backend), _library=lib) as d:
        assert d.ids() == [r.id_bytes(i).decode() for r in res for i in range(r.n_ids)]
        assert d.comments() == [r.comment_bytes(i).decode() for r in res for i in range(r.n_comments)]


@pytest.mark.parametrize("backend", BACKENDS)
def test_rows(backend, job_files):
    lib = library(backend)
    res, recs = host_job(job_files, lib)
    n = len(recs)
    rng = np.random.default_rng(7)
    bounds = np.cumsum([r.n_lengths for r in res])
    with N.decode_to_device(job_files, device=device_of(backend), _library=lib) as d:
        for length in (1, 15, 16, 17, 150, 1000):
            picks = rng.integers(0, n, 300)
            table = [(int(r), int(rng.integers(0, max(len(recs[r][0]), 1)))) for r in picks]      # inside the record, often truncated
            table += [(int(r), max(len(recs[r][0]) - k, 0)) for r in picks[:40] for k in (1, 3)]   # the last residues
            for b in bounds[:-1]:                                                                  # consecutive rows across archives
                table += [(int(b) - 1, 0), (int(b), 0), (int(b) - 1, 5)]
            table += [(int(r), len(recs[r][0]) + k) for r in picks[:20] for k in (0, 1, 100)]      # start at / past the end
            table += [(int(r), -k) for r in picks[:10] for k in (1, 2 ** 40)]                      # negative start
            table += [(-1, 0), (n, 0), (n + 5, 3), (-(2 ** 62), 0), (2 ** 62, 0)]                  # records out of range
            rows = torch.tensor(table, dtype=torch.int64, device=d.device)
            for field, tab, pad in (("sequence", None, 0), ("sequence", "dna5", 9), ("quality", "phred33", 255)):
                got = cpu(d.rows(rows, length, field=field, table=tab, pad=pad))
                want = ref_rows(recs, table, length, 0 if field == "sequence" else 1, tab, pad)
                assert np.array_equal(got, want), (length, field)
        assert d.rows(torch.zeros((0, 2), dtype=torch.int64, device=d.device), 16).shape == (0, 16)
        assert d.rows(rows, 0).shape == (len(table), 0)
        for bad in (rows.to(torch.int32), rows[:, :1], rows.t(), rows.reshape(-1)):
            with pytest.raises(ValueError):
                d.rows(bad, 16)
        with pytest.raises(ValueError):
            d.rows(rows, 16, field="ids")


def ref_windows(lens, length, stride, drop_last):
    rows = []
    for r, L in enumerate(lens):
        s = 0
        while s < L and (not drop_last or s + length <= L):
            rows.append((r, s))
            s += stride
    return rows


@pytest.mark.parametrize("backend", BACKENDS)
def test_windows_and_padded(backend):
    lib = library(backend)
    files = [K.multi_record_dna(11, 60, 400, level=3, empty_every=5), K.fastq_reads(3, 200)]
    _, recs = host_job(files, lib)
    lens = [len(s) for s, _ in recs]
    with N.decode_to_device(files, device=device_of(backend), _library=lib) as d:
        for length in (16, 17, 150):
            for stride in (length // 2, length, length + 7):
                for drop_last in (False, True):
                    tok, rows = d.windows(length, stride, table="dna5", pad=4, drop_last=drop_last)
                    want_rows = ref_windows(lens, length, stride, drop_last)
                    assert cpu(rows).tolist() == [list(x) for x in want_rows], (length, stride, drop_last)
                    assert np.array_equal(cpu(tok), ref_rows(recs, want_rows, length, 0, "dna5", 4))
        tok, rows = d.windows(100)
        assert np.array_equal(cpu(rows), ref_windows(lens, 100, 100, False))
        p = d.padded()
        assert p.shape == (len(recs), max(lens))
        assert np.array_equal(cpu(p), ref_rows(recs, [(r, 0) for r in range(len(recs))], max(lens), 0, None, 0))
        q = d.padded(150, field="quality", pad=255)
        assert np.array_equal(cpu(q), ref_rows(recs, [(r, 0) for r in range(len(recs))], 150, 1, "phred33", 255))


@pytest.mark.parametrize("backend", BACKENDS)
def test_field_skipping_and_refused_exports(backend):
    lib = library(backend)
    files = [K.fastq_reads(5, 300), read_golden("phix.naf")]
    res, recs = host_job(files, lib)
    with N.decode_to_device(files, sequence=False, device=device_of(backend), _library=lib) as d:
        assert np.array_equal(cpu(d.quality(None)), mapped(b"".join(r.quality for r in res), None))
        assert np.array_equal(cpu(d.lengths), [len(q) for _, q in recs])
        for export in (d.sequence, d.ids, d.comments, lambda: d.padded(8)):
            with pytest.raises(N.NafError) as e:
                export()
            assert e.value.status == _ffi.ERR_ARGUMENT
    # the same refusals through Context-level calls
    ctx = N.Context(0, lib)
    spec = _ffi.Export()
    spec.field, spec.layout = _ffi.SEC_SEQUENCE, _ffi.EXPORT_FLAT
    with pytest.raises(N.NafError, match="not been run"):
        ctx.export(spec)
    ctx.prepare([N.parse_archive(f, lib) for f in files], _ffi.WANT_ALL)
    ctx.run()
    counts = ctx.counts()
    total = sum(c.total_residues for c in counts)
    assert [c.status for c in counts] == [0, 0] and total == sum(len(s) for s, _ in recs)
    buf = torch.empty(total, dtype=torch.uint8, device=device_of(backend))
    spec.out, spec.out_bytes = buf.data_ptr(), total - 1
    with pytest.raises(N.NafError, match="out_bytes") as e:
        ctx.export(spec)
    assert e.value.status == _ffi.ERR_ARGUMENT
    spec.layout, spec.field, spec.n_rows, spec.row_length, spec.rows = _ffi.EXPORT_ROWS, _ffi.SEC_ID, 1, 1, buf.data_ptr()
    with pytest.raises(N.NafError, match="ids or comments"):
        ctx.export(spec)
    spec.field, spec.rows = _ffi.SEC_SEQUENCE, None
    with pytest.raises(N.NafError, match="row table"):
        ctx.export(spec)
    spec.layout, spec.field, spec.out_bytes = _ffi.EXPORT_FLAT, _ffi.SEC_SEQUENCE, total
    C.memmove(spec.table, bytes(range(256)), 256)
    ctx.export(spec)
    assert buf.cpu().numpy().tobytes() == b"".join(s for s, _ in recs)
    ctx.close()


@pytest.mark.parametrize("backend", BACKENDS)
def test_empty_job_and_archives_without_records(backend):
    lib = library(backend)
    empty = O.encode(ids=[], sequences=[], level=3)
    with N.decode_to_device([], device=device_of(backend), _library=lib) as d:
        assert d.n_records == 0 and cpu(d.offsets).tolist() == [0] and d.sequence().numel() == 0
        assert d.padded().shape == (0, 0) and d.windows(8)[0].shape == (0, 8)
    files = [empty, read_golden("masked.naf"), empty]
    res, recs = host_job(files, lib)
    with N.decode_to_device(files, id=True, device=device_of(backend), _library=lib) as d:
        assert d.archive_records == [0, 0, res[1].n_lengths, res[1].n_lengths]
        assert cpu(d.sequence()).tobytes() == res[1].sequence
        assert d.ids() == [res[1].id_bytes(i).decode() for i in range(res[1].n_ids)]


@pytest.mark.parametrize("backend", BACKENDS)
def test_a_corrupt_archive_of_the_batch(backend):
    lib = library(backend)
    arcs = [K.genome(700 + i, 20_000 + 777 * i, level=3, records=3) for i in range(3)]
    corrupt = bytearray(arcs[1])
    s2 = O.parse(arcs[1]).sec[4]
    corrupt[s2.offset + 2] = 0xFF                                    # first block header: reserved type / absurd size
    batch = [arcs[0], bytes(corrupt), arcs[2]]
    with pytest.raises(N.NafIoError, match="archive 1"):
        N.decode_to_device(batch, device=device_of(backend), _library=lib)
    good, recs = host_job([arcs[0], arcs[2]], lib)
    with N.decode_to_device(batch, strict=False, device=device_of(backend), _library=lib) as d:
        assert d.status[0] == 0 and d.status[2] == 0 and d.status[1] in (_ffi.ERR_INVALID_DATA, _ffi.ERR_UNEXPECTED_EOF)
        assert d.archive_records == [0, good[0].n_lengths, good[0].n_lengths, good[0].n_lengths + good[1].n_lengths]
        assert cpu(d.sequence()).tobytes() == good[0].sequence + good[1].sequence
        assert np.array_equal(cpu(d.offsets), np.concatenate([[0], np.cumsum([len(s) for s, _ in recs])]))
        rows = torch.tensor([[r, 0] for r in range(len(recs))], dtype=torch.int64, device=d.device)
        assert np.array_equal(cpu(d.rows(rows, 64)), ref_rows(recs, rows.tolist(), 64, 0, None, 0))


@pytest.mark.parametrize("backend", BACKENDS)
def test_bad_utf8_is_raised_at_the_same_record(backend):
    lib = library(backend)
    seqs = [b"MKV", b"protein text", b"bad \xff\xfe text", b"after"]
    data = K.text_archive(seqs, sequence_type=O.PROTEIN)
    host = N.decode_batch([data], _library=lib)[0]
    assert host.first_bad_record == 2
    files = [read_golden("LuxC.naf"), data]
    with pytest.raises(N.NafUnicodeError) as e:
        N.decode_to_device(files, device=device_of(backend), _library=lib)
    assert (e.value.archive, e.value.record) == (1, 2)
    with N.decode_to_device(files, strict=False, device=device_of(backend), _library=lib) as d:
        assert d.first_bad_record == [None, 2] and d.status == [0, 0]
        luxc = N.decode_batch([files[0]], _library=lib)[0]
        assert cpu(d.sequence()).tobytes() == luxc.sequence + host.sequence


@pytest.mark.parametrize("backend", BACKENDS)
def test_two_live_jobs(backend):
    lib = library(backend)
    fa, fb = [K.multi_record_dna(21, 40, 700, level=3)], [read_golden("phix.naf"), K.fastq_reads(9, 100)]
    ra, _ = host_job(fa, lib)
    rb, _ = host_job(fb, lib)
    a = N.decode_to_device(fa, device=device_of(backend), _library=lib)
    b = N.decode_to_device(fb, device=device_of(backend), _library=lib)
    for _ in range(2):
        assert cpu(a.sequence()).tobytes() == ra[0].sequence
        assert cpu(b.sequence()).tobytes() == b"".join(r.sequence for r in rb)
    a.close()
    assert cpu(b.quality(None)).tobytes() == b"".join(r.quality for r in rb)
    with pytest.raises(ValueError, match="closed"):
        a.sequence()
    b.close()


def test_product_library_refuses_a_host_device():
    with pytest.raises(ValueError, match="CUDA"):
        N.decode_to_device(read_golden("phix.naf"), device="cpu")


@pytest.mark.gpu
def test_export_on_a_side_stream_then_the_next_job_at_once():
    """The export waits for the run on the context's stream, and the next prepare + run on the same context waits for the
    export on the caller's stream: a run that overwrote the arena early would change the exported bytes."""
    lib = library("cuda")
    files = [K.genome(31, 3_000_000, level=3)]
    other = [N.parse_archive(K.genome(32, 3_000_000, level=3), lib)]
    want = N.decode_batch(files, _library=lib)[0].sequence
    d = N.decode_to_device(files, quality=False, _library=lib)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                  # holds the export back on the side stream (~0.1 s)
        x = d.sequence("dna5")
        y = d.rows(torch.tensor([[0, 1000]], dtype=torch.int64, device="cuda"), 4096)
    d._ctx.prepare(other, _ffi.WANT_SEQUENCE)              # before anyone synchronises
    d._ctx.run()
    side.synchronize()
    assert np.array_equal(x.cpu().numpy(), mapped(want, "dna5"))
    assert y.cpu().numpy().tobytes() == want[1000:5096]
    d.close()


@pytest.mark.gpu
@pytest.mark.slow
def test_cfg2_batch_and_cfg3_crops():
    """The 256-archive cfg2 batch (8 distinct 5 Mbp archives, cycled, as bench.py builds it) flat, and 10^4 random 1024 bp
    crops of the 250 Mbp cfg3 chromosome, against the host path."""
    lib = library("cuda")
    uniq = [K.cached(f"cfg2_s{s}_n5000000_l19.naf", lambda s=s: K.genome(s, 5_000_000, level=19, mask=True, records=1))[0]
            for s in range(1000, 1008)]
    batch = [uniq[i % 8] for i in range(256)]
    host = [r.sequence for r in N.decode_batch(uniq, quality=False, _library=lib)]
    with N.decode_to_device(batch, quality=False, _library=lib) as d:
        got = d.sequence().cpu().numpy().tobytes()
        assert got == b"".join(host[i % 8] for i in range(256))
    data = K.cached("cfg3_n250000000_s3_l19.naf", lambda: K.cfg3_chromosome(250_000_000, workers=0))[0]
    seq = N.decode_batch([data], quality=False, _library=lib)[0].sequence
    with N.decode_to_device(data, quality=False, _library=lib) as d:
        starts = torch.randint(0, len(seq) - 1024, (10_000,), generator=torch.Generator().manual_seed(3))
        rows = torch.stack([torch.zeros_like(starts), starts], 1).cuda()
        crops = d.rows(rows, 1024, table="dna5").cpu().numpy()
    t = np.frombuffer(N.TABLES["dna5"], np.uint8)
    for k, s in enumerate(starts.tolist()):
        assert np.array_equal(crops[k], t[np.frombuffer(seq[s:s + 1024], np.uint8)]), k

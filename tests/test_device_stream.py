"""Streaming a collection into device memory (nafcodec_b200.stream_to_device, nafgpu_pipeline_submit_device / _wait_counts /
_export): the sub-batches, concatenated, equal decode_to_device of the whole list and the oracle; the cuts, the flow control,
the lifetime of tickets and lanes, strict errors and the C ABI's refusals.  Under the emulator the "device" is host memory, so
the emul backend uses device="cpu"."""
import ctypes as C
import gc
import threading
import weakref

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
FIELDS = dict(id=True, comment=True, sequence=True, quality=True, mask=True)


def device_of(backend):
    return "cuda:0" if backend == "cuda" else "cpu"


def cpu(x):
    return x.cpu().numpy()


@pytest.fixture(scope="module")
def files():
    return [read_golden(n) for n in GOLDEN] + [K.multi_record_dna(3 + i, 4 + 3 * i, 700, level=3, empty_every=5) for i in range(3)] + \
        [K.fastq_reads(5, 40), K.fastq_reads(6, 7, read_len=90)]


def expected_cuts(sizes, batch_bytes, max_archives=65535):
    """(first, count) of every sub-batch by the rule stream_to_device documents."""
    cuts, first, size = [], 0, 0
    for i, s in enumerate(sizes):
        if i > first and (size + s > batch_bytes or i - first == max_archives):
            cuts.append((first, i - first))
            first, size = i, 0
        size += s
    if sizes:
        cuts.append((first, len(sizes) - first))
    return cuts


def concat(stream):
    """Every export the parity test compares, concatenated over the sub-batches (offsets made global), and the cuts."""
    out = {k: [] for k in ("seq", "dna5", "qual", "ids", "comments", "offsets")}
    cuts, base = [], 0
    for r in stream:
        cuts.append((r.first_archive, len(r.status)))
        out["seq"].append(cpu(r.sequence()).tobytes())
        out["dna5"].append(cpu(r.sequence("dna5")))
        out["qual"].append(cpu(r.quality()))
        out["ids"] += r.ids()
        out["comments"] += r.comments()
        off = cpu(r.offsets)
        out["offsets"].append(off[:-1] + base)
        base += int(off[-1])
        r.close()
    out["offsets"].append(np.array([base]))
    return {"seq": b"".join(out["seq"]), "dna5": np.concatenate(out["dna5"]), "qual": np.concatenate(out["qual"]),
            "ids": out["ids"], "comments": out["comments"], "offsets": np.concatenate(out["offsets"])}, cuts


@pytest.mark.parametrize("backend", BACKENDS)
def test_sub_batches_equal_the_whole_job_and_the_oracle(backend, files, monkeypatch):
    lib = library(backend)
    dev = device_of(backend)
    with N.decode_to_device(files, device=dev, _library=lib, **FIELDS) as w:
        whole = {"seq": cpu(w.sequence()).tobytes(), "dna5": cpu(w.sequence("dna5")), "qual": cpu(w.quality()), "ids": w.ids(),
                 "comments": w.comments(), "offsets": cpu(w.offsets)}
    oracle = [O.decode(f) for f in files]
    assert whole["seq"] == b"".join(d.sequence or b"" for d in oracle)
    assert whole["ids"] == [d.id(i).decode() for d in oracle for i in range(d.n) if d.id_present[i]]
    sizes = [len(f) for f in files]
    runs = [(k, 1 << 40) for k in (1, 2, 3)]                                           # cut by the archive count
    runs += [(65535, b) for b in (int(np.median(sizes) * 1.5), max(sizes) // 3, 1)]    # cut by bytes
    for k, batch_bytes in runs:
        monkeypatch.setattr(N.device, "_MAX_SUB_BATCH", k)
        cuts_want = expected_cuts(sizes, batch_bytes, k)
        for lanes in (1, 2, 3):
            got, cuts = concat(N.stream_to_device(files, batch_bytes=batch_bytes, lanes=lanes, device=dev, _library=lib, **FIELDS))
            assert cuts == cuts_want, (k, batch_bytes)
            label = (k, batch_bytes, lanes)
            assert got["seq"] == whole["seq"] and got["ids"] == whole["ids"] and got["comments"] == whole["comments"], label
            for key in ("dna5", "qual", "offsets"):
                assert np.array_equal(got[key], whole[key]), (key,) + label
    assert len({n for _, n in expected_cuts(sizes, int(np.median(sizes) * 1.5))}) > 1          # uneven sub-batches


@pytest.mark.parametrize("backend", BACKENDS)
def test_cuts_oversized_archives_and_lazy_input(backend, files):
    lib = library(backend)
    big = read_golden("NZ_AAEN01000029.naf")
    small = [K.multi_record_dna(40 + i, 3, 200, level=3) for i in range(5)]
    seq = [small[0], small[1], big, small[2], small[3], big, big, small[4]]
    batch_bytes = sum(len(s) for s in small[:3])
    assert len(big) > batch_bytes
    got = []
    for r in N.stream_to_device(seq, batch_bytes=batch_bytes, device=device_of(backend), _library=lib):
        got.append((r.first_archive, len(r.status)))
        r.close()
    assert got == [(0, 2), (2, 1), (3, 2), (5, 1), (6, 1), (7, 1)] == expected_cuts([len(s) for s in seq], batch_bytes)

    consumed = []

    def counting():
        for i, f in enumerate(files):
            consumed.append(i)
            yield f
    lanes = 2
    s = N.stream_to_device(counting(), batch_bytes=1, lanes=lanes, device=device_of(backend), _library=lib)
    assert consumed == []                           # nothing is read before the first next()
    for k in range(len(files)):
        r = next(s)
        assert r.first_archive == k
        assert len(consumed) <= k + lanes + 1       # the sub-batches in flight, and one archive to know where the last one ends
        r.close()
    with pytest.raises(StopIteration):
        next(s)
    assert len(consumed) == len(files)


@pytest.mark.parametrize("backend", BACKENDS)
def test_lanes_are_handed_back_and_early_exits_leave_nothing_behind(backend, files, monkeypatch):
    lib = library(backend)
    dev = device_of(backend)
    want = [cpu(N.decode_to_device(f, device=dev, _library=lib).sequence()).tobytes() for f in files[:4]]
    submitted, released = [], []
    submit, release = N.Pipeline.submit_device, N.Pipeline.release

    def spy_submit(self, *a):
        t = submit(self, *a)
        submitted.append(t[0])
        return t

    def spy_release(self, ticket):
        released.append(ticket)
        return release(self, ticket)
    monkeypatch.setattr(N.Pipeline, "submit_device", spy_submit)
    monkeypatch.setattr(N.Pipeline, "release", spy_release)
    threads = threading.active_count()

    # holding `lanes` DeviceRecords open: the next one raises (and does not wait), and the stream goes on after a close
    s = N.stream_to_device(files[:4], batch_bytes=1, lanes=2, device=dev, _library=lib)
    a, b = next(s), next(s)
    x = a.sequence()
    with pytest.raises(RuntimeError, match="close a DeviceRecords before asking for more than lanes=2"):
        next(s)
    a.close()
    assert np.array_equal(cpu(x), np.frombuffer(want[0], np.uint8))     # exported before close: still valid
    with pytest.raises(ValueError, match="closed"):
        a.sequence()
    c = next(s)
    assert (b.first_archive, c.first_archive) == (1, 2)
    assert cpu(c.sequence()).tobytes() == want[2]
    pipe = weakref.ref(s._pipe)
    s.close()                                       # c and b were open: closed with the stream, their tickets released
    assert not b._finalizer.alive and not c._finalizer.alive and not pipe()._p
    assert sorted(released) == sorted(submitted)

    # an early break, then the stream is collected
    submitted.clear(), released.clear()
    for r in N.stream_to_device(files, batch_bytes=1, lanes=3, device=dev, _library=lib):
        pipe = weakref.ref(r._ctx.pipe)
        if r.first_archive == 1:
            break
        r.close()
    del r
    gc.collect()
    assert pipe() is None or not pipe()._p
    assert len(submitted) == 4 and sorted(released) == sorted(submitted)

    # an exception in the loop body: the generator-like cleanup runs when the stream goes
    submitted.clear(), released.clear()
    with pytest.raises(KeyError):
        with N.stream_to_device(files, batch_bytes=1, lanes=2, device=dev, _library=lib) as s:
            for r in s:
                raise KeyError("consumer")
    assert not s._pipe._p and sorted(released) == sorted(submitted) and len(submitted) == 2
    assert threading.active_count() == threads


def corrupt(data: bytes) -> bytes:
    bad = bytearray(data)
    bad[O.parse(data).sec[4].offset + 2] = 0xFF             # first block header: reserved type / absurd size
    return bytes(bad)


@pytest.mark.parametrize("backend", BACKENDS)
def test_a_corrupt_archive_in_the_middle_sub_batch(backend):
    lib = library(backend)
    dev = device_of(backend)
    arcs = [K.genome(700 + i, 20_000 + 777 * i, level=3, records=3) for i in range(5)]
    batch = arcs[:3] + [corrupt(arcs[3])] + arcs[4:]
    batch_bytes = len(arcs[2]) + len(arcs[3]) + 10
    assert expected_cuts([len(a) for a in batch], batch_bytes) == [(0, 2), (2, 2), (4, 1)]
    host = [r.sequence for r in N.decode_batch(arcs, quality=False, _library=lib)]
    s = N.stream_to_device(batch, batch_bytes=batch_bytes, device=dev, _library=lib)
    r = next(s)
    assert cpu(r.sequence()).tobytes() == host[0] + host[1]
    r.close()
    with pytest.raises(N.NafIoError, match=r"archive 3 of the input") as e:
        next(s)
    assert e.value.status in (_ffi.ERR_INVALID_DATA, _ffi.ERR_UNEXPECTED_EOF)
    with pytest.raises(StopIteration):              # an error ends the stream
        next(s)
    assert not s._pipe._p

    got = []
    for r in N.stream_to_device(batch, batch_bytes=batch_bytes, strict=False, device=dev, _library=lib):
        got.append((r.first_archive, r.status, cpu(r.sequence()).tobytes()))
        r.close()
    assert [(f, st[0] == 0, len(st)) for f, st, _ in got] == [(0, True, 2), (2, True, 2), (4, True, 1)]
    assert got[1][1][1] in (_ffi.ERR_INVALID_DATA, _ffi.ERR_UNEXPECTED_EOF)
    assert [x for _, _, x in got] == [host[0] + host[1], host[2], host[4]]

    # an input that is not an archive: the sub-batches before it are yielded, then it raises naming its index
    s = N.stream_to_device(arcs[:2] + [b"not an archive"] + arcs[2:], batch_bytes=1, device=dev, _library=lib)
    assert [next(s).first_archive, next(s).first_archive] == [0, 1]
    with pytest.raises(N.NafParseError, match="archive 2 of the input"):
        next(s)


@pytest.mark.parametrize("backend", BACKENDS)
def test_bad_utf8_is_raised_at_the_same_record(backend):
    lib = library(backend)
    dev = device_of(backend)
    data = K.text_archive([b"MKV", b"protein text", b"bad \xff\xfe text", b"after"], sequence_type=O.PROTEIN)
    files = [read_golden("LuxC.naf"), read_golden("masked.naf"), read_golden("LuxC.naf"), data]
    with pytest.raises(N.NafUnicodeError) as whole:
        N.decode_to_device(files, device=dev, _library=lib)
    s = N.stream_to_device(files, batch_bytes=len(files[0]) + len(files[1]), device=dev, _library=lib)
    r = next(s)
    assert r.first_archive == 0
    r.close()
    with pytest.raises(N.NafUnicodeError) as e:
        next(s)
    assert (e.value.archive, e.value.record) == (whole.value.archive, whole.value.record) == (3, 2)
    seen = []
    for r in N.stream_to_device(files, batch_bytes=1, strict=False, device=dev, _library=lib):
        seen.append((r.first_archive, r.first_bad_record, r.status))
        r.close()
    assert seen == [(0, [None], [0]), (1, [None], [0]), (2, [None], [0]), (3, [2], [0])]


@pytest.mark.parametrize("backend", BACKENDS)
def test_c_abi_refusals_and_host_tickets_between_device_tickets(backend, files):
    lib = library(backend)
    dll = lib.dll
    archives = [N.parse_archive(f, lib) for f in files[:4]]
    host = N.decode_batch(files[:4], _library=lib)
    p = N.Pipeline(0, 2, lib)

    def refused(rc, match):
        assert rc == _ffi.ERR_ARGUMENT
        assert match in dll.nafgpu_pipeline_last_error(p._p).decode()

    spec = _ffi.Export()
    spec.field, spec.layout = _ffi.SEC_SEQUENCE, _ffi.EXPORT_FLAT
    C.memmove(spec.table, bytes(range(256)), 256)
    part_a, part_b = archives[:2], archives[2:]
    td, arr_d = p.submit_device(part_a, _ffi.WANT_ALL)                       # device, host, device, host in one queue
    th, arr_h, _ = p._submit(part_b, _ffi.WANT_ALL)
    refused(dll.nafgpu_pipeline_export(p._p, td, C.byref(spec), None), "not waited for")
    refused(dll.nafgpu_pipeline_wait(p._p, td, (_ffi.Result * 2)(), 2), "device ticket")
    refused(dll.nafgpu_pipeline_wait_counts(p._p, th, (_ffi.Counts * 2)(), 2), "host ticket")
    refused(dll.nafgpu_pipeline_export(p._p, th, C.byref(spec), None), "host ticket")
    counts = p.wait_counts(td, 2)
    assert [c.total_residues for c in counts] == [h.total_residues for h in host[:2]]
    out = torch.empty(sum(c.total_residues for c in counts), dtype=torch.uint8, device=device_of(backend))
    spec.out, spec.out_bytes = out.data_ptr(), out.numel()
    p.export(td, spec)
    if backend == "cuda":
        torch.cuda.synchronize()
    assert cpu(out).tobytes() == host[0].sequence + host[1].sequence
    spec.out_bytes = out.numel() - 1                                          # a refusal of nafgpu_job_export, passed on
    with pytest.raises(N.NafArgumentError, match="out_bytes"):
        p.export(td, spec)
    spec.out_bytes = out.numel()
    p.release(td)
    refused(dll.nafgpu_pipeline_export(p._p, td, C.byref(spec), None), "released")
    res = (_ffi.Result * 2)()
    assert dll.nafgpu_pipeline_wait(p._p, th, res, 2) == 0
    assert [C.string_at(res[i].sequence, res[i].total_residues) for i in range(2)] == [h.sequence for h in host[2:]]
    td2, arr_d2 = p.submit_device(part_b, _ffi.WANT_SEQUENCE)
    p.release(th)
    counts = p.wait_counts(td2, 2)
    out = torch.empty(sum(c.total_residues for c in counts), dtype=torch.uint8, device=device_of(backend))
    spec.out, spec.out_bytes = out.data_ptr(), out.numel()
    spec.field = _ffi.SEC_QUALITY
    with pytest.raises(N.NafArgumentError, match="not decoded"):              # want bits of the ticket
        p.export(td2, spec)
    spec.field = _ffi.SEC_SEQUENCE
    p.export(td2, spec)
    if backend == "cuda":
        torch.cuda.synchronize()
    assert cpu(out).tobytes() == host[2].sequence + host[3].sequence
    p.release(td2)
    refused(dll.nafgpu_pipeline_wait_counts(p._p, td2, (_ffi.Counts * 2)(), 2), "unknown ticket")
    p.close()


@pytest.mark.gpu
def test_export_on_a_side_stream_then_the_next_ticket_at_once():
    """Ticket k's export is held back on a side stream, ticket k is released at once and its lane decodes ticket k + lanes
    while the export waits: the lane's prepare waits for the export, so the bytes are ticket k's."""
    lib = library("cuda")
    files = [K.genome(31, 3_000_000, level=3), K.genome(32, 3_000_000, level=3)]
    want = [r.sequence for r in N.decode_batch(files, quality=False, _library=lib)]
    s = N.stream_to_device(files, batch_bytes=1, lanes=1, quality=False, _library=lib)
    r = next(s)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                  # holds the export back on the side stream (~0.1 s)
        x = r.sequence("dna5")
        y = r.rows(torch.tensor([[0, 1000]], dtype=torch.int64, device="cuda"), 4096)
    r.close()                                           # the lane takes ticket 1 before anyone synchronises
    r1 = next(s)
    side.synchronize()
    t = np.frombuffer(N.TABLES["dna5"], np.uint8)
    assert np.array_equal(x.cpu().numpy(), t[np.frombuffer(want[0], np.uint8)])
    assert y.cpu().numpy().tobytes() == want[0][1000:5096]
    assert r1.sequence().cpu().numpy().tobytes() == want[1]
    r1.close()
    s.close()


@pytest.mark.gpu
@pytest.mark.slow
def test_cfg5_shaped_collection():
    """300 archives of the RefSeq-collection shape (24 unique 2-6 Mbp level-19 genomes, cycled) in 64 MB sub-batches on two
    lanes, against the host path."""
    from concurrent.futures import ThreadPoolExecutor
    import os
    lib = library("cuda")
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        uniq = list(ex.map(lambda i: K.cached(f"cfg5_i{i}_l19.naf", lambda: K.cfg5_member(i))[0], range(24)))
    host = [r.sequence for r in N.decode_batch(uniq, quality=False, _library=lib)]
    batch = [uniq[i % 24] for i in range(300)]
    n = 0
    for r in N.stream_to_device(batch, batch_bytes=64 << 20, lanes=2, quality=False, _library=lib):
        k = len(r.status)
        assert r.first_archive == n and r.status == [0] * k
        assert r.sequence().cpu().numpy().tobytes() == b"".join(host[(n + a) % 24] for a in range(k))
        n += k
        r.close()
    assert n == 300

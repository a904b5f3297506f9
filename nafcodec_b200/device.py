"""Decode into CUDA tensors: the decoded job stays in device memory and is handed to PyTorch where it already sits.

`decode_to_device` decodes one archive or a list of them as one job and returns a `DeviceRecords`.  Every export from it
(nafgpu_job_export, include/nafgpu.h) runs sm_100a kernels that write into a tensor allocated with `torch.empty` on the
current torch stream of the device, through a 256-entry byte table: the ASCII itself, or tokens (`TABLES`).  Records are
numbered across the job: archive 0's records first, then archive 1's; an archive that failed contributes none.

    recs = decode_to_device(files)                  # sequence + quality, one job
    tokens = recs.sequence(table="dna5")            # uint8 [total residues]
    x, rows = recs.windows(1024, stride=512, table="dna5")

The job stays in HBM while `recs` lives, so any number of exports can be taken from one decode.  `recs` owns a context for
that time; closing or collecting it returns the context to a small per-device pool, so batch after batch allocates device
memory once.

`stream_to_device` does the same for a collection of any size: it cuts the input into sub-batches and decodes them on the
lanes of a pipeline (nafgpu_pipeline_submit_device), so that the header walk and H2D of one sub-batch overlap the kernels of
another, and yields one `DeviceRecords` per sub-batch, backed by its pipeline ticket instead of a pooled context.

    for recs in stream_to_device(files, batch_bytes=256 << 20, lanes=2):
        x, rows = recs.windows(1024, table="dna5")
        recs.close()                                # hands the lane back
"""
import ctypes as C
import threading
import weakref
from collections import deque
from typing import List, Optional

import numpy as np

from . import _ffi
from .decoder import Context, Pipeline, _read_all, _want_bits, parse_archive
from .errors import NafError, NafUnicodeError, raise_for_status


def _presets():
    b = np.arange(256)
    dna5 = np.full(256, 4, np.uint8)                     # A C G T/U -> 0..3 in either case, anything else -> 4
    for code, ch in enumerate(b"ACGT"):
        dna5[ch] = dna5[ch + 32] = code
    dna5[ord("U")] = dna5[ord("u")] = 3
    iupac = np.full(256, 15, np.uint8)                   # the NAF 4-bit code (read_nucleotide's "-TGKCYSBAWRDMHVN"), case folded; else N
    for code, ch in enumerate(b"-TGKCYSBAWRDMHVN"):
        iupac[ch] = code
        if ch != ord("-"):
            iupac[ch + 32] = code
    iupac[ord("U")] = iupac[ord("u")] = 1
    mask = ((b >= ord("a")) & (b <= ord("z"))).astype(np.uint8)     # soft-masked (lower case) -> 1
    phred33 = ((b - 33) & 0xFF).astype(np.uint8)                        # quality score (b - 33, modulo 256)
    return {"dna5": dna5.tobytes(), "iupac": iupac.tobytes(), "mask": mask.tobytes(), "phred33": phred33.tobytes()}


TABLES = _presets()
_IDENTITY = bytes(range(256))
_DEFAULT = object()           # table default: identity for the sequence, "phred33" for the quality
_FIELDS = {"sequence": _ffi.SEC_SEQUENCE, "quality": _ffi.SEC_QUALITY}


def _table(t) -> bytes:
    """None (identity), a preset name, or any 256-entry bytes / numpy / torch table of values in [0, 255]."""
    if t is None:
        return _IDENTITY
    if isinstance(t, str):
        if t not in TABLES:
            raise ValueError(f"unknown table {t!r}: one of {sorted(TABLES)}, or 256 bytes")
        return TABLES[t]
    if isinstance(t, (bytes, bytearray)):
        a = np.frombuffer(bytes(t), np.uint8)
    elif isinstance(t, np.ndarray):
        a = t
    elif type(t).__module__.startswith("torch"):
        a = t.detach().cpu().numpy()
    else:
        raise TypeError(f"table must be None, a preset name, bytes, a numpy array or a torch tensor, not {type(t).__name__}")
    if a.size != 256 or a.dtype.kind not in "ui" or (a.size and (a.min() < 0 or a.max() > 255)):
        raise ValueError("a table has 256 integer entries in [0, 255]")
    return a.astype(np.uint8).reshape(256).tobytes()


# ---- context pool (as detail::ContextPool in include/nafgpu.hpp): contexts keep their device buffers between jobs -------------
_POOL_MAX = 4
_pool = {}
_pool_lock = threading.Lock()


def _take(lib, index) -> Context:
    with _pool_lock:
        idle = _pool.get((lib.path, index))
        if idle:
            return idle.pop()
    return Context(index, lib)


def _give(key, ctx):
    with _pool_lock:
        idle = _pool.setdefault(key, [])
        if len(idle) < _POOL_MAX:
            idle.append(ctx)
            return
    ctx.close()


def _resolve_device(device, lib):
    import torch
    dev = torch.device(device)
    if lib.path == _ffi.LIB_PATH:
        if dev.type != "cuda":
            raise ValueError(f"decode_to_device writes CUDA tensors: {dev} is not a CUDA device")
        index = dev.index if dev.index is not None else torch.cuda.current_device()
        return torch.device("cuda", index), index
    if dev.type != "cpu":              # a library built for tests (the SIMT emulator): its "device memory" is host memory
        raise ValueError(f"{lib.path} writes host memory: use device='cpu'")
    return dev, 0


class _Ticket:
    """A device ticket of a pipeline, as what backs a DeviceRecords: its exports run on the ticket's lane."""

    def __init__(self, pipe: Pipeline, ticket: int):
        self.pipe, self.ticket = pipe, ticket

    def export(self, spec, stream=0):
        self.pipe.export(self.ticket, spec, stream)


class DeviceRecords:
    """A decoded job kept in device memory; every method returns torch tensors on `device` (see the module docstring).
    `first_archive` is the input index of the job's archive 0 (nonzero for the sub-batches of stream_to_device)."""

    def __init__(self, ctx, archives, want: int, device, counts, release=None, first_archive: int = 0):
        self.device = device
        self._ctx = ctx                 # what holds the decoded job: a pooled Context, or a pipeline ticket (_Ticket)
        self._want = want
        self.first_archive = first_archive
        self._finalizer = weakref.finalize(self, *(release or (_give, (ctx.lib.path, ctx.device), ctx)))
        self._counts = counts
        self.status = [c.status for c in counts]
        self.first_bad_record = [None if c.first_bad_record == _ffi.NO_RECORD else int(c.first_bad_record) for c in counts]
        arch = np.zeros(len(counts) + 1, np.int64)
        arch[1:] = np.cumsum([c.n_lengths for c in counts])
        self.archive_records = arch.tolist()            # job records of archive a: [archive_records[a], archive_records[a + 1])
        self.n_records = self.archive_records[-1]
        # residues per archive in a flat export of the sequence / quality: an archive without that section contributes none
        self._has = {f: [bool(a.sections[f].present and a.sections[_ffi.SEC_LENGTH].present) for a in archives]
                     for f in (_ffi.SEC_SEQUENCE, _ffi.SEC_QUALITY)}
        self.offsets = self._export(_ffi.EXPORT_OFFSETS, 0, (self.n_records + 1,), "int64")
        self._lengths = None

    # -- life time -----------------------------------------------------------------------------------------------------------
    def close(self):
        """Returns the context to the pool, or the ticket to its pipeline, and with it the decoded job; tensors already exported
        stay valid."""
        self._finalizer()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    @property
    def lengths(self):
        if self._lengths is None:
            self._lengths = self.offsets.diff()
        return self._lengths

    # -- exports -------------------------------------------------------------------------------------------------------------
    def _export(self, layout, field, shape, dtype, table=None, pad=0, rows=None, row_length=0):
        import torch
        if not self._finalizer.alive:
            raise ValueError("DeviceRecords is closed")
        out = torch.empty(shape, dtype=getattr(torch, dtype), device=self.device)
        spec = _ffi.Export()
        spec.field, spec.layout = field, layout
        C.memmove(spec.table, _table(table), 256)
        spec.pad = pad
        spec.out, spec.out_bytes = out.data_ptr() or None, out.numel() * out.element_size()
        if rows is not None:
            spec.rows, spec.n_rows, spec.row_length = rows.data_ptr() or None, rows.shape[0], row_length
        stream = 0
        if self.device.type == "cuda":
            # 0 is torch's legacy default stream, where the C ABI reads NULL as the context's own stream: cudaStreamLegacy (1)
            stream = torch.cuda.current_stream(self.device).cuda_stream or 1
        self._ctx.export(spec, stream)
        return out

    def _flat(self, field, table):
        n = sum(c.total_residues for c, has in zip(self._counts, self._has[field]) if has)
        return self._export(_ffi.EXPORT_FLAT, field, (n,), "uint8", table)

    def sequence(self, table=None):
        """uint8 [residues]: the sequences of all records, concatenated in job order, through `table` (None: the ASCII)."""
        return self._flat(_ffi.SEC_SEQUENCE, table)

    def quality(self, table="phred33"):
        """uint8 [residues]: the qualities of all records, concatenated in job order, through `table` (default: scores)."""
        return self._flat(_ffi.SEC_QUALITY, table)

    def rows(self, rows, length: int, field: str = "sequence", table=_DEFAULT, pad: int = 0):
        """uint8 [m, length]: row i holds residues [start, start + length) of job record `record`, (record, start) = rows[i],
        `pad` past the record's end.  A row whose record is out of range, or whose start is negative or not below the record's
        length, is all `pad`.  `rows`: a contiguous int64 [m, 2] tensor on this device."""
        import torch
        if field not in _FIELDS:
            raise ValueError(f"field must be one of {sorted(_FIELDS)}, not {field!r}")
        if not isinstance(rows, torch.Tensor) or rows.dtype != torch.int64 or rows.dim() != 2 or rows.shape[1] != 2:
            raise ValueError("rows must be an int64 tensor of shape [m, 2] (record, start)")
        if not rows.is_contiguous() or rows.device != self.device:
            raise ValueError(f"rows must be contiguous and on {self.device}")
        length = int(length)
        if length < 0 or not 0 <= int(pad) <= 255:
            raise ValueError("length must be >= 0 and pad in [0, 255]")
        if table is _DEFAULT:
            table = "phred33" if field == "quality" else None
        return self._export(_ffi.EXPORT_ROWS, _FIELDS[field], (rows.shape[0], length), "uint8", table, int(pad), rows, length)

    def padded(self, length: Optional[int] = None, field: str = "sequence", table=_DEFAULT, pad: int = 0):
        """uint8 [N, length]: every record from its first residue, cut or padded to `length` (None: the longest record)."""
        import torch
        if length is None:
            length = int(self.lengths.max()) if self.n_records else 0
        rec = torch.arange(self.n_records, dtype=torch.int64, device=self.device)
        rows = torch.stack([rec, torch.zeros_like(rec)], 1)
        return self.rows(rows, length, field, table, pad)

    def windows(self, length: int, stride: Optional[int] = None, field: str = "sequence", table=_DEFAULT, pad: int = 0,
                drop_last: bool = False):
        """(tokens [m, length], rows [m, 2]): windows of every record starting at 0, stride, 2 * stride, ... (stride defaults
        to length).  A window starts inside its record and is padded past its end; with drop_last only whole windows are kept."""
        import torch
        length = int(length)
        stride = length if stride is None else int(stride)
        if length <= 0 or stride <= 0:
            raise ValueError("length and stride must be positive")
        lens = self.lengths
        if drop_last:
            n = torch.where(lens >= length, (lens - length) // stride + 1, torch.zeros_like(lens))
        else:
            n = (lens + stride - 1) // stride
        total = int(n.sum()) if self.n_records else 0
        rec = torch.repeat_interleave(torch.arange(self.n_records, dtype=torch.int64, device=self.device), n, output_size=total)
        first = torch.cumsum(n, 0) - n
        k = torch.arange(total, dtype=torch.int64, device=self.device) - first[rec]
        rows = torch.stack([rec, k * stride], 1).contiguous()
        return self.rows(rows, length, field, table, pad), rows

    def _strings(self, field, size_of, count_of) -> List[str]:
        blob = self._export(_ffi.EXPORT_FLAT, field, (sum(size_of(c) for c in self._counts),), "uint8").cpu().numpy().tobytes()
        out, at = [], 0
        for c in self._counts:
            part = blob[at:at + size_of(c)]
            at += size_of(c)
            try:
                out += [s.decode("utf-8") for s in part.split(b"\0")[:count_of(c)]]
            except UnicodeDecodeError as e:
                raise NafUnicodeError("failed to decode UTF-8 data") from e
        return out

    def ids(self) -> List[str]:
        """The ids of every archive, in job order (an archive contributes its n_ids ids)."""
        return self._strings(_ffi.SEC_ID, lambda c: c.id_bytes, lambda c: c.n_ids)

    def comments(self) -> List[str]:
        """The comments of every archive, in job order (an archive contributes its n_comments comments)."""
        return self._strings(_ffi.SEC_COMMENT, lambda c: c.comment_bytes, lambda c: c.n_comments)


def decode_to_device(files, *, id: bool = False, comment: bool = False, sequence: bool = True, quality: bool = True,
                     mask: bool = True, device="cuda:0", strict: bool = True, _library=None) -> DeviceRecords:
    """Decodes one archive (bytes, path or file object) or a list of them as one job and keeps the result in device memory.
    strict=True raises as Context.decode does for a corrupt archive, and NafUnicodeError for text that is not UTF-8; with
    strict=False such an archive carries its `status` / `first_bad_record` and a failed one contributes no records."""
    lib = _library or _ffi.default_library()
    dev, index = _resolve_device(device, lib)
    datas = [_read_all(f) for f in (files if isinstance(files, (list, tuple)) else [files])]
    archives = [parse_archive(d, lib) for d in datas]
    want = _want_bits(id, comment, sequence, quality, mask)
    ctx = _take(lib, index)
    try:
        ctx.prepare(archives, want)
        ctx.run()
        counts = ctx.counts()           # (the compressed bytes of `archives` have crossed to the device after this)
    except BaseException:
        _give((lib.path, index), ctx)
        raise
    recs = DeviceRecords(ctx, archives, want, dev, counts)
    if strict:
        n = len(counts)
        try:
            _raise_for_counts(lib, counts, 0, lambda i: f"archive {i} of {n}" if n > 1 else "")
        except BaseException:
            recs.close()
            raise
    return recs


# ---- streaming a collection through the pipeline's device tickets ------------------------------------------------------------
_MAX_SUB_BATCH = 65535            # archives of one job (nafgpu_decode_batch)


def _sub_batches(files, batch_bytes, lib):
    """(first input index, [archive], exception) for contiguous runs of `files`, read one archive ahead of the sub-batch being
    cut.  A sub-batch ends where the next archive would take it past batch_bytes of compressed input, or at 65535 archives; an
    input that cannot be read or parsed ends the runs with (its index, [], the exception)."""
    part, first, size = [], 0, 0
    for i, f in enumerate(files):
        try:
            data = _read_all(f)
            a = parse_archive(data, lib)
        except Exception as e:
            if part:
                yield first, part, None
            yield i, [], e
            return
        if part and (size + len(data) > batch_bytes or len(part) == _MAX_SUB_BATCH):
            yield first, part, None
            part, first, size = [], i, 0
        part.append(a)
        size += len(data)
    if part:
        yield first, part, None


def _shutdown(pipe, inflight, yielded):
    """Ends a stream: every ticket in flight is waited for and released, every yielded DeviceRecords still open is closed, and
    the pipeline (its lane threads and contexts) is destroyed."""
    try:
        for _, part, ticket, _ in inflight:
            if part is None:
                continue
            try:
                pipe.wait_counts(ticket, len(part))
            except Exception:
                pass                    # (a failed sub-batch is released all the same)
            pipe.release(ticket)
        inflight.clear()
        for ref in yielded:
            r = ref()
            if r is not None:
                r.close()
        yielded.clear()
    finally:
        pipe.close()


class DeviceStream:
    """The iterator stream_to_device returns (see there).  close() ends it early; so do an exception and garbage collection."""

    def __init__(self, files, batch_bytes, lanes, device, want, strict, lib):
        self.lanes = lanes
        self._lib, self._want, self._strict = lib, want, strict
        self._device, index = _resolve_device(device, lib)
        self._pieces = _sub_batches(files, batch_bytes, lib)
        self._pending = None            # a sub-batch read but not submitted (all lanes were held)
        self._exhausted = False
        self._pipe = Pipeline(index, lanes, lib)
        self._inflight = deque()        # (first, [archive], ticket, archive array) submitted; (first, None, None, exception)
        self._yielded = []              # weak references to the DeviceRecords yielded (open until closed or collected)
        self._finalizer = weakref.finalize(self, _shutdown, self._pipe, self._inflight, self._yielded)

    def __iter__(self):
        return self

    def close(self):
        self._finalizer()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    def _open(self):
        self._yielded[:] = [r for r in self._yielded if r() is not None and r()._finalizer.alive]
        return len(self._yielded) + sum(1 for e in self._inflight if e[1] is not None)

    def _fill(self):
        """Submits sub-batches while fewer than `lanes` tickets are in flight or yielded and open."""
        while not self._exhausted:
            if self._pending is None:
                if self._inflight and self._open() >= self.lanes:
                    return              # (with nothing in flight, one sub-batch is read to tell the input's end from held lanes)
                self._pending = next(self._pieces, None)
                if self._pending is None:
                    self._exhausted = True
                    return
            first, part, err = self._pending
            if err is not None:
                self._inflight.append((first, None, None, err))
                self._pending = None
                continue
            if self._open() >= self.lanes:
                return
            ticket, arr = self._pipe.submit_device(part, self._want)
            self._inflight.append((first, part, ticket, arr))
            self._pending = None

    def __next__(self) -> DeviceRecords:
        if not self._finalizer.alive:
            raise StopIteration
        try:
            self._fill()
            if not self._inflight:
                if self._exhausted:
                    raise StopIteration
                raise _AllLanesHeld(f"{self.lanes} DeviceRecords of this stream are open: close a DeviceRecords before asking for "
                                    f"more than lanes={self.lanes}")
            first, part, ticket, arr = self._inflight.popleft()
            if part is None:
                raise _at_input(arr, first)
            try:
                counts = self._pipe.wait_counts(ticket, len(part))
            except BaseException:
                self._pipe.release(ticket)
                raise
            recs = DeviceRecords(_Ticket(self._pipe, ticket), part, self._want, self._device, counts,
                                 release=(self._pipe.release, ticket), first_archive=first)
            self._yielded.append(weakref.ref(recs))
            if self._strict:
                _raise_for_counts(self._lib, counts, first, lambda i: f"archive {first + i} of the input")
            return recs
        except _AllLanesHeld:
            raise                       # the stream goes on once a DeviceRecords is closed
        except BaseException:
            self.close()
            raise


class _AllLanesHeld(RuntimeError):
    pass


def _at_input(e, index):
    """The exception reading or parsing input `index` raised, naming the index."""
    if isinstance(e, NafError):
        named = type(e)(f"{e} [archive {index} of the input]")
        named.status = e.status
        named.__cause__ = e
        return named
    e.add_note(f"reading archive {index} of the input")
    return e


def _raise_for_counts(lib, counts, first, label):
    """strict=True: the first failed archive raises as Context.decode does (its message ends with label(i)), then the first
    text that is not UTF-8 (NafUnicodeError with .archive = first + i and .record)."""
    for i, c in enumerate(counts):
        if c.status:
            raise_for_status(lib, c.status, None, label(i))
    for i, c in enumerate(counts):
        if c.record_status:
            e = NafUnicodeError(f"failed to decode UTF-8 data [archive {first + i}, record {c.first_bad_record}]")
            e.status, e.archive, e.record = c.record_status, first + i, int(c.first_bad_record)
            raise e


def stream_to_device(files, *, batch_bytes: int = 256 << 20, lanes: int = 2, device="cuda:0", id: bool = False,
                     comment: bool = False, sequence: bool = True, quality: bool = True, mask: bool = True, strict: bool = True,
                     _library=None) -> DeviceStream:
    """Decodes a collection of archives into device memory in sub-batches, yielding one DeviceRecords per sub-batch in input
    order.  `files` is any iterable of archives (bytes, paths or file objects), read lazily.  A sub-batch is a contiguous run
    of the input that ends where the next archive would take it past `batch_bytes` of compressed input, or at 65535 archives;
    an archive larger than batch_bytes is a sub-batch of its own.  `recs.first_archive` is the input index of the sub-batch's
    first archive, so input archive recs.first_archive + a holds records [recs.archive_records[a], recs.archive_records[a + 1]).

    The sub-batches are decoded on `lanes` lanes of a pipeline.  At most `lanes` of them are in flight or yielded and not yet
    closed: close each DeviceRecords when done with it (that hands its lane back; tensors already exported stay valid).  Asking
    for the next one while `lanes` are open raises RuntimeError and the stream goes on once one is closed.  When the stream
    ends (exhausted, an exception, close() or garbage collection) every ticket in flight is released, every DeviceRecords it
    yielded is closed and the pipeline's threads are gone.

    strict=True raises as decode_to_device does at the sub-batch that holds a corrupt archive or text that is not UTF-8, after
    the sub-batches before it have been yielded, naming the input index; with strict=False statuses are carried as there.
    An input that cannot be read or is not a NAF archive raises at its sub-batch either way."""
    lib = _library or _ffi.default_library()
    if int(batch_bytes) <= 0:
        raise ValueError("batch_bytes must be positive")
    if not 1 <= int(lanes) <= 64:
        raise ValueError("lanes must be in [1, 64]")
    return DeviceStream(files, int(batch_bytes), int(lanes), device, _want_bits(id, comment, sequence, quality, mask), strict, lib)

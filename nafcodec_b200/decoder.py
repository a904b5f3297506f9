"""Host-side mirror of the reference decoder surface over the nafgpu C ABI.

* `DecoderBuilder` / `Decoder` follow nafcodec/src/decoder/mod.rs:53-461 (builder knobs, opt-out fields, iterator that
  stops after header.number_of_sequences, ExactSizeIterator == __len__).
* The keyword constructor, properties, `read()` and context-manager protocol follow the Python binding
  (nafcodec-py/nafcodec/lib.rs:324-461, lib.pyi:36-70).

What differs from the reference by construction: the six per-section streaming zstd readers are replaced by ONE device
decode of the whole archive (ids, comments, lengths, mask, sequence, quality) on first access; records are then sliced
out of the structure-of-arrays result.  Errors the reference raises lazily at a record (invalid UTF-8 text) are raised
at that same record; corrupt compressed data is raised at the first record.
"""
import ctypes as C
import io
import os
import threading
from typing import Iterable, List, Optional

import numpy as np

from . import _ffi
from .data import Flag, Flags, FormatVersion, Header, Record, SequenceType
from .errors import NafArgumentError, NafIoError, raise_for_status

_SEQTYPE_NAMES = {0: "dna", 1: "rna", 2: "protein", 3: "text"}


class Context:
    """One nafgpu context (CUDA stream + arenas).  Not thread-safe: guarded by a lock."""

    def __init__(self, device: int = 0, library: Optional[_ffi.Library] = None):
        self.lib = library or _ffi.default_library()
        self.device = device
        self._ctx = C.c_void_p()
        self._lock = threading.Lock()
        raise_for_status(self.lib, self.lib.dll.nafgpu_ctx_create(device, C.byref(self._ctx)), what="nafgpu_ctx_create")

    def close(self):
        if self._ctx:
            self.lib.dll.nafgpu_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- parsing (host only) ------------------------------------------------------------------------------------
    def parse(self, buf) -> "_ffi.Archive":
        return parse_archive(buf, self.lib)

    # -- decode --------------------------------------------------------------------------------------------------
    def decode(self, archives: List["_ffi.Archive"], want: int = _ffi.WANT_ALL, strict: bool = True) -> List["ArchiveResult"]:
        """Decodes a batch in one set of kernel launches.  Archives fail independently (like separate reference Decoders):
        with strict=True the first corrupt archive raises; with strict=False its ArchiveResult carries `.status` /
        `.error` and the others are returned normally."""
        n = len(archives)
        arr = (_ffi.Archive * n)(*archives)
        res = (_ffi.Result * n)()
        with self._lock:
            rc = self.lib.dll.nafgpu_decode_batch(self._ctx, arr, n, want, res)
            raise_for_status(self.lib, rc, self._ctx)
            if strict:
                for i in range(n):
                    if res[i].status:
                        raise_for_status(self.lib, res[i].status, self._ctx, f"archive {i} of {n}" if n > 1 else "")
            return [ArchiveResult._copy_from(archives[i].header, res[i]) for i in range(n)]

    def format(self, archives: List["_ffi.Archive"], want: int = _ffi.WANT_ALL, format: int = _ffi.TEXT_AUTO,
               line_length: Optional[int] = None) -> List[bytes]:
        """FASTA / FASTQ text of every archive, formatted on the device (nafgpu_format_batch): '>' / '@' + id + separator +
        comment, the sequence wrapped at `line_length` (None: the header's; 0: one line), '+' and the quality for FASTQ."""
        n = len(archives)
        arr = (_ffi.Archive * n)(*archives)
        res = (_ffi.Text * n)()
        ll = _ffi.LINE_LENGTH_FROM_HEADER if line_length is None else int(line_length)
        with self._lock:
            rc = self.lib.dll.nafgpu_format_batch(self._ctx, arr, n, want, format, ll, res)
            raise_for_status(self.lib, rc, self._ctx)
            out = []
            for i in range(n):
                raise_for_status(self.lib, res[i].status, self._ctx if res[i].status != _ffi.ERR_UTF8 else None,
                                 f"record {res[i].first_bad_record}" if res[i].status == _ffi.ERR_UTF8 else f"archive {i}")
                out.append(C.string_at(res[i].data, int(res[i].size)) if res[i].size else b"")
            return out

    def zstd_decompress(self, frame: bytes, regen_size: int) -> bytes:
        """One magicless zstd frame -> bytes (the pure-zstd boundary; used by the parity tests against libzstd)."""
        src = (C.c_uint8 * max(len(frame), 1)).from_buffer_copy(frame or b"\0")
        dst = (C.c_uint8 * max(regen_size, 1))()
        with self._lock:
            rc = self.lib.dll.nafgpu_zstd_decompress(self._ctx, src, len(frame), regen_size, dst)
            raise_for_status(self.lib, rc, self._ctx)
        return C.string_at(dst, regen_size)          # (one copy: a slice of a ctypes array is a list of ints)

    # staged API (bench / profiling)
    def prepare(self, archives, want=_ffi.WANT_ALL):
        n = len(archives)
        self._arr = (_ffi.Archive * n)(*archives)
        self._n = n
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_prepare(self._ctx, self._arr, n, want), self._ctx)

    def run(self):
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_run(self._ctx), self._ctx)

    def sync(self):
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_sync(self._ctx), self._ctx)

    def fetch_raw(self):
        res = (_ffi.Result * self._n)()
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_fetch(self._ctx, res, self._n), self._ctx)
        return res

    def fetch_window(self, archive: int, first: int, count: int, max_bytes: int = 0) -> "ArchiveResult":
        """Records [first, first + count) of one archive of the job that was run, through a pinned buffer of that window only
        (nafgpu_job_fetch_window): the decoded archive stays in HBM between calls."""
        res = _ffi.Result()
        with self._lock:
            rc = self.lib.dll.nafgpu_job_fetch_window(self._ctx, archive, first, count, max_bytes, C.byref(res))
            raise_for_status(self.lib, rc, self._ctx)
            return ArchiveResult._copy_from(self._arr[archive].header, res)

    def fetch(self):
        res = self.fetch_raw()
        return [ArchiveResult._copy_from(self._arr[i].header, res[i]) for i in range(self._n)]

    def counts(self) -> List["_ffi.Counts"]:
        """Per-archive counters of the job that was run (nafgpu_job_counts: one small copy and a synchronise per run)."""
        res = (_ffi.Counts * self._n)()
        with self._lock:
            self._check_export(self.lib.dll.nafgpu_job_counts(self._ctx, res, self._n))
        return list(res)

    def export(self, spec: "_ffi.Export", stream: int = 0):
        """Enqueues one export of the job that was run into device memory (nafgpu_job_export) on `stream` (a cudaStream_t
        handle; 0 = the context's own stream).  A refused export raises NafArgumentError."""
        with self._lock:
            self._check_export(self.lib.dll.nafgpu_job_export(self._ctx, C.byref(spec), stream or None))

    def _check_export(self, rc):
        if rc == _ffi.ERR_ARGUMENT:
            e = NafArgumentError(self.lib.strerror(rc) + ": " + self.lib.dll.nafgpu_last_error(self._ctx).decode())
            e.status = rc
            raise e
        raise_for_status(self.lib, rc, self._ctx)

    def stats(self) -> "_ffi.JobStats":
        s = _ffi.JobStats()
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_get_stats(self._ctx, C.byref(s)), self._ctx)
        return s

    def time_runs(self, iters: int, flush_l2: bool = True) -> float:
        """Total device milliseconds of `iters` runs of the prepared job (CUDA events on the launch stream)."""
        ms = C.c_float()
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_time(self._ctx, iters, int(flush_l2), C.byref(ms)), self._ctx)
        return ms.value

    def profile_stages(self):
        n = self.stats().n_stages
        arr = (C.c_float * n)()
        raise_for_status(self.lib, self.lib.dll.nafgpu_job_run_profiled(self._ctx, arr, n), self._ctx)
        return [(self.lib.dll.nafgpu_stage_name(i).decode(), arr[i]) for i in range(n)]


def parse_archive(buf, lib: Optional[_ffi.Library] = None) -> "_ffi.Archive":
    """parser::header + setup_block! section table (parser.rs:101-139, mod.rs:169-242).  `buf` must stay alive while the
    returned struct is used (its section pointers point into it)."""
    lib = lib or _ffi.default_library()
    a = _ffi.Archive()
    if isinstance(buf, (bytes, bytearray)):
        keep = (C.c_uint8 * max(len(buf), 1)).from_buffer_copy(bytes(buf) or b"\0")
        n = len(buf)
    else:  # numpy uint8 array (e.g. a view of pinned memory)
        keep = buf
        n = buf.size
    ptr = C.cast(keep, C.c_void_p) if not isinstance(keep, np.ndarray) else C.c_void_p(keep.ctypes.data)
    rc = lib.dll.nafgpu_parse_archive(ptr, n, C.byref(a))
    raise_for_status(lib, rc, what="header")
    a._keep = keep
    return a


def _np_copy(ptr, count, dtype):
    if not ptr or count == 0:
        return np.zeros(count, dtype=dtype)
    nbytes = count * np.dtype(dtype).itemsize
    return np.frombuffer(C.string_at(ptr, nbytes), dtype=dtype)


class _FieldView:
    """One field of an ArchiveResult for iteration: text(i) is record i's string or None (None-ness rules of mod.rs:356-399)."""
    __slots__ = ("n", "off", "str", "blob", "trim")

    def __init__(self, blob, offsets, n, trim):
        self.n = n if (blob is not None and offsets is not None) else 0
        self.off = offsets.tolist() if self.n else None
        self.blob = blob
        self.str = blob.decode("ascii") if (self.n and blob.isascii()) else None      # (1 byte = 1 character: slice the text)
        self.trim = trim                                                                # ids / comments: the NUL

    def text(self, i):
        if i >= self.n:
            return None
        a, b = self.off[i], self.off[i + 1] - self.trim
        t = self.str
        return t[a:b] if t is not None else self.blob[a:b].decode("utf-8")


class ArchiveResult:
    """Structure-of-arrays result of one archive, copied out of the context's pinned buffers."""

    @classmethod
    def _copy_from(cls, hdr, r):
        self = cls()
        self.n_records = r.n_records
        self.status = r.status                       # 0, or why this archive of the batch could not be decoded
        self.n_ids, self.n_comments, self.n_lengths = r.n_ids, r.n_comments, r.n_lengths
        self.total_residues = r.total_residues
        self.first_bad_record = None if r.first_bad_record == _ffi.NO_RECORD else r.first_bad_record
        self.record_status = r.record_status
        # the offset tables hold n_ids + 1 / n_comments + 1 / n_lengths + 1 entries (include/nafgpu.h): number_of_sequences
        # is whatever the header claims
        self.id_offsets = _np_copy(r.id_offsets, self.n_ids + 1, np.uint64) if r.ids else None
        self.ids = C.string_at(r.ids, int(self.id_offsets[self.n_ids])) if r.ids and self.n_ids else (b"" if r.ids else None)
        self.comment_offsets = _np_copy(r.comment_offsets, self.n_comments + 1, np.uint64) if r.comments else None
        self.comments = C.string_at(r.comments, int(self.comment_offsets[self.n_comments])) if r.comments and self.n_comments else (b"" if r.comments else None)
        self.lengths = _np_copy(r.lengths, self.n_lengths, np.uint64) if r.lengths else None
        self.record_offsets = _np_copy(r.record_offsets, self.n_lengths + 1, np.uint64) if r.record_offsets else None
        self.sequence = C.string_at(r.sequence, r.total_residues) if r.sequence else None
        self.quality = C.string_at(r.quality, r.total_residues) if r.quality else None
        return self

    def views(self):
        """Per-field views for record iteration (built once): offsets as Python ints and, where a blob is pure ASCII, its text
        decoded once, so that a record costs four string slices instead of four numpy reads, byte slices and decodes."""
        v = getattr(self, "_views", None)
        if v is None:
            nl = self.n_lengths if self.lengths is not None else 0
            v = self._views = (_FieldView(self.ids, self.id_offsets, self.n_ids, 1), _FieldView(self.comments, self.comment_offsets, self.n_comments, 1),
                               _FieldView(self.sequence, self.record_offsets, nl, 0), _FieldView(self.quality, self.record_offsets, nl, 0),
                               self.lengths.tolist() if self.lengths is not None else [], nl)
        return v

    # field accessors with the reference's None-ness rules (mod.rs:356-399)
    def id_bytes(self, i):
        if self.ids is None or i >= self.n_ids:
            return None
        return self.ids[int(self.id_offsets[i]):int(self.id_offsets[i + 1]) - 1]

    def comment_bytes(self, i):
        if self.comments is None or i >= self.n_comments:
            return None
        return self.comments[int(self.comment_offsets[i]):int(self.comment_offsets[i + 1]) - 1]

    def length(self, i):
        if self.lengths is None or i >= self.n_lengths:
            return None
        return int(self.lengths[i])

    def sequence_bytes(self, i):
        if self.sequence is None or i >= self.n_lengths:
            return None
        return self.sequence[int(self.record_offsets[i]):int(self.record_offsets[i + 1])]

    def quality_bytes(self, i):
        if self.quality is None or i >= self.n_lengths:
            return None
        return self.quality[int(self.record_offsets[i]):int(self.record_offsets[i + 1])]


_contexts = {}
_contexts_lock = threading.Lock()


def shared_context(device: int = 0, library: Optional[_ffi.Library] = None) -> Context:
    lib = library or _ffi.default_library()
    key = (lib.path, device)
    with _contexts_lock:
        if key not in _contexts:
            _contexts[key] = Context(device, lib)
        return _contexts[key]


def _want_bits(id, comment, sequence, quality, mask):
    return ((_ffi.WANT_ID if id else 0) | (_ffi.WANT_COMMENT if comment else 0) | (_ffi.WANT_SEQUENCE if sequence else 0) |
            (_ffi.WANT_QUALITY if quality else 0) | (_ffi.WANT_MASK if mask else 0))


class Decoder:
    """A decoder for Nucleotide Archive Format files running on a B200 (surface of nafcodec.Decoder)."""

    def __init__(self, file, *, id: bool = True, comment: bool = True, sequence: bool = True, quality: bool = True,
                 mask: bool = True, buffer_size: Optional[int] = None, device: int = 0, _library=None):
        # buffer_size (DecoderBuilder::buffer_size, decoder/mod.rs:105-112): the reference reads every section through
        # BufReaders of this many bytes, so its memory is bounded whatever the archive.  Here an explicit buffer_size bounds the
        # HOST side the same way: the archive is decoded once into HBM and the records cross PCIe in windows of about
        # buffer_size decoded bytes (at least one record), a path is mapped instead of read, and the first record is
        # yielded after the first window.  Without it the whole result is copied back in one go (fastest for whole-file reads).
        self._buffer_size = buffer_size if buffer_size is not None else io.DEFAULT_BUFFER_SIZE
        self._window_bytes = max(int(buffer_size), 1) if buffer_size is not None else 0
        self._window_first = 0
        self._window_ctx: Optional[Context] = None
        self._file = file
        if hasattr(file, "read"):
            data = file.read()
        else:
            path = os.fspath(file)
            with open(path, "rb") as f:      # FileNotFoundError / IsADirectoryError as in lib.rs:363-376
                if self._window_bytes and os.fstat(f.fileno()).st_size:
                    data = np.memmap(f, dtype=np.uint8, mode="r")     # compressed sections go page cache -> device
                else:
                    data = f.read()
        self._library = _library or _ffi.default_library()
        if len(data) == 0:
            # Decoder::new on empty input: Io(UnexpectedEof) "failed to read header" (mod.rs:181-186, test mod.rs:470-476)
            e = NafIoError("failed to read header")
            e.status = _ffi.ERR_UNEXPECTED_EOF
            raise e
        self._archive = parse_archive(data, self._library)
        h = self._archive.header
        self._header = Header(FormatVersion(h.format_version), SequenceType(h.sequence_type), Flags(h.flags),
                              chr(h.name_separator), h.line_length, h.number_of_sequences)
        self._want = _want_bits(id, comment, sequence, quality, mask)
        self._device = device
        self._n = 0
        self._run = None
        self._result: Optional[ArchiveResult] = None

    # -- Rust-style constructors -----------------------------------------------------------------------------------
    @classmethod
    def from_path(cls, path, **kw):          # mod.rs:304-306
        return cls(path, **kw)

    @classmethod
    def new(cls, reader, **kw):              # mod.rs:315-317
        return cls(reader, **kw)

    # -- header ----------------------------------------------------------------------------------------------------
    def header(self) -> Header:              # mod.rs:326-328
        return self._header

    @property
    def sequence_type(self) -> str:          # lib.rs:417-420 (Python surface returns the lowercase name)
        return _SEQTYPE_NAMES[int(self._header.sequence_type)]

    @property
    def format_version(self) -> str:
        return "v1" if self._header.format_version == FormatVersion.V1 else "v2"

    @property
    def line_length(self) -> int:
        return self._header.line_length

    @property
    def name_separator(self) -> str:
        return self._header.name_separator

    @property
    def number_of_sequences(self) -> int:
        return self._header.number_of_sequences

    def into_inner(self):                    # mod.rs:343-350
        return self._file

    # -- iteration -------------------------------------------------------------------------------------------------
    def _decoded(self) -> ArchiveResult:
        if self._result is None:
            ctx = shared_context(self._device, self._library)
            self._result = ctx.decode([self._archive], self._want)[0]
        return self._result

    def _window(self, i: int) -> ArchiveResult:
        """The window holding record i (windowed mode): the archive is decoded into HBM at the first call and stays there, on a
        context of this decoder's own, until the last record has been fetched."""
        if self._window_ctx is None:
            self._window_ctx = Context(self._device, self._library)
            self._window_ctx.prepare([self._archive], self._want)
            self._window_ctx.run()
        r = self._result
        if r is None or not (self._window_first <= i < self._window_first + r.n_records):
            r = self._result = self._window_ctx.fetch_window(0, i, self._header.number_of_sequences - i, self._window_bytes)
            self._window_first = i
        return r

    def close(self):
        """Releases the device memory of a windowed decoder early (otherwise released with the object)."""
        if self._window_ctx is not None:
            self._window_ctx.close()
            self._window_ctx = None

    def __iter__(self):
        return self

    def __len__(self):                       # ExactSizeIterator (mod.rs:453-459)
        return self._header.number_of_sequences - self._n

    def __next__(self) -> Record:
        run = self._run
        if run is not None:                                # records [i, stop) of the current result without a stop in between:
            try:                                           # a generator with everything in locals (~1 us per record)
                return next(run)
            except StopIteration:
                self._run = None
        if self._n >= self._header.number_of_sequences:    # mod.rs:447-449
            if self._window_bytes:
                self.close()
            raise StopIteration
        if self._window_bytes:
            r = self._window(self._n)
            base = self._window_first
        else:
            r = self._decoded()
            base = 0
        i = self._n - base
        bad = r.first_bad_record
        if bad is not None and i == bad:
            self._n += 1
            raise_for_status(self._library, r.record_status)
        stop = min(r.n_records, self._header.number_of_sequences - base)
        if bad is not None and i < bad < stop:
            stop = bad
        self._run = self._records(r, i, stop)
        return next(self._run)

    def _records(self, r: ArchiveResult, i: int, stop: int):
        """Records [i, stop) of one result (or window), None-ness as in mod.rs:356-399."""
        idv, comv, seqv, qualv, lengths, nl = r.views()
        id_n, id_off, id_str, id_blob = idv.n, idv.off, idv.str, idv.blob
        com_n, com_off, com_str, com_blob = comv.n, comv.off, comv.str, comv.blob
        seq_n, seq_str, seq_blob = seqv.n, seqv.str, seqv.blob
        qual_n, qual_str, qual_blob = qualv.n, qualv.str, qualv.blob
        rec_off = seqv.off if seq_n else qualv.off
        new = Record.__new__
        while i < stop:
            rec = new(Record)
            if i < id_n:
                a, b = id_off[i], id_off[i + 1] - 1
                rec.id = id_str[a:b] if id_str is not None else id_blob[a:b].decode("utf-8")
            else:
                rec.id = None
            if i < com_n:
                a, b = com_off[i], com_off[i + 1] - 1
                rec.comment = com_str[a:b] if com_str is not None else com_blob[a:b].decode("utf-8")
            else:
                rec.comment = None
            if i < nl:
                rec.length = lengths[i]
                if rec_off is not None:
                    a, b = rec_off[i], rec_off[i + 1]
                    rec.sequence = (seq_str[a:b] if seq_str is not None else seq_blob[a:b].decode("utf-8")) if seq_n else None
                    rec.quality = (qual_str[a:b] if qual_str is not None else qual_blob[a:b].decode("utf-8")) if qual_n else None
                else:
                    rec.sequence = rec.quality = None
            else:
                rec.length = rec.sequence = rec.quality = None
            i += 1
            self._n += 1
            yield rec

    def read(self) -> Optional[Record]:      # lib.rs:452-460
        try:
            return self.__next__()
        except StopIteration:
            return None

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc_value, traceback):
        return False


def _make_record(id, comment, sequence, quality, length) -> Record:
    r = Record.__new__(Record)
    r.id, r.comment, r.sequence, r.quality, r.length = id, comment, sequence, quality, length
    return r


class DecoderBuilder:
    """Builder with opt-out fields (nafcodec/src/decoder/mod.rs:53-257)."""

    def __init__(self):                      # DecoderBuilder::new (mod.rs:66-75)
        self._buffer_size = 4096
        self._id = self._comment = self._sequence = self._quality = self._mask = True
        self._device = 0
        self._library = None

    @classmethod
    def new(cls):
        return cls()

    @classmethod
    def from_flags(cls, flags):              # mod.rs:93-101 (quirk kept: never clears `id`)
        flags = int(flags)
        b = cls()
        b.quality(bool(flags & Flag.Quality))
        b.sequence(bool(flags & Flag.Sequence))
        b.mask(bool(flags & Flag.Mask))
        b.comment(bool(flags & Flag.Comment))
        return b

    def buffer_size(self, n):
        self._buffer_size = n
        return self

    def id(self, v):
        self._id = v
        return self

    def comment(self, v):
        self._comment = v
        return self

    def sequence(self, v):
        self._sequence = v
        return self

    def quality(self, v):
        self._quality = v
        return self

    def mask(self, v):
        self._mask = v
        return self

    def device(self, index):                 # extension: which GPU
        self._device = index
        return self

    def _kw(self):
        return dict(id=self._id, comment=self._comment, sequence=self._sequence, quality=self._quality, mask=self._mask,
                    buffer_size=self._buffer_size, device=self._device, _library=self._library)

    def with_bytes(self, data: bytes) -> Decoder:        # mod.rs:151-156
        return Decoder(io.BytesIO(data), **self._kw())

    def with_path(self, path) -> Decoder:                # mod.rs:159-166
        return Decoder(path, **self._kw())

    def with_reader(self, reader) -> Decoder:            # mod.rs:169-257
        return Decoder(reader, **self._kw())


class Pipeline:
    """The C ABI's pipeline (nafgpu_pipeline_*, include/nafgpu.h): `lanes` contexts and host threads inside the library, so
    that the H2D copy of one sub-batch, the kernels of another and the D2H copy of a third overlap.  This class only cuts
    batches into sub-batches and keeps a few tickets in flight; a Rust or C++ caller uses the same three calls."""

    def __init__(self, device: int = 0, lanes: int = 3, library: Optional[_ffi.Library] = None):
        self.lib = library or _ffi.default_library()
        self.lanes = lanes
        self._p = C.c_void_p()
        raise_for_status(self.lib, self.lib.dll.nafgpu_pipeline_create(device, lanes, C.byref(self._p)), what="nafgpu_pipeline_create")

    def _raise(self, rc):
        if rc:
            msg = self.lib.dll.nafgpu_pipeline_last_error(self._p).decode()
            raise_for_status(self.lib, rc, None, msg)

    def _submit(self, part, want, submit=None):
        cnt = len(part)
        arr = (_ffi.Archive * cnt)(*part)
        t = (submit or self.lib.dll.nafgpu_pipeline_submit)(self._p, arr, cnt, want)
        if t < 0:
            self._raise(int(t))
        return t, arr, cnt

    def _finish(self, ticket, cnt, each):
        res = (_ffi.Result * cnt)()
        rc = self.lib.dll.nafgpu_pipeline_wait(self._p, ticket, res, cnt)
        try:
            self._raise(rc)
            for i in range(cnt):
                if res[i].status:
                    raise_for_status(self.lib, res[i].status, None, f"archive {i} of the sub-batch")
                each(i, res[i])
        finally:
            self.lib.dll.nafgpu_pipeline_release(self._p, ticket)

    def decode(self, archives, want: int = _ffi.WANT_ALL, consume=None):
        """Decodes `archives` (list of _ffi.Archive) in `lanes` sub-batches.  `consume(index, result_struct)` is called for
        every archive while its pinned buffers are valid; without it the results are copied out as ArchiveResult objects."""
        n, lanes = len(archives), self.lanes
        bounds = [(n * k) // lanes for k in range(lanes + 1)]
        out = [None] * n
        inflight = [(lo,) + self._submit(archives[lo:hi], want) for lo, hi in zip(bounds, bounds[1:]) if hi > lo]
        err = None
        for lo, t, arr, cnt in inflight:
            def each(i, r, lo=lo):
                if consume is not None:
                    consume(lo + i, r)
                else:
                    out[lo + i] = ArchiveResult._copy_from(archives[lo + i].header, r)
            try:
                self._finish(t, cnt, each)
            except Exception as e:              # every ticket is waited for and released, then the first error is raised
                err = err or e
        if err is not None:
            raise err
        return out

    def decode_stream(self, batches, want: int = _ffi.WANT_ALL, consume=None, sub_batch: Optional[int] = None):
        """Decodes a sequence of batches (each a list of _ffi.Archive) as ONE stream of work: every batch is cut into
        sub-batches that are submitted ahead of the consumer (2 x lanes tickets in flight, no barrier between batches), so the
        header walk, H2D and kernels of one sub-batch always overlap the D2H of another.  `consume(batch_index, index,
        result_struct)` runs while the pinned buffers of that sub-batch are valid.  Returns the number of archives decoded."""
        from collections import deque
        lanes = self.lanes

        def pieces():
            for bi, archives in enumerate(batches):
                n = len(archives)
                step = sub_batch or max(1, -(-n // lanes))
                for lo in range(0, n, step):
                    yield bi, lo, archives[lo:lo + step]

        it = pieces()
        inflight = deque()
        done = 0
        err = None
        while True:
            while len(inflight) < 2 * lanes and err is None:
                nxt = next(it, None)
                if nxt is None:
                    break
                bi, lo, part = nxt
                inflight.append((bi, lo) + self._submit(part, want))
            if not inflight:
                break
            bi, lo, t, arr, cnt = inflight.popleft()

            def each(i, r, bi=bi, lo=lo):
                if consume is not None:
                    consume(bi, lo + i, r)
            try:
                self._finish(t, cnt, each)
                done += cnt
            except Exception as e:
                err = err or e
        if err is not None:
            raise err
        return done

    # -- device tickets (nafgpu_pipeline_submit_device / _wait_counts / _export): the sub-batch stays in the lane's arena -------
    def submit_device(self, archives, want: int = _ffi.WANT_ALL):
        """Submits a device ticket; returns (ticket, archive array).  The array and the archives' bytes are borrowed until
        wait_counts returns."""
        return self._submit(archives, want, self.lib.dll.nafgpu_pipeline_submit_device)[:2]

    def wait_counts(self, ticket: int, n: int) -> List["_ffi.Counts"]:
        """Blocks until the device ticket is decoded: n per-archive counters (a corrupt archive only sets its own status)."""
        res = (_ffi.Counts * n)()
        self._raise(self.lib.dll.nafgpu_pipeline_wait_counts(self._p, ticket, res, n))
        return list(res)

    def export(self, ticket: int, spec: "_ffi.Export", stream: int = 0):
        """nafgpu_job_export on the ticket's lane (as Context.export); a refused export raises NafArgumentError."""
        rc = self.lib.dll.nafgpu_pipeline_export(self._p, ticket, C.byref(spec), stream or None)
        if rc == _ffi.ERR_ARGUMENT:
            e = NafArgumentError(self.lib.strerror(rc) + ": " + self.lib.dll.nafgpu_pipeline_last_error(self._p).decode())
            e.status = rc
            raise e
        self._raise(rc)

    def release(self, ticket: int):
        if self._p:                     # (after close the tickets went with the pipeline)
            self._raise(self.lib.dll.nafgpu_pipeline_release(self._p, ticket))

    def stats(self):
        out = []
        for k in range(self.lanes):
            s = _ffi.JobStats()
            self.lib.dll.nafgpu_pipeline_lane_stats(self._p, k, C.byref(s))
            out.append(s)
        return out

    def close(self):
        if self._p:
            self.lib.dll.nafgpu_pipeline_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def decode_batch(files: Iterable, *, id=True, comment=True, sequence=True, quality=True, mask=True, device: int = 0,
                 _library=None) -> List[ArchiveResult]:
    """Decode many independent archives in one set of kernel launches (the RefSeq-collection shape)."""
    lib = _library or _ffi.default_library()
    archives = []
    for f in files:
        if isinstance(f, (bytes, bytearray)):
            data = bytes(f)
        elif hasattr(f, "read"):
            data = f.read()
        else:
            with open(os.fspath(f), "rb") as fh:
                data = fh.read()
        archives.append(parse_archive(data, lib))
    return shared_context(device, lib).decode(archives, _want_bits(id, comment, sequence, quality, mask))


_TEXT_FORMATS = {"auto": _ffi.TEXT_AUTO, "fasta": _ffi.TEXT_FASTA, "fastq": _ffi.TEXT_FASTQ}


def _read_all(f) -> bytes:
    if isinstance(f, (bytes, bytearray, memoryview)):
        return bytes(f)
    if hasattr(f, "read"):
        return f.read()
    with open(os.fspath(f), "rb") as fh:
        return fh.read()


def to_text(files, format: str = "auto", *, line_length: Optional[int] = None, comment: bool = True, mask: bool = True,
            device: int = 0, _library=None):
    """Archive(s) -> FASTA / FASTQ text (bytes), formatted on the GPU; what upstream `unnaf` prints.  `files` is one
    archive (bytes, path or file object) or a list of them (one set of kernel launches for the whole list).
    format: "fasta", "fastq", or "auto" (FASTQ when the archive stores qualities).  line_length: None = the header's
    (Header.line_length, data.rs:198-236), 0 = unwrapped.  mask=False gives upper-case sequences; comment=False names only."""
    lib = _library or _ffi.default_library()
    single = not isinstance(files, (list, tuple))
    datas = [_read_all(f) for f in ([files] if single else files)]
    archives = [parse_archive(d, lib) for d in datas]
    fmt = _TEXT_FORMATS[format]
    want = _want_bits(True, comment, True, fmt != _ffi.TEXT_FASTA, mask)
    out = shared_context(device, lib).format(archives, want, fmt, line_length)
    return out[0] if single else out


def to_fasta(files, **kw):
    return to_text(files, "fasta", **kw)


def to_fastq(files, **kw):
    return to_text(files, "fastq", **kw)

/*
 * nafgpu.h -- C ABI of the B200-native backend for the nafcodec decode hot path.
 *
 * This is the boundary a Rust `extern "C"` block (rust_shim/ffi.rs) or any other FFI binds.  It replaces, for
 * one NAF archive or a batch of archives, the six per-section streaming readers the reference builds in
 * `setup_block!` (nafcodec/src/decoder/mod.rs:199-242: BufReader<zstd::Decoder<BufReader<IoSlice<R>>>>,
 * type alias at mod.rs:32) and everything `Decoder::next_record` / `mask_sequence` (mod.rs:356-441) and the
 * readers of nafcodec/src/decoder/reader.rs compute from them.  Plain pointers and sizes only; no C++ types,
 * no exceptions cross this boundary.  Every entry point returns 0 or a negative nafgpu_status.
 *
 * There is NO CPU fallback: without the CUDA library / a device, nafgpu_ctx_create fails with
 * NAFGPU_ERR_NO_DEVICE and nothing else can be called.
 */
#ifndef NAFGPU_H
#define NAFGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Status codes.  Mapping onto the reference's `Error` (nafcodec/src/error.rs:4-11) is given per code. */
typedef enum nafgpu_status {
    NAFGPU_OK = 0,
    NAFGPU_ERR_UNEXPECTED_EOF = -1, /* Error::Io(UnexpectedEof): truncated header/section/stream, "failed to get mask unit" (mod.rs:431-434) */
    NAFGPU_ERR_INVALID_DATA = -2,   /* Error::Io(InvalidData): corrupt zstd data (what zstd-rs reports) */
    NAFGPU_ERR_PARSE = -3,          /* Error::Nom: bad format descriptor / version / sequence type / separator (parser.rs:50-91) */
    NAFGPU_ERR_UTF8 = -4,           /* Error::Io(InvalidData) from String::from_utf8 (reader.rs:108-109); ids/comments: reference panics (mod.rs:362,368) */
    NAFGPU_ERR_CUDA = -5,           /* Error::Io(Other): CUDA runtime failure */
    NAFGPU_ERR_NOMEM = -6,          /* Error::Io(OutOfMemory) */
    NAFGPU_ERR_ARGUMENT = -7,       /* caller bug (NULL pointer, bad index) */
    NAFGPU_ERR_NO_DEVICE = -8,      /* no CUDA device: there is no CPU fallback */
    NAFGPU_ERR_UNSUPPORTED = -9     /* valid zstd the backend does not handle (dictionaries) */
} nafgpu_status;

/* Header (nafcodec/src/data.rs:198-205, parsed by decoder/parser.rs:101-123). */
typedef struct nafgpu_header {
    int32_t format_version;        /* 1 | 2 (data.rs:46-50) */
    int32_t sequence_type;         /* 0 dna, 1 rna, 2 protein, 3 text (data.rs:56-62) */
    uint32_t flags;                /* Flag bits (data.rs:80-97): Quality 1, Sequence 2, Mask 4, Length 8, Comment 0x10, Id 0x20, Title 0x40, Extended 0x80 */
    int32_t name_separator;
    uint64_t line_length;
    uint64_t number_of_sequences;
} nafgpu_header;

/* Section order is fixed: Id, Comment, Length, Mask, Sequence, Quality (decoder/mod.rs:237-242). */
enum { NAFGPU_SEC_ID = 0, NAFGPU_SEC_COMMENT = 1, NAFGPU_SEC_LENGTH = 2, NAFGPU_SEC_MASK = 3, NAFGPU_SEC_SEQUENCE = 4, NAFGPU_SEC_QUALITY = 5, NAFGPU_N_SECTIONS = 6 };

/* One compressed section as `setup_block!` finds it: (original_size, compressed_size) varints + byte range. */
typedef struct nafgpu_section {
    const uint8_t* data;           /* HOST pointer to the compressed bytes (one magicless zstd frame); borrowed during the call */
    uint64_t compressed_size;
    uint64_t original_size;        /* Sequence: residues (encoder/counter.rs:25-34); other sections: bytes */
    int32_t present;               /* flag set in the header */
    int32_t _pad;
} nafgpu_section;

typedef struct nafgpu_archive {
    nafgpu_header header;
    nafgpu_section sections[NAFGPU_N_SECTIONS];
} nafgpu_archive;

/* Field selection == DecoderBuilder::{id,comment,sequence,quality,mask} (decoder/mod.rs:117-148).  Lengths are
 * always decoded (mod.rs:239). */
enum { NAFGPU_WANT_ID = 1, NAFGPU_WANT_COMMENT = 2, NAFGPU_WANT_SEQUENCE = 4, NAFGPU_WANT_QUALITY = 8, NAFGPU_WANT_MASK = 16, NAFGPU_WANT_ALL = 31 };

/* Decoded archive, structure-of-arrays.  Pointers are HOST pointers into pinned memory owned by the context,
 * valid until the next nafgpu_decode* / nafgpu_job_prepare on that context or its destruction.
 * Record i (0 <= i < n_records) as the reference's iterator would yield it (mod.rs:356-399):
 *   id       = i < n_ids      ? ids[id_offsets[i] .. id_offsets[i+1]-1)            : None   (NUL stripped)
 *   comment  = i < n_comments ? comments[comment_offsets[i] .. comment_offsets[i+1]-1) : None
 *   length   = i < n_lengths  ? lengths[i] : None
 *   sequence = (i < n_lengths && sequence) ? sequence[record_offsets[i] .. record_offsets[i+1]) : None
 *   quality  = (i < n_lengths && quality)  ? quality [record_offsets[i] .. record_offsets[i+1]) : None
 * A NULL blob pointer means the field is absent from the archive or was not requested.
 * n_records is the header's number_of_sequences, which a file may overstate at will: the offset tables hold n_ids + 1,
 * n_comments + 1 and n_lengths + 1 entries (a stream of b bytes cannot hold more than b strings or b / 4 lengths). */
typedef struct nafgpu_result {
    uint64_t n_records;
    uint64_t n_ids, n_comments, n_lengths;
    uint64_t total_residues;            /* == record_offsets[n_lengths] */
    const uint8_t* ids;
    const uint64_t* id_offsets;         /* n_ids + 1 entries */
    const uint8_t* comments;
    const uint64_t* comment_offsets;    /* n_comments + 1 entries */
    const uint64_t* lengths;            /* n_lengths entries */
    const uint64_t* record_offsets;     /* n_lengths + 1 entries (exclusive prefix sum of lengths) */
    const uint8_t* sequence;            /* ASCII, soft-masked; total_residues bytes */
    const uint8_t* quality;             /* total_residues bytes */
    uint64_t first_bad_record;          /* UINT64_MAX, or the first record whose text is not UTF-8: records before it are valid,
                                           the reference yields an error AT that record (reader.rs:108-109) */
    int32_t record_status;              /* status to raise at first_bad_record (NAFGPU_ERR_UTF8) or 0 */
    int32_t status;                     /* 0, or why THIS archive could not be decoded (corrupt / truncated data): its pointers are
                                           NULL then.  Archives of a batch fail independently, like separate reference Decoders */
} nafgpu_result;

/* Sizes of the last prepared job, for throughput arithmetic (SURVEY 8d: B_alg). */
typedef struct nafgpu_job_stats {
    uint64_t n_archives, n_frames, n_blocks, n_sequences;
    uint64_t compressed_bytes;          /* sum of compressed sizes of the decoded sections */
    uint64_t section_bytes;             /* regenerated bytes of all decoded sections */
    uint64_t ascii_bytes;               /* sequence ASCII bytes (capacity from the headers) */
    uint64_t quality_bytes, id_bytes, comment_bytes;
    uint64_t algorithmic_bytes;         /* compressed in + every output byte once + 8*(n_records+1) offsets */
    uint64_t h2d_bytes, d2h_bytes;      /* bytes copied per decode */
    uint32_t kernel_launches;           /* kernels enqueued by one nafgpu_job_run */
    uint32_t n_stages;                  /* entries nafgpu_job_run_profiled writes */
    uint32_t lz_handover;               /* nonzero if the last fetched run left LZ matches to the ordered finisher (k_lz_finish): the round it gave up at */
    uint32_t lz_rounds;                 /* dependency rounds the LZ stage of the last fetched run took */
    uint32_t lz_unresolved;             /* bytes the finisher's first level left to its cross-chunk level (0 without a hand-over) */
    float text_kernel_ms;               /* device time of the last nafgpu_job_format's kernels (CUDA events on the context's stream) */
    uint64_t text_bytes;                /* bytes of text the last nafgpu_job_format produced */
    uint32_t lz_pending[24];            /* matches still waiting after dependency round 1, 2, ... of the last fetched run (0 past the last round) */
    uint32_t lz_flow;                   /* the in-order match kernel (k_lz_flow) in the last fetched run: bit 0 = the rounds handed chains of a few dozen generations to it;
                                           bit 1 = it ran before the rounds (a job of a few thousand matches) and met its deadline */
    uint32_t _pad;
} nafgpu_job_stats;

/* ---- host-only helpers -------------------------------------------------------------------------------- */

/* parser::header + title + the setup_block! section table over an in-memory archive (parser.rs:101-139,
 * mod.rs:169-242).  Section data pointers point into `bytes`.  No GPU needed. */
int nafgpu_parse_archive(const uint8_t* bytes, uint64_t len, nafgpu_archive* out);
/* parser::variable_u64 (parser.rs:27-48): returns bytes consumed (>0) or a negative status. */
int nafgpu_variable_u64(const uint8_t* bytes, uint64_t len, uint64_t* value);

const char* nafgpu_strerror(int status);
const char* nafgpu_version(void);

/* ---- context --------------------------------------------------------------------------------------------- */
typedef struct nafgpu_ctx nafgpu_ctx;

/* One context per Decoder (or per worker thread); owns a CUDA stream, device arenas and pinned result buffers.
 * Replaces the construction / drop of the six `BufReader<zstd::Decoder<BufReader<IoSlice<R>>>>` section readers that
 * `setup_block!` builds in DecoderBuilder::with_reader (nafcodec/src/decoder/mod.rs:32,199-242).
 * Not thread-safe; distinct contexts may be used concurrently from distinct threads (cudaSetDevice at every entry). */
int nafgpu_ctx_create(int device, nafgpu_ctx** out);
void nafgpu_ctx_destroy(nafgpu_ctx* ctx);
const char* nafgpu_last_error(const nafgpu_ctx* ctx);   /* the message of the last failure (the io::Error text of error.rs:4-11) */

/* Pinned host memory for callers that want zero staging copies (optional). */
void* nafgpu_host_alloc(size_t bytes);
void nafgpu_host_free(void* p);

/* ---- decode ------------------------------------------------------------------------------------------------ */

/* Whole path, host buffers in, host buffers out: walk frames, H2D, kernels, D2H, synchronise.  Replaces, for ALL records of
 * the archive at once, what Decoder::next_record (decoder/mod.rs:356-399) pulls from the readers: CStringReader::next
 * (reader.rs:20-31), LengthReader::next (46-68), SequenceReader::next / read_nucleotide / read_text (88-172),
 * MaskReader::next (196-231), Decoder::mask_sequence (mod.rs:402-441), and the zstd inflate underneath (mod.rs:221-223). */
int nafgpu_decode(nafgpu_ctx* ctx, const nafgpu_archive* archive, uint32_t want, nafgpu_result* out);
/* Same for n independent archives in ONE set of kernel launches (the batch / RefSeq-collection shape); n <= 65535 per
 * call (larger collections: several calls, or the pipeline below).  The return value reports failures of the CALL (bad
 * arguments, CUDA, memory); a corrupt or truncated archive only sets its own out[i].status (for n == 1 that status is
 * also the return value) and nafgpu_last_error names the first such archive. */
int nafgpu_decode_batch(nafgpu_ctx* ctx, const nafgpu_archive* archives, uint32_t n, uint32_t want, nafgpu_result* out);

/* One magicless zstd frame -> exactly regen_size bytes at dst (host memory).  The pure-zstd boundary: what
 * zstd::stream::read::Decoder + include_magicbytes(false) (decoder/mod.rs:221-223) yields for one section. */
int nafgpu_zstd_decompress(nafgpu_ctx* ctx, const uint8_t* frame, uint64_t frame_size, uint64_t regen_size, uint8_t* dst);

/* The same pipeline in three steps, so the device-resident part can be timed on its own:
 *   prepare: host frame walk + H2D of compressed sections and descriptors (asynchronous on the context's stream)
 *   run:     enqueue every kernel (asynchronous); may be called repeatedly on a prepared job
 *   fetch:   D2H of the results + synchronise + validate; fills n results */
int nafgpu_job_prepare(nafgpu_ctx* ctx, const nafgpu_archive* archives, uint32_t n, uint32_t want);
int nafgpu_job_run(nafgpu_ctx* ctx);
int nafgpu_job_fetch(nafgpu_ctx* ctx, nafgpu_result* out, uint32_t n);
int nafgpu_job_sync(nafgpu_ctx* ctx);
/* Bounded-memory fetch: records [first, first + count) of archive `archive` of the job that was run, as a result of their
 * own (out->n_records = records in the window, offsets relative to the window's first byte, first_bad_record relative to
 * `first`), through a pinned buffer that holds this window only.  max_bytes != 0 shrinks the window to the records that fit
 * in max_bytes of decoded data (never below one record).  The decoded archive stays in device memory between calls, so a
 * consumer that walks the archive in windows needs host memory for one window, as the reference needs it for its 4 KiB
 * BufReaders (decoder/mod.rs:69,105-112,221-223: DecoderBuilder::buffer_size), and gets record `first` after one window has
 * crossed PCIe.  Pointers are valid until the next fetch of either kind on the context.  Returns the archive's status. */
int nafgpu_job_fetch_window(nafgpu_ctx* ctx, uint32_t archive, uint64_t first, uint64_t count, uint64_t max_bytes, nafgpu_result* out);
int nafgpu_job_get_stats(const nafgpu_ctx* ctx, nafgpu_job_stats* out);

/* Runs the prepared job `iters` times back to back and returns the elapsed device time in milliseconds, measured
 * with CUDA events on the context's own stream (where the kernels are launched). If flush_l2 != 0 a buffer larger
 * than L2 is overwritten before every iteration, outside the timed intervals (per-iteration events are summed). */
int nafgpu_job_time(nafgpu_ctx* ctx, int iters, int flush_l2, float* total_ms);
/* One serial run with an event after every stage (the last entry is the dominant kernel alone: the Huffman decode of the
 * big streams, k_huf_decode_block or k_huf_decode_big depending on the job size);
 * stage_ms must hold stats.n_stages floats. Stage names: nafgpu_stage_name. */
int nafgpu_job_run_profiled(nafgpu_ctx* ctx, float* stage_ms, uint32_t n_stages);
const char* nafgpu_stage_name(uint32_t stage);

/* ---- FASTA / FASTQ text (SURVEY 8f rank 1) --------------------------------------------------------------------------
 * The reference crate yields Records and only CARRIES what a formatter needs, Header::line_length and
 * Header::name_separator (nafcodec/src/data.rs:198-236; accessors decoder/mod.rs:319-328); the text is what upstream
 * `unnaf` prints and the reference's fixtures hold (data/masked.fna, data/LuxC.faa, data/phix.fastq):
 *   FASTA  '>' id [sep comment] '\n' sequence wrapped at line_length (0 = one line) '\n'
 *   FASTQ  '@' id [sep comment] '\n' sequence '\n' '+' '\n' quality '\n'
 * (separator + comment only when the comment is not empty; absent fields are empty).  Formatted on the device from the
 * job that was just run; only the text is copied back. */
enum { NAFGPU_TEXT_AUTO = 0 /* FASTQ iff quality was decoded */, NAFGPU_TEXT_FASTA = 1, NAFGPU_TEXT_FASTQ = 2 };
#define NAFGPU_LINE_LENGTH_FROM_HEADER UINT64_MAX

typedef struct nafgpu_text {
    const uint8_t* data;                /* HOST pointer into pinned memory owned by the context (valid until its next call) */
    uint64_t size;
    int32_t format;                     /* NAFGPU_TEXT_FASTA | NAFGPU_TEXT_FASTQ, as written */
    int32_t status;                     /* 0; NAFGPU_ERR_UTF8: the reference fails AT first_bad_record (reader.rs:108-109); any other
                                           code: this archive could not be decoded (data NULL), the rest of the batch is unaffected */
    uint64_t first_bad_record;
} nafgpu_text;

/* After nafgpu_job_run: text of every archive of the job (sequence must have been decoded; FASTQ also needs quality). */
int nafgpu_job_format(nafgpu_ctx* ctx, int format, uint64_t line_length, nafgpu_text* out, uint32_t n);
/* prepare + run + format in one call. */
int nafgpu_format_batch(nafgpu_ctx* ctx, const nafgpu_archive* archives, uint32_t n, uint32_t want, int format,
                        uint64_t line_length, nafgpu_text* out);

/* ---- pipeline ----------------------------------------------------------------------------------------------------------
 * The reference seam is an iterator a consumer drives (Decoder::next, nafcodec/src/decoder/mod.rs:444-457); a device backend
 * called synchronously leaves the copy engines idle while kernels run.  A pipeline owns `lanes` contexts and host threads:
 * batches are submitted without waiting, and the H2D copy of one batch, the kernels of another and the D2H copy of a third
 * overlap.  Typical use (a collection of archives, cfg5): submit every sub-batch, then wait / consume / release in order.
 *   submit   returns a ticket (>= 0) at once; `archives` and the compressed bytes they point to are borrowed until wait returns
 *   wait     blocks until the ticket is decoded; `out` gets n results whose pointers stay valid until release
 *   release  hands the lane's pinned buffers back (a lane takes no new batch before its last ticket is released)
 * At most `lanes` tickets can be decoded-but-unreleased at a time; thread-safe. */
typedef struct nafgpu_pipeline nafgpu_pipeline;
int nafgpu_pipeline_create(int device, uint32_t lanes, nafgpu_pipeline** out);
void nafgpu_pipeline_destroy(nafgpu_pipeline* p);
int64_t nafgpu_pipeline_submit(nafgpu_pipeline* p, const nafgpu_archive* archives, uint32_t n, uint32_t want);
int nafgpu_pipeline_wait(nafgpu_pipeline* p, int64_t ticket, nafgpu_result* out, uint32_t n);
int nafgpu_pipeline_release(nafgpu_pipeline* p, int64_t ticket);
const char* nafgpu_pipeline_last_error(const nafgpu_pipeline* p);
uint32_t nafgpu_pipeline_lanes(const nafgpu_pipeline* p);
int nafgpu_pipeline_lane_stats(nafgpu_pipeline* p, uint32_t lane, nafgpu_job_stats* out);   /* sizes of the lane's last batch */


/* ---- encode side (SURVEY 8f rank 4) -----------------------------------------------------------------------------------
 * What the reference's writers compute per record before the bytes reach the zstd compressors, for all records of an
 * archive at once:
 *   SequenceWriter::encode / write / into_inner (nafcodec/src/encoder/writer.rs:21-90): IUPAC -> 4 bit, first residue in the
 *     LOW nibble, the odd-length `cache` carried into the next record, the last nibble padded with 0;
 *   write_length (nafcodec/src/encoder/mod.rs:37-44): u32 LE words, 0xFFFFFFFF continues a length;
 *   and the soft-mask extraction the reference never wrote (its mask writer is commented out, encoder/mod.rs:240, and
 *   SequenceWriter rejects lower case): with extract_mask the lower-case runs come back as the bytes of a Mask section in
 *   the format MaskReader decodes (decoder/reader.rs:196-231), and the residues are packed as their upper-case codes.
 * zstd compression of these streams stays with the caller (the CPU, as in the reference: encoder/mod.rs:147-154,365). */
typedef struct nafgpu_pack_input {
    const uint8_t* sequence;            /* HOST: the residues of all records, concatenated (ASCII) */
    const uint64_t* lengths;            /* HOST: n_records lengths; their sum must be n_residues (else Error::InvalidLength) */
    uint64_t n_records;
    uint64_t n_residues;
    int32_t sequence_type;              /* 0 dna ('T'), 1 rna ('U'); protein / text are written verbatim by the reference: not packed */
    int32_t extract_mask;               /* 0: lower case is "unexpected sequence character" like the reference; 1: see above */
} nafgpu_pack_input;

typedef struct nafgpu_pack_result {
    const uint8_t* packed;              /* HOST (pinned, owned by the context): (n_residues + 1) / 2 bytes of the Sequence stream */
    uint64_t packed_size;
    const uint8_t* length_words;        /* the Length stream: length_size bytes (4 per word) */
    uint64_t length_size;
    const uint8_t* mask;                /* the Mask stream (NULL without extract_mask): mask_size bytes, n_mask_runs runs */
    uint64_t mask_size;
    uint64_t n_mask_runs;
    uint64_t first_invalid;             /* UINT64_MAX, or the index (in the concatenation) of the first character SequenceWriter::encode
                                           rejects: Error::InvalidSequence (encoder/mod.rs:283-286); the call returns NAFGPU_ERR_INVALID_DATA */
} nafgpu_pack_result;

int nafgpu_pack(nafgpu_ctx* ctx, const nafgpu_pack_input* in, nafgpu_pack_result* out);

/* Device pointers of the last run's outputs, for callers that keep results in HBM (device-resident variant). */
int nafgpu_job_device_result(nafgpu_ctx* ctx, uint32_t archive, const uint8_t** sequence_dev, uint64_t* capacity_bytes);

/* ---- device-resident export -------------------------------------------------------------------------------------------
 * The decoded job, from the context's arena into DEVICE memory the caller owns, as tokens: every decoded byte goes through a
 * 256-entry table (identity = ASCII; the soft mask is the case of the ASCII).  Records are numbered across the job: archive 0's
 * n_lengths records first, then archive 1's, and so on; an archive whose status is nonzero contributes none.
 * After nafgpu_job_run; the job stays in device memory until the next prepare / run on the context, so one decode serves
 * any number of exports. */

/* Per-archive counters of the job that was run (read once per run: one small D2H and a synchronise, as for
 * nafgpu_job_fetch_window). */
typedef struct nafgpu_counts {
    uint64_t n_records, n_ids, n_comments, n_lengths, total_residues;
    uint64_t id_bytes, comment_bytes;     /* decoded size of the ids / comments streams: what a FLAT export of that field writes */
    uint64_t first_bad_record;            /* as in nafgpu_result */
    int32_t record_status, status;        /* as in nafgpu_result: a failed archive has status != 0 and contributes no records */
} nafgpu_counts;
int nafgpu_job_counts(nafgpu_ctx* ctx, nafgpu_counts* out, uint32_t n);

/* FLAT    one field of every archive, concatenated in job order: sequence / quality total_residues bytes per archive, ids /
 *         comments id_bytes / comment_bytes (NUL-terminated strings).  An archive without that section contributes no bytes.
 * ROWS    uint8 [n_rows, row_length]: row i holds residues [start, start + row_length) of job record `record` of the sequence or
 *         quality, for (record, start) = rows[2i], rows[2i + 1]; `pad` past the record's end.  A row whose record is out of
 *         range or lacks the field, or whose start is negative or not below the record's length, is all `pad`.
 * OFFSETS int64 [N + 1] job-global exclusive record offsets (N = the job's records); lengths are their differences. */
enum { NAFGPU_EXPORT_FLAT = 0, NAFGPU_EXPORT_ROWS = 1, NAFGPU_EXPORT_OFFSETS = 2 };
typedef struct nafgpu_export {
    int32_t field;                 /* NAFGPU_SEC_ID | _COMMENT | _SEQUENCE | _QUALITY (FLAT); _SEQUENCE | _QUALITY (ROWS); ignored (OFFSETS) */
    int32_t layout;
    uint8_t table[256];            /* out byte = table[decoded byte]; by value, so no copy and no lifetime */
    uint8_t pad;                   /* ROWS */
    uint8_t _pad[7];
    void* out;                     /* DEVICE memory of the caller (8-byte aligned for OFFSETS) */
    uint64_t out_bytes;            /* its capacity: checked against what the export writes */
    const int64_t* rows;           /* DEVICE, ROWS: n_rows (record, start) pairs */
    uint64_t n_rows, row_length;
} nafgpu_export;
/* Enqueues the export on `stream` (a cudaStream_t; NULL = the context's stream).  The kernels wait for the job's run (an event
 * on the context's stream), and the context's next call waits for them (an event on `stream`), so the caller may prepare
 * the next job right away.  Asynchronous: no host sync unless the counters have not been read for this run yet.
 * NAFGPU_ERR_ARGUMENT: no run, a field that was not requested (want bits), ROWS of ids / comments, out_bytes too small,
 * rows NULL with n_rows > 0.  An empty job, or an archive without records, exports zero bytes (OFFSETS: the one entry 0). */
int nafgpu_job_export(nafgpu_ctx* ctx, const nafgpu_export* spec, void* stream);

/* ---- pipeline device tickets ------------------------------------------------------------------------------------------
 * The pipeline's lanes, but the decoded sub-batch stays in the lane's device arena, for consumers on the GPU (the
 * nafgpu_job_export surface above, per ticket).  Host and device tickets may be interleaved on one pipeline; at most `lanes`
 * tickets of either kind are decoded-but-unreleased at a time.
 *   submit_device  as nafgpu_pipeline_submit; the lane runs prepare + run + nafgpu_job_counts and copies no result back
 *   wait_counts    blocks until the ticket is decoded; `out` gets n per-archive counters, as nafgpu_job_counts.  `archives` and
 *                  the bytes they point to are borrowed until it returns (the counters' read synchronises the lane's stream,
 *                  so the sub-batch's H2D has completed).  A corrupt archive only sets its own out[i].status (it contributes
 *                  no records); a CUDA, memory or argument failure of the sub-batch is the return value
 *   export         nafgpu_job_export on the ticket's lane: same spec, same stream semantics, same errors.  Exports of one
 *                  ticket may come from several threads (they take turns on a per-lane mutex)
 *   release        (nafgpu_pipeline_release, for both kinds) hands the lane back.  The lane's next prepare is enqueued on its
 *                  context's stream, which waits for every export already enqueued from the ticket, so releasing right after
 *                  an export on another stream is safe
 * NAFGPU_ERR_ARGUMENT with a message in nafgpu_pipeline_last_error: nafgpu_pipeline_wait on a device ticket, wait_counts on a
 * host ticket, an export from a ticket that was not waited for, whose decode failed, or that was released. */
int64_t nafgpu_pipeline_submit_device(nafgpu_pipeline* p, const nafgpu_archive* archives, uint32_t n, uint32_t want);
int nafgpu_pipeline_wait_counts(nafgpu_pipeline* p, int64_t ticket, nafgpu_counts* out, uint32_t n);
int nafgpu_pipeline_export(nafgpu_pipeline* p, int64_t ticket, const nafgpu_export* spec, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NAFGPU_H */

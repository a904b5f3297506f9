// naf_kernels.cuh -- the NAF layer on the device: what nafcodec/src/decoder/reader.rs and Decoder::mask_sequence
// (decoder/mod.rs:402-441) compute per record on the CPU, restated as whole-archive data-parallel kernels.
#pragma once
#include "cuda_compat.h"
#include <stdint.h>

namespace nk {

enum : uint32_t { HAS_IDS = 1, HAS_COMMENTS = 2, HAS_LENGTHS = 4, HAS_MASK = 8, HAS_SEQUENCE = 16, HAS_QUALITY = 32 };

constexpr uint32_t UNPACK_T = 256;                     // threads of an unpack CTA
constexpr uint32_t UNPACK_W = 2;                       // adjacent mask words (of 32 residues) per thread
constexpr uint32_t CHUNK_WORDS = UNPACK_W * UNPACK_T;  // mask words per unpack CTA
constexpr uint32_t CHUNK_RESIDUES = CHUNK_WORDS * 32;
constexpr uint64_t NO_RECORD = ~0ull;
constexpr uint32_t NAF_SLICE = 32768;                  // section bytes per CTA of k_naf_scan (ids, comments, lengths, mask alike)
constexpr uint32_t NAF_AGG_BYTES = 16;                 // per (archive, task, slice) when a job has more than one slice: (count, sum)

// Per-archive counters, device-written, copied back with the results (80 bytes).
struct NafCounts {
    uint64_t n_ids;            // NUL-terminated strings found in the ids stream
    uint64_t n_comments;
    uint64_t n_lengths;        // lengths available for records (min(#terminated lengths, n_records))
    uint64_t total_residues;   // sum of those lengths == bytes of sequence / quality output
    uint64_t n_mask_runs;
    uint64_t mask_sum;
    uint64_t first_bad_record; // first record whose text failed UTF-8 validation (NO_RECORD if none)
    uint64_t nonascii;         // bit f set: field f (0 ids, 1 comments, 2 text sequence, 3 quality) has bytes >= 0x80
    uint64_t status;           // zc::E_* bits raised by the NAF kernels for THIS archive (the job-wide word keeps their OR)
    uint64_t _pad;
};

// One per archive of the job.  All *_off fields are byte offsets into the job arena (16 B aligned at least).
struct NafDev {
    uint64_t n_records;
    uint32_t seq_type;         // 0 dna, 1 rna, 2 protein, 3 text (data.rs:56-62)
    uint32_t has;              // HAS_* bits: sections that were decoded
    uint64_t seq_residues;     // Sequence section original_size (residues; bytes for protein/text)
    uint64_t ids_off, ids_size, com_off, com_size, len_off, len_size, mask_off, mask_size;
    uint64_t seq_off, seq_size, qual_off, qual_size;
    uint64_t counts_off, id_offsets_off, com_offsets_off, lengths_off, rec_offsets_off, ascii_off;
    uint64_t mask_bits_off, mask_bounds_off, chunk_par_off;
    uint32_t n_chunks;         // ceil((seq_residues + 1) / CHUNK_RESIDUES) when sequence is decoded
    uint32_t _pad;
};

// Enqueues the NAF stage for n_archives archives on `stream`.  max_* are maxima over the archives (grid sizing).
// max_scan_bytes: largest ids / comments / lengths / mask section of the job; scan_agg: n_archives x 4 x slices x NAF_AGG_BYTES of
// scratch when that is more than one NAF_SLICE.  Returns the number of kernels launched; `ev` (optional) gets one mark per stage (NAF_STAGES).
// any_mask: some archive decodes sequence + mask; any_text_mask: one of those is protein/text.  sms: the device's multiprocessors.
int launch_naf_stage(uint8_t* arena, const NafDev* archives_dev, uint32_t n_archives, uint64_t max_records, uint64_t max_scan_bytes, void* scan_agg,
                     uint32_t max_chunks, uint64_t max_text_bytes, bool any_mask, bool any_text_mask, uint32_t* status, uint32_t sms,
                     cudaStream_t stream, StageEvents* ev);
constexpr int NAF_STAGES = 5;

}  // namespace nk

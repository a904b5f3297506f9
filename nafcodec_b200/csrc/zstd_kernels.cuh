// zstd_kernels.cuh -- device-side view of a decode job and the launch entry points of the zstd stage.
#pragma once
#include "cuda_compat.h"
#include <stddef.h>
#include <stdint.h>

#include <optional>

#include "zstd_core.cuh"
#include "zstd_format.h"

namespace fw { struct JobPlan; }

namespace zk {

constexpr uint32_t HUF_SMALL_SYMBOLS = 2048;   // blocks whose streams regenerate <= this many symbols each go to the four-warp kernel

// Everything the zstd kernels need, by value.  All pointers are device pointers.
struct JobDev {
    const uint8_t* comp;              // compressed sections, each frame 16 B aligned, COMP_PAD slack at the end
    uint8_t* out;                     // regenerated sections (frame f at frames[f].dst_off)
    uint8_t* lit;                     // literal staging for blocks with Huffman literals AND sequences
    const zf::FrameDesc* frames;
    const zf::BlockDesc* blocks;
    zf::BlockState* bstate;
    zc::SeqCell* tables;              // n_slots * FSE_SLOT_CELLS
    uint8_t* table_al;                // accuracy log per slot
    uint8_t* huf_weights;             // n_huf_slots x 256 weights (k_build_tables decodes every tree description once)
    uint8_t* huf_meta;                // n_huf_slots x {n_symbols - 1, max_bits}; max_bits == 0: bad tree
    zf::SeqRec* seq;                  // one 32-byte record per sequence (written by k_decode_sequences / k_lz_literals)
    uint32_t lz_small;                // nonzero: the match stage runs in one CTA (k_lz_small): at most 8192 matches, arena below 4 GB
    uint32_t tiny_blocks;             // nonzero: blocks of at most 32 sequences / 2 KiB of literals go through the warp-per-block kernels
    const uint32_t* seq_big_list;     // with tiny_blocks: the blocks k_decode_sequences takes (more than 32 sequences), host-built
    const uint32_t* lit_big_list;     // with tiny_blocks: the blocks k_lz_literals takes
    uint32_t n_seq_big, n_lit_big;
    uint32_t seq_stage_bytes;         // shared-memory staging size of k_decode_sequences (largest sequence bitstream, capped)
    uint32_t* seq_done;               // 0 = pending, else the pass that executed the match
    uint32_t* lz_idx;                 // per frame, per 4 KB of output: first match ending after the start of the cell (k_lz_index)
    uint32_t* lz_blocker;             // per match: the unfinished match it was last found waiting for (0xFFFFFFFF: none yet)
    uint32_t* frame_bad;              // per frame: non-zero once anything in it failed validation
    uint32_t* status;                 // OR of zc::E_* bits
    unsigned long long* debug_seq;    // optional cycle accounting of k_decode_sequences and k_lz_small (8 counters), else null
    uint32_t* lz_list[3];             // rotating worklists of matches still pending (n_seq entries each)
    uint32_t* lz_count;               // [3] their lengths
    uint32_t* lz_rounds;              // rounds k_lz_first + k_lz_resolve ran (statistics)
    uint32_t* lz_handover;            // set by k_lz_resolve when it leaves work to k_lz_finish
    uint32_t* lz_flow;                // [0] set by k_lz_resolve: k_lz_flow takes the rest; [1] its ticket counter; [2] its abort flag
    uint32_t lz_flow_early;           // host: k_lz_flow also runs before the rounds (jobs of 2 K .. 64 K matches), words [3] ticket, [4] abort
    uint32_t lz_flow_on, flow_ctas;   // host: launch configuration: launch k_lz_flow (jobs with more than a few thousand matches); its grid
    uint32_t* lz_pending;             // [24] matches still pending after round 1, 2, ... (statistics)
    uint32_t coop_ctas;               // host: launch configuration: co-resident CTAs for k_lz_resolve's grid barrier
    uint32_t fin_cost_us;             // estimated cost of the finisher kernels on this job (hand-over decision)
    // finisher (k_lz_finish, k_lz_finish2): the frames cut into 64 KB chunks
    const uint32_t* fin_chunk_first;  // [n_frames + 1] first chunk of every frame (host-filled)
    uint32_t fin_total_chunks;
    uint32_t fin_ctas, fin2_ctas;     // host: launch configuration: grid sizes (one CTA per SM; co-resident CTAs of the cooperative level 2)
    uint32_t* fin_g;                  // one u32 per byte of every frame: distance of an unresolved byte to its source, 0 = final
    uint32_t* fin_ext;                // [fin_total_chunks x 2048] bitmap of a chunk's external roots (written by level 1 for chunks it flags)
    const uint64_t* fin_g_base;       // [n_frames] first entry of every frame in fin_g (host-filled; frames are packed, 16-entry aligned)
    uint32_t* fin_chunk_flag;         // [fin_total_chunks] chunk has unresolved bytes (zeroed every run)
    uint32_t* fin_unresolved;         // unresolved bytes after level 1
    uint32_t* fin_count;              // [3] rotating per-round counters of level 2
    const zf::HufItem* huf_items;     // one per Huffman bitstream
    uint32_t* huf_bounds;             // [n_huf_big x 256] k_huf_scout -> k_huf_decode_block: output offset << 4 | start offset of every range
    uint32_t huf_block_min;           // host: launch configuration: jobs with at least this many big blocks use k_huf_decode_block (0: default)
    uint32_t n_huf_items, n_huf_big;  // items [0, n_huf_big): streams of 4-stream blocks, four per block (k_huf_scout + k_huf_decode_block, or k_huf_decode_big); the rest: k_huf_decode_small
    uint32_t max_huf_stream, max_huf_small;   // largest stream (bytes) in each class
    const zf::FsTile* fs_tiles;       // tiles of the frames with more than FS_BIG_FRAME blocks (host-filled)
    const zf::FsBigFrame* fs_big;
    zf::FsTileState* fs_state;
    uint32_t n_fs_tiles, n_fs_big;
    uint32_t fs_big_frame;            // frames with more blocks than this are scanned by tiles
    uint32_t n_frames, n_blocks, n_slots;
    uint32_t n_checksums;             // frames with a content checksum (k_frame_checksum runs only if any)
    uint64_t n_seq;
};

// The job's counter words: one device allocation, zeroed before every run and copied back with the results.  The fixed part
// comes first; behind it, two tails whose lengths depend on the job: frame_bad[n_frames], then fin_chunk_flag[fin_total_chunks].
struct JobWords {
    uint32_t status;                  // JobDev::status
    uint32_t lz_count[3];
    uint32_t lz_handover, lz_rounds, fin_unresolved;
    uint32_t fin_count[3];
    uint32_t lz_flow[8];              // k_lz_flow: [0] the rounds' hand-over, [1] ticket, [2] abort; [3] early ticket, [4] early abort
    uint32_t lz_pending[24];
    uint32_t* frame_bad() { return reinterpret_cast<uint32_t*>(this + 1); }
    const uint32_t* frame_bad() const { return reinterpret_cast<const uint32_t*>(this + 1); }
    uint32_t* fin_chunk_flag(size_t n_frames) { return frame_bad() + n_frames; }
    static size_t words(size_t n_frames, size_t chunks) { return sizeof(JobWords) / 4 + n_frames + chunks; }
};
static_assert(sizeof(JobWords) == 42 * 4, "JobWords: 42 fixed words");

// Test and probe overrides, from the environment.  Read once per nafgpu_job_prepare / nafgpu_zstd_decompress (not once per
// process: tests change them between calls).  Unset, the job's own size decides.
//   NAFGPU_TINY_BLOCKS=n      n != 0: the warp-per-block kernels for tiny blocks; 0: never (default: 4096+ tiny blocks)
//                             test_parity, test_zstd_sequences, test_job_plan
//   NAFGPU_LZ_SMALL=n         k_lz_small for jobs of at most n matches, n clamped to [0, 8192] (default 2048).  Set at all, it
//                             also turns the early k_lz_flow off, so that tests forcing the general rounds keep them.
//                             test_parity, test_zstd_sequences, test_job_plan
//   NAFGPU_LZ_FLOW=n          0: never k_lz_flow after the rounds; 2: whenever the rounds would go on (default: 8192+ matches)
//                             test_parity
//   NAFGPU_LZ_FLOW_EARLY=n    n != 0: k_lz_flow also before the rounds; 0: never (default: 2 K .. 64 K matches)
//                             test_parity, test_job_plan
//   NAFGPU_FIN_COST_US=us     the finisher's estimated cost, which sets the rounds' hand-over deadline (probing: 100000000
//                             never hands over)                                                     test_parity
//   NAFGPU_HUF_BLOCK_MIN=n    k_huf_decode_block from n big blocks on, n >= 1 (default 296)
//                             test_parity, test_zstd_sequences, test_job_plan
//   NAFGPU_FS_TILE=n          frame scan tiles of n >= 1 blocks, for frames of more than 2n (default FS_TILE, FS_BIG_FRAME)
//                             test_parity, test_zstd_sequences, test_job_plan
//   NAFGPU_WALK_SPLIT=n       n > 0: walk sections in parts of n blocks, even short ones; n <= 0: never in parts
//                             test_parity, test_zstd_sequences, test_job_plan
//   NAFGPU_DEBUG_HUF          any value: cycle counters of k_decode_sequences and k_lz_small on stderr at fetch (tools/lat_debug.py)
//   NAFGPU_DEBUG_PREP         any value: phase times of the job's preparation on stderr (tools/prep_probe.py)
struct Overrides {
    std::optional<uint32_t> tiny_blocks, lz_small, lz_flow, lz_flow_early, fin_cost_us, huf_block_min, fs_tile;
    std::optional<int> walk_split;
    bool debug_huf = false, debug_prep = false;
};

// Every path decision of the zstd stage that launch_zstd_stage does not find in JobDev: grids, shared memory, kernel shapes.
struct Launch {
    bool huf_side = false;            // small Huffman streams beside the big ones (given a third stream)
    bool huf_per_block = false;       // big streams: k_huf_decode_block (one CTA per block) rather than k_huf_decode_big
    uint32_t huf_small_smem = 0, huf_big_smem = 0, huf_scout_smem = 0;
    bool seq_side = false;            // k_decode_sequences beside the tiny blocks' kernel (given a third stream)
    uint32_t lit_blocks = 0, lit_split = 0;   // k_lz_literals grid (blocks x split); lit_few: the <4> shape
    bool lit_few = false;
    uint32_t lz_small_smem = 0;
    uint32_t first_ctas = 0, resolve_ctas = 0;    // k_lz_first; k_lz_resolve (cooperative)
    bool finish = false;              // the finisher kernels run
    uint32_t finish_ctas = 0, finish2_ctas = 0;   // k_lz_finish; k_lz_finish2 (cooperative)
};

// The context's streams and the fork / join events that order them: `st` carries the job; st2 the Huffman branch beside the
// FSE branch (pair 0); st3 the small Huffman streams beside the big ones (pair 1) and the general sequence kernel beside the
// tiny blocks' (pair 2).
struct Streams {
    cudaStream_t st = 0, st2 = 0, st3 = 0;
    cudaEvent_t fork[3] = {nullptr, nullptr, nullptr}, join[3] = {nullptr, nullptr, nullptr};
    bool create();
    void destroy();
};

// Sets the path choices of a job in J (tiny_blocks, lz_small, seq_stage_bytes, the lz_flow fields, fin_cost_us, huf_block_min)
// and returns the rest.  J's counts, coop_ctas and fin_* must be set.  `sms`: the device's multiprocessor count.
Launch choose_paths(JobDev& J, const fw::JobPlan& plan, const Overrides& ov, uint32_t sms, uint64_t arena_size);
// Enqueues the whole zstd stage for a job (no host synchronisation); returns the number of kernels launched.  `ev` (optional)
// gets one mark per stage (ZSTD_STAGES); a profiled run is serial, on S.st alone, so that every stage has its own interval.
int launch_zstd_stage(const JobDev& J, const Launch& L, const Streams& S, StageEvents* ev);
// Co-resident CTAs (whole device) for the cooperative match-resolution kernel.
uint32_t lz_resolve_max_ctas(int device);
void lz_finish_ctas(int device, uint32_t* level1, uint32_t* level2);
constexpr int ZSTD_STAGES = 8;

}  // namespace zk

// nafgpu_api.cu -- the extern "C" layer of include/nafgpu.h: context, job planning (arena layout + host frame
// walk), stream orchestration, result marshalling.  The reference-side seam it stands behind is the generic
// reader parameter of nafcodec/src/decoder/reader.rs instantiated with ZstdDecoder in setup_block!
// (nafcodec/src/decoder/mod.rs:32,218-226) and consumed by next_record / mask_sequence (mod.rs:356-441).
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <memory>
#include <mutex>
#include <optional>
#include <thread>
#include <string>
#include <vector>

#include "../../include/nafgpu.h"
#include "cuda_compat.h"
#include "frame_walk.h"
#include "naf_export.cuh"
#include "naf_kernels.cuh"
#include "naf_pack.cuh"
#include "naf_text.cuh"
#include "zstd_kernels.cuh"

namespace {

constexpr uint64_t ALIGN = 128;
inline uint64_t align_up(uint64_t v, uint64_t a = ALIGN) { return (v + a - 1) / a * a; }
constexpr int N_STAGES = zk::ZSTD_STAGES + nk::NAF_STAGES;
constexpr size_t FLUSH_BYTES = 256u << 20;          // > 126 MB L2

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool ensure(size_t n) {
        if (n <= cap) return true;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 256;
        if (cudaMalloc(&p, want) != cudaSuccess) { p = nullptr; cudaGetLastError(); return false; }
        cap = want;
        return true;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    ~DevBuf() { release(); }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool ensure(size_t n) {
        if (n <= cap) return true;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 256;
        if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { p = nullptr; cudaGetLastError(); return false; }
        cap = want;
        return true;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    ~PinBuf() { release(); }
};

struct ArchPlan {
    uint64_t n_records = 0;
    bool dec[6] = {false, false, false, false, false, false};
    uint64_t blob_off[6] = {0, 0, 0, 0, 0, 0};   // arena offset of each regenerated section
    uint64_t blob_size[6] = {0, 0, 0, 0, 0, 0};
    bool nucleotide = true;
    uint64_t line_length = 0;                    // Header::line_length / name_separator (data.rs:198-236): for the text formatter
    uint32_t sep = ' ';
    uint32_t first_frame = 0, n_frames = 0;      // the archive's frames in the job plan (per-archive status)
    int host_status = 0;                         // failure found on the host (frame walk, validation): the archive is not decoded
    std::string host_msg;
};

// One compressed section (= one zstd frame) of the job: at comp_off in `comp`, regenerating dst_size bytes at dst_off in the arena.
struct Section { uint32_t arch = 0; int sec = 0; const uint8_t* data = nullptr; uint64_t comp_off = 0, comp_size = 0, dst_off = 0, dst_size = 0; };

// A section in the header walk's first pass: the chain of its block headers, cut every so many blocks when it is long.
struct SecRef : Section { std::vector<uint64_t> cuts; uint64_t n_blocks = 0; int chain_rc = 0; std::string chain_err; };

// One section, or part of one, walked into its own plan, so that the sections of a job can be walked by several host threads
// (a FASTQ archive flushed per record has 10^6 block headers per section: 30 ns each on one core was as long as the whole
// device decode); the plans are then laid end to end, block descriptors going straight into the pinned staging buffer with
// their indices rebased.
struct WalkTask : Section {
    fw::JobPlan plan;
    int rc = 0;
    std::string err;
    bool live = true;
    size_t bo = 0;                     // first block of the task among the job's blocks
    uint32_t so = 0, slot_off = 0, ho = 0;
    uint64_t lo = 0;
    // a long section walked in parts (frame_walk.h): [p_begin, p_end) of the frame, and what the part inherits from the parts
    // before it: the task that last defined a Huffman tree / an FSE table of each kind (-1: none, -2: a predefined table) and the
    // index there; made absolute (abs_*) once the tasks' offsets are known
    uint64_t p_begin = 0, p_end = 0;
    bool first = true, last = true, heavy = false;
    fw::RangeState st;
    int carry_huf_task = -1, carry_tbl_task[3] = {-1, -1, -1};
    uint32_t carry_huf_block = 0, carry_huf_slot = 0, carry_tbl_slot[3] = {0, 0, 0};
    uint32_t abs_huf_block = zf::NO_BLOCK, abs_huf_slot = 0, abs_tbl[3] = {zf::NO_SLOT, zf::NO_SLOT, zf::NO_SLOT};

    // Starts the task afresh on [begin, end) of section S (0, 0: all of it): nothing walked, nothing inherited yet.
    void start(const Section& S, bool first_part, bool last_part, uint64_t begin = 0, uint64_t end = 0, bool heavy_part = false) {
        static_cast<Section&>(*this) = S;
        plan.clear(); rc = 0; err.clear(); live = true;
        first = first_part; last = last_part; p_begin = begin; p_end = end; heavy = heavy_part;
        carry_huf_task = -1; carry_tbl_task[0] = carry_tbl_task[1] = carry_tbl_task[2] = -1;
        abs_huf_block = zf::NO_BLOCK; abs_tbl[0] = abs_tbl[1] = abs_tbl[2] = zf::NO_SLOT;
    }
};

// Phase times of the job's preparation on stderr (NAFGPU_DEBUG_PREP)
struct PrepClock {
    bool on;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(const char* what) {
        if (!on) return;
        const auto n = std::chrono::steady_clock::now();
        fprintf(stderr, "[prepare] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
        t = n;
    }
};

// A block descriptor goes to the pinned staging buffer with non-temporal stores where the host has them: the buffer is written
// once and read by the copy engine, and a cached store would first read every line it overwrites (160 MB of descriptors for a
// 10^6-read FASTQ archive: 6.3 ms on 8 threads with plain stores).
static_assert(sizeof(zf::BlockDesc) % 16 == 0, "store_desc writes 16 bytes at a time");
#if defined(__SSE2__) && !defined(__CUDA_ARCH__)
inline void store_desc(zf::BlockDesc* dst, const zf::BlockDesc& b) {
    if (((uintptr_t)dst & 15) == 0) {
        const __m128i* s = (const __m128i*)&b;
        __m128i* d = (__m128i*)dst;
        for (size_t k = 0; k < sizeof(zf::BlockDesc) / 16; k++) _mm_stream_si128(d + k, _mm_loadu_si128(s + k));
    } else {
        *dst = b;
    }
}
inline void desc_fence() { _mm_sfence(); }
#else
inline void store_desc(zf::BlockDesc* dst, const zf::BlockDesc& b) { *dst = b; }
inline void desc_fence() {}
#endif

// Host threads a big job may use for its header walk and descriptor copy: three quarters of the cores, at most 12, less what the
// other contexts of the process (the lanes of a pipeline) are using at this moment; never fewer than one.
static std::atomic<int> g_helpers_busy{0};
struct HelperLease {
    unsigned n = 1;
    HelperLease() {
        const int hw = (int)std::max(1u, std::thread::hardware_concurrency());
        const int cap = std::min(12, std::max(1, hw * 3 / 4));
        const int got = std::max(1, std::min(cap, hw - g_helpers_busy.load(std::memory_order_relaxed)));
        g_helpers_busy.fetch_add(got, std::memory_order_relaxed);
        n = (unsigned)got;
    }
    ~HelperLease() { g_helpers_busy.fetch_sub((int)n, std::memory_order_relaxed); }
    HelperLease(const HelperLease&) = delete;
    HelperLease& operator=(const HelperLease&) = delete;
};

// fn(i) for i in [0, n) on up to `max_threads` host threads (inline when that is one).
template <class F>
void parallel_for(size_t n, unsigned max_threads, F fn) {
    if (n <= 1 || max_threads <= 1) { for (size_t i = 0; i < n; i++) fn(i); return; }
    const unsigned w = (unsigned)std::min<size_t>(n, max_threads);
    std::atomic<size_t> next{0};
    auto body = [&] { for (;;) { const size_t i = next.fetch_add(1); if (i >= n) return; fn(i); } };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < w; t++) th.emplace_back(body);
    body();
    for (std::thread& t : th) t.join();
}

}  // namespace

struct nafgpu_ctx {
    int device = 0;
    uint32_t sms = 1;                  // the device's multiprocessors (grid sizes)
    zk::Streams streams;
    cudaEvent_t ev_block = nullptr, ev_d2h = nullptr;
    std::string err;
    DevBuf comp, arena, lit, desc, bstate, hufw, fsstate, lzidx, scanagg, debug, tables, table_al, seq32, seq64, misc, flush, text, fin_g, pack_in, pack_out;
    size_t o_frames = 0, o_naf = 0, o_huf = 0, o_chunks = 0, o_gbase = 0, o_tiles = 0, o_big = 0, o_bigseq = 0, o_biglit = 0;   // layout of `desc` (blocks at 0): one H2D copy for all descriptors
    PinBuf stage, result, misc_host, text_host, text_stage, pack_host;
    fw::JobPlan plan;                  // frames, Huffman items and totals of the job (block descriptors live in the tasks)
    std::vector<WalkTask> tasks;       // [0, n_tasks) belong to the current job
    size_t n_tasks = 0;
    std::vector<nk::NafDev> arch;
    std::vector<ArchPlan> aplan;
    zk::JobDev J;
    zk::Launch launch;                 // path choices of the prepared job that JobDev does not hold
    uint64_t z1_size = 0, z2_off = 0, z2_size = 0, arena_size = 0, counts_size = 0;
    uint64_t max_records = 0, max_text = 0, max_mask = 0, max_scan = 0;
    uint32_t max_chunks = 0;
    bool any_mask = false, any_text_mask = false;
    size_t misc_words = 0;             // zk::JobWords of the prepared job, in `misc` and `misc_host`
    nafgpu_job_stats stats;
    bool prepared = false, ran = false;
    bool win_counts = false;           // counts + status of the last run are on the host (windowed fetch)
    PinBuf win;                        // the current window of a job that is read in windows (nafgpu_job_fetch_window)
    uint32_t want = 0;                 // the want bits of the prepared job
    // device-resident export (nafgpu_job_export): the archives' counters and the export descriptors of the last run, built and
    // uploaded once per run by the first export: [ExpRec x n_exp_rec | ExpSpan x n_exp_span[f] for ids, comments, sequence, quality]
    bool exp_ready = false;
    std::vector<nafgpu_counts> counts;
    DevBuf exp_desc;
    PinBuf exp_stage;
    uint32_t n_exp_rec = 0, n_exp_span[4] = {0, 0, 0, 0};
    uint64_t o_exp_span[4] = {0, 0, 0, 0}, exp_bytes[4] = {0, 0, 0, 0}, exp_records = 0, exp_residues = 0;
    cudaEvent_t ev_exp_ready = nullptr, ev_exp_done = nullptr;
    cudaEvent_t ev[N_STAGES + 3];
    bool ev_ok = false;
#if !defined(NAFGPU_EMULATE)
    cudaGraphExec_t graph = nullptr;
#endif
};

namespace {

int fail(nafgpu_ctx* c, int code, const std::string& msg) {
    c->err = msg;
    return code;
}

#define CUDA_TRY(c, expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
    char _b[256]; snprintf(_b, sizeof _b, "%s failed: %s", #expr, cudaGetErrorString(_e)); return fail((c), NAFGPU_ERR_CUDA, _b); } } while (0)

void drop_graph(nafgpu_ctx* c) {
#if !defined(NAFGPU_EMULATE)
    if (c->graph) { cudaGraphExecDestroy(c->graph); c->graph = nullptr; }
#else
    (void)c;
#endif
}

// Enqueue one full decode of the prepared job.
int enqueue_run(nafgpu_ctx* c, StageEvents* ev) {
    cudaStream_t st = c->streams.st;
    CUDA_TRY(c, cudaMemsetAsync(c->misc.p, 0, c->misc_words * 4, st));
    if (c->J.n_seq && !c->J.lz_small) {             // (k_lz_small keeps these in shared memory and writes seq_done itself)
        CUDA_TRY(c, cudaMemsetAsync(c->J.seq_done, 0, c->J.n_seq * 4, st));
        CUDA_TRY(c, cudaMemsetAsync(c->J.lz_blocker, 0xFF, c->J.n_seq * 4, st));
    }
    CUDA_TRY(c, cudaMemsetAsync(c->arena.p, 0, c->counts_size, st));
    if (c->z2_size) CUDA_TRY(c, cudaMemsetAsync((uint8_t*)c->arena.p + c->z2_off, 0, c->z2_size, st));
    int launches = zk::launch_zstd_stage(c->J, c->launch, c->streams, ev);
    launches += nk::launch_naf_stage((uint8_t*)c->arena.p, (const nk::NafDev*)((const uint8_t*)c->desc.p + c->o_naf), (uint32_t)c->arch.size(), c->max_records, c->max_scan, c->scanagg.p,
                                     c->max_chunks, c->max_text, c->any_mask, c->any_text_mask, c->J.status, c->sms, st, ev);
    c->stats.kernel_launches = (uint32_t)launches;
    CUDA_TRY(c, cudaGetLastError());
    c->ran = true;
    c->win_counts = false;
    c->exp_ready = false;
    return NAFGPU_OK;
}

// The host copy of the job's counter words (misc_host), as the last copy back left them.
const zk::JobWords& words(const nafgpu_ctx* c) { return *(const zk::JobWords*)c->misc_host.p; }

void read_lz_stats(nafgpu_ctx* c) {
    const zk::JobWords& w = words(c);
    c->stats.lz_handover = w.lz_handover; c->stats.lz_rounds = w.lz_rounds; c->stats.lz_unresolved = w.fin_unresolved;
    c->stats.lz_flow = w.lz_flow[0] | ((c->J.lz_flow_early && w.lz_flow[4] == 0) ? 2u : 0u);   // bit 0: chosen by the rounds; bit 1: ran before them to the end
    memcpy(c->stats.lz_pending, w.lz_pending, sizeof w.lz_pending);
}

int status_to_code(uint32_t s, std::string& msg) {
    using namespace zc;
    if (s == 0) return NAFGPU_OK;
    char b[96];
    snprintf(b, sizeof b, " (device status 0x%x)", s);
    if (s & (E_FSE_TABLE | E_HUF_TREE | E_HUF_STREAM | E_SEQ_STREAM | E_LITERALS | E_OFFSET | E_NO_TABLE | E_INTERNAL)) {
        msg = std::string("corrupt zstd stream") + b; return NAFGPU_ERR_INVALID_DATA;
    }
    if (s & E_CHECKSUM) { msg = std::string("zstd frame checksum mismatch") + b; return NAFGPU_ERR_INVALID_DATA; }
    if (s & E_SIZE) { msg = std::string("section does not regenerate the size its header states") + b; return NAFGPU_ERR_INVALID_DATA; }
    if (s & E_LENGTHS) { msg = std::string("record lengths exceed the sequence/quality stream") + b; return NAFGPU_ERR_UNEXPECTED_EOF; }
    if (s & E_MASK) { msg = std::string("failed to get mask unit") + b; return NAFGPU_ERR_UNEXPECTED_EOF; }
    if (s & E_NUL) { msg = std::string("id/comment stream is not NUL terminated") + b; return NAFGPU_ERR_INVALID_DATA; }
    if (s & E_UTF8) { msg = std::string("invalid utf-8") + b; return NAFGPU_ERR_UTF8; }
    msg = std::string("unknown device status") + b;
    return NAFGPU_ERR_INVALID_DATA;
}

// Result copies of concurrent contexts on one device take turns.  Issued together they share the PCIe link, every lane
// finishes at the same time, and all of them then walk headers and run kernels together while the copy engine idles
// (measured: 8.2 ms per 320 MB step whatever the number of lanes).  One at a time each copy runs at the full rate and
// the lanes stay staggered, so the link is always busy (tools/e2e_probe.py).
static std::mutex g_d2h_turn[16];

// Waiting for the context's stream.  A big job waits on an event created with cudaEventBlockingSync: the thread sleeps
// instead of spinning.  With 8 GPUs x 4 lanes on a 32-vCPU host, 32 threads spinning in cudaStreamSynchronize next to the
// header walks halved the end-to-end rate per GPU (round 1: 49.5 -> 11 GB/s per GPU at N = 8).  Small jobs keep spinning:
// a wake-up costs tens of microseconds, which is the whole decode of a 5 Mbp archive.
static cudaError_t wait_stream(nafgpu_ctx* c) {
    if (c->z1_size < (8u << 20) || !c->ev_block) return cudaStreamSynchronize(c->streams.st);
    cudaError_t e = cudaEventRecord(c->ev_block, c->streams.st);
    return e != cudaSuccess ? e : cudaEventSynchronize(c->ev_block);
}

// The turns are taken on the DEVICE: a lane enqueues its copy behind the previous lane's (an event of that lane's stream), so the
// copy engine goes from one result to the next without waiting for a host thread to wake up, release a lock and enqueue
// (blocking-sync wake-ups cost tens of microseconds each).  The mutex only orders the enqueues.
static cudaEvent_t g_last_d2h[16];

static int d2h_results(nafgpu_ctx* c) {
    if (!c->result.ensure(c->z1_size + 64)) return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
    c->win_counts = false;
    CUDA_TRY(c, wait_stream(c));                                // kernels first: a copy queued behind running kernels would hold up the lanes behind it
    {
        std::lock_guard<std::mutex> turn(g_d2h_turn[c->device & 15]);
        cudaEvent_t prev = g_last_d2h[c->device & 15];
        if (prev && prev != c->ev_d2h && c->ev_d2h) CUDA_TRY(c, cudaStreamWaitEvent(c->streams.st, prev, 0));
        CUDA_TRY(c, cudaMemcpyAsync(c->misc_host.p, c->misc.p, c->misc_words * 4, cudaMemcpyDeviceToHost, c->streams.st));
        CUDA_TRY(c, cudaMemcpyAsync(c->result.p, c->arena.p, c->z1_size, cudaMemcpyDeviceToHost, c->streams.st));
        if (c->ev_d2h) { CUDA_TRY(c, cudaEventRecord(c->ev_d2h, c->streams.st)); g_last_d2h[c->device & 15] = c->ev_d2h; }
        else { CUDA_TRY(c, wait_stream(c)); return NAFGPU_OK; }   // (no event: the old way, the turn held until the copy is done)
    }
    CUDA_TRY(c, wait_stream(c));
    return NAFGPU_OK;
}

struct Copy { const uint8_t* src; uint64_t dst, size; };

// NAFGPU_* test and probe overrides (zstd_kernels.cuh, zk::Overrides: what each one forces): the one place that reads them.
zk::Overrides read_overrides() {
    const auto num = [](const char* name) -> std::optional<int> {
        const char* e = getenv(name);
        return e ? std::optional<int>(atoi(e)) : std::nullopt;
    };
    zk::Overrides o;
    if (const auto v = num("NAFGPU_TINY_BLOCKS")) o.tiny_blocks = (uint32_t)*v;
    if (const auto v = num("NAFGPU_LZ_SMALL")) o.lz_small = (uint32_t)std::min(8192, std::max(0, *v));
    if (const auto v = num("NAFGPU_LZ_FLOW")) o.lz_flow = (uint32_t)*v;
    if (const auto v = num("NAFGPU_LZ_FLOW_EARLY")) o.lz_flow_early = (uint32_t)*v;
    if (const auto v = num("NAFGPU_FIN_COST_US")) o.fin_cost_us = (uint32_t)*v;
    if (const auto v = num("NAFGPU_HUF_BLOCK_MIN")) o.huf_block_min = (uint32_t)std::max(1, *v);
    if (const auto v = num("NAFGPU_FS_TILE")) o.fs_tile = (uint32_t)std::max(1, *v);
    o.walk_split = num("NAFGPU_WALK_SPLIT");
    o.debug_huf = getenv("NAFGPU_DEBUG_HUF") != nullptr;
    o.debug_prep = getenv("NAFGPU_DEBUG_PREP") != nullptr;
    return o;
}

// Forgets the previous job (plans, counters, graph) before a job of n archives is laid out.
void reset_job(nafgpu_ctx* c, uint32_t n, uint32_t want) {
    c->prepared = false; c->ran = false;
    drop_graph(c);
    c->want = want;
    c->plan.clear();
    c->arch.assign(n, nk::NafDev());
    c->aplan.assign(n, ArchPlan());
    memset(&c->stats, 0, sizeof c->stats);
    c->max_records = 0; c->max_chunks = 0; c->max_text = 0; c->max_mask = 0; c->max_scan = 0; c->any_mask = false; c->any_text_mask = false;
    c->misc_words = 0;
}

// Checks the header fields that size the arena (a zstd frame regenerates at most 128 KB per 3-byte block header): 0, or why not.
int validate_archive(const nafgpu_archive& A, std::string& why) {
    constexpr uint64_t MAX_SECTION = 1ull << 38;                    // 256 GB: more than a B200 holds
    if (A.header.sequence_type < 0 || A.header.sequence_type > 3) { why = "bad sequence type"; return NAFGPU_ERR_ARGUMENT; }
    for (int s = 0; s < 6; s++) {
        const nafgpu_section& S = A.sections[s];
        if (!S.present) continue;
        if (!S.data) { why = "present section without data"; return NAFGPU_ERR_ARGUMENT; }
        const uint64_t regen = (s == NAFGPU_SEC_SEQUENCE && A.header.sequence_type <= 1) ? S.original_size / 2 + (S.original_size & 1) : S.original_size;
        if (S.compressed_size > MAX_SECTION || regen > MAX_SECTION || regen > (S.compressed_size / 3 + 1) * (uint64_t)zf::BLOCK_MAX) {
            static const char* names[6] = {"ids", "comments", "lengths", "mask", "sequence", "quality"};
            why = std::string(names[s]) + " section: the header states a size its zstd frame cannot regenerate";
            return NAFGPU_ERR_INVALID_DATA;
        }
    }
    return 0;
}

// Validates the archives and lays out the arena.
int lay_out_arena(nafgpu_ctx* c, const nafgpu_archive* archives, uint32_t n, uint32_t want) {
    // Z1 (copied back): counts[n] | per archive: lengths, record offsets, id offsets, comment offsets, ids, comments, quality,
    // sequence ASCII.  Z2 (zeroed every run): mask toggle bitmaps.  Z3: device-only sections.  Sizes are validated first, record
    // counts are clamped by what the sections can hold, and a job whose arena would not fit any device is refused.
    c->counts_size = align_up((uint64_t)n * sizeof(nk::NafCounts));
    uint64_t off = c->counts_size;
    for (uint32_t a = 0; a < n; a++) {
        const nafgpu_archive& A = archives[a];
        ArchPlan& P = c->aplan[a];
        nk::NafDev& D = c->arch[a];
        memset(&D, 0, sizeof D);
        const uint64_t nrec = A.header.number_of_sequences;
        P.n_records = nrec;
        P.nucleotide = A.header.sequence_type <= 1;
        P.line_length = A.header.line_length; P.sep = (uint32_t)(A.header.name_separator & 0xFF);
        {
            std::string why;
            const int rc = validate_archive(A, why);
            if (rc == NAFGPU_ERR_ARGUMENT || (rc && n == 1)) return fail(c, rc, why);
            if (rc) { P.host_status = rc; P.host_msg = why; }       // one bad archive does not fail the batch: it is skipped and reported
        }
        const uint64_t nrec_dev = P.host_status ? 0 : nrec;
        const bool live = P.host_status == 0;
        const bool has_len = live && A.sections[NAFGPU_SEC_LENGTH].present;
        P.dec[NAFGPU_SEC_ID] = live && A.sections[NAFGPU_SEC_ID].present && (want & NAFGPU_WANT_ID);
        P.dec[NAFGPU_SEC_COMMENT] = live && A.sections[NAFGPU_SEC_COMMENT].present && (want & NAFGPU_WANT_COMMENT);
        P.dec[NAFGPU_SEC_LENGTH] = has_len;                                                  // mod.rs:239: always
        P.dec[NAFGPU_SEC_SEQUENCE] = has_len && A.sections[NAFGPU_SEC_SEQUENCE].present && (want & NAFGPU_WANT_SEQUENCE);
        P.dec[NAFGPU_SEC_QUALITY] = has_len && A.sections[NAFGPU_SEC_QUALITY].present && (want & NAFGPU_WANT_QUALITY);
        P.dec[NAFGPU_SEC_MASK] = P.dec[NAFGPU_SEC_SEQUENCE] && A.sections[NAFGPU_SEC_MASK].present && (want & NAFGPU_WANT_MASK);
        for (int s = 0; s < 6; s++) {
            uint64_t o = A.sections[s].original_size;
            P.blob_size[s] = !P.dec[s] ? 0 : ((s == NAFGPU_SEC_SEQUENCE && P.nucleotide) ? o / 2 + (o & 1) : o);
        }
        for (int k = 0; k < 4; k++) c->max_scan = std::max(c->max_scan, P.blob_size[k]);      // ids, comments, lengths, mask: the streaming scans
        const uint64_t residues = P.dec[NAFGPU_SEC_SEQUENCE] ? A.sections[NAFGPU_SEC_SEQUENCE].original_size : 0;
        // number_of_sequences is whatever the header says (2^61 is a valid varint); a stream of b bytes holds at most b
        // NUL-terminated strings / b/4 length words, so the offset tables are sized by that, not by the header
        const uint64_t nrec_ids = std::min<uint64_t>(nrec, P.blob_size[0]), nrec_com = std::min<uint64_t>(nrec, P.blob_size[1]);
        const uint64_t nrec_len = std::min<uint64_t>(nrec, P.blob_size[2] / 4);
        D.n_records = nrec_dev;
        D.seq_type = (uint32_t)A.header.sequence_type;
        D.has = (P.dec[0] ? nk::HAS_IDS : 0) | (P.dec[1] ? nk::HAS_COMMENTS : 0) | (P.dec[2] ? nk::HAS_LENGTHS : 0) |
                (P.dec[3] ? nk::HAS_MASK : 0) | (P.dec[4] ? nk::HAS_SEQUENCE : 0) | (P.dec[5] ? nk::HAS_QUALITY : 0);
        D.seq_residues = residues;
        D.counts_off = (uint64_t)a * sizeof(nk::NafCounts);
        D.lengths_off = off; off = align_up(off + 8 * (nrec_len + 1));
        D.rec_offsets_off = off; off = align_up(off + 8 * (nrec_len + 1));
        D.id_offsets_off = off; if (P.dec[0]) off = align_up(off + 8 * (nrec_ids + 1));
        D.com_offsets_off = off; if (P.dec[1]) off = align_up(off + 8 * (nrec_com + 1));
        auto place = [&](int s) { P.blob_off[s] = off; off = align_up(off + P.blob_size[s] + 32); };
        if (P.dec[0]) place(0);
        if (P.dec[1]) place(1);
        if (P.dec[5]) place(5);
        if (P.dec[4]) {
            if (P.nucleotide) { D.ascii_off = off; off = align_up(off + align_up(residues, 32) + 32); }
            else { place(4); D.ascii_off = P.blob_off[4]; }
        }
        c->max_records = std::max(c->max_records, std::max(nrec_len, std::max(nrec_ids, nrec_com)));
        if (P.dec[4]) {
            D.n_chunks = (uint32_t)((residues + 1 + nk::CHUNK_RESIDUES - 1) / nk::CHUNK_RESIDUES);
            c->max_chunks = std::max(c->max_chunks, D.n_chunks);
            if (P.dec[3]) { c->any_mask = true; c->max_mask = std::max(c->max_mask, P.blob_size[3]); if (!P.nucleotide) c->any_text_mask = true; }
            if (!P.nucleotide) c->max_text = std::max(c->max_text, P.blob_size[4]);
        }
        if (P.dec[5]) c->max_text = std::max(c->max_text, P.blob_size[5]);
        c->stats.ascii_bytes += residues;
        c->stats.quality_bytes += P.blob_size[5];
        c->stats.id_bytes += P.blob_size[0];
        c->stats.comment_bytes += P.blob_size[1];
        c->stats.algorithmic_bytes += residues + P.blob_size[5] + P.blob_size[0] + P.blob_size[1] + 8 * (nrec_len + 1);
        if (off > (1ull << 40)) return fail(c, NAFGPU_ERR_NOMEM, "job does not fit the device: split the batch");
    }
    c->z1_size = off;
    c->z2_off = off;
    for (uint32_t a = 0; a < n; a++) {
        ArchPlan& P = c->aplan[a];
        nk::NafDev& D = c->arch[a];
        D.mask_bits_off = off;
        if (P.dec[3]) off = align_up(off + 4 * ((D.seq_residues + 32) / 32 + 1));
        D.chunk_par_off = off;
        if (P.dec[3]) off = align_up(off + 4 * ((uint64_t)D.n_chunks + 1));
    }
    c->z2_size = off - c->z2_off;
    for (uint32_t a = 0; a < n; a++) {
        ArchPlan& P = c->aplan[a];
        nk::NafDev& D = c->arch[a];
        auto place = [&](int s) { P.blob_off[s] = off; off = align_up(off + P.blob_size[s] + 32); };
        if (P.dec[2]) place(2);
        if (P.dec[3]) place(3);
        if (P.dec[4] && P.nucleotide) place(4);
        D.mask_bounds_off = off; if (P.dec[3]) off = align_up(off + 8 * (P.blob_size[3] + 2));
        D.ids_off = P.blob_off[0]; D.ids_size = P.blob_size[0];
        D.com_off = P.blob_off[1]; D.com_size = P.blob_size[1];
        D.len_off = P.blob_off[2]; D.len_size = P.blob_size[2];
        D.mask_off = P.blob_off[3]; D.mask_size = P.blob_size[3];
        D.seq_off = P.blob_off[4]; D.seq_size = P.blob_size[4];
        D.qual_off = P.blob_off[5]; D.qual_size = P.blob_size[5];
    }
    c->arena_size = off + 256;
    return NAFGPU_OK;
}

// The sections the job decodes and the copies that bring them to `comp`; returns the end of the compressed bytes there.
uint64_t gather_sections(nafgpu_ctx* c, const nafgpu_archive* archives, uint32_t n, std::vector<SecRef>& secs, std::vector<Copy>& copies) {
    uint64_t comp_off = 16;          // gathers may read up to 15 bytes below a literal run: keep them inside the allocation
    for (uint32_t a = 0; a < n; a++) {
        const nafgpu_archive& A = archives[a];
        const ArchPlan& P = c->aplan[a];
        const size_t copies_mark = copies.size();
        for (int s = 0; s < 6; s++) {
            if (!P.dec[s]) continue;
            const nafgpu_section& S = A.sections[s];
            // Sections that follow one another in the caller's buffer (the sections of a NAF file do, a few header bytes
            // apart) keep their relative positions on the device and travel in one copy, gap bytes included.
            bool merged = false;
            if (copies.size() > copies_mark) {                  // (only within ONE archive: two archives may sit in adjacent allocations)
                Copy& L = copies.back();
                const uint8_t* lend = L.src + L.size;
                if (S.data >= lend && (uint64_t)(S.data - lend) <= 64) {
                    comp_off = L.dst + (uint64_t)(S.data - L.src);
                    L.size = (uint64_t)(S.data - L.src) + S.compressed_size;
                    merged = true;
                }
            }
            if (!merged) {
                if (!copies.empty()) comp_off = align_up(copies.back().dst + copies.back().size + zf::COMP_PAD, 16);
                copies.push_back({S.data, comp_off, S.compressed_size});
            }
            secs.push_back({{a, s, S.data, comp_off, S.compressed_size, P.blob_off[s], P.blob_size[s]}});
        }
    }
    return copies.empty() ? comp_off : align_up(copies.back().dst + copies.back().size + zf::COMP_PAD, 16);
}

// The host frame walk: chain pass over the long sections, the tasks (a long section as up to 8 parts), the walk of every task.
void walk_sections(nafgpu_ctx* c, std::vector<SecRef>& secs, const zk::Overrides& ov, PrepClock& clk) {
    // pass 1 over the long sections: the chain of block headers alone, a cut every `every` blocks
    uint32_t split_min = 200000, every = 16384;                  // (sections of fewer blocks are walked in one piece)
    uint64_t long_bytes = 4u << 20;
    if (ov.walk_split && *ov.walk_split <= 0) long_bytes = UINT64_MAX;
    else if (ov.walk_split) { every = (uint32_t)*ov.walk_split; split_min = every; long_bytes = 0; }
    bool any_long = false;
    for (const SecRef& R : secs) any_long = any_long || R.comp_size > long_bytes;
    std::unique_ptr<HelperLease> walk_lease;
    if (any_long) walk_lease.reset(new HelperLease);              // (held to the end of the walk)
    const unsigned hw_threads = walk_lease ? walk_lease->n : 1u;
    {
        std::vector<size_t> longs;
        for (size_t i = 0; i < secs.size(); i++) if (secs[i].comp_size > long_bytes) longs.push_back(i);
        parallel_for(longs.size(), hw_threads, [&](size_t i) {
            SecRef& R = secs[longs[i]];
            R.chain_rc = fw::chain_blocks(R.data, R.comp_size, R.dst_size, every, R.cuts, R.n_blocks, R.chain_err);
            if (R.chain_rc || R.n_blocks < split_min) R.cuts.clear();       // (an error is found again, and reported, by the walk proper)
        });
    }
    clk.lap("block chains");
    size_t n_tasks = 0;                                         // (tasks are reused from call to call: their plans keep their capacity)
    uint32_t heavy = 0;
    for (SecRef& R : secs) {
        const size_t n_cuts = R.cuts.size();
        const size_t parts = std::min<size_t>(n_cuts + 1, ov.walk_split ? n_cuts + 1 : std::max(8u, hw_threads));
        for (size_t k = 0; k < parts; k++) {
            if (n_tasks == c->tasks.size()) c->tasks.emplace_back();
            WalkTask& T = c->tasks[n_tasks++];
            // part k covers cuts [k * (n_cuts + 1) / parts, (k + 1) * (n_cuts + 1) / parts) of the n_cuts + 1 stretches between cuts
            const size_t lo = k * (n_cuts + 1) / parts, hi = (k + 1) * (n_cuts + 1) / parts;
            T.start(R, k == 0, k + 1 == parts, lo ? R.cuts[lo - 1] : 0, hi <= n_cuts ? R.cuts[hi - 1] : 0, R.comp_size > (8u << 20) || parts > 1);
            if (T.heavy) heavy++;
        }
    }
    c->n_tasks = n_tasks;
    auto walk = [&](size_t t) {
        WalkTask& T = c->tasks[t];
        T.rc = fw::walk_frame_part(T.data, T.comp_off, T.comp_size, T.dst_off, T.dst_size, T.p_begin, T.p_end, T.first, T.last, T.st, T.plan, T.err);
    };
    // (threads only when at least two tasks are big enough to hold 10^5+ block headers: starting threads costs more than
    // walking the ~30 headers of a genome section)
    const unsigned threads = heavy >= 2 ? std::min(heavy, hw_threads) : 1u;
    if (threads > 1) {
        std::vector<size_t> big, small;
        for (size_t t = 0; t < n_tasks; t++) (c->tasks[t].heavy ? big : small).push_back(t);
        std::thread rest([&] { for (size_t t : small) walk(t); });
        parallel_for(big.size(), threads, [&](size_t i) { walk(big[i]); });
        rest.join();
    } else {
        for (size_t t = 0; t < n_tasks; t++) walk(t);
    }
}

// What every part of a section walked in parts inherits from the parts before it, and the checks that span a whole frame.
void resolve_parts(nafgpu_ctx* c) {
    const size_t n_tasks = c->n_tasks;
    for (size_t t0 = 0; t0 < n_tasks;) {
        size_t t1 = t0 + 1;
        while (t1 < n_tasks && !c->tasks[t1].first) t1++;
        int huf_task = -1, tbl_task[3] = {-1, -1, -1};
        uint32_t huf_block = 0, huf_slot = 0, tbl_slot[3] = {0, 0, 0};
        uint64_t n_seq = 0, known = 0;
        int rc = 0;
        std::string err;
        for (size_t t = t0; t < t1 && !rc; t++) {
            WalkTask& T = c->tasks[t];
            if (T.rc) { rc = T.rc; err = T.err; break; }
            if (!T.first) {
                T.carry_huf_task = huf_task; T.carry_huf_block = huf_block; T.carry_huf_slot = huf_slot;
                for (int k = 0; k < 3; k++) { T.carry_tbl_task[k] = tbl_task[k]; T.carry_tbl_slot[k] = tbl_slot[k]; }
                if (T.st.used_prev_huf && huf_task < 0) { rc = NAFGPU_ERR_INVALID_DATA; err = "zstd literals: treeless block without a previous tree"; }
                for (int k = 0; k < 3; k++) if (T.st.used_prev_tbl[k] && tbl_task[k] == -1) { rc = NAFGPU_ERR_INVALID_DATA; err = "zstd sequences: repeat mode without a previous table"; }
            }
            if (T.st.last_huf != fw::PREV_BLOCK && T.st.last_huf != zf::NO_BLOCK) { huf_task = (int)t; huf_block = T.st.last_huf; huf_slot = T.st.last_huf_slot; }
            for (int k = 0; k < 3; k++) {
                const uint32_t v = T.st.cur_tbl[k];
                if (v == fw::PREV_SLOT || v == zf::NO_SLOT) continue;
                tbl_task[k] = v < 3 ? -2 : (int)t; tbl_slot[k] = v;
            }
            n_seq += T.st.n_seq; known += T.st.known_total;
        }
        if (!rc) rc = fw::check_frame_total(n_seq, known, c->tasks[t0].dst_size, err);
        if (rc) { c->tasks[t0].rc = rc; c->tasks[t0].err = err; }
        for (size_t t = t0 + 1; t < t1; t++) { c->tasks[t].comp_size = 0; c->tasks[t].dst_size = 0; }      // (counted once, with the first part)
        t0 = t1;
    }
}

// Closes the archives whose walk failed (a single archive fails the job), then numbers every archive's frames in the job plan.
int close_failed_archives(nafgpu_ctx* c, uint32_t n) {
    static const char* names[6] = {"ids", "comments", "lengths", "mask", "sequence", "quality"};
    uint32_t frames_so_far = 0;
    size_t t = 0;
    for (uint32_t a = 0; a < n; a++) {
        ArchPlan& P = c->aplan[a];
        const size_t t0 = t;
        while (t < c->n_tasks && c->tasks[t].arch == a) t++;
        int bad_rc = 0;
        for (size_t k = t0; k < t && !bad_rc; k++) {
            if (c->tasks[k].rc) { bad_rc = c->tasks[k].rc; P.host_msg = std::string(names[c->tasks[k].sec]) + " section: " + c->tasks[k].err; }
        }
        if (bad_rc) {
            if (n == 1) return fail(c, bad_rc, P.host_msg);
            // a batch goes on without this archive: none of it is decoded, its result carries the status (its bytes still travel)
            P.host_status = bad_rc;
            c->arch[a].has = 0; c->arch[a].n_records = 0;
            for (int k = 0; k < 6; k++) P.dec[k] = false;
            for (size_t k = t0; k < t; k++) c->tasks[k].live = false;
        }
        P.first_frame = frames_so_far;
        P.n_frames = 0;
        for (size_t k = t0; k < t; k++) {
            if (!c->tasks[k].live) continue;
            P.n_frames += (uint32_t)c->tasks[k].plan.frames.size();
            c->stats.compressed_bytes += c->tasks[k].comp_size;
            c->stats.section_bytes += c->tasks[k].dst_size;
        }
        frames_so_far += P.n_frames;
    }
    c->stats.algorithmic_bytes += c->stats.compressed_bytes;
    return NAFGPU_OK;
}

// Lays the tasks' plans end to end into the job plan (block descriptors stay in the tasks); nb: the job's blocks.
int merge_plans(nafgpu_ctx* c, size_t& nb) {
    nb = 0;
    fw::JobPlan& G = c->plan;
    for (size_t ti = 0; ti < c->n_tasks; ti++) {
        WalkTask& T = c->tasks[ti];
        if (!T.live) continue;
        const fw::JobPlan& L = T.plan;
        T.bo = nb; T.so = (uint32_t)G.seq_total; T.lo = G.lit_total - 16; T.slot_off = G.n_slots - 3; T.ho = G.n_huf_slots;
        if (G.seq_total + L.seq_total > 0xFFFFFFF0ull || nb + L.blocks.size() > 0xFFFFFFF0ull) return fail(c, NAFGPU_ERR_UNSUPPORTED, "job has too many blocks or sequences: split the batch");
        for (zf::FrameDesc F : L.frames) { F.first_block += (uint32_t)T.bo; F.first_seq += T.so; G.frames.push_back(F); }
        if (!T.first) {                // a continuation part: its blocks and sequences belong to the frame the first part opened
            zf::FrameDesc& F = G.frames.back();
            F.n_blocks += T.st.n_blocks; F.n_seq += T.st.n_seq;
            if (T.last) { F.has_checksum = T.st.has_checksum; F.checksum = T.st.checksum; }
            if (T.carry_huf_task >= 0) { const WalkTask& S = c->tasks[T.carry_huf_task]; T.abs_huf_block = (uint32_t)S.bo + T.carry_huf_block; T.abs_huf_slot = S.ho + T.carry_huf_slot; }
            for (int k = 0; k < 3; k++) {
                if (T.carry_tbl_task[k] == -2) T.abs_tbl[k] = T.carry_tbl_slot[k];
                else if (T.carry_tbl_task[k] >= 0) T.abs_tbl[k] = c->tasks[T.carry_tbl_task[k]].slot_off + T.carry_tbl_slot[k];
            }
        }
        for (zf::HufItem it : L.huf_items) { it.block += (uint32_t)T.bo; G.huf_items.push_back(it); }
        for (uint32_t b : L.big_seq) G.big_seq.push_back(b + (uint32_t)T.bo);
        for (uint32_t b : L.big_lit) G.big_lit.push_back(b + (uint32_t)T.bo);
        G.seq_total += L.seq_total; G.lit_total += L.lit_total - 16; G.n_slots += L.n_slots - 3; G.n_huf_slots += L.n_huf_slots;
        G.n_huf_blocks += L.n_huf_blocks; G.n_seq_blocks += L.n_seq_blocks; G.n_checksums += L.n_checksums;
        G.max_seq_section = std::max(G.max_seq_section, L.max_seq_section);
        G.max_seq_section_big = std::max(G.max_seq_section_big, L.max_seq_section_big); G.n_tiny_seq_blocks += L.n_tiny_seq_blocks;
        nb += L.blocks.size();
    }
    G.finalize(zk::HUF_SMALL_SYMBOLS);
    return NAFGPU_OK;
}

// What stage_descriptors leaves for bind_job besides the layout of `desc` (c->o_*).
struct Staged {
    uint32_t total_chunks = 0;         // the finisher's 64 KB chunks, all frames
    uint64_t g_entries = 0;            // fin_g entries, all frames
    uint32_t n_tiles = 0, n_bigs = 0, fs_big = 0;   // frame-scan tiles, the frames they cover, and the frame size (blocks) above which a frame is tiled
    uint64_t h2d = 0;                  // bytes copied to the device
};

// Sizes the device buffers, stages the job's descriptors in pinned memory and uploads them in one H2D copy.
int stage_descriptors(nafgpu_ctx* c, uint32_t n, size_t nb, const std::vector<Copy>& copies, uint64_t comp_end, bool copies_enqueued,
                      const zk::Overrides& ov, PrepClock& clk, Staged& S) {
    const fw::JobPlan& pl = c->plan;
    const size_t nf = pl.frames.size(), nh = pl.huf_items.size();
    // descriptors: [blocks | frames | NafDev | HufItem | chunk table | fin_g bases | tiles | big frames | big-block lists], the same
    // layout in `stage` and `desc`, so that they go up in ONE copy (a burst of small H2D copies is time-sliced against other
    // contexts' result copies); then the compressed sections, unless they went before the walk
    c->o_frames = align_up(nb * sizeof(zf::BlockDesc), 16);
    c->o_naf = c->o_frames + align_up(nf * sizeof(zf::FrameDesc), 16);
    c->o_huf = c->o_naf + align_up((size_t)n * sizeof(nk::NafDev), 16);
    c->o_chunks = c->o_huf + align_up(nh * sizeof(zf::HufItem), 16);
    // finisher chunk table: first 64 KB chunk of every frame (zstd_kernels.cu, k_lz_finish)
    std::vector<uint32_t> chunk_first(nf + 1, 0);
    for (size_t f = 0; f < nf; f++) {
        const uint64_t nchunks = (pl.frames[f].dst_size + 65535) >> 16;
        if ((uint64_t)chunk_first[f] + nchunks > 0x7FFFFFFFull) return fail(c, NAFGPU_ERR_UNSUPPORTED, "job too large for the chunk table");
        chunk_first[f + 1] = chunk_first[f] + (uint32_t)nchunks;
    }
    S.total_chunks = chunk_first[nf];
    std::vector<uint64_t> g_base(nf + 1, 0);             // fin_g: one entry per byte of every frame, frames packed (16-entry aligned)
    for (size_t f = 0; f < nf; f++) g_base[f + 1] = g_base[f] + ((pl.frames[f].dst_size + 15) & ~(uint64_t)15);
    S.g_entries = g_base[nf];
    c->o_gbase = c->o_chunks + align_up((nf + 1) * 4, 16);
    // tiles of the frames that are too long for one scanning CTA
    std::vector<zf::FsTile> tiles;
    std::vector<zf::FsBigFrame> bigs;
    const uint32_t fs_tile = ov.fs_tile ? *ov.fs_tile : zf::FS_TILE;
    S.fs_big = ov.fs_tile ? 2 * fs_tile : zf::FS_BIG_FRAME;
    for (size_t f = 0; f < nf; f++) {
        const zf::FrameDesc& F = pl.frames[f];
        if (F.n_blocks <= S.fs_big) continue;
        bigs.push_back({(uint32_t)f, (uint32_t)tiles.size(), (F.n_blocks + fs_tile - 1) / fs_tile, 0u});
        for (uint32_t b = 0; b < F.n_blocks; b += fs_tile) tiles.push_back({(uint32_t)f, F.first_block + b, std::min(fs_tile, F.n_blocks - b), 0u});
    }
    S.n_tiles = (uint32_t)tiles.size(); S.n_bigs = (uint32_t)bigs.size();
    c->o_tiles = c->o_gbase + align_up((nf + 1) * 8, 16);
    c->o_big = c->o_tiles + align_up(tiles.size() * sizeof(zf::FsTile), 16);
    c->o_bigseq = c->o_big + align_up(bigs.size() * sizeof(zf::FsBigFrame), 16);
    c->o_biglit = c->o_bigseq + align_up(pl.big_seq.size() * 4, 16);
    const size_t stage_bytes = c->o_biglit + align_up(pl.big_lit.size() * 4, 16);
    c->misc_words = zk::JobWords::words(nf, S.total_chunks);
    const uint64_t nseq = pl.seq_total;
    bool ok = c->comp.ensure(comp_end + 64) && c->arena.ensure(c->arena_size) && c->lit.ensure(pl.lit_total + 64) &&
              c->desc.ensure(stage_bytes + 64) && c->fin_g.ensure((size_t)g_base[nf] * 4 + 256 + (size_t)S.total_chunks * 8192) &&
              c->bstate.ensure(nb * sizeof(zf::BlockState) + 64) && c->fsstate.ensure(tiles.size() * sizeof(zf::FsTileState) + 64) && c->lzidx.ensure(((size_t)S.total_chunks * 16 + nf + 16) * 4) &&
              c->scanagg.ensure((size_t)n * 4 * ((c->max_scan + nk::NAF_SLICE - 1) / nk::NAF_SLICE + 1) * nk::NAF_AGG_BYTES + 64) && c->hufw.ensure((size_t)pl.n_huf_slots * 258 + 64) &&
              c->tables.ensure((size_t)pl.n_slots * zf::FSE_SLOT_CELLS * sizeof(zc::SeqCell)) && c->table_al.ensure(pl.n_slots + 64) &&
              c->seq32.ensure(nseq * 5 * 4 + 64) && c->seq64.ensure(nseq * sizeof(zf::SeqRec) + 64) && c->misc.ensure(c->misc_words * 4);
    if (!ok) return fail(c, NAFGPU_ERR_NOMEM, "device allocation failed");
    clk.lap("merge + device buffers");
    if (!c->stage.ensure(stage_bytes + 64) || !c->result.ensure(c->counts_size + 64) || !c->misc_host.ensure(c->misc_words * 4 + 64))   // (the whole-result buffer is taken at the first full fetch: a job read in windows never needs it)
        return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");

    uint8_t* sp = (uint8_t*)c->stage.p;
    {
        // block descriptors: every task's blocks to their place, indices rebased to the job (frames, sequences, literal staging,
        // FSE table slots, Huffman weight records)
        std::vector<uint32_t> frame_off(c->n_tasks, 0);
        { uint32_t fo = 0; for (size_t t = 0; t < c->n_tasks; t++) { frame_off[t] = c->tasks[t].first ? fo : fo - 1; if (c->tasks[t].live) fo += (uint32_t)c->tasks[t].plan.frames.size(); } }
        unsigned threads = 1;
        std::unique_ptr<HelperLease> lease;
        if (nb > 200000) { lease.reset(new HelperLease); threads = lease->n; }
        struct Chunk { size_t task, begin, end; };
        std::vector<Chunk> chunks;
        for (size_t t = 0; t < c->n_tasks; t++) {
            if (!c->tasks[t].live) continue;
            const size_t cnt = c->tasks[t].plan.blocks.size();
            for (size_t b = 0; b < cnt; b += 65536) chunks.push_back({t, b, std::min(cnt, b + 65536)});
        }
        parallel_for(chunks.size(), threads, [&](size_t ci) {
            const Chunk& K = chunks[ci];
            const WalkTask& T = c->tasks[K.task];
            zf::BlockDesc* out = (zf::BlockDesc*)sp + T.bo;
            const zf::BlockDesc* in = T.plan.blocks.data();
            const uint32_t fo = frame_off[K.task];
            for (size_t i = K.begin; i < K.end; i++) {
                zf::BlockDesc b = in[i];
                b.frame += fo;
                if (b.n_seq) b.seq_base += T.so;
                if (b.huf_block == fw::PREV_BLOCK) { b.lit_base += T.lo; b.huf_block = T.abs_huf_block; b.huf_slot = T.abs_huf_slot; }     // treeless, the tree from an earlier part
                else {
                    if (b.lit_type >= zf::LT_HUF && b.btype == zf::BT_COMPRESSED) { b.lit_base += T.lo; b.huf_slot += T.ho; }
                    if (b.huf_block != zf::NO_BLOCK) b.huf_block += (uint32_t)T.bo;
                }
                for (int k = 0; k < 3; k++) {
                    if (b.tbl[k] == fw::PREV_SLOT) b.tbl[k] = T.abs_tbl[k];
                    else if (b.tbl[k] != zf::NO_SLOT && b.tbl[k] >= 3) b.tbl[k] += T.slot_off;
                }
                store_desc(out + i, b);
            }
            desc_fence();
        });
    }
    clk.lap("pinned staging + block copy");
    if (nf) memcpy(sp + c->o_frames, pl.frames.data(), nf * sizeof(zf::FrameDesc));
    if (n) memcpy(sp + c->o_naf, c->arch.data(), (size_t)n * sizeof(nk::NafDev));
    if (nh) memcpy(sp + c->o_huf, pl.huf_items.data(), nh * sizeof(zf::HufItem));
    memcpy(sp + c->o_chunks, chunk_first.data(), (nf + 1) * 4);
    memcpy(sp + c->o_gbase, g_base.data(), (nf + 1) * 8);
    if (!pl.big_seq.empty()) memcpy(sp + c->o_bigseq, pl.big_seq.data(), pl.big_seq.size() * 4);
    if (!pl.big_lit.empty()) memcpy(sp + c->o_biglit, pl.big_lit.data(), pl.big_lit.size() * 4);
    if (!tiles.empty()) { memcpy(sp + c->o_tiles, tiles.data(), tiles.size() * sizeof(zf::FsTile)); memcpy(sp + c->o_big, bigs.data(), bigs.size() * sizeof(zf::FsBigFrame)); }
    if (stage_bytes) CUDA_TRY(c, cudaMemcpyAsync(c->desc.p, sp, stage_bytes, cudaMemcpyHostToDevice, c->streams.st));
    S.h2d = stage_bytes;
    for (const Copy& cp : copies) {
        if (!copies_enqueued) CUDA_TRY(c, cudaMemcpyAsync((uint8_t*)c->comp.p + cp.dst, cp.src, cp.size, cudaMemcpyHostToDevice, c->streams.st));
        S.h2d += cp.size;
    }
    clk.lap("H2D enqueue");
    return NAFGPU_OK;
}

// Points JobDev into the job's buffers and descriptor tables, then lets choose_paths make the job's path decisions.
int bind_job(nafgpu_ctx* c, size_t nb, const Staged& S, const zk::Overrides& ov) {
    const fw::JobPlan& pl = c->plan;
    const size_t nf = pl.frames.size(), nh = pl.huf_items.size();
    const uint64_t nseq = pl.seq_total;
    const uint8_t* desc = (const uint8_t*)c->desc.p;
    zk::JobDev& J = c->J;
    J.comp = (const uint8_t*)c->comp.p; J.out = (uint8_t*)c->arena.p; J.lit = (uint8_t*)c->lit.p;
    J.frames = (const zf::FrameDesc*)(desc + c->o_frames); J.blocks = (const zf::BlockDesc*)desc;
    J.bstate = (zf::BlockState*)c->bstate.p; J.tables = (zc::SeqCell*)c->tables.p; J.table_al = (uint8_t*)c->table_al.p;
    J.seq_done = (uint32_t*)c->seq32.p;
    J.lz_list[0] = J.seq_done + nseq; J.lz_list[1] = J.seq_done + 2 * nseq; J.lz_list[2] = J.seq_done + 3 * nseq; J.lz_blocker = J.seq_done + 4 * nseq;
    J.seq = (zf::SeqRec*)c->seq64.p;
    J.seq_big_list = (const uint32_t*)(desc + c->o_bigseq); J.n_seq_big = (uint32_t)pl.big_seq.size();
    J.lit_big_list = (const uint32_t*)(desc + c->o_biglit); J.n_lit_big = (uint32_t)pl.big_lit.size();
    zk::JobWords* w = (zk::JobWords*)c->misc.p;
    J.status = &w->status; J.lz_count = w->lz_count; J.lz_handover = &w->lz_handover; J.lz_rounds = &w->lz_rounds;
    J.fin_unresolved = &w->fin_unresolved; J.fin_count = w->fin_count; J.lz_flow = w->lz_flow; J.lz_pending = w->lz_pending;
    J.frame_bad = w->frame_bad(); J.fin_chunk_flag = w->fin_chunk_flag(nf);
    J.fin_chunk_first = (const uint32_t*)(desc + c->o_chunks); J.fin_total_chunks = S.total_chunks;
    J.lz_idx = (uint32_t*)c->lzidx.p;
    J.fin_g = (uint32_t*)c->fin_g.p; J.fin_ext = (uint32_t*)c->fin_g.p + S.g_entries + 64;
    J.fin_g_base = (const uint64_t*)(desc + c->o_gbase);
    J.huf_weights = (uint8_t*)c->hufw.p; J.huf_meta = (uint8_t*)c->hufw.p + (size_t)pl.n_huf_slots * 256;
    J.huf_items = (const zf::HufItem*)(desc + c->o_huf); J.n_huf_items = (uint32_t)nh; J.n_huf_big = pl.n_huf_big; J.max_huf_stream = pl.max_huf_stream; J.max_huf_small = pl.max_huf_small;
    J.debug = nullptr; J.debug_seq = nullptr;
    if (ov.debug_huf && nh) {
        if (!c->debug.ensure(nh * 64 + 64)) return fail(c, NAFGPU_ERR_NOMEM, "debug buffer");
        cudaMemsetAsync(c->debug.p, 0, nh * 64 + 64, c->streams.st);
        J.debug = (unsigned long long*)c->debug.p;
        J.debug_seq = J.debug + nh * 8;
    }
    J.fs_tiles = (const zf::FsTile*)(desc + c->o_tiles); J.fs_big = (const zf::FsBigFrame*)(desc + c->o_big);
    J.fs_state = (zf::FsTileState*)c->fsstate.p; J.n_fs_tiles = S.n_tiles; J.n_fs_big = S.n_bigs; J.fs_big_frame = S.fs_big;
    J.n_frames = (uint32_t)nf; J.n_blocks = (uint32_t)nb; J.n_slots = pl.n_slots; J.n_seq = nseq; J.n_checksums = pl.n_checksums;
    c->launch = zk::choose_paths(J, pl, ov, c->sms, c->arena_size);
    return NAFGPU_OK;
}

// The walked job to the device: the plans merged, descriptors and sections uploaded, JobDev bound and its paths chosen.
int finish_prepare(nafgpu_ctx* c, const std::vector<Copy>& copies, uint64_t comp_end, uint32_t n, bool copies_enqueued,
                   const zk::Overrides& ov, PrepClock& clk) {
    size_t nb = 0;
    Staged S;
    int rc = merge_plans(c, nb);
    if (!rc) rc = stage_descriptors(c, n, nb, copies, comp_end, copies_enqueued, ov, clk, S);
    if (!rc) rc = bind_job(c, nb, S, ov);
    if (rc) return rc;
    c->stats.n_archives = n; c->stats.n_frames = c->plan.frames.size(); c->stats.n_blocks = nb; c->stats.n_sequences = c->plan.seq_total;
    c->stats.h2d_bytes = S.h2d; c->stats.d2h_bytes = c->z1_size + c->misc_words * 4;
    c->stats.n_stages = N_STAGES + 1;
    c->prepared = true;
    return NAFGPU_OK;
}

// What fetch, format, export and fetch-window report for one archive after a run (counters only when it did not fail).
struct Outcome {
    int status = 0;
    std::string msg;                   // "archive <a>: ..." when status != 0
    const nk::NafCounts* C = nullptr;
    uint64_t n_ids = 0, n_comments = 0;          // clamped to the header's record count
    uint64_t first_bad_record = nk::NO_RECORD;
    int record_status = 0;             // NAFGPU_ERR_UTF8 when first_bad_record is a record
};

Outcome archive_outcome(nafgpu_ctx* c, uint32_t a) {
    const ArchPlan& P = c->aplan[a];
    Outcome o;
    // status: what the host found (validation, frame walk), else the OR of the device status of its frames and of its NAF-level
    // checks (NafCounts::status); UTF-8 is reported per record, as first_bad_record
    o.C = (const nk::NafCounts*)((const uint8_t*)c->result.p + c->arch[a].counts_off);
    uint32_t s = (uint32_t)o.C->status;
    for (uint32_t f = P.first_frame; f < P.first_frame + P.n_frames; f++) s |= words(c).frame_bad()[f];
    o.status = P.host_status ? P.host_status : status_to_code(s & ~zc::E_UTF8, o.msg);
    if (o.status) {
        char b[48];
        snprintf(b, sizeof b, "archive %u: ", a);
        o.msg = b + (P.host_status ? P.host_msg : o.msg);
        return o;
    }
    o.n_ids = std::min<uint64_t>(o.C->n_ids, P.n_records);
    o.n_comments = std::min<uint64_t>(o.C->n_comments, P.n_records);
    o.first_bad_record = o.C->first_bad_record;
    o.record_status = o.first_bad_record != nk::NO_RECORD ? NAFGPU_ERR_UTF8 : 0;
    return o;
}

// Status words and the archives' counters of the last run on the host, once per run (a synchronise on the context's stream).
int read_counts(nafgpu_ctx* c) {
    if (c->win_counts) return NAFGPU_OK;
    CUDA_TRY(c, wait_stream(c));
    CUDA_TRY(c, cudaMemcpyAsync(c->misc_host.p, c->misc.p, c->misc_words * 4, cudaMemcpyDeviceToHost, c->streams.st));
    CUDA_TRY(c, cudaMemcpyAsync(c->result.p, c->arena.p, c->counts_size, cudaMemcpyDeviceToHost, c->streams.st));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    read_lz_stats(c);
    c->win_counts = true;
    return NAFGPU_OK;
}

// The counters of every archive and the export descriptors of the last run (include/nafgpu.h, nafgpu_job_export): built on the
// host from the counters and uploaded in one copy on the context's stream.  They stay unchanged until the next run, which the
// context's stream only starts once the exports that read them are done.
int export_tables(nafgpu_ctx* c) {
    if (c->exp_ready) return NAFGPU_OK;
    { int rc = read_counts(c); if (rc) return rc; }
    const uint32_t n = (uint32_t)c->arch.size();
    c->counts.assign(n, nafgpu_counts());
    std::vector<nk::ExpRec> recs;
    std::vector<nk::ExpSpan> spans[4];
    uint64_t records = 0, residues = 0, bytes[4] = {0, 0, 0, 0};
    for (uint32_t a = 0; a < n; a++) {
        const nk::NafDev& D = c->arch[a];
        const ArchPlan& P = c->aplan[a];
        nafgpu_counts& k = c->counts[a];
        memset(&k, 0, sizeof k);
        k.n_records = P.n_records;
        const Outcome o = archive_outcome(c, a);
        k.status = o.status;
        k.first_bad_record = o.first_bad_record;
        k.record_status = o.record_status;
        if (k.status) continue;
        k.n_ids = P.dec[0] ? o.n_ids : 0;
        k.n_comments = P.dec[1] ? o.n_comments : 0;
        k.n_lengths = P.dec[2] ? o.C->n_lengths : 0;
        k.total_residues = P.dec[2] ? o.C->total_residues : 0;
        k.id_bytes = P.dec[0] ? D.ids_size : 0;
        k.comment_bytes = P.dec[1] ? D.com_size : 0;
        if (k.n_lengths)
            recs.push_back({records, residues, D.rec_offsets_off, {P.dec[4] ? D.ascii_off : nk::NO_FIELD, P.dec[5] ? D.qual_off : nk::NO_FIELD}, 0});
        const uint64_t field_bytes[4] = {k.id_bytes, k.comment_bytes, P.dec[4] ? k.total_residues : 0, P.dec[5] ? k.total_residues : 0};
        const uint64_t field_off[4] = {D.ids_off, D.com_off, D.ascii_off, D.qual_off};
        for (int f = 0; f < 4; f++) {
            if (!field_bytes[f]) continue;
            spans[f].push_back({bytes[f], field_off[f]});
            bytes[f] += field_bytes[f];
        }
        records += k.n_lengths;
        residues += k.total_residues;
    }
    uint64_t off = align_up(recs.size() * sizeof(nk::ExpRec), 16);
    for (int f = 0; f < 4; f++) { c->o_exp_span[f] = off; off += align_up(spans[f].size() * sizeof(nk::ExpSpan), 16); }
    if (!c->exp_desc.ensure(off + 64)) return fail(c, NAFGPU_ERR_NOMEM, "device allocation failed");
    if (!c->exp_stage.ensure(off + 64)) return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
    uint8_t* S = (uint8_t*)c->exp_stage.p;       // (free: the stream was synchronised above, after the last copy from it)
    if (!recs.empty()) memcpy(S, recs.data(), recs.size() * sizeof(nk::ExpRec));
    for (int f = 0; f < 4; f++) if (!spans[f].empty()) memcpy(S + c->o_exp_span[f], spans[f].data(), spans[f].size() * sizeof(nk::ExpSpan));
    if (off) CUDA_TRY(c, cudaMemcpyAsync(c->exp_desc.p, S, off, cudaMemcpyHostToDevice, c->streams.st));
    c->n_exp_rec = (uint32_t)recs.size();
    for (int f = 0; f < 4; f++) { c->n_exp_span[f] = (uint32_t)spans[f].size(); c->exp_bytes[f] = bytes[f]; }
    c->exp_records = records;
    c->exp_residues = residues;
    c->exp_ready = true;
    return NAFGPU_OK;
}

}  // namespace

extern "C" {

int nafgpu_ctx_create(int device, nafgpu_ctx** out) {
    if (!out) return NAFGPU_ERR_ARGUMENT;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); return NAFGPU_ERR_NO_DEVICE; }
    if (device < 0 || device >= n) return NAFGPU_ERR_ARGUMENT;
    if (cudaSetDevice(device) != cudaSuccess) return NAFGPU_ERR_CUDA;
    nafgpu_ctx* c = new nafgpu_ctx();
    c->device = device;
    memset(&c->stats, 0, sizeof c->stats);
    memset(&c->J, 0, sizeof c->J);
    if (!c->streams.create()) { c->streams.destroy(); delete c; return NAFGPU_ERR_CUDA; }
    if (cudaEventCreateWithFlags(&c->ev_block, cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) { c->ev_block = nullptr; cudaGetLastError(); }
    if (cudaEventCreateWithFlags(&c->ev_d2h, cudaEventDisableTiming) != cudaSuccess) { c->ev_d2h = nullptr; cudaGetLastError(); }
    if (cudaEventCreateWithFlags(&c->ev_exp_ready, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&c->ev_exp_done, cudaEventDisableTiming) != cudaSuccess) { delete c; return NAFGPU_ERR_CUDA; }
    for (int i = 0; i < N_STAGES + 3; i++) if (cudaEventCreate(&c->ev[i]) != cudaSuccess) { delete c; return NAFGPU_ERR_CUDA; }
    c->ev_ok = true;
#if defined(NAFGPU_EMULATE)
    c->sms = 148;                      // (the emulator runs the grids of a B200)
#else
    { int sms = 0; if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) c->sms = (uint32_t)sms; }
#endif
    c->J.coop_ctas = zk::lz_resolve_max_ctas(device);                  // (the grids of the device: set once, every job keeps them)
    zk::lz_finish_ctas(device, &c->J.fin_ctas, &c->J.fin2_ctas);
    *out = c;
    return NAFGPU_OK;
}

void nafgpu_ctx_destroy(nafgpu_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->streams.st);
    drop_graph(c);
    DevBuf* d[] = {&c->comp, &c->arena, &c->lit, &c->desc, &c->bstate, &c->hufw, &c->fsstate, &c->lzidx, &c->scanagg, &c->debug, &c->tables, &c->table_al, &c->seq32, &c->seq64, &c->misc, &c->flush, &c->text, &c->fin_g, &c->pack_in, &c->pack_out, &c->exp_desc};
    for (DevBuf* b : d) b->release();
    c->stage.release(); c->result.release(); c->misc_host.release(); c->text_host.release(); c->text_stage.release(); c->pack_host.release(); c->win.release();
    c->exp_stage.release();
    if (c->ev_exp_ready) cudaEventDestroy(c->ev_exp_ready);
    if (c->ev_exp_done) cudaEventDestroy(c->ev_exp_done);
    if (c->ev_ok) for (int i = 0; i < N_STAGES + 3; i++) cudaEventDestroy(c->ev[i]);
    if (c->ev_block) cudaEventDestroy(c->ev_block);
    if (c->ev_d2h) {
        { std::lock_guard<std::mutex> turn(g_d2h_turn[c->device & 15]); if (g_last_d2h[c->device & 15] == c->ev_d2h) g_last_d2h[c->device & 15] = nullptr; }
        cudaEventDestroy(c->ev_d2h);
    }
    c->streams.destroy();
    delete c;
}

const char* nafgpu_last_error(const nafgpu_ctx* c) { return c ? c->err.c_str() : "null context"; }

void* nafgpu_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void nafgpu_host_free(void* p) { if (p) cudaFreeHost(p); }

int nafgpu_job_prepare(nafgpu_ctx* c, const nafgpu_archive* archives, uint32_t n, uint32_t want) {
    if (!c || (!archives && n)) return NAFGPU_ERR_ARGUMENT;
    if (n > 65535u) return fail(c, NAFGPU_ERR_ARGUMENT, "at most 65535 archives per job (the archive index is a grid dimension): split the batch");
    CUDA_TRY(c, cudaSetDevice(c->device));
    // the previous job may still be in flight on the stream and owns the staging buffers
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    reset_job(c, n, want);
    const zk::Overrides ov = read_overrides();
    { const int rc = lay_out_arena(c, archives, n, want); if (rc) return rc; }
    std::vector<Copy> copies;
    std::vector<SecRef> secs;
    const uint64_t comp_end = gather_sections(c, archives, n, secs, copies);
    PrepClock clk{ov.debug_prep};
    // The compressed sections do not wait for the header walk: their copies go first, so that they cross PCIe while the host walks
    // (512 archives: 520 MB, 9.5 ms of copies beside 4.5 ms of walk).  The stream was synchronised above: nothing reads `comp`.
    bool copies_enqueued = false;
    if (c->comp.ensure(comp_end + 64)) {
        for (const Copy& cp : copies) CUDA_TRY(c, cudaMemcpyAsync((uint8_t*)c->comp.p + cp.dst, cp.src, cp.size, cudaMemcpyHostToDevice, c->streams.st));
        copies_enqueued = true;
    }                                                          // (else: finish_prepare reports the failed allocation)
    // (a failed prepare must not leave copies from the caller's buffers in flight: every error return below waits for them)
    struct CopyGuard { cudaStream_t st; bool armed; ~CopyGuard() { if (armed) cudaStreamSynchronize(st); } } copy_guard{c->streams.st, copies_enqueued};
    clk.lap("compressed sections enqueued");
    walk_sections(c, secs, ov, clk);
    resolve_parts(c);
    clk.lap("header walk");
    { const int rc = close_failed_archives(c, n); if (rc) return rc; }
    const int rc = finish_prepare(c, copies, comp_end, n, copies_enqueued, ov, clk);
    if (rc == NAFGPU_OK) copy_guard.armed = false;
    return rc;
}

// One magicless zstd frame -> regen_size bytes at dst (host).  The pure-zstd boundary of the reference
// (zstd::stream::read::Decoder, decoder/mod.rs:221-223), exposed for parity tests against libzstd.
int nafgpu_zstd_decompress(nafgpu_ctx* c, const uint8_t* frame, uint64_t frame_size, uint64_t regen_size, uint8_t* dst) {
    if (!c || !frame || (!dst && regen_size)) return NAFGPU_ERR_ARGUMENT;
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    reset_job(c, 0, 0);
    const zk::Overrides ov = read_overrides();
    c->counts_size = ALIGN;
    c->z1_size = align_up(ALIGN + regen_size + 32);
    c->z2_off = c->z1_size; c->z2_size = 0;
    c->arena_size = c->z1_size + 256;
    if (c->tasks.empty()) c->tasks.emplace_back();
    c->n_tasks = 1;
    WalkTask& T = c->tasks[0];
    T.start({0, 0, frame, 16, frame_size, ALIGN, regen_size}, true, true);
    T.rc = fw::walk_frame(frame, 16, frame_size, ALIGN, regen_size, T.plan, T.err);
    if (T.rc) return fail(c, T.rc, T.err);
    c->stats.compressed_bytes = frame_size; c->stats.section_bytes = regen_size;
    c->stats.algorithmic_bytes = frame_size + regen_size;
    PrepClock clk{ov.debug_prep};
    int rc = finish_prepare(c, {{frame, 16, frame_size}}, 16 + align_up(frame_size + zf::COMP_PAD, 16), 0, false, ov, clk);
    if (rc) return rc;
    rc = enqueue_run(c, nullptr);
    if (rc) return rc;
    rc = d2h_results(c);
    if (rc) return rc;
    std::string msg;
    const int code = status_to_code(words(c).status, msg);
    read_lz_stats(c);
    if (code) return fail(c, code, msg);
    if (regen_size) memcpy(dst, (const uint8_t*)c->result.p + ALIGN, regen_size);
    return NAFGPU_OK;
}

int nafgpu_job_run(nafgpu_ctx* c) {
    if (!c) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared) return fail(c, NAFGPU_ERR_ARGUMENT, "no prepared job");
    CUDA_TRY(c, cudaSetDevice(c->device));
    return enqueue_run(c, nullptr);
}

int nafgpu_job_sync(nafgpu_ctx* c) {
    if (!c) return NAFGPU_ERR_ARGUMENT;
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    return NAFGPU_OK;
}

int nafgpu_job_fetch(nafgpu_ctx* c, nafgpu_result* out, uint32_t n) {
    if (!c || (!out && n)) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared || !c->ran) return fail(c, NAFGPU_ERR_ARGUMENT, "job has not been run");
    if (n != c->arch.size()) return fail(c, NAFGPU_ERR_ARGUMENT, "result count differs from the prepared job");
    CUDA_TRY(c, cudaSetDevice(c->device));
    { int rc_d2h = d2h_results(c); if (rc_d2h) return rc_d2h; }
    CUDA_TRY(c, cudaGetLastError());
    if (c->J.debug) {
        size_t nh = c->J.n_huf_items;
        std::vector<unsigned long long> d(nh * 8 + 8);
        cudaMemcpy(d.data(), c->J.debug, nh * 64 + 64, cudaMemcpyDeviceToHost);
        const unsigned long long* q = d.data() + nh * 8;
        double ph[6] = {0, 0, 0, 0, 0, 0}, iters = 0, maxit = 0;
        size_t cnt = 0;
        for (size_t i = 0; i < c->J.n_huf_big; i++) {
            if (!d[i * 8 + 6]) continue;
            for (int k = 0; k < 6; k++) ph[k] += (double)(d[i * 8 + k + 1] - d[i * 8 + k]);
            iters += (double)d[i * 8 + 7]; if ((double)d[i * 8 + 7] > maxit) maxit = (double)d[i * 8 + 7];
            cnt++;
        }
        if (q[4]) fprintf(stderr, "[seq debug] %llu sequences: producer %.0f cycles work + %.0f waiting, consumer %.0f work + %.0f waiting (per sequence)\n", q[4],
                          (double)q[0] / q[4], (double)q[1] / q[4], (double)q[2] / q[4], (double)q[3] / q[4]);
        if (q[7]) fprintf(stderr, "[lz small debug] cycles: probe %llu, copy %llu, all rounds %llu\n", q[5], q[6], q[7]);
        if (cnt) fprintf(stderr, "[huf debug] big CTAs %zu: cycles stage+weights %.0f, table %.0f, sync %.0f (iters avg %.2f max %.0f), scan %.0f, write %.0f, flush %.0f\n",
                         cnt, ph[0] / cnt, ph[1] / cnt, ph[2] / cnt, iters / cnt, maxit, ph[3] / cnt, ph[4] / cnt, ph[5] / cnt);
    }
    read_lz_stats(c);
    const uint8_t* R = (const uint8_t*)c->result.p;
    int first_code = 0;
    for (uint32_t a = 0; a < n; a++) {
        const nk::NafDev& D = c->arch[a];
        const ArchPlan& P = c->aplan[a];
        nafgpu_result& r = out[a];
        memset(&r, 0, sizeof r);
        r.n_records = P.n_records;
        const Outcome o = archive_outcome(c, a);
        r.first_bad_record = o.first_bad_record;
        r.record_status = o.record_status;
        if (o.status) {
            r.status = o.status;
            if (!first_code) { first_code = o.status; c->err = o.msg; }
            continue;
        }
        r.n_ids = o.n_ids;
        r.n_comments = o.n_comments;
        r.n_lengths = o.C->n_lengths;
        r.total_residues = o.C->total_residues;
        if (P.dec[0]) { r.ids = R + D.ids_off; r.id_offsets = (const uint64_t*)(R + D.id_offsets_off); }
        if (P.dec[1]) { r.comments = R + D.com_off; r.comment_offsets = (const uint64_t*)(R + D.com_offsets_off); }
        if (P.dec[2]) { r.lengths = (const uint64_t*)(R + D.lengths_off); r.record_offsets = (const uint64_t*)(R + D.rec_offsets_off); }
        if (P.dec[4]) r.sequence = R + D.ascii_off;
        if (P.dec[5]) r.quality = R + D.qual_off;
    }
    return (n == 1) ? first_code : NAFGPU_OK;
}

// FASTA / FASTQ text of the job that was just run, formatted on the device (naf_text.cu); only the text crosses PCIe.
int nafgpu_job_format(nafgpu_ctx* c, int format, uint64_t line_length, nafgpu_text* out, uint32_t n) {
    if (!c || (!out && n)) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared || !c->ran) return fail(c, NAFGPU_ERR_ARGUMENT, "job has not been run");
    if (n != c->arch.size()) return fail(c, NAFGPU_ERR_ARGUMENT, "result count differs from the prepared job");
    if (format != NAFGPU_TEXT_AUTO && format != NAFGPU_TEXT_FASTA && format != NAFGPU_TEXT_FASTQ) return fail(c, NAFGPU_ERR_ARGUMENT, "bad text format");
    CUDA_TRY(c, cudaSetDevice(c->device));
    // layout of the text buffer: sizes[n] | text of every archive (copied back) | record offsets (device only)
    std::vector<nk::TextDev> td(n);
    uint64_t off = align_up((uint64_t)n * 8), max_cap = 0;
    for (uint32_t a = 0; a < n; a++) {
        const ArchPlan& P = c->aplan[a];
        const nk::NafDev& D = c->arch[a];
        const bool skipped = P.host_status != 0;          // (not decoded: no text, its status is reported; D.n_records is 0)
        if (!skipped && !P.dec[NAFGPU_SEC_SEQUENCE]) return fail(c, NAFGPU_ERR_ARGUMENT, "text output needs the sequence (and lengths) decoded");
        const bool fastq = format == NAFGPU_TEXT_FASTQ || (format == NAFGPU_TEXT_AUTO && P.dec[NAFGPU_SEC_QUALITY]);
        if (!skipped && fastq && !P.dec[NAFGPU_SEC_QUALITY]) return fail(c, NAFGPU_ERR_ARGUMENT, "FASTQ output needs the quality section decoded");
        if (D.n_records > (1ull << 36)) return fail(c, NAFGPU_ERR_NOMEM, "text of an archive with more than 2^36 records does not fit the device");
        nk::TextDev& T = td[a];
        T.fastq = fastq ? 1u : 0u;
        T.sep = P.sep;
        T.line_length = fastq ? 0 : (line_length == NAFGPU_LINE_LENGTH_FROM_HEADER ? P.line_length : line_length);
        const uint64_t nrec = D.n_records, res = D.seq_residues;
        T.cap = 3 * nrec + P.blob_size[0] + P.blob_size[1] +
                (fastq ? 2 * res + 4 * nrec : res + (T.line_length ? res / T.line_length + nrec : nrec)) + 16;
        T.text_off = off;
        off = align_up(off + T.cap);
        max_cap = std::max(max_cap, T.cap);
    }
    const uint64_t copy_size = off;
    for (uint32_t a = 0; a < n; a++) { td[a].offs_off = off; off = align_up(off + 8 * (c->arch[a].n_records + 1)); }
    if (!c->text.ensure(off + 64 + (uint64_t)n * sizeof(nk::TextDev))) return fail(c, NAFGPU_ERR_NOMEM, "device allocation failed");
    if (!c->text_host.ensure(copy_size + 64) || !c->text_stage.ensure((uint64_t)n * sizeof(nk::TextDev) + 64) || !c->result.ensure(c->counts_size + 64))
        return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));                  // text_stage may still feed an earlier call's copy
    uint8_t* tdev = (uint8_t*)c->text.p + off;                  // descriptors behind the offsets (off is 128 B aligned)
    if (n) {
        memcpy(c->text_stage.p, td.data(), (size_t)n * sizeof(nk::TextDev));
        CUDA_TRY(c, cudaMemcpyAsync(tdev, c->text_stage.p, (size_t)n * sizeof(nk::TextDev), cudaMemcpyHostToDevice, c->streams.st));
    }
    CUDA_TRY(c, cudaEventRecord(c->ev[0], c->streams.st));
    nk::launch_text_stage((uint8_t*)c->arena.p, (const nk::NafDev*)((const uint8_t*)c->desc.p + c->o_naf), (uint8_t*)c->text.p,
                          (const nk::TextDev*)tdev, n, max_cap, c->J.status, c->streams.st);
    CUDA_TRY(c, cudaEventRecord(c->ev[1], c->streams.st));
    CUDA_TRY(c, cudaGetLastError());
    {
        CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
        std::lock_guard<std::mutex> turn(g_d2h_turn[c->device & 15]);
        CUDA_TRY(c, cudaMemcpyAsync(c->misc_host.p, c->misc.p, c->misc_words * 4, cudaMemcpyDeviceToHost, c->streams.st));
        CUDA_TRY(c, cudaMemcpyAsync(c->result.p, c->arena.p, c->counts_size, cudaMemcpyDeviceToHost, c->streams.st));
        CUDA_TRY(c, cudaMemcpyAsync(c->text_host.p, c->text.p, copy_size, cudaMemcpyDeviceToHost, c->streams.st));
        CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    }
    read_lz_stats(c);
    if (words(c).status & zc::E_INTERNAL) return fail(c, NAFGPU_ERR_INVALID_DATA, "text layout exceeded its bound");
    const uint8_t* H = (const uint8_t*)c->text_host.p;
    c->stats.text_kernel_ms = 0; c->stats.text_bytes = 0;
    cudaEventElapsedTime(&c->stats.text_kernel_ms, c->ev[0], c->ev[1]);
    int first_code = 0;
    for (uint32_t a = 0; a < n; a++) {
        nafgpu_text& t = out[a];
        memset(&t, 0, sizeof t);
        t.format = td[a].fastq ? NAFGPU_TEXT_FASTQ : NAFGPU_TEXT_FASTA;
        const Outcome o = archive_outcome(c, a);
        t.first_bad_record = o.first_bad_record;
        if (o.status) {
            t.status = o.status;
            if (!first_code) { first_code = o.status; c->err = o.msg; }
            continue;
        }
        t.data = H + td[a].text_off;
        t.size = ((const uint64_t*)H)[a];
        c->stats.text_bytes += t.size;
        t.status = o.record_status;
    }
    return (n == 1) ? first_code : NAFGPU_OK;
}

int nafgpu_format_batch(nafgpu_ctx* c, const nafgpu_archive* archives, uint32_t n, uint32_t want, int format, uint64_t line_length, nafgpu_text* out) {
    int rc = nafgpu_job_prepare(c, archives, n, want);
    if (rc) return rc;
    rc = nafgpu_job_run(c);
    if (rc) return rc;
    return nafgpu_job_format(c, format, line_length, out, n);
}

int nafgpu_decode_batch(nafgpu_ctx* c, const nafgpu_archive* archives, uint32_t n, uint32_t want, nafgpu_result* out) {
    int rc = nafgpu_job_prepare(c, archives, n, want);
    if (rc) return rc;
    rc = nafgpu_job_run(c);
    if (rc) return rc;
    return nafgpu_job_fetch(c, out, n);
}

int nafgpu_decode(nafgpu_ctx* c, const nafgpu_archive* archive, uint32_t want, nafgpu_result* out) {
    return nafgpu_decode_batch(c, archive, 1, want, out);
}

int nafgpu_job_get_stats(const nafgpu_ctx* c, nafgpu_job_stats* out) {
    if (!c || !out) return NAFGPU_ERR_ARGUMENT;
    *out = c->stats;
    return NAFGPU_OK;
}

int nafgpu_job_time(nafgpu_ctx* c, int iters, int flush_l2, float* total_ms) {
    if (!c || !total_ms || iters <= 0) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared) return fail(c, NAFGPU_ERR_ARGUMENT, "no prepared job");
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (flush_l2 && !c->flush.ensure(FLUSH_BYTES)) return fail(c, NAFGPU_ERR_NOMEM, "flush buffer allocation failed");
#if !defined(NAFGPU_EMULATE)
    // Capture one decode into a CUDA graph so that the timed interval holds device work, not launch latency.
    if (!c->graph) {
        cudaGraph_t g = nullptr;
        CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
        CUDA_TRY(c, cudaStreamBeginCapture(c->streams.st, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_run(c, nullptr);
        cudaError_t e = cudaStreamEndCapture(c->streams.st, &g);
        if (rc) { if (g) cudaGraphDestroy(g); return rc; }
        if (e != cudaSuccess) return fail(c, NAFGPU_ERR_CUDA, std::string("graph capture failed: ") + cudaGetErrorString(e));
        e = cudaGraphInstantiate(&c->graph, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) { c->graph = nullptr; return fail(c, NAFGPU_ERR_CUDA, std::string("graph instantiate failed: ") + cudaGetErrorString(e)); }
    }
#endif
    double total = 0;
    for (int i = 0; i < iters; i++) {
        if (flush_l2) CUDA_TRY(c, cudaMemsetAsync(c->flush.p, i & 0xFF, FLUSH_BYTES, c->streams.st));
        CUDA_TRY(c, cudaEventRecord(c->ev[0], c->streams.st));
#if !defined(NAFGPU_EMULATE)
        CUDA_TRY(c, cudaGraphLaunch(c->graph, c->streams.st));
        c->ran = true;
#else
        int rc = enqueue_run(c, nullptr);
        if (rc) return rc;
#endif
        CUDA_TRY(c, cudaEventRecord(c->ev[1], c->streams.st));
        CUDA_TRY(c, cudaEventSynchronize(c->ev[1]));
        float ms = 0;
        CUDA_TRY(c, cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
        total += ms;
    }
    *total_ms = (float)total;
    return NAFGPU_OK;
}

int nafgpu_job_run_profiled(nafgpu_ctx* c, float* stage_ms, uint32_t n_stages) {
    if (!c || !stage_ms || n_stages < (uint32_t)N_STAGES + 1) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared) return fail(c, NAFGPU_ERR_ARGUMENT, "no prepared job");
    CUDA_TRY(c, cudaSetDevice(c->device));
    // memsets first, then the start mark, so that stage 0 is the first kernel only
    StageEvents se;
    se.ev = c->ev + 1; se.cap = N_STAGES; se.st = c->streams.st;
    se.kb = c->ev[N_STAGES + 1]; se.ke = c->ev[N_STAGES + 2];
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    // enqueue_run issues its memsets before the first kernel; record the start after them by splitting here:
    CUDA_TRY(c, cudaEventRecord(c->ev[0], c->streams.st));
    int rc = enqueue_run(c, &se);
    if (rc) return rc;
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    for (int i = 0; i < N_STAGES; i++) {
        float ms = 0;
        if (i < se.n) CUDA_TRY(c, cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]));
        stage_ms[i] = ms;
    }
    stage_ms[N_STAGES] = 0;                       // the dominant kernel alone (the Huffman kernel of the big streams)
    if (se.k_used) CUDA_TRY(c, cudaEventElapsedTime(&stage_ms[N_STAGES], se.kb, se.ke));
    return NAFGPU_OK;
}

const char* nafgpu_stage_name(uint32_t s) {
    static const char* names[N_STAGES] = {"memset+huf_decode", "build_tables", "decode_sequences", "frame_scan", "lz_literals", "lz_first",
                                          "lz_resolve", "lz_finish", "naf_scan", "mask_fix", "-", "unpack", "utf8_check"};
    return s < (uint32_t)N_STAGES ? names[s] : (s == (uint32_t)N_STAGES ? "huf_big_kernel" : "?");
}

// Encode side: pack + length words + mask runs of one archive's records (include/nafgpu.h).
int nafgpu_pack(nafgpu_ctx* c, const nafgpu_pack_input* in, nafgpu_pack_result* out) {
    if (!c || !in || !out) return NAFGPU_ERR_ARGUMENT;
    if ((in->n_residues && !in->sequence) || (in->n_records && !in->lengths)) return fail(c, NAFGPU_ERR_ARGUMENT, "null input");
    if (in->sequence_type < 0 || in->sequence_type > 1) return fail(c, NAFGPU_ERR_ARGUMENT, "only nucleotide sequences are packed (protein / text go to the compressor verbatim)");
    if (in->n_residues > (1ull << 38) || in->n_records > (1ull << 36)) return fail(c, NAFGPU_ERR_NOMEM, "archive does not fit the device");
    memset(out, 0, sizeof *out);
    out->first_invalid = ~0ull;
    uint64_t total = 0, n_words = 0;
    for (uint64_t i = 0; i < in->n_records; i++) {
        if (in->lengths[i] > in->n_residues - total) return fail(c, NAFGPU_ERR_ARGUMENT, "record lengths exceed the sequence (Error::InvalidLength)");
        total += in->lengths[i];
        n_words += in->lengths[i] / 0xFFFFFFFFull + 1;
    }
    if (total != in->n_residues) return fail(c, NAFGPU_ERR_ARGUMENT, "record lengths do not add up to the sequence (Error::InvalidLength)");
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    const uint64_t nres = in->n_residues, npacked = (nres + 1) / 2;
    // device input: [sequence (padded to 32) | lengths]; device output: [counters 4 x u64 | length words | packed | mask | flag words]
    const uint64_t i_len = align_up(nres + 32), in_bytes = i_len + 8 * in->n_records + 64;
    const uint64_t o_words = 64, o_packed = align_up(o_words + 4 * n_words), o_mask = align_up(o_packed + npacked + 16);
    const uint64_t mask_cap = in->extract_mask ? nres / 255 + nres + 16 : 0;     // every residue its own run, at worst
    const uint64_t o_low = align_up(o_mask + mask_cap), out_bytes = o_low + (in->extract_mask ? 4 * ((nres + 31) / 32) : 0) + 64;
    if (!c->pack_in.ensure(in_bytes) || !c->pack_out.ensure(out_bytes)) return fail(c, NAFGPU_ERR_NOMEM, "device allocation failed");
    uint8_t* di = (uint8_t*)c->pack_in.p;
    uint8_t* dout = (uint8_t*)c->pack_out.p;
    if (nres) CUDA_TRY(c, cudaMemcpyAsync(di, in->sequence, nres, cudaMemcpyHostToDevice, c->streams.st));
    if (in->n_records) CUDA_TRY(c, cudaMemcpyAsync(di + i_len, in->lengths, 8 * in->n_records, cudaMemcpyHostToDevice, c->streams.st));
    CUDA_TRY(c, cudaMemsetAsync(dout, 0xFF, 8, c->streams.st));                          // first invalid residue: none
    CUDA_TRY(c, cudaMemsetAsync(dout + 8, 0, 24, c->streams.st));
    nk::launch_pack_stage(di, nres, (uint32_t)in->sequence_type, in->extract_mask != 0, dout + o_packed, (uint32_t*)(dout + o_low),
                          (const uint64_t*)(di + i_len), in->n_records, (uint32_t*)(dout + o_words), dout + o_mask,
                          (unsigned long long*)dout, c->streams.st);
    CUDA_TRY(c, cudaGetLastError());
    // the counters first (the mask size is only known now), then the streams themselves
    if (!c->pack_host.ensure(64)) return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
    CUDA_TRY(c, cudaMemcpyAsync(c->pack_host.p, dout, 32, cudaMemcpyDeviceToHost, c->streams.st));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    uint64_t cnt[4];
    memcpy(cnt, c->pack_host.p, 32);
    if (cnt[1] != n_words || cnt[2] > mask_cap) return fail(c, NAFGPU_ERR_CUDA, "pack stage produced inconsistent sizes");
    const uint64_t mask_size = in->extract_mask ? cnt[2] : 0;
    const uint64_t h_words = 64, h_packed = align_up(h_words + 4 * n_words), h_mask = align_up(h_packed + npacked + 16);
    if (!c->pack_host.ensure(h_mask + mask_size + 64)) return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
    uint8_t* H = (uint8_t*)c->pack_host.p;
    {
        std::lock_guard<std::mutex> turn(g_d2h_turn[c->device & 15]);
        if (n_words) CUDA_TRY(c, cudaMemcpyAsync(H + h_words, dout + o_words, 4 * n_words, cudaMemcpyDeviceToHost, c->streams.st));
        if (npacked) CUDA_TRY(c, cudaMemcpyAsync(H + h_packed, dout + o_packed, npacked, cudaMemcpyDeviceToHost, c->streams.st));
        if (mask_size) CUDA_TRY(c, cudaMemcpyAsync(H + h_mask, dout + o_mask, mask_size, cudaMemcpyDeviceToHost, c->streams.st));
        CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    }
    out->packed = H + h_packed; out->packed_size = npacked;
    out->length_words = H + h_words; out->length_size = 4 * n_words;
    if (in->extract_mask) { out->mask = H + h_mask; out->mask_size = mask_size; out->n_mask_runs = cnt[3]; }
    out->first_invalid = cnt[0];
    if (cnt[0] != ~0ull) {
        char b[96];
        snprintf(b, sizeof b, "unexpected sequence character at residue %llu", (unsigned long long)cnt[0]);
        return fail(c, NAFGPU_ERR_INVALID_DATA, b);
    }
    return NAFGPU_OK;
}

// Records [first, first + count) of one archive of the job that was run, through a pinned buffer that holds this window only:
// the result stays in HBM and crosses PCIe a window at a time, so the host memory a decode needs is bounded by the window,
// as the reference's is by its 4 KiB BufReaders (decoder/mod.rs:69,221-223), and record `first` is available after
// copying one window instead of the whole archive.  Two copies: the slices of the offset tables, then the bytes they span.
int nafgpu_job_fetch_window(nafgpu_ctx* c, uint32_t archive, uint64_t first, uint64_t count, uint64_t max_bytes, nafgpu_result* out) {
    if (!c || !out) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared || !c->ran) return fail(c, NAFGPU_ERR_ARGUMENT, "job has not been run");
    if (archive >= c->arch.size()) return fail(c, NAFGPU_ERR_ARGUMENT, "bad archive index");
    CUDA_TRY(c, cudaSetDevice(c->device));
    { int rc = read_counts(c); if (rc) return rc; }
    const nk::NafDev& D = c->arch[archive];
    const ArchPlan& P = c->aplan[archive];
    nafgpu_result& r = *out;
    memset(&r, 0, sizeof r);
    r.first_bad_record = nk::NO_RECORD;
    const Outcome o = archive_outcome(c, archive);
    if (o.status) { r.status = o.status; r.n_records = P.n_records; return fail(c, o.status, o.msg); }
    first = std::min<uint64_t>(first, P.n_records);
    count = std::min<uint64_t>(count, P.n_records - first);
    if (max_bytes) count = std::min<uint64_t>(count, max_bytes / 32 + 1);       // (a record takes 32 bytes of tables at least)
    const uint64_t n_ids = o.n_ids, n_com = o.n_comments, n_len = o.C->n_lengths;
    struct Slice { bool on; uint64_t lo, hi, src, dst; } id{P.dec[0], 0, 0, D.id_offsets_off, 0}, co{P.dec[1], 0, 0, D.com_offsets_off, 0}, le{P.dec[2], 0, 0, D.rec_offsets_off, 0};
    auto clampw = [&](Slice& s, uint64_t n) { s.lo = std::min(first, n); s.hi = std::min(first + count, n); };
    clampw(id, n_ids); clampw(co, n_com); clampw(le, n_len);
    // ---- copy 1: table slices (hi - lo + 1 offsets each; lengths hi - lo) ----
    uint64_t need = 0;
    for (Slice* s : {&id, &co, &le}) if (s->on) { s->dst = need; need += align_up((s->hi - s->lo + 1) * 8, 64); }
    const uint64_t len_dst = need;
    if (le.on) need += align_up((le.hi - le.lo) * 8 + 8, 64);
    const uint64_t tables_bytes = need;
    if (!c->win.ensure(tables_bytes + 64)) return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
    uint8_t* W = (uint8_t*)c->win.p;
    const uint8_t* A = (const uint8_t*)c->arena.p;
    for (Slice* s : {&id, &co, &le}) if (s->on) CUDA_TRY(c, cudaMemcpyAsync(W + s->dst, A + s->src + s->lo * 8, (s->hi - s->lo + 1) * 8, cudaMemcpyDeviceToHost, c->streams.st));
    if (le.on && le.hi > le.lo) CUDA_TRY(c, cudaMemcpyAsync(W + len_dst, A + D.lengths_off + le.lo * 8, (le.hi - le.lo) * 8, cudaMemcpyDeviceToHost, c->streams.st));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    // ---- fit the window to max_bytes (never less than one record) ----
    auto span = [&](const Slice& s, uint64_t k) -> uint64_t {      // bytes of the first k records of the window in this field
        if (!s.on) return 0;
        const uint64_t* o = (const uint64_t*)(W + s.dst);
        const uint64_t kk = std::min(k, s.hi - s.lo);
        return o[kk] - o[0];
    };
    const uint64_t per_res = (P.dec[4] ? 1 : 0) + (P.dec[5] ? 1 : 0);
    auto bytes_of = [&](uint64_t k) { return span(id, k) + span(co, k) + span(le, k) * per_res + k * 32; };
    if (max_bytes && count > 1 && bytes_of(count) > max_bytes) {
        uint64_t lo = 1, hi = count;                                 // largest k in [1, count] with bytes_of(k) <= max_bytes (bytes_of is monotone)
        while (lo < hi) { const uint64_t mid = (lo + hi + 1) / 2; if (bytes_of(mid) <= max_bytes) lo = mid; else hi = mid - 1; }
        count = lo;
        clampw(id, n_ids); clampw(co, n_com); clampw(le, n_len);
    }
    // ---- copy 2: the bytes the slices span ----
    const uint64_t id_bytes = span(id, count), co_bytes = span(co, count), res = span(le, count);
    const uint64_t id0 = id.on ? *(const uint64_t*)(W + id.dst) : 0, co0 = co.on ? *(const uint64_t*)(W + co.dst) : 0, r0 = le.on ? *(const uint64_t*)(W + le.dst) : 0;
    if (id0 + id_bytes > D.ids_size || co0 + co_bytes > D.com_size || (P.dec[4] && r0 + res > D.seq_residues) || (P.dec[5] && r0 + res > D.qual_size)) return fail(c, NAFGPU_ERR_INVALID_DATA, "offset tables exceed their sections");
    uint64_t o_ids = tables_bytes, o_com = o_ids + align_up(id_bytes + 1, 64), o_seq = o_com + align_up(co_bytes + 1, 64), o_qual = o_seq + (P.dec[4] ? align_up(res + 1, 64) : 0);
    need = o_qual + (P.dec[5] ? align_up(res + 1, 64) : 0);
    if (need + 64 > c->win.cap) {           // grow, keeping the tables
        std::vector<uint8_t> keep(W, W + tables_bytes);
        if (!c->win.ensure(need + 64)) return fail(c, NAFGPU_ERR_NOMEM, "pinned host allocation failed");
        W = (uint8_t*)c->win.p;
        memcpy(W, keep.data(), tables_bytes);
    }
    if (id_bytes) CUDA_TRY(c, cudaMemcpyAsync(W + o_ids, A + D.ids_off + id0, id_bytes, cudaMemcpyDeviceToHost, c->streams.st));
    if (co_bytes) CUDA_TRY(c, cudaMemcpyAsync(W + o_com, A + D.com_off + co0, co_bytes, cudaMemcpyDeviceToHost, c->streams.st));
    if (P.dec[4] && res) CUDA_TRY(c, cudaMemcpyAsync(W + o_seq, A + D.ascii_off + r0, res, cudaMemcpyDeviceToHost, c->streams.st));
    if (P.dec[5] && res) CUDA_TRY(c, cudaMemcpyAsync(W + o_qual, A + D.qual_off + r0, res, cudaMemcpyDeviceToHost, c->streams.st));
    CUDA_TRY(c, cudaStreamSynchronize(c->streams.st));
    // ---- the window as a result of its own: offsets rebased to the window's first byte ----
    for (Slice* s : {&id, &co, &le}) if (s->on) {
        uint64_t* o = (uint64_t*)(W + s->dst);
        const uint64_t base = o[0], n = s->hi - s->lo;
        for (uint64_t k = 0; k <= n; k++) o[k] -= base;
    }
    r.n_records = count;
    r.n_ids = id.hi - id.lo; r.n_comments = co.hi - co.lo; r.n_lengths = le.hi - le.lo;
    r.total_residues = res;
    if (id.on) { r.ids = W + o_ids; r.id_offsets = (const uint64_t*)(W + id.dst); }
    if (co.on) { r.comments = W + o_com; r.comment_offsets = (const uint64_t*)(W + co.dst); }
    if (le.on) { r.lengths = (const uint64_t*)(W + len_dst); r.record_offsets = (const uint64_t*)(W + le.dst); }
    if (P.dec[4]) r.sequence = W + o_seq;
    if (P.dec[5]) r.quality = W + o_qual;
    const uint64_t fb = o.first_bad_record;
    if (fb != nk::NO_RECORD && fb >= first && fb < first + count) { r.first_bad_record = fb - first; r.record_status = NAFGPU_ERR_UTF8; }
    return NAFGPU_OK;
}

int nafgpu_job_device_result(nafgpu_ctx* c, uint32_t archive, const uint8_t** sequence_dev, uint64_t* capacity_bytes) {
    if (!c || !sequence_dev || !capacity_bytes) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared || archive >= c->arch.size()) return fail(c, NAFGPU_ERR_ARGUMENT, "bad archive index");
    *sequence_dev = (const uint8_t*)c->arena.p + c->arch[archive].ascii_off;
    *capacity_bytes = c->arch[archive].seq_residues;
    return NAFGPU_OK;
}

int nafgpu_job_counts(nafgpu_ctx* c, nafgpu_counts* out, uint32_t n) {
    if (!c || (!out && n)) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared || !c->ran) return fail(c, NAFGPU_ERR_ARGUMENT, "job has not been run");
    if (n != c->arch.size()) return fail(c, NAFGPU_ERR_ARGUMENT, "count differs from the prepared job");
    CUDA_TRY(c, cudaSetDevice(c->device));
    { int rc = export_tables(c); if (rc) return rc; }
    if (n) memcpy(out, c->counts.data(), (size_t)n * sizeof(nafgpu_counts));
    return NAFGPU_OK;
}

int nafgpu_job_export(nafgpu_ctx* c, const nafgpu_export* spec, void* stream) {
    if (!c || !spec) return NAFGPU_ERR_ARGUMENT;
    if (!c->prepared || !c->ran) return fail(c, NAFGPU_ERR_ARGUMENT, "job has not been run");
    const int field = spec->field, layout = spec->layout;
    if (layout != NAFGPU_EXPORT_FLAT && layout != NAFGPU_EXPORT_ROWS && layout != NAFGPU_EXPORT_OFFSETS) return fail(c, NAFGPU_ERR_ARGUMENT, "bad export layout");
    int f = -1;                                         // index of the field among ids, comments, sequence, quality
    if (layout != NAFGPU_EXPORT_OFFSETS) {
        static const int fields[4] = {NAFGPU_SEC_ID, NAFGPU_SEC_COMMENT, NAFGPU_SEC_SEQUENCE, NAFGPU_SEC_QUALITY};
        static const uint32_t want_bit[4] = {NAFGPU_WANT_ID, NAFGPU_WANT_COMMENT, NAFGPU_WANT_SEQUENCE, NAFGPU_WANT_QUALITY};
        for (int k = 0; k < 4; k++) if (field == fields[k]) f = k;
        if (f < 0) return fail(c, NAFGPU_ERR_ARGUMENT, "bad export field");
        if (layout == NAFGPU_EXPORT_ROWS && f < 2) return fail(c, NAFGPU_ERR_ARGUMENT, "rows export of ids or comments: only sequence and quality have residues");
        if (!(c->want & want_bit[f])) return fail(c, NAFGPU_ERR_ARGUMENT, "export of a field that was not decoded (want bits of the job)");
    }
    if (layout == NAFGPU_EXPORT_ROWS && !spec->rows && spec->n_rows) return fail(c, NAFGPU_ERR_ARGUMENT, "rows export without a row table");
    if (layout == NAFGPU_EXPORT_ROWS && spec->row_length && spec->n_rows > UINT64_MAX / spec->row_length) return fail(c, NAFGPU_ERR_ARGUMENT, "rows export larger than 2^64 bytes");
    if (layout == NAFGPU_EXPORT_OFFSETS && ((uintptr_t)spec->out & 7)) return fail(c, NAFGPU_ERR_ARGUMENT, "offsets export: out must be 8-byte aligned");
    CUDA_TRY(c, cudaSetDevice(c->device));
    { int rc = export_tables(c); if (rc) return rc; }
    const uint64_t need = layout == NAFGPU_EXPORT_FLAT ? c->exp_bytes[f] : layout == NAFGPU_EXPORT_ROWS ? spec->n_rows * spec->row_length : 8 * (c->exp_records + 1);
    if (spec->out_bytes < need || (!spec->out && need)) {
        char b[128];
        snprintf(b, sizeof b, "export needs %llu bytes of output, out_bytes is %llu", (unsigned long long)need, (unsigned long long)spec->out_bytes);
        return fail(c, NAFGPU_ERR_ARGUMENT, b);
    }
    // ordering: the caller's stream waits for the run (and the descriptors' upload); the context's stream, where every later
    // call on this context enqueues its work, waits for the export
    cudaStream_t st = stream ? (cudaStream_t)stream : c->streams.st;
    if (st != c->streams.st) {
        CUDA_TRY(c, cudaEventRecord(c->ev_exp_ready, c->streams.st));
        CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_exp_ready, 0));
    }
    nk::ExpTable table;
    memcpy(table.b, spec->table, 256);
    bool identity = true;
    for (int i = 0; i < 256; i++) identity = identity && spec->table[i] == (uint8_t)i;
    const uint8_t* arena = (const uint8_t*)c->arena.p;
    const uint8_t* desc = (const uint8_t*)c->exp_desc.p;
    const nk::ExpRec* recs = (const nk::ExpRec*)desc;
    if (layout == NAFGPU_EXPORT_FLAT)
        nk::launch_export_flat(arena, (const nk::ExpSpan*)(desc + c->o_exp_span[f]), c->n_exp_span[f], need, table, identity, (uint8_t*)spec->out, c->sms, st);
    else if (layout == NAFGPU_EXPORT_ROWS)
        nk::launch_export_rows(arena, recs, c->n_exp_rec, c->exp_records, f == 3 ? 1u : 0u, spec->rows, spec->n_rows, spec->row_length, table, identity,
                               spec->pad, (uint8_t*)spec->out, c->sms, st);
    else
        nk::launch_export_offsets(arena, recs, c->n_exp_rec, c->exp_records, c->exp_residues, (int64_t*)spec->out, c->sms, st);
    CUDA_TRY(c, cudaGetLastError());
    if (st != c->streams.st) {
        CUDA_TRY(c, cudaEventRecord(c->ev_exp_done, st));
        CUDA_TRY(c, cudaStreamWaitEvent(c->streams.st, c->ev_exp_done, 0));
    }
    return NAFGPU_OK;
}

}  // extern "C"

// nafgpu_pipeline.cpp -- the overlap of H2D, kernels and D2H for callers of the C ABI (include/nafgpu.h, "pipeline").
//
// The reference seam is an iterator that a consumer drives (Decoder::next, nafcodec/src/decoder/mod.rs:444-457); a device
// backend that is only ever called synchronously leaves the copy engines idle while kernels run and the SMs idle while
// results travel.  A pipeline owns `lanes` contexts (each with its own streams, arenas and pinned result buffers) and as
// many host threads; batches are submitted without waiting, and while one lane copies its results back another walks
// headers, uploads and decodes.  This used to live in the Python mirror only (threads around nafgpu_decode_batch); a Rust or
// C++ caller now gets the same thing from three calls: submit, wait, release.
//
// A device ticket ends one step earlier: the lane decodes into its context's arena, reads the per-archive counters and leaves
// the sub-batch there; the caller exports from it (nafgpu_job_export on the lane's context) until it releases the ticket.
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nafgpu.h"

namespace {

struct Ticket {
    int64_t id = 0;
    const nafgpu_archive* archives = nullptr;
    uint32_t n = 0, want = 0;
    int rc = 0;
    int lane = -1;
    bool device = false;                       // a device ticket: the result stays in the lane's arena (counts, no D2H)
    bool done = false;
    bool waited = false;                       // a device ticket's counts were read by the caller: exports may follow
    std::vector<nafgpu_result> results;
    std::vector<nafgpu_counts> counts;
    std::string err;
    nafgpu_job_stats stats{};
};

}  // namespace

struct nafgpu_pipeline {
    int device = 0;
    std::vector<nafgpu_ctx*> ctx;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::deque<Ticket*> queue;                 // submitted, not yet taken by a lane
    std::deque<Ticket*> tickets;               // every ticket that has not been released
    int64_t next_id = 0;
    bool stop = false;
    std::string err;
    std::vector<nafgpu_job_stats> lane_stats;
    std::vector<char> lane_holds;             // lane's pinned buffers hold the results of a ticket that has not been released
    // exports of a device ticket run on the lane's context from the caller's threads: one at a time per lane, and never while
    // release hands the lane back to its thread (a context is not thread-safe)
    std::vector<std::unique_ptr<std::mutex>> lane_export;
};

// Decode a device ticket on its lane: prepare + run + counts, nothing copied back.
static int decode_device(nafgpu_ctx* c, Ticket* t) {
    t->counts.assign(t->n, nafgpu_counts{});
    int rc = nafgpu_job_prepare(c, t->archives, t->n, t->want);
    if (!rc) rc = nafgpu_job_run(c);
    if (!rc) rc = nafgpu_job_counts(c, t->counts.data(), t->n);
    return rc;
}

static void lane_main(nafgpu_pipeline* p, int lane) {
    for (;;) {
        Ticket* t = nullptr;
        {
            std::unique_lock<std::mutex> lk(p->mu);
            p->cv_work.wait(lk, [&] { return p->stop || !p->queue.empty(); });
            if (p->stop && p->queue.empty()) return;
            t = p->queue.front();
            p->queue.pop_front();
            t->lane = lane;
        }
        int rc;
        if (t->device) {
            rc = decode_device(p->ctx[lane], t);
        } else {
            t->results.assign(t->n, nafgpu_result{});
            rc = nafgpu_decode_batch(p->ctx[lane], t->archives, t->n, t->want, t->results.data());
        }
        nafgpu_job_stats st{};
        nafgpu_job_get_stats(p->ctx[lane], &st);
        {
            std::unique_lock<std::mutex> lk(p->mu);
            t->rc = rc;
            if (rc) t->err = nafgpu_last_error(p->ctx[lane]);
            t->stats = st;
            p->lane_stats[lane] = st;
            t->done = true;
            p->lane_holds[lane] = 1;
            p->cv_done.notify_all();
            // the lane's pinned buffers (a device ticket: its arena) hold this ticket's results: it takes no new work before
            // they are released
            // (the ticket itself belongs to the caller from here on: release frees it)
            p->cv_done.wait(lk, [&] { return !p->lane_holds[lane] || p->stop; });
        }
    }
}

extern "C" {

int nafgpu_pipeline_create(int device, uint32_t lanes, nafgpu_pipeline** out) {
    if (!out || lanes == 0 || lanes > 64) return NAFGPU_ERR_ARGUMENT;
    *out = nullptr;
    nafgpu_pipeline* p = new nafgpu_pipeline();
    p->device = device;
    p->lane_stats.assign(lanes, nafgpu_job_stats{});
    p->lane_holds.assign(lanes, 0);
    for (uint32_t i = 0; i < lanes; i++) p->lane_export.emplace_back(new std::mutex());
    for (uint32_t i = 0; i < lanes; i++) {
        nafgpu_ctx* c = nullptr;
        const int rc = nafgpu_ctx_create(device, &c);
        if (rc) {
            for (nafgpu_ctx* x : p->ctx) nafgpu_ctx_destroy(x);
            delete p;
            return rc;
        }
        p->ctx.push_back(c);
    }
    for (uint32_t i = 0; i < lanes; i++) p->workers.emplace_back(lane_main, p, (int)i);
    *out = p;
    return NAFGPU_OK;
}

void nafgpu_pipeline_destroy(nafgpu_pipeline* p) {
    if (!p) return;
    {
        std::unique_lock<std::mutex> lk(p->mu);
        p->stop = true;
        p->cv_work.notify_all();
        p->cv_done.notify_all();
    }
    for (std::thread& t : p->workers) t.join();
    for (Ticket* t : p->tickets) delete t;
    for (nafgpu_ctx* c : p->ctx) nafgpu_ctx_destroy(c);
    delete p;
}

static int64_t submit(nafgpu_pipeline* p, const nafgpu_archive* archives, uint32_t n, uint32_t want, bool device) {
    if (!p || (!archives && n)) return NAFGPU_ERR_ARGUMENT;
    Ticket* t = new Ticket();
    t->archives = archives; t->n = n; t->want = want; t->device = device;
    std::unique_lock<std::mutex> lk(p->mu);
    t->id = p->next_id++;
    p->tickets.push_back(t);
    p->queue.push_back(t);
    p->cv_work.notify_one();
    return t->id;
}

int64_t nafgpu_pipeline_submit(nafgpu_pipeline* p, const nafgpu_archive* archives, uint32_t n, uint32_t want) {
    return submit(p, archives, n, want, false);
}

int64_t nafgpu_pipeline_submit_device(nafgpu_pipeline* p, const nafgpu_archive* archives, uint32_t n, uint32_t want) {
    return submit(p, archives, n, want, true);
}

static Ticket* find_ticket(nafgpu_pipeline* p, int64_t id) {
    for (Ticket* t : p->tickets) if (t->id == id) return t;
    return nullptr;
}

int nafgpu_pipeline_wait(nafgpu_pipeline* p, int64_t ticket, nafgpu_result* out, uint32_t n) {
    if (!p || (!out && n)) return NAFGPU_ERR_ARGUMENT;
    std::unique_lock<std::mutex> lk(p->mu);
    Ticket* t = find_ticket(p, ticket);
    if (!t || t->n != n) { p->err = "unknown ticket or wrong result count"; return NAFGPU_ERR_ARGUMENT; }
    if (t->device) { p->err = "nafgpu_pipeline_wait on a device ticket: use nafgpu_pipeline_wait_counts"; return NAFGPU_ERR_ARGUMENT; }
    p->cv_done.wait(lk, [&] { return t->done; });
    for (uint32_t i = 0; i < n; i++) out[i] = t->results[i];
    if (t->rc) p->err = t->err;
    return t->rc;
}

int nafgpu_pipeline_wait_counts(nafgpu_pipeline* p, int64_t ticket, nafgpu_counts* out, uint32_t n) {
    if (!p || (!out && n)) return NAFGPU_ERR_ARGUMENT;
    std::unique_lock<std::mutex> lk(p->mu);
    Ticket* t = find_ticket(p, ticket);
    if (!t || t->n != n) { p->err = "unknown ticket or wrong count"; return NAFGPU_ERR_ARGUMENT; }
    if (!t->device) { p->err = "nafgpu_pipeline_wait_counts on a host ticket: use nafgpu_pipeline_wait"; return NAFGPU_ERR_ARGUMENT; }
    p->cv_done.wait(lk, [&] { return t->done; });
    for (uint32_t i = 0; i < n; i++) out[i] = t->counts[i];
    t->waited = true;
    if (t->rc) p->err = t->err;
    return t->rc;
}

int nafgpu_pipeline_export(nafgpu_pipeline* p, int64_t ticket, const nafgpu_export* spec, void* stream) {
    if (!p || !spec) return NAFGPU_ERR_ARGUMENT;
    std::unique_lock<std::mutex> lk(p->mu);
    Ticket* t = find_ticket(p, ticket);
    const char* why = !t ? "export from an unknown or released ticket"
                    : !t->device ? "export from a host ticket"
                    : !t->waited ? "export from a ticket that was not waited for (nafgpu_pipeline_wait_counts)"
                    : t->rc ? "export from a ticket whose decode failed" : nullptr;
    if (why) { p->err = why; return NAFGPU_ERR_ARGUMENT; }
    nafgpu_ctx* c = p->ctx[t->lane];
    std::unique_lock<std::mutex> turn(*p->lane_export[t->lane]);   // (taken under mu: release cannot slip in between)
    lk.unlock();
    const int rc = nafgpu_job_export(c, spec, stream);
    if (rc) {
        const std::string msg = nafgpu_last_error(c);
        turn.unlock();                                              // (release takes mu, then the turn: never the other way)
        lk.lock();
        p->err = msg;
    }
    return rc;
}

int nafgpu_pipeline_release(nafgpu_pipeline* p, int64_t ticket) {
    if (!p) return NAFGPU_ERR_ARGUMENT;
    std::unique_lock<std::mutex> lk(p->mu);
    for (auto it = p->tickets.begin(); it != p->tickets.end(); ++it) {
        if ((*it)->id != ticket) continue;
        Ticket* t = *it;
        if (!t->done) { p->err = "ticket released before it was waited for"; return NAFGPU_ERR_ARGUMENT; }
        { std::lock_guard<std::mutex> turn(*p->lane_export[t->lane]); }    // an export of this ticket in flight ends first
        p->lane_holds[t->lane] = 0;
        p->tickets.erase(it);
        p->cv_done.notify_all();
        lk.unlock();
        delete t;
        return NAFGPU_OK;
    }
    p->err = "unknown ticket";
    return NAFGPU_ERR_ARGUMENT;
}

const char* nafgpu_pipeline_last_error(const nafgpu_pipeline* p) { return p ? p->err.c_str() : "null pipeline"; }

uint32_t nafgpu_pipeline_lanes(const nafgpu_pipeline* p) { return p ? (uint32_t)p->ctx.size() : 0; }

int nafgpu_pipeline_lane_stats(nafgpu_pipeline* p, uint32_t lane, nafgpu_job_stats* out) {
    if (!p || !out || lane >= p->ctx.size()) return NAFGPU_ERR_ARGUMENT;
    std::unique_lock<std::mutex> lk(p->mu);
    *out = p->lane_stats[lane];
    return NAFGPU_OK;
}

}  // extern "C"

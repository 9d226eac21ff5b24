/* nnsp_group.cpp -- several devices behind one handle: streams block-partitioned over the GPUs of one box, one host
 * thread per device, no inter-GPU traffic (SURVEY.md section 8e: the streams are independent, weights are replicated,
 * a stream's state stays on its GPU for its lifetime).
 *
 * What it stands for in the reference: nothing -- the reference is one instance on one core (nn_speech.c:74-127,
 * evb/src/nnCntrlClass.c:152-272). A member of the group IS an nnsp_b200_batch / nnsp_b200_cascade handle (the batched
 * NNSPClass_exec / nnCntrlClass_exec); the group only hands each member its slice of the caller's host buffers:
 * member k owns streams [S k / G, S (k + 1) / G).
 *
 * Host code only (C++ threads over the library's own C ABI): no CUDA call is made here, and no collective exists. */
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <mutex>
#include <new>
#include <thread>
#include <utility>
#include <vector>

#include "nnsp_b200.h"
#include "nnsp_model.h"

namespace {

struct Command {
    enum Kind { EXEC, RESET, QUIT, RESET_STREAMS, IMPORT_STREAMS, EXPORT_STREAMS } kind;
    const int16_t *pcm;
    long long stride;
    int n_frames;                    /* RESET_STREAMS: the mode */
    void *results;                   /* EXPORT_STREAMS: the caller's records */
    long long seq;                   /* RESET_ / IMPORT_STREAMS: complete once recorded and the call before it is complete */
    std::vector<int32_t> streams;    /* *_STREAMS: the member's own streams, in its numbering */
    std::vector<int32_t> where;      /* EXPORT_STREAMS: the record of streams[i] is record where[i] of the caller's */
    std::vector<unsigned char> records;   /* IMPORT_STREAMS: the records of streams, a copy */
};

struct Member {
    int device = 0, first = 0, count = 0;
    nnsp_b200_batch *batch = nullptr;
    nnsp_b200_cascade *cascade = nullptr;
    std::thread thread;
    std::mutex mu;
    std::condition_variable cv_cmd, cv_done;
    std::deque<Command> queue;
    long long done_seq = 0;          /* every command up to this one is complete (results in the caller's buffer) */
    int status = NNSP_B200_OK;       /* first error of this member */
    char error[256] = { 0 };
};

}  // namespace

struct nnsp_b200_group {
    bool is_cascade = false;
    int n_streams = 0;
    long long seq = 0;
    std::vector<Member *> members;
};

namespace {

int member_exec_async(Member *m, const Command &c, long long *ticket)
{
    const int16_t *pcm = c.pcm + (long long)m->first * c.stride;
    if (m->cascade) {
        nnsp_b200_cascade_result *r = c.results ? (nnsp_b200_cascade_result *)c.results + (size_t)m->first * c.n_frames : nullptr;
        return nnsp_b200_cascade_exec_host_async(m->cascade, pcm, c.stride, c.n_frames, r, ticket);
    }
    nnsp_b200_result *r = c.results ? (nnsp_b200_result *)c.results + (size_t)m->first * c.n_frames : nullptr;
    return nnsp_b200_batch_exec_host_async(m->batch, pcm, c.stride, c.n_frames, r, ticket);
}
int member_wait(Member *m, long long ticket)
{
    return m->cascade ? nnsp_b200_cascade_wait_host(m->cascade, ticket) : nnsp_b200_batch_wait_host(m->batch, ticket);
}

/* One host thread per device. A call is queued on the device asynchronously and completed (results waited for) only
 * when the next command is there or nothing else is: the H2D of call n + 1 then overlaps the tail of call n, exactly
 * like the two-buffer serving loop of INTEGRATION.md, on every device at once. */
void worker(Member *m)
{
    long long inflight_seq = 0, inflight_ticket = 0;
    long long passed_seq = 0;        /* a reset recorded while a call was in flight: complete when that call is */
    auto fail = [&](int rc) {
        std::lock_guard<std::mutex> lk(m->mu);
        if (m->status == NNSP_B200_OK) {
            m->status = rc;
            snprintf(m->error, sizeof m->error, "device %d: %s", m->device, nnsp_b200_last_error());
        }
    };
    auto finish_inflight = [&]() {
        if (!inflight_seq) return;
        const int rc = member_wait(m, inflight_ticket);
        if (rc) fail(rc);
        {
            std::lock_guard<std::mutex> lk(m->mu);
            m->done_seq = passed_seq > inflight_seq ? passed_seq : inflight_seq;
        }
        m->cv_done.notify_all();
        inflight_seq = 0;
        passed_seq = 0;
    };
    for (;;) {
        Command c;
        {
            std::unique_lock<std::mutex> lk(m->mu);
            if (m->queue.empty() && inflight_seq) {            /* nothing to overlap with: complete what is in flight */
                lk.unlock();
                finish_inflight();
                lk.lock();
            }
            m->cv_cmd.wait(lk, [&] { return !m->queue.empty(); });
            c = std::move(m->queue.front());
            m->queue.pop_front();
        }
        if (c.kind == Command::QUIT) { finish_inflight(); return; }
        if (c.kind == Command::RESET_STREAMS || c.kind == Command::IMPORT_STREAMS) {   /* recorded on the handle, applied by its next call */
            const int rc = c.kind == Command::RESET_STREAMS
                               ? nnsp_b200_cascade_reset_streams(m->cascade, c.streams.data(), (int)c.streams.size(), c.n_frames)
                               : nnsp_b200_cascade_import_streams(m->cascade, c.streams.data(), (int)c.streams.size(), c.records.data());
            if (rc) fail(rc);
            if (inflight_seq) { passed_seq = c.seq; continue; }
            { std::lock_guard<std::mutex> lk(m->mu); m->done_seq = c.seq; }
            m->cv_done.notify_all();
            continue;
        }
        if (c.kind == Command::EXPORT_STREAMS) {                /* synchronous: the member's device is idle afterwards */
            finish_inflight();
            const size_t rb = nnsp_b200_cascade_stream_state_bytes(m->cascade), n = c.streams.size();
            unsigned char *out = static_cast<unsigned char *>(c.results);
            int rc = NNSP_B200_OK;
            if (n && c.where[n - 1] - c.where[0] + 1 == (int32_t)n)   /* the member's records are one range of the caller's */
                rc = nnsp_b200_cascade_export_streams(m->cascade, c.streams.data(), (int)n, out + rb * (size_t)c.where[0]);
            else if (n) {
                std::vector<unsigned char> tmp(rb * n);
                rc = nnsp_b200_cascade_export_streams(m->cascade, c.streams.data(), (int)n, tmp.data());
                for (size_t i = 0; !rc && i < n; i++) memcpy(out + rb * (size_t)c.where[i], tmp.data() + rb * i, rb);
            }
            if (rc) fail(rc);
            { std::lock_guard<std::mutex> lk(m->mu); m->done_seq = c.seq; }
            m->cv_done.notify_all();
            continue;
        }
        if (c.kind == Command::RESET) {
            finish_inflight();
            const int rc = m->cascade ? nnsp_b200_cascade_reset(m->cascade) : nnsp_b200_batch_reset(m->batch);
            if (rc) fail(rc);
            { std::lock_guard<std::mutex> lk(m->mu); m->done_seq = c.seq; }
            m->cv_done.notify_all();
            continue;
        }
        long long ticket = 0;
        const int rc = member_exec_async(m, c, &ticket);       /* queued behind the call in flight, on the device's own streams */
        finish_inflight();
        if (rc) {
            fail(rc);
            { std::lock_guard<std::mutex> lk(m->mu); m->done_seq = c.seq; }
            m->cv_done.notify_all();
        } else {
            inflight_seq = c.seq;
            inflight_ticket = ticket;
        }
    }
}

int post(nnsp_b200_group *g, Command c, long long *ticket)
{
    c.seq = ++g->seq;
    for (Member *m : g->members) {
        { std::lock_guard<std::mutex> lk(m->mu); m->queue.push_back(c); }
        m->cv_cmd.notify_one();
    }
    if (ticket) *ticket = c.seq;
    return NNSP_B200_OK;
}

int create(nnsp_b200_group *g, int n_streams, const int *devices, int n_devices)
{
    if (n_streams < n_devices) { nnsp_set_error("group: fewer streams (%d) than devices (%d)", n_streams, n_devices); return NNSP_B200_ERR_ARG; }
    g->n_streams = n_streams;
    for (int k = 0; k < n_devices; k++) {
        Member *m = new (std::nothrow) Member();
        if (!m) return NNSP_B200_ERR_NOMEM;
        m->device = devices[k];
        m->first = (int)((long long)n_streams * k / n_devices);
        m->count = (int)((long long)n_streams * (k + 1) / n_devices) - m->first;
        g->members.push_back(m);
    }
    return NNSP_B200_OK;
}

}  // namespace

extern "C" {

int nnsp_b200_group_create_batch(const nnsp_b200_model *model, int n_streams, const int *devices, int n_devices,
                                 int16_t thresh_prob, int16_t th_count_trigger, nnsp_b200_group **out)
{
    if (!model || !devices || !out || n_devices < 1 || n_streams < 1) return NNSP_B200_ERR_ARG;
    nnsp_b200_group *g = new (std::nothrow) nnsp_b200_group();
    if (!g) return NNSP_B200_ERR_NOMEM;
    int rc = create(g, n_streams, devices, n_devices);
    for (Member *m : g->members)
        if (!rc) rc = nnsp_b200_batch_create(model, m->count, m->device, thresh_prob, th_count_trigger, &m->batch);
    if (rc) { nnsp_b200_group_destroy(g); return rc; }
    for (Member *m : g->members) m->thread = std::thread(worker, m);
    *out = g;
    return NNSP_B200_OK;
}

int nnsp_b200_group_create_cascade(const nnsp_b200_model *const models[3], const int *seq, int len_seq,
                                   const nnsp_b200_cascade_params *params, int n_streams, const int *devices, int n_devices,
                                   nnsp_b200_group **out)
{
    if (!models || !seq || !devices || !out || n_devices < 1 || n_streams < 1) return NNSP_B200_ERR_ARG;
    nnsp_b200_group *g = new (std::nothrow) nnsp_b200_group();
    if (!g) return NNSP_B200_ERR_NOMEM;
    g->is_cascade = true;
    int rc = create(g, n_streams, devices, n_devices);
    for (Member *m : g->members)
        if (!rc) rc = nnsp_b200_cascade_create(models, seq, len_seq, params, m->count, m->device, &m->cascade);
    if (rc) { nnsp_b200_group_destroy(g); return rc; }
    for (Member *m : g->members) m->thread = std::thread(worker, m);
    *out = g;
    return NNSP_B200_OK;
}

int nnsp_b200_group_size(const nnsp_b200_group *g) { return g ? (int)g->members.size() : NNSP_B200_ERR_ARG; }

int nnsp_b200_group_range(const nnsp_b200_group *g, int member, int *device, int *first_stream, int *n_streams)
{
    if (!g || member < 0 || member >= (int)g->members.size()) return NNSP_B200_ERR_ARG;
    const Member *m = g->members[member];
    if (device) *device = m->device;
    if (first_stream) *first_stream = m->first;
    if (n_streams) *n_streams = m->count;
    return NNSP_B200_OK;
}

int nnsp_b200_group_exec_host_async(nnsp_b200_group *g, const int16_t *pcm, long long stream_stride, int n_frames,
                                    void *results, long long *ticket)
{
    if (!g || !pcm || n_frames <= 0) return NNSP_B200_ERR_ARG;
    Command c{ Command::EXEC, pcm, stream_stride, n_frames, results, 0, {}, {}, {} };
    return post(g, c, ticket);
}

int nnsp_b200_group_wait(nnsp_b200_group *g, long long ticket)
{
    if (!g || ticket <= 0 || ticket > g->seq) return NNSP_B200_ERR_ARG;
    int rc = NNSP_B200_OK;
    for (Member *m : g->members) {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv_done.wait(lk, [&] { return m->done_seq >= ticket; });
        if (m->status != NNSP_B200_OK && rc == NNSP_B200_OK) { rc = m->status; nnsp_set_error("%s", m->error); }
    }
    return rc;
}

int nnsp_b200_group_exec_host(nnsp_b200_group *g, const int16_t *pcm, long long stream_stride, int n_frames, void *results)
{
    long long t = 0;
    const int rc = nnsp_b200_group_exec_host_async(g, pcm, stream_stride, n_frames, results, &t);
    return rc ? rc : nnsp_b200_group_wait(g, t);
}

int nnsp_b200_group_reset(nnsp_b200_group *g)
{
    if (!g) return NNSP_B200_ERR_ARG;
    long long t = 0;
    Command c{ Command::RESET, nullptr, 0, 0, nullptr, 0, {}, {}, {} };
    post(g, c, &t);
    return nnsp_b200_group_wait(g, t);
}

/* nnsp_b200_cascade_set_stream_params over the group's global stream numbering: every command issued so far completes
 * first, then each member takes the part of the range it owns (the workers are idle, the handles are the caller's). */
int nnsp_b200_group_set_stream_params(nnsp_b200_group *g, int first_stream, int n_streams, const nnsp_b200_cascade_params *params)
{
    if (!g || !g->is_cascade || !params || first_stream < 0 || n_streams < 0 || (long long)first_stream + n_streams > g->n_streams) {
        nnsp_set_error("group_set_stream_params: a cascade group and a stream range inside it are required");
        return NNSP_B200_ERR_ARG;
    }
    if (g->seq > 0) { const int rc = nnsp_b200_group_wait(g, g->seq); if (rc) return rc; }
    for (Member *m : g->members) {
        const int lo = first_stream > m->first ? first_stream : m->first;
        const int hi = (first_stream + n_streams) < (m->first + m->count) ? (first_stream + n_streams) : (m->first + m->count);
        if (hi <= lo) continue;
        const int rc = nnsp_b200_cascade_set_stream_params(m->cascade, lo - m->first, hi - lo, params + (lo - first_stream));
        if (rc) return rc;
    }
    return NNSP_B200_OK;
}

int nnsp_b200_group_reset_streams(nnsp_b200_group *g, const int32_t *streams, int n, int mode)
{
    if (!g || !g->is_cascade || n < 0 || (n > 0 && !streams) || (mode != NNSP_B200_RESET_INSTANCE && mode != NNSP_B200_RESET_FRESH)) {
        nnsp_set_error("group_reset_streams: a cascade group, n >= 0 and a known mode are required");
        return NNSP_B200_ERR_ARG;
    }
    for (int i = 0; i < n; i++)
        if (streams[i] < 0 || streams[i] >= g->n_streams) {
            nnsp_set_error("group_reset_streams: streams[%d] = %d is outside [0, %d)", i, (int)streams[i], g->n_streams);
            return NNSP_B200_ERR_ARG;
        }
    /* every member gets the command (its own streams, maybe none) and the sequence number, so that waiting for the
     * group's latest command (nnsp_b200_group_set_stream_params, group_wait) also waits until it is recorded */
    const long long seq = ++g->seq;
    for (Member *m : g->members) {
        Command c{ Command::RESET_STREAMS, nullptr, 0, mode, nullptr, seq, {}, {}, {} };
        for (int i = 0; i < n; i++)
            if (streams[i] >= m->first && streams[i] < m->first + m->count) c.streams.push_back(streams[i] - m->first);
        { std::lock_guard<std::mutex> lk(m->mu); m->queue.push_back(std::move(c)); }
        m->cv_cmd.notify_one();
    }
    return NNSP_B200_OK;
}

size_t nnsp_b200_group_stream_state_bytes(const nnsp_b200_group *g)
{
    return (g && g->is_cascade) ? nnsp_b200_cascade_stream_state_bytes(g->members[0]->cascade) : 0;
}

/* the checks of nnsp_b200_cascade_export_streams / _import_streams over the group's numbering (cascade groups) */
static int group_check_ids(const nnsp_b200_group *g, const int32_t *streams, int n, bool unique, const char *fn)
{
    if (!g || !g->is_cascade || n < 0 || (n > 0 && !streams)) {
        nnsp_set_error("%s: a cascade group and n >= 0 are required", fn);
        return NNSP_B200_ERR_ARG;
    }
    std::vector<char> seen(unique ? (size_t)g->n_streams : 0);
    for (int i = 0; i < n; i++) {
        if (streams[i] < 0 || streams[i] >= g->n_streams) {
            nnsp_set_error("%s: streams[%d] = %d is outside [0, %d)", fn, i, (int)streams[i], g->n_streams);
            return NNSP_B200_ERR_ARG;
        }
        if (unique && seen[(size_t)streams[i]]++) { nnsp_set_error("%s: stream %d listed twice", fn, (int)streams[i]); return NNSP_B200_ERR_ARG; }
    }
    return NNSP_B200_OK;
}

int nnsp_b200_group_export_streams(nnsp_b200_group *g, const int32_t *streams, int n, void *records)
{
    int rc = group_check_ids(g, streams, n, false, "group_export_streams");
    if (rc) return rc;
    if (n > 0 && !records) { nnsp_set_error("group_export_streams: null records"); return NNSP_B200_ERR_ARG; }
    const long long seq = ++g->seq;
    for (Member *m : g->members) {
        Command c{ Command::EXPORT_STREAMS, nullptr, 0, 0, records, seq, {}, {}, {} };
        for (int i = 0; i < n; i++)
            if (streams[i] >= m->first && streams[i] < m->first + m->count) { c.streams.push_back(streams[i] - m->first); c.where.push_back(i); }
        { std::lock_guard<std::mutex> lk(m->mu); m->queue.push_back(std::move(c)); }
        m->cv_cmd.notify_one();
    }
    return nnsp_b200_group_wait(g, seq);
}

int nnsp_b200_group_import_streams(nnsp_b200_group *g, const int32_t *streams, int n, const void *records)
{
    int rc = group_check_ids(g, streams, n, true, "group_import_streams");
    if (rc) return rc;
    if ((rc = nnsp_cascade_check_records(g->members[0]->cascade, records, n))) return rc;   /* every member takes the same records */
    const size_t rb = nnsp_b200_cascade_stream_state_bytes(g->members[0]->cascade);
    const unsigned char *in = static_cast<const unsigned char *>(records);
    const long long seq = ++g->seq;                                   /* in order with the calls, like RESET_STREAMS */
    for (Member *m : g->members) {
        Command c{ Command::IMPORT_STREAMS, nullptr, 0, 0, nullptr, seq, {}, {}, {} };
        for (int i = 0; i < n; i++)
            if (streams[i] >= m->first && streams[i] < m->first + m->count) {
                c.streams.push_back(streams[i] - m->first);
                c.records.insert(c.records.end(), in + rb * (size_t)i, in + rb * (size_t)(i + 1));
            }
        { std::lock_guard<std::mutex> lk(m->mu); m->queue.push_back(std::move(c)); }
        m->cv_cmd.notify_one();
    }
    return NNSP_B200_OK;
}

void nnsp_b200_group_destroy(nnsp_b200_group *g)
{
    if (!g) return;
    for (Member *m : g->members) {
        if (m->thread.joinable()) {
            { std::lock_guard<std::mutex> lk(m->mu); m->queue.push_back(Command{ Command::QUIT, nullptr, 0, 0, nullptr, 0, {}, {}, {} }); }
            m->cv_cmd.notify_one();
            m->thread.join();
        }
        if (m->batch) nnsp_b200_batch_destroy(m->batch);
        if (m->cascade) nnsp_b200_cascade_destroy(m->cascade);
        delete m;
    }
    delete g;
}

}  /* extern "C" */

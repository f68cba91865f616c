/*
 * xm_stream.h -- the chunked walk: two host streams of any length are sent
 * through the GPU in bounded chunks, records aligned by index, the six bins
 * appended in order.  This is what replaces the reference's lockstep reader
 * on real files (getReadPairs, xm.py:95-118, driven by main(), xm.py:702-740).
 *
 * Step k walks two device buffers, each = [carry of step k-1][new bytes]:
 *
 *   - New bytes are cut after their last '\n', so a step only ever sees
 *     complete lines; the cut-off tail is sent again with the next chunk.
 *   - The two streams hold different numbers of records per byte.  A step
 *     yields n = min(records of both buffers); the surplus records of the
 *     longer buffer are carried (device-to-device) to the front of its next
 *     buffer.
 *   - The last yielded record is carried too, as record 0 of the next step
 *     ("halo"): the pair predicate (xm.py:402) and the run-skipping reader
 *     (xm.py:110-114) look at the previous record.  The kernels do not
 *     classify a halo record again.
 *   - The walk ends like the reference's (xm.py:105): at the first blank line
 *     or at the end of either stream.
 *
 * The host-to-device copy of step k+1 never waits for the kernels of step k:
 * new bytes go to a staging buffer on the device as soon as the host has them
 * (their place in the walk buffer depends on the carry, which is only known
 * when step k is done; moving them there is a device-to-device copy of a
 * fraction of a millisecond).  Descriptor sources are read ahead by a thread
 * of their own into a ring of pinned buffers (FdFeeder), so pread, H2D, the
 * kernels, D2H and the writes of the bins all overlap.
 *
 * Written against the same Backend interface as xm_walk.h plus
 *     int upload(void *dev_dst, const void *host_src, size_t n)   asynchronous H2D
 *     int upload_wait()
 *     int copy_dd(void *dev_dst, const void *dev_src, size_t n)
 * so that the CPU emulation harness of the tests runs the same logic.
 */
#pragma once
#include <errno.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "xm_walk.h"

namespace xm {

/* bytes of [p, p + n) up to and including the last '\n', 0 if there is none */
inline uint64_t cut_after_last_newline(const uint8_t *p, uint64_t n)
{
    while (n > 0 && p[n - 1] != '\n') --n;
    return n;
}

/* read n bytes of a descriptor source at absolute offset `at` into dst; returns bytes read or -1 */
int64_t xm_pread_all(int fd, void *dst, uint64_t n, int64_t at);      /* xm_api.cu / the emulation harness */

/* the same with `threads` preads side by side (page-cache and tmpfs reads are memcpy-bound per thread) */
inline int64_t xm_pread_parallel(int fd, void *dst, uint64_t n, int64_t at, int threads)
{
    const uint64_t min_part = 8ull << 20;
    if (threads <= 1 || n < 2 * min_part) return xm_pread_all(fd, dst, n, at);
    const uint64_t parts = std::min<uint64_t>((uint64_t)threads, n / min_part);
    const uint64_t per = ((n + parts - 1) / parts + 4095) & ~4095ull;
    std::vector<int64_t> got(parts, 0);
    std::vector<std::thread> th;
    for (uint64_t k = 0; k < parts; ++k) {
        const uint64_t lo = k * per, m = lo < n ? std::min<uint64_t>(per, n - lo) : 0;
        th.emplace_back([=, &got] { got[k] = m ? xm_pread_all(fd, (uint8_t *)dst + lo, m, at + (int64_t)lo) : 0; });
    }
    for (auto &t : th) t.join();
    int64_t total = 0;
    for (uint64_t k = 0; k < parts; ++k) {
        if (got[k] < 0) return -1;
        total += got[k];
        const uint64_t lo = k * per, m = lo < n ? std::min<uint64_t>(per, n - lo) : 0;
        if ((uint64_t)got[k] < m) break;           /* the file ends inside this part: what the later parts read is not contiguous */
    }
    return total;
}

/*
 * Reads a descriptor ahead of the walk.  A thread of its own fills a ring of pinned slots; every slot holds whole
 * lines only (the tail behind a slot's last newline opens the next slot), the last one whatever is left.
 */
struct FdFeeder {
    struct Slot { uint8_t *p = nullptr; uint64_t n = 0, used = 0; bool last = false; int state = 0; /* 0 free, 1 filled, 2 drained (an H2D copy may still read it) */ };
    int fd = -1;
    int64_t off = 0;
    uint64_t len = 0, slot_cap = 0;
    int threads = 1;                    /* preads side by side per slot */
    bool seekable = true;               /* false: a pipe or socket, read() in order, length unknown until it ends */
    std::vector<uint8_t> pre;           /* bytes already taken from a pipe (behind its header): the stream starts with them */
    std::vector<Slot> ring;
    size_t head = 0;                    /* slot the walk takes from */
    bool ended = false;                 /* the walk has taken the stream's last byte */
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    bool stop = false, failed = false, too_long = false;

    void start() { th = std::thread([this] { run(); }); }
    void run()
    {
        uint64_t pos = 0;               /* bytes of the source read so far */
        std::vector<uint8_t> tail;
        tail.swap(pre);                 /* a pipe's first bytes were read with its header */
        size_t k = 0;
        for (;;) {
            Slot *s;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || ring[k].state == 0; });
                if (stop) return;
                s = &ring[k];
            }
            /* what is left over from before (the tail behind the last slot's final newline; a pipe's first bytes) comes
             * first, as much of it as fits */
            uint64_t have = std::min<uint64_t>(tail.size(), slot_cap);
            if (have) memcpy(s->p, tail.data(), have);
            tail.erase(tail.begin(), tail.begin() + (long)have);
            const uint64_t want = tail.empty() ? std::min<uint64_t>(slot_cap - have, len - pos) : 0;
            int64_t got = 0;
            if (want && seekable) got = xm_pread_parallel(fd, s->p + have, want, off + (int64_t)pos, threads);
            else if (want) {
                /* a pipe: whatever arrives, until the slot is full or the writer closes its end */
                while ((uint64_t)got < want) {
                    const ssize_t r = read(fd, s->p + have + (uint64_t)got, (size_t)std::min<uint64_t>(want - (uint64_t)got, 1u << 30));
                    if (r < 0) { if (errno == EINTR) continue; got = -1; break; }
                    if (r == 0) break;
                    got += r;
                }
            }
            if (got < 0) { std::lock_guard<std::mutex> lk(mu); failed = true; s->n = 0; s->last = true; s->state = 1; cv.notify_all(); return; }
            if ((uint64_t)got < want) len = pos + (uint64_t)got;                 /* the source ends here (a pipe's length is only known now) */
            pos += (uint64_t)got;
            have += (uint64_t)got;
            const bool eof = pos >= len && tail.empty();
            uint64_t n = have;
            if (!eof) {
                n = cut_after_last_newline(s->p, have);
                if (n == 0) { std::lock_guard<std::mutex> lk(mu); too_long = true; s->n = 0; s->last = true; s->state = 1; cv.notify_all(); return; }
                tail.insert(tail.begin(), s->p + n, s->p + have);
            }
            {
                std::lock_guard<std::mutex> lk(mu);
                s->n = n; s->used = 0; s->last = eof; s->state = 1;
            }
            cv.notify_all();
            if (eof) return;
            k = (k + 1) % ring.size();
        }
    }
    /* the bytes the walk may take next: pointer, count, and whether they are the stream's last */
    bool peek(const uint8_t *&p, uint64_t &avail, bool &last)
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return ring[head].state == 1; });
        Slot &s = ring[head];
        p = s.p + s.used; avail = s.n - s.used; last = s.last;
        return !failed && !too_long;
    }
    void consume(uint64_t n)
    {
        std::lock_guard<std::mutex> lk(mu);
        Slot &s = ring[head];
        s.used += n;
        if (s.used == s.n) {
            if (s.last) ended = true;
            else { s.state = 2; head = (head + 1) % ring.size(); }
        }
    }
    /* every upload issued so far has completed: drained slots go back to the reader */
    void release_drained()
    {
        { std::lock_guard<std::mutex> lk(mu); for (auto &s : ring) if (s.state == 2) s.state = 0; }
        cv.notify_all();
    }
    void shutdown()
    {
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv.notify_all();
        if (th.joinable()) th.join();
    }
};

/* a source that puts whole lines straight into a device buffer (BAM input: records rendered as SAM text on the GPU) */
struct DevSource {
    virtual ~DevSource() {}
    /* up to max_bytes of SAM text into dev_dst; n = bytes written, final = the stream ends with them.  Returns an xm_status. */
    virtual int next(uint8_t *dev_dst, uint64_t max_bytes, uint64_t &n, bool &final, std::string &err) = 0;
    bool ended = false;
};

/* one input stream on the host */
struct HostIn {
    const uint8_t *mem = nullptr;      /* memory source (pageable or pinned) ... */
    uint64_t len = 0;
    FdFeeder *feed = nullptr;          /* ... or a descriptor read ahead by its own thread ... */
    DevSource *prod = nullptr;         /* ... or a producer of device-resident text */
    uint64_t pos = 0;                  /* next byte to send */
    bool exhausted() const { return prod ? prod->ended : (feed ? feed->ended : pos >= len); }
};

/* device side of one input stream: two walk buffers and two staging buffers used alternately */
struct DevIn {
    uint8_t *buf[2] = {nullptr, nullptr};
    uint8_t *stage[2] = {nullptr, nullptr};
    uint64_t cap = 0;                  /* of each of the four */
    uint64_t len = 0;                  /* bytes of the current walk buffer */
};

struct StreamPlan {
    uint64_t chunk = 256ull << 20;     /* new bytes per stream and step */
};

/*
 * The chunked walk.  `outs[set][b]` are two sets of six device output buffers of `out_cap[b]` bytes each;
 * `emit(set, bin, dev_ptr, nbytes)` is called for every bin with new bytes after a step, then once with bin -1, and
 * must have consumed (or queued a copy of) them before the same set is written again two steps later --
 * `emit_wait(set)` is called for that.  Returns an xm_status; *res holds the totals of the whole walk.
 */
template <class BE, class Emit, class EmitWait>
inline int walk_stream(BE &be, Scratch &sc, HostIn in[2], DevIn dev[2], uint8_t *const outs[2][6], const uint64_t out_cap[6],
                       const xm_opts &o, uint32_t debug, const StreamPlan &plan, Emit emit, EmitWait emit_wait,
                       xm_result *res, std::string &errmsg, int first_is_context = 0)
{
    memset(res, 0, sizeof *res);
    res->err_stream = -1;
    uint64_t carry_off[2] = {0, 0}, carry_len[2] = {0, 0};      /* in the previous walk buffer */
    uint64_t staged[2][2] = {{0, 0}, {0, 0}};                   /* [slot][stream]: bytes waiting in the staging buffer */
    bool staged_final[2][2] = {{false, false}, {false, false}};
    bool final_sent[2] = {false, false};
    int halo = first_is_context ? 1 : 0;                      /* sharded walks: the caller's buffers open with the record before its range */
    int io_rc = XM_OK;

    /* send the next bytes of both streams towards staging buffer `slot`; room[s]: what the next walk buffer can take
     * behind its carry (the carry is not known yet: the whole of the buffer being walked is allowed for) */
    auto stage_next = [&](int slot, const uint64_t room[2]) {
        for (int s = 0; s < 2; ++s) {
            staged[slot][s] = 0; staged_final[slot][s] = false;
            if (in[s].exhausted()) continue;
            if (in[s].prod) {
                uint64_t n = 0;
                bool fin = false;
                const int prc = in[s].prod->next(dev[s].stage[slot], std::min<uint64_t>(room[s], plan.chunk), n, fin, errmsg);
                if (prc) { io_rc = prc; return; }
                staged[slot][s] = n; staged_final[slot][s] = fin;
                in[s].prod->ended = fin;
                in[s].pos += n;
                continue;
            }
            const uint8_t *src = nullptr;
            uint64_t avail = 0;
            bool last_piece = false;
            if (in[s].feed) {
                if (!in[s].feed->peek(src, avail, last_piece)) {
                    io_rc = in[s].feed->too_long ? XM_ERR_UNSUPPORTED : XM_ERR_IO;
                    errmsg = in[s].feed->too_long ? "a line is longer than the staging buffer (" + std::to_string(in[s].feed->slot_cap) + " bytes)" : "read failed";
                    return;
                }
            } else {
                avail = in[s].len - in[s].pos;
                src = in[s].mem + in[s].pos;
                last_piece = true;
            }
            uint64_t take = std::min<uint64_t>(std::min<uint64_t>(room[s], plan.chunk), avail);
            if (!(last_piece && take == avail)) {
                uint64_t cut = cut_after_last_newline(src, take);
                if (cut == 0 && !in[s].feed) {
                    /* a line longer than the chunk: take it whole if the buffer has room for it */
                    const uint64_t lim = std::min<uint64_t>(room[s], avail);
                    const void *nl = lim > take ? memchr(src + take, '\n', lim - take) : nullptr;
                    if (nl) cut = (uint64_t)((const uint8_t *)nl - src) + 1;
                }
                take = cut;             /* 0: no complete line fits behind the carry this time; the other stream moves on */
            }
            if (take && be.upload(dev[s].stage[slot], src, take)) { io_rc = XM_ERR_CUDA; errmsg = "H2D copy failed: " + be.last_error(); return; }
            staged[slot][s] = take;
            staged_final[slot][s] = last_piece && take == avail;
            if (in[s].feed) in[s].feed->consume(take);
            in[s].pos += take;
        }
    };

    {
        const uint64_t room0[2] = {dev[0].cap, dev[1].cap};
        stage_next(0, room0);
        if (io_rc) { be.upload_wait(); return res->status = io_rc; }
    }
    for (uint64_t step = 0;; ++step) {
        const int cur = (int)(step & 1), prev = cur ^ 1;
        if (be.upload_wait()) { errmsg = "H2D copy failed: " + be.last_error(); return res->status = XM_ERR_CUDA; }
        for (int s = 0; s < 2; ++s) if (in[s].feed) in[s].feed->release_drained();
        /* this step's buffers: carry to the front, the staged bytes behind it */
        uint64_t fresh_bytes = 0;
        for (int s = 0; s < 2; ++s) {
            if (carry_len[s] && be.copy_dd(dev[s].buf[cur], dev[s].buf[prev] + carry_off[s], carry_len[s])) { errmsg = "carry copy failed: " + be.last_error(); return res->status = XM_ERR_CUDA; }
            const uint64_t take = staged[cur][s];
            if (take && be.copy_dd(dev[s].buf[cur] + carry_len[s], dev[s].stage[cur], take)) { errmsg = "staging copy failed: " + be.last_error(); return res->status = XM_ERR_CUDA; }
            dev[s].len = carry_len[s] + take;
            fresh_bytes += take;
            final_sent[s] = final_sent[s] || staged_final[cur][s] || (in[s].len == 0);
        }
        /* the next step's bytes leave the host now, while this step's kernels run */
        uint64_t next_bytes = 0;
        staged[prev][0] = staged[prev][1] = 0; staged_final[prev][0] = staged_final[prev][1] = false;
        if (!in[0].exhausted() || !in[1].exhausted()) {
            const uint64_t room[2] = {dev[0].cap - dev[0].len, dev[1].cap - dev[1].len};
            stage_next(prev, room);
            if (io_rc) { be.upload_wait(); return res->status = io_rc; }
            next_bytes = staged[prev][0] + staged[prev][1];
        }
        if (step >= 2) emit_wait(cur);

        /* walk the two buffers */
        xm_result r;
        WalkCtl ctl;
        ctl.halo = halo;
        ctl.want_tail = true;
        std::string msg;
        const int rc = walk_resident(be, sc, StreamBuf{dev[0].buf[cur], dev[0].len}, StreamBuf{dev[1].buf[cur], dev[1].len}, o,
                                     outs[cur], out_cap, debug, &r, msg, &ctl);
        res->n_launches += r.n_launches;
        res->ms_scan += r.ms_scan; res->ms_classify += r.ms_classify; res->ms_total += r.ms_total;
        if (rc == XM_ERR_CUDA || rc == XM_ERR_NOMEM || rc == XM_ERR_ARG) { be.upload_wait(); errmsg = msg; return res->status = rc; }
        const uint64_t n = r.n_records;                              /* includes the halo record */
        const uint64_t fresh = n - (uint64_t)(n ? halo : 0);
        for (int k = 0; k < 36; ++k) res->counts[k] += r.counts[k];
        for (int b = 0; b < 6; ++b) {
            if (r.out_len[b]) emit(cur, b, outs[cur][b], r.out_len[b]);
            res->out_len[b] += r.out_len[b];
        }
        emit(cur, -1, nullptr, 0);                                   /* the step's bins are all handed over */
        if (rc != XM_OK) {
            /* a failing record: everything before it has been produced (the reference's streaming writes) */
            errmsg = msg;
            res->err_stream = r.err_stream;
            res->err_record = res->n_records + (r.err_record - (uint64_t)halo);
            res->n_records += r.err_record - (uint64_t)halo;
            be.upload_wait();
            return res->status = rc;
        }
        res->n_records += fresh;
        /* the end of the walk (xm.py:105): the lockstep reader reaches a blank line, or the end of a stream */
        bool done = false;
        for (int s = 0; s < 2; ++s) {
            const bool drained = ctl.n_stream[s] == n;                   /* every record of this buffer was yielded */
            if (drained && ctl.stopped[s]) done = true;
            if (drained && final_sent[s]) done = true;
        }
        for (int s = 0; s < 2; ++s) {
            const uint64_t last = s ? ctl.last_s : ctl.last_p;
            if (n > 0) res->bytes_in[s] += done ? (ctl.n_stream[s] == n ? ctl.end_off[s] : last) : last;
        }
        if (done) { be.upload_wait(); break; }
        if (fresh == 0 && (dev[0].len == dev[0].cap || dev[1].len == dev[1].cap)) {
            be.upload_wait();
            errmsg = "no complete record fits the staging buffers";
            return res->status = XM_ERR_UNSUPPORTED;
        }
        if (fresh == 0 && fresh_bytes == 0 && next_bytes == 0) {
            /* nothing was yielded, nothing new was staged and nothing new is on its way: the next step would be this
             * one again.  A line that does not fit a staging step ends here. */
            be.upload_wait();
            errmsg = "a line is longer than the staging buffer (" + std::to_string(plan.chunk) + " bytes per step)";
            return res->status = XM_ERR_UNSUPPORTED;
        }
        /* carry: from the last yielded record (the next step's halo) to the end of each buffer */
        if (n > 0) {
            carry_off[0] = ctl.last_p; carry_off[1] = ctl.last_s;
            halo = 1;
        } else {
            carry_off[0] = carry_off[1] = 0;            /* nothing was yielded: the buffers (halo included) are carried whole */
        }
        for (int s = 0; s < 2; ++s) carry_len[s] = dev[s].len - carry_off[s];
    }
    return res->status = XM_OK;
}

}  // namespace xm

// capture_frontend.cpp -- the SDRplay-format front end of the batched engine (SURVEY.md 8f.1) and an in-memory
// message store behind add_message (8f.2).  Host code only; no CUDA in this file.
//
// nvx_capture replaces, for S radios at once, the reference's capture plumbing:
//   producer  StreamACallback  receiver/capt_sched.c:105-148  (xi[], xq[] int16 arrays, numSamples per callback,
//                                                              interleaved into one ring of shorts under a mutex)
//   consumer  main loop        receiver/capt_sched.c:484-528  (every 50 ms: drain the ring, sample_in_1 per I,Q pair)
// Here every stream has its own ring of interleaved int16 I,Q; the consumer ("pump") takes what ALL streams have in
// common, rounded down to a multiple of 280 samples, lays it out stream-major and pushes it as one int16 block.
// nvx_capture_create_u8 makes the same front end for RTL-SDR radios: rings of interleaved 8-bit I,Q bytes (the buffer
// rtlsdr_read_async hands its callback), pumped with nvx_engine_push_host_u8.
//
// nvx_store mirrors message_store.c:59-97: add = "delete from messages where bbbb = ?; insert (bbbb, message,
// timestamp, 'NEW', freq)" with the reference's UTC "%Y-%m-%d %H:%M" stamp, keyed additionally by stream; purge drops
// messages older than MESSAGE_PURGE_AGE (72 h, message_store.c:13).
#include <stdio.h>
#include <string.h>
#include <time.h>

#include <atomic>
#include <chrono>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/navtex_b200.h"

struct nvx_capture {
    nvx_engine* eng = nullptr;
    int S = 0;
    long long ring = 0;                    // samples per stream
    long long max_block = 0;
    bool u8 = false;                       // 8-bit I,Q pairs (nvx_capture_create_u8), else int16
    size_t bps = 4;                        // bytes per I,Q pair in the rings and the staging buffers
    struct Ring {
        std::vector<uint8_t> buf;          // ring * bps bytes of interleaved I,Q
        long long head = 0, tail = 0;      // absolute sample counts written / consumed
        std::mutex mu;                     // in_mutex of capt_sched.c:109-112
        long long dropped = 0;
    };
    std::vector<Ring> rings;
    // [S][n] staging, stream-major: two page-locked buffers (nvx_pinned_alloc), so that the engine's H2D copy of pump k is
    // asynchronous and overlaps the ring drain of pump k + 1
    uint8_t* block[2] = {nullptr, nullptr};
    long long block_push[2] = {-1, -1};    // index of the engine host push that last read each buffer
    unsigned pumps = 0;
    std::thread poller;
    std::atomic<bool> stop{false};
    std::mutex pump_mu;
    int pump_rc = 0;
};

namespace {
long long pump_locked(nvx_capture* c) {
    long long n = c->max_block;
    for (auto& r : c->rings) {
        std::lock_guard<std::mutex> lk(r.mu);
        const long long avail = r.head - r.tail;
        if (avail < n) n = avail;
    }
    n -= n % NVX_BLOCK_ALIGN;
    if (n <= 0) return 0;
    const unsigned which = c->pumps++ & 1;
    uint8_t* const blk = c->block[which];
    // the copy that last read this buffer was queued two pumps ago; make sure it is over before the buffer is refilled (the copy
    // of the previous pump, out of the other buffer, keeps running meanwhile)
    if (c->block_push[which] >= 0)
        if (const int rc = nvx_engine_wait_ingest_of(c->eng, c->block_push[which])) return rc;
    for (int s = 0; s < c->S; ++s) {
        auto& r = c->rings[(size_t)s];
        uint8_t* dst = blk + (size_t)s * c->bps * (size_t)n;
        // the producer only ever writes beyond head, so [tail, tail + n) is stable without the lock
        long long at = r.tail % c->ring;
        long long first = n < c->ring - at ? n : c->ring - at;
        memcpy(dst, r.buf.data() + c->bps * at, c->bps * (size_t)first);
        if (first < n) memcpy(dst + c->bps * first, r.buf.data(), c->bps * (size_t)(n - first));
        std::lock_guard<std::mutex> lk(r.mu);
        r.tail += n;
    }
    c->block_push[which] = nvx_engine_host_pushes(c->eng);
    const int rc = c->u8 ? nvx_engine_push_host_u8(c->eng, blk, n) : nvx_engine_push_host_s16(c->eng, reinterpret_cast<const int16_t*>(blk), n);
    if (rc != 0) { c->block_push[which] = -1; return rc; }
    return n;
}
int create(nvx_engine* e, int n_streams, long long max_block, long long ring_samples, bool u8, nvx_capture** out) {
    if (!e || !out || n_streams <= 0 || max_block <= 0 || max_block % NVX_BLOCK_ALIGN != 0 || ring_samples < 2 * max_block) return NVX_ERR_ARG;
    nvx_capture* c = new nvx_capture();
    c->eng = e;
    c->S = n_streams;
    c->ring = ring_samples;
    c->max_block = max_block;
    c->u8 = u8;
    c->bps = u8 ? 2 : 4;
    c->rings = std::vector<nvx_capture::Ring>((size_t)n_streams);
    for (auto& r : c->rings) r.buf.assign(c->bps * (size_t)ring_samples, 0);
    for (int k = 0; k < 2; ++k) {
        void* p = nullptr;
        if (const int rc = nvx_pinned_alloc((size_t)n_streams * c->bps * (size_t)max_block, 0, &p)) {
            nvx_pinned_free(c->block[0]);
            delete c;
            return rc;
        }
        c->block[k] = static_cast<uint8_t*>(p);
    }
    *out = c;
    return 0;
}

// reserve room for num_samples in the ring of `stream`; put(at, i, k) stores samples i .. i + k - 1 at ring position `at`
// (k contiguous ring slots).  Unlike the reference ring (which silently overwrites unread samples when the consumer lags,
// capt_sched.c:120-128) an overrun is reported: the samples that do not fit are dropped and counted.
template <typename Put>
int write_ring(nvx_capture* c, int stream, unsigned num_samples, Put put) {
    auto& r = c->rings[(size_t)stream];
    long long head, tail;
    {
        std::lock_guard<std::mutex> lk(r.mu);
        head = r.head;
        tail = r.tail;
    }
    long long room = c->ring - (head - tail);
    unsigned take = num_samples;
    int rc = 0;
    if ((long long)take > room) { take = (unsigned)(room > 0 ? room : 0); rc = NVX_ERR_OVERFLOW; }
    const long long at = head % c->ring;
    const unsigned first = (long long)take < c->ring - at ? take : (unsigned)(c->ring - at);
    put(r.buf.data() + c->bps * (size_t)at, 0u, first);
    if (first < take) put(r.buf.data(), first, take - first);
    std::lock_guard<std::mutex> lk(r.mu);
    r.head = head + take;
    r.dropped += num_samples - take;
    return rc;
}
}  // namespace

extern "C" {

int nvx_capture_create(nvx_engine* e, int n_streams, long long max_block, long long ring_samples, nvx_capture** out) {
    return create(e, n_streams, max_block, ring_samples, false, out);
}

int nvx_capture_create_u8(nvx_engine* e, int n_streams, long long max_block, long long ring_samples, nvx_capture** out) {
    return create(e, n_streams, max_block, ring_samples, true, out);
}

int nvx_capture_write(nvx_capture* c, int stream, const short* xi, const short* xq, unsigned num_samples) {
    if (!c || c->u8 || stream < 0 || stream >= c->S || (!xi && num_samples) || (!xq && num_samples)) return NVX_ERR_ARG;
    return write_ring(c, stream, num_samples, [&](uint8_t* dst, unsigned i0, unsigned k) {
        int16_t* d = reinterpret_cast<int16_t*>(dst);
        for (unsigned i = 0; i < k; ++i) {
            d[2 * i] = xi[i0 + i];
            d[2 * i + 1] = xq[i0 + i];
        }
    });
}

int nvx_capture_write_u8(nvx_capture* c, int stream, const unsigned char* iq, unsigned num_samples) {
    if (!c || !c->u8 || stream < 0 || stream >= c->S || (!iq && num_samples)) return NVX_ERR_ARG;
    return write_ring(c, stream, num_samples, [&](uint8_t* dst, unsigned i0, unsigned k) { memcpy(dst, iq + 2 * (size_t)i0, 2 * (size_t)k); });
}

long long nvx_capture_pump(nvx_capture* c) {
    if (!c) return NVX_ERR_ARG;
    std::lock_guard<std::mutex> lk(c->pump_mu);
    return pump_locked(c);
}

int nvx_capture_start(nvx_capture* c, int poll_ms) {
    if (!c || c->poller.joinable()) return NVX_ERR_ARG;
    if (poll_ms <= 0) poll_ms = 50;                      // usleep(50000), capt_sched.c:489
    c->stop = false;
    c->poller = std::thread([c, poll_ms] {
        while (!c->stop) {
            std::this_thread::sleep_for(std::chrono::milliseconds(poll_ms));
            std::lock_guard<std::mutex> lk(c->pump_mu);
            long long n;
            while ((n = pump_locked(c)) > 0) {}
            if (n < 0 && !c->pump_rc) c->pump_rc = (int)n;
        }
    });
    return 0;
}

int nvx_capture_stop(nvx_capture* c) {
    if (!c) return NVX_ERR_ARG;
    if (c->poller.joinable()) {
        c->stop = true;
        c->poller.join();
    }
    std::lock_guard<std::mutex> lk(c->pump_mu);
    long long n;
    while ((n = pump_locked(c)) > 0) {}
    nvx_engine_wait_ingest(c->eng);
    const int rc = c->pump_rc ? c->pump_rc : (n < 0 ? (int)n : 0);
    c->pump_rc = 0;
    return rc;
}

long long nvx_capture_dropped(nvx_capture* c, int stream) {
    if (!c || stream < 0 || stream >= c->S) return NVX_ERR_ARG;
    std::lock_guard<std::mutex> lk(c->rings[(size_t)stream].mu);
    return c->rings[(size_t)stream].dropped;
}

void nvx_capture_destroy(nvx_capture* c) {
    if (!c) return;
    if (c->poller.joinable()) {
        c->stop = true;
        c->poller.join();
    }
    nvx_pinned_free(c->block[0]);      // cudaFreeHost waits for a copy still reading the buffer
    nvx_pinned_free(c->block[1]);
    delete c;
}

}  // extern "C"

// ---------------------------------------------------------------- message store
struct nvx_store {
    struct Row {
        int stream, freq;
        std::string bbbb, text, stamp;
        time_t when;
        long long id;
    };
    std::vector<Row> rows;
    std::mutex mu;
    long long next_id = 1;
};

extern "C" {

nvx_store* nvx_store_create(void) { return new nvx_store(); }
void nvx_store_destroy(nvx_store* s) { delete s; }

int nvx_store_add_at(nvx_store* s, int stream, const char* bbbb, const char* message, int freq, long long unix_time) {
    if (!s || !bbbb || !message) return -1;                // message_store.c:69-73: -1 = store unavailable
    char stamp[20];
    const time_t t = (time_t)unix_time;
    struct tm tmv;
    gmtime_r(&t, &tmv);
    strftime(stamp, sizeof stamp, "%Y-%m-%d %H:%M", &tmv); // message_store.c:30
    std::lock_guard<std::mutex> lk(s->mu);
    for (size_t k = 0; k < s->rows.size();) {              // "delete from messages where bbbb = ?1" (message_store.c:75)
        if (s->rows[k].stream == stream && s->rows[k].bbbb == bbbb) s->rows.erase(s->rows.begin() + (long)k);
        else ++k;
    }
    s->rows.push_back({stream, freq, bbbb, message, stamp, t, s->next_id++});
    return 0;
}

int nvx_store_add(nvx_store* s, int stream, const char* bbbb, const char* message, int freq) {
    return nvx_store_add_at(s, stream, bbbb, message, freq, (long long)time(nullptr));
}

// nvx_message_cb-shaped adapter: nvx_engine_set_message_callback(e, nvx_store_sink, store)
int nvx_store_sink(void* store, int stream, char* bbbb, char* message, int freq) {
    return nvx_store_add(static_cast<nvx_store*>(store), stream, bbbb, message, freq);
}

size_t nvx_store_count(nvx_store* s) {
    if (!s) return 0;
    std::lock_guard<std::mutex> lk(s->mu);
    return s->rows.size();
}

int nvx_store_get(nvx_store* s, size_t k, int* stream, int* freq, char bbbb[8], char stamp[20], const char** text) {
    if (!s) return NVX_ERR_ARG;
    std::lock_guard<std::mutex> lk(s->mu);
    if (k >= s->rows.size()) return NVX_ERR_ARG;
    const auto& r = s->rows[k];
    if (stream) *stream = r.stream;
    if (freq) *freq = r.freq;
    if (bbbb) { memset(bbbb, 0, 8); strncpy(bbbb, r.bbbb.c_str(), 7); }
    if (stamp) { memset(stamp, 0, 20); strncpy(stamp, r.stamp.c_str(), 19); }
    if (text) *text = r.text.c_str();                      // valid until the next add / purge / destroy
    return 0;
}

// message_store.c purge_old_messages: drop rows older than max_age_s (72 h in the reference); returns the number dropped
int nvx_store_purge(nvx_store* s, long long now_unix, long long max_age_s) {
    if (!s) return NVX_ERR_ARG;
    std::lock_guard<std::mutex> lk(s->mu);
    int dropped = 0;
    for (size_t k = 0; k < s->rows.size();) {
        if ((long long)s->rows[k].when + max_age_s < now_unix) { s->rows.erase(s->rows.begin() + (long)k); ++dropped; }
        else ++k;
    }
    return dropped;
}

// id,stream,freq,bbbb,timestamp,"text" with embedded quotes doubled and newlines as \n
int nvx_store_dump_csv(nvx_store* s, const char* path) {
    if (!s || !path) return NVX_ERR_ARG;
    FILE* f = fopen(path, "w");
    if (!f) return NVX_ERR_ARG;
    std::lock_guard<std::mutex> lk(s->mu);
    fprintf(f, "id,stream,freq,bbbb,timestamp,message\n");
    for (const auto& r : s->rows) {
        fprintf(f, "%lld,%d,%d,%s,%s,\"", r.id, r.stream, r.freq, r.bbbb.c_str(), r.stamp.c_str());
        for (char ch : r.text) {
            if (ch == '"') fputs("\"\"", f);
            else if (ch == '\n') fputs("\\n", f);
            else fputc(ch, f);
        }
        fputs("\"\n", f);
    }
    fclose(f);
    return 0;
}

}  // extern "C"

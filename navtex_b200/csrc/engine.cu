// engine.cu -- the C ABI of include/navtex_b200.h: per-GPU engine that owns the carried state of
// S independent streams and queues, per pushed block, the FIR path (the fused cascade and its tail carry, or the
// three long-tap stage kernels), the demod / bit-sync / state-machine kernels and the event
// download; host side it runs the message assembler on a worker thread.
//
// Call contract it replaces: capt_sched.c:552-555 (init_dsp), :612 (init_fir2_wrapper) and the
// consumer loop :484-528 that calls sample_in_1 once per IQ pair.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/navtex_b200.h"
#include "demod.cuh"
#include "fir_cascade.cuh"
#include "fir_long.cuh"
#include "message_assembler.h"
#include "resample.cuh"

namespace {

thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define CU_TRY(expr)                                                                              \
    do {                                                                                          \
        cudaError_t e__ = (expr);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return fail(NVX_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

// nvx_config.nco_hz entry f -> its NCO row; false if f is off the 0.5 Hz grid or outside +-31.5 kHz
bool nco_entry(double f, nvx::NcoChan* out) {
    const double twice = 2.0 * f;
    if (!(fabs(f) < 31500.0) || twice != nearbyint(twice)) return false;
    long long num = (long long)twice % nvx::kNcoDen;
    if (num < 0) num += nvx::kNcoDen;
    out->num = (int)num;
    out->phase0 = 0;
    // same expression as fir2cpp.C:105-106 for table entry 1, rounded once to float
    out->step = make_float2((float)cos((2 * M_PI * 1 * f) / 63000), (float)-sin((2 * M_PI * 1 * f) / 63000));
    return true;
}

// One stream's record of saved state (nvx_engine_save_streams), in 32-bit words: the FIR path's carried rows, then per channel
// the y3 and correlation histories, ClockState, FsmState, epoch and, for general-NCO engines, the NcoChan row, then, on engines
// fed at another input rate, the resampler's history.  The offsets inside a channel's part are fixed; the rest follows from the
// path's CarriedRows, the channel count, the NCO kind and the resampler's history words (0 on engines fed at 252 kS/s).
constexpr int kRecY3 = 0, kRecCorr = kRecY3 + 2 * nvx::kHistY, kRecClock = kRecCorr + 2 * nvx::kHistC;
constexpr int kRecFsm = kRecClock + (int)sizeof(nvx::ClockState) / 4, kRecEpoch = kRecFsm + (int)sizeof(nvx::FsmState) / 4;
constexpr int kRecNco = kRecEpoch + 2, kRecNcoWords = (int)sizeof(nvx::NcoChan) / 4;
static_assert(sizeof(nvx::ClockState) % 4 == 0 && sizeof(nvx::FsmState) % 4 == 0 && sizeof(nvx::NcoChan) % 4 == 0, "word records");
struct StateLayout {
    long long rows[3];                  // offset of each carried region
    long long chan;                     // offset of channel 0's part
    long long ch_words;                 // words per channel
    long long pre;                      // offset of the resampler's history
    long long words;                    // the whole record
};
StateLayout state_layout(const long long words[3], int C, bool gen_nco, long long pre_words) {
    StateLayout l;
    long long at = 0;
    for (int k = 0; k < 3; ++k) { l.rows[k] = at; at += words[k]; }
    l.chan = (at + 1) & ~1LL;
    l.ch_words = kRecNco + (gen_nco ? kRecNcoWords : 0);
    l.pre = l.chan + C * l.ch_words;
    l.words = l.pre + pre_words;
    return l;
}

// Everything the next block would carry over from the past of the listed streams.  A reset clears it so that each stream restarts
// as an engine created at its epoch e0 (nvx_engine_reset_streams); a load writes a saved record over it (nvx_engine_load_streams);
// a save copies it out (nvx_engine_save_streams).  Resets and loads are queued on the engine stream in push order, after the
// previous block's sequential demod kernels (they still read its y3 buffer and the decoder state) and before this block's cascade.
struct ResetArgs {
    const int* streams;                 // [gridDim.x] local stream indices
    const int* recs;                    // [gridDim.x] record each stream loads, -1 = reset (null when saving)
    uint32_t* rec;                      // records [][lay.words]: a load's input, a save's output (record k = streams[k])
    StateLayout lay;
    int C;                              // channels per stream
    long long e0;                       // the new epoch, 900 Hz samples (a multiple of 567)
    nvx::CarriedRows rows;              // what the engine's FIR path carries into the next block
    nvx::CarriedRows pre;               // what the resampler carries (region 0; nothing on engines fed at 252 kS/s)
    float2* y3_prev;                    // the previous block's y3 / corr buffers, whose ends become this block's histories
    long long y3_pitch;
    double* corr_prev;
    long long corr_pitch;
    int n_prev;
    nvx::ClockState* clock;
    nvx::FsmState* fsm;
    long long* epoch;
    nvx::NcoChan* nco;                  // general-NCO rows (their phase origin moves to e0), or null: the reference table
};

template <bool kSave>
__device__ void move_words(uint32_t* state, uint32_t* rec, long long n) {
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
        if (kSave) rec[i] = state[i];
        else state[i] = rec[i];
    }
}

// stream s's carried state -> rec (kSave) or back; the addresses are those reset_streams_kernel clears
template <bool kSave>
__device__ void move_stream(const ResetArgs& a, int s, uint32_t* rec) {
    for (int k = 0; k < 3; ++k) move_words<kSave>(a.rows.base[k] + (size_t)s * a.rows.words[k], rec + a.lay.rows[k], a.rows.words[k]);
    move_words<kSave>(a.pre.base[0] + (size_t)s * a.pre.words[0], rec + a.lay.pre, a.pre.words[0]);
    for (int c = 0; c < a.C; ++c) {
        const size_t ch = (size_t)s * a.C + c;
        uint32_t* r = rec + a.lay.chan + c * a.lay.ch_words;
        move_words<kSave>(reinterpret_cast<uint32_t*>(a.y3_prev + ch * a.y3_pitch + a.n_prev), r + kRecY3, 2 * nvx::kHistY);
        move_words<kSave>(reinterpret_cast<uint32_t*>(a.corr_prev + ch * a.corr_pitch + a.n_prev), r + kRecCorr, 2 * nvx::kHistC);
        move_words<kSave>(reinterpret_cast<uint32_t*>(a.clock + ch), r + kRecClock, kRecFsm - kRecClock);
        move_words<kSave>(reinterpret_cast<uint32_t*>(a.fsm + ch), r + kRecFsm, kRecEpoch - kRecFsm);
        move_words<kSave>(reinterpret_cast<uint32_t*>(a.epoch + ch), r + kRecEpoch, 2);
        if (a.nco) move_words<kSave>(reinterpret_cast<uint32_t*>(a.nco + ch), r + kRecNco, kRecNcoWords);
    }
}

// one CTA per listed stream: record k <- stream streams[k]
__global__ void save_streams_kernel(const ResetArgs a) { move_stream<true>(a, a.streams[blockIdx.x], a.rec + (size_t)blockIdx.x * a.lay.words); }

// one CTA per listed stream: its record, or the state of an engine created at e0
__global__ void reset_streams_kernel(const ResetArgs a) {
    const int s = a.streams[blockIdx.x];
    if (a.recs[blockIdx.x] >= 0) {
        move_stream<false>(a, s, a.rec + (size_t)a.recs[blockIdx.x] * a.lay.words);
        return;
    }
    const int t = threadIdx.x, nt = blockDim.x;
    for (int k = 0; k < 3; ++k)
        for (long long i = t; i < a.rows.words[k]; i += nt) a.rows.base[k][(size_t)s * a.rows.words[k] + i] = a.rows.fill[k];
    for (long long i = t; i < a.pre.words[0]; i += nt) a.pre.base[0][(size_t)s * a.pre.words[0] + i] = a.pre.fill[0];
    for (int c = 0; c < a.C; ++c) {
        const size_t ch = (size_t)s * a.C + c;
        for (int i = t; i < nvx::kHistY; i += nt) a.y3_prev[ch * a.y3_pitch + a.n_prev + i] = make_float2(0.f, 0.f);
        for (int i = t; i < nvx::kHistC; i += nt) a.corr_prev[ch * a.corr_pitch + a.n_prev + i] = 0.0;
    }
    if (t < a.C) {
        const size_t ch = (size_t)s * a.C + t;
        a.clock[ch] = nvx::clock_state_init();
        a.fsm[ch] = nvx::fsm_state_init();
        a.epoch[ch] = a.e0;
        if (a.nco) {     // the stage-1 output at e0 is number 70 e0; its phase becomes 0
            const long long k0 = a.e0 * (nvx::kSuper / NVX_D1) % nvx::kNcoDen;
            const int p = (int)(k0 * a.nco[ch].num % nvx::kNcoDen);
            a.nco[ch].phase0 = p ? nvx::kNcoDen - p : 0;
        }
    }
}

}  // namespace

constexpr int kBuf = 3;   // blocks in flight: cascade of block i+1/i+2 overlaps demod + event download of block i

struct nvx_engine {
    nvx_config cfg;
    int S = 0, P_max = 0, channels = 0;
    int C = 2;                            // channels per stream (nvx_config.n_channels)
    cudaStream_t stream = nullptr;        // FIR path, ingest copies / conversion
    cudaStream_t stream_demod = nullptr;  // demod kernels + event download, one block behind
    float2* y3buf[kBuf] = {};
    uint8_t* pickbuf[kBuf] = {};
    cudaEvent_t demod_done[kBuf] = {}, ff_done[kBuf] = {};
    long long blocks = 0;
    int last_buf = 0;
    int fmt = -1;                         // -1 = nothing pushed since create/reset, else the nvx::SampleFmt of the pushes
    nvx::DemodBuffers db = {};
    double* corrbuf[2] = {nullptr, nullptr};   // |mask correlation| rows, alternating per block (each block reads its history from the other)
    uint8_t* d_events[kBuf] = {}; int* d_ev_count[kBuf] = {}; int ev_cap = 0;
    char* d_bits = nullptr; float* d_disc = nullptr; int* d_bit_count = nullptr; int bit_cap = 0;
    uint8_t* h_events[kBuf] = {}; int* h_ev_count[kBuf] = {};
    // host ingest: two device staging slots filled by a copy stream, so the H2D copy of block k+1 runs beside the
    // kernels of block k
    cudaStream_t stream_copy = nullptr;
    void* stage[2] = {nullptr, nullptr};
    size_t stage_bytes[2] = {0, 0};
    cudaEvent_t copy_done[2] = {}, stage_free[2] = {};
    long long host_pushes = 0;
    long long sb_abs = 0;
    int last_P = 0;
    nvx::NcoChan* d_nco_ch = nullptr;     // [S][C] per-stream NCO parameters (nvx_config.nco_hz), else null: the reference table
    std::vector<nvx::NcoChan> nco_host;   // the same rows with phase origin 0 (retunes edit them here first)
    // the FIR path, one of the two: the fused cascade (fir_cascade.cuh), or the three stage kernels of tap sets too long for it
    // (fir_long.cuh)
    nvx::CascadePath* cp = nullptr;
    nvx::LongPath* lp = nullptr;
    // in front of it, on engines fed at another rate than 252 kS/s (nvx_config.input_rate_hz), the resampler; null otherwise
    nvx::ResamplePath* rp = nullptr;
    int rate = 0;                         // that input rate, 0 = 252 kS/s
    int up = 1, down = 1;                 // 252000 / rate = up / down
    long long align = nvx::kSuper;        // push lengths and max_block are multiples of this many input samples
    int path = 0;                         // what saved state records: 0 / 1 = the fused path's tap class, 2 = the long-tap path
    std::vector<int> stream_tag;          // optional [S][C] message tags (read by the worker; changed through markers)
    // per-stream resets, retunes and loads asked for since the last push; the next push applies them
    struct TagChange { int stream; std::vector<int> tags; };
    enum { kListed = 1, kNewNco = 2, kLoad = 4 };
    std::vector<int> pend_streams;        // in call order, each once
    std::vector<uint8_t> pend_flags;      // [S] kListed | kNewNco | kLoad
    std::vector<TagChange> pend_tags;
    std::vector<int> pend_rec;            // [S] with kLoad: the stream's record in pend_records / pend_text
    std::vector<uint32_t> pend_records;   // loaded records [][layout words], epochs and NCO phases already moved to this engine
    std::vector<std::vector<nvx::MessageAssembler::Channel>> pend_text;   // [record][C] the loaded partial lines and messages
    bool adopted = false;                 // a load placed this engine, which had pushed nothing, at the saved position
    int* d_reset_list = nullptr;          // [2 S] the streams of one push's reset kernel, then the record each loads (-1: none)
    void* h_reset = nullptr;              // pinned: [S][C] NcoChan rows to upload, then [2 S] ints (the list)
    cudaEvent_t reset_copied = nullptr;   // the copies out of h_reset are over
    uint32_t* d_records = nullptr;        // records of one save (gather output) or of one push's loads; grown on demand
    size_t records_cap = 0;               // bytes
    // what the worker does before it assembles block `block`: drop the reset streams' partial lines and messages, put in the
    // loaded streams' ones, switch tags
    struct Loaded { int stream; std::vector<nvx::MessageAssembler::Channel> text; };
    struct Marker { long long block; std::vector<int> streams; std::vector<TagChange> tags; std::vector<Loaded> loads; };
    std::deque<Marker> markers;           // guarded by mu, in push order
    nvx::MessageAssembler assembler;
    std::vector<nvx::AssembledMessage> ready, handed;
    std::vector<nvx_message> view;
    nvx_message_cb cb = nullptr; void* cb_user = nullptr;
    // host-side message assembly runs on a worker thread, one block after the other, off the push path
    std::thread worker;
    std::mutex mu;
    std::condition_variable cv;
    long long queued = 0, drained = 0;      // blocks handed to / finished by the worker
    long long delivered = 0;                // messages completed so far (callback or queue)
    bool stop = false;
    int worker_rc = 0;
    // timing
    int timing = 0;                       // 0 off, 1 = cascade span only, 2 = every demod stage too
    std::vector<cudaEvent_t> ev_pool;
    struct Span { int a, b, kind; };
    std::vector<Span> spans;
    size_t ev_used = 0;
    std::vector<float> cascade_spans_ms;  // every timed cascade launch since the last nvx_engine_get_stats(reset)
    nvx_stats stats = {};
};

namespace {

int free_engine(nvx_engine* e) {
    if (!e) return 0;
    cudaSetDevice(e->cfg.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->stream_demod) cudaStreamSynchronize(e->stream_demod);
    if (e->worker.joinable()) {
        {
            std::lock_guard<std::mutex> lk(e->mu);
            e->stop = true;
        }
        e->cv.notify_all();
        e->worker.join();
    }
    for (cudaEvent_t ev : e->ev_pool) cudaEventDestroy(ev);
    cudaFree(e->corrbuf[0]); cudaFree(e->corrbuf[1]); cudaFree(e->db.clock); cudaFree(e->db.fsm);
    cudaFree(e->db.bitpos); cudaFree(e->db.bitval); cudaFree(e->db.nbits);
    cudaFree(e->d_bits); cudaFree(e->d_disc); cudaFree(e->d_bit_count);
    if (e->stream_copy) cudaStreamSynchronize(e->stream_copy);
    for (int k = 0; k < 2; ++k) {
        cudaFree(e->stage[k]);
        if (e->copy_done[k]) cudaEventDestroy(e->copy_done[k]);
        if (e->stage_free[k]) cudaEventDestroy(e->stage_free[k]);
    }
    if (e->stream_copy) cudaStreamDestroy(e->stream_copy);
    cudaFree(e->d_nco_ch);
    cudaFree(e->db.epoch); cudaFree(e->d_reset_list); cudaFreeHost(e->h_reset); cudaFree(e->d_records);
    if (e->reset_copied) cudaEventDestroy(e->reset_copied);
    nvx::cascade_path_free(e->cp);
    nvx::long_path_free(e->lp);
    nvx::resample_path_free(e->rp);
    for (int k = 0; k < kBuf; ++k) {
        cudaFree(e->y3buf[k]); cudaFree(e->d_events[k]); cudaFree(e->d_ev_count[k]);
        cudaFreeHost(e->h_events[k]); cudaFreeHost(e->h_ev_count[k]);
        if (e->demod_done[k]) cudaEventDestroy(e->demod_done[k]);
        if (e->ff_done[k]) cudaEventDestroy(e->ff_done[k]);
        cudaFree(e->pickbuf[k]);
    }
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->stream_demod) cudaStreamDestroy(e->stream_demod);
    delete e;
    return 0;
}

void set_tags(nvx_engine* e, const nvx_engine::TagChange& t) {
    if (e->stream_tag.empty())
        for (int ch = 0; ch < e->channels; ++ch) e->stream_tag.push_back(e->cfg.freq_tag[(ch % e->C) & 1]);
    std::copy(t.tags.begin(), t.tags.end(), e->stream_tag.begin() + (size_t)t.stream * e->C);
}

int reset_state(nvx_engine* e) {
    e->fmt = -1;                                    // the next push fixes the format
    // per-stream resets still pending are part of this one; their new tags take effect now, their offsets are in nco_host
    for (const auto& t : e->pend_tags) set_tags(e, t);
    for (int s : e->pend_streams) e->pend_flags[(size_t)s] = 0;
    e->pend_streams.clear();
    e->pend_tags.clear();
    e->pend_records.clear();
    e->pend_text.clear();
    e->adopted = false;
    if (e->d_nco_ch)   // every row's phase origin back to 0
        CU_TRY(cudaMemcpyAsync(e->d_nco_ch, e->nco_host.data(), e->nco_host.size() * sizeof(nvx::NcoChan), cudaMemcpyHostToDevice, e->stream));
    if (e->lp) CU_TRY(nvx::long_path_reset(e->lp, e->stream));
    else nvx::cascade_path_reset(e->cp);
    if (e->rp) CU_TRY(nvx::resample_path_reset(e->rp, e->stream));
    for (int k = 0; k < kBuf; ++k) {
        e->db.y3 = e->y3buf[k];
        e->db.picks = e->pickbuf[k];
        e->db.corr = e->corrbuf[k & 1];
        CU_TRY(nvx::demod_init_state(e->db, e->channels, e->stream));
    }
    CU_TRY(cudaStreamSynchronize(e->stream));
    e->sb_abs = 0;
    e->last_P = 0;
    e->blocks = 0;
    e->last_buf = 0;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->queued = e->drained = 0;
        e->worker_rc = 0;
        e->markers.clear();
    }
    e->assembler.reset();
    e->ready.clear();
    return 0;
}

constexpr int kSpanResample = 8;          // span kinds: 0 cascade, 1 demod chain, 2 .. 7 demod stages, 8 resampler

cudaEvent_t next_event(nvx_engine* e) {
    if (e->ev_used == e->ev_pool.size()) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        e->ev_pool.push_back(ev);
    }
    return e->ev_pool[e->ev_used++];
}

void collect_spans(nvx_engine* e) {
    if (!e->timing || e->spans.empty()) return;
    for (const auto& sp : e->spans) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e->ev_pool[sp.a], e->ev_pool[sp.b]);
        if (sp.kind == 0) {
            e->stats.cascade_ms += ms;
            if (e->cascade_spans_ms.size() < (1u << 20)) e->cascade_spans_ms.push_back(ms);
            if (e->stats.cascade_ms_min == 0.0 || ms < e->stats.cascade_ms_min) e->stats.cascade_ms_min = ms;
            if (ms > e->stats.cascade_ms_max) e->stats.cascade_ms_max = ms;
        }
        else if (sp.kind == 1) e->stats.demod_ms += ms;
        else if (sp.kind == kSpanResample) e->stats.resample_ms += ms;
        else e->stats.demod_stage_ms[sp.kind - 2] += ms;
    }
    e->spans.clear();
    e->ev_used = 0;
}

// host half of one block (worker thread): wait for its demod_done event, then assemble messages
int drain_events(nvx_engine* e, int b) {
    int rc = 0;
    std::vector<nvx::AssembledMessage> out;
    for (int ch = 0; ch < e->channels; ++ch) {
        int n = e->h_ev_count[b][ch];
        if (n > e->ev_cap) { n = e->ev_cap; rc = NVX_ERR_OVERFLOW; }
        if (n > 0)
            e->assembler.feed(ch, e->cfg.first_stream_id + ch / e->C, e->stream_tag.empty() ? e->cfg.freq_tag[(ch % e->C) & 1] : e->stream_tag[ch],
                              e->h_events[b] + (size_t)ch * e->ev_cap,
                              (size_t)n, &out);
    }
    if (!out.empty()) {
        // With a callback installed the messages are delivered right here, on the worker thread, as soon as the block that
        // completed them has drained -- the reference calls add_message the moment NNNN or an abort is seen
        // (nav_b_sm.C:47-50, :82-88).  Without one they queue for nvx_engine_poll_messages.
        nvx_message_cb cb;
        void* user;
        {
            std::lock_guard<std::mutex> lk(e->mu);
            cb = e->cb; user = e->cb_user;
            if (!cb) for (auto& m : out) e->ready.push_back(std::move(m));
            e->delivered += (long long)out.size();
        }
        if (cb)
            for (auto& m : out) {
                std::string bb = m.bbbb, t = m.text;
                cb(user, m.stream, &bb[0], &t[0], m.freq);
            }
    }
    return rc;
}

void worker_main(nvx_engine* e) {
    cudaSetDevice(e->cfg.device);
    for (;;) {
        long long blk;
        {
            std::unique_lock<std::mutex> lk(e->mu);
            e->cv.wait(lk, [&] { return e->stop || e->drained < e->queued; });
            if (e->drained >= e->queued) return;      // stop requested and nothing left
            blk = e->drained;
        }
        const int b = (int)(blk % kBuf);
        std::vector<nvx_engine::Marker> take;
        {
            std::lock_guard<std::mutex> lk(e->mu);
            while (!e->markers.empty() && e->markers.front().block <= blk) {
                take.push_back(std::move(e->markers.front()));
                e->markers.pop_front();
            }
        }
        for (const auto& m : take) {       // blocks before this one were assembled under the old state and tags
            for (int s : m.streams)
                for (int c = 0; c < e->C; ++c) e->assembler.reset_channel(s * e->C + c);
            for (const auto& l : m.loads)
                for (int c = 0; c < e->C; ++c) e->assembler.set_channel(l.stream * e->C + c, l.text[(size_t)c]);
            for (const auto& t : m.tags) set_tags(e, t);
        }
        int rc = 0;
        if (cudaEventSynchronize(e->demod_done[b]) != cudaSuccess) rc = NVX_ERR_CUDA;
        else rc = drain_events(e, b);
        {
            std::lock_guard<std::mutex> lk(e->mu);
            if (rc && !e->worker_rc) e->worker_rc = rc;
            e->drained = blk + 1;
        }
        e->cv.notify_all();
    }
}

// wait until the worker has drained every block up to (not including) `upto`
void wait_drained(nvx_engine* e, long long upto) {
    std::unique_lock<std::mutex> lk(e->mu);
    e->cv.wait(lk, [&] { return e->drained >= upto; });
}

// messages that were queued before a callback was installed
void deliver_callbacks(nvx_engine* e) {
    std::vector<nvx::AssembledMessage> take;
    nvx_message_cb cb;
    void* user;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        cb = e->cb; user = e->cb_user;
        if (!cb) return;
        take.swap(e->ready);
    }
    for (auto& m : take) {
        std::string bb = m.bbbb, t = m.text;
        cb(user, m.stream, &bb[0], &t[0], m.freq);
    }
}

int sync_engine(nvx_engine* e) {
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->stream_copy));
    CU_TRY(cudaStreamSynchronize(e->stream));
    CU_TRY(cudaStreamSynchronize(e->stream_demod));
    collect_spans(e);
    wait_drained(e, e->blocks);
    deliver_callbacks(e);
    int rc;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        rc = e->worker_rc;
        e->worker_rc = 0;
    }
    if (rc == NVX_ERR_OVERFLOW) return fail(rc, "an event buffer overflowed");
    if (rc) return fail(rc, "event download failed");
    return 0;
}

// what the FIR path reports goes into this engine's nvx_stats and nvx_last_error()
int path_report(nvx_engine* e, int rc, const nvx::PathReport& rep) {
    e->stats.aux_launches += rep.launches;
    e->stats.long_tc_fallbacks += rep.fallbacks;
    if (rep.msg[0]) fail(rc, "%s", rep.msg);
    return rc;
}

// the addresses of every stream's carried state as the next block reads it (list, records and e0 are the caller's)
ResetArgs state_args(nvx_engine* e) {
    using namespace nvx;
    ResetArgs a = {};
    a.C = e->C;
    a.rows = e->lp ? long_path_carried(e->lp) : cascade_path_carried(e->cp);
    if (e->rp) a.pre = resample_path_carried(e->rp);
    a.lay = state_layout(a.rows.words, e->C, e->d_nco_ch != nullptr, a.pre.words[0]);
    a.y3_prev = e->y3buf[(e->blocks + kBuf - 1) % kBuf];
    a.y3_pitch = kHistY + e->P_max;
    a.corr_prev = e->corrbuf[(e->blocks & 1) ^ 1];
    a.corr_pitch = kHistC + e->P_max + kPadC;
    a.n_prev = e->last_P;
    a.clock = e->db.clock; a.fsm = e->db.fsm; a.epoch = e->db.epoch;
    a.nco = e->d_nco_ch;
    return a;
}

int reset_buffers(nvx_engine* e) {
    if (e->d_reset_list) return 0;
    CU_TRY(cudaMalloc(&e->d_reset_list, 2 * (size_t)e->S * sizeof(int)));
    CU_TRY(cudaHostAlloc(&e->h_reset, (size_t)e->S * e->C * sizeof(nvx::NcoChan) + 2 * (size_t)e->S * sizeof(int), cudaHostAllocDefault));
    CU_TRY(cudaEventCreateWithFlags(&e->reset_copied, cudaEventDisableTiming));
    CU_TRY(cudaEventRecord(e->reset_copied, e->stream));
    return 0;
}

// d_records holds at least `bytes` (the engine stream's earlier work on it is over before it is replaced)
int records_buffer(nvx_engine* e, size_t bytes) {
    if (e->records_cap >= bytes) return 0;
    CU_TRY(cudaStreamSynchronize(e->stream));
    cudaFree(e->d_records);
    e->d_records = nullptr;
    e->records_cap = 0;
    CU_TRY(cudaMalloc(&e->d_records, bytes));
    e->records_cap = bytes;
    return 0;
}

// the resets and loads asked for since the last push, queued in front of this block: NCO rows of retuned and loaded streams, the
// loaded records, the reset kernel, and the marker that tells the worker from which block on the streams' messages start over
// (or go on from the loaded partial lines and messages)
int apply_resets(nvx_engine* e) {
    using namespace nvx;
    const int count = (int)e->pend_streams.size();
    if (!count) return 0;
    const size_t rows_bytes = (size_t)e->S * e->C * sizeof(NcoChan);
    if (int rc = reset_buffers(e)) return rc;
    CU_TRY(cudaEventSynchronize(e->reset_copied));      // the previous copies out of h_reset are over
    NcoChan* h_rows = static_cast<NcoChan*>(e->h_reset);
    int* h_list = reinterpret_cast<int*>(static_cast<char*>(e->h_reset) + rows_bytes);
    int retuned = 0;
    nvx_engine::Marker mk;
    for (int i = 0; i < count; ++i) {
        const int s = e->pend_streams[(size_t)i];
        const uint8_t f = e->pend_flags[(size_t)s];
        h_list[i] = s;
        h_list[count + i] = f & nvx_engine::kLoad ? e->pend_rec[(size_t)s] : -1;
        if (f & nvx_engine::kNewNco) {
            NcoChan* src = h_rows + (size_t)retuned++ * e->C;
            memcpy(src, &e->nco_host[(size_t)s * e->C], e->C * sizeof(NcoChan));
            CU_TRY(cudaMemcpyAsync(e->d_nco_ch + (size_t)s * e->C, src, e->C * sizeof(NcoChan), cudaMemcpyHostToDevice, e->stream));
        }
        if (f & nvx_engine::kLoad) mk.loads.push_back({s, std::move(e->pend_text[(size_t)e->pend_rec[(size_t)s]])});
        else mk.streams.push_back(s);
        e->pend_flags[(size_t)s] = 0;
    }
    CU_TRY(cudaMemcpyAsync(e->d_reset_list, h_list, 2 * (size_t)count * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    CU_TRY(cudaEventRecord(e->reset_copied, e->stream));
    ResetArgs ra = state_args(e);
    if (!e->pend_records.empty()) {
        const size_t bytes = e->pend_records.size() * sizeof(uint32_t);
        if (int rc = records_buffer(e, bytes)) return rc;
        CU_TRY(cudaMemcpyAsync(e->d_records, e->pend_records.data(), bytes, cudaMemcpyHostToDevice, e->stream));
        ra.rec = e->d_records;
    }
    if (e->blocks > 0) CU_TRY(cudaStreamWaitEvent(e->stream, e->demod_done[e->last_buf], 0));
    ra.streams = e->d_reset_list;
    ra.recs = e->d_reset_list + count;
    ra.e0 = e->sb_abs - e->sb_abs % kCorrLen;
    reset_streams_kernel<<<(unsigned)count, 256, 0, e->stream>>>(ra);
    CU_TRY(cudaGetLastError());
    e->stats.aux_launches++;
    mk.block = e->blocks;
    mk.tags = std::move(e->pend_tags);
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->markers.push_back(std::move(mk));
    }
    e->pend_streams.clear();
    e->pend_tags.clear();
    e->pend_records.clear();
    e->pend_text.clear();
    return 0;
}

int process_block(nvx_engine* e, const void* d_x, long long n, nvx::SampleFmt fmt) {
    using namespace nvx;
    if (e->fmt >= 0 && e->fmt != (int)fmt)
        return fail(NVX_ERR_ARG, "sample format changed between pushes (float, int16 and 8-bit blocks cannot be mixed without a reset)");
    if (n <= 0 || n % e->align != 0) return fail(NVX_ERR_ARG, "block length %lld is not a positive multiple of %lld", n, e->align);
    if (n > e->cfg.max_block) return fail(NVX_ERR_ARG, "block length %lld exceeds max_block %lld", n, e->cfg.max_block);
    if (((uintptr_t)d_x & 15) != 0) return fail(NVX_ERR_ARG, "device block is not 16-byte aligned");
    e->fmt = (int)fmt;                              // only a block that is accepted fixes the format
    const int b = (int)(e->blocks % kBuf);
    wait_drained(e, e->blocks - kBuf + 1);          // block (blocks - kBuf) used these buffers: long finished, normally
    if (int rc = apply_resets(e)) return rc;
    if (e->timing && e->ev_used > 4000) {            // bound the event pool in long timed runs
        CU_TRY(cudaStreamSynchronize(e->stream));
        CU_TRY(cudaStreamSynchronize(e->stream_demod));
        collect_spans(e);
    }
    // the FIR path runs at 252 kS/s: on the resampler's float output when the engine is fed at another rate
    const void* x = d_x;
    long long n_fir = n;
    SampleFmt fir_fmt = fmt;
    if (e->rp) {
        PathReport rrep;
        const float2* y = nullptr;
        if (e->timing) {
            e->spans.push_back({(int)e->ev_used, (int)e->ev_used + 1, kSpanResample});
            CU_TRY(cudaEventRecord(next_event(e), e->stream));
        }
        const int rc = resample_path_run(e->rp, d_x, n, fmt, e->stream, &y, &n_fir, &rrep);
        if (path_report(e, rc, rrep)) return rc;
        if (e->timing) CU_TRY(cudaEventRecord(next_event(e), e->stream));
        x = y;
        fir_fmt = SampleFmt::F32;
    }
    const int n_super = (int)(n_fir / kSuper);

    cudaEvent_t t0 = nullptr, t1 = nullptr, marks[8] = {};
    if (e->timing) {
        const int base = (int)e->ev_used;
        t0 = next_event(e); t1 = next_event(e);
        e->spans.push_back({base, base + 1, 0});
        if (e->timing > 1) {
            for (int k = 0; k < 8; ++k) marks[k] = next_event(e);
            e->spans.push_back({base + 2, base + 9, 1});                                      // whole demod chain
            for (int k = 0; k < 3; ++k) e->spans.push_back({base + 2 + k, base + 3 + k, 2 + k});   // angle, sums, carry
            for (int k = 0; k < 3; ++k) e->spans.push_back({base + 6 + k, base + 7 + k, 5 + k});   // clock, decide, fsm
        }
        CU_TRY(cudaEventRecord(t0, e->stream));
    }
    PathReport rep;
    const long long y3_pitch = kHistY + e->P_max;
    const int rc = e->lp ? long_path_run(e->lp, x, n_fir, fir_fmt, e->sb_abs, e->y3buf[b], y3_pitch, kHistY, e->stream, t1, &rep)
                         : cascade_path_run(e->cp, x, n_fir, fir_fmt, e->sb_abs, e->y3buf[b], y3_pitch, kHistY, e->stream, t1, &rep);
    if (path_report(e, rc, rep)) return rc;

    // demod of this block runs on its own stream, overlapping the next block's cascade
    DemodArgs da;
    da.b = e->db;
    da.b.y3 = e->y3buf[b];
    da.b.picks = e->pickbuf[b];
    da.b.corr = e->corrbuf[e->blocks & 1];
    da.y3_prev = e->y3buf[(b + kBuf - 1) % kBuf];
    da.corr_prev = e->corrbuf[(e->blocks & 1) ^ 1];
    da.n_prev = e->last_P;
    da.n_new = n_super; da.channels = e->channels; da.seen = e->sb_abs;
    da.events = e->d_events[b]; da.ev_count = e->d_ev_count[b]; da.ev_cap = e->ev_cap;
    da.bits = e->d_bits; da.disc = e->d_disc; da.bit_count = e->d_bit_count; da.bit_cap = e->bit_cap;
    // The feed-forward demod kernels are short whole-GPU kernels (0.25 ms of FP64 work per 10 s block of 2048 channels); beside
    // the cascade (one warp per SM sub-partition, little latency slack) they cost it about what they take alone, so they follow
    // it on the main stream and only the sequential symbol-clock / state-machine kernels (64 warps on the SMs the cascade grid
    // leaves free) overlap the next block's cascade (the whole chain beside it measured no faster: DESIGN.md §3.3).  The main
    // stream also orders their look-back into the previous block's y3 buffer before the cascade two blocks on, which
    // overwrites it.
    CU_TRY(demod_launch(da, e->stream, e->stream_demod, e->ff_done[b], e->timing > 1 ? marks : nullptr));
    CU_TRY(cudaMemcpyAsync(e->h_ev_count[b], e->d_ev_count[b], sizeof(int) * e->channels, cudaMemcpyDeviceToHost, e->stream_demod));
    CU_TRY(cudaMemcpyAsync(e->h_events[b], e->d_events[b], (size_t)e->channels * e->ev_cap, cudaMemcpyDeviceToHost, e->stream_demod));
    CU_TRY(cudaEventRecord(e->demod_done[b], e->stream_demod));
    // the next block's cascade may overwrite neither this block's input staging nor (two blocks on) its y3
    // buffer before the demod has consumed them: the staging buffers are only touched on e->stream (ordered),
    // the y3 buffer is protected by the demod_done wait above
    e->last_buf = b;
    e->blocks++;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->queued = e->blocks;
    }
    e->cv.notify_all();
    e->sb_abs += n_super;
    e->last_P = n_super;
    e->stats.cascade_launches++;
    e->stats.demod_launches += nvx::demod_launches_per_block();
    e->stats.samples += n * e->S;
    return 0;
}

// H2D on the copy stream into staging slot k % 2, then the block's kernels on the main stream
int push_host(nvx_engine* e, const void* iq, long long n, nvx::SampleFmt fmt) {
    if (n <= 0 || n % e->align != 0 || n > e->cfg.max_block) return fail(NVX_ERR_ARG, "bad block length %lld (a positive multiple of %lld up to max_block)", n, e->align);
    CU_TRY(cudaSetDevice(e->cfg.device));
    const size_t bytes = (size_t)e->S * (size_t)n * nvx::sample_bytes(fmt);
    const int slot = (int)(e->host_pushes % 2);
    if (e->stage_bytes[slot] < bytes) {
        CU_TRY(cudaStreamSynchronize(e->stream_copy));
        CU_TRY(cudaStreamSynchronize(e->stream));
        cudaFree(e->stage[slot]);
        e->stage[slot] = nullptr; e->stage_bytes[slot] = 0;
        CU_TRY(cudaMalloc(&e->stage[slot], bytes));
        e->stage_bytes[slot] = bytes;
    }
    CU_TRY(cudaStreamWaitEvent(e->stream_copy, e->stage_free[slot], 0));     // the block that used this slot two pushes ago
    CU_TRY(cudaMemcpyAsync(e->stage[slot], iq, bytes, cudaMemcpyHostToDevice, e->stream_copy));
    CU_TRY(cudaEventRecord(e->copy_done[slot], e->stream_copy));
    CU_TRY(cudaStreamWaitEvent(e->stream, e->copy_done[slot], 0));
    if (int rc = process_block(e, e->stage[slot], n, fmt)) return rc;
    CU_TRY(cudaEventRecord(e->stage_free[slot], e->stream));
    e->host_pushes++;
    return 0;
}

// ---- saved stream state (nvx_engine_save_streams): header | count device records of rec_words words | per record and channel:
// tag, in_message, the lengths of line / text / bbbb, then their bytes.  Native byte order.
constexpr uint32_t kStateMagic = 0x5358564eu;      // "NVXS"
constexpr uint32_t kStateVersion = 1;
constexpr long long kStateGrid = (long long)nvx::kCorrLen * nvx::kSuper;     // 158760: positions must agree modulo this
struct StateHeader {
    uint32_t magic, version;
    uint64_t bytes;                     // the whole state
    uint64_t checksum;                  // hash_bytes of every byte but these eight
    long long position;                 // E: input samples per stream pushed before the save
    long long words[3];                 // the FIR path's CarriedRows words
    uint64_t taps;                      // the path's tap hash
    long long rec_words;                // words per device record
    int32_t count, n_channels, fmt, path, gen_nco;
    int32_t rate;                       // input rate of an engine that resamples (nvx_config.input_rate_hz), 0 = 252 kS/s
};
static_assert(sizeof(StateHeader) == 96, "state header layout");
constexpr size_t kChecksumAt = offsetof(StateHeader, checksum);
using ChannelText = nvx::MessageAssembler::Channel;

uint64_t state_checksum(const uint8_t* p, size_t n) {
    return nvx::hash_bytes(p + kChecksumAt + 8, n - kChecksumAt - 8, nvx::hash_bytes(p, kChecksumAt));
}

// input samples per stream pushed so far, and the restart grid, in input samples (158760 x down / up)
long long in_position(const nvx_engine* e) { return e->sb_abs * nvx::kSuper / e->up * e->down; }
long long in_grid(const nvx_engine* e) { return kStateGrid / e->up * e->down; }

// words of the resampler's history per stream at that input rate (0 = 252 kS/s); -1 for a rate no engine takes
long long resampler_words(int rate) {
    if (rate == 0) return 0;
    nvx::ResampleDesign d;
    const char* why = "";
    if (rate == NVX_FS_HZ || !nvx::resample_geometry(rate, &d, &why)) return -1;
    return 2LL * (d.J - 1);
}

const char* path_name(int path) { return path == 0 ? "fused path (reference tap class)" : path == 1 ? "fused path (medium tap class)" : "long-tap path"; }

// validates a saved state completely (nothing is half-applied) and returns its header and [record][channel] texts and tags
int parse_state(const void* state, size_t size, StateHeader* h, std::vector<std::vector<ChannelText>>* text, std::vector<std::vector<int>>* tags) {
    if (!state || size < sizeof(StateHeader)) return fail(NVX_ERR_ARG, "saved stream state: %zu bytes, shorter than its %zu-byte header", state ? size : 0, sizeof(StateHeader));
    const uint8_t* p = static_cast<const uint8_t*>(state);
    memcpy(h, p, sizeof *h);
    if (h->magic != kStateMagic) return fail(NVX_ERR_ARG, "saved stream state: bad magic number 0x%08x", h->magic);
    if (h->version != kStateVersion) return fail(NVX_ERR_ARG, "saved stream state: version %u, this library reads version %u", h->version, kStateVersion);
    if (h->bytes != size) return fail(NVX_ERR_ARG, "saved stream state: %zu bytes given, the state has %llu (truncated?)", size, (unsigned long long)h->bytes);
    if (state_checksum(p, size) != h->checksum) return fail(NVX_ERR_ARG, "saved stream state: checksum mismatch (the bytes were altered)");
    const long long pre_words = resampler_words(h->rate);
    if (pre_words < 0) return fail(NVX_ERR_ARG, "saved stream state: inconsistent header");
    nvx::ResampleDesign rd;
    const char* why = "";
    nvx::resample_geometry(h->rate ? h->rate : NVX_FS_HZ, &rd, &why);
    const long long rec_words = state_layout(h->words, h->n_channels, h->gen_nco != 0, pre_words).words;
    if (h->count < 0 || h->n_channels < 1 || h->n_channels > nvx::kMaxChannels || h->fmt < 0 || h->fmt >= nvx::kSampleFmts || h->path < 0 ||
        h->path > 2 || (h->gen_nco != 0 && h->gen_nco != 1) || h->position < 0 || h->position % rd.align || h->words[0] < 0 ||
        h->words[1] < 0 || h->words[2] < 0 || h->rec_words != rec_words)
        return fail(NVX_ERR_ARG, "saved stream state: inconsistent header");
    size_t at = sizeof(StateHeader);
    if ((size - at) / sizeof(uint32_t) / (size_t)rec_words < (size_t)h->count) return fail(NVX_ERR_ARG, "saved stream state: records cut short");
    at += (size_t)h->count * rec_words * sizeof(uint32_t);
    text->assign((size_t)h->count, std::vector<ChannelText>((size_t)h->n_channels));
    tags->assign((size_t)h->count, std::vector<int>((size_t)h->n_channels));
    for (int k = 0; k < h->count; ++k)
        for (int c = 0; c < h->n_channels; ++c) {
            int32_t v[5];
            if (size - at < sizeof v) return fail(NVX_ERR_ARG, "saved stream state: message part cut short");
            memcpy(v, p + at, sizeof v);
            at += sizeof v;
            ChannelText& t = (*text)[(size_t)k][(size_t)c];
            (*tags)[(size_t)k][(size_t)c] = v[0];
            t.in_message = v[1] != 0;
            std::string* str[3] = {&t.line, &t.text, &t.bbbb};
            for (int i = 0; i < 3; ++i) {
                if (v[2 + i] < 0 || (size_t)v[2 + i] > size - at) return fail(NVX_ERR_ARG, "saved stream state: message part cut short");
                str[i]->assign(reinterpret_cast<const char*>(p + at), (size_t)v[2 + i]);
                at += (size_t)v[2 + i];
            }
        }
    if (at != size) return fail(NVX_ERR_ARG, "saved stream state: %zu bytes after the last record", size - at);
    return 0;
}

// streams[0..count) are local streams, each listed once
int check_stream_list(const nvx_engine* e, const int* streams, int count) {
    std::vector<char> seen((size_t)e->S, 0);
    for (int i = 0; i < count; ++i) {
        if (streams[i] < 0 || streams[i] >= e->S) return fail(NVX_ERR_ARG, "stream %d outside 0..%d", streams[i], e->S - 1);
        if (seen[(size_t)streams[i]]++) return fail(NVX_ERR_ARG, "stream %d is listed twice", streams[i]);
    }
    return 0;
}

}  // namespace

namespace nvx {
long long engine_block_align(const nvx_engine* e) { return e->align; }
}  // namespace nvx

extern "C" {

const char* nvx_last_error(void) { return g_err; }

void nvx_default_config(nvx_config* cfg) {
    memset(cfg, 0, sizeof *cfg);
    cfg->n_streams = 1;
    cfg->max_block = 252000;
    cfg->freq_tag[0] = 518;   // nav_sched.C:10-11
    cfg->freq_tag[1] = 490;
}

int nvx_resampler_info(int input_rate_hz, int* up, int* down, long long* block_align, double* h, size_t cap, size_t* n_taps) {
    nvx::ResampleDesign d;
    const char* why = "";
    if (!(h ? nvx::resample_design(input_rate_hz, &d, &why) : nvx::resample_geometry(input_rate_hz, &d, &why)))
        return fail(NVX_ERR_ARG, "input rate %d: %s", input_rate_hz, why);
    if (up) *up = d.L;
    if (down) *down = d.M;
    if (block_align) *block_align = d.align;
    if (n_taps) *n_taps = (size_t)d.L * d.J;
    if (!h) return 0;
    if (cap < d.h.size()) return fail(NVX_ERR_OVERFLOW, "the resampler has %zu taps, the buffer holds %zu", d.h.size(), cap);
    memcpy(h, d.h.data(), d.h.size() * sizeof(double));
    return 0;
}

int nvx_engine_create(const nvx_config* cfg, nvx_engine** out) {
    if (!cfg || !out) return fail(NVX_ERR_ARG, "null argument");
    // input rate: 252 kS/s as it is, or resampled on the device; every count of samples below is in input samples
    nvx::ResampleDesign rd;
    const char* why = "";
    if (cfg->input_rate_hz != 0 && !nvx::resample_geometry(cfg->input_rate_hz, &rd, &why))
        return fail(NVX_ERR_ARG, "input_rate_hz %d: %s", cfg->input_rate_hz, why);
    if (cfg->n_streams <= 0 || cfg->max_block <= 0 || cfg->max_block % rd.align != 0)
        return fail(NVX_ERR_ARG, "n_streams must be > 0 and max_block a positive multiple of %lld", rd.align);
    const long long max_fir = cfg->max_block / rd.M * rd.L;       // the largest block at 252 kS/s
    if (cfg->n_streams > 32767)       // channel rows index the y dimension of the demod grids (65535 max)
        return fail(NVX_ERR_ARG, "n_streams %d exceeds 32767 per engine: shard the streams over more engines", cfg->n_streams);
    if (max_fir / nvx::kSuper > (1 << 24))
        return fail(NVX_ERR_ARG, "max_block %lld is too long (at most %d samples per push at 252 kS/s)", cfg->max_block, nvx::kSuper << 24);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev)
        return fail(NVX_ERR_CUDA, "no usable CUDA device %d (%d visible): this library has no CPU path", cfg->device, ndev);
    CU_TRY(cudaSetDevice(cfg->device));
    nvx_engine* e = new nvx_engine();
    e->cfg = *cfg;
    if (e->cfg.freq_tag[0] == 0 && e->cfg.freq_tag[1] == 0) { e->cfg.freq_tag[0] = 518; e->cfg.freq_tag[1] = 490; }
    e->cfg.h1 = e->cfg.h2 = e->cfg.h3 = nullptr;    // copied to the device below, not retained
    e->cfg.nco_hz = nullptr;
    e->cfg.stream_freq_tag = nullptr;
    const int C = cfg->n_channels ? cfg->n_channels : 2;
    if (C < 1 || C > nvx::kMaxChannels) { delete e; return fail(NVX_ERR_ARG, "n_channels %d outside 1..%d", C, nvx::kMaxChannels); }
    if (C != 2 && !cfg->nco_hz) { delete e; return fail(NVX_ERR_ARG, "n_channels = %d needs nco_hz (only the reference's two channels have default offsets)", C); }
    if ((long long)C * cfg->n_streams > 65535) { delete e; return fail(NVX_ERR_ARG, "n_streams x n_channels = %lld exceeds 65535 channel rows per engine", (long long)C * cfg->n_streams); }
    e->C = C;
    e->rate = rd.L != rd.M ? cfg->input_rate_hz : 0;
    e->up = rd.L; e->down = rd.M; e->align = rd.align;
    if (cfg->stream_freq_tag) e->stream_tag.assign(cfg->stream_freq_tag, cfg->stream_freq_tag + (size_t)C * (size_t)cfg->n_streams);
    if (cfg->nco_hz) {
        e->nco_host.resize((size_t)cfg->n_streams * C);
        for (int k = 0; k < C * cfg->n_streams; ++k)
            if (!nco_entry(cfg->nco_hz[k], &e->nco_host[(size_t)k])) {
                delete e;
                return fail(NVX_ERR_ARG, "nco_hz[%d] = %g is not a multiple of 0.5 Hz inside +-31.5 kHz", k, cfg->nco_hz[k]);
            }
    }
    e->S = cfg->n_streams;
    e->channels = C * e->S;
    e->pend_flags.assign((size_t)e->S, 0);
    e->pend_rec.assign((size_t)e->S, -1);
    e->P_max = (int)(max_fir / nvx::kSuper);
    // tap counts: reference lengths unless given; sets up to 37/47/71 and up to 61/75/111 run through the fused kernel
    // (zero-padded to the class), longer ones through the long-tap path
    const int n[3] = {cfg->n1 ? cfg->n1 : NVX_T1, cfg->n2 ? cfg->n2 : NVX_T2, cfg->n3 ? cfg->n3 : NVX_T3};
    if ((cfg->n1 && !cfg->h1) || (cfg->n2 && !cfg->h2) || (cfg->n3 && !cfg->h3)) {
        delete e;
        return fail(NVX_ERR_ARG, "a tap count was given without its tap array");
    }
    for (int k = 0; k < 3; ++k)
        if (n[k] < 1 || n[k] > nvx::kLongMaxTaps) { delete e; return fail(NVX_ERR_ARG, "tap count %d outside 1..%d", n[k], nvx::kLongMaxTaps); }
    // the FIR path: the fused cascade for sets it takes, else the long-tap path; only the fused reference class serves other than
    // the reference's two channels
    const int tap_class = nvx::cascade_tap_class(n[0], n[1], n[2]);
    e->path = tap_class >= 0 ? tap_class : 2;
    if (C != 2 && tap_class != 0) {
        delete e;
        return fail(NVX_ERR_ARG, "n_channels = %d is served by the fused kernel's reference tap class only (up to %d / %d / %d taps)", C, NVX_T1, NVX_T2, NVX_T3);
    }
    // per block and channel: at most one character plus one abort per 14 bits ... generous bound
    e->ev_cap = 2 * (e->P_max / 63 + 2) + 8;
    e->bit_cap = cfg->keep_bits ? e->P_max / 8 + 2 : 0;      // the symbol clock may run one sample per bit fast while it slews
#define CREATE_TRY(expr)                                                                                      \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess) {                                                                             \
            fail(NVX_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__));                              \
            free_engine(e);                                                                                   \
            return e__ == cudaErrorMemoryAllocation ? NVX_ERR_NOMEM : NVX_ERR_CUDA;                           \
        }                                                                                                     \
    } while (0)
    {   // the short demod kernels of block i get the leftover SM resources first while block i+1's cascade runs
        int lo = 0, hi = 0;
        CREATE_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CREATE_TRY(cudaStreamCreateWithPriority(&e->stream, cudaStreamNonBlocking, lo));
        CREATE_TRY(cudaStreamCreateWithFlags(&e->stream_copy, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            CREATE_TRY(cudaEventCreateWithFlags(&e->copy_done[k], cudaEventDisableTiming));
            CREATE_TRY(cudaEventCreateWithFlags(&e->stage_free[k], cudaEventDisableTiming));
        }
        CREATE_TRY(cudaStreamCreateWithPriority(&e->stream_demod, cudaStreamNonBlocking, hi));
    }
    for (int k = 0; k < kBuf; ++k) {
        CREATE_TRY(cudaEventCreateWithFlags(&e->demod_done[k], cudaEventDisableTiming));
        CREATE_TRY(cudaEventCreateWithFlags(&e->ff_done[k], cudaEventDisableTiming));
    }
    e->db.p_max = e->P_max;
    for (int k = 0; k < kBuf; ++k) CREATE_TRY(cudaMalloc(&e->y3buf[k], (size_t)e->channels * (nvx::kHistY + e->P_max) * sizeof(float2)));
    for (int k = 0; k < 2; ++k) CREATE_TRY(cudaMalloc(&e->corrbuf[k], (size_t)e->channels * (nvx::kHistC + e->P_max + nvx::kPadC) * sizeof(double)));
    for (int k = 0; k < kBuf; ++k) CREATE_TRY(cudaMalloc(&e->pickbuf[k], (size_t)e->channels * nvx::demod_pick_pitch(e->P_max)));
    CREATE_TRY(cudaMalloc(&e->db.bitpos, (size_t)e->channels * nvx::demod_bit_pitch(e->P_max) * sizeof(int)));
    CREATE_TRY(cudaMalloc(&e->db.bitval, (size_t)e->channels * nvx::demod_bit_pitch(e->P_max)));
    CREATE_TRY(cudaMalloc(&e->db.nbits, (size_t)e->channels * sizeof(int)));
    CREATE_TRY(cudaMemset(e->db.nbits, 0, (size_t)e->channels * sizeof(int)));
    CREATE_TRY(cudaMalloc(&e->db.clock, (size_t)e->channels * sizeof(nvx::ClockState)));
    CREATE_TRY(cudaMalloc(&e->db.fsm, (size_t)e->channels * sizeof(nvx::FsmState)));
    CREATE_TRY(cudaMalloc(&e->db.epoch, (size_t)e->channels * sizeof(long long)));
    for (int k = 0; k < kBuf; ++k) {
        CREATE_TRY(cudaMalloc(&e->d_events[k], (size_t)e->channels * e->ev_cap));
        CREATE_TRY(cudaMalloc(&e->d_ev_count[k], sizeof(int) * e->channels));
        CREATE_TRY(cudaMemset(e->d_ev_count[k], 0, sizeof(int) * e->channels));
        CREATE_TRY(cudaMallocHost(&e->h_events[k], (size_t)e->channels * e->ev_cap));
        CREATE_TRY(cudaMallocHost(&e->h_ev_count[k], sizeof(int) * e->channels));
        memset(e->h_ev_count[k], 0, sizeof(int) * e->channels);
    }
    if (cfg->keep_bits) {
        CREATE_TRY(cudaMalloc(&e->d_bits, (size_t)e->channels * e->bit_cap));
        CREATE_TRY(cudaMalloc(&e->d_disc, (size_t)e->channels * e->bit_cap * 4 * sizeof(float)));
        CREATE_TRY(cudaMalloc(&e->d_bit_count, sizeof(int) * e->channels));
        CREATE_TRY(cudaMemset(e->d_bit_count, 0, sizeof(int) * e->channels));
    }
    if (!e->nco_host.empty()) CREATE_TRY(cudaMalloc(&e->d_nco_ch, e->nco_host.size() * sizeof(nvx::NcoChan)));   // filled by reset_state
#undef CREATE_TRY
    {
        const double* const h[3] = {cfg->h1, cfg->h2, cfg->h3};
        nvx::PathReport rep;
        const int rc = tap_class >= 0
                           ? nvx::cascade_path_create(e->S, C, n, h, e->d_nco_ch, cfg->device, nvx::demod_reserved_sms(e->channels), &e->cp, &rep)
                           : nvx::long_path_create(e->S, max_fir, n, h, e->d_nco_ch, e->stream, &e->lp, &rep);
        if (path_report(e, rc, rep)) { free_engine(e); return rc; }
    }
    if (e->rate) {
        nvx::PathReport rep;
        const int rc = nvx::resample_path_create(e->rate, e->S, cfg->max_block, &e->rp, &rep);
        if (path_report(e, rc, rep)) { free_engine(e); return rc; }
    }
    e->assembler.resize(e->channels);
    if (int rc = reset_state(e)) { free_engine(e); return rc; }
    e->worker = std::thread(worker_main, e);
    *out = e;
    return 0;
}

void nvx_engine_destroy(nvx_engine* e) { free_engine(e); }

int nvx_engine_reset(nvx_engine* e) {
    if (!e) return fail(NVX_ERR_ARG, "null engine");
    CU_TRY(cudaSetDevice(e->cfg.device));
    const int rc_sync = sync_engine(e);
    if (rc_sync == NVX_ERR_CUDA) return rc_sync;   // a dead context cannot be reset; an event-buffer overflow of the old run can
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->ready.clear();
    }
    return reset_state(e);
}

int nvx_engine_reset_streams(nvx_engine* e, const int* streams, int count) {
    if (!e || count < 0 || (count && !streams)) return fail(NVX_ERR_ARG, "bad argument");
    for (int i = 0; i < count; ++i)
        if (streams[i] < 0 || streams[i] >= e->S) return fail(NVX_ERR_ARG, "stream %d outside 0..%d", streams[i], e->S - 1);
    for (int i = 0; i < count; ++i) {
        uint8_t& f = e->pend_flags[(size_t)streams[i]];
        if (!(f & nvx_engine::kListed)) e->pend_streams.push_back(streams[i]);
        f = (uint8_t)((f | nvx_engine::kListed) & ~nvx_engine::kLoad);     // a reset after a load wins
    }
    return 0;
}

int nvx_engine_retune_stream(nvx_engine* e, int stream, const double* nco_hz, const int* freq_tag) {
    if (!e || !nco_hz || stream < 0 || stream >= e->S) return fail(NVX_ERR_ARG, "bad argument");
    if (e->nco_host.empty()) return fail(NVX_ERR_ARG, "engine was created without nco_hz: its reference-table channels cannot be retuned");
    std::vector<nvx::NcoChan> rows((size_t)e->C);
    for (int c = 0; c < e->C; ++c)
        if (!nco_entry(nco_hz[c], &rows[(size_t)c]))
            return fail(NVX_ERR_ARG, "nco_hz[%d] = %g is not a multiple of 0.5 Hz inside +-31.5 kHz", c, nco_hz[c]);
    std::copy(rows.begin(), rows.end(), e->nco_host.begin() + (size_t)stream * e->C);
    if (freq_tag) e->pend_tags.push_back({stream, std::vector<int>(freq_tag, freq_tag + e->C)});
    e->pend_flags[(size_t)stream] |= nvx_engine::kNewNco;
    return nvx_engine_reset_streams(e, &stream, 1);
}

int nvx_engine_save_streams(nvx_engine* e, const int* streams, int count, void* out, size_t cap, size_t* size) {
    if (!e || !size || count < 0 || (count && !streams)) return fail(NVX_ERR_ARG, "bad argument");
    if (int rc = check_stream_list(e, streams, count)) return rc;
    if (int rc = sync_engine(e)) return rc;
    if (e->blocks == 0) return fail(NVX_ERR_ARG, "nothing has been pushed since create or reset: there is no stream state to save");
    for (int i = 0; i < count; ++i)
        if (e->pend_flags[(size_t)streams[i]])
            return fail(NVX_ERR_ARG, "stream %d has a reset, retune or load pending: push a block before saving it", streams[i]);
    ResetArgs a = state_args(e);
    std::vector<uint8_t> msg;           // the message part: tags and the assembler's partial lines and messages
    for (int i = 0; i < count; ++i)
        for (int c = 0; c < e->C; ++c) {
            const size_t ch = (size_t)streams[i] * e->C + c;
            const ChannelText& t = e->assembler.channel((int)ch);
            const int32_t v[5] = {e->stream_tag.empty() ? e->cfg.freq_tag[c & 1] : e->stream_tag[ch], t.in_message ? 1 : 0,
                                  (int32_t)t.line.size(), (int32_t)t.text.size(), (int32_t)t.bbbb.size()};
            const uint8_t* pv = reinterpret_cast<const uint8_t*>(v);
            msg.insert(msg.end(), pv, pv + sizeof v);
            for (const std::string* str : {&t.line, &t.text, &t.bbbb}) msg.insert(msg.end(), str->begin(), str->end());
        }
    const size_t rec_bytes = (size_t)count * a.lay.words * sizeof(uint32_t);
    *size = sizeof(StateHeader) + rec_bytes + msg.size();
    if (!out) return 0;
    if (cap < *size) return fail(NVX_ERR_OVERFLOW, "the saved state needs %zu bytes, the buffer holds %zu", *size, cap);
    uint8_t* o = static_cast<uint8_t*>(out);
    if (count) {
        if (int rc = reset_buffers(e)) return rc;
        if (int rc = records_buffer(e, rec_bytes)) return rc;
        CU_TRY(cudaMemcpyAsync(e->d_reset_list, streams, (size_t)count * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        a.streams = e->d_reset_list;
        a.rec = e->d_records;
        save_streams_kernel<<<(unsigned)count, 256, 0, e->stream>>>(a);
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaMemcpyAsync(o + sizeof(StateHeader), e->d_records, rec_bytes, cudaMemcpyDeviceToHost, e->stream));
        CU_TRY(cudaStreamSynchronize(e->stream));
    }
    StateHeader h = {};
    h.magic = kStateMagic;
    h.version = kStateVersion;
    h.bytes = *size;
    h.position = in_position(e);
    for (int k = 0; k < 3; ++k) h.words[k] = a.rows.words[k];
    h.taps = e->lp ? nvx::long_path_taps_hash(e->lp) : nvx::cascade_path_taps_hash(e->cp);
    if (e->rp) h.taps = nvx::hash_bytes(&h.taps, sizeof h.taps, nvx::resample_path_taps_hash(e->rp));
    h.rate = e->rate;
    h.rec_words = a.lay.words;
    h.count = count;
    h.n_channels = e->C;
    h.fmt = e->fmt;
    h.path = e->path;
    h.gen_nco = e->d_nco_ch != nullptr;
    memcpy(o, &h, sizeof h);
    if (!msg.empty()) memcpy(o + sizeof h + rec_bytes, msg.data(), msg.size());
    h.checksum = state_checksum(o, *size);
    memcpy(o + kChecksumAt, &h.checksum, sizeof h.checksum);
    return 0;
}

int nvx_engine_load_streams(nvx_engine* e, const int* streams, int count, const void* state, size_t size) {
    using namespace nvx;
    if (!e || count < 0 || (count && !streams)) return fail(NVX_ERR_ARG, "bad argument");
    StateHeader h;
    std::vector<std::vector<ChannelText>> text;
    std::vector<std::vector<int>> tags;
    if (int rc = parse_state(state, size, &h, &text, &tags)) return rc;
    if (h.count != count) return fail(NVX_ERR_ARG, "the saved state holds %d streams, %d were listed", h.count, count);
    if (int rc = check_stream_list(e, streams, count)) return rc;
    const bool gen = e->d_nco_ch != nullptr;
    if (h.rate != e->rate)
        return fail(NVX_ERR_ARG, "the state was saved on an engine fed at %d S/s, this engine is fed at %d S/s", h.rate ? h.rate : NVX_FS_HZ,
                    e->rate ? e->rate : NVX_FS_HZ);
    if (h.path != e->path) return fail(NVX_ERR_ARG, "the state was saved on the %s, this engine runs the %s", path_name(h.path), path_name(e->path));
    uint64_t taps = e->lp ? long_path_taps_hash(e->lp) : cascade_path_taps_hash(e->cp);
    if (e->rp) taps = hash_bytes(&taps, sizeof taps, resample_path_taps_hash(e->rp));
    if (h.taps != taps) return fail(NVX_ERR_ARG, "the state was saved with another tap set");
    if (h.n_channels != e->C) return fail(NVX_ERR_ARG, "the state has %d channels per stream, this engine %d", h.n_channels, e->C);
    if ((h.gen_nco != 0) != gen)
        return fail(NVX_ERR_ARG, "the state was saved %s, this engine runs %s", h.gen_nco ? "with per-stream NCO offsets" : "on the reference NCO table",
                    gen ? "per-stream NCO offsets" : "the reference NCO table");
    if (e->fmt >= 0 && e->fmt != h.fmt) return fail(NVX_ERR_ARG, "the state holds sample format %d, this engine takes format %d", h.fmt, e->fmt);
    // an engine that has pushed nothing since create or reset adopts the saved position; any other must be on the same grid
    const bool adopt = e->blocks == 0 && !e->adopted;
    const long long here = adopt ? h.position : in_position(e);
    if ((here - h.position) % in_grid(e))
        return fail(NVX_ERR_ARG, "the state was saved after input sample %lld, this engine is at %lld: the two must agree modulo %lld (567 x 280 at 252 kS/s)",
                    (long long)h.position, here, in_grid(e));
    CU_TRY(cudaSetDevice(e->cfg.device));
    if (e->cp) {      // a fresh engine's tails take the saved format now (it would fill them with its silence at the first push)
        PathReport rep;
        const int rc = cascade_path_prepare(e->cp, e->rp ? SampleFmt::F32 : (SampleFmt)h.fmt, e->stream, &rep);
        if (path_report(e, rc, rep)) return rc;
    }
    const CarriedRows rows = e->lp ? long_path_carried(e->lp) : cascade_path_carried(e->cp);
    for (int k = 0; k < 3; ++k)
        if (rows.words[k] != h.words[k])
            return fail(NVX_ERR_ARG, "the state carries %lld words of FIR stage %d per stream, this engine %lld", (long long)h.words[k], k + 1, rows.words[k]);

    // accepted: nothing below fails
    if (adopt) {      // its other streams start as streams reset at the saved position
        e->sb_abs = h.position / e->down * e->up / kSuper;
        e->adopted = true;
        for (int s = 0; s < e->S; ++s) nvx_engine_reset_streams(e, &s, 1);
    }
    e->fmt = h.fmt;
    const StateLayout lay = state_layout(h.words, e->C, gen, resampler_words(h.rate));
    const long long d_out = (here - h.position) / e->down * e->up;             // the same distance at 252 kS/s
    const long long d_sb = d_out / kSuper;                                      // epochs: 900 Hz samples
    const long long d_tick = (d_out / NVX_D1) % kNcoDen;                        // NCO phases: 63 kHz ticks
    const uint32_t* recs = reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(state) + sizeof(StateHeader));
    for (int k = 0; k < count; ++k) {
        const int s = streams[k];
        const size_t r0 = e->pend_records.size();
        e->pend_records.resize(r0 + (size_t)lay.words);
        memcpy(&e->pend_records[r0], recs + (size_t)k * lay.words, (size_t)lay.words * sizeof(uint32_t));
        for (int c = 0; c < e->C; ++c) {
            uint32_t* r = &e->pend_records[r0 + (size_t)(lay.chan + c * lay.ch_words)];
            long long epoch;
            memcpy(&epoch, r + kRecEpoch, sizeof epoch);
            epoch += d_sb;
            memcpy(r + kRecEpoch, &epoch, sizeof epoch);
            if (gen) {     // the row keeps its phase: (tick + d_tick) num + phase0' = tick num + phase0
                NcoChan n;
                memcpy(&n, r + kRecNco, sizeof n);
                n.phase0 = (int)(((n.phase0 - (d_tick + kNcoDen) % kNcoDen * n.num) % kNcoDen + kNcoDen) % kNcoDen);
                memcpy(r + kRecNco, &n, sizeof n);
                e->nco_host[(size_t)s * e->C + c] = {n.num, 0, n.step};     // a later reset or nvx_engine_reset keeps the offsets
            }
        }
        uint8_t& f = e->pend_flags[(size_t)s];
        if (!(f & nvx_engine::kListed)) e->pend_streams.push_back(s);
        f |= nvx_engine::kListed | nvx_engine::kLoad | (gen ? nvx_engine::kNewNco : 0);
        e->pend_rec[(size_t)s] = (int)e->pend_text.size();
        e->pend_text.push_back(std::move(text[(size_t)k]));
        e->pend_tags.push_back({s, std::move(tags[(size_t)k])});
    }
    return 0;
}

int nvx_stream_state_info(const void* state, size_t size, int* count, long long* position, int* n_channels, int* sample_format) {
    StateHeader h;
    std::vector<std::vector<ChannelText>> text;
    std::vector<std::vector<int>> tags;
    if (int rc = parse_state(state, size, &h, &text, &tags)) return rc;
    if (count) *count = h.count;
    if (position) *position = h.position;
    if (n_channels) *n_channels = h.n_channels;
    if (sample_format) *sample_format = h.fmt;
    return 0;
}

int nvx_engine_push_device_f32(nvx_engine* e, const void* d_iq, long long n) {
    if (!e || !d_iq) return fail(NVX_ERR_ARG, "null argument");
    CU_TRY(cudaSetDevice(e->cfg.device));
    return process_block(e, d_iq, n, nvx::SampleFmt::F32);
}

int nvx_engine_push_device_s16(nvx_engine* e, const void* d_iq, long long n) {
    if (!e || !d_iq) return fail(NVX_ERR_ARG, "null argument");
    CU_TRY(cudaSetDevice(e->cfg.device));
    return process_block(e, d_iq, n, nvx::SampleFmt::S16);
}

int nvx_engine_push_device_u8(nvx_engine* e, const void* d_iq, long long n) {
    if (!e || !d_iq) return fail(NVX_ERR_ARG, "null argument");
    CU_TRY(cudaSetDevice(e->cfg.device));
    return process_block(e, d_iq, n, nvx::SampleFmt::U8);
}

int nvx_engine_push_host_f32(nvx_engine* e, const float* iq, long long n) {
    if (!e || !iq) return fail(NVX_ERR_ARG, "null argument");
    return push_host(e, iq, n, nvx::SampleFmt::F32);
}

int nvx_engine_push_host_s16(nvx_engine* e, const int16_t* iq, long long n) {
    if (!e || !iq) return fail(NVX_ERR_ARG, "null argument");
    return push_host(e, iq, n, nvx::SampleFmt::S16);
}

int nvx_engine_push_host_u8(nvx_engine* e, const uint8_t* iq, long long n) {
    if (!e || !iq) return fail(NVX_ERR_ARG, "null argument");
    return push_host(e, iq, n, nvx::SampleFmt::U8);
}

int nvx_engine_wait_ingest(nvx_engine* e) {
    if (!e) return fail(NVX_ERR_ARG, "null engine");
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaStreamSynchronize(e->stream_copy));
    return 0;
}

long long nvx_engine_host_pushes(nvx_engine* e) { return e ? e->host_pushes : NVX_ERR_ARG; }

int nvx_engine_wait_ingest_of(nvx_engine* e, long long push_index) {
    if (!e || push_index < 0) return fail(NVX_ERR_ARG, "bad argument");
    if (push_index >= e->host_pushes) return fail(NVX_ERR_ARG, "host push %lld has not been made yet (%lld so far)", push_index, e->host_pushes);
    // copies run in order on one stream into two alternating staging slots: pushes older than the last two are necessarily over
    if (push_index < e->host_pushes - 2) return 0;
    CU_TRY(cudaSetDevice(e->cfg.device));
    CU_TRY(cudaEventSynchronize(e->copy_done[push_index % 2]));
    return 0;
}

int nvx_engine_sync(nvx_engine* e) {
    if (!e) return fail(NVX_ERR_ARG, "null engine");
    return sync_engine(e);
}

int nvx_engine_poll_messages(nvx_engine* e, const nvx_message** msgs, size_t* count) {
    if (!e || !msgs || !count) return fail(NVX_ERR_ARG, "null argument");
    int rc = sync_engine(e);
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->handed.swap(e->ready);
        e->ready.clear();
    }
    e->view.clear();
    for (const auto& m : e->handed) {
        nvx_message v;
        v.stream = m.stream; v.freq = m.freq;
        memset(v.bbbb, 0, sizeof v.bbbb);
        strncpy(v.bbbb, m.bbbb.c_str(), sizeof v.bbbb - 1);
        v.text = m.text.c_str(); v.text_len = m.text.size();
        e->view.push_back(v);
    }
    *msgs = e->view.data();
    *count = e->view.size();
    return rc;
}

int nvx_engine_try_poll_messages(nvx_engine* e, const nvx_message** msgs, size_t* count) {
    if (!e || !msgs || !count) return fail(NVX_ERR_ARG, "null argument");
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->handed.swap(e->ready);
        e->ready.clear();
    }
    e->view.clear();
    for (const auto& m : e->handed) {
        nvx_message v;
        v.stream = m.stream; v.freq = m.freq;
        memset(v.bbbb, 0, sizeof v.bbbb);
        strncpy(v.bbbb, m.bbbb.c_str(), sizeof v.bbbb - 1);
        v.text = m.text.c_str(); v.text_len = m.text.size();
        e->view.push_back(v);
    }
    *msgs = e->view.data();
    *count = e->view.size();
    return 0;
}

int nvx_engine_set_message_callback(nvx_engine* e, nvx_message_cb cb, void* user) {
    if (!e) return fail(NVX_ERR_ARG, "null engine");
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->cb = cb; e->cb_user = user;
    }
    deliver_callbacks(e);                  // anything queued before the callback existed goes out first, in order
    return 0;
}

int nvx_engine_read_y3(nvx_engine* e, float* out, size_t cap_floats, size_t* n_per_channel) {
    if (!e || !out || !n_per_channel) return fail(NVX_ERR_ARG, "null argument");
    int rc = sync_engine(e);
    const size_t P = (size_t)e->last_P;
    *n_per_channel = P;
    if (cap_floats < (size_t)e->channels * P * 2) return fail(NVX_ERR_ARG, "y3 buffer too small");
    if (P)
        CU_TRY(cudaMemcpy2D(out, P * sizeof(float2), e->y3buf[e->last_buf] + nvx::kHistY, (size_t)(nvx::kHistY + e->P_max) * sizeof(float2),
                            P * sizeof(float2), (size_t)e->channels, cudaMemcpyDeviceToHost));
    return rc;
}

int nvx_engine_read_bits(nvx_engine* e, int stream, int ch, char* bits, float* sums, size_t cap, size_t* count) {
    if (!e || !bits || !count || stream < 0 || stream >= e->S || ch < 0 || ch >= e->C) return fail(NVX_ERR_ARG, "bad argument");
    if (!e->d_bits) return fail(NVX_ERR_ARG, "engine was created without keep_bits");
    int rc = sync_engine(e);
    const int c = stream * e->C + ch;
    int n = 0;
    CU_TRY(cudaMemcpy(&n, e->d_bit_count + c, sizeof n, cudaMemcpyDeviceToHost));
    if (n > e->bit_cap) { n = e->bit_cap; rc = fail(NVX_ERR_OVERFLOW, "bit buffer overflow"); }
    if ((size_t)n > cap) return fail(NVX_ERR_ARG, "bit buffer too small (%d needed)", n);
    *count = (size_t)n;
    if (n) {
        CU_TRY(cudaMemcpy(bits, e->d_bits + (size_t)c * e->bit_cap, (size_t)n, cudaMemcpyDeviceToHost));
        if (sums) CU_TRY(cudaMemcpy(sums, e->d_disc + (size_t)c * e->bit_cap * 4, (size_t)n * 4 * sizeof(float), cudaMemcpyDeviceToHost));
    }
    return rc;
}

int nvx_engine_read_events(nvx_engine* e, int stream, int ch, char* ev, size_t cap, size_t* count) {
    if (!e || !ev || !count || stream < 0 || stream >= e->S || ch < 0 || ch >= e->C) return fail(NVX_ERR_ARG, "bad argument");
    int rc = sync_engine(e);
    const int c = stream * e->C + ch;
    int n = e->h_ev_count[e->last_buf][c];
    if (n > e->ev_cap) n = e->ev_cap;
    if ((size_t)n > cap) return fail(NVX_ERR_ARG, "event buffer too small (%d needed)", n);
    memcpy(ev, e->h_events[e->last_buf] + (size_t)c * e->ev_cap, (size_t)n);
    *count = (size_t)n;
    return rc;
}

int nvx_engine_enable_timing(nvx_engine* e, int on) {
    if (!e) return fail(NVX_ERR_ARG, "null engine");
    int rc = sync_engine(e);
    e->timing = on < 0 ? 0 : on;
    return rc;
}

int nvx_engine_get_stats(nvx_engine* e, nvx_stats* out, int reset) {
    if (!e || !out) return fail(NVX_ERR_ARG, "null argument");
    int rc = sync_engine(e);
    *out = e->stats;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        out->messages = e->delivered;
    }
    if (reset) { e->stats = nvx_stats{}; e->cascade_spans_ms.clear(); }
    return rc;
}

int nvx_engine_get_cascade_spans(nvx_engine* e, float* ms, size_t cap, size_t* count) {
    if (!e || !count || (!ms && cap)) return fail(NVX_ERR_ARG, "null argument");
    int rc = sync_engine(e);
    *count = e->cascade_spans_ms.size();
    const size_t n = *count < cap ? *count : cap;
    if (n) memcpy(ms, e->cascade_spans_ms.data(), n * sizeof(float));
    return rc;
}

int nvx_engine_fence(nvx_engine* e) {
    if (!e) return fail(NVX_ERR_ARG, "null engine");
    CU_TRY(cudaSetDevice(e->cfg.device));
    if (e->blocks > 0) CU_TRY(cudaStreamWaitEvent(e->stream, e->demod_done[e->last_buf], 0));
    return 0;
}

int nvx_pinned_alloc(size_t bytes, int write_combined, void** out) {
    if (!out || !bytes) return fail(NVX_ERR_ARG, "bad argument");
    void* p = nullptr;
    const cudaError_t err = cudaHostAlloc(&p, bytes, cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0));
    if (err != cudaSuccess) return fail(err == cudaErrorMemoryAllocation ? NVX_ERR_NOMEM : NVX_ERR_CUDA, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(err));
    *out = p;
    return 0;
}

int nvx_pinned_free(void* p) {
    if (!p) return 0;
    CU_TRY(cudaFreeHost(p));
    return 0;
}

void* nvx_engine_stream(nvx_engine* e) { return e ? (void*)e->stream : nullptr; }

int nvx_host_assemble(const unsigned char* events, size_t n, int stream, int freq, nvx_message_cb cb, void* user) {
    if ((!events && n) || !cb) return fail(NVX_ERR_ARG, "null argument");
    nvx::MessageAssembler as;
    as.resize(1);
    std::vector<nvx::AssembledMessage> out;
    as.feed(0, stream, freq, events, n, &out);
    for (auto& m : out) {
        std::string b = m.bbbb, t = m.text;
        cb(user, m.stream, &b[0], &t[0], m.freq);
    }
    return (int)out.size();
}

int nvx_debug_long_tc_band(int decimation, const double* h, int n_taps, int* geometry, float* g_hi, float* g_lo, size_t capacity) {
    nvx::TcBand b;
    if (!h || n_taps < 1 || !geometry || !nvx::long_tc_band(decimation, n_taps, h, &b))
        return fail(NVX_ERR_ARG, "no tensor-core band matrix for decimation %d, %d taps", decimation, n_taps);
    geometry[0] = b.T; geometry[1] = b.N; geometry[2] = b.chunks; geometry[3] = b.J; geometry[4] = b.copies;
    if (g_hi && g_lo) {
        if (capacity < b.gh.size()) return fail(NVX_ERR_ARG, "the band matrix needs %zu floats per part", b.gh.size());
        memcpy(g_hi, b.gh.data(), b.gh.size() * sizeof(float));
        memcpy(g_lo, b.gl.data(), b.gl.size() * sizeof(float));
    }
    return (int)b.gh.size();
}

}  // extern "C"

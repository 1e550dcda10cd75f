// engine.cu -- the C ABI of include/navtex_b200.h: per-GPU engine that owns the carried state of
// S independent streams and queues, per pushed block, the fused FIR cascade (or the three long-tap
// stage kernels), the tail carry, the demod / bit-sync / state-machine kernels and the event
// download; host side it runs the message assembler on a worker thread.
//
// Call contract it replaces: capt_sched.c:552-555 (init_dsp), :612 (init_fir2_wrapper) and the
// consumer loop :484-528 that calls sample_in_1 once per IQ pair.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/navtex_b200.h"
#include "demod.cuh"
#include "fir_cascade.cuh"
#include "fir_long.cuh"
#include "message_assembler.h"

namespace nvx {
int cascade_box_elems(SampleFmt f);
int cascade_tap_class(int n1, int n2, int n3);
int cascade_warm_super(int tap_class);
void cascade_fill_taps(int tap_class, const double* h1, int n1, const double* h2, int n2, const double* h3, int n3, CascadeTaps* out);
cudaError_t cascade_launch(const CascadeArgs& a, const CascadeTaps& taps, int tap_class, bool custom_taps, SampleFmt f, int n_ch, cudaStream_t stream);
int cascade_target_warps(int device, int reserved_sms, SampleFmt f, int tap_class, bool heavy);
}  // namespace nvx

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

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;

int load_encode() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
        return fail(NVX_ERR_CUDA, "cuTensorMapEncodeTiled not available: %s", cudaGetErrorString(e));
    g_encode = (EncodeTiledFn)fn;
    return 0;
}

// 32-bit-element view of a stream-major sample array: [rows][2 * cols] floats for float2 samples, [rows][cols] words for
// short2 samples (one word = one I,Q pair), [rows][cols / 2] words for 8-bit pairs (one word = two pairs; cols is a multiple
// of 280); box = one ring stage x 32 rows
int encode_rows(CUtensorMap* map, const void* base, long long cols, long long rows, nvx::SampleFmt f) {
    if (int rc = load_encode()) return rc;
    const long long row_bytes = cols * nvx::sample_bytes(f);
    cuuint64_t dims[2] = {(cuuint64_t)(row_bytes / 4), (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
    cuuint32_t box[2] = {(cuuint32_t)nvx::cascade_box_elems(f), 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(map, f == nvx::SampleFmt::F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NVX_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) cols=%lld rows=%lld", (int)r, cols, rows);
    return 0;
}

// new_tail[s] = last `halo` samples of (old_tail[s] ++ x[s][0..n)); kPer samples (16 bytes) per thread
template <typename Sample>
__global__ void tail_carry_kernel(const Sample* __restrict__ old_tail, const Sample* __restrict__ x, Sample* __restrict__ new_tail,
                                  int streams, long long n, int halo) {
    constexpr int kPer = 16 / (int)sizeof(Sample);
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long per = halo / kPer;
    if (idx >= per * streams) return;
    const int s = (int)(idx / per);
    const long long k = (idx % per) * kPer;
    const long long p = n - halo + k;                                            // n and halo are multiples of 280
    const int4* src = p >= 0 ? reinterpret_cast<const int4*>(x + (size_t)s * n + p)
                             : reinterpret_cast<const int4*>(old_tail + (size_t)s * halo + (halo + p));
    *reinterpret_cast<int4*>(new_tail + (size_t)s * halo + k) = *src;
}

// long-tap path, 8-bit input: out = (u - 128) as short2, 8 samples (16 bytes in, 32 out) per thread; count = S n, a multiple of 280
__global__ void widen_u8_kernel(const uchar2* __restrict__ in, short2* __restrict__ out, long long count) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i >= count) return;
    const int4 v = *reinterpret_cast<const int4*>(in + i);
    const unsigned w[4] = {(unsigned)v.x, (unsigned)v.y, (unsigned)v.z, (unsigned)v.w};
    int o[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {       // bytes I0 Q0 I1 Q1 of a word -> two short2 words
        o[2 * k] = (int)(((w[k] & 0xFFu) - 128u) & 0xFFFFu) | (int)(((((w[k] >> 8) & 0xFFu) - 128u) & 0xFFFFu) << 16);
        o[2 * k + 1] = (int)((((w[k] >> 16) & 0xFFu) - 128u) & 0xFFFFu) | (int)((((w[k] >> 24) - 128u) & 0xFFFFu) << 16);
    }
    int4* dst = reinterpret_cast<int4*>(out + i);
    dst[0] = make_int4(o[0], o[1], o[2], o[3]);
    dst[1] = make_int4(o[4], o[5], o[6], o[7]);
}

}  // namespace

constexpr int kBuf = 3;   // blocks in flight: cascade of block i+1/i+2 overlaps demod + event download of block i

struct nvx_engine {
    nvx_config cfg;
    int S = 0, P_max = 0, channels = 0;
    int C = 2;                            // channels per stream (nvx_config.n_channels)
    cudaStream_t stream = nullptr;        // cascade, tail carry, ingest copies / conversion
    cudaStream_t stream_demod = nullptr;  // demod kernels + event download, one block behind
    float2* y3buf[kBuf] = {};
    uint8_t* pickbuf[kBuf] = {};
    cudaEvent_t casc_done[kBuf] = {}, demod_done[kBuf] = {}, ff_done[kBuf] = {};
    long long blocks = 0;
    int last_buf = 0;
    int tap_class = 0;                    // fused-kernel tap-length class (fir_cascade.cuh), -1 = long-tap path
    int halo = 1960;                      // carried input samples per stream: 280 x the class's warm-up superblocks
    // carried input tail, ping-pong, in the sample format being pushed: [S][halo] float2, short2 or 8-bit pairs
    void* tail[nvx::kSampleFmts][2] = {};                            // [format][ping-pong]
    CUtensorMap map_tail[nvx::kSampleFmts][2];
    int tail_cur = 0;
    int fmt = -1;                         // -1 = nothing pushed since create/reset, else the nvx::SampleFmt of the pushes
    short2* u8_wide = nullptr;            // long-tap path, 8-bit input: [S][max_block] short2 (u - 128), allocated on first use
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
    bool custom_taps = false;
    nvx::CascadeTaps taps;                // this engine's filter constants: passed in the parameter block of every cascade launch
    nvx::NcoParam* d_nco = nullptr;       // per-stream NCO parameters, two-channel layout of the long-tap path, else null
    nvx::NcoChan* d_nco_ch = nullptr;     // per (stream, channel) NCO parameters of the fused kernel's general-NCO variants, else null
    // long-tap path (tap counts other than 37 / 47 / 71): per-stage kernels, intermediates and histories in HBM
    bool long_taps = false;
    nvx::LongStage lst[3];
    float2* lhist[3][2] = {};             // [stage][ping-pong]: [rows][H]
    float2 *y1buf = nullptr, *y2buf = nullptr;
    int lcur = 0;
    nvx::LongTcStage* ltc[2] = {nullptr, nullptr};   // tensor-core variants of stages 1 and 2 (null: CUDA-core kernel)
    bool mix_on_load = false;             // long path, reference NCO table, streaming tensor-core stage 2: stage 1 writes ONE un-mixed row per stream
    bool ltc_wanted[2] = {false, false};  // the tensor-core kernel was asked for (NVX_LONG_TC mask) for that stage
    nvx::LongStageTaps ltaps[3];          // this engine's long-path taps: passed in the parameter block of every stage launch
    std::vector<int> stream_tag;          // optional [S][2] message tags
    bool serial = false;                  // NVX_PIPELINE=serial: the next cascade waits for this block's whole demod
    bool ff_on_main = true;               // feed-forward demod kernels follow the cascade on the main stream
    int target_warps[nvx::kSampleFmts] = {576, 576, 576};   // resident cascade warps per sample format
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
    for (int f = 0; f < nvx::kSampleFmts; ++f) { cudaFree(e->tail[f][0]); cudaFree(e->tail[f][1]); }
    cudaFree(e->u8_wide);
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
    cudaFree(e->d_nco);
    cudaFree(e->d_nco_ch);
    for (int k = 0; k < 3; ++k) { cudaFree(e->lhist[k][0]); cudaFree(e->lhist[k][1]); }
    cudaFree(e->y1buf); cudaFree(e->y2buf);
    nvx::long_tc_free(e->ltc[0]); nvx::long_tc_free(e->ltc[1]);
    for (int k = 0; k < kBuf; ++k) {
        cudaFree(e->y3buf[k]); cudaFree(e->d_events[k]); cudaFree(e->d_ev_count[k]);
        cudaFreeHost(e->h_events[k]); cudaFreeHost(e->h_ev_count[k]);
        if (e->casc_done[k]) cudaEventDestroy(e->casc_done[k]);
        if (e->demod_done[k]) cudaEventDestroy(e->demod_done[k]);
        if (e->ff_done[k]) cudaEventDestroy(e->ff_done[k]);
        cudaFree(e->pickbuf[k]);
    }
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->stream_demod) cudaStreamDestroy(e->stream_demod);
    delete e;
    return 0;
}

int reset_state(nvx_engine* e) {
    // the warm-up before the first block sees silence: the value 0, which is the byte 128 in 8-bit offset binary
    for (int f = 0; f < nvx::kSampleFmts; ++f)
        for (int k = 0; k < 2; ++k)
            CU_TRY(cudaMemsetAsync(e->tail[f][k], (nvx::SampleFmt)f == nvx::SampleFmt::U8 ? 128 : 0,
                                   (size_t)e->S * e->halo * nvx::sample_bytes((nvx::SampleFmt)f), e->stream));
    e->fmt = -1;
    if (e->long_taps)
        for (int k = 0; k < 3; ++k)
            for (int q = 0; q < 2; ++q)
                CU_TRY(cudaMemsetAsync(e->lhist[k][q], 0, (size_t)(k == 0 ? e->S : e->channels) * e->lst[k].H * sizeof(float2), e->stream));
    e->lcur = 0;
    for (int k = 0; k < kBuf; ++k) {
        e->db.y3 = e->y3buf[k];
        e->db.picks = e->pickbuf[k];
        e->db.corr = e->corrbuf[k & 1];
        CU_TRY(nvx::demod_init_state(e->db, e->channels, e->stream));
    }
    CU_TRY(cudaStreamSynchronize(e->stream));
    e->tail_cur = 0;
    e->sb_abs = 0;
    e->last_P = 0;
    e->blocks = 0;
    e->last_buf = 0;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->queued = e->drained = 0;
        e->worker_rc = 0;
    }
    e->assembler.reset();
    e->ready.clear();
    return 0;
}

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

// a long-tap stage that was meant for the tensor cores ran on the CUDA-core kernel: counted, and explained in nvx_last_error()
void note_tc_fallback(nvx_engine* e, int stage, const char* why) {
    e->stats.long_tc_fallbacks++;
    fail(0, "note: long-tap stage %d ran on the CUDA-core kernel: %s", stage, why);
}

int process_block(nvx_engine* e, const void* d_x, long long n, nvx::SampleFmt fmt) {
    using namespace nvx;
    if (e->fmt >= 0 && e->fmt != (int)fmt)
        return fail(NVX_ERR_ARG, "sample format changed between pushes (float, int16 and 8-bit blocks cannot be mixed without a reset)");
    e->fmt = (int)fmt;
    if (n <= 0 || n % kSuper != 0) return fail(NVX_ERR_ARG, "block length %lld is not a positive multiple of %d", n, kSuper);
    if (n > e->cfg.max_block) return fail(NVX_ERR_ARG, "block length %lld exceeds max_block %lld", n, e->cfg.max_block);
    if (((uintptr_t)d_x & 15) != 0) return fail(NVX_ERR_ARG, "device block is not 16-byte aligned");
    const int b = (int)(e->blocks % kBuf);
    wait_drained(e, e->blocks - kBuf + 1);          // block (blocks - kBuf) used these buffers: long finished, normally
    if (e->timing && e->ev_used > 4000) {            // bound the event pool in long timed runs
        CU_TRY(cudaStreamSynchronize(e->stream));
        CU_TRY(cudaStreamSynchronize(e->stream_demod));
        collect_spans(e);
    }
    CascadeArgs ca;
    if (int rc = encode_rows(&ca.map_x, d_x, n, e->S, fmt)) return rc;
    ca.map_tail = e->map_tail[(int)fmt][e->tail_cur];
    const int n_super = (int)(n / kSuper);
    const int groups = (e->S + 31) / 32;
    // time segments: enough warps to fill the machine once, but keep the 7-superblock warm-up small
    int segs = e->target_warps[(int)fmt] / groups;            // never more warps than are resident at once (no second wave)
    const int min_seg = 63;
    if (segs > n_super / min_seg) segs = n_super / min_seg;
    if (segs < 1) segs = 1;
    const int seg_super = (n_super + segs - 1) / segs;
    segs = (n_super + seg_super - 1) / seg_super;
    ca.y3 = e->y3buf[b];
    ca.n = n;
    ca.streams = e->S;
    ca.segs = segs;
    ca.seg_super = seg_super;
    ca.n_super = n_super;
    ca.sb_phase = (int)(e->sb_abs % kNcoPeriod);
    ca.sb_abs = e->sb_abs;
    ca.nco = e->d_nco_ch;
    ca.y3_pitch = nvx::kHistY + e->P_max;
    ca.y3_off = nvx::kHistY;
    ca.ch_total = e->C;
    ca.ch0 = 0;

    // this block's FIR output goes into the y3 buffer block (blocks - 3) used -- long drained, see wait_drained above -- whose
    // last samples the feed-forward kernels of block (blocks - 2) read as their history: when those run on the demod stream
    // nothing else orders them before this launch
    if (!e->ff_on_main && e->blocks >= 2) CU_TRY(cudaStreamWaitEvent(e->stream, e->ff_done[(b + 1) % kBuf], 0));
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
    if (e->long_taps) {
        // 8-bit input: widened to the int16 values u - 128 in front of the unchanged int16 long path (same results bit for bit)
        if (fmt == SampleFmt::U8) {
            if (!e->u8_wide) CU_TRY(cudaMalloc(&e->u8_wide, (size_t)e->S * e->cfg.max_block * sizeof(short2)));
            const long long count = (long long)e->S * n;
            widen_u8_kernel<<<(unsigned)((count / 8 + 255) / 256), 256, 0, e->stream>>>(static_cast<const uchar2*>(d_x), e->u8_wide, count);
            CU_TRY(cudaGetLastError());
            e->stats.aux_launches++;
            d_x = e->u8_wide;
        }
        const int s16 = fmt != SampleFmt::F32;
        const int cur = e->lcur, nx = cur ^ 1;
        const long long p1 = e->cfg.max_block / NVX_D1, p2 = e->cfg.max_block / (NVX_D1 * NVX_D2);
        LongArgs la = {};
        la.in = d_x; la.hist = e->lhist[0][cur]; la.out = e->y1buf; la.n_in = n; la.out_pitch = p1; la.out_off = 0;
        la.rows_in = e->S; la.stage = 0; la.s16 = s16; la.k_abs = e->sb_abs * (kSuper / NVX_D1); la.nco = e->d_nco;
        la.plain = e->mix_on_load;                 // stage 2 mixes while it loads: one un-mixed 63 kHz row per stream
        cudaError_t tc = e->ltc[0] ? long_tc_launch(e->ltc[0], la, e->lst[0], n, e->stream) : cudaErrorNotSupported;
        if (tc == cudaErrorNotSupported) {         // 252 k -> 63 k, mixed: one row per channel
            if (e->ltc_wanted[0]) note_tc_fallback(e, 1, e->ltc[0] ? "this block cannot be described to the TMA unit (pointer or pitch not 16-byte aligned)"
                                                                    : "the tap set does not fit the tensor-core tile");
            tc = long_launch(la, e->lst[0], e->ltaps[0], n, e->stream);
        }
        CU_TRY(tc);
        CU_TRY(long_carry(e->lhist[0][cur], d_x, n, e->lhist[0][nx], e->S, e->lst[0].H, n, s16, e->stream));
        la.in = e->y1buf; la.hist = e->lhist[1][cur]; la.out = e->y2buf; la.n_in = n / NVX_D1; la.out_pitch = p2;
        la.rows_in = e->channels; la.stage = 1; la.s16 = 0; la.nco = nullptr;
        la.plain = 0; la.mix_in = e->mix_on_load;   // (k_abs: the block's first stage-2 INPUT sample sits at that 63 kHz tick)
        tc = e->ltc[1] ? long_tc_launch(e->ltc[1], la, e->lst[1], p1, e->stream) : cudaErrorNotSupported;
        if (tc == cudaErrorNotSupported && e->mix_on_load)      // (cannot happen: y1buf and its pitch are 16-byte aligned)
            return fail(NVX_ERR_CUDA, "long-tap stage 2: the tensor-core kernel refused the block and the stage-1 output is un-mixed");
        if (tc == cudaErrorNotSupported) {         // 63 k -> 9 k
            if (e->ltc_wanted[1]) note_tc_fallback(e, 2, e->ltc[1] ? "this block cannot be described to the TMA unit (pointer or pitch not 16-byte aligned)"
                                                                    : "the tap set does not fit the tensor-core tile");
            tc = long_launch(la, e->lst[1], e->ltaps[1], p1, e->stream);
        }
        CU_TRY(tc);
        CU_TRY(long_carry(e->lhist[1][cur], e->y1buf, p1, e->lhist[1][nx], e->mix_on_load ? e->S : e->channels, e->lst[1].H, n / NVX_D1, 0, e->stream));
        la.mix_in = 0;
        la.in = e->y2buf; la.hist = e->lhist[2][cur]; la.out = e->y3buf[b]; la.n_in = n / (NVX_D1 * NVX_D2);
        la.out_pitch = ca.y3_pitch; la.out_off = ca.y3_off; la.stage = 2;
        CU_TRY(long_launch(la, e->lst[2], e->ltaps[2], p2, e->stream));                // 9 k -> 900
        CU_TRY(long_carry(e->lhist[2][cur], e->y2buf, p2, e->lhist[2][nx], e->channels, e->lst[2].H, la.n_in, 0, e->stream));
        e->lcur = nx;
        e->stats.aux_launches += 5;
    } else {
        // up to four channels share one pass over the input (stage 1 computed once for all of them); five to eight take two
        for (int c0 = 0; c0 < e->C;) {
            const int left = e->C - c0;
            const int n_ch = left <= nvx::kMaxFusedCh ? left : (left + 1) / 2;      // 5 = 3 + 2, 6 = 3 + 3, 7 = 4 + 3, 8 = 4 + 4
            ca.ch0 = c0;
            CU_TRY(cascade_launch(ca, e->taps, e->tap_class, e->custom_taps, fmt, n_ch, e->stream));
            if (c0) e->stats.aux_launches++;
            c0 += n_ch;
        }
    }
    if (e->timing) CU_TRY(cudaEventRecord(t1, e->stream));

    const int nxt = e->tail_cur ^ 1;
    if (!e->long_taps) {
        const long long work = (long long)e->S * (e->halo / (16 / sample_bytes(fmt)));
        const unsigned grid = (unsigned)((work + 255) / 256);
        const void* old_tail = e->tail[(int)fmt][e->tail_cur];
        void* new_tail = e->tail[(int)fmt][nxt];
        if (fmt == SampleFmt::U8)
            tail_carry_kernel<uchar2><<<grid, 256, 0, e->stream>>>(static_cast<const uchar2*>(old_tail), static_cast<const uchar2*>(d_x),
                                                                   static_cast<uchar2*>(new_tail), e->S, n, e->halo);
        else if (fmt == SampleFmt::S16)
            tail_carry_kernel<short2><<<grid, 256, 0, e->stream>>>(static_cast<const short2*>(old_tail), static_cast<const short2*>(d_x),
                                                                   static_cast<short2*>(new_tail), e->S, n, e->halo);
        else
            tail_carry_kernel<float2><<<grid, 256, 0, e->stream>>>(static_cast<const float2*>(old_tail), static_cast<const float2*>(d_x),
                                                                   static_cast<float2*>(new_tail), e->S, n, e->halo);
        CU_TRY(cudaGetLastError());
    }
    e->tail_cur = nxt;

    CU_TRY(cudaEventRecord(e->casc_done[b], e->stream));

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
    // the cascade (one warp per SM sub-partition, little latency slack) they cost it about what they take alone, so by default
    // they follow it on the main stream and only the sequential symbol-clock / state-machine kernels (64 warps on the SMs the
    // cascade grid leaves free) overlap the next block's cascade.  NVX_PIPELINE=overlap moves them to the demod stream too.
    cudaStream_t s_ff = e->ff_on_main ? e->stream : e->stream_demod;
    if (!e->ff_on_main) CU_TRY(cudaStreamWaitEvent(e->stream_demod, e->casc_done[b], 0));
    CU_TRY(demod_launch(da, s_ff, e->stream_demod, e->ff_done[b], e->timing > 1 ? marks : nullptr));
    CU_TRY(cudaMemcpyAsync(e->h_ev_count[b], e->d_ev_count[b], sizeof(int) * e->channels, cudaMemcpyDeviceToHost, e->stream_demod));
    CU_TRY(cudaMemcpyAsync(e->h_events[b], e->d_events[b], (size_t)e->channels * e->ev_cap, cudaMemcpyDeviceToHost, e->stream_demod));
    CU_TRY(cudaEventRecord(e->demod_done[b], e->stream_demod));
    if (e->serial) CU_TRY(cudaStreamWaitEvent(e->stream, e->demod_done[b], 0));
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
    e->stats.aux_launches++;
    e->stats.samples += n * e->S;
    return 0;
}

// H2D on the copy stream into staging slot k % 2, then the block's kernels on the main stream
int push_host(nvx_engine* e, const void* iq, long long n, nvx::SampleFmt fmt) {
    if (n <= 0 || n % nvx::kSuper != 0 || n > e->cfg.max_block) return fail(NVX_ERR_ARG, "bad block length %lld", n);
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

}  // namespace

extern "C" {

const char* nvx_last_error(void) { return g_err; }

void nvx_default_config(nvx_config* cfg) {
    memset(cfg, 0, sizeof *cfg);
    cfg->n_streams = 1;
    cfg->max_block = 252000;
    cfg->freq_tag[0] = 518;   // nav_sched.C:10-11
    cfg->freq_tag[1] = 490;
}

int nvx_engine_create(const nvx_config* cfg, nvx_engine** out) {
    if (!cfg || !out) return fail(NVX_ERR_ARG, "null argument");
    if (cfg->n_streams <= 0 || cfg->max_block <= 0 || cfg->max_block % nvx::kSuper != 0)
        return fail(NVX_ERR_ARG, "n_streams must be > 0 and max_block a positive multiple of %d", nvx::kSuper);
    if (cfg->n_streams > 32767)       // channel rows index the y dimension of the demod grids (65535 max)
        return fail(NVX_ERR_ARG, "n_streams %d exceeds 32767 per engine: shard the streams over more engines", cfg->n_streams);
    if (cfg->max_block / nvx::kSuper > (1 << 24))
        return fail(NVX_ERR_ARG, "max_block %lld is too long (at most %d samples per push)", cfg->max_block, nvx::kSuper << 24);
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
    if (cfg->stream_freq_tag) e->stream_tag.assign(cfg->stream_freq_tag, cfg->stream_freq_tag + (size_t)C * (size_t)cfg->n_streams);
    std::vector<nvx::NcoParam> nco;
    std::vector<nvx::NcoChan> nco_ch;
    if (cfg->nco_hz) {
        nco_ch.resize((size_t)cfg->n_streams * C);
        if (C == 2) nco.resize((size_t)cfg->n_streams);
        for (int k = 0; k < C * cfg->n_streams; ++k) {
            const double f = cfg->nco_hz[k], twice = 2.0 * f;
            if (!(fabs(f) < 31500.0) || twice != nearbyint(twice)) {
                delete e;
                return fail(NVX_ERR_ARG, "nco_hz[%d] = %g is not a multiple of 0.5 Hz inside +-31.5 kHz", k, f);
            }
            long long num = (long long)twice % nvx::kNcoDen;
            if (num < 0) num += nvx::kNcoDen;
            // same expression as fir2cpp.C:105-106 for table entry 1, rounded once to float
            const float2 step = make_float2((float)cos((2 * M_PI * 1 * f) / 63000), (float)-sin((2 * M_PI * 1 * f) / 63000));
            nco_ch[(size_t)k].num = (int)num;
            nco_ch[(size_t)k].step = step;
            if (C == 2) { nco[(size_t)k / 2].num[k & 1] = (int)num; nco[(size_t)k / 2].step[k & 1] = step; }
        }
    }
    e->S = cfg->n_streams;
    e->channels = C * e->S;
    e->P_max = (int)(cfg->max_block / nvx::kSuper);
    e->custom_taps = cfg->h1 || cfg->h2 || cfg->h3;
    // tap counts: reference lengths unless given; sets up to 37/47/71 and up to 61/75/111 run through the fused kernel
    // (zero-padded to the class), longer ones through the long-tap path
    const int n[3] = {cfg->n1 ? cfg->n1 : NVX_T1, cfg->n2 ? cfg->n2 : NVX_T2, cfg->n3 ? cfg->n3 : NVX_T3};
    if ((cfg->n1 && !cfg->h1) || (cfg->n2 && !cfg->h2) || (cfg->n3 && !cfg->h3)) {
        delete e;
        return fail(NVX_ERR_ARG, "a tap count was given without its tap array");
    }
    for (int k = 0; k < 3; ++k)
        if (n[k] < 1 || n[k] > nvx::kLongMaxTaps) { delete e; return fail(NVX_ERR_ARG, "tap count %d outside 1..%d", n[k], nvx::kLongMaxTaps); }
    e->tap_class = nvx::cascade_tap_class(n[0], n[1], n[2]);
    e->long_taps = e->tap_class < 0;
    if (C != 2 && e->tap_class != 0) {
        delete e;
        return fail(NVX_ERR_ARG, "n_channels = %d is served by the fused kernel's reference tap class only (up to %d / %d / %d taps)", C, NVX_T1, NVX_T2, NVX_T3);
    }
    e->halo = nvx::kSuper * nvx::cascade_warm_super(e->tap_class);
    if (e->long_taps) {
        const int D[3] = {NVX_D1, NVX_D2, NVX_D3};
        for (int k = 0; k < 3; ++k) e->lst[k] = nvx::long_stage(D[k], n[k]);
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
        // tuning knob NVX_PIPELINE: default "main" = the feed-forward demod kernels follow the cascade on the main stream and only
        // the sequential kernels run beside the next cascade; "overlap" = the whole demod chain of block i runs on the demod
        // stream beside the cascade of block i + 1 (A/B on one box, 30 steps each, twice: 3.81 / 3.84 ms per step against 3.86 /
        // 3.81 -- no difference beyond the noise, while the cascade itself slows from 3.48 to 3.71 ms); "serial" = the next
        // cascade waits for the whole demod
        const char* mode = getenv("NVX_PIPELINE");
        e->serial = mode && !strcmp(mode, "serial");
        e->ff_on_main = !(mode && !strcmp(mode, "overlap"));
    }
    for (int k = 0; k < kBuf; ++k) {
        CREATE_TRY(cudaEventCreateWithFlags(&e->casc_done[k], cudaEventDisableTiming));
        CREATE_TRY(cudaEventCreateWithFlags(&e->demod_done[k], cudaEventDisableTiming));
        CREATE_TRY(cudaEventCreateWithFlags(&e->ff_done[k], cudaEventDisableTiming));
    }
    for (int f = 0; f < nvx::kSampleFmts; ++f)
        for (int k = 0; k < 2; ++k)
            CREATE_TRY(cudaMalloc(&e->tail[f][k], (size_t)e->S * e->halo * nvx::sample_bytes((nvx::SampleFmt)f)));
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
    if (e->long_taps) {
        static const double d1[NVX_T1] = {NVX_H1_VALUES}, d2[NVX_T2] = {NVX_H2_VALUES}, d3[NVX_T3] = {NVX_H3_VALUES};
        const double* hh[3] = {cfg->h1 ? cfg->h1 : d1, cfg->h2 ? cfg->h2 : d2, cfg->h3 ? cfg->h3 : d3};
        for (int k = 0; k < 3; ++k)
            if (!nvx::long_fill_taps(e->lst[k], hh[k], &e->ltaps[k])) { free_engine(e); return fail(NVX_ERR_ARG, "stage %d: %d taps do not fit the long-tap kernel", k + 1, e->lst[k].T); }
        for (int k = 0; k < 3; ++k)
            for (int q = 0; q < 2; ++q)
                CREATE_TRY(cudaMalloc(&e->lhist[k][q], (size_t)(k == 0 ? e->S : e->channels) * e->lst[k].H * sizeof(float2)));
        // stages 1 and 2 on the tensor cores where the band matrix fits (fir_long_tc.cu); NVX_LONG_TC is a mask (bit 0: stage
        // 1, bit 1: stage 2; 0 keeps the CUDA-core kernels, whose output is bit-identical across blockings)
        const int tc_mask = getenv("NVX_LONG_TC") ? atoi(getenv("NVX_LONG_TC")) : 3;
        e->ltc_wanted[0] = (tc_mask & 1) != 0;
        e->ltc_wanted[1] = (tc_mask & 2) != 0;
        if (tc_mask & 1) e->ltc[0] = nvx::long_tc_prepare(NVX_D1, e->lst[0].T, hh[0], e->stream);
        if (tc_mask & 2) e->ltc[1] = nvx::long_tc_prepare(NVX_D2, e->lst[1].T, hh[1], e->stream);
        // a stage the tensor-core kernel does not serve (e.g. stage 2 beyond 959 taps) runs on the CUDA-core kernel: same
        // results to rounding, about half the speed.  Not an error, but never silent: nvx_last_error() says so after create
        // and nvx_stats.long_tc_fallbacks counts every such stage launch.
        for (int k = 0; k < 2; ++k)
            if (e->ltc_wanted[k] && !e->ltc[k])
                fail(0, "note: long-tap stage %d (%d taps) is not served by the tensor-core kernel and runs on the CUDA-core kernel", k + 1, e->lst[k].T);
        CREATE_TRY(cudaMalloc(&e->y1buf, (size_t)e->channels * (cfg->max_block / NVX_D1) * sizeof(float2)));
        // "mix on load": with the reference offsets (no per-stream NCO) and stage 2 on the streaming tensor-core kernel, stage 1
        // writes one un-mixed 63 kHz row per stream and stage 2 rotates while it converts: y1 crosses HBM once per stream instead
        // of once per channel, in both directions.  NVX_LONG_MIX=stage1 keeps the rotation in the stage-1 epilogue (A/B measurements).
        e->mix_on_load = nco.empty() && nvx::long_tc_mixes_on_load(e->ltc[1]) && (cfg->max_block / NVX_D1) % 2 == 0 &&
                         !(getenv("NVX_LONG_MIX") && !strcmp(getenv("NVX_LONG_MIX"), "stage1"));
        CREATE_TRY(cudaMalloc(&e->y2buf, (size_t)e->channels * (cfg->max_block / (NVX_D1 * NVX_D2)) * sizeof(float2)));
    } else {
        nvx::cascade_fill_taps(e->tap_class, cfg->h1, n[0], cfg->h2, n[1], cfg->h3, n[2], &e->taps);
    }
    if (!nco.empty()) {
        CREATE_TRY(cudaMalloc(&e->d_nco, nco.size() * sizeof(nvx::NcoParam)));
        CREATE_TRY(cudaMemcpy(e->d_nco, nco.data(), nco.size() * sizeof(nvx::NcoParam), cudaMemcpyHostToDevice));
    }
    if (!nco_ch.empty()) {
        CREATE_TRY(cudaMalloc(&e->d_nco_ch, nco_ch.size() * sizeof(nvx::NcoChan)));
        CREATE_TRY(cudaMemcpy(e->d_nco_ch, nco_ch.data(), nco_ch.size() * sizeof(nvx::NcoChan), cudaMemcpyHostToDevice));
    }
#undef CREATE_TRY
    for (int f = 0; f < nvx::kSampleFmts; ++f)
        for (int k = 0; k < 2; ++k)
            if (int rc = encode_rows(&e->map_tail[f][k], e->tail[f][k], e->halo, e->S, (nvx::SampleFmt)f)) { free_engine(e); return rc; }
    for (int f = 0; f < nvx::kSampleFmts; ++f)
        e->target_warps[f] = nvx::cascade_target_warps(cfg->device, nvx::demod_reserved_sms(e->channels), (nvx::SampleFmt)f, e->tap_class, C > 2);
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

int nvx_engine_push_device_f32(nvx_engine* e, const void* d_iq, long long n) {
    if (!e || !d_iq) return fail(NVX_ERR_ARG, "null argument");
    CU_TRY(cudaSetDevice(e->cfg.device));
    return process_block(e, d_iq, n, nvx::SampleFmt::F32);
}

int nvx_engine_push_device_s16(nvx_engine* e, const void* d_iq, long long n) {
    if (!e || !d_iq) return fail(NVX_ERR_ARG, "null argument");
    if (((uintptr_t)d_iq & 15) != 0) return fail(NVX_ERR_ARG, "device block is not 16-byte aligned");
    CU_TRY(cudaSetDevice(e->cfg.device));
    return process_block(e, d_iq, n, nvx::SampleFmt::S16);
}

int nvx_engine_push_device_u8(nvx_engine* e, const void* d_iq, long long n) {
    if (!e || !d_iq) return fail(NVX_ERR_ARG, "null argument");
    if (((uintptr_t)d_iq & 15) != 0) return fail(NVX_ERR_ARG, "device block is not 16-byte aligned");
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

/* navtex_b200.h -- C ABI of the batched, B200-native NAVTEX receive chain.
 *
 * One engine = one GPU = S independent 252 kS/s zero-IF IQ streams, each carrying the 518 kHz
 * (+14 kHz) and 490 kHz (-14 kHz) channels.  It replaces, for all S streams at once, the
 * reference's per-sample push chain (all citations relative to receiver/ in bartelvdh/Navtex):
 *
 *   init_fir_filter1()            fir1cpp.h:2   -> nvx_engine_create / nvx_engine_reset
 *   init_fir2_wrapper()           nav_sched.h:1 -> nvx_engine_create / nvx_engine_reset
 *   sample_in_1(double I,double Q) fir1cpp.h:3, called per sample at capt_sched.c:511
 *                                               -> nvx_engine_push_* (a whole [S][n] block per call)
 *   fir_filter3::sample_in        fir3cpp.h:100 -> stage taps via nvx_engine_read_y3
 *   decoder::sample_in            decoder.h:85  -> bit taps via nvx_engine_read_bits
 *   byte_state_machine::receive_bit nav_b_sm.h:127 -> events, nvx_engine_read_events
 *   add_message(bbbb,message,freq) nav_b_sm.C:4, message_store.h:7
 *                                               -> nvx_engine_poll_messages / nvx_message_cb
 *
 * The legacy symbol names themselves are provided by libnavtex_compat.so (navtex_compat.h), a
 * one-stream adapter over this ABI, so a host written against the reference headers relinks
 * unchanged.  There is no CPU fallback: every entry point needs a CUDA device and fails with
 * NVX_ERR_CUDA otherwise.
 *
 * Conventions: plain pointers and sizes only; the caller owns every buffer it passes; the engine
 * owns all device state; one caller thread per engine; return 0 on success, negative nvx_status
 * otherwise (nvx_last_error() gives a message).  Sample blocks are stream-major:
 * element (s, k) of a block of n samples per stream is at base[(s * n + k) * 2 + {0 = I, 1 = Q}].
 * n must be a multiple of NVX_BLOCK_ALIGN (280 = 4*7*10, one 900 Hz output); on an engine fed at another rate
 * (nvx_config.input_rate_hz) n counts input samples and must be a multiple of that rate's alignment.
 */
#ifndef NAVTEX_B200_H
#define NAVTEX_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define NVX_BLOCK_ALIGN 280
#define NVX_FS_HZ 252000

typedef enum {
    NVX_OK = 0,
    NVX_ERR_ARG = -1,      /* bad argument (null, misaligned n, wrong engine state) */
    NVX_ERR_CUDA = -2,     /* CUDA runtime/driver failure, including "no device" */
    NVX_ERR_NOMEM = -3,
    NVX_ERR_OVERFLOW = -4  /* a per-block output buffer was too small; results up to that point are valid */
} nvx_status;

typedef struct nvx_engine nvx_engine;

typedef struct {
    int device;                 /* CUDA device ordinal */
    int n_streams;              /* S */
    long long max_block;        /* largest n a push will carry (samples per stream) */
    int freq_tag[2];            /* tags handed to add_message for channel 0 (+14 kHz) / 1 (-14 kHz); 0,0 = 518,490 */
    /* optional replacement tap sets (NULL = reference taps), lengths n1 / n2 / n3 (0 = the reference length 37 / 47 / 71).
     * Sets of up to 37 / 47 / 71 taps and "medium" sets of up to 61 / 75 / 111 taps run through the fused cascade kernel
     * (zero-padded to the class; the medium class is where it turns from HBM-bound to FP32-bound); longer ones (up to
     * 1024 per stage, e.g. the 255-tap stress designs) take the long-tap path: one register-tiled FIR kernel per stage,
     * intermediates in HBM.
     * Tap sets are per engine (they travel in the kernel parameter block of every launch): engines with different
     * filters can be alive on one device at the same time.
     * Tap order: h[0] weighs the newest sample: y[k] = sum_i h[i] x[D (k + 1) - 1 - i] (D = 4, 7, 10 for h1, h2, h3; the
     * order matters for asymmetric filters, e.g. minimum-phase designs) */
    const double *h1, *h2, *h3;
    int keep_bits;              /* record 'B'/'Y' decisions and discriminator sums for nvx_engine_read_bits */
    int first_stream_id;        /* global id of stream 0 (multi-GPU sharding; only used to label messages) */
    /* optional per-stream channel offsets [n_streams][2] in Hz (multiples of 0.5 Hz, |f| < 31500): channel c of stream
     * s is mixed down by nco_hz[2 s + c].  NULL = the reference's +14000 / -14000 with its 9-entry table
     * (fir2cpp.C:12-14, :104-107); a non-NULL array selects the general-NCO kernel variant for every stream */
    const double *nco_hz;
    /* optional per-stream tags [n_streams][2] handed to add_message instead of freq_tag (e.g. 4209 for 4209.5 kHz) */
    const int *stream_freq_tag;
    /* tap counts of h1 / h2 / h3; 0 = reference length.  Up to 61 / 75 / 111 taps the fused kernel serves them (results do not
     * depend on how the samples are cut into blocks); longer sets, up to 1024 per stage, run one kernel per stage, stages 1
     * and 2 on the tensor cores (3xTF32, equal to the FP64 oracle to 1e-5; different blockings agree to rounding, not bit
     * for bit -- set NVX_LONG_TC=0 in the environment for the CUDA-core kernels if block-invariant bits matter) */
    int n1, n2, n3;
    /* channels per capture sharing stage 1 (SURVEY.md 8f.4): 0 = 2 (the reference's pair, nav_sched.C:10-16).  1 .. 8 channels
     * need nco_hz [n_streams][n_channels] (and stream_freq_tag [n_streams][n_channels] if the messages are to be told apart);
     * up to four are computed in ONE pass over the input -- stage 1 runs once, the mix and stages 2 / 3 once per channel, all
     * in registers -- five to eight in two passes.  Reference tap class only (up to 37 / 47 / 71 taps).  Results are laid out
     * [stream][channel] everywhere (y3, bits, events, messages). */
    int n_channels;
    /* the radio's sample rate in S/s: 0 or NVX_FS_HZ (252000) = the engine's own rate, pushed as it is (no extra launch, no
     * extra allocation).  Any other multiple of 100 in [96000, 3200000] is resampled on the device to 252 kS/s in front of
     * the FIR path (nvx_resampler_info gives the filter); other rates return NVX_ERR_ARG.  On such an engine every count of
     * samples is in input samples at this rate: max_block, the n of every push, nvx_stats.samples and every stream position
     * (E in nvx_engine_reset_streams, the saved states' positions).  n and max_block must be multiples of the rate's
     * alignment r / gcd(r, 900), the smallest input count that makes a whole number of 280-sample blocks at 252 kS/s, and
     * the 158760-sample restart grid of nvx_engine_reset_streams is 0.63 r input samples. */
    int input_rate_hz;
} nvx_config;

typedef struct {
    int stream;                 /* global stream id */
    int freq;                   /* 518 / 490 */
    char bbbb[8];               /* B1B2B3B4, NUL terminated */
    const char *text;           /* message text, NUL terminated; valid until the next poll/destroy */
    size_t text_len;
} nvx_message;

/* add_message-shaped callback (nav_b_sm.C:4): strings are borrowed for the duration of the call */
typedef int (*nvx_message_cb)(void *user, int stream, char *bbbb, char *message, int freq);

void nvx_default_config(nvx_config *cfg);

/* host-only (no GPU): the rational resampler an engine with nvx_config.input_rate_hz = input_rate_hz runs.  252000 / r = up /
 * down in lowest terms; output k at 252 kS/s (absolute, since create) is y[k] = sum_j h[p + j up] x[t - j], t = floor(k down /
 * up), p = k down - t up, input samples before the first being 0 -- scipy.signal.upfirdn(h, x, up, down)[k].  h: a
 * Kaiser-windowed sinc at up x r, pass band +-31.5 kHz (ripple <= 0.01 dB), stop band from min(r, 252000) - 31.5 kHz at
 * least 80 dB down, each of its up polyphase branches summing to 1 within 1e-3; the kernel uses the float rounding of these
 * FP64 taps and accumulates in FP32.  *block_align = r / gcd(r, 900), the multiple every push length and max_block must be.
 * h may be NULL (or cap too small: NVX_ERR_OVERFLOW) to query *n_taps; any other output may be NULL.  252000 gives 1 / 1 / 280
 * and one unit tap; an unsupported rate returns NVX_ERR_ARG. */
int nvx_resampler_info(int input_rate_hz, int *up, int *down, long long *block_align, double *h, size_t cap, size_t *n_taps);
const char *nvx_last_error(void);

int nvx_engine_create(const nvx_config *cfg, nvx_engine **out);
void nvx_engine_destroy(nvx_engine *e);
/* back to the state right after create (zero FIR history, decoder INIT, phasing search) */
int nvx_engine_reset(nvx_engine *e);

/* ---- per-stream lifecycle: one radio reconnects or is retuned while the others keep decoding ----------------------------
 * streams[0..count): local indices 0..S-1 (duplicates are fine).  Each listed stream restarts as if the engine had just been
 * created for it: zero FIR history, decoder INIT, phasing search, its partly received line and message dropped without being
 * delivered (like nvx_engine_reset).  Takes effect at the start of the next push; every other stream is untouched.  Messages
 * the stream completed in blocks pushed before still arrive.  Callable before the first push (harmless).
 *
 * The demod grids are absolute and shared by all channels (evaluation samples at 900 Hz index = 6 mod 9, the 567-sample
 * correlation ring, the order of its FP64 sums), so a reset stream restarts on that grid: a reset that takes effect at input
 * sample E (the total pushed per stream so far) restarts the stream at E0 = E - (E mod 158760), 158760 = 567 x 280.  From
 * then on the stream is, bit for bit, what a freshly created engine produces when fed Z = E - E0 zero samples followed by the
 * stream's input from E on: y3, bits, discriminator sums, events and messages (the Z < 158760 zeros make no decision: the
 * ring is not full before 574 samples at 900 Hz).  On the long-tap path with its tensor-core stages "bit for bit" reads
 * "to rounding", as for any change of blocking there (see n1 / n2 / n3).  The extra work -- one small kernel -- is only
 * queued on pushes that carry a reset; it waits for the previous block's demod. */
int nvx_engine_reset_streams(nvx_engine *e, const int *streams, int count);
/* new channel offsets nco_hz[n_channels] (same rules as nvx_config.nco_hz) and optionally new tags freq_tag[n_channels]
 * (NULL = keep the current ones) for one stream.  Implies nvx_engine_reset_streams for that stream, whose rule also places
 * the new NCO's phase origin: phase 0 at E0.  Messages of blocks pushed before carry the old tags.  Returns NVX_ERR_ARG if
 * the engine was created without nco_hz (reference-table engines cannot be retuned). */
int nvx_engine_retune_stream(nvx_engine *e, int stream, const double *nco_hz, const int *freq_tag);

/* ---- saved stream state: a stream survives an engine restart or moves to another engine ---------------------------------
 * A stream saved after input sample E (the total pushed per stream) and loaded into an engine created with the same
 * configuration continues bit for bit as the uninterrupted stream would: y3, bits, discriminator sums, events and messages.  A
 * bulletin in flight at the save completes on the destination, its full text delivered once, labelled with the destination's
 * stream id and the tags the state carries.  This holds on both FIR paths, the long-tap tensor-core stages included, as long as
 * the blocks pushed after the load are those the source would have pushed.
 *
 * Position rule: the demod grids and the reference NCO table are absolute, so a load is accepted only where the destination's
 * pushed total E' satisfies E' = E (mod 158760), 158760 = 567 x 280 as in nvx_engine_reset_streams.  An engine that has pushed
 * nothing since create or reset adopts E instead (this is what a restart uses): its streams that are not loaded start as
 * streams reset at E, and a second load before its first push must agree with the first modulo 158760.  Epochs move by E' - E
 * and general-NCO rows keep their phase.
 * Compatibility: the state records the FIR path (fused reference or medium tap class, or long-tap path), the tap values as
 * the kernels read them, what the path carries per stream, n_channels, reference table or per-stream NCO offsets, and the sample
 * format.  A load into an engine that differs in any of these, or whose pushes already fixed another sample format, returns
 * NVX_ERR_ARG and changes nothing; so does a state whose magic number, version or checksum is wrong (a truncated or altered
 * state is never half-applied).  The bytes are in the host's byte order.
 *
 * Loading a stream into one engine while another engine still runs it delivers its bulletins twice: reset or detach the source.
 * Like every call, a load belongs to the engine's one caller thread; a capture poller (nvx_capture_start) pushing on another
 * thread meanwhile is outside that contract: stop it first. */
/* State of streams[0..count) (each listed once) after the last pushed block (implies nvx_engine_sync), as one self-contained
 * byte string.  out = NULL or cap too small: *size receives the bytes needed, NVX_ERR_OVERFLOW if out was given.  Read-only:
 * the engine and the listed streams carry on untouched.  NVX_ERR_ARG if nothing was pushed since create or reset, or if a listed
 * stream has a reset, retune or load pending. */
int nvx_engine_save_streams(nvx_engine *e, const int *streams, int count, void *out, size_t cap, size_t *size);
/* Record k of the state goes to local stream streams[k] (count = the number of records in it; each stream listed once).  Takes
 * effect at the start of the next push, like nvx_engine_reset_streams; per stream, the last reset / retune / load called before
 * a push wins.  A load also gives the stream the saved channel offsets and tags, which a later reset or retune keeps unless it
 * replaces them.  Messages the stream completed in blocks pushed before the load still arrive under the old state. */
int nvx_engine_load_streams(nvx_engine *e, const int *streams, int count, const void *state, size_t size);
/* host-only (no GPU): validate a saved state and report its record count, input position E (samples per stream), channels per
 * stream and sample format (0 = float, 1 = int16, 2 = 8-bit); any output may be NULL */
int nvx_stream_state_info(const void *state, size_t size, int *count, long long *position, int *n_channels, int *sample_format);

/* ---- ingest: n samples for every stream.  Host variants copy H2D on a copy stream into one of two staging slots, so
 * the copy of block k+1 overlaps the kernels of block k.  A pageable buffer may be reused as soon as the call returns;
 * a pinned (cudaHostAlloc / cudaHostRegister) buffer is read asynchronously and must stay unchanged until
 * nvx_engine_wait_ingest() or nvx_engine_sync() returns.  One engine takes one sample format between resets. */
int nvx_engine_push_host_f32(nvx_engine *e, const float *iq, long long n);
int nvx_engine_push_host_s16(nvx_engine *e, const int16_t *iq, long long n);   /* SDRplay / WAV sample format */
/* RTL-SDR sample format (rtlsdr_read_async / rtl_tcp): unsigned 8-bit offset-binary I,Q bytes, block [S][n][2] stream-major.
 * Sample value = u - 128 exactly, a float in [-128, 127].  128 rather than the converter's mid-scale 127.5 keeps the values
 * integers: the same capture pushed as int16 (u - 128) gives bit-identical results.  The -0.5 LSB DC offset this leaves
 * sits at -+14 kHz after the mix, where the channel filter removes it. */
int nvx_engine_push_host_u8(nvx_engine *e, const uint8_t *iq, long long n);
int nvx_engine_wait_ingest(nvx_engine *e);                                      /* every host buffer pushed so far has been read */
long long nvx_engine_host_pushes(nvx_engine *e);                                /* host pushes made so far (the next one has this index) */
int nvx_engine_wait_ingest_of(nvx_engine *e, long long push_index);             /* the buffer of that host push (0-based) has been read */
/* device-resident float2 block [S][n], 16-byte aligned; processed in place, asynchronously on the
 * engine's stream (ordered after everything previously queued on it) */
int nvx_engine_push_device_f32(nvx_engine *e, const void *d_iq, long long n);
int nvx_engine_push_device_s16(nvx_engine *e, const void *d_iq, long long n);
int nvx_engine_push_device_u8(nvx_engine *e, const void *d_iq, long long n);    /* 8-bit I,Q bytes [S][n][2], 16-byte aligned */
/* wait for everything pushed so far and run the host-side message assembly */
int nvx_engine_sync(nvx_engine *e);

/* ---- results -------------------------------------------------------------------------------- */
/* messages completed since the previous poll (implies sync); pointers valid until the next poll */
int nvx_engine_poll_messages(nvx_engine *e, const nvx_message **msgs, size_t *count);
/* same without waiting: whatever the blocks already finished have completed (the pipeline keeps running) */
int nvx_engine_try_poll_messages(nvx_engine *e, const nvx_message **msgs, size_t *count);
/* alternatively deliver them through an add_message-shaped callback.  The callback runs on the engine's worker thread as
 * soon as the block that completed a message (NNNN line or abort, nav_b_sm.C:47-50, :82-88) has drained -- no sync or poll
 * needed, so a capture poller + nvx_store_sink see rows while the capture runs.  Calls are serialised (never two at a
 * time per engine); nvx_engine_sync returns after every callback of the blocks pushed so far has returned.  The
 * callback must not call back into the same engine.  Messages queued before the callback was installed are delivered
 * from this call; cb = NULL goes back to queueing for poll. */
int nvx_engine_set_message_callback(nvx_engine *e, nvx_message_cb cb, void *user);

/* taps of the LAST pushed block (imply sync).  y3: [S][n_channels][n/280] float pairs (I,Q) at 900 Hz */
int nvx_engine_read_y3(nvx_engine *e, float *out, size_t cap_floats, size_t *n_per_channel);
/* bits decided during the last block for (stream, ch): 'B'/'Y'; sums = 4 floats per bit (BR BI YR YI), may be NULL */
int nvx_engine_read_bits(nvx_engine *e, int stream, int ch, char *bits, float *sums, size_t cap, size_t *count);
/* character / '\n' (line complete) / 0x18 (abort) events of the last block for (stream, ch) */
int nvx_engine_read_events(nvx_engine *e, int stream, int ch, char *ev, size_t cap, size_t *count);

/* ---- measurement hooks (bench.py) --------------------------------------------------------- */
typedef struct {
    double cascade_ms;          /* sum of fused-FIR kernel time since the last call, CUDA events on the engine stream */
    double demod_ms;            /* same for the demod/bit-sync/FSM kernel */
    long long cascade_launches;
    long long demod_launches;
    long long aux_launches;     /* tail carry, second pass of five to eight channels, long-tap stages, 8-bit -> int16 widening (long-tap path),
                                 * per-stream resets, the resampler (engines with an input_rate_hz other than 252000; one launch per
                                 * block, outside the cascade_ms spans) */
    long long samples;          /* IQ samples (all streams) pushed, at the input rate */
    double demod_stage_ms[6];   /* split of demod_ms: angle/correlation, per-offset sums + arg max, history carry | symbol clock, bit decisions, SITOR-B state machine */
    long long long_tc_fallbacks;/* long-tap stage launches that were meant for the tensor-core kernel but ran on the CUDA-core one
                                 * (tap set outside its tile geometry, or a block the TMA unit cannot address); nvx_last_error() says why */
    long long messages;         /* messages completed (delivered to the callback or queued for poll) */
    double cascade_ms_min, cascade_ms_max;   /* fastest / slowest single launch of the fused-FIR kernel (or the long-path stage trio) */
    double resample_ms;         /* sum of the resampler kernel's time (engines with an input_rate_hz other than 252000), CUDA events
                                 * around its launch on the engine stream while timing is on; not part of cascade_ms */
} nvx_stats;
/* on: 0 = off, 1 = time the fused-FIR kernel (two event records per block) and the resampler (two more, where there is one),
 * 2 = also every demod stage */
int nvx_engine_enable_timing(nvx_engine *e, int on);
int nvx_engine_get_stats(nvx_engine *e, nvx_stats *out, int reset);
/* the per-launch times behind cascade_ms (milliseconds, in launch order, since the last get_stats(reset)); *count = how many
 * there are, at most cap are copied */
int nvx_engine_get_cascade_spans(nvx_engine *e, float *ms, size_t cap, size_t *count);
/* device-side fence, no host wait: whatever is queued on nvx_engine_stream() after this call runs after EVERY kernel and
 * copy of the blocks pushed so far (the demod / state-machine kernels and the event download run on a second stream) */
int nvx_engine_fence(nvx_engine *e);
/* page-locked host memory for the push_host_* calls (cudaHostAlloc, portable; write_combined != 0: write-combined pages, faster
 * for the device to read on some hosts, slow for the CPU to read back) */
int nvx_pinned_alloc(size_t bytes, int write_combined, void **out);
int nvx_pinned_free(void *p);
/* the CUDA stream everything is queued on (cudaStream_t as void*), for callers that produce input on the device */
void *nvx_engine_stream(nvx_engine *e);

/* host-only helper (no GPU needed): run the line / ZCZC / NNNN / abort assembly of nav_b_sm.C:44-97 over one
 * channel's event bytes; calls cb once per completed message and returns their number */
int nvx_host_assemble(const unsigned char *events, size_t n, int stream, int freq, nvx_message_cb cb, void *user);

/* host-only test hook (no GPU needed): the operand the tensor-core long-tap kernel (stage with the given decimation, 4 or 7)
 * builds from n_taps taps h.  geometry[5] = { taps after zero padding, outputs per tile N, K chunks per tile, band rows J per
 * copy, copies }; g_hi / g_lo (may be NULL to query the size) receive the TF32 high / low parts as [copies][J][32] floats.
 * Chunk c of a tile multiplies 32 window columns (D = 4: 32 samples; D = 7: 28 samples + 4 zero columns) with rows
 * [8 ((chunks - 1) / copies - c / copies), + N) of copy c % copies.  Returns the float count per part, or NVX_ERR_ARG when
 * the stage is not served by that kernel. */
int nvx_debug_long_tc_band(int decimation, const double *h, int n_taps, int *geometry, float *g_hi, float *g_lo, size_t capacity);

/* ---- SDRplay-format front end (host): replaces the ring buffer + 50 ms consumer loop of capt_sched.c:105-148, :484-528 --- */
typedef struct nvx_capture nvx_capture;
/* one ring of ring_samples int16 I,Q pairs per stream (>= 2 max_block); max_block <= the engine's */
int nvx_capture_create(nvx_engine *e, int n_streams, long long max_block, long long ring_samples, nvx_capture **out);
/* same for RTL-SDR radios: the rings hold 8-bit I,Q pairs and the pump pushes with nvx_engine_push_host_u8 */
int nvx_capture_create_u8(nvx_engine *e, int n_streams, long long max_block, long long ring_samples, nvx_capture **out);
void nvx_capture_destroy(nvx_capture *c);
/* producer (the radio callback of stream `stream`, capt_sched.c:105: separate xi[] / xq[] arrays); one producer thread per
 * stream.  NVX_ERR_OVERFLOW = the ring was full, the excess was dropped (and counted) instead of overwriting unread data */
int nvx_capture_write(nvx_capture *c, int stream, const short *xi, const short *xq, unsigned num_samples);
/* producer of an 8-bit capture: num_samples interleaved I,Q byte pairs, exactly as the rtlsdr_read_async callback hands them
 * over (len = 2 num_samples).  Writing int16 to an 8-bit capture or 8-bit pairs to an int16 capture returns NVX_ERR_ARG;
 * overflow as for nvx_capture_write */
int nvx_capture_write_u8(nvx_capture *c, int stream, const unsigned char *iq, unsigned num_samples);
/* consumer: push what every attached stream has in common (a multiple of the engine's alignment -- 280, or the input rate's,
 * see nvx_resampler_info -- <= max_block) as one block in the capture's format.  Rings and max_block count input samples; create
 * returns NVX_ERR_ARG unless max_block is a multiple of that alignment.
 * Returns samples per stream pushed, 0 if there was less than one aligned block, or a negative nvx_status */
long long nvx_capture_pump(nvx_capture *c);
/* or let a poller thread pump every poll_ms (<= 0: 50 ms, capt_sched.c:489); stop() drains what is left */
int nvx_capture_start(nvx_capture *c, int poll_ms);
int nvx_capture_stop(nvx_capture *c);
long long nvx_capture_dropped(nvx_capture *c, int stream);
/* a radio that stops delivering: a detached stream no longer holds the pump back.  Its rows of each pumped block are silence
 * (0 for int16, 0x80 for 8-bit), and writes to it return NVX_ERR_ARG (nothing is counted as dropped).  attach flushes its ring
 * and resets the stream in the engine (nvx_engine_reset_streams), ordered between two pumps: the radio's first samples after
 * attach start a fresh decoder.  Detaching a detached or attaching an attached stream does nothing.  The pump returns 0
 * while every stream is detached. */
int nvx_capture_detach(nvx_capture *c, int stream);
int nvx_capture_attach(nvx_capture *c, int stream);

/* ---- in-memory message store behind add_message (message_store.c:59-97): newest message per (stream, B1B2B3B4) -------- */
typedef struct nvx_store nvx_store;
nvx_store *nvx_store_create(void);
void nvx_store_destroy(nvx_store *s);
/* 0, or -1 like message_store.c:69-73 when the store is unusable; replaces an older message with the same bbbb */
int nvx_store_add(nvx_store *s, int stream, const char *bbbb, const char *message, int freq);
int nvx_store_add_at(nvx_store *s, int stream, const char *bbbb, const char *message, int freq, long long unix_time);
/* nvx_message_cb-shaped: nvx_engine_set_message_callback(e, nvx_store_sink, store) */
int nvx_store_sink(void *store, int stream, char *bbbb, char *message, int freq);
size_t nvx_store_count(nvx_store *s);
/* row k in insertion order; stamp = UTC "%Y-%m-%d %H:%M" (message_store.c:30); *text valid until the next add/purge */
int nvx_store_get(nvx_store *s, size_t k, int *stream, int *freq, char bbbb[8], char stamp[20], const char **text);
int nvx_store_purge(nvx_store *s, long long now_unix, long long max_age_s);   /* reference: 72 h, message_store.c:13 */
int nvx_store_dump_csv(nvx_store *s, const char *path);

/* ---- synthetic captures on the device (bench / tests): SITOR-B FSK + AWGN, int16-valued float2 - */
typedef struct {
    const uint8_t *bits;        /* host: concatenated per-stream bit strings (1 = 'Y'), 100 baud */
    const long long *bit_off;   /* host: [S+1] offsets into bits */
    const float *offset_hz;     /* host: [S] channel offset (+14000 / -14000) */
    const float *start_s;       /* host: [S] emission start time */
    const float *amplitude;     /* host: [S] */
    const float *noise_sigma;   /* host: [S] per-component AWGN sigma (0 = none) */
    unsigned long long seed;
} nvx_synth_desc;
/* fill d_iq ([S][n] float2, device) with samples [t0, t0+n) of every stream's capture */
int nvx_synth_fill_device(int device, const nvx_synth_desc *d, int n_streams, long long t0, long long n,
                          void *d_iq, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif

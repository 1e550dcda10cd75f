// demod.cuh -- buffers, per-channel persistent state and launch arguments of the demodulator /
// bit synchroniser / SITOR-B state machine kernels (demod.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nvx {

constexpr int kSpb = 9;                 // samples per bit at 900 Hz (decoder.h:21)
constexpr int kCorrLen = 63 * kSpb;     // 567 (decoder.h:23-24)
constexpr int kEvAbort = 0x18;          // event byte: message_abort() (nav_b_sm.C:44-52)

// Every per-sample array keeps a short history of the previous block in front of the new samples,
// so the feed-forward kernels are stateless: element for block-relative sample m lives at [hist + m].
constexpr int kHistY = 16;              // 900 Hz samples (angle needs 1, mask correlation 8 more, decisions look back 4)
constexpr int kHistC = 640;             // |mask correlation| values (the per-offset sum threads reach back up to 628)
constexpr int kPadC = 64;               // readable slack behind the new samples (a thread's running prefix may run 46 past the block)

enum { DS_INIT = 0, DS_WAIT = 1, DS_PENDING = 2 };   // decoder.h:16-19 (BIT_START / RECEIVING folded into PENDING)
enum { BY_WAIT = 1, BY_GOT_DX = 2, BY_GOT_RX = 3 };  // nav_b_sm.h:41-43

// What decoder.{h,C} keeps per channel and that is genuinely sequential: the slew-limited offset tracker and the
// symbol clock of the mark/space discriminator (decoder.C:73-137, :217-249), in event form.
struct ClockState {
    int last_pick;            // prev_offset (decoder.C:247), -1 = none
    // dstate INIT / WAIT (searching the sample whose tick equals offs, from `cur` on) / PENDING (bit triggered
    // at sample `pend`, decided 7 samples later); indices are relative to the start of the next block
    int dstate, offs, next_offs, cur, pend;
};

// SITOR-B state machine (nav_b_sm.h:92-116), arrays packed into words
struct FsmState {
    int match;                // phasing pattern bits matched (status)
    int byte_state, figures, nbits, shift;
    unsigned dx_ring;         // 3 bytes, slot k at bits [8k, 8k+8)
    int dx_at, dx_full;
    unsigned err_mask;        // bit k set = error_buffer[k] holds an invalid code
    int err_at, err_full, err_count;
    int eoe_count, prev_dx_alpha, holdoff, enabled;
};

// a channel's state at create: decoder::decoder (decoder.C:6-39) and byte_state_machine::init (nav_b_sm.C:16-42)
__host__ __device__ inline ClockState clock_state_init() {
    ClockState c = {};
    c.last_pick = -1;
    c.dstate = DS_INIT;
    return c;
}
__host__ __device__ inline FsmState fsm_state_init() {
    FsmState s = {};
    s.byte_state = BY_WAIT;
    return s;
}

struct DemodBuffers {
    float2* y3;               // [channels][kHistY + p_max]   (the cascade kernel writes at +kHistY); one per block in flight
    double* corr;             // [channels][kHistC + p_max + kPadC]   |mask correlation| per sample (two buffers, alternating per block)
    uint8_t* picks;           // [channels][pick pitch]  arg max offset of every evaluation sample of the block; one per block in flight
    int* bitpos;              // [channels][bit pitch]   first sample of the 5-sample window of every bit of the block
    uint8_t* bitval;          // [channels][bit pitch]   1 = 'Y', 0 = 'B'
    int* nbits;               // [channels]              bits decided in the block
    ClockState* clock;        // [channels]
    FsmState* fsm;            // [channels]
    // [channels] the channel's epoch: the 900 Hz sample its decoder (re)started at -- 0 from create and nvx_engine_reset, the
    // E0 of nvx_engine_reset_streams after that.  Warm-up conditions count from it; the sample grids stay absolute.
    long long* epoch;
    int p_max;
};

struct DemodArgs {
    DemodBuffers b;           // b.y3 / b.picks = the buffers of this block
    const float2* y3_prev;    // y3 buffer of the PREVIOUS block: its last kHistY samples are this block's history
    const double* corr_prev;  // corr buffer of the previous block, likewise (last kHistC values)
    int n_prev;               // 900 Hz samples per channel of the previous block (0 right after a reset: zero history)
    int n_new;                // new 900 Hz samples per channel in this block
    int channels;             // streams * 2
    long long seen;           // 900 Hz samples consumed before this block (same for every channel)
    // per-launch outputs
    uint8_t* events;          // [channels][ev_cap]: appended characters, '\n' = line complete, 0x18 = abort
    int* ev_count;            // [channels]
    int ev_cap;
    char* bits;               // optional [channels][bit_cap] 'B'/'Y' decisions (parity taps), may be null
    float* disc;              // optional [channels][bit_cap][4] BR BI YR YI at each decision, may be null
    int* bit_count;           // [channels] (required if bits != null)
    int bit_cap;
};

size_t demod_pick_pitch(int p_max);  // row pitch of DemodBuffers::picks in bytes
size_t demod_bit_pitch(int p_max);   // row pitch of DemodBuffers::bitpos / bitval in elements
// SMs the sequential kernels want for themselves (the cascade grid is sized to leave them free)
int demod_reserved_sms(int channels);
// Queues the feed-forward kernels (angle/correlation incl. the history hand-over, per-offset sums + arg max) on s_ff and the
// sequential symbol clock, the per-bit window decisions and the SITOR-B state machine on s_seq (ordered after them
// through ff_done when the two streams differ).  marks: optional 8 events recorded around the kernels (timing mode).
cudaError_t demod_launch(const DemodArgs& a, cudaStream_t s_ff, cudaStream_t s_seq, cudaEvent_t ff_done, cudaEvent_t* marks = nullptr);
cudaError_t demod_init_state(const DemodBuffers& b, int channels, cudaStream_t stream);
int demod_launches_per_block();

}  // namespace nvx

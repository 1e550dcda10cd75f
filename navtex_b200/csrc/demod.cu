// demod.cu -- FSK discriminator, bit synchroniser, mark/space decision and SITOR-B byte state
// machine for [channels] independent 900 Hz complex streams.
//
// Replaces, per channel and per block instead of per sample,
//   decoder::sample_in            receiver/decoder.C:42-59    (delay-conjugate product + atan2)
//   decoder::bs_decoded_sample_in receiver/decoder.C:142-255  (bit-sync timing recovery)
//   decoder::bd_decoded_sample_in receiver/decoder.C:73-137   (mark/space energy discriminator)
//   byte_state_machine::receive_bit / receive_rxdx_byte / message_byte_out
//                                 receiver/nav_b_sm.C:266-634, :150-262, :100-145
// Line assembly, the ZCZC/NNNN regexes and add_message (nav_b_sm.C:56-97, :44-52) stay on the
// host (message_assembler.cpp); the last kernel emits the character/line/abort event stream they
// consume.
//
// The reference interleaves everything per sample, but almost all of it is feed-forward in time.  Per block:
//   angle_corr_kernel   thread = sample: FP64 angle of y[n] conj(y[n-1]) and the 9-tap transition mask
//                       correlation, in the reference's operation order;
//   offset_sum_kernel   thread = (channel, ring revolution, offset class): the 63-term per-offset sums "as the
//                       567-ring stood at that sample" in the reference's summation order, and the first-maximum
//                       arg max over the nine sums at every evaluation sample (nine neighbouring lanes);
//   symbol_clock_kernel lane = channel: the slew-limited offset tracking and the WAIT / BIT_START / RECEIVING
//                       symbol clock in event form -- it only decides WHICH five samples make up each bit;
//   bit_decide_kernel   thread = bit: the mark/space decision of that window with the reference's mixed
//                       float/double accumulator arithmetic (_rn intrinsics, no FMA contraction);
//   fsm_kernel          lane = channel: the SITOR-B byte state machine over the block's bits.
// The two lane-per-channel kernels are latency-bound and tiny (64 warps for 2048 channels); they are shaped as
// 16-warp CTAs with a shared-memory footprint that cannot share an SM with the cascade kernel, so that they run on
// the few SMs the cascade grid leaves free instead of fighting its single warp per SM sub-partition.
#include "demod.cuh"

#include <math.h>
#include <stdlib.h>

namespace nvx {

namespace {

constexpr int kThreads = 128;           // feed-forward kernels: one warp per SM sub-partition
constexpr int kPer = 3;                 // samples per thread (independent dependency chains)
constexpr int kTile = kThreads * kPer;  // samples per CTA

__constant__ unsigned char c_ltrs[128];
__constant__ unsigned char c_figs[128];
__constant__ float c_tone_r[5];
__constant__ float c_tone_i[5];
__constant__ double c_tone_rd[5];   // the same tones widened to double
__constant__ double c_tone_id[5];

struct Emit {
    uint8_t* ev; int* ev_n; int ev_cap; int n;
    bool writer;
    const unsigned char *ltrs, *figs;      // code tables in shared memory (per-lane indices would serialise the constant cache)
    __device__ __forceinline__ void put(int c) {
        if (writer && n < ev_cap) ev[n] = (uint8_t)c;
        ++n;
    }
};

// byte_state_machine::init, nav_b_sm.C:16-42 (the error ring contents survive, only its counters reset)
__device__ __forceinline__ void fsm_reset(FsmState& s) {
    s.match = 0; s.byte_state = BY_WAIT; s.figures = 0; s.nbits = 0;
    s.dx_at = 0; s.dx_full = 0;
    s.err_count = 0; s.err_at = 0; s.err_full = 0;
    s.eoe_count = 0; s.prev_dx_alpha = 0;
    s.holdoff = 0; s.enabled = 0;
}

// message_byte_out, nav_b_sm.C:100-145; code 0 = "no valid copy" -> '*'
__device__ __forceinline__ void fsm_char(FsmState& s, Emit& e, int code) {
    if (code == 0) { e.put('*'); return; }
    const int l = e.ltrs[code];
    if (l == 'l') { s.figures = 0; return; }
    if (l == 'f') { s.figures = 1; return; }
    if (l == 'n') { e.put('\n'); return; }
    if (l == 'r' || l == 'p' || l == 'q') return;
    e.put(s.figures ? e.figs[code] : l);
}

// message_abort, nav_b_sm.C:44-52: the host decides whether a message was in progress
__device__ __forceinline__ void fsm_abort(FsmState& s, Emit& e) {
    e.put(kEvAbort);
    fsm_reset(s);
}

// receive_rxdx_byte, nav_b_sm.C:150-262
__device__ __forceinline__ void fsm_byte(FsmState& s, Emit& e, int b) {
    if (s.byte_state == BY_WAIT) {
        if (b == 0x07) s.byte_state = BY_GOT_RX;
        if (b == 0x4c) s.byte_state = BY_GOT_DX;
    } else if (s.byte_state == BY_GOT_RX) {           // byte in the DX slot
        s.dx_ring = (s.dx_ring & ~(0xffu << (8 * s.dx_at))) | ((unsigned)b << (8 * s.dx_at));
        if (++s.dx_at == 3) { s.dx_at = 0; s.dx_full = 1; }
        bool stopped = false;
        if (b == 0x07) {
            if (s.prev_dx_alpha && ++s.eoe_count == 2) { fsm_abort(s, e); stopped = true; }   // end of emission
            if (!stopped) s.prev_dx_alpha = 1;
        } else {
            s.prev_dx_alpha = 0;
        }
        if (!stopped) s.byte_state = BY_GOT_DX;
    } else {                                           // BY_GOT_DX: byte in the RX slot
        if (s.dx_full) {
            const int dx = (s.dx_ring >> (8 * s.dx_at)) & 0x7f;
            if (e.ltrs[b] != '_') fsm_char(s, e, b);
            else if (e.ltrs[dx] != '_') fsm_char(s, e, dx);
            else fsm_char(s, e, 0);
        }
        s.byte_state = BY_GOT_RX;
    }
    // 20-byte sliding window of invalid codes (nav_b_sm.C:235-261)
    const unsigned bit = 1u << s.err_at;
    if (s.err_full && (s.err_mask & bit)) s.err_count--;
    const bool bad = e.ltrs[b] == '_';
    s.err_mask = bad ? (s.err_mask | bit) : (s.err_mask & ~bit);
    if (bad) s.err_count++;
    if (++s.err_at == 20) { s.err_at = 0; s.err_full = 1; }
    if (s.err_count > 12) {
        fsm_char(s, e, 0);
        fsm_abort(s, e);
    }
}

// receive_bit, nav_b_sm.C:266-634, in two halves so that the lanes of a warp (32 channels with 32 different byte phases) can meet
// at the expensive one.  First half (:269-286): shift the bit in; true = this bit completes a 7-bit byte, which the caller must
// hand to fsm_byte() BEFORE the second half of the same bit.  is_y: 'Y' (=1) else 'B'.
__device__ __forceinline__ bool fsm_bit_shift(FsmState& s, bool is_y, int& byte) {
    if (!s.enabled) return false;
    s.shift = ((s.shift << 1) | (is_y ? 1 : 0)) & 0x7f;
    if (++s.nbits < 7) return false;
    byte = s.shift;
    s.nbits = 0;
    s.shift = 0;
    return true;
}
// second half (:288-633): detector hold-off and the 30-bit phasing pattern
__device__ __forceinline__ void fsm_bit_phasing(FsmState& s, bool is_y) {
    if (s.holdoff != 0) { s.holdoff--; return; }
    // 30-bit phasing pattern BBBBBB YYYY BB YY BBBBBB YYYY BB YY BB, bit k of the mask = 1 for 'Y'
    // positions of 'Y': 6-9, 12-13, 20-23, 26-27
    constexpr unsigned kYmask = (0xFu << 6) | (0x3u << 12) | (0xFu << 20) | (0x3u << 26);
    if (s.match == 29) {
        if (!is_y) { s.enabled = 1; s.nbits = 0; s.shift = 0; s.holdoff = 1100; }   // nav_b_sm.h:52
        s.match = 0;
    } else if ((((kYmask >> s.match) & 1u) != 0) == is_y) {
        s.match++;
    } else if (s.match != 6) {          // extra B's are tolerated only after the first BBBBBB (nav_b_sm.C:363-372)
        s.match = 0;
    }
}


__device__ __forceinline__ size_t pitch_y(int p_max) { return (size_t)kHistY + p_max; }
__device__ __forceinline__ size_t pitch_c(int p_max) { return (size_t)kHistC + p_max + kPadC; }
__host__ __device__ __forceinline__ size_t pitch_p(int p_max) { return ((size_t)p_max / kSpb + 2 + 15) & ~(size_t)15; }   // picks (bytes)
// bits per block: a bit normally takes 9 samples, but while the tracked offset slews by -1 per evaluation the next trigger comes
// 8 samples after the previous one (decoder.C:217-249), so a block of P samples can hold up to P / 8 + 1 bits
__host__ __device__ __forceinline__ size_t pitch_b(int p_max) { return ((size_t)p_max / (kSpb - 1) + 2 + 15) & ~(size_t)15; }   // bits (elements)

// decoder.C:48-52
__device__ __forceinline__ double angle_of(float2 cur, float2 prev) {
    const double yi = cur.x, yq = cur.y, pi = prev.x, pq = prev.y;
    const double re = __dadd_rn(__dmul_rn(yi, pi), __dmul_rn(yq, pq));
    const double im = __dsub_rn(__dmul_rn(yq, pi), __dmul_rn(yi, pq));
    return atan2(im, re);
}

// grid (tiles, channels), block kThreads: |mask correlation| for samples [tile0, tile0 + kTile); every thread owns three
// samples (strided by kThreads) so that one resident warp per SM sub-partition still has independent work in flight
// The CTA of tile 0 also hands the histories over: the last kHistY samples / kHistC correlation values of the previous block
// (which live at the end of ITS buffers) become the front of this block's buffers.  Nobody else touches those fronts in this
// kernel (only tile 0 looks back past sample 0), and every later kernel of the block is ordered behind it.
__global__ void __launch_bounds__(kThreads) angle_corr_kernel(const DemodArgs a) {
    __shared__ double s_ang[kTile + 8];
    const int ch = blockIdx.y, tile0 = blockIdx.x * kTile, t = threadIdx.x;
    float2* ybuf = a.b.y3 + (size_t)ch * pitch_y(a.b.p_max);
    const float2* y = ybuf + kHistY;                                          // y[m], m >= -kHistY
    if (blockIdx.x == 0) {
        const float2* yp = a.y3_prev + (size_t)ch * pitch_y(a.b.p_max) + a.n_prev;
        if (t < kHistY) ybuf[t] = yp[t];
        double* c = a.b.corr + (size_t)ch * pitch_c(a.b.p_max);
        const double* cp = a.corr_prev + (size_t)ch * pitch_c(a.b.p_max) + a.n_prev;
        for (int k = t; k < kHistC; k += kThreads) c[k] = cp[k];
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
        const int m = tile0 + t + u * kThreads;
        if (m < a.n_new) s_ang[8 + t + u * kThreads] = angle_of(y[m], y[m - 1]);
    }
    if (t < 8) s_ang[t] = angle_of(y[tile0 - 8 + t], y[tile0 - 9 + t]);
    __syncthreads();
    double* corr = a.b.corr + (size_t)ch * pitch_c(a.b.p_max) + kHistC;
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
        const int i = t + u * kThreads, m = tile0 + i;
        if (m >= a.n_new) break;
        // mask {0,1,1,1,0,-1,-1,-1,0} over angles n-8 .. n, oldest first (decoder.C:161-170); s_ang[8 + i - k] = angle[m - k]
        double c = s_ang[i + 1];
        c = __dadd_rn(c, s_ang[i + 2]);
        c = __dadd_rn(c, s_ang[i + 3]);
        c = __dsub_rn(c, s_ang[i + 5]);
        c = __dsub_rn(c, s_ang[i + 6]);
        c = __dsub_rn(c, s_ang[i + 7]);
        corr[m] = fabs(c);
    }
}

// mark/space decision of the window y[0..4] (decoder.C:109-133).  Returns true for 'Y'.
// Reference arithmetic per sample (SURVEY.md A.3): acc = (float)((double)acc + ((double)((float)sR * f_a) +- sI * (double)f_b)).
// (float)sR is the stored float itself, (float)(-sR) * f = -((float)sR * f) exactly, and the float accumulators are
// carried as doubles holding float-representable values, so only the four roundings to float cost conversions.
__device__ __forceinline__ bool window_is_y(const float2* __restrict__ y, float* sums) {
    double br = 0.0, bi = 0.0, yr = 0.0, yi = 0.0;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const float srf = y[k].x;
        const double si = (double)y[k].y;
        const float fr = c_tone_r[k], fi = c_tone_i[k];
        const double pr = (double)__fmul_rn(srf, fr), pim = (double)__fmul_rn(srf, fi);
        const double qi = __dmul_rn(si, c_tone_id[k]), qr = __dmul_rn(si, c_tone_rd[k]);
        yr = (double)(float)__dadd_rn(yr, __dsub_rn(pr, qi));
        yi = (double)(float)__dadd_rn(yi, __dadd_rn(pim, qr));
        br = (double)(float)__dadd_rn(br, __dadd_rn(pr, qi));
        bi = (double)(float)__dadd_rn(bi, __dsub_rn(qr, pim));      // (-pim) + qr
    }
    const float brf = (float)br, bif = (float)bi, yrf = (float)yr, yif = (float)yi;
    if (sums) { sums[0] = brf; sums[1] = bif; sums[2] = yrf; sums[3] = yif; }
    const float eb = __fadd_rn(__fmul_rn(brf, brf), __fmul_rn(bif, bif));
    const float ey = __fadd_rn(__fmul_rn(yrf, yrf), __fmul_rn(yif, yif));
    return !(eb > ey);
}

// Per-offset sums + arg max (decoder.C:181-215).  At sample n the reference adds up the 63 ring slots j, j + 9, ...
// (j = (n - 7) mod 9) in ascending slot order, the ring standing as it did after sample n's own write.  Those slots
// hold one residue class of samples -- the newest written at n - 8 -- and slot order is "from the value in slot j
// forward in time to the newest, then from the oldest forward".  With K = the 567-sample ring revolution and
// r = 0..62 the position of the newest class member inside it (n = 16 + 567 K + j + 9 r):
//     sum(n) = ((cur[0] + ... + cur[r]) + prev[r + 1]) + ... + prev[62],
// cur[i] = corr[n - 8 - 9 (r - i)] (this revolution), prev[i] = cur[i] one revolution earlier.  The prefix over cur is a
// running sum along r, so ONE THREAD owns (channel, revolution K, class j), walks r = 0..62 and spends 1 + (62 - r)
// FP64 adds per sample instead of 63 -- every add in the reference's order, so the sums are bit-identical to a
// literal transcription.  Seven consecutive r are in flight at once (seven independent DADD chains, each prev[] value
// loaded once per seven).
// The arg max taken at evaluation sample n = 24 + 567 K + 9 r compares the sums made at samples n - 8 .. n, which are
// exactly the nine classes j = 0..8 at the same (K, r): nine neighbouring lanes.  They exchange through a per-warp
// shared-memory patch; lanes 0..20 then each resolve one (revolution, r) arg max (first maximum wins, j ascending,
// seed -1.0 as decoder.C:207-215) and store the pick of that evaluation sample.
// Warp = 3 revolutions x 9 classes (27 lanes); (channel, revolution) pairs are flattened over warps.
constexpr int kSumWarps = 4;
constexpr int kGroup = 7;                                  // r values in flight per thread
__global__ void __launch_bounds__(kSumWarps * 32) offset_sum_kernel(const DemodArgs a, int k_lo, int n_rev) {
    __shared__ double s_os[kSumWarps][3][kGroup][kSpb];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kk = lane / kSpb, j = lane - kk * kSpb;       // lanes 27..31: kk == 3, idle
    const long long unit = ((long long)blockIdx.x * kSumWarps + warp) * 3 + kk;     // (channel, revolution) pair
    const bool mine = kk < 3 && unit < (long long)a.channels * n_rev;
    const int ch = mine ? (int)(unit / n_rev) : 0;
    const int K = k_lo + (mine ? (int)(unit % n_rev) : 0);
    // first block-relative sample whose ring is full (decoder.C:181), counted from the channel's epoch (nvx_engine_reset_streams)
    const int m_full = (int)max(kCorrLen + 7 - (a.seen - a.b.epoch[ch]), -(1ll << 30));
    // block-relative sample of the evaluation r = 0 of this thread; its class members sit 8 samples earlier
    const int m_first = (int)(16 + (long long)kCorrLen * K + j - a.seen);
    const double* cur = a.b.corr + (size_t)ch * pitch_c(a.b.p_max) + kHistC + (m_first - 8);
    const double* prev = cur - kCorrLen;
    // the lane that resolves arg maxima: (revolution kk2, r offset u2) of this warp
    const int kk2 = lane / kGroup, u2 = lane - kk2 * kGroup;
    const long long unit2 = ((long long)blockIdx.x * kSumWarps + warp) * 3 + kk2;
    const bool judge = kk2 < 3 && unit2 < (long long)a.channels * n_rev;
    const int ch2 = judge ? (int)(unit2 / n_rev) : 0;
    const int w_full = (int)max(kCorrLen + 15 - (a.seen - a.b.epoch[ch2]), -(1ll << 30));     // first evaluation with a pick
    const int w_first = (int)(24 + (long long)kCorrLen * (k_lo + (judge ? (int)(unit2 % n_rev) : 0)) - a.seen);
    uint8_t* picks2 = a.b.picks + (size_t)ch2 * pitch_p(a.b.p_max);     // evaluation samples of a block: e0 + 9 q

    double run = 0.0;
#pragma unroll 1
    for (int g = 0; g < kCorrLen / kSpb / kGroup; ++g) {
        const int r0 = g * kGroup;
        const int m0 = m_first + kSpb * r0;                 // sample of evaluation r0
        double acc[kGroup];
        if (mine && m0 < a.n_new) {
#pragma unroll
            for (int u = 0; u < kGroup; ++u) {
                run = __dadd_rn(run, __ldg(cur + kSpb * (r0 + u)));
                acc[u] = run;
            }
        } else {
#pragma unroll
            for (int u = 0; u < kGroup; ++u) acc[u] = 0.0;
        }
        // only groups with a sample inside [-8, n_new) matter (arg max windows reach 8 samples back)
        if (mine && m0 < a.n_new && m0 + kSpb * (kGroup - 1) >= -8) {
            const double* p = prev + kSpb * (r0 + 1);
            double v[kGroup - 1];
#pragma unroll
            for (int t = 0; t < kGroup - 1; ++t) v[t] = __ldg(p + kSpb * t);
#pragma unroll
            for (int u = 0; u < kGroup - 1; ++u) {
#pragma unroll
                for (int t = u; t < kGroup - 1; ++t) acc[u] = __dadd_rn(acc[u], v[t]);
            }
            p += kSpb * (kGroup - 1);
            const int rest = kCorrLen / kSpb - kGroup - r0;   // 56, 49, ..., 0: prev[r0 + 7 .. 62] go to all seven
#pragma unroll 1
            for (int i = 0; i < rest; i += kGroup, p += kSpb * kGroup) {
                double x[kGroup];
#pragma unroll
                for (int t = 0; t < kGroup; ++t) x[t] = __ldg(p + kSpb * t);
#pragma unroll
                for (int t = 0; t < kGroup; ++t) {
#pragma unroll
                    for (int u = 0; u < kGroup; ++u) acc[u] = __dadd_rn(acc[u], x[t]);
                }
            }
        }
        if (kk < 3) {
#pragma unroll
            for (int u = 0; u < kGroup; ++u) {
                const int m = m0 + kSpb * u;
                const bool ok = mine && m < a.n_new && m >= m_full;
                s_os[warp][kk][u][j] = ok ? acc[u] : 0.0;
            }
        }
        __syncwarp();
        if (judge) {
            const int w = w_first + kSpb * (r0 + u2);
            if (w >= 0 && w < a.n_new && w >= w_full) {
                double best = -1.0;
                int pick = 0;
#pragma unroll
                for (int i = 0; i < kSpb; ++i) {
                    const double x = s_os[warp][kk2][u2][i];
                    if (x > best) { best = x; pick = i; }
                }
                picks2[w / kSpb] = (uint8_t)pick;
            }
        }
        __syncwarp();
    }
}

// ---- sequential part --------------------------------------------------------------------------------------------
// lane = channel, warp = 32 channels, CTA = kSeqWarps warps.  Per-channel byte rows (picks, bit values) are staged
// through shared memory in chunks, coalesced, with an odd word pitch so that the per-lane reads are conflict free.
constexpr int kSeqWarps = 16;
constexpr int kSeqChunk = 256;                                // bytes of every channel's row staged at a time
constexpr int kSeqPitch = kSeqChunk + 4;                      // 65 words
constexpr int kSeqSmem = kSeqWarps * 32 * kSeqPitch;          // 133 KB: no room left for a cascade CTA on the same SM

__device__ __forceinline__ void stage_rows(uint8_t* s_rows, const uint8_t* src, size_t pitch, int ch0, int channels,
                                           int c0, int count, int lane) {
    // rows [ch0, ch0 + 32), bytes [c0, c0 + count) (c0 and the pitch are multiples of 4)
    __syncwarp();
    const int words = (count + 3) >> 2;
    for (int r = 0; r < 32 && ch0 + r < channels; ++r) {
        const uint32_t* g = reinterpret_cast<const uint32_t*>(src + (size_t)(ch0 + r) * pitch + c0);
        uint32_t* d = reinterpret_cast<uint32_t*>(s_rows + r * kSeqPitch);
        for (int k = lane; k < words; k += 32) d[k] = g[k];
    }
    __syncwarp();
}

// Symbol clock, one iteration per BIT:
//   trigger t0 = first sample >= cur whose (n + 1) mod 9 equals the bit-sync offset (decoder.C:83-90);
//   the samples t0, t0+1, t0+2 are burnt, t0+3 .. t0+7 integrated, the bit is decided at t0+7 (decoder.C:91-135);
//   every evaluation sample <= t0+7 has by then updated next_offs (bs_ runs before bd_, decoder.C:57-58).
// Output: the window start t0+3 of every bit decided in this block.
__global__ void __launch_bounds__(kSeqWarps * 32) symbol_clock_kernel(const DemodArgs a) {
    extern __shared__ __align__(16) uint8_t s_seq[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ch0 = (blockIdx.x * kSeqWarps + warp) * 32, ch = ch0 + lane;
    if (ch0 >= a.channels) return;
    const bool live = ch < a.channels;
    uint8_t* rows = s_seq + (size_t)warp * 32 * kSeqPitch;
    const uint8_t* my_row = rows + lane * kSeqPitch;
    ClockState s = {};
    if (live) s = a.b.clock[ch];
    int* bitpos = a.b.bitpos + (size_t)(live ? ch : 0) * pitch_b(a.b.p_max);
    const int cap = (int)pitch_b(a.b.p_max);
    int nb = 0;

    // evaluation samples of this block (decoder.C:204): w = e0 + 9 q with absolute index == 6 (mod 9), from 582 on
    const int seen9 = (int)(a.seen % kSpb);
    const int e0 = (6 - seen9 + kSpb) % kSpb;
    const int n_eval = e0 < a.n_new ? (a.n_new - 1 - e0) / kSpb + 1 : 0;
    int q = n_eval;
    if (live) {     // the first evaluation after the channel's ring filled (its epoch: nvx_engine_reset_streams)
        const long long need = kCorrLen + 15 - (a.seen - a.b.epoch[ch]) - e0;
        q = need > 0 ? (int)min((need + kSpb - 1) / kSpb, (long long)n_eval) : 0;
    }
    const int q_warp = __reduce_min_sync(0xffffffffu, q);         // the chunks are staged by the whole warp
    for (int c0 = (q_warp / kSeqChunk) * kSeqChunk; c0 < n_eval || c0 == 0; c0 += kSeqChunk) {
        const int c1 = min(n_eval, c0 + kSeqChunk);
        if (c1 > c0) stage_rows(rows, a.b.picks, pitch_p(a.b.p_max), ch0, a.channels, c0, c1 - c0, lane);
        const int lim = c1 == n_eval ? a.n_new : e0 + kSpb * c1;          // samples whose evaluations are staged
        auto do_eval = [&](int qq) {
            int pick = my_row[qq - c0];
            if (s.last_pick != -1 && pick != s.last_pick) {        // slew one step the short way round (decoder.C:217-246)
                bool up;
                if (pick > s.last_pick) up = !(pick - s.last_pick > 4);
                else up = (s.last_pick - pick > 4);
                pick = up ? (s.last_pick + 1) % kSpb : (s.last_pick - 1 + kSpb) % kSpb;
            }
            s.last_pick = pick;
            const int offs = (pick + 5) % kSpb;                    // decoder.C:249
            if (s.dstate == DS_INIT) { s.dstate = DS_WAIT; s.offs = offs; s.cur = e0 + kSpb * qq; }   // decoder.C:62-70
            s.next_offs = offs;
        };
        while (live) {
            if (s.dstate == DS_INIT) {
                if (q >= c1) break;
                do_eval(q);
                ++q;
                if (s.dstate == DS_INIT) continue;
            }
            if (s.dstate == DS_WAIT) {
                const int tick = (seen9 + s.cur + 1) % kSpb;
                const int t0 = s.cur + (s.offs - tick + kSpb) % kSpb;
                if (t0 >= a.n_new) break;
                s.dstate = DS_PENDING;
                s.pend = t0;
            }
            const int td = s.pend + 7;
            if (td >= lim) break;
            while (q < c1 && e0 + kSpb * q <= td) { do_eval(q); ++q; }
            if (nb < cap) bitpos[nb] = s.pend + 3;
            ++nb;
            s.offs = s.next_offs;
            s.dstate = DS_WAIT;
            s.cur = td + 1;
        }
        // what is left of the chunk precedes the next bit decision (or no further bit ends in this block)
        if (live) while (q < c1) { do_eval(q); ++q; }
        if (c1 == n_eval) break;
    }
    if (!live) return;
    if (s.dstate == DS_PENDING) s.pend -= a.n_new;
    s.cur = s.cur > a.n_new ? s.cur - a.n_new : 0;
    a.b.clock[ch] = s;
    a.b.nbits[ch] = nb;
    if (a.bit_count) a.bit_count[ch] = nb;
}

// grid (tiles, channels), block 128: thread = one bit of the block -> its mark/space decision
__global__ void __launch_bounds__(128) bit_decide_kernel(const DemodArgs a) {
    const int ch = blockIdx.y, k = blockIdx.x * 128 + threadIdx.x;
    const int nb = min(a.b.nbits[ch], (int)pitch_b(a.b.p_max));
    if (k >= nb) return;
    const int w = a.b.bitpos[(size_t)ch * pitch_b(a.b.p_max) + k];
    const float2* y = a.b.y3 + (size_t)ch * pitch_y(a.b.p_max) + kHistY + w;
    const bool tap = a.bits && k < a.bit_cap;
    const bool is_y = window_is_y(y, tap && a.disc ? a.disc + ((size_t)ch * a.bit_cap + k) * 4 : nullptr);
    a.b.bitval[(size_t)ch * pitch_b(a.b.p_max) + k] = is_y ? 1 : 0;
    if (tap) a.bits[(size_t)ch * a.bit_cap + k] = is_y ? 'Y' : 'B';
}

// lane = channel: receive_bit (nav_b_sm.C:266-634) over the bits of the block
__global__ void __launch_bounds__(kSeqWarps * 32) fsm_kernel(const DemodArgs a) {
    extern __shared__ __align__(16) uint8_t s_seq[];
    __shared__ unsigned char s_ltrs[128], s_figs[128];      // per-lane indices would serialise the constant cache
    for (int k = threadIdx.x; k < 128; k += blockDim.x) { s_ltrs[k] = c_ltrs[k]; s_figs[k] = c_figs[k]; }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ch0 = (blockIdx.x * kSeqWarps + warp) * 32, ch = ch0 + lane;
    if (ch0 >= a.channels) return;
    const bool live = ch < a.channels;
    uint8_t* rows = s_seq + (size_t)warp * 32 * kSeqPitch;
    const uint8_t* my_row = rows + lane * kSeqPitch;
    FsmState s = {};
    if (live) s = a.b.fsm[ch];
    Emit em;
    em.ev = a.events + (size_t)(live ? ch : 0) * a.ev_cap; em.ev_cap = a.ev_cap; em.n = 0; em.writer = live;
    em.ltrs = s_ltrs; em.figs = s_figs;
    const int nb = live ? min(a.b.nbits[ch], (int)pitch_b(a.b.p_max)) : 0;
    const int nb_max = __reduce_max_sync(0xffffffffu, nb);
    for (int c0 = 0; c0 < nb_max; c0 += kSeqChunk) {
        const int c1 = min(nb_max, c0 + kSeqChunk);
        stage_rows(rows, a.b.bitval, pitch_b(a.b.p_max), ch0, a.channels, c0, c1 - c0, lane);
        const int mine = min(nb, c1);
        // The lane's row of the chunk (one byte per bit) is packed into eight 32-bit words first -- 64 independent loads instead of
        // one dependent byte load per bit -- and written back over the front of its own row.
        {
            uint32_t pk[kSeqChunk / 32];
            const uint32_t* rw = reinterpret_cast<const uint32_t*>(my_row);
#pragma unroll
            for (int w = 0; w < kSeqChunk / 32; ++w) {
                uint32_t acc = 0;
#pragma unroll
                for (int q4 = 0; q4 < 8; ++q4)      // four bytes holding 0 / 1 -> four bits
                    acc |= ((((rw[w * 8 + q4] & 0x01010101u) * 0x01020408u) >> 24) & 0xFu) << (4 * q4);
                pk[w] = acc;
            }
            uint32_t* ww = reinterpret_cast<uint32_t*>(rows + lane * kSeqPitch);
#pragma unroll
            for (int w = 0; w < kSeqChunk / 32; ++w) ww[w] = pk[w];
        }
        const uint32_t* wrow = reinterpret_cast<const uint32_t*>(my_row);
        // Every lane runs through at most seven of its bits, stopping at (the first half of) the one that completes a byte; then
        // the whole warp does receive_rxdx_byte together and finishes that bit.  After the first round the byte phases of the 32
        // channels of a warp are aligned, so the expensive byte path runs once per seven bits instead of at every bit.
        int k = c0;
        uint32_t word = k < mine ? wrow[0] : 0u;
        for (;;) {
            int byte = 0;
            bool pending = false, y = false;
#pragma unroll 1
            for (int i = 0; i < 7 && k < mine; ++i) {
                y = (word & 1u) != 0;
                word >>= 1;
                ++k;
                if (((k - c0) & 31) == 0) word = wrow[(k - c0) >> 5];      // (index 8 at the end of a full chunk: the row's pad word)
                pending = fsm_bit_shift(s, y, byte);
                if (pending) break;
                fsm_bit_phasing(s, y);
            }
            if (pending) {
                fsm_byte(s, em, byte);
                fsm_bit_phasing(s, y);
            }
            if (!__any_sync(0xffffffffu, k < mine)) break;       // every lane has used up the chunk
        }
    }
    if (!live) return;
    a.b.fsm[ch] = s;
    a.ev_count[ch] = em.n;
}

__global__ void init_state_kernel(ClockState* clock, FsmState* fsm, int channels) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= channels) return;
    // decoder::decoder (decoder.C:6-39) and byte_state_machine::init (nav_b_sm.C:16-42)
    clock[ch] = clock_state_init();
    fsm[ch] = fsm_state_init();
}

}  // namespace

int demod_launches_per_block() { return 5; }
size_t demod_pick_pitch(int p_max) { return pitch_p(p_max); }
size_t demod_bit_pitch(int p_max) { return pitch_b(p_max); }
int demod_reserved_sms(int channels) {
    const int ctas = (channels + kSeqWarps * 32 - 1) / (kSeqWarps * 32);
    return ctas < 4 ? ctas : 4;
}

cudaError_t demod_init_state(const DemodBuffers& b, int channels, cudaStream_t stream) {
    {   // constant-bank tables are per device: (re)loaded with every engine create / reset
        // CCIR 476 tables as (code, letters, figures); see nav_b_sm.h:60-83 -- every other code is invalid '_'.
        static const struct { unsigned char code; char l, f; } codes[] = {
            {0x07, 'p', 'p'}, {0x0b, 'J', 'b'}, {0x0d, 'W', '2'}, {0x0e, 'A', '-'}, {0x13, 'F', '*'},
            {0x15, 'Y', '6'}, {0x16, 'S', '\''}, {0x19, '-', '-'}, {0x1a, 'D', '%'}, {0x1c, 'Z', '+'},
            {0x1d, '_', ' '}, {0x23, 'C', ':'}, {0x25, 'P', '0'}, {0x26, 'I', '8'}, {0x29, 'G', '*'},
            {0x2a, 'R', '4'}, {0x2c, 'L', ')'}, {0x31, 'M', '.'}, {0x32, 'N', ','}, {0x34, 'H', '*'},
            {0x38, 'O', '9'}, {0x43, 'K', '('}, {0x45, 'Q', '1'}, {0x46, 'U', '7'}, {0x49, 'f', 'f'},
            {0x4a, 'E', '3'}, {0x4c, 'q', 'q'}, {0x51, 'X', '/'}, {0x52, 'l', 'l'}, {0x58, 'B', '?'},
            {0x5c, ' ', ' '}, {0x61, 'V', '='}, {0x62, ' ', ' '}, {0x64, 'n', 'n'}, {0x68, 'T', '5'},
            {0x70, 'r', 'r'},
        };
        unsigned char ltrs[128], figs[128];
        for (int i = 0; i < 128; ++i) ltrs[i] = figs[i] = '_';
        for (const auto& c : codes) { ltrs[c.code] = (unsigned char)c.l; figs[c.code] = (unsigned char)c.f; }
        float tr[5], ti[5];
        for (int i = 0; i < 5; ++i) {
            const float ang = (float)((i * 2 * 3.1415 * 85) / 900);     // decoder.C:25: 3.1415, float angle
            tr[i] = cosf(ang);
            ti[i] = sinf(ang);
        }
        cudaError_t e;
        if ((e = cudaMemcpyToSymbol(c_ltrs, ltrs, sizeof ltrs)) != cudaSuccess) return e;
        if ((e = cudaMemcpyToSymbol(c_figs, figs, sizeof figs)) != cudaSuccess) return e;
        if ((e = cudaMemcpyToSymbol(c_tone_r, tr, sizeof tr)) != cudaSuccess) return e;
        if ((e = cudaMemcpyToSymbol(c_tone_i, ti, sizeof ti)) != cudaSuccess) return e;
        double trd[5], tid[5];
        for (int i = 0; i < 5; ++i) { trd[i] = tr[i]; tid[i] = ti[i]; }
        if ((e = cudaMemcpyToSymbol(c_tone_rd, trd, sizeof trd)) != cudaSuccess) return e;
        if ((e = cudaMemcpyToSymbol(c_tone_id, tid, sizeof tid)) != cudaSuccess) return e;
    }
    cudaError_t e;
    if ((e = cudaMemsetAsync(b.y3, 0, sizeof(float2) * (size_t)channels * (kHistY + b.p_max), stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(b.corr, 0, sizeof(double) * (size_t)channels * (kHistC + b.p_max + kPadC), stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(b.picks, 0, (size_t)channels * pitch_p(b.p_max), stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(b.epoch, 0, sizeof(long long) * (size_t)channels, stream)) != cudaSuccess) return e;
    init_state_kernel<<<(channels + 127) / 128, 128, 0, stream>>>(b.clock, b.fsm, channels);
    return cudaGetLastError();
}

cudaError_t demod_launch(const DemodArgs& a, cudaStream_t s_ff, cudaStream_t s_seq, cudaEvent_t ff_done, cudaEvent_t* marks) {
    if (a.n_new <= 0 || a.channels <= 0) return cudaSuccess;
    auto mark = [&](int k, cudaStream_t st) { if (marks) cudaEventRecord(marks[k], st); };
    // feed-forward part (thread = sample / ring revolution): whole-GPU kernels, ~0.3 ms per 10 s block of 2048 channels
    mark(0, s_ff);
    angle_corr_kernel<<<dim3((a.n_new + kTile - 1) / kTile, a.channels), kThreads, 0, s_ff>>>(a);
    mark(1, s_ff);
    // Ring revolutions with an evaluation sample in [-8, n_new): samples 16 + 567 K .. 582 + 567 K.  The revolutions are counted
    // on the absolute grid, whatever the channels' epochs: epochs are multiples of 567, so a channel's revolutions are the ones a
    // fresh engine would walk, and those before its ring filled produce sums and picks that its epoch-relative gates discard.
    {
        const long long lo = a.seen - 8 - (kCorrLen + 15), hi = a.seen + a.n_new - 17;
        const int k_lo = lo <= 0 ? 0 : (int)((lo + kCorrLen - 1) / kCorrLen);
        if (hi >= 0 && (int)(hi / kCorrLen) >= k_lo) {
            const int n_rev = (int)(hi / kCorrLen) - k_lo + 1;
            const long long units = (long long)a.channels * n_rev;
            offset_sum_kernel<<<(unsigned)((units + 3 * kSumWarps - 1) / (3 * kSumWarps)), kSumWarps * 32, 0, s_ff>>>(a, k_lo, n_rev);
        }
    }
    mark(2, s_ff);
    mark(3, s_ff);      // (the history carry used to be a kernel of its own here; angle_corr_kernel does it now)
    // sequential part: few warps, latency-bound, runs beside the next block's cascade on the SMs it leaves free
    {   // ff_done also tells the engine when this block's look-back into the previous block's y3 buffer is over
        cudaError_t e = cudaEventRecord(ff_done, s_ff);
        if (e != cudaSuccess) return e;
        if (s_seq != s_ff && (e = cudaStreamWaitEvent(s_seq, ff_done, 0)) != cudaSuccess) return e;
    }
    {   // per device, and a few hundred nanoseconds: not cached
        cudaError_t e = cudaFuncSetAttribute(symbol_clock_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSeqSmem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSeqSmem);
        if (e != cudaSuccess) return e;
    }
    const unsigned seq_ctas = (a.channels + kSeqWarps * 32 - 1) / (kSeqWarps * 32);
    mark(4, s_seq);
    symbol_clock_kernel<<<seq_ctas, kSeqWarps * 32, kSeqSmem, s_seq>>>(a);
    mark(5, s_seq);
    bit_decide_kernel<<<dim3((unsigned)((a.n_new / (kSpb - 1) + 2 + 127) / 128), a.channels), 128, 0, s_seq>>>(a);
    mark(6, s_seq);
    fsm_kernel<<<seq_ctas, kSeqWarps * 32, kSeqSmem, s_seq>>>(a);
    mark(7, s_seq);
    return cudaGetLastError();
}

}  // namespace nvx

// fir_cascade.cuh -- fused stage-1 FIR (/4) -> NCO mix (two channels) -> stage-2 FIR (/7) ->
// stage-3 FIR (/10) for batches of independent IQ streams, sm_100a.
//
// Replaces, for [streams x samples] at once, the reference's per-sample push chain
//   sample_in_1   receiver/fir1cpp.C:80-136   (37 taps, /4)
//   sample_in_2   receiver/fir2cpp.C:112-128  (mix by e^{-+j 2 pi k 2/9})
//   fir_in_2 / fir_in_2_490   fir2cpp.C:131-215 (47 taps, /7, per channel)
//   fir_filter3::sample_in    fir3cpp.C:22-60   (71 taps, /10, per channel)
// and emits the 900 Hz complex samples that decoder::sample_in (decoder.C:42) consumes.
//
// Mapping (B200-first, not the reference's ring buffers):
//   * one THREAD owns one (stream, time-segment) "row"; a warp is 32 rows.  Every FIR stage
//     runs in transposed (scatter) polyphase form: an arriving sample is multiply-added into
//     the few output accumulators it belongs to, so the whole cascade state is 9 + 2*6 + 2*8
//     complex partial sums in registers and no intermediate (63 kHz, 9 kHz) sample ever
//     touches shared memory or HBM.
//   * I and Q ride in one 64-bit register pair and every tap is one FFMA2 (fma.rn.f32x2) with
//     the tap as a 32-bit immediate / uniform operand: 2 FMAs per lane per issue slot.
//   * a warp's 32 rows are 32 consecutive streams at the same time segment, so the samples they
//     need for two 28-sample steps form a [32 streams x 448 B] box of the stream-major input
//     (224 B when the input is int16 pairs, 112 B for 8-bit pairs): ONE TMA tensor copy (cp.async.bulk.tensor.2d ->
//     UTMALDG) per warp per stage into a per-warp ring of shared-memory stages, completion
//     tracked by one mbarrier per stage.  Each lane then reads its own row with LDS.128.
//   * variants (template flags): taps as immediates or from the constant bank (replacement tap
//     sets), the reference's 9-entry NCO table or an exact per-stream NCO, float2, short2 or 8-bit input (SampleFmt).
//   * time segments are made independent by recomputing a 7-superblock (1960-sample) warm-up
//     from the raw input that precedes the segment (previous segment, or the carried tail of
//     the previous chunk); since every 900 Hz output depends on exactly 2181 inputs
//     (SURVEY.md A.5) the results are bit-identical to an unsegmented pass.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/navtex_taps.h"

namespace nvx {

constexpr int kSuper = NVX_D1 * NVX_D2 * NVX_D3;   // 280 inputs per 900 Hz output
constexpr int kStepIn = NVX_D1 * NVX_D2;           // 28 inputs per 9 kHz output ("step")
constexpr int kStepsPerSuper = NVX_D3;             // 10
// warm-up superblocks / carried input samples per stream are per tap-length class: Geo<>::kWarm (7 -> 1960 samples for the
// reference lengths: ceil(1901 / 280))
constexpr int kNcoPeriod = 9;                      // fir2cpp.C:12-14
// Tunables (see DESIGN.md "input staging"): how many 28-sample steps one TMA box carries per stream row, how many
// extra floats pad each row in shared memory (bank-conflict control), ring depth and CTA shape.  Measured on B200
// (profiles/r1_staging_sweep.md): HBM efficiency of the [32 streams x B bytes] access pattern rises with B
// (224 B: 6.2 TB/s, 448 B: 6.9 TB/s with no compute at all), the FMA pipe wants the same number of warps on each of
// the four SM sub-partitions (4 or 8 warps per SM), and the third ring stage matters more than a second warp per
// sub-partition.  Default: 448-byte rows (+16 B pad), 3 stages, 4 warps, 1 CTA per SM = 178 KB of shared memory.
#ifndef NVX_STEPS_PER_STAGE
#define NVX_STEPS_PER_STAGE 2
#endif
#ifndef NVX_ROW_PAD_FLOATS
#define NVX_ROW_PAD_FLOATS 4
#endif
#ifndef NVX_STAGES
#define NVX_STAGES 3
#endif
#ifndef NVX_WARPS_PER_CTA
#define NVX_WARPS_PER_CTA 4
#endif
#ifndef NVX_CTAS_PER_SM
#define NVX_CTAS_PER_SM 1
#endif
#ifndef NVX_S16_STEPS_PER_STAGE
#define NVX_S16_STEPS_PER_STAGE 2
#endif
#ifndef NVX_S16_ROW_PAD_BYTES
#define NVX_S16_ROW_PAD_BYTES 16
#endif
#ifndef NVX_S16_STAGES
#define NVX_S16_STAGES 2
#endif
#ifndef NVX_S16_WARPS_PER_CTA
#define NVX_S16_WARPS_PER_CTA 12
#endif
#ifndef NVX_U8_ROW_PAD_BYTES
#define NVX_U8_ROW_PAD_BYTES 32
#endif
#ifndef NVX_U8_STAGES
#define NVX_U8_STAGES 2
#endif
#ifndef NVX_U8_WARPS_PER_CTA
#define NVX_U8_WARPS_PER_CTA 12
#endif
constexpr int kCtasPerSm = NVX_CTAS_PER_SM;

// The sample formats an engine accepts (one between resets).  Every layer -- the fused kernel's staging geometry and
// conversion, the tensor maps, the tail buffers, the host staging -- takes its decision from this one enum.
//   F32: float2 I,Q
//   S16: int16 I,Q pairs (the SDRplay's / WAV's own samples, capt_sched.c:120-128), value = the int16
//   U8:  unsigned 8-bit offset-binary I,Q pairs (the RTL-SDR's rtlsdr_read_async / rtl_tcp format), value = u - 128 exactly.
//        128 rather than the converter's mid-scale 127.5 keeps the values integers, so the same capture pushed as int16 (or
//        fed to the reference) gives bit-identical results; the -0.5 LSB DC offset this leaves sits at -+14 kHz after the
//        mix, where the channel filter removes it.
enum class SampleFmt : int { F32 = 0, S16 = 1, U8 = 2 };
constexpr int kSampleFmts = 3;
__host__ __device__ constexpr int sample_bytes(SampleFmt f) { return f == SampleFmt::F32 ? 8 : f == SampleFmt::S16 ? 4 : 2; }

// Staging geometry per input sample format.  float2 input: 8 B / sample, 2 steps = 448 B (+16 B pad) per row.
// short2 input: 4 B / sample, 2 steps = 224 B (+16 B pad) per row.  8-bit input: 2 B / sample, 2 steps = 112 B (+32 B pad)
// per row; a 28-sample step is 56 B, not a whole number of 16-byte reads, so the 8-bit rows are read per 2-step stage
// (7 x LDS.128).  All three pads make the per-lane LDS.128 row reads bank-conflict free (row pitch = 4 or 28 words mod
// 32).  The int16 variant is FP32-issue-bound, not HBM-bound (4.06 B / sample), so short rows cost it nothing, while a loop
// body of more than two steps would outgrow the 32 KB L1.5 instruction cache -- with one warp per SM sub-partition an
// instruction fetch from L2 is not hidden (measured: 5 steps per stage = 5.3 ms, 2 steps = 3.3 ms per block).  Being
// issue-bound it also wants more warps per sub-partition: 12 warps x 2 stages = 2.77 ms, 8 x 3 = 2.90 ms, 16 x 1 = 2.81 ms,
// 4 warps x 6 stages = 3.27 ms.  The 8-bit variant runs the same arithmetic on half the bytes; its CTA shapes are the int16
// ones (DESIGN.md 3.1 has the sweep).
template <SampleFmt kFmt, int kClass = 0, int kCh = 2>
struct InFmt {
    static constexpr bool kF32 = kFmt == SampleFmt::F32;
    static constexpr int kSteps = kF32 ? NVX_STEPS_PER_STAGE : NVX_S16_STEPS_PER_STAGE;   // 28-sample steps per TMA box row
    static constexpr int kSampleBytes = sample_bytes(kFmt);
    static constexpr int kStepBytes = kStepIn * kSampleBytes;
    static constexpr int kStageIn = kSteps * kStepIn;                                     // input samples per stream per stage
    static constexpr int kPadBytes = kF32 ? NVX_ROW_PAD_FLOATS * 4 : kFmt == SampleFmt::S16 ? NVX_S16_ROW_PAD_BYTES : NVX_U8_ROW_PAD_BYTES;
    static constexpr int kRowBytes = kSteps * kStepBytes + kPadBytes;
    static constexpr int kBoxElems = kRowBytes / 4;                                       // TMA box width in 32-bit elements (pad over-fetched)
    static constexpr int kStageBytes = 32 * kRowBytes;                                    // per warp per stage
    // the medium tap class needs ~250 registers per thread: 4 warps per CTA for either format; three or four channels sharing
    // stage 1 need ~200: at most 8 warps per CTA
    static constexpr int kStages = kF32 ? NVX_STAGES : (kClass != 0 ? 6 : kCh > 2 ? 3 : kFmt == SampleFmt::S16 ? NVX_S16_STAGES : NVX_U8_STAGES);
    static constexpr int kWarps = kF32 ? NVX_WARPS_PER_CTA : (kClass != 0 ? 4 : kCh > 2 ? 8 : kFmt == SampleFmt::S16 ? NVX_S16_WARPS_PER_CTA : NVX_U8_WARPS_PER_CTA);      // per CTA
    static constexpr int kSmemBytes = kWarps * kStages * kStageBytes + kWarps * kStages * 8;
    static_assert(kStepsPerSuper % kSteps == 0, "a stage must not straddle superblocks");
    static_assert(kRowBytes % 16 == 0 && kStageBytes % 128 == 0 && kBoxElems <= 256, "TMA box alignment");
    static_assert((kSteps * kStepBytes) % 16 == 0, "a stage row is read in whole 16-byte loads");
    static_assert(kSmemBytes <= 227 * 1024, "shared memory per CTA");
};
// Tap-length classes of the fused kernel.  Class 0 = the reference lengths 37 / 47 / 71 (taps may be immediates); class 1 =
// "medium" replacement sets up to 61 / 75 / 111 taps (1.6x the reference: ~83 flop per input sample, which is where the
// kernel turns from HBM-bound to FP32-bound).  Shorter sets are zero-padded at the old end; longer ones take the long-tap
// path (fir_long.cu).  Everything the kernel needs follows from the three lengths:
template <int kClass> struct TapClass;
template <> struct TapClass<0> { static constexpr int T1 = NVX_T1, T2 = NVX_T2, T3 = NVX_T3; };
template <> struct TapClass<1> { static constexpr int T1 = 61, T2 = 75, T3 = 111; };
constexpr int kTapClasses = 2;
template <int kClass>
struct Geo {
    static constexpr int T1 = TapClass<kClass>::T1, T2 = TapClass<kClass>::T2, T3 = TapClass<kClass>::T3;
    // partial sums carried between 28-sample steps (transposed form): outputs still waiting for newer samples
    static constexpr int kLive1 = (T1 - 1) / NVX_D1, kLive2 = (T2 - 1) / NVX_D2, kLive3 = (T3 - 1) / NVX_D3 + 1;
    // a 900 Hz output depends on (T3 - 1) 28 + (T2 - 1) 4 + T1 input samples, 280 of them in its own superblock
    static constexpr int kWarm = ((T3 - 1) * kStepIn + (T2 - 1) * NVX_D1 + T1 - kSuper + kSuper - 1) / kSuper;
};
static_assert(Geo<0>::kLive1 == 9 && Geo<0>::kLive2 == 6 && Geo<0>::kLive3 == 8 && Geo<0>::kWarm == 7, "reference geometry");
constexpr int kMaxWarm = Geo<kTapClasses - 1>::kWarm;

__device__ constexpr double kH1[NVX_T1] = {NVX_H1_VALUES};
__device__ constexpr double kH2[NVX_T2] = {NVX_H2_VALUES};

// runtime tap sets (constant bank, uniform operands), zero-padded to the class lengths
template <int kClass>
struct TapSet {
    float h1[Geo<kClass>::T1 + 3];
    float h2[Geo<kClass>::T2 + 1];
    // stage-3 taps regrouped per step position: h3t[r][j] = h3[10 j + 9 - r] (0 where that index is beyond the set),
    // so the taps one step needs are a few aligned 16-byte uniform loads
    float h3t[NVX_D3][(Geo<kClass>::kLive3 + 3) / 4 * 4];
};
// (cos, -sin) of 2 pi k 14000 / 63000, k = 0..8, repeated so that [phase + q], q < 7 needs no wrap
struct NcoTable { float2 w[kNcoPeriod + NVX_D2]; };


// Per-stream channel offsets other than the reference's +-14 kHz (fir2cpp.C:12-14 generalised): the phase of stage-1
// output k is k * f / 63000 turns, tracked exactly as an integer numerator over 126000 (f on a 0.5 Hz grid); every
// 28-sample step re-seeds the phasor from that exact phase (sincospif) and advances it by six complex multiplies.
constexpr int kNcoDen = 126000;
// one entry per (stream, channel), [S][channels]: any number of channels can share stage 1 (SURVEY.md 8f.4); the fused kernel's
// general-NCO variants and the long-tap path's stage 1 (two channels: entries 2 row + c) read the same array
struct NcoChan {
    int num;           // (2 f) mod 126000
    // (-(E0 / 4) num) mod 126000, added to every exact phase numerator: the row's phase is 0 at its epoch E0 (input samples;
    // nvx_engine_reset_streams), as in an engine created there.  0 from create and nvx_engine_reset.
    int phase0;
    float2 step;       // (cos, -sin)(2 pi f / 63000)
};
constexpr int kMaxFusedCh = 4;   // channels one pass of the fused kernel carries in registers (9 + 14 per channel complex partial sums)
constexpr int kMaxChannels = 8;  // per capture: more than four take two passes over the input

struct CascadeArgs {
    CUtensorMap map_x;    // 32-bit view [S][2 n] (float2 input), [S][n] (short2) or [S][n / 2] (8-bit pairs) of this chunk, box InFmt::kBoxElems x 32
    CUtensorMap map_tail; // same view of [S][halo]: the halo = 280 kWarm samples that preceded the chunk (zeros at start)
    float2* y3;           // [S][2][y3_pitch] 900 Hz output; this chunk's samples start at y3_off
    long long n;          // samples per stream in this chunk (multiple of kSuper)
    int streams;
    int segs;             // time segments per stream
    int seg_super;        // superblocks per segment (last one may be short)
    int n_super;          // n / kSuper
    int sb_phase;         // (absolute superblock index of chunk start) mod 9
    long long sb_abs;     // absolute superblock index of chunk start
    const NcoChan* nco;   // [S][ch_total] per-stream NCO (kernel variants with kGenNco), else null
    long long y3_pitch;
    long long y3_off;
    int ch_total;         // channels per stream (rows of y3 per stream)
    int ch0;              // first channel this launch computes (it computes kCh of them)
};

// Everything a launch needs travels in the kernel parameter block (constant bank 0, __grid_constant__): the tap set and the NCO
// table are PER ENGINE, so engines with different filters can be alive on one device at the same time.  Taps are read as
// constant-bank operands of the FFMA2s exactly as they would be from a __constant__ symbol.
template <int kClass>
struct CascadeParams {
    CascadeArgs a;
    TapSet<kClass> taps;
    NcoTable nco;
};
static_assert(sizeof(CascadeParams<kTapClasses - 1>) <= 4096, "kernel parameter block");

// ---- host side (fir_cascade.cu) ----
// what a call of either FIR path (the fused one below, the long-tap one of fir_long.cuh) reports to the engine
struct PathReport {
    long long launches = 0;   // nvx_stats.aux_launches: every launch of the call but the fused path's first channel pass
    long long fallbacks = 0;  // stage launches meant for the tensor-core kernel that ran on the CUDA-core one (nvx_stats.long_tc_fallbacks)
    char msg[256] = "";       // for nvx_last_error(): why the call failed, else a "note: ..." about a tensor-core fallback, else empty
};
int say(PathReport* rep, int code, const char* fmt, ...);     // rep->msg = the formatted message; returns code
// what a path carries into the next block: region k of stream s is base[k][s words[k] .. + words[k]); setting a stream's regions
// to fill[k] restarts its filters after silence (nvx_engine_reset_streams)
struct CarriedRows { uint32_t* base[3]; long long words[3]; uint32_t fill[3]; };

// the driver's tiled tensor-map encoder (looked up once), or null when the driver has none
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder();
// entry k of the reference's NCO table: (cos, -sin)(2 pi k 14000 / 63000), fir2cpp.C:105-106, rounded once to float
float2 reference_nco(int k);
extern const double* const kRefTaps[3];      // the reference tap sets of stages 1, 2 and 3 (NVX_H*_VALUES)
// 64-bit hash of n bytes, continuing from h: every step is a bijection of the running value, so changing any one 8-byte word
// (or tail byte) changes the result (saved stream state: checksum and tap fingerprint)
constexpr uint64_t kHashSeed = 1469598103934665603ULL;
uint64_t hash_bytes(const void* p, size_t n, uint64_t h = kHashSeed);

int cascade_tap_class(int n1, int n2, int n3);   // tap class a set of lengths needs, or -1 if it takes the long-tap path

// ---- the fused path of one engine (S streams, C channels each): it owns the tap set, the carried input tail with its tensor
// maps, and the launch policy (time segments, channel passes) ----
struct CascadePath;
// n[k] taps of stage k + 1, h[k] = null for the reference taps; nco = the engine's [S][C] per-stream offsets, or null for the
// reference table (not owned: retunes and resets write it); reserved_sms SMs are left to the sequential demod kernels.  Returns 0
// or an NVX_ERR_* code.
int cascade_path_create(int S, int C, const int n[3], const double* const h[3], const NcoChan* nco, int device, int reserved_sms,
                        CascadePath** out, PathReport* rep);
void cascade_path_reset(CascadePath* cp);        // the next block starts after silence, in whatever format it comes
// the carried tails hold format fmt: if they hold another (or none), both are filled with its silence and described to the TMA
// unit again, queued on `stream`.  Every run does this first; a load of saved state into a fresh engine does it before the
// state's tails are written.  Returns 0 or an NVX_ERR_* code.
int cascade_path_prepare(CascadePath* cp, SampleFmt fmt, cudaStream_t stream, PathReport* rep);
CarriedRows cascade_path_carried(const CascadePath* cp);
uint64_t cascade_path_taps_hash(const CascadePath* cp);   // of the tap set as the kernels read it (class, zero padding included)
// one block x[S][n] in format fmt that starts at 900 Hz sample sb_abs; the 900 Hz output goes to y3[C S][y3_pitch] from y3_off
// on.  after_fir (if not null) is recorded once the FIR work is queued, before the tail carry.  Returns 0 or an NVX_ERR_* code.
int cascade_path_run(CascadePath* cp, const void* x, long long n, SampleFmt fmt, long long sb_abs, float2* y3, long long y3_pitch,
                     long long y3_off, cudaStream_t stream, cudaEvent_t after_fir, PathReport* rep);
void cascade_path_free(CascadePath* cp);

#ifdef NVX_CASCADE_DEVICE_CODE

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

template <bool kImm, int kClass> __device__ __forceinline__ float tap1(const TapSet<kClass>& ts, int i) { return kImm ? (float)kH1[i] : ts.h1[i]; }
template <bool kImm, int kClass> __device__ __forceinline__ float tap2(const TapSet<kClass>& ts, int i) { return kImm ? (float)kH2[i] : ts.h2[i]; }

__device__ __forceinline__ float2 fma2(float2 a, float s, float2 c) { return __ffma2_rn(a, make_float2(s, s), c); }

template <int kClass, int kCh>
struct CascadeState {
    float2 a1[Geo<kClass>::kLive1];
    float2 a2[kCh][Geo<kClass>::kLive2];
    float2 a3[kCh][Geo<kClass>::kLive3];
};

// One step: 28 inputs of one row -> 7 stage-1 outputs -> mix -> one stage-2 output per channel ->
// scattered into the stage-3 partial sums.  r10 = position of this step inside its superblock.
// y3 is written when r10 == 9 completed a 900 Hz sample.
// Per-lane phasors of the general NCO (unused by the reference-table variants)
template <int kCh>
struct NcoLane {
    float2 w[kCh];    // current (cos, -sin) per channel
    float2 step[kCh];
};

// (double)short of capt_sched.c:511, exact in float, without the quarter-rate I2F unit: flip the sign bits (offset
// binary u = v + 32768), drop each half under the exponent of 2^23 (PRMT), subtract 2^23 + 32768 with one packed add
__device__ __forceinline__ float2 iq_of(int packed) {
    const unsigned w = (unsigned)packed ^ 0x80008000u;
    const float2 biased = make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7610)),
                                      __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7632)));
    return __fadd2_rn(biased, make_float2(-8421376.0f, -8421376.0f));
}

// 8-bit offset binary u -> u - 128, exact, also without I2F: PRMT puts u in the low mantissa byte of 2^23 (2^23 + u), one
// packed add of -(2^23 + 128) per I,Q pair finishes it.  No sign flip: the data is offset binary already.
__device__ __forceinline__ float2 iq_of_u8(unsigned w, unsigned sel_i, unsigned sel_q) {
    const float2 biased = make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, sel_i)), __uint_as_float(__byte_perm(w, 0x4B000000u, sel_q)));
    return __fadd2_rn(biased, make_float2(-8388736.0f, -8388736.0f));
}

// the four input samples that complete stage-1 output q of step u, read from this lane's row of the ring stage
template <SampleFmt kFmt>
__device__ __forceinline__ void load_quad(const uint8_t* stage_row, int u, int q, float2 (&xs)[4]) {
    if constexpr (kFmt == SampleFmt::F32) {
        const float4* row = reinterpret_cast<const float4*>(stage_row + u * InFmt<kFmt>::kStepBytes);
        const float4 v0 = row[2 * q], v1 = row[2 * q + 1];
        xs[0] = make_float2(v0.x, v0.y); xs[1] = make_float2(v0.z, v0.w);
        xs[2] = make_float2(v1.x, v1.y); xs[3] = make_float2(v1.z, v1.w);
    } else if constexpr (kFmt == SampleFmt::S16) {
        const int4 v = reinterpret_cast<const int4*>(stage_row + u * InFmt<kFmt>::kStepBytes)[q];
        xs[0] = iq_of(v.x); xs[1] = iq_of(v.y); xs[2] = iq_of(v.z); xs[3] = iq_of(v.w);
    } else {
        // 8 B per quad: quad c = 7 u + q of the stage is one half of the stage row's 16-byte word c / 2 (u and q are
        // compile-time constants, so the two halves of a word come from the same LDS.128)
        const int c = 7 * u + q;
        const int4 v = reinterpret_cast<const int4*>(stage_row)[c >> 1];
        const unsigned w0 = (unsigned)((c & 1) ? v.z : v.x), w1 = (unsigned)((c & 1) ? v.w : v.y);
        xs[0] = iq_of_u8(w0, 0x7440, 0x7441); xs[1] = iq_of_u8(w0, 0x7442, 0x7443);
        xs[2] = iq_of_u8(w1, 0x7440, 0x7441); xs[3] = iq_of_u8(w1, 0x7442, 0x7443);
    }
}

template <bool kImm, bool kGenNco, SampleFmt kFmt, int kClass, int kCh>
__device__ __forceinline__ void cascade_step(const TapSet<kClass>& ts, const NcoTable& nco, CascadeState<kClass, kCh>& st,
                                             const uint8_t* __restrict__ stage_row, const int u, int nco_phase, const int r10, float2 (&y3)[kCh], NcoLane<kCh>& nl) {
    using G = Geo<kClass>;
    constexpr int kLive1 = G::kLive1, kLive2 = G::kLive2, kLive3 = G::kLive3;
    static_assert(!kImm || kClass == 0, "immediate taps are the reference set");
    static_assert(kGenNco || kCh == 2, "the reference's 9-entry table serves exactly its two channels (+14 kHz and its conjugate)");
    float2 w[kLive1 + NVX_D2];
#pragma unroll
    for (int j = 0; j < kLive1; ++j) w[j] = st.a1[j];
#pragma unroll
    for (int j = kLive1; j < kLive1 + NVX_D2; ++j) w[j] = make_float2(0.f, 0.f);

    float2 b[kCh][kLive2 + 1];
#pragma unroll
    for (int c = 0; c < kCh; ++c) {
#pragma unroll
        for (int j = 0; j < kLive2; ++j) b[c][j] = st.a2[c][j];
        b[c][kLive2] = make_float2(0.f, 0.f);
    }

#pragma unroll
    for (int q = 0; q < NVX_D2; ++q) {
        // four inputs complete stage-1 output q of this step
        float2 xs[4];
        load_quad<kFmt>(stage_row, u, q, xs);
#pragma unroll
        for (int r = 0; r < NVX_D1; ++r) {
#pragma unroll
            for (int j = 0; 4 * j + 3 - r < G::T1; ++j) w[q + j] = fma2(xs[r], tap1<kImm, kClass>(ts, 4 * j + 3 - r), w[q + j]);
        }
        const float2 y1 = w[q];
        // NCO mix (fir2cpp.C:115-124): ch0 = y1 * (re + j im), ch1 = y1 * (re - j im), (re, im) = (cos, -sin)
        float2 m[kCh];
        if (kGenNco) {
#pragma unroll
            for (int c = 0; c < kCh; ++c) {
                const float2 rot = nl.w[c];
                m[c] = make_float2(fmaf(-y1.y, rot.y, y1.x * rot.x), fmaf(y1.x, rot.y, y1.y * rot.x));
                if (q + 1 < NVX_D2)     // advance the phasor: w *= step
                    nl.w[c] = make_float2(fmaf(-rot.y, nl.step[c].y, rot.x * nl.step[c].x), fmaf(rot.x, nl.step[c].y, rot.y * nl.step[c].x));
            }
        } else {
            const float2 rot = nco.w[nco_phase + q];
            const float ar = y1.x * rot.x, br = y1.y * rot.x;
            m[0] = make_float2(fmaf(-y1.y, rot.y, ar), fmaf(y1.x, rot.y, br));
            m[kCh - 1] = make_float2(fmaf(y1.y, rot.y, ar), fmaf(-y1.x, rot.y, br));
        }
#pragma unroll
        for (int c = 0; c < kCh; ++c) {
#pragma unroll
            for (int j = 0; 7 * j + 6 - q < G::T2; ++j) b[c][j] = fma2(m[c], tap2<kImm, kClass>(ts, 7 * j + 6 - q), b[c][j]);
        }
    }
#pragma unroll
    for (int j = 0; j < kLive1; ++j) st.a1[j] = w[j + NVX_D2];

#pragma unroll
    for (int c = 0; c < kCh; ++c) {
        const float2 y2 = b[c][0];
#pragma unroll
        for (int j = 0; j < kLive2; ++j) st.a2[c][j] = b[c][j + 1];
        // stage 3: sample 10p + r10 feeds outputs p + j with tap 10 j + 9 - r10 (table row r10; the last j only
        // carries a non-zero tap for the largest r10)
#pragma unroll
        for (int j = 0; j < kLive3; ++j) st.a3[c][j] = fma2(y2, ts.h3t[r10][j], st.a3[c][j]);
    }
    if (r10 == NVX_D3 - 1) {
#pragma unroll
        for (int c = 0; c < kCh; ++c) {
            y3[c] = st.a3[c][0];
#pragma unroll
            for (int j = 1; j < kLive3; ++j) st.a3[c][j - 1] = st.a3[c][j];
            st.a3[c][kLive3 - 1] = make_float2(0.f, 0.f);
        }
    }
}

#endif  // NVX_CASCADE_DEVICE_CODE

}  // namespace nvx

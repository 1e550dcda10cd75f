// fir_cascade.cu -- kernel + launcher for the fused FIR cascade (see fir_cascade.cuh).
#define NVX_CASCADE_DEVICE_CODE
#include "fir_cascade.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "../../include/navtex_b200.h"

namespace nvx {

template <bool kImm, bool kGenNco, SampleFmt kFmt, int kClass, int kCh>
__global__ void __launch_bounds__(InFmt<kFmt, kClass, kCh>::kWarps * 32, kCtasPerSm) fir_cascade_kernel(const __grid_constant__ CascadeParams<kClass> prm) {
    const CascadeArgs& a = prm.a;
    using F = InFmt<kFmt, kClass, kCh>;
    using G = Geo<kClass>;
    constexpr int kWarmSuper = G::kWarm, kHalo = G::kWarm * kSuper, kLive1 = G::kLive1, kLive2 = G::kLive2, kLive3 = G::kLive3;
    constexpr int kWarpsPerCta = F::kWarps;
    constexpr int kStages = F::kStages, kStageBytes = F::kStageBytes, kStepsPerStage = F::kSteps, kStageIn = F::kStageIn;
    constexpr int kRowBytes = F::kRowBytes;
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* const wbase = smem + (size_t)warp * (kStages * kStageBytes);
    const uint32_t wbase_s = smem_u32(wbase);
    const uint32_t bar0 = smem_u32(smem + (size_t)kWarpsPerCta * kStages * kStageBytes) + warp * kStages * 8;

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    // warp -> (group of 32 consecutive streams, time segment); lane -> stream inside the group
    const int groups = (a.streams + 31) >> 5;
    const long long wg = (long long)blockIdx.x * kWarpsPerCta + warp;
    if (wg >= (long long)groups * a.segs) return;
    const int seg = (int)(wg / groups);
    const int strm0 = (int)(wg % groups) * 32;
    const int strm = strm0 + lane;
    const int first_sb = seg * a.seg_super;
    int my_super = a.n_super - first_sb;
    my_super = my_super > a.seg_super ? a.seg_super : my_super;
    if (strm >= a.streams) my_super = 0;          // padding lanes compute on TMA zero fill, store nothing

    const int warp_stages = (kWarmSuper + a.seg_super) * (kStepsPerSuper / kStepsPerStage);
    // first input sample of this segment's warm-up, relative to the chunk start (negative = carried tail)
    const long long pos0 = ((long long)first_sb - kWarmSuper) * kSuper;

    // sample position -> 32-bit element of the tensor map (8-bit pairs: two samples per element; stage positions and the halo
    // are multiples of 56, so the division is exact)
    auto elem = [](long long p) { return (int)(p * F::kSampleBytes / 4); };
    auto issue = [&](int t, int stage) {
        if (lane == 0) {
            const uint32_t bar = bar0 + 8 * stage;
            const long long p = pos0 + (long long)t * kStageIn;
            mbar_arrive_expect_tx(bar, kStageBytes);
            if (p < 0) tma_load_2d(wbase_s + stage * kStageBytes, &a.map_tail, elem(p + kHalo), strm0, bar);
            else       tma_load_2d(wbase_s + stage * kStageBytes, &a.map_x, elem(p), strm0, bar);
        }
    };

#pragma unroll
    for (int s = 0; s < kStages; ++s)
        if (s < warp_stages) issue(s, s);

    CascadeState<kClass, kCh> st;
#pragma unroll
    for (int j = 0; j < kLive1; ++j) st.a1[j] = make_float2(0.f, 0.f);
#pragma unroll
    for (int c = 0; c < kCh; ++c) {
#pragma unroll
        for (int j = 0; j < kLive2; ++j) st.a2[c][j] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < kLive3; ++j) st.a3[c][j] = make_float2(0.f, 0.f);
    }

    // NCO phase of the first stage-1 output of a step: (70 sb_abs + 7 r10) mod 9, sb_abs = absolute
    // superblock index; identical for every lane (same time position, all streams share the chunk clock).
    int phase = (7 * ((a.sb_phase + first_sb + 9 * kWarmSuper - kWarmSuper) % kNcoPeriod)) % kNcoPeriod;
    // general NCO: exact phase numerators of this lane's two channels at the first stage-1 output of the warm-up
    NcoLane<kCh> nl = {};
    int nco_idx[kCh] = {}, nco_adv[kCh] = {};
    if (kGenNco) {
        const NcoChan* np = a.nco + (size_t)(strm < a.streams ? strm : a.streams - 1) * a.ch_total + a.ch0;
        long long k0 = ((a.sb_abs + first_sb - kWarmSuper) * (long long)(kSuper / NVX_D1)) % kNcoDen;    // 70 outputs per superblock
        if (k0 < 0) k0 += kNcoDen;
#pragma unroll
        for (int c = 0; c < kCh; ++c) {
            const NcoChan pc = np[c];
            nco_idx[c] = (int)((k0 * pc.num + pc.phase0) % kNcoDen);
            nco_adv[c] = (int)(((long long)NVX_D2 * pc.num) % kNcoDen);
            nl.step[c] = pc.step;
        }
    }
    int stage = 0;
    uint32_t parity = 0;
    float2* const y3row = a.y3 + ((size_t)strm * a.ch_total + a.ch0) * a.y3_pitch + a.y3_off + first_sb;

    float2 y3[kCh];
#pragma unroll
    for (int c = 0; c < kCh; ++c) y3[c] = make_float2(0.f, 0.f);
    int r10 = 0, out = -kWarmSuper;
    for (int t = 0; t < warp_stages; ++t) {
        mbar_wait(bar0 + 8 * stage, parity);
        const uint8_t* rowb = wbase + stage * kStageBytes + lane * kRowBytes;
#pragma unroll
        for (int u = 0; u < kStepsPerStage; ++u) {
            if (kGenNco) {
#pragma unroll
                for (int c = 0; c < kCh; ++c) {
                    float t = (float)nco_idx[c] * (2.0f / kNcoDen);      // turns * 2, in [0, 2)
                    if (t > 1.0f) t -= 2.0f;
                    float sn, cs;
                    sincospif(t, &sn, &cs);
                    nl.w[c] = make_float2(cs, -sn);
                    nco_idx[c] += nco_adv[c];
                    if (nco_idx[c] >= kNcoDen) nco_idx[c] -= kNcoDen;
                }
            }
            cascade_step<kImm, kGenNco, kFmt, kClass, kCh>(prm.taps, prm.nco, st, rowb, u, phase, r10 + u, y3, nl);
            phase += 7;
            if (phase >= kNcoPeriod) phase -= kNcoPeriod;
        }
        __syncwarp();
        if (t + kStages < warp_stages) issue(t + kStages, stage);
        if (++stage == kStages) { stage = 0; parity ^= 1; }
        r10 += kStepsPerStage;
        if (r10 == kStepsPerSuper) {
            r10 = 0;
            if (out >= 0 && out < my_super) {
#pragma unroll
                for (int c = 0; c < kCh; ++c) y3row[c * a.y3_pitch + out] = y3[c];
            }
            ++out;
        }
    }
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
template <typename Sample>
static cudaError_t tail_carry(const void* old_tail, const void* x, void* new_tail, int streams, long long n, int halo, cudaStream_t stream) {
    const long long work = (long long)streams * (halo / (16 / (int)sizeof(Sample)));
    tail_carry_kernel<Sample><<<(unsigned)((work + 255) / 256), 256, 0, stream>>>(static_cast<const Sample*>(old_tail), static_cast<const Sample*>(x),
                                                                                 static_cast<Sample*>(new_tail), streams, n, halo);
    return cudaGetLastError();
}

int say(PathReport* rep, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(rep->msg, sizeof rep->msg, fmt, ap);
    va_end(ap);
    return code;
}
static int check(PathReport* rep, cudaError_t e, const char* what) {
    return e == cudaSuccess ? 0 : say(rep, NVX_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
}

EncodeTiledFn tensor_map_encoder() {
    static const EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        const cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
        return e == cudaSuccess && q == cudaDriverEntryPointSuccess ? (EncodeTiledFn)p : nullptr;
    }();
    return fn;
}

float2 reference_nco(int k) { return make_float2((float)cos((2 * M_PI * k * 14000) / 63000), (float)-sin((2 * M_PI * k * 14000) / 63000)); }

static const double kRef1[NVX_T1] = {NVX_H1_VALUES}, kRef2[NVX_T2] = {NVX_H2_VALUES}, kRef3[NVX_T3] = {NVX_H3_VALUES};
const double* const kRefTaps[3] = {kRef1, kRef2, kRef3};

uint64_t hash_bytes(const void* p, size_t n, uint64_t h) {
    const uint8_t* b = static_cast<const uint8_t*>(p);
    for (; n >= 8; n -= 8, b += 8) {
        uint64_t w;
        memcpy(&w, b, 8);
        h = (h ^ w) * 0x100000001b3ULL;
        h ^= h >> 29;
    }
    for (; n; --n, ++b) {
        h = (h ^ *b) * 0x100000001b3ULL;
        h ^= h >> 29;
    }
    return h;
}

// 32-bit-element view of a stream-major sample array: [rows][2 * cols] floats for float2 samples, [rows][cols] words for
// short2 samples (one word = one I,Q pair), [rows][cols / 2] words for 8-bit pairs (one word = two pairs; cols is a multiple
// of 280); box = one ring stage x 32 rows
static int encode_rows(CUtensorMap* map, const void* base, long long cols, long long rows, SampleFmt f, PathReport* rep) {
    const EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return say(rep, NVX_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    const long long row_bytes = cols * sample_bytes(f);
    const int box_elems = f == SampleFmt::F32 ? InFmt<SampleFmt::F32>::kBoxElems : f == SampleFmt::S16 ? InFmt<SampleFmt::S16>::kBoxElems : InFmt<SampleFmt::U8>::kBoxElems;
    cuuint64_t dims[2] = {(cuuint64_t)(row_bytes / 4), (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
    cuuint32_t box[2] = {(cuuint32_t)box_elems, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, f == SampleFmt::F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return say(rep, NVX_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) cols=%lld rows=%lld", (int)r, cols, rows);
    return 0;
}

// host-side copy of an engine's filter constants (both classes' layouts; only the engine's own class is filled)
struct CascadeTaps {
    TapSet<0> t0;
    TapSet<1> t1;
    NcoTable nco;
};

// pad a tap set with zeros at the old end up to the class length (a shorter FIR is the same FIR with zero taps)
template <int kClass>
static void fill_taps(const double* h1, int n1, const double* h2, int n2, const double* h3, int n3, TapSet<kClass>* t) {
    using G = Geo<kClass>;
    for (int i = 0; i < G::T1 + 3; ++i) t->h1[i] = i < n1 ? (float)h1[i] : 0.f;
    for (int i = 0; i < G::T2 + 1; ++i) t->h2[i] = i < n2 ? (float)h2[i] : 0.f;
    for (int r = 0; r < NVX_D3; ++r)
        for (int j = 0; j < (int)(sizeof t->h3t[0] / sizeof(float)); ++j) {
            const int i = 10 * j + 9 - r;
            t->h3t[r][j] = i < n3 ? (float)h3[i] : 0.f;
        }
}

int cascade_tap_class(int n1, int n2, int n3) {
    if (n1 <= Geo<0>::T1 && n2 <= Geo<0>::T2 && n3 <= Geo<0>::T3) return 0;
    if (n1 <= Geo<1>::T1 && n2 <= Geo<1>::T2 && n3 <= Geo<1>::T3) return 1;
    return -1;
}

template <SampleFmt kFmt, int kClass, int kCh>
static cudaError_t launch_fmt(const CascadeArgs& a, const CascadeTaps& taps, bool custom_taps, cudaStream_t stream) {
    const size_t smem = InFmt<kFmt, kClass, kCh>::kSmemBytes;
    // more than two channels always run the general (per-channel) NCO; two channels use the reference's table unless offsets were given
    const bool gen = a.nco != nullptr;
    // immediates only for the reference taps themselves; every other set (class 0 or 1) reads the constant bank
    constexpr bool kCanImm = kClass == 0;
    constexpr bool kTable = kCh == 2;          // the table variants exist for exactly two channels
    auto kern = (gen || !kTable)
                    ? ((custom_taps || !kCanImm) ? fir_cascade_kernel<false, true, kFmt, kClass, kCh> : fir_cascade_kernel<kCanImm, true, kFmt, kClass, kCh>)
                    : ((custom_taps || !kCanImm) ? fir_cascade_kernel<false, !kTable, kFmt, kClass, kCh> : fir_cascade_kernel<kCanImm, !kTable, kFmt, kClass, kCh>);
    if (!gen && !kTable) return cudaErrorInvalidValue;
    {   // function attributes are per device: set on every launch (cheap) rather than cached process-wide
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    constexpr int kWarpsPerCta = InFmt<kFmt, kClass, kCh>::kWarps;
    const long long warps = (long long)((a.streams + 31) / 32) * a.segs;
    const unsigned grid = (unsigned)((warps + kWarpsPerCta - 1) / kWarpsPerCta);
    CascadeParams<kClass> prm;
    prm.a = a;
    if constexpr (kClass == 1) prm.taps = taps.t1; else prm.taps = taps.t0;
    prm.nco = taps.nco;
    kern<<<grid, kWarpsPerCta * 32, smem, stream>>>(prm);
    return cudaGetLastError();
}

template <int kClass, int kCh>
static cudaError_t launch_cls(SampleFmt f, const CascadeArgs& a, const CascadeTaps& taps, bool custom_taps, cudaStream_t stream) {
    switch (f) {
        case SampleFmt::F32: return launch_fmt<SampleFmt::F32, kClass, kCh>(a, taps, custom_taps, stream);
        case SampleFmt::S16: return launch_fmt<SampleFmt::S16, kClass, kCh>(a, taps, custom_taps, stream);
        default: return launch_fmt<SampleFmt::U8, kClass, kCh>(a, taps, custom_taps, stream);
    }
}

// n_ch = channels of this launch (a.ch0 .. a.ch0 + n_ch - 1): 2 in either tap class, 1 / 3 / 4 in the reference class
static cudaError_t cascade_launch(const CascadeArgs& a, const CascadeTaps& taps, int tap_class, bool custom_taps, SampleFmt f, int n_ch, cudaStream_t stream) {
    if (tap_class == 1) {
        if (n_ch != 2) return cudaErrorInvalidValue;
        return launch_cls<1, 2>(f, a, taps, true, stream);
    }
    switch (n_ch) {
        case 1: return launch_cls<0, 1>(f, a, taps, custom_taps, stream);
        case 2: return launch_cls<0, 2>(f, a, taps, custom_taps, stream);
        case 3: return launch_cls<0, 3>(f, a, taps, custom_taps, stream);
        case 4: return launch_cls<0, 4>(f, a, taps, custom_taps, stream);
        default: return cudaErrorInvalidValue;
    }
}

// warps that are resident at once across the device, leaving `reserved_sms` SMs to the sequential demod kernels:
// the host sizes the grid to at most one full wave
template <SampleFmt kFmt, int kClass, int kCh>
static int target_warps_fmt(int device, int reserved_sms) {
    using F = InFmt<kFmt, kClass, kCh>;
    int sms = 148, per_sm = kCtasPerSm;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    auto kern = fir_cascade_kernel<false, true, kFmt, kClass, kCh>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, F::kSmemBytes);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, F::kWarps * 32, F::kSmemBytes) != cudaSuccess || per_sm < 1)
        per_sm = kCtasPerSm;
    if (sms - reserved_sms >= 8) sms -= reserved_sms;
    return sms * per_sm * F::kWarps;
}
template <int kClass, int kCh>
static int target_warps_cls(int device, int reserved_sms, SampleFmt f) {
    switch (f) {
        case SampleFmt::F32: return target_warps_fmt<SampleFmt::F32, kClass, kCh>(device, reserved_sms);
        case SampleFmt::S16: return target_warps_fmt<SampleFmt::S16, kClass, kCh>(device, reserved_sms);
        default: return target_warps_fmt<SampleFmt::U8, kClass, kCh>(device, reserved_sms);
    }
}
// heavy = a launch carries three or four channels (different CTA shape for integer input)
static int target_warps(int device, int reserved_sms, SampleFmt f, int tap_class, bool heavy) {
    if (tap_class == 1) return target_warps_cls<1, 2>(device, reserved_sms, f);
    if (heavy) return target_warps_cls<0, 4>(device, reserved_sms, f);
    return target_warps_cls<0, 2>(device, reserved_sms, f);
}

// ---- the fused path of one engine ----

struct CascadePath {
    int S = 0, C = 2;                     // streams, channels per stream
    int tap_class = 0;                    // 0 or 1 (Geo<>)
    bool custom_taps = false;             // not the reference set: the taps come from the constant bank, not immediates
    CascadeTaps taps;                     // passed in the parameter block of every launch
    int halo = 0;                         // carried input samples per stream: 280 x the class's warm-up superblocks
    // carried input tail, ping-pong, in the sample format being pushed: [S][halo] float2, short2 or 8-bit pairs (each buffer
    // sized for float2); filled with silence and described to the TMA unit when a block in another format arrives
    void* tail[2] = {};
    CUtensorMap map_tail[2];
    int cur = 0;
    int fmt = -1;                         // the SampleFmt the tails hold, -1 = none (after create and reset)
    int target_warps[kSampleFmts] = {};   // resident cascade warps per sample format
    const NcoChan* nco = nullptr;         // the engine's [S][C] per-stream offsets, or null: the reference table
};

int cascade_path_create(int S, int C, const int n[3], const double* const h[3], const NcoChan* nco, int device, int reserved_sms,
                        CascadePath** out, PathReport* rep) {
    const int cls = cascade_tap_class(n[0], n[1], n[2]);
    if (cls < 0) return say(rep, NVX_ERR_ARG, "%d / %d / %d taps do not fit the fused kernel", n[0], n[1], n[2]);
    const double* hh[3] = {h[0] ? h[0] : kRefTaps[0], h[1] ? h[1] : kRefTaps[1], h[2] ? h[2] : kRefTaps[2]};
    CascadePath* cp = new CascadePath();
    cp->S = S; cp->C = C; cp->nco = nco;
    cp->tap_class = cls;
    cp->custom_taps = h[0] || h[1] || h[2];
    if (cls == 1) fill_taps<1>(hh[0], n[0], hh[1], n[1], hh[2], n[2], &cp->taps.t1);
    else fill_taps<0>(hh[0], n[0], hh[1], n[1], hh[2], n[2], &cp->taps.t0);
    for (int i = 0; i < kNcoPeriod + NVX_D2; ++i) cp->taps.nco.w[i] = reference_nco(i % kNcoPeriod);
    cp->halo = kSuper * (cls == 1 ? Geo<1>::kWarm : Geo<0>::kWarm);
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaMalloc(&cp->tail[k], (size_t)S * cp->halo * sample_bytes(SampleFmt::F32));
    if (e != cudaSuccess) {
        cascade_path_free(cp);
        return say(rep, e == cudaErrorMemoryAllocation ? NVX_ERR_NOMEM : NVX_ERR_CUDA, "fused path: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    for (int f = 0; f < kSampleFmts; ++f) cp->target_warps[f] = target_warps(device, reserved_sms, (SampleFmt)f, cls, C > 2);
    *out = cp;
    return 0;
}

void cascade_path_reset(CascadePath* cp) {
    cp->cur = 0;
    cp->fmt = -1;
}

// the tail the next block reads; nothing while the tails hold no format: the next block fills them with silence anyway
CarriedRows cascade_path_carried(const CascadePath* cp) {
    if (cp->fmt < 0) return {};
    const SampleFmt f = (SampleFmt)cp->fmt;
    return {{static_cast<uint32_t*>(cp->tail[cp->cur])}, {(long long)cp->halo * sample_bytes(f) / 4}, {f == SampleFmt::U8 ? 0x80808080u : 0u}};
}

// the first launch is nvx_stats.cascade_launches; the second channel pass and the tail carry count in rep->launches
int cascade_path_prepare(CascadePath* cp, SampleFmt fmt, cudaStream_t stream, PathReport* rep) {
    if (cp->fmt == (int)fmt) return 0;
    // the warm-up before the first block sees silence: the value 0, which is the byte 128 in 8-bit offset binary
    for (int k = 0; k < 2; ++k) {
        if (int rc = check(rep, cudaMemsetAsync(cp->tail[k], fmt == SampleFmt::U8 ? 128 : 0, (size_t)cp->S * cp->halo * sample_bytes(fmt), stream),
                           "fused path: filling the input tail"))
            return rc;
        if (int rc = encode_rows(&cp->map_tail[k], cp->tail[k], cp->halo, cp->S, fmt, rep)) return rc;
    }
    cp->fmt = (int)fmt;
    return 0;
}

uint64_t cascade_path_taps_hash(const CascadePath* cp) {
    return cp->tap_class == 1 ? hash_bytes(&cp->taps.t1, sizeof cp->taps.t1) : hash_bytes(&cp->taps.t0, sizeof cp->taps.t0);
}

int cascade_path_run(CascadePath* cp, const void* x, long long n, SampleFmt fmt, long long sb_abs, float2* y3, long long y3_pitch,
                     long long y3_off, cudaStream_t stream, cudaEvent_t after_fir, PathReport* rep) {
    if (int rc = cascade_path_prepare(cp, fmt, stream, rep)) return rc;
    CascadeArgs ca;
    if (int rc = encode_rows(&ca.map_x, x, n, cp->S, fmt, rep)) return rc;
    ca.map_tail = cp->map_tail[cp->cur];
    const int n_super = (int)(n / kSuper);
    const int groups = (cp->S + 31) / 32;
    // time segments: enough warps to fill the machine once, but keep the 7-superblock warm-up small
    int segs = cp->target_warps[(int)fmt] / groups;            // never more warps than are resident at once (no second wave)
    const int min_seg = 63;
    if (segs > n_super / min_seg) segs = n_super / min_seg;
    if (segs < 1) segs = 1;
    const int seg_super = (n_super + segs - 1) / segs;
    segs = (n_super + seg_super - 1) / seg_super;
    ca.y3 = y3;
    ca.n = n;
    ca.streams = cp->S;
    ca.segs = segs;
    ca.seg_super = seg_super;
    ca.n_super = n_super;
    ca.sb_phase = (int)(sb_abs % kNcoPeriod);
    ca.sb_abs = sb_abs;
    ca.nco = cp->nco;
    ca.y3_pitch = y3_pitch;
    ca.y3_off = y3_off;
    ca.ch_total = cp->C;
    // up to four channels share one pass over the input (stage 1 computed once for all of them); five to eight take two
    for (int c0 = 0; c0 < cp->C;) {
        const int left = cp->C - c0;
        const int n_ch = left <= kMaxFusedCh ? left : (left + 1) / 2;      // 5 = 3 + 2, 6 = 3 + 3, 7 = 4 + 3, 8 = 4 + 4
        ca.ch0 = c0;
        if (int rc = check(rep, cascade_launch(ca, cp->taps, cp->tap_class, cp->custom_taps, fmt, n_ch, stream), "fused cascade launch")) return rc;
        if (c0) rep->launches++;
        c0 += n_ch;
    }
    if (int rc = check(rep, after_fir ? cudaEventRecord(after_fir, stream) : cudaSuccess, "cudaEventRecord")) return rc;
    const auto carry = fmt == SampleFmt::U8 ? tail_carry<uchar2> : fmt == SampleFmt::S16 ? tail_carry<short2> : tail_carry<float2>;
    if (int rc = check(rep, carry(cp->tail[cp->cur], x, cp->tail[cp->cur ^ 1], cp->S, n, cp->halo, stream), "fused path: tail carry")) return rc;
    rep->launches++;
    cp->cur ^= 1;
    return 0;
}

void cascade_path_free(CascadePath* cp) {
    if (!cp) return;
    cudaFree(cp->tail[0]); cudaFree(cp->tail[1]);
    delete cp;
}

}  // namespace nvx

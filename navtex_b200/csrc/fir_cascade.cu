// fir_cascade.cu -- kernel + launcher for the fused FIR cascade (see fir_cascade.cuh).
#define NVX_CASCADE_DEVICE_CODE
#include "fir_cascade.cuh"

#include <math.h>
#include <stdio.h>

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
            nco_idx[c] = (int)((k0 * pc.num) % kNcoDen);
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
#ifdef NVX_ROLL_STEPS
#pragma unroll 1
#else
#pragma unroll
#endif
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

int cascade_box_elems(SampleFmt f) {
    return f == SampleFmt::F32 ? InFmt<SampleFmt::F32>::kBoxElems : f == SampleFmt::S16 ? InFmt<SampleFmt::S16>::kBoxElems : InFmt<SampleFmt::U8>::kBoxElems;
}

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

// tap class a set of lengths needs, or -1 if it takes the long-tap path
int cascade_tap_class(int n1, int n2, int n3) {
    if (n1 <= Geo<0>::T1 && n2 <= Geo<0>::T2 && n3 <= Geo<0>::T3) return 0;
    if (n1 <= Geo<1>::T1 && n2 <= Geo<1>::T2 && n3 <= Geo<1>::T3) return 1;
    return -1;
}
int cascade_warm_super(int tap_class) { return tap_class == 1 ? Geo<1>::kWarm : Geo<0>::kWarm; }

// the filter constants of one engine (host side; they travel in the kernel parameter block of every launch)
void cascade_fill_taps(int tap_class, const double* h1, int n1, const double* h2, int n2, const double* h3, int n3, CascadeTaps* out) {
    static const double d1[NVX_T1] = {NVX_H1_VALUES};
    static const double d2[NVX_T2] = {NVX_H2_VALUES};
    static const double d3[NVX_T3] = {NVX_H3_VALUES};
    if (!h1) { h1 = d1; n1 = NVX_T1; }
    if (!h2) { h2 = d2; n2 = NVX_T2; }
    if (!h3) { h3 = d3; n3 = NVX_T3; }
    *out = CascadeTaps{};
    if (tap_class == 1) fill_taps<1>(h1, n1, h2, n2, h3, n3, &out->t1);
    else fill_taps<0>(h1, n1, h2, n2, h3, n3, &out->t0);
    for (int i = 0; i < kNcoPeriod + NVX_D2; ++i) {
        const int k = i % kNcoPeriod;
        // same expression as fir2cpp.C:105-106, rounded once to float
        out->nco.w[i].x = (float)cos((2 * M_PI * k * 14000) / 63000);
        out->nco.w[i].y = (float)-sin((2 * M_PI * k * 14000) / 63000);
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
int cascade_target_warps(int device, int reserved_sms, SampleFmt f, int tap_class, bool heavy) {
    if (tap_class == 1) return target_warps_cls<1, 2>(device, reserved_sms, f);
    if (heavy) return target_warps_cls<0, 4>(device, reserved_sms, f);
    return target_warps_cls<0, 2>(device, reserved_sms, f);
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
cudaError_t cascade_launch(const CascadeArgs& a, const CascadeTaps& taps, int tap_class, bool custom_taps, SampleFmt f, int n_ch, cudaStream_t stream) {
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

}  // namespace nvx

// fir_long.cu -- register-tiled polyphase decimating FIR kernels for long tap sets, and the long-tap path of an engine that
// runs them (see fir_long.cuh).
#include "fir_long.cuh"

#include <stdlib.h>
#include <string.h>

#include "../../include/navtex_b200.h"

namespace nvx {

namespace {

// taps of one stage regrouped per decimation phase + the reference NCO table: passed by value in the kernel parameter block
constexpr int kLongTapSlots = 1152;             // D * J <= 1024 + D * kLongR
struct LongStageTaps {
    float h[kLongTapSlots];
    float2 nco[kNcoPeriod];
};

// The taps of the launched stage and the reference NCO table travel in the kernel parameter block (constant bank 0,
// __grid_constant__): per engine, so engines with different tap sets can be alive on one device, and still warp-uniform
// constant-bank operands for the FFMA2 loops.

__device__ __forceinline__ float2 ffma2s(float2 a, float s, float2 c) { return __ffma2_rn(a, make_float2(s, s), c); }

__device__ __forceinline__ float2 load_sample(const LongArgs& a, int row, long long in_pitch, int H, long long g) {
    if (g < 0) return a.hist[(size_t)row * H + (H + g)];
    if (g >= a.n_in) return make_float2(0.f, 0.f);
    if (a.s16) {
        const short2 v = static_cast<const short2*>(a.in)[(size_t)row * in_pitch + g];
        return make_float2((float)v.x, (float)v.y);
    }
    return static_cast<const float2*>(a.in)[(size_t)row * in_pitch + g];
}

// Shared-memory layout of a tile: the inputs in their natural (interleaved) order, f = sample index relative to the
// tile's first input, with one pad slot after every 8 D samples: slot(f) = f + f / (8 D).  A thread's outputs are 8
// apart from its neighbour's, i.e. 8 D inputs: the pad turns that lane stride into 8 D + 1 (odd), so both the staging
// stores (consecutive f) and the window loads (fixed phase, lane stride 8 D + 1) are bank-conflict free, and the
// staging needs no de-interleaving arithmetic.
template <int D>
__device__ __forceinline__ int slot(int f) { return f + f / (kLongR * D); }

// grid (tiles, input rows).  STAGE 0 (the first stage) writes TWO output rows per input row: its 63 kHz outputs rotated by
// each channel's NCO (fir2cpp.C:112-128), so that the second stage is a plain FIR over channel rows.
template <int D, int STAGE>
__global__ void __launch_bounds__(long_threads(D)) fir_long_kernel(const LongArgs a, const int J, const long long in_pitch,
                                                                   const __grid_constant__ LongStageTaps tp) {
    constexpr int kLongThreads = long_threads(D), kLongTile = long_tile(D);
    extern __shared__ __align__(16) float2 s_x[];
    const int H = D * J;
    const int F = D * (kLongTile + J - 1);                    // inputs staged per tile
    const int row_in = blockIdx.y;
    const long long k0 = (long long)blockIdx.x * kLongTile;  // first output of the tile
    const long long n_out = a.n_in / D;
    const long long g0 = (long long)D * (k0 - J + 1);        // first input the tile needs (oldest tap of output k0)

    // ---- stage the tile: a pure copy, so float2 sources go through cp.async (every load of the tile in flight at once);
    // int16 input is converted on the way and keeps the register path ----
    if (a.s16) {
        constexpr int kBatch = 8;
        for (int base = 0; base < F; base += kLongThreads * kBatch) {
            float2 v[kBatch];
#pragma unroll
            for (int i = 0; i < kBatch; ++i) {
                const int f = base + i * kLongThreads + (int)threadIdx.x;
                v[i] = f < F ? load_sample(a, row_in, in_pitch, H, g0 + f) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < kBatch; ++i) {
                const int f = base + i * kLongThreads + (int)threadIdx.x;
                if (f < F) s_x[slot<D>(f)] = v[i];
            }
        }
    } else {
        const float2* blk = static_cast<const float2*>(a.in) + (size_t)row_in * in_pitch;
        const float2* hist = a.hist + (size_t)row_in * H + H;
        if (g0 >= 0 && g0 + F <= a.n_in) {
            // interior tile (all but the first and the last of a row): no history, no zero fill, and the pad slot of every
            // kLongR * D samples kept incrementally -- the general loop below costs ~20 instructions per sample, which at 65 taps
            // was more than the filter itself (ncu: 4 000 instructions per warp and tile for 640 FFMA2)
            constexpr int kG = kLongR * D, kStepG = kLongThreads / kG, kStepR = kLongThreads % kG;
            int grp = (int)threadIdx.x / kG, rem = (int)threadIdx.x % kG;
            const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(s_x);
            const float2* src = blk + g0 + threadIdx.x;
#pragma unroll 4
            for (int f = threadIdx.x; f < F; f += kLongThreads, src += kLongThreads) {
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s0 + 8u * (uint32_t)(f + grp)), "l"(src) : "memory");
                grp += kStepG;
                rem += kStepR;
                if (rem >= kG) { rem -= kG; ++grp; }
            }
        } else {
            for (int f = threadIdx.x; f < F; f += kLongThreads) {
                const long long g = g0 + f;
                float2* dst = s_x + slot<D>(f);
                if (g >= a.n_in) { *dst = make_float2(0.f, 0.f); continue; }
                const float2* src = g < 0 ? hist + g : blk + g;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();

    // ---- R consecutive outputs per thread ----
    // Output k0 + R t + u, tap j = jb + jj of phase p reads position R (q - 1) + (u - jj + R - 1) of that phase, q = t +
    // (J - jb) / R, i.e. input f = D pos + p.  The window win[i] holds positions R (q - 1) + i, i < 2 R - 1; since
    // D i + p < 8 D exactly when i < 8, its slots are (8 D + 1)(q - 1) + D i + p + (i >= 8).
    const int t = threadIdx.x;
    float2 acc[kLongR];
#pragma unroll
    for (int u = 0; u < kLongR; ++u) acc[u] = make_float2(0.f, 0.f);
    const float* taps = tp.h;
    constexpr int kLane = kLongR * D + 1;
#pragma unroll 1
    for (int p = 0; p < D; ++p) {
        const float* hp = taps + p * J;
        const float2* sp = s_x + kLane * (t + J / kLongR - 1) + p;     // window base of tap block 0
        float2 win[2 * kLongR - 1];
#pragma unroll
        for (int i = 0; i < 2 * kLongR - 1; ++i) win[i] = sp[D * i + (i >= kLongR)];
#pragma unroll 1
        for (int jb = 0; jb < J; jb += kLongR) {
#pragma unroll
            for (int jj = 0; jj < kLongR; ++jj) {
                const float h = hp[jb + jj];
#pragma unroll
                for (int u = 0; u < kLongR; ++u) acc[u] = ffma2s(win[u - jj + kLongR - 1], h, acc[u]);
            }
            // slide one tap block towards older samples
            sp -= kLane;
#pragma unroll
            for (int i = 2 * kLongR - 2; i >= kLongR; --i) win[i] = win[i - kLongR];
            if (jb + kLongR < J) {
#pragma unroll
                for (int i = 0; i < kLongR; ++i) win[i] = sp[D * i];
            }
        }
    }
    if (STAGE == 0 && !a.plain) {
        // NCO mix: output k sits at 63 kHz clock tick k_abs + k; channel c gets y1 * (cos - j sin)(2 pi tick f_c / 63000)
        float2* out0 = a.out + (size_t)(2 * row_in) * a.out_pitch + a.out_off + k0 + (long long)kLongR * t;
        float2* out1 = out0 + a.out_pitch;
        int num[2] = {0, 0}, phase0[2] = {0, 0};
        if (a.nco)
            for (int c = 0; c < 2; ++c) { num[c] = a.nco[2 * row_in + c].num; phase0[c] = a.nco[2 * row_in + c].phase0; }
        const long long tick0 = a.k_abs + k0 + (long long)kLongR * t;
        long long r9 = tick0 % kNcoPeriod, rden = tick0 % kNcoDen;
        int k9 = (int)(r9 < 0 ? r9 + kNcoPeriod : r9), kden = (int)(rden < 0 ? rden + kNcoDen : rden);
#pragma unroll
        for (int u = 0; u < kLongR; ++u) {
            float2 rot[2];
            if (a.nco) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const int ph = (int)(((long long)kden * num[c] + phase0[c]) % kNcoDen);
                    float tt = (float)ph * (2.0f / kNcoDen);
                    if (tt > 1.0f) tt -= 2.0f;
                    float sn, cs;
                    sincospif(tt, &sn, &cs);
                    rot[c] = make_float2(cs, -sn);
                }
            } else {
                rot[0] = tp.nco[k9];
                rot[1] = make_float2(rot[0].x, -rot[0].y);     // "490": conjugate rotation (fir2cpp.C:121-124)
            }
            if (k0 + (long long)kLongR * t + u < n_out) {
                const float2 y = acc[u];
                out0[u] = make_float2(fmaf(-y.y, rot[0].y, y.x * rot[0].x), fmaf(y.x, rot[0].y, y.y * rot[0].x));
                out1[u] = make_float2(fmaf(-y.y, rot[1].y, y.x * rot[1].x), fmaf(y.x, rot[1].y, y.y * rot[1].x));
            }
            if (++k9 == kNcoPeriod) k9 = 0;
            if (++kden == kNcoDen) kden = 0;
        }
    } else {
        float2* out = a.out + (size_t)row_in * a.out_pitch + a.out_off + k0 + (long long)kLongR * t;
#pragma unroll
        for (int u = 0; u < kLongR; ++u)
            if (k0 + (long long)kLongR * t + u < n_out) out[u] = acc[u];
    }
}

template <typename Sample>
__global__ void long_carry_kernel(const float2* __restrict__ old_hist, const Sample* __restrict__ block, long long pitch,
                                  float2* __restrict__ new_hist, int rows, int H, long long n) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)rows * H) return;
    const int row = (int)(idx / H), i = (int)(idx % H);
    const long long src = n - H + i;
    float2 v;
    if (src >= 0) {
        const Sample s = block[(size_t)row * pitch + src];
        v = make_float2((float)s.x, (float)s.y);
    } else {
        v = old_hist[(size_t)row * H + (H + src)];
    }
    new_hist[(size_t)row * H + i] = v;
}

template <int D, int STAGE>
cudaError_t launch_one(const LongArgs& a, const LongStage& st, const LongStageTaps& tp, long long in_pitch, cudaStream_t stream) {
    constexpr int kLongThreads = long_threads(D), kLongTile = long_tile(D);
    const int F = D * (kLongTile + st.J - 1);
    const size_t smem = (size_t)(F + F / (kLongR * D) + 2) * sizeof(float2);
    {   // per device: not cached
        cudaError_t e = cudaFuncSetAttribute(fir_long_kernel<D, STAGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long long n_out = a.n_in / D;
    fir_long_kernel<D, STAGE><<<dim3((unsigned)((n_out + kLongTile - 1) / kLongTile), (unsigned)a.rows_in), kLongThreads, smem, stream>>>(
        a, st.J, in_pitch, tp);
    return cudaGetLastError();
}

// 8-bit input: out = (u - 128) as short2, 8 samples (16 bytes in, 32 out) per thread; count = S n, a multiple of 280
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

LongStage long_stage(int D, int T) {
    LongStage s;
    s.D = D;
    s.T = T;
    const int per_phase = (T + D - 1) / D;
    s.J = (per_phase + kLongR - 1) / kLongR * kLongR;
    s.H = D * s.J;
    return s;
}

// host side of one stage's tap block: [p * J + j] = h[D j + D - 1 - p] (0 beyond the set), plus the reference NCO table
bool long_fill_taps(const LongStage& st, const double* h, LongStageTaps* out) {
    if (st.T < 1 || st.T > kLongMaxTaps || st.D * st.J > kLongTapSlots) return false;
    for (int k = 0; k < kLongTapSlots; ++k) out->h[k] = 0.f;
    for (int p = 0; p < st.D; ++p)
        for (int j = 0; j < st.J; ++j) {
            const int i = st.D * j + st.D - 1 - p;
            out->h[p * st.J + j] = i < st.T ? (float)h[i] : 0.f;
        }
    for (int k = 0; k < kNcoPeriod; ++k) out->nco[k] = reference_nco(k);
    return true;
}

cudaError_t long_launch(const LongArgs& a, const LongStage& st, const LongStageTaps& tp, long long in_pitch, cudaStream_t stream) {
    switch (a.stage) {
        case 0: return launch_one<NVX_D1, 0>(a, st, tp, in_pitch, stream);
        case 1: return launch_one<NVX_D2, 1>(a, st, tp, in_pitch, stream);
        default: return launch_one<NVX_D3, 2>(a, st, tp, in_pitch, stream);
    }
}

// new_hist = last H samples of (old_hist ++ block[.][0..n)) per row; block rows are `pitch` samples apart, short2 if s16
cudaError_t long_carry(const float2* old_hist, const void* block, long long pitch, float2* new_hist, int rows, int H, long long n,
                       int s16, cudaStream_t stream) {
    const long long work = (long long)rows * H;
    const unsigned grid = (unsigned)((work + 255) / 256);
    if (s16)
        long_carry_kernel<short2><<<grid, 256, 0, stream>>>(old_hist, static_cast<const short2*>(block), pitch, new_hist, rows, H, n);
    else
        long_carry_kernel<float2><<<grid, 256, 0, stream>>>(old_hist, static_cast<const float2*>(block), pitch, new_hist, rows, H, n);
    return cudaGetLastError();
}

}  // namespace

// ---- the long-tap path of one engine ----

struct LongPath {
    int S = 0;                            // streams; stages 2 and 3 run over the 2 S channel rows
    long long max_block = 0;
    const NcoChan* nco = nullptr;         // the engine's [S][2] per-stream offsets, or null: the reference table
    LongStage st[3];
    LongStageTaps taps[3];                // passed in the parameter block of every stage launch
    float2* hist[3][2] = {};              // [stage][ping-pong]: [rows][H]
    int cur = 0;
    float2 *y1 = nullptr, *y2 = nullptr;  // 63 kHz and 9 kHz intermediates, [2 S][max_block / 4] and [2 S][max_block / 28]
    LongTcStage* tc[3] = {};              // tensor-core variants of stages 1 and 2 (null: CUDA-core kernel; stage 3 has none)
    bool tc_wanted[3] = {};               // the tensor-core kernel was asked for (NVX_LONG_TC mask) for that stage
    bool mix_on_load = false;             // stage 1 writes ONE un-mixed row per stream, stage 2 rotates while it loads
    short2* u8_wide = nullptr;            // 8-bit input: [S][max_block] short2 (u - 128), allocated on first use
};

namespace {

size_t hist_bytes(const LongPath* lp, int k) { return (size_t)(k == 0 ? lp->S : 2 * lp->S) * lp->st[k].H * sizeof(float2); }

// stage k + 1: on the tensor cores where they serve it, else on the CUDA-core kernel (counted and explained when the tensor cores
// were asked for); then its history carry, the last H inputs of each of `rows` rows (S stream rows of y1 when stage 2 mixes on load)
int run_stage(LongPath* lp, int k, const LongArgs& a, long long in_pitch, int rows, cudaStream_t stream, PathReport* rep) {
    cudaError_t e = lp->tc[k] ? long_tc_launch(lp->tc[k], a, lp->st[k], in_pitch, stream) : cudaErrorNotSupported;
    if (e == cudaErrorNotSupported && a.mix_in)      // (cannot happen: y1 and its pitch are 16-byte aligned)
        return say(rep, NVX_ERR_CUDA, "long-tap stage 2: the tensor-core kernel refused the block and the stage-1 output is un-mixed");
    if (e == cudaErrorNotSupported) {
        if (lp->tc_wanted[k]) {
            rep->fallbacks++;
            say(rep, 0, "note: long-tap stage %d ran on the CUDA-core kernel: %s", k + 1, lp->tc[k] ? "this block cannot be described to the TMA unit (pointer or pitch not 16-byte aligned)"
                                                                                         : "the tap set does not fit the tensor-core tile");
        }
        e = long_launch(a, lp->st[k], lp->taps[k], in_pitch, stream);
    }
    if (e == cudaSuccess) e = long_carry(a.hist, a.in, in_pitch, lp->hist[k][lp->cur ^ 1], rows, lp->st[k].H, a.n_in, a.s16, stream);
    return e == cudaSuccess ? 0 : say(rep, NVX_ERR_CUDA, "long-tap stage %d failed: %s", k + 1, cudaGetErrorString(e));
}

}  // namespace

int long_path_create(int S, long long max_block, const int n[3], const double* const h[3], const NcoChan* nco, cudaStream_t stream,
                     LongPath** out, PathReport* rep) {
    const double* hh[3] = {h[0] ? h[0] : kRefTaps[0], h[1] ? h[1] : kRefTaps[1], h[2] ? h[2] : kRefTaps[2]};
    const int D[3] = {NVX_D1, NVX_D2, NVX_D3};
    LongPath* lp = new LongPath();
    lp->S = S; lp->max_block = max_block; lp->nco = nco;
    for (int k = 0; k < 3; ++k) {
        lp->st[k] = long_stage(D[k], n[k]);
        if (!long_fill_taps(lp->st[k], hh[k], &lp->taps[k])) { long_path_free(lp); return say(rep, NVX_ERR_ARG, "stage %d: %d taps do not fit the long-tap kernel", k + 1, n[k]); }
    }
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 3; ++k)
        for (int q = 0; q < 2 && e == cudaSuccess; ++q) e = cudaMalloc(&lp->hist[k][q], hist_bytes(lp, k));
    if (e == cudaSuccess) e = cudaMalloc(&lp->y1, (size_t)2 * S * (max_block / NVX_D1) * sizeof(float2));
    if (e == cudaSuccess) e = cudaMalloc(&lp->y2, (size_t)2 * S * (max_block / (NVX_D1 * NVX_D2)) * sizeof(float2));
    if (e != cudaSuccess) {
        long_path_free(lp);
        return say(rep, e == cudaErrorMemoryAllocation ? NVX_ERR_NOMEM : NVX_ERR_CUDA, "long-tap path: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    // stages 1 and 2 on the tensor cores where the band matrix fits (fir_long_tc.cu); NVX_LONG_TC is a mask (bit 0: stage
    // 1, bit 1: stage 2; 0 keeps the CUDA-core kernels, whose output is bit-identical across blockings)
    const int tc_mask = getenv("NVX_LONG_TC") ? atoi(getenv("NVX_LONG_TC")) : 3;
    for (int k = 0; k < 2; ++k) {
        lp->tc_wanted[k] = (tc_mask >> k & 1) != 0;
        if (lp->tc_wanted[k]) lp->tc[k] = long_tc_prepare(D[k], n[k], hh[k], stream);
        // a stage the tensor-core kernel does not serve (e.g. stage 2 beyond 959 taps) runs on the CUDA-core kernel: same
        // results to rounding, about half the speed.  Not an error, but never silent: nvx_last_error() says so after create
        // and nvx_stats.long_tc_fallbacks counts every such stage launch.
        if (lp->tc_wanted[k] && !lp->tc[k])
            say(rep, 0, "note: long-tap stage %d (%d taps) is not served by the tensor-core kernel and runs on the CUDA-core kernel", k + 1, n[k]);
    }
    // "mix on load": with the reference offsets (no per-stream NCO) and stage 2 on the streaming tensor-core kernel, stage 1
    // writes one un-mixed 63 kHz row per stream and stage 2 rotates while it converts: y1 crosses HBM once per stream instead
    // of once per channel, in both directions.  NVX_LONG_MIX=stage1 keeps the rotation in the stage-1 epilogue (A/B measurements).
    const char* mix = getenv("NVX_LONG_MIX");
    lp->mix_on_load = !nco && long_tc_mixes_on_load(lp->tc[1]) && (max_block / NVX_D1) % 2 == 0 && !(mix && !strcmp(mix, "stage1"));
    *out = lp;
    return 0;
}

cudaError_t long_path_reset(LongPath* lp, cudaStream_t stream) {
    lp->cur = 0;
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 3; ++k)
        for (int q = 0; q < 2 && e == cudaSuccess; ++q) e = cudaMemsetAsync(lp->hist[k][q], 0, hist_bytes(lp, k), stream);
    return e;
}

CarriedRows long_path_carried(const LongPath* lp) {
    CarriedRows r = {};
    for (int k = 0; k < 3; ++k) {      // per stream: 1 or 2 rows of H float2 (two words each), zeroed
        r.base[k] = reinterpret_cast<uint32_t*>(lp->hist[k][lp->cur]);
        r.words[k] = 2LL * (k == 0 || (k == 1 && lp->mix_on_load) ? 1 : 2) * lp->st[k].H;
    }
    return r;
}

uint64_t long_path_taps_hash(const LongPath* lp) {
    uint64_t h = kHashSeed;
    for (int k = 0; k < 3; ++k) {
        h = hash_bytes(&lp->st[k], sizeof lp->st[k], h);
        h = hash_bytes(lp->taps[k].h, sizeof lp->taps[k].h, h);
    }
    return h;
}

// 3 stage launches, 3 history carries and, for 8-bit input, the widening kernel: all in rep->launches
int long_path_run(LongPath* lp, const void* x, long long n, SampleFmt fmt, long long sb_abs, float2* y3, long long y3_pitch,
                  long long y3_off, cudaStream_t stream, cudaEvent_t after_fir, PathReport* rep) {
    const int S = lp->S;
    // 8-bit input: widened to the int16 values u - 128 in front of the unchanged int16 path (same results bit for bit)
    if (fmt == SampleFmt::U8) {
        const long long count = (long long)S * n;
        cudaError_t e = lp->u8_wide ? cudaSuccess : cudaMalloc(&lp->u8_wide, (size_t)S * lp->max_block * sizeof(short2));
        if (e == cudaSuccess) widen_u8_kernel<<<(unsigned)((count / 8 + 255) / 256), 256, 0, stream>>>(static_cast<const uchar2*>(x), lp->u8_wide, count);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) return say(rep, NVX_ERR_CUDA, "long-tap path, 8-bit input: %s", cudaGetErrorString(e));
        rep->launches++;
        x = lp->u8_wide;
    }
    const long long tick = sb_abs * (kSuper / NVX_D1);                                       // the block's first 63 kHz output
    const long long p1 = lp->max_block / NVX_D1, p2 = lp->max_block / (NVX_D1 * NVX_D2);     // row pitches of y1 and y2
    LongArgs a1 = {};         // 252 k -> 63 k: mixed, one row per channel, or un-mixed, one row per stream (mix on load)
    a1.in = x; a1.hist = lp->hist[0][lp->cur]; a1.out = lp->y1; a1.n_in = n; a1.out_pitch = p1;
    a1.rows_in = S; a1.stage = 0; a1.s16 = fmt != SampleFmt::F32; a1.k_abs = tick; a1.nco = lp->nco; a1.plain = lp->mix_on_load;
    if (int rc = run_stage(lp, 0, a1, n, S, stream, rep)) return rc;
    LongArgs a2 = {};         // 63 k -> 9 k (k_abs: the block's first stage-2 INPUT sample sits at that 63 kHz tick)
    a2.in = lp->y1; a2.hist = lp->hist[1][lp->cur]; a2.out = lp->y2; a2.n_in = n / NVX_D1; a2.out_pitch = p2;
    a2.rows_in = 2 * S; a2.stage = 1; a2.k_abs = tick; a2.mix_in = lp->mix_on_load;
    if (int rc = run_stage(lp, 1, a2, p1, lp->mix_on_load ? S : 2 * S, stream, rep)) return rc;
    LongArgs a3 = {};         // 9 k -> 900
    a3.in = lp->y2; a3.hist = lp->hist[2][lp->cur]; a3.out = y3; a3.n_in = n / (NVX_D1 * NVX_D2); a3.out_pitch = y3_pitch; a3.out_off = y3_off;
    a3.rows_in = 2 * S; a3.stage = 2;
    if (int rc = run_stage(lp, 2, a3, p2, 2 * S, stream, rep)) return rc;
    lp->cur ^= 1;
    rep->launches += 6;
    const cudaError_t e = after_fir ? cudaEventRecord(after_fir, stream) : cudaSuccess;
    return e == cudaSuccess ? 0 : say(rep, NVX_ERR_CUDA, "cudaEventRecord failed: %s", cudaGetErrorString(e));
}

void long_path_free(LongPath* lp) {
    if (!lp) return;
    for (auto& h : lp->hist) { cudaFree(h[0]); cudaFree(h[1]); }
    cudaFree(lp->y1); cudaFree(lp->y2); cudaFree(lp->u8_wide);
    long_tc_free(lp->tc[0]); long_tc_free(lp->tc[1]);
    delete lp;
}

}  // namespace nvx

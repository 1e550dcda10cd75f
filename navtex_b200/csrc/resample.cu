// resample.cu -- the rational resampler in front of the FIR paths (see resample.cuh): design, kernel and the path that runs it.
#include "resample.cuh"

#include <math.h>
#include <stdint.h>

#include "../../include/navtex_b200.h"

namespace nvx {

namespace {

constexpr int kResampleThreads = 256;                                  // one output per thread and tile
constexpr int kResampleTiles = 8;                                      // tiles per CTA, which stages the taps once
// Tap tables up to this size are staged in shared memory by every CTA; larger ones (L up to 2520 branches: 100 S/s steps of the
// rate make L = 2520 / gcd(2520, r / 100)) are read through L1 from global memory, so every accepted rate launches
constexpr size_t kResampleSmemTaps = 96 * 1024;

struct ResampleArgs {
    const void* x;            // this block, [S][n] in the pushed format, 16-byte aligned
    long long n;              // input samples per stream (a multiple of align)
    long long total;          // S n: the block's last sample; words past it are not read
    const float2* hist_in;    // [S][H] float2: the H = J - 1 samples before the block
    float2* hist_out;         // [S][H]: the H samples before the next block
    int H;
    float2* out;              // [S][n_out] at 252 kS/s
    long long n_out;
    const float* taps;        // [L][Jp]: branch p, tap j = h[p + j L], zero for j >= J
    int L, M, J, Jp;          // Jp = J padded to 1 mod 32: the taps lanes of different branches read sit in different banks
    int tile_q, tile_r;       // kResampleThreads M / L, kResampleThreads M % L
};
template <SampleFmt kFmt> struct Words;
template <> struct Words<SampleFmt::F32> {
    static constexpr int kPer = 2;
    __device__ static void get(const int4& v, float2 (&s)[kPer]) {
        s[0] = make_float2(__int_as_float(v.x), __int_as_float(v.y));
        s[1] = make_float2(__int_as_float(v.z), __int_as_float(v.w));
    }
};
template <> struct Words<SampleFmt::S16> {
    static constexpr int kPer = 4;
    __device__ static void get(const int4& v, float2 (&s)[kPer]) {
        const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] = make_float2((float)(short)(w[i] & 0xFFFF), (float)(short)(w[i] >> 16));
    }
};
template <> struct Words<SampleFmt::U8> {
    static constexpr int kPer = 8;
    __device__ static void get(const int4& v, float2 (&s)[kPer]) {
        const unsigned w[4] = {(unsigned)v.x, (unsigned)v.y, (unsigned)v.z, (unsigned)v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            s[2 * i] = make_float2((float)(int)(w[i] & 0xFFu) - 128.f, (float)(int)((w[i] >> 8) & 0xFFu) - 128.f);
            s[2 * i + 1] = make_float2((float)(int)((w[i] >> 16) & 0xFFu) - 128.f, (float)(int)(w[i] >> 24) - 128.f);
        }
    }
};

// sample i of the block (stream-major index), converted exactly
template <SampleFmt kFmt>
__device__ float2 one_sample(const void* x, long long i) {
    if constexpr (kFmt == SampleFmt::F32) return __ldg(static_cast<const float2*>(x) + i);
    else if constexpr (kFmt == SampleFmt::S16) {
        const short2 v = static_cast<const short2*>(x)[i];
        return make_float2((float)v.x, (float)v.y);
    } else {
        const uchar2 v = static_cast<const uchar2*>(x)[i];
        return make_float2((float)(int)v.x - 128.f, (float)(int)v.y - 128.f);
    }
}

// dst[g - g0] = sample g of row s for g in [g_lo, g_hi) (all inside the block), read as whole aligned 16-byte words: a word
// holds 16 / sample_bytes whole samples, and words at the ends of the range may hold samples of no interest, which are skipped.
// A last word that would reach past the end of the block (S n sample_bytes not a multiple of 16) is read sample by sample.
template <SampleFmt kFmt>
__device__ void stage_block(const ResampleArgs& a, int s, long long g0, long long g_lo, long long g_hi, float2* dst) {
    using W = Words<kFmt>;
    if (g_lo >= g_hi) return;
    const long long row = (long long)s * a.n;
    const long long w_lo = (row + g_lo) / W::kPer, w_hi = (row + g_hi - 1) / W::kPer + 1;
    const int4* words = static_cast<const int4*>(a.x);
    for (long long w = w_lo + threadIdx.x; w < w_hi; w += kResampleThreads) {
        float2 v[W::kPer];
        if ((w + 1) * W::kPer <= a.total) W::get(__ldg(words + w), v);
        else {
#pragma unroll
            for (int i = 0; i < W::kPer; ++i) v[i] = w * W::kPer + i < a.total ? one_sample<kFmt>(a.x, w * W::kPer + i) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < W::kPer; ++i) {
            const long long g = w * W::kPer + i - row;
            if (g >= g_lo && g < g_hi) dst[g - g0] = v[i];
        }
    }
}

// grid (chunks of kResampleTiles tiles, streams).  kSmemTaps: the tap table is staged in shared memory, else read from global
template <SampleFmt kFmt, bool kSmemTaps>
__global__ void __launch_bounds__(kResampleThreads) resample_kernel(const ResampleArgs a) {
    extern __shared__ __align__(16) float smem[];
    float* const ts = smem;                                           // [L][Jp] (kSmemTaps)
    float2* const xs = reinterpret_cast<float2*>(smem + (kSmemTaps ? (a.L * a.Jp + 3) & ~3 : 0));   // the tile's window
    const int s = blockIdx.y;
    if (kSmemTaps)
        for (int i = threadIdx.x; i < a.L * a.Jp; i += kResampleThreads) ts[i] = __ldg(a.taps + i);
    // CTA 0 of the row carries the last H samples of (history ++ block) into the next block's history
    if (blockIdx.x == 0) {
        float2* hist = a.hist_out + (size_t)s * a.H;
        const long long first = a.n - a.H;
        for (int i = threadIdx.x; i < a.H && first + i < 0; i += kResampleThreads) hist[i] = a.hist_in[(size_t)s * a.H + a.H + first + i];
        stage_block<kFmt>(a, s, first, first > 0 ? first : 0, a.n, hist);
    }
    long long k0 = (long long)blockIdx.x * kResampleTiles * kResampleThreads;
    // the first tile's phase is the CTA's only 64-bit division; later tiles step it by (tile_q, tile_r)
    long long t0 = k0 * a.M / a.L;
    int p0 = (int)(k0 * a.M - t0 * a.L);
    float2* out = a.out + (size_t)s * a.n_out;
    for (int tile = 0; tile < kResampleTiles && k0 < a.n_out; ++tile) {
        const int count = a.n_out - k0 < kResampleThreads ? (int)(a.n_out - k0) : kResampleThreads;
        const long long g0 = t0 - (a.J - 1);                          // oldest input of the window, xs[0]
        const long long g1 = t0 + (p0 + (count - 1) * a.M) / a.L + 1;
        __syncthreads();                                              // the previous tile's window has been read
        for (long long g = g0 + threadIdx.x; g < 0 && g < g1; g += kResampleThreads) xs[g - g0] = a.hist_in[(size_t)s * a.H + a.H + g];
        stage_block<kFmt>(a, s, g0, g0 > 0 ? g0 : 0, g1, xs);
        __syncthreads();
        if ((int)threadIdx.x < count) {
            const int q = p0 + (int)threadIdx.x * a.M;                // < 2^31: kResampleThreads M < 2^23
            const int t = q / a.L, p = q - t * a.L;                   // relative to t0
            const float2* xp = xs + t + a.J - 1;                      // x[t0 + t - j] = xp[-j]
            const float* hp = (kSmemTaps ? ts : a.taps) + p * a.Jp;
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll 4
            for (int j = 0; j < a.J; ++j) {
                const float h = kSmemTaps ? hp[j] : __ldg(hp + j);
                acc = __ffma2_rn(xp[-j], make_float2(h, h), acc);
            }
            out[k0 + threadIdx.x] = acc;
        }
        k0 += kResampleThreads;
        t0 += a.tile_q;
        p0 += a.tile_r;
        if (p0 >= a.L) { p0 -= a.L; ++t0; }
    }
}

long long gcd_ll(long long a, long long b) {
    while (b) { const long long t = a % b; a = b; b = t; }
    return a;
}

// modified Bessel function of the first kind, order 0 (power series; converges for the window's arguments <= beta)
double bessel_i0(double x) {
    double sum = 1.0, term = 1.0;
    for (int k = 1; k < 200; ++k) {
        term *= (x / (2.0 * k)) * (x / (2.0 * k));
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

}  // namespace

// the Kaiser design's parameters (85 dB: at least 80 dB in the stop band, about 0.0005 dB pass-band ripple)
constexpr double kKaiserA = 85.0, kPassHz = 31500.0;

bool resample_geometry(int rate, ResampleDesign* d, const char** why) {
    *d = ResampleDesign();
    if (rate == NVX_FS_HZ) return true;
    if (rate < kResampleMinRate || rate > kResampleMaxRate || rate % 100 != 0) {
        *why = "input rates are multiples of 100 Hz in [96000, 3200000] S/s";
        return false;
    }
    const long long g = gcd_ll(NVX_FS_HZ, rate);
    d->L = (int)(NVX_FS_HZ / g);
    d->M = (int)(rate / g);
    d->align = rate / gcd_ll(rate, 900);
    // the length from Kaiser's formula, rounded up to whole branches
    const double fs = (double)d->L * rate, f_stop = (rate < NVX_FS_HZ ? rate : NVX_FS_HZ) - kPassHz;
    const double dw = 2.0 * M_PI * (f_stop - kPassHz) / fs;
    const long long n_min = (long long)ceil((kKaiserA - 7.95) / (2.285 * dw)) + 1;
    d->J = (int)((n_min + d->L - 1) / d->L);
    return true;
}

bool resample_design(int rate, ResampleDesign* d, const char** why) {
    if (!resample_geometry(rate, d, why)) return false;
    if (d->L == d->M) {
        d->h.assign(1, 1.0);
        return true;
    }
    // Kaiser window: beta from Kaiser's formula
    const double fs = (double)d->L * rate;
    const double f_pass = kPassHz, f_stop = (rate < NVX_FS_HZ ? rate : NVX_FS_HZ) - kPassHz;
    const double beta = 0.1102 * (kKaiserA - 8.7);
    const long long N = (long long)d->J * d->L;
    const double fc = 0.5 * (f_pass + f_stop) / fs;                   // cycles per sample at L r
    const double i0b = bessel_i0(beta);
    d->h.resize((size_t)N);
    double sum = 0.0;
    for (long long i = 0; i < N; ++i) {
        const double m = (double)i - 0.5 * (double)(N - 1);
        const double xx = 2.0 * fc * m;
        const double sinc = xx == 0.0 ? 1.0 : sin(M_PI * xx) / (M_PI * xx);
        const double r = 2.0 * (double)i / (double)(N - 1) - 1.0;
        const double w = bessel_i0(beta * sqrt(fmax(0.0, 1.0 - r * r))) / i0b;
        d->h[(size_t)i] = 2.0 * fc * sinc * w;
        sum += d->h[(size_t)i];
    }
    for (double& v : d->h) v *= d->L / sum;                          // DC gain L: each branch sums to about 1
    return true;
}

struct ResamplePath {
    int S = 0;
    ResampleDesign d;
    long long max_out = 0;                // outputs per stream of the largest block
    float* taps = nullptr;                // [L][Jp] float, zero-padded
    int Jp = 0;
    bool smem_taps = false;               // the table fits kResampleSmemTaps: every CTA stages it
    size_t smem = 0;                      // dynamic shared memory per CTA
    std::vector<float> taps_host;         // [L][J]: the float taps the kernel reads
    float2* hist[2] = {};                 // [S][H] float2, ping-pong
    int H = 0;
    int cur = 0;
    float2* out = nullptr;                // [S][max_out]
};

int resample_path_create(int rate, int S, long long max_block, ResamplePath** out, PathReport* rep) {
    ResamplePath* rp = new ResamplePath();
    const char* why = "";
    if (!resample_design(rate, &rp->d, &why) || rp->d.L == rp->d.M) {
        delete rp;
        return say(rep, NVX_ERR_ARG, "input rate %d: %s", rate, why);
    }
    const ResampleDesign& d = rp->d;
    rp->S = S;
    rp->H = d.J - 1;
    rp->max_out = max_block / d.M * d.L;
    rp->taps_host.resize((size_t)d.L * d.J);
    for (int p = 0; p < d.L; ++p)
        for (int j = 0; j < d.J; ++j) rp->taps_host[(size_t)p * d.J + j] = (float)d.h[(size_t)p + (size_t)j * d.L];
    rp->Jp = d.J + ((1 - d.J) % 32 + 32) % 32;
    // the taps (when staged), then the window of a full tile: the inputs of its outputs, (tile - 1) M / L + 1 of them at most,
    // and the J - 1 before them
    const size_t table = (size_t)((d.L * rp->Jp + 3) & ~3) * sizeof(float);
    const long long w_max = ((long long)(kResampleThreads - 1) * d.M + d.L - 1) / d.L + d.J + 1;
    rp->smem_taps = table <= kResampleSmemTaps;
    rp->smem = (rp->smem_taps ? table : 0) + (size_t)w_max * sizeof(float2);
    {
        int dev = 0, limit = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || rp->smem > (size_t)limit) {
            resample_path_free(rp);
            return say(rep, NVX_ERR_ARG, "input rate %d: the resampler needs %zu bytes of shared memory per CTA, the device allows %d", rate,
                       rp->smem, limit);
        }
    }
    std::vector<float> padded((size_t)d.L * rp->Jp, 0.f);
    for (int p = 0; p < d.L; ++p)
        for (int j = 0; j < d.J; ++j) padded[(size_t)p * rp->Jp + j] = rp->taps_host[(size_t)p * d.J + j];
    cudaError_t e = cudaMalloc(&rp->taps, padded.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(rp->taps, padded.data(), padded.size() * sizeof(float), cudaMemcpyHostToDevice);
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaMalloc(&rp->hist[k], (size_t)S * (rp->H > 0 ? rp->H : 1) * sizeof(float2));
    if (e == cudaSuccess) e = cudaMalloc(&rp->out, (size_t)S * rp->max_out * sizeof(float2));
    if (e != cudaSuccess) {
        resample_path_free(rp);
        return say(rep, e == cudaErrorMemoryAllocation ? NVX_ERR_NOMEM : NVX_ERR_CUDA, "resampler: %s", cudaGetErrorString(e));
    }
    *out = rp;
    return 0;
}

cudaError_t resample_path_reset(ResamplePath* rp, cudaStream_t stream) {
    rp->cur = 0;
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaMemsetAsync(rp->hist[k], 0, (size_t)rp->S * rp->H * sizeof(float2), stream);
    return e;
}

CarriedRows resample_path_carried(const ResamplePath* rp) {
    return {{reinterpret_cast<uint32_t*>(rp->hist[rp->cur])}, {2LL * rp->H}, {0u}};
}

uint64_t resample_path_taps_hash(const ResamplePath* rp) {
    const int geo[3] = {rp->d.L, rp->d.M, rp->d.J};
    return hash_bytes(rp->taps_host.data(), rp->taps_host.size() * sizeof(float), hash_bytes(geo, sizeof geo));
}

int resample_path_run(ResamplePath* rp, const void* x, long long n, SampleFmt fmt, cudaStream_t stream, const float2** y,
                      long long* n_out, PathReport* rep) {
    const ResampleDesign& d = rp->d;
    ResampleArgs a;
    a.x = x; a.n = n; a.total = (long long)rp->S * n;
    a.hist_in = rp->hist[rp->cur]; a.hist_out = rp->hist[rp->cur ^ 1]; a.H = rp->H;
    a.out = rp->out; a.n_out = n / d.M * d.L;
    a.taps = rp->taps; a.L = d.L; a.M = d.M; a.J = d.J; a.Jp = rp->Jp;
    a.tile_q = kResampleThreads * d.M / d.L; a.tile_r = kResampleThreads * d.M % d.L;
    const size_t smem = rp->smem;
    const long long chunk = (long long)kResampleTiles * kResampleThreads;
    const dim3 grid((unsigned)((a.n_out + chunk - 1) / chunk), (unsigned)rp->S);
    auto kern = rp->smem_taps ? (fmt == SampleFmt::U8 ? resample_kernel<SampleFmt::U8, true> : fmt == SampleFmt::S16 ? resample_kernel<SampleFmt::S16, true>
                                                                                          : resample_kernel<SampleFmt::F32, true>)
                              : (fmt == SampleFmt::U8 ? resample_kernel<SampleFmt::U8, false> : fmt == SampleFmt::S16 ? resample_kernel<SampleFmt::S16, false>
                                                                                          : resample_kernel<SampleFmt::F32, false>);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        kern<<<grid, kResampleThreads, smem, stream>>>(a);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return say(rep, NVX_ERR_CUDA, "resampler launch failed: %s", cudaGetErrorString(e));
    rep->launches++;
    rp->cur ^= 1;
    *y = rp->out;
    *n_out = a.n_out;
    return 0;
}

void resample_path_free(ResamplePath* rp) {
    if (!rp) return;
    cudaFree(rp->taps); cudaFree(rp->hist[0]); cudaFree(rp->hist[1]); cudaFree(rp->out);
    delete rp;
}

}  // namespace nvx

// resample.cuh -- rational resampler in front of the FIR paths: IQ at the radio's own rate r (a multiple of 100 Hz in
// [96 000, 3 200 000]) to the engine's 252 kS/s.
//
// With L / M = 252000 / r in lowest terms, output k (absolute 252 kS/s index since create) is
//   y[k] = sum_j h[p + j L] x[t - j],   t = floor(k M / L),  p = k M - t L,
// samples before the first input being 0: scipy.signal.upfirdn(h, x, L, M)[k].  h is a Kaiser-windowed sinc at L r of L J
// taps (J per polyphase branch): pass band +-31.5 kHz (every nco_hz offset may use it), stop band from min(r, 252000) -
// 31.5 kHz at least 80 dB down, every branch summing to 1 within 1e-3.  L divides 2520 because 100 divides r, so a block of
// a multiple of align = r / gcd(r, 900) input samples carries a whole number of 280-sample superblocks at 252 kS/s.
//
// Mapping: a CTA owns (stream row, 8 tiles of 256 consecutive outputs).  It stages the taps once, branch-major with each branch
// padded to 1 mod 32 words (lanes on different branches read different banks) -- when the table fits 96 KB; the larger tables of
// rates with many branches (L up to 2520) are read through L1 from global memory instead -- then per tile the tile's input window, the
// J - 1 samples before it included, as float2 converted exactly from the pushed format (8-bit: u - 128) with whole 16-byte
// loads, so every input sample is read from HBM once (ends of windows shared by two tiles come from L2).  Lane i of the tile
// computes output i, consecutive lanes reading nearly consecutive window samples, in FP32 with FFMA2 on (I, Q) in ascending j.
// The phase (t, p) of the CTA's first output is its one 64-bit division; tiles and lanes step from it in 32-bit integers.
// Every output is the same sum in the same order whatever the blocking, so the result is bit-identical for any cut of the
// input into aligned blocks.
// The J - 1 samples the next block needs are carried per stream (float2, ping-pong); CTA 0 of each row writes them.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "fir_cascade.cuh"

namespace nvx {

constexpr int kResampleMinRate = 96000, kResampleMaxRate = 3200000;

// the host-side design of one rate (nvx_resampler_info)
struct ResampleDesign {
    int L = 1, M = 1;                 // 252000 / r = L / M in lowest terms
    long long align = kSuper;         // input samples per smallest block: r / gcd(r, 900)
    int J = 1;                        // taps per polyphase branch
    std::vector<double> h;            // L J prototype taps (FP64; the kernel uses their float rounding)
};
// false (and *why set) for an unsupported rate; 252000 gives 1 / 1 / 280 and one unit tap
bool resample_design(int rate, ResampleDesign* d, const char** why);
// the same without the taps (d->h empty): L, M, align and J only
bool resample_geometry(int rate, ResampleDesign* d, const char** why);

// ---- the resampler of one engine (S streams): it owns the taps, the carried input history, the 252 kS/s buffer and the
// launch.  Same calls as the FIR paths (fir_cascade.cuh, fir_long.cuh).
struct ResamplePath;
// rate other than 252000; max_block in input samples.  Returns 0 or an NVX_ERR_* code.
int resample_path_create(int rate, int S, long long max_block, ResamplePath** out, PathReport* rep);
cudaError_t resample_path_reset(ResamplePath* rp, cudaStream_t stream);      // zero histories: the next block follows silence
// the history the next block reads: [S][J - 1] float2 per stream in region 0; zeroing a stream's row restarts it after silence
CarriedRows resample_path_carried(const ResamplePath* rp);
uint64_t resample_path_taps_hash(const ResamplePath* rp);                    // of L, M, J and the float taps the kernel reads
// one block x[S][n] (n a multiple of align) in format fmt -> *y = the float2 [S][*n_out] buffer at 252 kS/s.  One launch,
// counted in rep->launches.  Returns 0 or an NVX_ERR_* code.
int resample_path_run(ResamplePath* rp, const void* x, long long n, SampleFmt fmt, cudaStream_t stream, const float2** y,
                      long long* n_out, PathReport* rep);
void resample_path_free(ResamplePath* rp);

}  // namespace nvx

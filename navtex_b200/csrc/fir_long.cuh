// fir_long.cuh -- the three decimating FIR stages as separate, register-tiled kernels for tap sets LONGER than the
// reference's 37 / 47 / 71 (BASELINE.json configs[4]: "long-tap FIR stress, 255+ taps").
//
// Same arithmetic definition as the reference stages (SURVEY.md A.1):
//   y[k] = sum_{i < T} h[i] x[D (k + 1) - 1 - i]     fir1cpp.C:80-136 (D = 4), fir2cpp.C:131-215 (D = 7, after the
//                                                     NCO mix of fir2cpp.C:112-128), fir3cpp.C:22-60 (D = 10)
// but a different machine mapping from the fused cascade: with hundreds of taps the partial sums of the transposed
// form no longer fit the register file and the work is FP32-bound (~330 flop per input sample at 255 taps, 42 flop/B),
// so the intermediates may as well round-trip through HBM (+4.6 B per input sample) and every stage becomes a plain
// polyphase, register-tiled FIR:
//   * a CTA owns (row, tile of kLongTile consecutive outputs); the inputs that tile needs are staged in shared memory
//     de-interleaved by decimation phase (x_p[m] = x[D m + p]) so that lanes read consecutive addresses;
//   * a thread owns R = 8 consecutive outputs; per phase it slides an R-wide register window over x_p and applies the
//     taps of that phase (warp-uniform constant-bank operands) as packed FFMA2 on (I, Q): R * R FFMA2 per R loads;
//   * the stage-1 kernel applies the NCO rotation of both channels in its epilogue (9-entry table of the reference or
//     the exact per-stream phase of the general NCO) and writes one 63 kHz row per channel, so stages 2 and 3 are
//     plain FIRs over channel rows -- unless stage 2 runs on the streaming tensor-core kernel with the reference table:
//     then stage 1 writes ONE un-mixed row per stream and stage 2 rotates while it loads (LongArgs.plain / mix_in).
// History between blocks is carried per stage (last H inputs of each row), not recomputed.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "fir_cascade.cuh"

namespace nvx {

constexpr int kLongR = 8;                       // outputs per thread
// threads per CTA (each owns kLongR outputs).  The tile a CTA stages is D (tile + J - 1) samples: at D = 10 a 1024-output tile is
// 84 KB of shared memory, two CTAs = 8 warps per SM, and the kernel ran at 42 % FMA-pipe activity for lack of warps; 64 threads
// (512 outputs, 43 KB) put five CTAs on an SM and also waste less on the ragged last tile of a 9250-output row.
__host__ __device__ constexpr int long_threads(int D) { return D == NVX_D3 ? 64 : 128; }
__host__ __device__ constexpr int long_tile(int D) { return kLongR * long_threads(D); }   // outputs per CTA
constexpr int kLongMaxTaps = 1024;              // per stage

struct LongStage {
    int D;            // decimation
    int T;            // taps
    int J;            // taps per phase, padded to a multiple of kLongR: D * J >= T
    int H;            // history samples carried per row: D * J
};

struct LongArgs {
    const void* in;           // [rows_in][in_pitch] float2 (or short2 for stage 1 with s16 input), this block
    const float2* hist;       // [rows_in][H] float2: the H samples that preceded the block (always float2)
    float2* out;              // [rows_out][out_pitch], written at out_off + k; stage 1: rows_out = 2 rows_in (one per channel)
    long long n_in;           // input samples per row in this block (multiple of D)
    long long out_pitch, out_off;
    int rows_in;              // streams (stage 1) or channels (stages 2, 3)
    int stage;                // 0, 1, 2
    int s16;                  // stage 1 only: input block is short2
    long long k_abs;          // stage 1: absolute index of the block's first OUTPUT sample (63 kHz clock), for the NCO
    const NcoChan* nco;       // stage 1: [rows_in][2] per-stream general NCO or null (reference table)
    // "mix on load" (reference NCO table only): stage 1 leaves its output un-mixed, ONE 63 kHz row per stream (plain = 1), and the
    // tensor-core stage 2 applies the rotation of its row's channel while it converts the samples (mix_in = 1: the input has
    // rows_in / 2 rows, k_abs is the absolute index of the block's first INPUT sample) -- the same FP32 products in the same order
    // as the stage-1 epilogue, with half the y1 traffic on both sides
    int plain, mix_in;
};

// ---- tensor-core variant of stages 1 and 2 (fir_long_tc.cu): tcgen05 3xTF32 Toeplitz GEMM, same contract as the CUDA-core stages ----
struct LongTcStage;
struct TcBand {
    int T, N, chunks, J, copies;      // padded taps, outputs per tile, K chunks per tile, band rows per copy, copies
    bool streaming = false;           // served by the streaming kernel (every input chunk feeds the two tiles that contain it)
    std::vector<float> gh, gl;        // [copies][J][32] high / low TF32 parts
};
bool long_tc_band(int D, int T_taps, const double* h, TcBand* out);
// builds the Toeplitz operand of one stage (D = 4 or 7, T taps) on the device; nullptr when the stage does not fit the kernel
LongTcStage* long_tc_prepare(int D, int T, const double* h, cudaStream_t stream);
void long_tc_free(LongTcStage* s);
bool long_tc_mixes_on_load(const LongTcStage* s);      // stage 2 served by the streaming kernel: LongArgs.mix_in is available
cudaError_t long_tc_launch(const LongTcStage* s, const LongArgs& a, const LongStage& st, long long in_pitch, cudaStream_t stream);

// ---- the long-tap path of one engine (S streams, two channels each) ----
// It owns the stage taps, the per-stage histories, the y1 / y2 intermediates, the tensor-core stages and the choice of mix on
// load.  Same calls as the fused path (fir_cascade.cuh); create and run report to the engine through a PathReport.
struct LongPath;
// n[k] taps of stage k + 1, h[k] = null for the reference taps; nco = the engine's [S][2] per-stream offsets, or null for the
// reference table.  Reads NVX_LONG_TC and NVX_LONG_MIX.  Returns 0 or an NVX_ERR_* code.
int long_path_create(int S, long long max_block, const int n[3], const double* const h[3], const NcoChan* nco, cudaStream_t stream,
                     LongPath** out, PathReport* rep);
cudaError_t long_path_reset(LongPath* lp, cudaStream_t stream);     // zero histories: the next block starts after silence
// the histories the next block reads: stage k keeps per_stream[k] consecutive rows of H[k] float2 for each stream (1 for stage 1,
// 2 for stages 2 and 3 -- one per channel -- or 1 for stage 2 when it mixes on load); zeroing a stream's rows restarts its filters
CarriedRows long_path_carried(const LongPath* lp);
uint64_t long_path_taps_hash(const LongPath* lp);     // of the stage geometries and the tap blocks the kernels read
// one block x[S][n] in format fmt that starts at 900 Hz sample sb_abs; the 900 Hz output goes to y3[2 S][y3_pitch] from y3_off on.
// after_fir (if not null) is recorded after the last launch.  Returns 0 or an NVX_ERR_* code.
int long_path_run(LongPath* lp, const void* x, long long n, SampleFmt fmt, long long sb_abs, float2* y3, long long y3_pitch,
                  long long y3_off, cudaStream_t stream, cudaEvent_t after_fir, PathReport* rep);
void long_path_free(LongPath* lp);

}  // namespace nvx

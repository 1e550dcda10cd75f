// fir_long_tc.cu -- the first two long-tap decimating FIR stages (252 k -> 63 k, D = 4, with the NCO mix; 63 k -> 9 k, D = 7)
// on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// Same arithmetic definition as fir_long.cu / the reference stages (fir1cpp.C:80-136, fir2cpp.C:131-215):
//     y[k] = sum_{i < T} h[i] x[D (k + 1) - 1 - i].
// With hundreds of taps that is a dense contraction, and for a tile of N consecutive outputs of 128 rows (streams, or
// channel rows for stage 2) it is the GEMM
//     Y_p[128 x N] = X_p[128 x K] * B[N x K]^T,   p in {I, Q},  K = D (N - 1) + T rounded up to whole chunks,
// where X_p is the window of inputs the tile depends on and B[n][k] = h[D n + T - 1 - k] is the Toeplitz matrix of the
// taps.  B is the same for every tile.  A K chunk is 32 columns holding a whole number of outputs' worth of samples (D = 4:
// 32 samples = 8 outputs; D = 7: 28 samples = 4 outputs + 4 zero columns), so chunk c of B is chunk 0 shifted down by 8 c
// (4 c) rows: the whole operand is ONE band matrix G of N + 8 (chunks - 1) rows (D = 7: two copies, the one for odd chunks
// pre-shifted by 4 rows), kept in shared memory (TMA, SWIZZLE_128B) and addressed per chunk by moving the matrix
// descriptor's start address in whole 8-row swizzle atoms (1024 B).
// Precision: the north star's 1e-5 bar rules out plain TF32 (10-bit mantissa), so every product is the 3xTF32 split
// x_hi h_hi + x_lo h_hi + x_hi h_lo accumulated in FP32 in TMEM (measured 1.5e-6 relative to the FP64 oracle).
//
// Measured on B200 (tools/probes/umma_rate.cu, umma_ts_probe.cu): one tcgen05.mma.kind::tf32 with M = 128, K = 8 costs
// 52 / 59 / 73 cycles at N = 32 / 64 / 128 with both operands in shared memory (4 KB of A per instruction through the
// 128 B/clk pipe the converters' stores also need), but 23 / 36 / 64 with A in tensor memory.  Hence the DATA operand lives
// in tensor memory -- the converters write it with tcgen05.st -- and shared memory only serves the band matrix reads, the
// ring of raw input and the epilogue's dump.
//
// Two kernels share the machinery below.  fir_tcs_kernel<D, L> ("streaming", the default up to 516 taps at D = 4 and 903 at D = 7)
// cuts the input into one global grid of chunks and multiplies every chunk, loaded and converted ONCE, into the two or three tiles
// whose windows contain it (L live accumulator slots in tensor memory); its MMAs are trimmed to the non-zero columns of the band
// parallelogram and the issuer plans the next chunk between the batches of the current one -- see the comment above it.
// fir_tc_kernel<D, N> ("tile at a time") loads and converts each tile's whole window and serves the longer tap sets.
//
// One CTA = 16 warps, persistent over a contiguous range of (row block, output tile) work items:
//   * warp 9 (one thread, TMA) and warps 10..11 (cp.async loaders): stream the raw input through a ring of [128 rows x 128 B]
//     slots, alternating chunks between one 2-D TMA box per slot (SWIZZLE_128B) and 16-byte cp.async copies written in the same
//     XOR-swizzled layout, both completing on the slot's mbarrier; the swizzle lets a thread read ITS row conflict-free, and rows
//     past the last stream / samples past the block end are zero-filled.  (One 1-D bulk copy per row was measured at ~63 cycles
//     of the TMA unit each, whatever its size: 2.8x slower end to end.)  Chunks that lie in the carried history skip the copies
//     and the converters call the general loader instead; the ring protocol is the same;
//   * warps 0..7, converters: thread = row (TMEM lane) x half of the chunk; reads its 16 samples from the slot,
//     de-interleaves I and Q, splits them into TF32 high and low parts and writes the four A tiles (I_hi, I_lo, Q_hi, Q_lo;
//     32 columns each) of one of the A sets into tensor memory with tcgen05.st;
//   * warp 8, issuer: the whole warp runs the loop, one elect.sync-elected lane issues the 2 planes x 3 terms x 4 k-steps
//     tcgen05.mma.kind::tf32 (A in TMEM, B = band matrix in shared memory) per chunk and tile and commits them to the A set's
//     empty barrier; the last chunk of a tile also commits to the tile barrier.  (Issued from an "if (lane == 0)" branch, ptxas
//     wraps every MMA in an R2UR waterfall loop -- ~80 cycles per MMA, which bounded the first versions of this kernel; 64-bit
//     divisions and per-MMA descriptor arithmetic on this thread bounded the next ones: everything it does per chunk is
//     incremental 32-bit arithmetic now.);
//   * warps 12..15, epilogue: dump the tile's accumulator columns to shared memory (tcgen05.ld, lane = row) and release the
//     accumulators, then, lane = output, apply the NCO rotation of both channels (stage 1 with per-stream offsets,
//     fir2cpp.C:112-128) and store 256 contiguous bytes per instruction.  With the reference offsets the rotation moves into
//     the stage-2 converters instead ("mix on load", kMixIn below): stage 1 stores one plain row per stream.
// TMEM map (512 columns): accumulators (I | Q per tile) at the bottom, A sets of 4 x 32 columns above them.
// The accumulation order inside the tensor core is fixed per tile position, so results are deterministic for a given
// blocking but not bit-identical across blockings (tile boundaries move); the tests hold this path to the 1e-5 bar.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#include "fir_long.cuh"

namespace nvx {

namespace {

constexpr int kRows = 128;                 // M: rows per CTA tile
constexpr int kKB = 32;                    // floats per 128-byte swizzle row = samples per K chunk
constexpr int kUmmaK = 8;                  // tf32: 32 bytes per instruction along K
constexpr int kConvWarps = 8;
constexpr int kIssuerWarp = kConvWarps;
constexpr int kTmaWarp = kConvWarps + 1;
constexpr int kLoaderWarp0 = kConvWarps + 2;
constexpr int kLoaderWarps = 2;
constexpr int kEpiWarp0 = kLoaderWarp0 + kLoaderWarps;
constexpr int kTcThreads = 32 * (kConvWarps + 2 + kLoaderWarps + 4);
constexpr int kSlotBytes = kRows * 128;    // one raw-input slot: [128 rows x 128 B]
constexpr int kMaxSlots = 8;
constexpr int kDumpPad = 4;                // epilogue dump: [128 rows][2 NP + 4] floats (row pitch = 4 words mod 32: conflict-free)
// NP: outputs dumped per epilogue pass.  Stage 2 (D = 7) dumps 32 at a time: its two band copies leave little shared memory, and
// two more raw-input slots are worth more than a one-pass epilogue
// (the same holds for the streaming kernel with three live tiles, L = 3, whose band is long)
__host__ __device__ constexpr int dump_outputs(int D, int N, int L = 2) { return (D == NVX_D2 || L == 3) ? 32 : (N > 64 ? 64 : N); }
constexpr int kSmemLimit = 227 * 1024;
// A K chunk is 32 columns holding the largest whole number of outputs' worth of samples: D = 4: 32 samples = 8 outputs; D = 7:
// 28 samples = 4 outputs and 4 zero columns.  The band matrix moves 8 / 4 rows per chunk; descriptors can only move in whole
// 8-row atoms, so D = 7 keeps two copies of the band (even / odd chunks, the odd one pre-shifted by 4 rows).
__host__ __device__ constexpr int chunk_samples(int D) { return kKB / D * D; }
__host__ __device__ constexpr int band_copies(int D) { return 8 / (chunk_samples(D) / D); }
constexpr int kMaxSets = 3;                // A sets in tensor memory
constexpr uint32_t kSetCols = 128;         // {I_hi, I_lo, Q_hi, Q_lo} x 32 columns

struct TcArgs {
    CUtensorMap map_gh, map_gl;            // band matrix G[J][32], high / low TF32 parts
    CUtensorMap map_x;                     // this block as [rows][2 n_in] floats / shorts, box = one slot (128 B x 128 rows, SWIZZLE_128B)
    const void* in;
    const float2* hist;
    float2* out;
    long long n_in, in_pitch, out_pitch, out_off, k_abs;
    const NcoChan* nco;
    int rows, s16, T, H, chunks, J, slots, box_rows, mix;
    int rows_src;                          // rows of the input: rows, or rows / 2 stream rows when the stage mixes on load
    int cpt, lead;                         // streaming kernel: chunks per tile advance (D N / chunk samples), chunks a window leads its tile by
    long long tiles_per_block;             // output tiles per row block
    long long work;                        // row blocks * tiles_per_block
    float2 nco_tab[kNcoPeriod + 16];       // (cos, -sin)(2 pi k 14000 / 63000), fir2cpp.C:104-107, continued periodically (mix on load)
};

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in [0,14),
// leading byte offset (unused here) [16,30), stride byte offset = 8 rows x 128 B = 1024 >> 4 in [32,46), version 1 in
// [46,48), layout type SWIZZLE_128B = 2 in [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void bar_wait(uint32_t bar, uint32_t parity) {
    asm volatile("{\n.reg .pred p;\nW_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra D_%=;\nbra W_%=;\nD_%=:\n}\n"
                 ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(p));
    return p != 0;
}
__device__ __forceinline__ void bar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void umma_ts_tf32(uint32_t d_tmem, uint32_t a_tmem, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}\n"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
                   "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]) : "memory");
}

// general loader for tiles that touch the carried history
__device__ __noinline__ float2 tc_load(const TcArgs& a, int row, long long g) {
    if (row >= a.rows_src || g >= a.n_in || g < -(long long)a.H) return make_float2(0.f, 0.f);   // (older than the history: only zero-padded taps reach there)
    if (g < 0) return a.hist[(size_t)row * a.H + (a.H + g)];
    if (a.s16) {
        const short2 v = static_cast<const short2*>(a.in)[(size_t)row * a.in_pitch + g];
        return make_float2((float)v.x, (float)v.y);
    }
    return static_cast<const float2*>(a.in)[(size_t)row * a.in_pitch + g];
}

// 32 accumulator columns of this warp's 32 TMEM lanes
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr));
}

// mbarriers: band matrix loaded; per raw slot full (TMA -> converters) / empty (converters -> producer); per A set full
// (converters -> issuer) / empty (tensor core -> converters); tile accumulated (tensor core -> epilogue) / accumulators
// dumped (epilogue -> issuer)
enum {
    kBarG = 0,
    kBarRawFull = 1,
    kBarRawEmpty = kBarRawFull + kMaxSlots,
    kBarAFull = kBarRawEmpty + kMaxSlots,
    kBarAEmpty = kBarAFull + kMaxSets,
    kBarTile = kBarAEmpty + kMaxSets,      // (streaming kernel: one per accumulator slot, up to three)
    kBarTmemFree = kBarTile + 3,
    kBars = kBarTmemFree + 3
};

// round to TF32 (10-bit mantissa, nearest, ties away) with integer ops; the remainder is exact in FP32
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
    lo = x - hi;
}

// one sample times the NCO rotation rot = (cos, -sin) of its tick, or its conjugate for the "490" channel (fir2cpp.C:115-124):
// exactly the two FP32 operations per component of the stage-1 epilogues
__device__ __forceinline__ float2 mix_sample(float2 y, float2 rot, bool conj) {
    const float sn = conj ? -rot.y : rot.y;
    return make_float2(__fmaf_rn(-y.y, sn, __fmul_rn(y.x, rot.x)), __fmaf_rn(y.x, sn, __fmul_rn(y.y, rot.x)));
}

template <int D, int N>
__global__ void __launch_bounds__(kTcThreads, 1) fir_tc_kernel(const __grid_constant__ TcArgs a) {
    constexpr int kCS = chunk_samples(D);                   // samples per chunk
    constexpr int kCopies = band_copies(D);
    extern __shared__ __align__(1024) uint8_t smem[];
    // TMEM map: accumulators (I | Q) in columns [0, 2 N), A sets of 128 columns at the top.  Three A sets, not two plus a
    // second accumulator buffer: the round trip "MMAs of a set done -> converters refill it -> next MMAs issued" is a multiple
    // of the ~870 cycles the MMAs of one chunk take (N = 64), so two sets leave the tensor core idle much of the time, while
    // the accumulators are only held for the few hundred cycles the epilogue needs to dump them to shared memory.
    constexpr int kSets = (512 - 2 * N) / (int)kSetCols < kMaxSets ? (512 - 2 * N) / (int)kSetCols : kMaxSets;
    constexpr uint32_t kACol0 = 512 - kSets * kSetCols;
    constexpr int NP = dump_outputs(D, N);                      // the epilogue dumps and stores the tile in N / NP passes
    constexpr int kDumpPitch = 2 * NP + kDumpPad;            // floats per dump row: NP I columns, NP Q columns, padding
    const int g_bytes = kCopies * a.J * 128;                // one part of the band matrix (a multiple of 1024), all copies
    uint8_t* s_gh = smem;
    uint8_t* s_gl = smem + g_bytes;
    uint8_t* s_raw = smem + 2 * g_bytes;                    // ring of raw-input slots
    float* s_dump = reinterpret_cast<float*>(s_raw + a.slots * kSlotBytes);      // the tile's accumulators, [row][I cols | Q cols]
    float2* s_nco = reinterpret_cast<float2*>(s_dump + kRows * kDumpPitch);      // the 9-entry reference NCO table
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_nco + 16);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kBars);
    const uint32_t bar0 = s_u32(bars);
    // warp index made provably warp-uniform: the issuer warp below runs its loops on all lanes and elects one to issue, so that
    // the descriptors are computed in uniform registers (a lane == 0 branch makes ptxas wrap every tcgen05.mma in a
    // R2UR "waterfall" loop: ~15 instructions and ~80 cycles per MMA, which was the kernel's bound)
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
    // float2 input: a slot is 16 samples and each half of the converters owns one slot of a chunk; short2: 32 samples, shared
    const int slots_per_chunk = a.s16 ? 1 : 2;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kBars; ++i) {
            int count = 1;
            // chunks alternate between the cp.async loaders (one arrival per thread) and the TMA thread (which arrives for as many)
            if (i >= kBarRawFull && i < kBarRawFull + kMaxSlots) count = 32 * kLoaderWarps;
            if (i >= kBarRawEmpty && i < kBarRawEmpty + kMaxSlots) count = kConvWarps / slots_per_chunk;
            if (i >= kBarAFull && i < kBarAFull + kMaxSets) count = kConvWarps;
            if (i >= kBarTmemFree) count = 4;
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8 * i), "r"(count));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < kNcoPeriod) s_nco[threadIdx.x] = a.nco_tab[threadIdx.x];
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(s_u32(tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = *tmem_slot;

    // a contiguous range of work items per CTA: consecutive tiles of a row block overlap in a third to two thirds of their
    // inputs, which the CTA's own previous tile left in L2 (DRAM reads 1.02x the input; interleaving the tiles over the CTAs
    // was measured at 1.86x and 5 % slower)
    const long long per = (a.work + gridDim.x - 1) / gridDim.x;
    const long long w_lo = (long long)blockIdx.x * per, w_hi = w_lo + per < a.work ? w_lo + per : a.work;

    // The raw window of a tile goes through the slot ring chunk by chunk; chunks are numbered g = 0, 1, ... across the CTA's
    // tiles and alternate between two independent paths into the same swizzled layout -- even g: one 2-D TMA box per slot
    // (its 128-byte rows cap the TMA unit near 14 B/clk per SM), odd g: 16-byte cp.async pieces from two loader warps (capped
    // at about the same rate by the SM's outstanding-load limit) -- because neither alone keeps up with the tensor core.
    const int ring_chunks = a.slots / slots_per_chunk;
    if (warp == kTmaWarp) {
        if (lane == 0) {
            int ring_at = 0;                                // ring position of chunk g, kept incrementally (no 64-bit divisions per chunk)
            uint32_t ring_ph = 0, odd = 0;
            for (long long w = w_lo; w < w_hi; ++w) {
                const int rb = (int)(w / a.tiles_per_block);
                const long long n0 = (w % a.tiles_per_block) * N;
                const long long t_base = (long long)D * n0 + D - a.T;      // first input of the tile's window (block-relative)
                const bool fast = t_base >= 0;
                for (int c = 0; c < a.chunks; ++c) {
                    const int slot = ring_at * slots_per_chunk;
                    const uint32_t ph = ring_ph;
                    const bool mine = !odd && kCS == kKB;   // 28-sample chunks are not whole 128-byte box rows: cp.async only
                    odd ^= 1;
                    if (++ring_at == ring_chunks) { ring_at = 0; ring_ph ^= 1; }
                    if (!mine) continue;
                    for (int h = 0; h < slots_per_chunk; ++h) {
                        const uint32_t full = bar0 + 8 * (kBarRawFull + slot + h);
                        bar_wait(bar0 + 8 * (kBarRawEmpty + slot + h), ph ^ 1);
                        if (fast) {
                            // x coordinate in 32-bit (float) / 16-bit (short) elements, two per sample; rows past the last
                            // stream and samples past the block end are zero-filled by the TMA unit
                            const int x0 = (int)(2 * (t_base + (long long)c * kCS + h * 16));
                            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(kSlotBytes) : "memory");
                            asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                                         ::"r"(s_u32(s_raw + (slot + h) * kSlotBytes)), "l"(&a.map_x), "r"(x0), "r"(rb * kRows), "r"(full) : "memory");
                            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(32 * kLoaderWarps - 1) : "memory");
                        } else {                            // the converters load this chunk themselves
                            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(32 * kLoaderWarps) : "memory");
                        }
                    }
                }
            }
        }
    } else if (warp >= kLoaderWarp0 && warp < kLoaderWarp0 + kLoaderWarps) {
        // loaders: 16-byte cp.async pieces (L1 bypassed), zero fill past the last stream / the block end, written in the
        // 128-byte-swizzled slot layout: piece (row r, unit u) -> r * 128 + ((u ^ (r % 8)) * 16)
        const int tid = (warp - kLoaderWarp0) * 32 + lane;
        constexpr int kLoaders = 32 * kLoaderWarps;
        const int units = 8 * slots_per_chunk;                    // 16-byte pieces per row per chunk
        const int u16 = tid % units, r0 = tid / units, r_step = kLoaders / units;
        const int esz = a.s16 ? 4 : 8;                            // bytes per sample
        const int per_piece = 16 / esz;                           // samples per piece
        int ring_at = 0;
        uint32_t ring_ph = 0, odd = 0;
        for (long long w = w_lo; w < w_hi; ++w) {
            const int rb = (int)(w / a.tiles_per_block);
            const long long n0 = (w % a.tiles_per_block) * N;
            const long long t_base = (long long)D * n0 + D - a.T;
            const bool fast = t_base >= 0;
            for (int c = 0; c < a.chunks; ++c) {
                const int slot = ring_at * slots_per_chunk;
                const uint32_t ph = ring_ph;
                const bool mine = odd || kCS != kKB;
                odd ^= 1;
                if (++ring_at == ring_chunks) { ring_at = 0; ring_ph ^= 1; }
                if (!mine) continue;
                bar_wait(bar0 + 8 * (kBarRawEmpty + slot), ph ^ 1);
                if (slots_per_chunk == 2) bar_wait(bar0 + 8 * (kBarRawEmpty + slot + 1), ph ^ 1);
                if (fast) {
                    const long long t = t_base + (long long)c * kCS + u16 * per_piece;       // first sample of this thread's pieces
                    const bool t_ok = t + per_piece <= a.n_in && u16 * per_piece < kCS;
                    const uint8_t* src = static_cast<const uint8_t*>(a.in) + ((size_t)(rb * kRows + r0) * a.in_pitch + t) * esz;
                    const size_t src_step = (size_t)r_step * a.in_pitch * esz;
                    const uint32_t dst0 = s_u32(s_raw + (slot + (u16 >> 3)) * kSlotBytes);
#pragma unroll 4
                    for (int r = r0; r < kRows; r += r_step, src += src_step) {
                        const uint32_t dst = dst0 + r * 128 + (((u16 & 7) ^ (r & 7)) << 4);
                        const int bytes = (t_ok && rb * kRows + r < a.rows) ? 16 : 0;
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(bytes ? src : static_cast<const uint8_t*>(a.in)), "r"(bytes) : "memory");
                    }
                    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar0 + 8 * (kBarRawFull + slot)) : "memory");
                    if (slots_per_chunk == 2)
                        asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar0 + 8 * (kBarRawFull + slot + 1)) : "memory");
                } else {
                    bar_arrive(bar0 + 8 * (kBarRawFull + slot));               // the converters load this chunk themselves
                    if (slots_per_chunk == 2) bar_arrive(bar0 + 8 * (kBarRawFull + slot + 1));
                }
            }
        }
    } else if (warp == kIssuerWarp) {
        const bool leader = elect_one();
        if (leader) {
            // the constant band matrix, once per CTA (TMA boxes of box_rows <= 256 rows, a divisor of J)
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * kBarG), "r"(2 * g_bytes) : "memory");
            for (int j = 0; j < kCopies * a.J; j += a.box_rows) {
                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                             ::"r"(s_u32(s_gh + j * 128)), "l"(&a.map_gh), "r"(0), "r"(j), "r"(bar0 + 8 * kBarG) : "memory");
                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                             ::"r"(s_u32(s_gl + j * 128)), "l"(&a.map_gl), "r"(0), "r"(j), "r"(bar0 + 8 * kBarG) : "memory");
            }
        }
        // cute::UMMA::InstrDescriptor: c_format F32 = 1 at [4,6), a / b format TF32 = 2 at [7,10) / [10,13), K-major both,
        // n_dim = N >> 3 at [17,23), m_dim = 128 >> 4 at [24,29)
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24);
        bar_wait(bar0 + 8 * kBarG, 0);
        uint32_t s = 0, ph = 0, tile = 0;
        for (long long w = w_lo; w < w_hi; ++w, ++tile) {
            bar_wait(bar0 + 8 * kBarTmemFree, (tile & 1) ^ 1);            // the epilogue has dumped the previous tile
            asm volatile("tcgen05.fence::after_thread_sync;");
            const uint32_t acc = tmem;
            for (int c = 0; c < a.chunks; ++c) {
                bar_wait(bar0 + 8 * (kBarAFull + s), ph);
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t at = tmem + kACol0 + s * kSetCols;
                // chunk c of B = copy c % kCopies of the band, moved up by whole atoms
                const uint32_t goff = (uint32_t)((a.chunks - 1) / kCopies - c / kCopies) * 1024 + (uint32_t)(c % kCopies) * (a.J * 128);
                // only the outputs n with a tap index D n + T - 1 - (chunk c + k) inside [0, T) see this chunk: the MMAs span those
                // columns of the tile, rounded out to 16 (see fir_tcs_kernel); the first MMA of the tile clears all N columns
                const int num = kCS * c - a.T + 1;
                const int n_lo = num <= 0 ? 0 : (num + D - 1) / D;
                int n_hi = (kCS * c + kCS - 1) / D;
                n_hi = n_hi > N - 1 ? N - 1 : n_hi;
                const bool trim = n_lo <= n_hi;
                const uint32_t c_off = trim ? ((uint32_t)n_lo & ~15u) : 0u;
                const uint32_t np = trim ? (((uint32_t)n_hi | 15u) + 1u) - c_off : (uint32_t)N;
                const uint32_t idesc_np = (idesc & ~(0x3Fu << 17)) | ((np >> 3) << 17);
                const uint32_t gh = s_u32(s_gh) + goff, gl = s_u32(s_gl) + goff;
                if (leader) {
#pragma unroll
                    for (int p = 0; p < 2; ++p)
#pragma unroll
                        for (int term = 0; term < 3; ++term)              // x_hi h_hi, x_lo h_hi, x_hi h_lo
#pragma unroll
                            for (int k = 0; k < kKB / kUmmaK; ++k) {
                                const bool clear = (c | term | k) == 0;
                                umma_ts_tf32(acc + p * N + (clear ? 0u : c_off), at + (2 * p + (term == 1 ? 1 : 0)) * 32 + k * kUmmaK,
                                             umma_desc((term == 2 ? gl : gh) + (clear ? 0u : c_off * 128u) + k * kUmmaK * 4),
                                             clear ? idesc : idesc_np, clear ? 0u : 1u);
                            }
                    umma_commit(bar0 + 8 * (kBarAEmpty + s));
                    if (c == a.chunks - 1) umma_commit(bar0 + 8 * kBarTile);
                }
                __syncwarp();
                if (++s == kSets) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp < kConvWarps) {
        // thread = TMEM lane = row 32 q + lane of the tile, samples [16 kh, 16 kh + 16) of every chunk
        const int q = warp & 3, kh = warp >> 2;
        const int r = q * 32 + lane;
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16) + kACol0 + kh * 16;
        int slot = a.s16 ? 0 : kh;                          // float2: this half's slot of chunk 0
        uint32_t sph = 0, s = 0, ph = 0;
        for (long long w = w_lo; w < w_hi; ++w) {
            const int rb = (int)(w / a.tiles_per_block);
            const long long n0 = (w % a.tiles_per_block) * N;
            const long long t_base = (long long)D * n0 + D - a.T;
            const bool fast = t_base >= 0;
            for (int c = 0; c < a.chunks; ++c) {
                bar_wait(bar0 + 8 * (kBarRawFull + slot), sph);                 // raw samples landed
                // read and split BEFORE waiting for the A set: the round trip "set free -> set full" is then only the
                // eight tcgen05.st of this thread (the conversion itself overlaps the MMAs that still read the set)
                const uint8_t* row = s_raw + slot * kSlotBytes + r * 128;
                float ih[16], il[16], qh[16], ql[16];
                if (fast) {
                    if (a.s16) {                                                // 16-byte units 4 kh .. 4 kh + 3: 4 samples each
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int4 v = *reinterpret_cast<const int4*>(row + (((4 * kh + u) ^ (r & 7)) << 4));
                            const int wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                split_tf32((float)(short)(wv[j] & 0xFFFF), ih[4 * u + j], il[4 * u + j]);
                                split_tf32((float)(wv[j] >> 16), qh[4 * u + j], ql[4 * u + j]);
                            }
                        }
                    } else {                                                    // 16-byte units 0 .. 7: 2 samples each
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            float4 v = *reinterpret_cast<const float4*>(row + ((u ^ (r & 7)) << 4));
                            if (kCS != kKB && kh * 16 + 2 * u >= kCS) v = make_float4(0.f, 0.f, 0.f, 0.f);     // zero columns
                            split_tf32(v.x, ih[2 * u], il[2 * u]);
                            split_tf32(v.y, qh[2 * u], ql[2 * u]);
                            split_tf32(v.z, ih[2 * u + 1], il[2 * u + 1]);
                            split_tf32(v.w, qh[2 * u + 1], ql[2 * u + 1]);
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float2 v = make_float2(0.f, 0.f);
                        if (kh * 16 + j < kCS) v = tc_load(a, rb * kRows + r, t_base + (long long)c * kCS + kh * 16 + j);
                        split_tf32(v.x, ih[j], il[j]);
                        split_tf32(v.y, qh[j], ql[j]);
                    }
                }
                __syncwarp();                                                   // every lane holds its samples in registers:
                if (lane == 0) bar_arrive(bar0 + 8 * (kBarRawEmpty + slot));    // the slot can be refilled already
                bar_wait(bar0 + 8 * (kBarAEmpty + s), ph ^ 1);                  // the MMAs that read this A set are done
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t col = lane_base + s * kSetCols;
                tmem_st16(col + 0 * 32, ih);
                tmem_st16(col + 1 * 32, il);
                tmem_st16(col + 2 * 32, qh);
                tmem_st16(col + 3 * 32, ql);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;");
                __syncwarp();
                if (lane == 0) bar_arrive(bar0 + 8 * (kBarAFull + s));
                if (++s == kSets) { s = 0; ph ^= 1; }
                slot += slots_per_chunk;
                if (slot >= a.slots) { slot -= a.slots; sph ^= 1; }
            }
        }
    } else {
        // epilogue warp: TMEM lanes 32 q .. 32 q + 31 (q = warp % 4, the lanes this warp may address) = rows of the tile.
        // Phase 1, lane = row: dump the row's 2 N accumulator columns to shared memory and release the accumulators.
        // Phase 2, lane = output: per row read (I, Q), apply the NCO rotation of both channels -- output k sits at 63 kHz
        // clock tick k_abs + k; channel c gets y * (cos - j sin)(2 pi tick f_c / 63000), fir2cpp.C:112-128 -- and store 256
        // contiguous bytes per instruction (one row per lane was measured 1.5x slower for the whole kernel).
        const int q = warp & 3;
        const long long n_out = a.n_in / D;
        float* my_row = s_dump + (q * 32 + lane) * kDumpPitch;
        const float* rows0 = s_dump + (q * 32) * kDumpPitch;
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16);
        uint32_t tile = 0;
        for (long long w = w_lo; w < w_hi; ++w, ++tile) {
            const int rb = (int)(w / a.tiles_per_block);
            const long long n0 = (w % a.tiles_per_block) * N;
            bar_wait(bar0 + 8 * kBarTile, tile & 1);
            asm volatile("tcgen05.fence::after_thread_sync;");
            const int row0 = rb * kRows + q * 32;
            const int r_max = a.rows - row0 < 32 ? a.rows - row0 : 32;
#pragma unroll 1
            for (int pass = 0; pass < N / NP; ++pass) {
            if (pass) __syncwarp();                         // the previous pass has been stored
#pragma unroll 1
            for (int h = 0; h < 2 * NP / 32; ++h) {
                uint32_t v[32];
                // dump column h * 32: I columns of this pass first, then its Q columns
                tmem_ld32(taddr + (h < NP / 32 ? pass * NP + h * 32 : N + pass * NP + (h - NP / 32) * 32), v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<uint4*>(my_row + h * 32 + 4 * j) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (pass == N / NP - 1) asm volatile("tcgen05.fence::before_thread_sync;");
            __syncwarp();
            if (pass == N / NP - 1 && lane == 0) bar_arrive(bar0 + 8 * kBarTmemFree);      // the accumulators may be overwritten
#pragma unroll 1
            for (int h = 0; h < NP / 32; ++h) {
                const int m = h * 32 + lane;                // column of the dump
                const int n = pass * NP + m;                // output of the tile
                if (n0 + n >= n_out) continue;
                const long long tick = a.k_abs + n0 + n;
                if (!a.mix) {                               // stage 2: one output row per input row, no rotation
                    float2* dst1 = a.out + (size_t)row0 * a.out_pitch + a.out_off + n0 + n;
#pragma unroll 4
                    for (int r = 0; r < r_max; ++r, dst1 += a.out_pitch)
                        *dst1 = make_float2(rows0[r * kDumpPitch + m], rows0[r * kDumpPitch + NP + m]);
                    continue;
                }
                float2* dst = a.out + (size_t)(2 * row0) * a.out_pitch + a.out_off + n0 + n;
                if (a.nco) {
                    const long long rden = tick % kNcoDen;
                    const long long kden = rden < 0 ? rden + kNcoDen : rden;
#pragma unroll 2
                    for (int r = 0; r < r_max; ++r, dst += 2 * a.out_pitch) {
                        const NcoChan nc[2] = {a.nco[2 * (row0 + r)], a.nco[2 * (row0 + r) + 1]};
                        const float2 y = make_float2(rows0[r * kDumpPitch + m], rows0[r * kDumpPitch + NP + m]);
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            const int phs = (int)((kden * nc[c].num + nc[c].phase0) % kNcoDen);
                            float tt = (float)phs * (2.0f / kNcoDen);
                            if (tt > 1.0f) tt -= 2.0f;
                            float sn, cs;
                            sincospif(tt, &sn, &cs);
                            dst[c * a.out_pitch] = make_float2(fmaf(y.y, sn, y.x * cs), fmaf(-y.x, sn, y.y * cs));
                        }
                    }
                } else {
                    const long long r9 = tick % kNcoPeriod;
                    const float2 rot = s_nco[r9 < 0 ? r9 + kNcoPeriod : r9];       // (cos, -sin); "490" uses the conjugate (fir2cpp.C:121-124)
#pragma unroll 4
                    for (int r = 0; r < r_max; ++r, dst += 2 * a.out_pitch) {
                        const float2 y = make_float2(rows0[r * kDumpPitch + m], rows0[r * kDumpPitch + NP + m]);
                        dst[0] = make_float2(fmaf(-y.y, rot.y, y.x * rot.x), fmaf(y.x, rot.y, y.y * rot.x));
                        dst[a.out_pitch] = make_float2(fmaf(y.y, rot.y, y.x * rot.x), fmaf(-y.x, rot.y, y.y * rot.x));
                    }
                }
            }
            }
            __syncwarp();                                   // the dump rows are overwritten by the next tile
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
}


// ---------------------------------------------------------------------------------------------------------------------------------
// Streaming variant (the default wherever a window spans at most two tiles: up to 260 taps at D = 4, 455 at D = 7).
//
// fir_tc_kernel above treats every tile on its own: it loads and converts the tile's whole window, D (N - 1) + T samples for
// D N new ones -- at 255 taps every input sample travels L2 -> shared memory -> registers -> tensor memory TWICE, and that
// traffic, not the tensor core, bounded the kernel (ncu: tensor pipe 51 % busy, converters waiting for raw input).  Here the
// input is cut into GLOBAL chunks G (chunk_samples(D) samples each, the same grid for every tile: the tap count is padded to
// T = D + lead * chunk so that tile t's window is exactly the chunks [cpt t - lead, cpt t + cpt), cpt = D N / chunk) and a CTA
// walks its contiguous range of tiles chunk by chunk: every chunk is loaded once, converted once, written to tensor memory
// once -- and multiplied into BOTH tiles whose windows contain it, the one that is finishing (band rows of its late chunks)
// and the one that is starting (band rows of its early chunks).  Two tiles are therefore live at a time:
//   TMEM: accumulator slot 0 in columns [0, 128), slot 1 in [128, 256) (I | Q, N = 64), two A sets of 128 columns above.
// The epilogue dumps a finished tile to shared memory while the MMAs of the next chunk's older tile run, and the slot is handed
// back before the tile after next needs it.  Per chunk the tensor core now has 48 MMAs to chew on instead of 24 while the
// converters refill the other A set, so two A sets are enough.  Everything else -- band matrix, descriptors, 3xTF32 split, slot
// ring, TMA / cp.async alternation, epilogue phases -- is as in fir_tc_kernel.
constexpr int kSN = 64;                    // outputs per tile of the streaming kernel

// L = live tiles = accumulator slots: 2 while a window spans at most two tiles (lead <= cpt: two A sets), 3 up to three tiles
// (cpt < lead <= 2 cpt, i.e. up to 516 taps at D = 4: the third slot takes the place of the second A set, so conversion and MMAs
// of consecutive chunks no longer overlap -- still far ahead of loading and converting every window three times).
// kMixIn ("mix on load", stage 2 with the reference NCO table): the input is the UN-mixed stage-1 output, one row per stream; a
// row block is 64 streams, CTA row r = stream (r & 63) of the block, channel r >> 6 (uniform per converter warp), and the converters
// rotate every sample by its channel's NCO phase (fir2cpp.C:112-128: "518" by (cos, -sin), "490" by the conjugate) before the
// TF32 split -- the same two FP32 operations per component as the stage-1 epilogue's mix, so the products are bit-identical,
// while y1 crosses HBM once per stream instead of once per channel on both sides.
// Converters: two warps per TMEM lane quarter, each converting 16 samples of a chunk per row, as in fir_tc_kernel.  The
// converters are a latency-bound chain of ~300 instructions per chunk and warp and set the chunk period of stage 2 (in-kernel
// trace, 65 taps: 1 470 cycles per chunk against 963 with conversion, loads and epilogue knocked out), so four per quarter were
// built and measured: 24 warps per CTA cap the kernel at 80 registers per thread, every role spills, and the whole chain is
// SLOWER (65 taps: 332 -> 315 Gsamples/s with stage 2 on four, 286 with both stages; 255 taps: 288 -> 276 / 260).
// Also built, measured and removed: one issuer warp per plane (I / Q: independent accumulators and A tiles) so that one thread's
// per-batch operand set-up (~130 instructions of moves into uniform registers, ~300 cycles in which the short MMA queue runs dry:
// 573 cycles of MMAs per 980-cycle chunk with every other role knocked out) overlaps the other's MMAs -- two interleaved MMA
// streams are slower than one (that floor rose to 1 204 cycles per chunk; 65 / 255 taps: 330 / 280 -> 278 / 249 Gsamples/s);
// and a host-built per-chunk plan table in the kernel parameters with 32-bit descriptor arithmetic (no measurable change).
// And: two converter groups taking ALTERNATE chunks (each thread all 32 columns, one A set per group, so that a chunk's chain of
// hand-overs has two chunk periods to complete) -- correct only with two A sets and an even number of chunks in the ring (a parity
// wait cannot tell phase k from phase k + 2), and slower where it applies (65 taps: 328 -> 319 Gsamples/s): the converters are
// bound by their instruction throughput, not by the latency of the hand-overs.
template <int D, int L, bool kMixIn = false>
__global__ void __launch_bounds__(kTcThreads, 1) fir_tcs_kernel(const __grid_constant__ TcArgs a) {
    constexpr int N = kSN;
    constexpr int kPer = kKB / 2;                            // samples (A columns) per converter thread and chunk
    constexpr int kInRows = kMixIn ? kRows / 2 : kRows;      // input rows per row block
    static_assert(!kMixIn || chunk_samples(D) % kNcoPeriod == 1, "mix on load: a chunk advances the NCO phase index by one");
    constexpr int kCS = chunk_samples(D);
    constexpr int kCopies = band_copies(D);
    constexpr uint32_t kSlotCols = 2 * N;
    constexpr int kSets = (512 - L * (int)kSlotCols) / (int)kSetCols;
    constexpr uint32_t kACol0 = L * kSlotCols;               // the A sets sit above the accumulator slots
    static_assert(kSets >= 1 && L >= 2 && L <= 3, "tensor memory budget");
    constexpr int NP = dump_outputs(D, N, L);
    constexpr int kDumpPitch = 2 * NP + kDumpPad;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int g_bytes = kCopies * a.J * 128;
    uint8_t* s_gh = smem;
    uint8_t* s_gl = smem + g_bytes;
    uint8_t* s_raw = smem + 2 * g_bytes;
    float* s_dump = reinterpret_cast<float*>(s_raw + a.slots * kSlotBytes);
    float2* s_nco = reinterpret_cast<float2*>(s_dump + kRows * kDumpPitch);
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_nco + 16);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kBars);
    const uint32_t bar0 = s_u32(bars);
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
    // a chunk is one 128-byte piece per row (int16 input) or two (float2 input): two ring slots -- except when mixing on load, where
    // a row block has only 64 input rows and both pieces share ONE slot (second piece at kHalfBytes), so the ring holds twice as
    // many chunks and as many bytes in flight as the 128-row layout
    const int pieces = a.s16 ? 1 : 2;
    const int slots_per_chunk = kMixIn ? 1 : pieces;
    constexpr int kHalfBytes = kInRows * 128;
    const int cpt = a.cpt, lead = a.lead;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kBars; ++i) {
            int count = 1;
            if (i >= kBarRawFull && i < kBarRawFull + kMaxSlots) count = 32 * kLoaderWarps;
            if (i >= kBarRawEmpty && i < kBarRawEmpty + kMaxSlots) count = kConvWarps / slots_per_chunk;
            if (i >= kBarAFull && i < kBarAFull + kMaxSets) count = kConvWarps;
            if (i >= kBarTmemFree) count = 4;
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8 * i), "r"(count));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < kNcoPeriod) s_nco[threadIdx.x] = a.nco_tab[threadIdx.x];
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(s_u32(tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = *tmem_slot;

    // a contiguous range of (row block, tile) items per CTA, walked as segments [ta, tb) of consecutive tiles of one row block;
    // only the first `lead` chunks of a segment are loaded without feeding a second tile (the neighbour CTA loads them too)
    const long long per = (a.work + gridDim.x - 1) / gridDim.x;
    const long long w_lo = (long long)blockIdx.x * per, w_hi = w_lo + per < a.work ? w_lo + per : a.work;
    const long long tpb = a.tiles_per_block;
    const int ring_chunks = a.slots / slots_per_chunk;

#define NVX_FOR_SEGMENTS(...)                                                                        \
    for (long long w_ = w_lo; w_ < w_hi;) {                                                          \
        const int rb = (int)(w_ / tpb);                                                              \
        const long long ta = w_ % tpb;                                                               \
        const long long tb = ta + (w_hi - w_) < tpb ? ta + (w_hi - w_) : tpb;                        \
        __VA_ARGS__                                                                                  \
        w_ += tb - ta;                                                                               \
    }

    if (warp == kTmaWarp) {
        if (lane == 0) {
            // ring position of chunk g, kept incrementally (no 64-bit divisions on any role's critical path)
            int ring_at = 0;
            uint32_t ring_ph = 0, odd = 0;
            NVX_FOR_SEGMENTS({
                for (long long G = cpt * ta - lead; G < cpt * tb; ++G) {
                    const int slot = ring_at * slots_per_chunk;
                    const uint32_t ph = ring_ph;
                    const bool mine = !odd;                 // odd chunks: the cp.async loaders
                    odd ^= 1;
                    if (++ring_at == ring_chunks) { ring_at = 0; ring_ph ^= 1; }
                    if (!mine) continue;
                    const bool fast = G >= 0;       // chunks before the block come from the carried history
                    if (kMixIn) {
                        const uint32_t full = bar0 + 8 * (kBarRawFull + slot);
                        bar_wait(bar0 + 8 * (kBarRawEmpty + slot), ph ^ 1);
                        if (fast) {
                            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(pieces * kHalfBytes) : "memory");
                            for (int h = 0; h < pieces; ++h)
                                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                                             ::"r"(s_u32(s_raw + slot * kSlotBytes + h * kHalfBytes)), "l"(&a.map_x), "r"((int)(2 * (G * kCS + h * 16))),
                                               "r"(rb * kInRows), "r"(full) : "memory");
                            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(32 * kLoaderWarps - 1) : "memory");
                        } else {
                            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(32 * kLoaderWarps) : "memory");
                        }
                        continue;
                    }
                    for (int h = 0; h < slots_per_chunk; ++h) {
                        const uint32_t full = bar0 + 8 * (kBarRawFull + slot + h);
                        bar_wait(bar0 + 8 * (kBarRawEmpty + slot + h), ph ^ 1);
                        if (fast) {
                            // x coordinate in 32-bit (float) / 16-bit (short) elements, two per sample.  D = 7: the second box of a
                            // 28-sample chunk over-fetches 4 samples of the next chunk (the converters zero those columns); rows past
                            // the last stream and samples past the block end are zero-filled by the TMA unit
                            const int x0 = (int)(2 * (G * kCS + h * 16));
                            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(kInRows * 128) : "memory");
                            asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                                         ::"r"(s_u32(s_raw + (slot + h) * kSlotBytes)), "l"(&a.map_x), "r"(x0), "r"(rb * kInRows), "r"(full) : "memory");
                            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(32 * kLoaderWarps - 1) : "memory");
                        } else {
                            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(full), "n"(32 * kLoaderWarps) : "memory");
                        }
                    }
                }
            })
        }
    } else if (warp >= kLoaderWarp0 && warp < kLoaderWarp0 + kLoaderWarps) {
        const int tid = (warp - kLoaderWarp0) * 32 + lane;
        constexpr int kLoaders = 32 * kLoaderWarps;
        const int units = 8 * pieces;
        const int u16 = tid % units, r0 = tid / units, r_step = kLoaders / units;
        const int esz = a.s16 ? 4 : 8;
        const int per_piece = 16 / esz;
        int ring_at = 0;
        uint32_t ring_ph = 0, odd = 0;
        NVX_FOR_SEGMENTS({
            for (long long G = cpt * ta - lead; G < cpt * tb; ++G) {
                const int slot = ring_at * slots_per_chunk;
                const uint32_t ph = ring_ph;
                const bool mine = odd != 0;
                odd ^= 1;
                if (++ring_at == ring_chunks) { ring_at = 0; ring_ph ^= 1; }
                if (!mine) continue;
                bar_wait(bar0 + 8 * (kBarRawEmpty + slot), ph ^ 1);
                if (slots_per_chunk == 2) bar_wait(bar0 + 8 * (kBarRawEmpty + slot + 1), ph ^ 1);
                if (G >= 0) {
                    const long long t = G * kCS + u16 * per_piece;
                    const bool t_ok = t + per_piece <= a.n_in && u16 * per_piece < kCS;
                    const uint8_t* src = static_cast<const uint8_t*>(a.in) + ((size_t)(rb * kInRows + r0) * a.in_pitch + t) * esz;
                    const size_t src_step = (size_t)r_step * a.in_pitch * esz;
                    const uint32_t dst0 = s_u32(s_raw + (kMixIn ? slot * kSlotBytes + (u16 >> 3) * kHalfBytes : (slot + (u16 >> 3)) * kSlotBytes));
#pragma unroll 4
                    for (int r = r0; r < kInRows; r += r_step, src += src_step) {
                        const uint32_t dst = dst0 + r * 128 + (((u16 & 7) ^ (r & 7)) << 4);
                        const int bytes = (t_ok && rb * kInRows + r < a.rows_src) ? 16 : 0;
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(bytes ? src : static_cast<const uint8_t*>(a.in)), "r"(bytes) : "memory");
                    }
                    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar0 + 8 * (kBarRawFull + slot)) : "memory");
                    if (slots_per_chunk == 2)
                        asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar0 + 8 * (kBarRawFull + slot + 1)) : "memory");
                } else {
                    bar_arrive(bar0 + 8 * (kBarRawFull + slot));
                    if (slots_per_chunk == 2) bar_arrive(bar0 + 8 * (kBarRawFull + slot + 1));
                }
            }
        })
    } else if (warp == kIssuerWarp) {
        const bool leader = elect_one();
        if (leader) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * kBarG), "r"(2 * g_bytes) : "memory");
            for (int j = 0; j < kCopies * a.J; j += a.box_rows) {
                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                             ::"r"(s_u32(s_gh + j * 128)), "l"(&a.map_gh), "r"(0), "r"(j), "r"(bar0 + 8 * kBarG) : "memory");
                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                             ::"r"(s_u32(s_gl + j * 128)), "l"(&a.map_gl), "r"(0), "r"(j), "r"(bar0 + 8 * kBarG) : "memory");
            }
        }
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24);
        bar_wait(bar0 + 8 * kBarG, 0);
        uint32_t s = 0, ph = 0;
        int q0 = 0;                                         // tiles of the segments already done (32-bit: a CTA walks < 2^31 tiles)
        uint64_t dh0[kKB / kUmmaK], dl0[kKB / kUmmaK];      // band descriptors at offset 0, one per k-step
#pragma unroll
        for (int k = 0; k < kKB / kUmmaK; ++k) {
            dh0[k] = umma_desc(s_u32(s_gh) + k * kUmmaK * 4);
            dl0[k] = umma_desc(s_u32(s_gl) + k * kUmmaK * 4);
        }
        // What one chunk contributes to one tile, worked out ahead of time (see below): chunk index c inside the tile's window,
        // accumulator slot, and the trimmed extent of its MMAs.
        // The band is a parallelogram: the samples of chunk c only reach the outputs n with a tap index D n + T - 1 - (chunk c + k)
        // inside [0, T), i.e. n in [opc (c - lead), opc c + opc - 1] (opc = outputs per chunk); every other row of the tile's B
        // slice is all zero.  So the MMAs of a chunk only span those output columns, rounded out to the instruction's N
        // granularity of 16: D, the band rows and N move together.  Early and late chunks of a window become N = 16 .. 48
        // instructions instead of 64: 37 % less tensor work at 255 taps, more for shorter filters.  The first MMA of a tile still
        // spans all 64 columns: it is the one that clears them (its chunk has column offset 0 anyway).
        struct Plan { uint32_t valid, c, slot, wait_par, d_off, idesc_np; uint64_t dadd; };
        auto plan = [&](int r, int t1, int which, int q0_, int n_tiles) {
            Plan p;
            const int t = t1 + which;
            const int c = r + lead - which * cpt;               // chunk index inside tile t's window, 0 .. chunks - 1
            p.valid = !(c < 0 || t < 0 || t >= n_tiles);
            const int q = q0_ + (t < 0 ? 0 : t);
            p.c = (uint32_t)c;
            p.slot = (uint32_t)(q % L);
            p.wait_par = (uint32_t)((q / L) & 1) ^ 1u;
            // chunk c of B = copy c % kCopies of the band, moved up by whole atoms: the descriptors are those of the band's first
            // rows plus the offset in their 16-byte address field (shared memory is far below its 14-bit range)
            const uint32_t goff = (uint32_t)((a.chunks - 1) / kCopies - c / kCopies) * 1024 + (uint32_t)(c % kCopies) * (a.J * 128);
            constexpr int kOpc = kCS / D;
            int n_lo = kOpc * (c - lead), n_hi = kOpc * c + kOpc - 1;
            n_lo = n_lo < 0 ? 0 : n_lo;
            n_hi = n_hi > N - 1 ? N - 1 : n_hi;
            const uint32_t off = (uint32_t)n_lo & ~15u;
            const uint32_t np = (((uint32_t)n_hi | 15u) + 1u) - off;
            p.d_off = p.slot * kSlotCols + off;
            p.idesc_np = (idesc & ~(0x3Fu << 17)) | ((np >> 3) << 17);
            p.dadd = (goff >> 4) + (uint64_t)off * 8;           // 16 rows of the band = two 1024-byte atoms
            return p;
        };
        auto issue = [&](const Plan& p, uint32_t at) {
            if (p.c == 0) {                                     // first chunk of the tile: its accumulator slot must have been dumped
                bar_wait(bar0 + 8 * (kBarTmemFree + p.slot), p.wait_par);
                asm volatile("tcgen05.fence::after_thread_sync;");
            }
            if (leader) {
#pragma unroll
                for (int pl = 0; pl < 2; ++pl)
#pragma unroll
                    for (int term = 0; term < 3; ++term)        // x_hi h_hi, x_lo h_hi, x_hi h_lo
#pragma unroll
                        for (int k = 0; k < kKB / kUmmaK; ++k) {
                            const bool clear = (p.c | (uint32_t)term | (uint32_t)k) == 0;     // c == 0: column offset 0
                            umma_ts_tf32(tmem + p.d_off + pl * N, at + (2 * pl + (term == 1 ? 1 : 0)) * 32 + k * kUmmaK,
                                         (term == 2 ? dl0[k] : dh0[k]) + p.dadd, clear ? idesc : p.idesc_np, clear ? 0u : 1u);
                        }
                if (p.c == (uint32_t)(a.chunks - 1)) umma_commit(bar0 + 8 * (kBarTile + p.slot));
            }
            __syncwarp();
        };
        NVX_FOR_SEGMENTS({
            // chunk G = cpt t1 + r: t1 is the tile that is finishing (its chunk index r + lead), t1 + 1 starts once r + lead >= cpt
            const int back = (lead + cpt - 1) / cpt;        // whole tiles the first chunk of the segment lies before tile ta
            int r = back * cpt - lead;
            int t1 = -back;                                 // relative to ta
            const int n_tiles = (int)(tb - ta);
            const int n_chunks = cpt * n_tiles + lead;
            // The contributions of chunk j + 1 are planned BETWEEN the MMA batches of chunk j: the issuing thread's integer
            // work (~300 cycles of dependent uniform-datapath instructions per chunk) then runs while the tensor core still has
            // the first batch queued, instead of leaving it idle between chunks.
            Plan pl[L];
#pragma unroll
            for (int w = 0; w < L; ++w) pl[w] = plan(r, t1, w, q0, n_tiles);
            for (int j = 0; j < n_chunks; ++j) {
                bar_wait(bar0 + 8 * (kBarAFull + s), ph);
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t at = tmem + kACol0 + s * kSetCols;
                if (pl[0].valid) issue(pl[0], at);
                int r2 = r + 1, t2 = t1;
                if (r2 == cpt) { r2 = 0; ++t2; }
                Plan nx[L];
#pragma unroll
                for (int w = 0; w < L; ++w) nx[w] = plan(r2, t2, w, q0, n_tiles);
#pragma unroll
                for (int w = 1; w < L; ++w)
                    if (pl[w].valid) issue(pl[w], at);
                if (leader) umma_commit(bar0 + 8 * (kBarAEmpty + s));
                if (++s == kSets) { s = 0; ph ^= 1; }
                r = r2; t1 = t2;
#pragma unroll
                for (int w = 0; w < L; ++w) pl[w] = nx[w];
            }
            q0 += n_tiles;
        })
    } else if (warp < kConvWarps) {
        const int q = warp & 3, kh = warp >> 2;              // TMEM lane quarter, column group of the chunk
        const int r = q * 32 + lane;
        const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16) + kACol0 + kh * kPer;
        // where this thread's kPer samples sit: float2 input = piece kh of two 128-byte pieces of 16 samples per row (two slots,
        // or -- mix on load -- two halves of one slot), int16 input = half kh of one piece of 32 samples
        const int piece = a.s16 ? 0 : kh;
        const int in_piece = a.s16 ? kh * kPer : 0;         // first sample inside the piece
        int slot = kMixIn ? 0 : piece;
        uint32_t sph = 0, s = 0, ph = 0;
        const int r_in = r & (kInRows - 1);                  // this thread's input row inside the row block
        const bool conj = kMixIn && q >= 2;                  // mix on load: rows 64..127 are the "490" channel (conjugate rotation)
        NVX_FOR_SEGMENTS({
            // mix on load: phase index of this thread's first sample of the chunk in the periodically continued NCO table; the
            // input sample at block index t sits at 63 kHz tick k_abs + t, and a chunk advances the phase by 28 mod 9 = 1
            int p9 = 0;
            if (kMixIn) {
                const long long t0 = (a.k_abs + (cpt * ta - lead) * kCS + kh * kPer) % kNcoPeriod;
                p9 = (int)(t0 < 0 ? t0 + kNcoPeriod : t0);
            }
            for (long long G = cpt * ta - lead; G < cpt * tb; ++G) {
                bar_wait(bar0 + 8 * (kBarRawFull + slot), sph);
                const uint8_t* row = s_raw + slot * kSlotBytes + (kMixIn ? piece * kHalfBytes : 0) + r_in * 128;
                float ih[kPer], il[kPer], qh[kPer], ql[kPer];
                if (G >= 0) {
                    if (a.s16) {
#pragma unroll
                        for (int u = 0; u < kPer / 4; ++u) {
                            const int4 v = *reinterpret_cast<const int4*>(row + (((in_piece / 4 + u) ^ (r & 7)) << 4));
                            const int wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                split_tf32((float)(short)(wv[j] & 0xFFFF), ih[4 * u + j], il[4 * u + j]);
                                split_tf32((float)(wv[j] >> 16), qh[4 * u + j], ql[4 * u + j]);
                            }
                        }
                    } else {
#pragma unroll
                        for (int u = 0; u < kPer / 2; ++u) {
                            float4 v = *reinterpret_cast<const float4*>(row + (((in_piece / 2 + u) ^ (r & 7)) << 4));
                            if (kCS != kKB && kh * kPer + 2 * u >= kCS) v = make_float4(0.f, 0.f, 0.f, 0.f);     // zero columns
                            if (kMixIn) {
                                const float2 m0 = mix_sample(make_float2(v.x, v.y), a.nco_tab[p9 + 2 * u], conj);
                                const float2 m1 = mix_sample(make_float2(v.z, v.w), a.nco_tab[p9 + 2 * u + 1], conj);
                                v = make_float4(m0.x, m0.y, m1.x, m1.y);
                            }
                            split_tf32(v.x, ih[2 * u], il[2 * u]);
                            split_tf32(v.y, qh[2 * u], ql[2 * u]);
                            split_tf32(v.z, ih[2 * u + 1], il[2 * u + 1]);
                            split_tf32(v.w, qh[2 * u + 1], ql[2 * u + 1]);
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < kPer; ++j) {
                        float2 v = make_float2(0.f, 0.f);
                        if (kh * kPer + j < kCS) v = tc_load(a, rb * kInRows + r_in, G * kCS + kh * kPer + j);
                        if (kMixIn) v = mix_sample(v, a.nco_tab[p9 + j], conj);
                        split_tf32(v.x, ih[j], il[j]);
                        split_tf32(v.y, qh[j], ql[j]);
                    }
                }
                if (kMixIn && ++p9 == kNcoPeriod) p9 = 0;
                __syncwarp();
                if (lane == 0) bar_arrive(bar0 + 8 * (kBarRawEmpty + slot));
                bar_wait(bar0 + 8 * (kBarAEmpty + s), ph ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t col = lane_base + s * kSetCols;
                tmem_st16(col + 0 * 32, ih);
                tmem_st16(col + 1 * 32, il);
                tmem_st16(col + 2 * 32, qh);
                tmem_st16(col + 3 * 32, ql);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;");
                __syncwarp();
                if (lane == 0) bar_arrive(bar0 + 8 * (kBarAFull + s));
                if (++s == kSets) { s = 0; ph ^= 1; }
                slot += slots_per_chunk;
                if (slot >= a.slots) { slot -= a.slots; sph ^= 1; }
            }
        })
    } else {
        // epilogue, as in fir_tc_kernel, on the accumulator slot of the tile
        const int q = warp & 3;
        const long long n_out = a.n_in / D;
        float* my_row = s_dump + (q * 32 + lane) * kDumpPitch;
        const float* rows0 = s_dump + (q * 32) * kDumpPitch;
        long long tq = 0;                                   // tiles handled so far (all segments)
        NVX_FOR_SEGMENTS({
            for (long long t = ta; t < tb; ++t, ++tq) {
                const uint32_t slot = (uint32_t)(tq % L);
                const long long n0 = t * N;
                const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + slot * kSlotCols;
                bar_wait(bar0 + 8 * (kBarTile + slot), (uint32_t)((tq / L) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;");
                // mix on load: this warp's 32 rows are the streams rb 64 + (q & 1) 32 .. of channel q >> 1; output rows are
                // channel rows, 2 stream + channel
                const int row0 = kMixIn ? rb * kInRows + (q & 1) * 32 : rb * kRows + q * 32;
                const int rows_left = (kMixIn ? a.rows_src : a.rows) - row0;
                const int r_max = rows_left < 32 ? rows_left : 32;
#pragma unroll 1
                for (int pass = 0; pass < N / NP; ++pass) {
                    if (pass) __syncwarp();
#pragma unroll 1
                    for (int h = 0; h < 2 * NP / 32; ++h) {
                        uint32_t v[32];
                        tmem_ld32(taddr + (h < NP / 32 ? pass * NP + h * 32 : N + pass * NP + (h - NP / 32) * 32), v);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            *reinterpret_cast<uint4*>(my_row + h * 32 + 4 * j) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    }
                    if (pass == N / NP - 1) asm volatile("tcgen05.fence::before_thread_sync;");
                    __syncwarp();
                    if (pass == N / NP - 1 && lane == 0) bar_arrive(bar0 + 8 * (kBarTmemFree + slot));
#pragma unroll 1
                    for (int h = 0; h < NP / 32; ++h) {
                        const int m = h * 32 + lane;
                        const int n = pass * NP + m;
                        if (n0 + n >= n_out) continue;
                        const long long tick = a.k_abs + n0 + n;
                        if (!a.mix) {
                            const long long out_step = kMixIn ? 2 * a.out_pitch : a.out_pitch;
                            float2* dst1 = a.out + (size_t)(kMixIn ? 2 * row0 + (q >> 1) : row0) * a.out_pitch + a.out_off + n0 + n;
#pragma unroll 4
                            for (int rr = 0; rr < r_max; ++rr, dst1 += out_step)
                                *dst1 = make_float2(rows0[rr * kDumpPitch + m], rows0[rr * kDumpPitch + NP + m]);
                            continue;
                        }
                        float2* dst = a.out + (size_t)(2 * row0) * a.out_pitch + a.out_off + n0 + n;
                        if (a.nco) {
                            const long long rden = tick % kNcoDen;
                            const long long kden = rden < 0 ? rden + kNcoDen : rden;
#pragma unroll 2
                            for (int rr = 0; rr < r_max; ++rr, dst += 2 * a.out_pitch) {
                                const NcoChan nc[2] = {a.nco[2 * (row0 + rr)], a.nco[2 * (row0 + rr) + 1]};
                                const float2 y = make_float2(rows0[rr * kDumpPitch + m], rows0[rr * kDumpPitch + NP + m]);
#pragma unroll
                                for (int c = 0; c < 2; ++c) {
                                    const int phs = (int)((kden * nc[c].num + nc[c].phase0) % kNcoDen);
                                    float tt = (float)phs * (2.0f / kNcoDen);
                                    if (tt > 1.0f) tt -= 2.0f;
                                    float sn, cs;
                                    sincospif(tt, &sn, &cs);
                                    dst[c * a.out_pitch] = make_float2(fmaf(y.y, sn, y.x * cs), fmaf(-y.x, sn, y.y * cs));
                                }
                            }
                        } else {
                            const long long r9 = tick % kNcoPeriod;
                            const float2 rot = s_nco[r9 < 0 ? r9 + kNcoPeriod : r9];
#pragma unroll 4
                            for (int rr = 0; rr < r_max; ++rr, dst += 2 * a.out_pitch) {
                                const float2 y = make_float2(rows0[rr * kDumpPitch + m], rows0[rr * kDumpPitch + NP + m]);
                                dst[0] = make_float2(fmaf(-y.y, rot.y, y.x * rot.x), fmaf(y.x, rot.y, y.y * rot.x));
                                dst[a.out_pitch] = make_float2(fmaf(y.y, rot.y, y.x * rot.x), fmaf(-y.x, rot.y, y.y * rot.x));
                            }
                        }
                    }
                }
                __syncwarp();
            }
        })
    }
#undef NVX_FOR_SEGMENTS
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
}

float tf32_rna(float x) {                  // round to nearest, ties away, 10-bit mantissa (cvt.rna.tf32.f32)
    uint32_t u;
    memcpy(&u, &x, 4);
    u = (u + 0x1000u) & 0xFFFFE000u;
    memcpy(&x, &u, 4);
    return x;
}

int tc_chunks(int D, int N, int T) { return (D * (N - 1) + T + chunk_samples(D) - 1) / chunk_samples(D); }
// streaming kernel geometry: chunks per tile advance, and the chunks a window leads its tile by for T_taps taps (the tap count is
// padded to D + lead * chunk so that tile windows are whole chunks of ONE global grid)
int tcs_cpt(int D) { return D * kSN / chunk_samples(D); }
int tcs_lead(int D, int T_taps) { return T_taps <= D ? 0 : (T_taps - D + chunk_samples(D) - 1) / chunk_samples(D); }
// rows of one copy of the band matrix: N plus one 8-row atom per further (group of) chunk(s)
int tc_band_rows(int D, int N, int T) { return N + 8 * ((tc_chunks(D, N, T) - 1) / band_copies(D)); }
size_t tc_smem(int D, int N, int T, int slots, int L = 2) {
    return (size_t)2 * band_copies(D) * tc_band_rows(D, N, T) * 128 + (size_t)slots * kSlotBytes + (size_t)kRows * (2 * dump_outputs(D, N, L) + kDumpPad) * 4 + 128 +
           kBars * 8 + 16;
}
int tc_box_rows(int J) {                   // whole swizzle atoms, at most 256 rows, dividing J
    int best = 1;
    for (int d = 1; d <= 32; ++d)
        if ((J / 8) % d == 0) best = d;
    return 8 * best;
}
int tc_slots(int D, int N, int T, int L = 2) {        // raw-input slots that fit beside the band matrix: even, >= 4 (0: the stage does not fit)
    for (int slots = kMaxSlots; slots >= 4; slots -= 2)
        if (tc_smem(D, N, T, slots, L) <= (size_t)kSmemLimit) return slots;
    return 0;
}

template <int D, int L, bool kMixIn = false>
cudaError_t launch_tcs(TcArgs& a, int sms, cudaStream_t stream) {
    a.slots = tc_slots(D, kSN, a.T, L);
    const size_t smem = tc_smem(D, kSN, a.T, a.slots, L);
    cudaError_t e = cudaFuncSetAttribute(fir_tcs_kernel<D, L, kMixIn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const long long grid = a.work < sms ? a.work : sms;
    fir_tcs_kernel<D, L, kMixIn><<<(unsigned)grid, kTcThreads, smem, stream>>>(a);
    return cudaGetLastError();
}

template <int D, int N>
cudaError_t launch_tc(TcArgs& a, int sms, cudaStream_t stream) {
    a.slots = tc_slots(D, N, a.T);
    const size_t smem = tc_smem(D, N, a.T, a.slots);
    cudaError_t e = cudaFuncSetAttribute(fir_tc_kernel<D, N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const long long grid = a.work < sms ? a.work : sms;
    fir_tc_kernel<D, N><<<(unsigned)grid, kTcThreads, smem, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace

// outputs per tile for (D, T); 0 = the stage is not served by the tensor-core kernel
int long_tc_tile(int D, int T) {
    if (D != NVX_D1 && D != NVX_D2) return 0;
    // measured with the data operand in tensor memory (tools/probes/umma_ts_probe.cu): 23 / 36 / 64 cycles per tcgen05.mma at
    // N = 32 / 64 / 128, i.e. 211 / 218 / 288 cycles per output column at 255 taps; N = 64 halves the re-read of N = 32.  N = 128
    // (stage 1 only: 1.5x instead of 2x re-read, but two A sets and a two-pass epilogue) wins from ~400 taps on: 511 taps 131
    // against 122 Gsamples/s, 255 taps 183 against 190.  No N = 32 kernel: at stage 1, N = 64 fits every tap count up to
    // kLongMaxTaps; stage 2 takes N = 64 only (fits up to 959 taps): with N = 32 tiles the CUDA-core kernel is faster
    if (D == NVX_D1 && T >= 384 && tc_slots(D, 128, T)) return 128;
    return tc_slots(D, 64, T) ? 64 : 0;
}

// the streaming kernel serves a stage when a window spans at most three tiles (lead <= 2 x chunks per tile) and its band fits
bool tcs_applies(int D, int T_taps) {
    if (D != NVX_D1 && D != NVX_D2) return false;
    const int lead = tcs_lead(D, T_taps);
    return lead <= 2 * tcs_cpt(D) && tc_slots(D, kSN, D + lead * chunk_samples(D), lead > tcs_cpt(D) ? 3 : 2) > 0;
}

struct LongTcStage {
    int D = 0, T = 0, N = 0, chunks = 0, J = 0, box_rows = 0;
    bool streaming = false;
    float *d_gh = nullptr, *d_gl = nullptr;
    CUtensorMap map_gh, map_gl;
};

// host side of the band matrix (no GPU needed; also behind nvx_debug_long_tc_band for the CPU tests): padded tap count, tile
// width, chunk count, rows per copy, copies, and the hi / lo TF32 parts [copies][J][32]
bool long_tc_band(int D, int T_taps, const double* h, TcBand* b) {
    // zero taps appended at the old end until the tile windows (first sample D n0 + D - T, n0 a multiple of 32) start on a whole
    // 32-byte sector = 4 samples: TMA box origins and cp.async pieces need 16-byte alignment, and aligned rows cost 8 sectors
    // instead of 9
    int T = T_taps;
    while ((D - T) & 3) ++T;
    int N;
    b->streaming = tcs_applies(D, T_taps);
    if (b->streaming) {        // streaming kernel: windows are whole chunks of one global grid, T = D + lead * chunk
        T = D + tcs_lead(D, T_taps) * chunk_samples(D);
        N = kSN;
    } else {
        N = long_tc_tile(D, T);
    }
    if (!N) return false;
    b->T = T; b->N = N;
    b->chunks = tc_chunks(D, N, T);
    b->J = tc_band_rows(D, N, T);
    b->copies = band_copies(D);
    const int P = b->copies, CS = chunk_samples(D), M1 = (b->chunks - 1) / P;
    b->gh.assign((size_t)P * b->J * kKB, 0.f);
    b->gl.assign((size_t)P * b->J * kKB, 0.f);
    for (int p = 0; p < P; ++p)
        for (int j = 0; j < b->J; ++j)
            for (int k = 0; k < CS; ++k) {
                // chunk c = P m + p reads copy p from atom M1 - m on: its row j is output n = j - 8 (M1 - m), whose tap for sample
                // k of the chunk is D n + T - 1 - (CS c + k) = D (j - 8 M1) + T - 1 - CS p - k   (8 D = CS P)
                const int i = D * (j - 8 * M1) + T - 1 - CS * p - k;
                if (i >= 0 && i < T_taps) {
                    const float t = (float)h[i];
                    b->gh[((size_t)p * b->J + j) * kKB + k] = tf32_rna(t);
                    b->gl[((size_t)p * b->J + j) * kKB + k] = t - tf32_rna(t);
                }
            }
    return true;
}

// builds the band matrix of the stage on the device; returns nullptr if the stage does not fit the tensor-core kernel
LongTcStage* long_tc_prepare(int D, int T_taps, const double* h, cudaStream_t stream) {
    TcBand band;
    if (!long_tc_band(D, T_taps, h, &band)) return nullptr;
    const EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return nullptr;
    LongTcStage* s = new LongTcStage();
    s->D = D; s->T = band.T; s->N = band.N;
    s->streaming = band.streaming;
    s->chunks = band.chunks;
    s->J = band.J;
    s->box_rows = tc_box_rows(s->J);
    const int P = band.copies;
    const std::vector<float>&gh = band.gh, &gl = band.gl;
    bool ok = cudaMalloc(&s->d_gh, gh.size() * 4) == cudaSuccess && cudaMalloc(&s->d_gl, gl.size() * 4) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->d_gh, gh.data(), gh.size() * 4, cudaMemcpyHostToDevice, stream) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(s->d_gl, gl.data(), gl.size() * 4, cudaMemcpyHostToDevice, stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(stream) == cudaSuccess;
    if (ok) {
        cuuint64_t dims[2] = {(cuuint64_t)kKB, (cuuint64_t)P * s->J};
        cuuint64_t strides[1] = {(cuuint64_t)kKB * 4};
        cuuint32_t box[2] = {kKB, (cuuint32_t)s->box_rows};
        cuuint32_t es[2] = {1, 1};
        ok = enc(&s->map_gh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, s->d_gh, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS &&
             enc(&s->map_gl, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, s->d_gl, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    }
    if (!ok) {
        cudaFree(s->d_gh); cudaFree(s->d_gl);
        delete s;
        return nullptr;
    }
    return s;
}

void long_tc_free(LongTcStage* s) {
    if (!s) return;
    cudaFree(s->d_gh); cudaFree(s->d_gl);
    delete s;
}

// same contract as long_launch (fir_long.cu) for stages 0 and 1; cudaErrorNotSupported = this block cannot be described to the TMA
// unit (misaligned pointer or pitch): the caller falls back to long_launch
bool long_tc_mixes_on_load(const LongTcStage* s) { return s && s->D == NVX_D2 && s->streaming; }

cudaError_t long_tc_launch(const LongTcStage* s, const LongArgs& la, const LongStage& st, long long in_pitch, cudaStream_t stream) {
    if (la.mix_in && !long_tc_mixes_on_load(s)) return cudaErrorInvalidValue;
    TcArgs a = {};
    a.map_gh = s->map_gh; a.map_gl = s->map_gl;
    a.in = la.in; a.hist = la.hist; a.out = la.out;
    a.n_in = la.n_in; a.in_pitch = in_pitch; a.out_pitch = la.out_pitch; a.out_off = la.out_off; a.k_abs = la.k_abs;
    a.nco = la.nco; a.rows = la.rows_in; a.s16 = la.s16; a.T = s->T; a.H = st.H; a.chunks = s->chunks; a.J = s->J; a.slots = 4; a.box_rows = s->box_rows;
    a.mix = la.stage == 0 && !la.plain;
    a.rows_src = la.mix_in ? la.rows_in / 2 : la.rows_in;
    for (int k = 0; k < kNcoPeriod + 16; ++k) a.nco_tab[k] = reference_nco(k % kNcoPeriod);
    // TMA boxes and 16-byte cp.async pieces: the block and its rows must start on 16-byte boundaries (tile windows do by
    // construction).  The block as a 2-D tensor of 32-bit (float2 input) or 16-bit (short2 input) elements, two per sample:
    if (((uintptr_t)la.in & 15) || ((in_pitch * (la.s16 ? 4 : 8)) & 15)) return cudaErrorNotSupported;
    a.cpt = tcs_cpt(s->D);
    a.lead = s->chunks - a.cpt;
    if (chunk_samples(s->D) == kKB || s->streaming) {
        const size_t esz = la.s16 ? 2 : 4;
        cuuint64_t dims[2] = {(cuuint64_t)(2 * la.n_in), (cuuint64_t)a.rows_src};
        cuuint64_t strides[1] = {(cuuint64_t)in_pitch * 2 * esz};
        cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)(la.mix_in ? kRows / 2 : kRows)};
        cuuint32_t es[2] = {1, 1};
        if (tensor_map_encoder()(&a.map_x, la.s16 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(la.in), dims, strides,
                   box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorNotSupported;
    }
    const long long n_out = la.n_in / s->D;
    a.tiles_per_block = (n_out + s->N - 1) / s->N;
    a.work = (long long)((la.rows_in + kRows - 1) / kRows) * a.tiles_per_block;
    if (a.work <= 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (s->streaming) {
        const bool three = a.lead > a.cpt;
        return s->D == NVX_D1 ? (three ? launch_tcs<NVX_D1, 3>(a, sms, stream) : launch_tcs<NVX_D1, 2>(a, sms, stream))
               : la.mix_in    ? (three ? launch_tcs<NVX_D2, 3, true>(a, sms, stream) : launch_tcs<NVX_D2, 2, true>(a, sms, stream))
                              : (three ? launch_tcs<NVX_D2, 3>(a, sms, stream) : launch_tcs<NVX_D2, 2>(a, sms, stream));
    }
    // the tile widths long_tc_tile picks
    if (s->D == NVX_D1 && s->N == 128) return launch_tc<NVX_D1, 128>(a, sms, stream);
    if (s->D == NVX_D1 && s->N == 64) return launch_tc<NVX_D1, 64>(a, sms, stream);
    if (s->D == NVX_D2 && s->N == 64) return launch_tc<NVX_D2, 64>(a, sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace nvx

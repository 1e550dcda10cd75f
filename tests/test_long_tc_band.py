"""Host logic of the tensor-core long-tap kernel (navtex_b200/csrc/fir_long_tc.cu), checked on the CPU: the band-matrix
operand and its chunk addressing must turn the decimating FIR of the reference stages

    y[k] = sum_{i < T} h[i] x[D (k + 1) - 1 - i]        fir1cpp.C:80-136 (D = 4), fir2cpp.C:131-215 (D = 7)

into the chunked GEMM the kernel issues: per tile of N outputs, for every K chunk c, [rows x 32 window columns] times
rows [8 ((chunks - 1) / copies - c / copies), + N) of band copy c % copies.  The GEMM is emulated in numpy (FP64, hi + lo
parts) exactly as the issuer warp addresses it; the GPU tests then cover the kernel itself."""
import numpy as np
import pytest
from scipy import signal

from navtex_b200 import engine


@pytest.mark.parametrize("D,T", [(4, 255), (4, 256), (4, 101), (4, 511), (4, 62), (7, 255), (7, 383), (7, 76), (7, 512)])
def test_band_gemm_equals_the_decimating_fir(D, T):
    rng = np.random.default_rng(D * 1000 + T)
    h = signal.firwin(T, 0.2 / D, window=("kaiser", 8.0)) + 1e-3 * rng.normal(size=T)      # no symmetry to hide an index flip
    geo, g_hi, g_lo = engine.long_tc_band(D, h)
    N, chunks, J, P, Tp = geo["n_tile"], geo["chunks"], geo["band_rows"], geo["copies"], geo["taps_padded"]
    cs = 32 // D * D                                            # samples per chunk
    cpt = D * N // cs                                           # chunks a tile advances by
    lead = -(-(T - D) // cs)
    if lead <= 2 * cpt and N == 64:                             # streaming kernel (two or three live tiles): windows are whole chunks of one global grid
        assert Tp == D + lead * cs and chunks == cpt + lead and chunks * cs == D * (N - 1) + Tp
    else:                                                       # tile-at-a-time kernel: windows start on whole 32-byte sectors
        assert (D - Tp) % 4 == 0 and T <= Tp < T + 4
    assert chunks * cs >= D * (N - 1) + Tp and J == N + 8 * ((chunks - 1) // P) and P == 8 // (cs // D)
    g = g_hi.astype(np.float64) + g_lo.astype(np.float64)
    assert not g[:, :, cs:].any()                               # the zero columns of a 28-sample chunk
    # TF32 split of the taps: hi has a 10-bit mantissa, hi + lo is the float tap
    assert np.all((g_hi.view(np.uint32) & 0x1FFF) == 0)
    n_tiles = 3
    x = rng.normal(size=D * N * n_tiles + 64)
    hist = Tp + 40                                              # samples before the block (the carried history)
    xx = np.concatenate([rng.normal(size=hist), x])
    for tile in range(n_tiles):
        n0 = tile * N
        t_base = D * n0 + D - Tp                                # first sample of the tile's window (block-relative)
        y = np.zeros(N)
        for c in range(chunks):
            a = np.zeros(32)
            w0 = hist + t_base + cs * c
            a[:cs] = xx[w0:w0 + cs]
            r0 = 8 * ((chunks - 1) // P - c // P)
            y += g[c % P, r0:r0 + N, :] @ a
        want = np.array([sum(h[i] * xx[hist + D * (n0 + n + 1) - 1 - i] for i in range(T)) for n in range(N)])
        assert np.abs(y - want).max() <= 2e-7 * np.abs(want).max() + 1e-9, (tile, np.abs(y - want).max())


def test_band_is_refused_where_the_kernel_does_not_apply():
    h = np.ones(300)
    with pytest.raises(engine.NvxError):
        engine.long_tc_band(10, h)                              # stage 3 stays on CUDA cores
    with pytest.raises(engine.NvxError):
        engine.long_tc_band(7, np.ones(1000))                   # stage 2 beyond 959 taps: only N = 32 tiles would fit
    geo, _, _ = engine.long_tc_band(4, np.ones(1000))
    assert geo["n_tile"] == 64
    geo, _, _ = engine.long_tc_band(4, np.ones(511))
    assert geo["n_tile"] == 64 and geo["taps_padded"] == 516 and geo["chunks"] == 24       # streaming with three live tiles: 8 + 16 chunks
    geo, _, _ = engine.long_tc_band(4, np.ones(540))
    assert geo["n_tile"] == 128                                 # beyond 516 taps: tile at a time, N = 128 while the band fits (to 548)
    geo, _, _ = engine.long_tc_band(4, np.ones(255))
    assert geo["n_tile"] == 64 and geo["taps_padded"] == 260 and geo["chunks"] == 16      # streaming: 8 + 8 chunks of 32 samples
    geo, _, _ = engine.long_tc_band(7, np.ones(255))
    assert geo["n_tile"] == 64 and geo["taps_padded"] == 259 and geo["chunks"] == 25      # streaming: 16 + 9 chunks of 28 samples
    geo, _, _ = engine.long_tc_band(7, np.ones(959))
    assert geo["n_tile"] == 64 and geo["copies"] == 2


def test_every_tap_count_lands_on_a_built_tile_width():
    # the tile-at-a-time kernel is only instantiated for N = 128 and 64 at D = 4 and N = 64 at D = 7 (the streaming kernel's
    # N is 64 too): every tap count the engine accepts, 1 .. 1024 per stage, must map to one of those or be refused
    for T in range(1, 1025):
        h = np.ones(T)
        geo, _, _ = engine.long_tc_band(4, h)
        assert geo["n_tile"] == (128 if 517 <= T <= 548 else 64), (T, geo)
        if T >= 960:
            with pytest.raises(engine.NvxError):
                engine.long_tc_band(7, h)
        else:
            geo, _, _ = engine.long_tc_band(7, h)
            assert geo["n_tile"] == 64, (T, geo)

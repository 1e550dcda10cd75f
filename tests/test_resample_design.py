"""The rational resampler of engines fed at another rate than 252 kS/s, on the host (no GPU): nvx_resampler_info's L / M,
alignment and taps, the taps' response, and the output formula the kernel is tested against, modelled in numpy."""
from math import gcd

import numpy as np
import pytest
from scipy import signal

from navtex_b200 import engine

# rate: (L, M, align, 252 k samples per align, restart grid in input samples)
TABLE = {
    96_000: (21, 8, 320, 840, 60_480), 192_000: (21, 16, 640, 840, 120_960), 250_000: (126, 125, 2_500, 2_520, 157_500),
    256_000: (63, 64, 2_560, 2_520, 161_280), 912_000: (21, 76, 3_040, 840, 574_560), 2_016_000: (1, 8, 2_240, 280, 1_270_080),
    2_048_000: (63, 512, 20_480, 2_520, 1_290_240), 2_400_000: (21, 200, 8_000, 840, 1_512_000),
    3_200_000: (63, 800, 32_000, 2_520, 2_016_000),
}

# many polyphase branches: L = 2520 at both ends of the range, L = 840 at a high rate
MANY_BRANCHES = (96_100, 2_000_100, 3_199_900)


@pytest.mark.parametrize("rate", sorted(TABLE))
def test_table(rate):
    L, M, align, per_align, grid = TABLE[rate]
    info = engine.resampler_info(rate)
    assert (info["up"], info["down"], info["align"]) == (L, M, align)
    assert align == rate // gcd(rate, 900) and align * L // M == per_align and per_align % 280 == 0
    assert 158_760 * M % L == 0 and 158_760 * M // L == grid == round(0.63 * rate)
    assert 2520 % L == 0                          # the cascade's 2520-sample period falls on whole input samples
    assert info["taps"].size % L == 0


def test_many_branches():
    for rate in MANY_BRANCHES:
        info = engine.resampler_info(rate)
        q = rate // 100
        assert info["up"] == 2520 // gcd(2520, q) and info["down"] == q // gcd(2520, q)
        assert info["align"] == rate // gcd(rate, 900)
    assert engine.resampler_info(96_100)["up"] == 2520 and engine.resampler_info(2_000_100)["up"] == 840


def test_native_and_rejected():
    info = engine.resampler_info(252_000)
    assert (info["up"], info["down"], info["align"]) == (1, 1, 280)
    assert info["taps"].tolist() == [1.0]
    for bad in (95_900, 3_200_100, 250_001, 0, -256_000, 3_300_000, 50_000):
        with pytest.raises(engine.NvxError, match="input rate"):
            engine.resampler_info(bad)


@pytest.mark.parametrize("rate", sorted(TABLE) + list(MANY_BRANCHES))
def test_response(rate):
    """Pass band +-31.5 kHz within 0.01 dB, stop band from min(r, 252000) - 31.5 kHz at least 80 dB down (relative to the DC gain
    L), every polyphase branch summing to 1 within 1e-3; and the same for the float rounding the kernel uses.  The response is
    sampled by an FFT zero-padded to at least 8 times the length (and at least 2^20 points)."""
    info = engine.resampler_info(rate)
    L, h = info["up"], info["taps"]
    assert h.size == info["up"] * (h.size // info["up"])
    fs = L * rate
    f_pass, f_stop = 31_500.0, min(rate, 252_000) - 31_500.0
    nfft = 1 << max(20, int(np.ceil(np.log2(8 * h.size))))
    f = np.arange(nfft // 2 + 1) * fs / nfft
    for taps in (h, h.astype(np.float32).astype(np.float64)):
        g = np.abs(np.fft.rfft(taps, nfft)) / L
        pb, sb = g[f <= f_pass], g[f >= f_stop]
        assert pb.size > 8
        assert 20 * np.log10(pb.max() / pb.min()) <= 0.01
        assert 20 * np.log10(sb.max()) <= -80.0, (rate, 20 * np.log10(sb.max()))
        sums = taps.reshape(-1, L).sum(axis=0)                # branch p = taps[p::L]
        assert np.abs(sums - 1).max() <= 1e-3


def model(h, L, M, x, k0, n_out, hist):
    """The kernel's formula for outputs k0 .. k0 + n_out - 1 (absolute): y[k] = sum_j h[p + j L] x[t - j], t = floor(k M / L),
    p = k M - t L, with x given from absolute index i0 = k0 M / L on and `hist` the samples before it."""
    J = h.size // L
    i0 = k0 * M // L
    xx = np.concatenate([hist, x])
    base = i0 - hist.size
    k = np.arange(k0, k0 + n_out)
    t, p = k * M // L, (k * M) % L
    y = np.zeros(n_out, dtype=np.complex128)
    for j in range(J):
        y += h[p + j * L] * xx[t - j - base]
    return y


@pytest.mark.parametrize("rate", [96_000, 250_000, 256_000, 912_000, 2_400_000, 96_100])
def test_formula_is_upfirdn(rate):
    """The formula equals scipy's upfirdn on random data, in one block and in uneven aligned blocks with the history carried."""
    info = engine.resampler_info(rate)
    L, M, align, h = info["up"], info["down"], info["align"], info["taps"]
    J = h.size // L
    rng = np.random.default_rng(rate)
    blocks = [align * k for k in (1, 3, 2, 5)]
    n = sum(blocks)
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    want = signal.upfirdn(h, x, L, M)[: n * L // M]
    one = model(h, L, M, x, 0, n * L // M, np.zeros(J - 1, complex))
    assert np.abs(one - want).max() <= 1e-12 * np.abs(want).max()
    got, hist, at = [], np.zeros(J - 1, complex), 0
    for b in blocks:
        got.append(model(h, L, M, x[at:at + b], at * L // M, b * L // M, hist))
        hist = np.concatenate([hist, x[at:at + b]])[-(J - 1):]
        at += b
    assert np.abs(np.concatenate(got) - want).max() <= 1e-12 * np.abs(want).max()

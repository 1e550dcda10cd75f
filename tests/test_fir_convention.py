"""CPU test: the tap order and NCO convention of the oracle (oracle/navtex_oracle.c), pinned against an independent numpy
float64 statement of the cascade with asymmetric taps.

The reference taps are symmetric, so the oracle's agreement with the compiled reference says nothing about which end of a
replacement tap set weighs the newest sample.  Here every stage is stated directly:

    y[k] = sum_i h[i] x[D (k + 1) - 1 - i]          (h[0] weighs the newest sample; zero history before the first input)

and channel c multiplies the 63 kHz sample k by exp(-2 pi i ((k f_c) mod 63000) / 63000) before its stage 2.  With random
taps a reversed, shifted or dropped tap moves every output by about 1 / sqrt(T) of its peak."""
import numpy as np
import pytest

import oracle_lib as ol

D1, D2, D3 = 4, 7, 10
REL = 1e-10          # float64 against float64: measured 1e-15, 1e-12 at -31 499.5 Hz (long NCO table period)


def decimating_fir(x, h, D):
    """y[k] = sum_i h[i] x[D (k + 1) - 1 - i] for k < len(x) // D, x zero before index 0."""
    full = np.convolve(x, h)                    # full[n] = sum_i h[i] x[n - i]
    return full[D - 1: D * (len(x) // D): D]


def mix(y1, f):
    k = np.arange(len(y1), dtype=np.float64)
    return y1 * np.exp(-2j * np.pi * np.mod(k * f, 63000.0) / 63000.0)


def rand_taps(rng, T):
    h = rng.normal(size=T)
    return h / np.abs(h).sum()


CASES = [((37, 47, 71), (14000.0, -14000.0, 5000.5)),
         ((255, 900, 112), (9500.0, -4500.5)),
         ((1, 1, 1), (0.5, -31499.5)),
         ((61, 75, 111), (-14000.0, 3.5, 20999.5))]


@pytest.mark.parametrize("lengths,nco", CASES, ids=["%d-%d-%d" % c[0] for c in CASES])
def test_oracle_tap_order_and_mix(lengths, nco):
    rng = np.random.default_rng(sum(lengths))
    h1, h2, h3 = (rand_taps(rng, T) for T in lengths)
    n = 280 * 300
    iq = np.rint(rng.normal(0.0, 3000.0, size=2 * n)).astype(np.int16)
    o = ol.run_oracle(iq, h1=h1, h2=h2, h3=h3, nco_hz=nco)

    x = iq[0::2].astype(np.float64) + 1j * iq[1::2].astype(np.float64)
    y1 = decimating_fir(x, h1, D1)
    assert len(o.y1) == len(y1)
    assert np.abs(o.y1 - y1).max() <= REL * np.abs(y1).max()
    for c, f in enumerate(nco):
        tag = ol.CHANNEL_KEYS[c]
        y2 = decimating_fir(mix(y1, f), h2, D2)
        y3 = decimating_fir(y2, h3, D3)
        assert len(o.y2[tag]) == len(y2) and len(o.y3[tag]) == len(y3) == n // 280
        assert np.abs(o.y2[tag] - y2).max() <= REL * np.abs(y2).max(), (tag, f)
        assert np.abs(o.y3[tag] - y3).max() <= REL * np.abs(y3).max(), (tag, f)


def test_reversed_taps_are_seen():
    """The statement above is not blind to tap order: reversing the stage-1 taps of an asymmetric set moves y3 by more than
    a percent of its peak."""
    rng = np.random.default_rng(5)
    h1, h2, h3 = (rand_taps(rng, T) for T in (37, 47, 71))
    x = rng.normal(size=280 * 50) + 1j * rng.normal(size=280 * 50)
    fwd = decimating_fir(decimating_fir(mix(decimating_fir(x, h1, D1), 14000.0), h2, D2), h3, D3)
    rev = decimating_fir(decimating_fir(mix(decimating_fir(x, h1[::-1], D1), 14000.0), h2, D2), h3, D3)
    assert np.abs(fwd - rev).max() > 1e-2 * np.abs(fwd).max()

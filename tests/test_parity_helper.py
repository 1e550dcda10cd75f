"""CPU test of tests/parity.py, the comparison behind every "1e-5 relative" claim: denominators, bit-decision bookkeeping and the
timing-slip attribution, on oracle output perturbed in known ways (no GPU involved)."""
import numpy as np

import cases
import oracle_lib as ol
import parity


def _as_gpu(o, scale_err=0.0, flip=None, seed=0, keys=ol.CHANNELS, err_rows=None):
    """Dress an oracle result up as GPU taps: complex64 samples (+ optional relative perturbation of the channel indices
    err_rows, default all), bits with optional flips."""
    rng = np.random.default_rng(seed)
    y3 = np.stack([o.y3[t] for t in keys]).astype(np.complex64)
    if scale_err:
        peak = np.abs(y3).max()
        rows = list(range(len(keys))) if err_rows is None else err_rows
        shape = (len(rows), y3.shape[1])
        y3[rows] += (scale_err * peak * (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / 4).astype(np.complex64)
    bits = {c: bytearray(o.bits[t]) for c, t in enumerate(keys)}
    for c, k in (flip or []):
        bits[c][k] = ord("B") if bits[c][k] == ord("Y") else ord("Y")
    return y3, {c: bytes(b) for c, b in bits.items()}, {c: o.disc[t].copy() for c, t in enumerate(keys)}


def test_identical_taps_pass_and_float32_rounding_is_measured():
    o = ol.run_oracle(cases.build("clean518"))
    y3, bits, disc = _as_gpu(o)
    cmp = parity.compare_stream(y3, bits, disc, o, {"518"})
    parity.assert_stream(cmp, {"518"})
    assert 0 < cmp["y3_rel_pair_peak"] < 1e-7                       # complex64 rounding of FP64 samples
    assert cmp["bit_mismatches"] == {"518": 0, "490": 0} and cmp["disc_rel"]["518"] == 0.0
    assert cmp["y3_rel_own_rms"]["518"] >= cmp["y3_rel_pair_peak"]   # the RMS of a channel is below the pair peak: the tighter bar


def test_errors_beyond_the_bar_and_flipped_decisions_fail():
    import pytest

    o = ol.run_oracle(cases.build("clean518"))
    y3, bits, disc = _as_gpu(o, scale_err=1e-4)
    with pytest.raises(AssertionError):
        parity.assert_stream(parity.compare_stream(y3, bits, disc, o, {"518"}), {"518"})
    y3, bits, disc = _as_gpu(o, flip=[(0, 100)])
    cmp = parity.compare_stream(y3, bits, disc, o, {"518"})
    assert cmp["bit_mismatches"]["518"] == 1 and len(cmp["mismatch_margins"]["518"]) == 1
    with pytest.raises(AssertionError):
        parity.assert_stream(cmp, {"518"})


def test_empty_channel_differences_are_reported_not_asserted():
    o = ol.run_oracle(cases.build("clean518"))
    y3, bits, disc = _as_gpu(o, flip=[(1, 50), (1, 51), (1, 52), (1, 400)])
    cmp = parity.compare_stream(y3, bits, disc, o, {"518"})
    parity.assert_stream(cmp, {"518"})                               # the empty channel's decisions are counted, not required equal
    assert cmp["bit_mismatches"]["490"] == 4 and len(cmp["mismatch_margins"]["490"]) == 4
    assert all(0.0 <= m <= 1.0 for m in cmp["mismatch_margins"]["490"])
    # two runs of differences, each attributed to the tightest arg max of the 64 evaluations before it
    assert len(cmp["timing_slip_pick_margins"]["490"]) == 2 and all(0.0 <= m <= 1.0 for m in cmp["timing_slip_pick_margins"]["490"])
    s = parity.summarise([cmp], [{"518"}])
    assert s["bit_mismatches_occupied"] == 0 and s["empty_channel_bit_mismatches"] == 4 and s["empty_channel_bits_compared"] == len(o.bits["490"])


def test_three_channels_every_channel_is_compared():
    """More than the reference pair (channels=CHANNEL_KEYS[:C]): the bulletin at +14 kHz sits in channel index 2 ("ch2"), the
    other two are empty.  An error or a flipped decision that touches only the third channel is caught; the empty channels'
    decisions are counted as for the pair."""
    import pytest

    keys = ol.CHANNEL_KEYS[:3]
    o = ol.run_oracle(cases.build("clean518"), nco_hz=(7000.0, -14000.0, 14000.0), freq_tag=(511, 490, 518))
    assert [m[0] for m in o.messages] == [518] and len(o.bits["ch2"]) > 0
    occ = {"ch2"}
    y3, bits, disc = _as_gpu(o, keys=keys)
    cmp = parity.compare_stream(y3, bits, disc, o, occ, channels=keys)
    parity.assert_stream(cmp, occ)
    assert set(cmp["bit_mismatches"]) == set(keys) and set(cmp["y3_rel_own_rms"]) == occ
    assert set(cmp["empty_rel_own_rms"]) == {"518", "490"} and cmp["disc_rel"]["ch2"] == 0.0
    assert 0 < cmp["y3_rel_pair_peak"] < 1e-7
    y3, bits, disc = _as_gpu(o, keys=keys, scale_err=1e-4, err_rows=[2])       # the third channel alone is off
    with pytest.raises(AssertionError):
        parity.assert_stream(parity.compare_stream(y3, bits, disc, o, occ, channels=keys), occ)
    y3, bits, disc = _as_gpu(o, keys=keys, flip=[(2, 100)])
    cmp = parity.compare_stream(y3, bits, disc, o, occ, channels=keys)
    assert cmp["bit_mismatches"]["ch2"] == 1
    with pytest.raises(AssertionError):
        parity.assert_stream(cmp, occ)
    y3, bits, disc = _as_gpu(o, keys=keys, flip=[(0, 50), (1, 60)])
    cmp = parity.compare_stream(y3, bits, disc, o, occ, channels=keys)
    parity.assert_stream(cmp, occ)                                           # empty channels: counted, not required equal
    y3, bits, disc = _as_gpu(o, keys=keys)
    bits[1] = bits[1][:-1]                                                   # ... but an empty channel must keep its length
    short = parity.compare_stream(y3, bits, disc, o, occ, channels=keys)
    with pytest.raises(AssertionError):
        parity.assert_stream(short, occ)
    parity.assert_stream(short, occ, unbounded={"490"})                      # unless it is tuned into the stage-1 stopband
    with pytest.raises(AssertionError):
        parity.assert_stream(short, occ, unbounded={"518"})
    assert short["bit_len_diff"]["490"] == -1 and short["length_slip"]["490"]["first_diverging_decision"] == len(bits[1]) - 1
    tie = short["length_slip"]["490"]["pick_margin"]                         # or the slip follows an arg max near-tie
    parity.assert_stream(short, occ, near_tie=tie)
    with pytest.raises(AssertionError):
        parity.assert_stream(short, occ, near_tie=tie / 2)
    s = parity.summarise([cmp], [occ])
    assert s["empty_channels"] == 2 and s["empty_channel_bit_mismatches"] == 2 and s["bit_mismatches_occupied"] == 0
    assert s["empty_channel_bits_compared"] == len(o.bits["518"]) + len(o.bits["490"])

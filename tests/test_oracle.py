"""CPU tests: the oracle (C restatement) against the golden fixtures generated from the unmodified
reference, and -- when the compiled reference is present (oracle/_ref) -- against the reference itself."""
import os

import numpy as np
import pytest

import cases
import oracle_lib as ol

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def golden_messages(g):
    return [(int(f), str(b), str(t)) for f, b, t in zip(g["msg_freq"], g["msg_bbbb"], g["msg_text"])]


@pytest.mark.parametrize("name", list(cases.CASES))
def test_oracle_matches_golden_exactly(name):
    g = load_golden(name)
    iq = cases.build(name)
    if cases.digest(iq) != str(g["sha256"]):
        pytest.skip("numpy regenerated a different capture than the fixture was made from")
    r = ol.run_oracle(iq)
    assert np.array_equal(r.y1[:4096], g["y1_head"])
    for tag in ol.CHANNELS:
        assert np.array_equal(r.y2[tag][:2048], g["y2_head_" + tag])
        y3 = g["y3_" + tag]                                                  # the first Y3_MAX samples (make_golden.py)
        assert len(r.y3[tag]) == int(g["n"]) // 280
        assert np.array_equal(r.y3[tag][:len(y3)], y3)                        # exact FP64 equality
        assert r.bits[tag] == g["bits_" + tag].tobytes()
        assert np.array_equal(r.bitpos[tag], g["bitpos_" + tag])
        assert np.array_equal(r.disc[tag], g["disc_" + tag])                  # float accumulators, bit-exact
    assert r.messages == golden_messages(g)


@pytest.mark.skipif(not ol.have_ref(), reason="compiled reference (oracle/_ref) not present")
def test_oracle_matches_compiled_reference_long_run():
    """36 s bulletin with end-of-emission: every stage tap, bit, discriminator sum and message equal."""
    from navtex_b200 import synth

    rng = np.random.default_rng(1)
    text, _ = synth.random_message(rng)
    x = synth.fsk_iq([synth.Emission(text, -14000.0, start_s=0.3)], duration_s=36.0, snr_db=-10.0, seed=3)
    iq = synth.quantise_s16(x)
    ref, o = ol.run_ref(iq), ol.run_oracle(iq)
    assert np.array_equal(ref.y1, o.y1)
    for tag in ol.CHANNELS:
        assert np.array_equal(ref.y2[tag], o.y2[tag])
        assert np.array_equal(ref.y3[tag], o.y3[tag])
        assert ref.bits[tag] == o.bits[tag]
        assert np.array_equal(ref.disc[tag], o.disc[tag])
    assert ref.messages == o.messages and len(o.messages) == 1
    assert o.messages[0][0] == 490 and o.messages[0][2] == text
    assert o.events["490"].endswith(b"\x18")          # end of emission -> message_abort


def test_oracle_generalised_nco_reduces_to_reference_table():
    """The restated NCO with f = +-14000 Hz must use the 9-entry table; other offsets get their own period."""
    iq = cases.build("clean518")[: 2 * 252000]
    a = ol.run_oracle(iq)
    b = ol.run_oracle(iq, nco_hz=(14000.0, -14000.0), nco_period=(9, 9))
    for tag in ol.CHANNELS:
        assert np.array_equal(a.y3[tag], b.y3[tag])
    # a channel placed at +10.5 kHz is only found when the NCO is told so
    from navtex_b200 import synth

    em = synth.Emission("ZCZC AB12\nTEST\nNNNN\n", 10500.0, start_s=0.2, n_phasing=16, n_tail=5)
    x = synth.quantise_s16(synth.fsk_iq([em], 8.0, snr_db=10.0, seed=5))
    hit = ol.run_oracle(x, nco_hz=(10500.0, -14000.0), record_taps=False)
    miss = ol.run_oracle(x, record_taps=False)
    assert [m[1] for m in hit.messages] == ["AB12"] and miss.messages == []


def test_oracle_long_taps_linear_phase():
    """Alternative (longer) tap sets: DC gain and delay behave as a decimating FIR should."""
    from scipy import signal

    h1 = signal.firwin(255, 23000, fs=252000, window=("kaiser", 8.0))
    h2 = signal.firwin(255, 2300, fs=63000, window=("kaiser", 8.0))
    h3 = signal.firwin(255, 250, fs=9000, window=("kaiser", 8.0))
    n = 280 * 400
    k = np.arange(n)
    x = 1000.0 * np.exp(2j * np.pi * 14000.0 * k / 252000)            # carrier exactly on the 518 channel
    iq = np.empty(2 * n)
    iq[0::2], iq[1::2] = x.real, x.imag
    r = ol.run_oracle(iq, h1=h1, h2=h2, h3=h3)
    tail = np.abs(r.y3["518"][-50:])
    assert np.allclose(tail, 1000.0, rtol=2e-3)                      # passband gain 1 after the transient
    assert np.all(np.abs(r.y3["490"][-50:]) < 1.0)                  # 28 kHz away: deep in the stop band

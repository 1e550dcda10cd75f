"""The 900 Hz rows of demod_inputs.py, checked on the oracle alone (no GPU): the oracle's 900 Hz entry is the chain with unit
taps and a 0 Hz mix, and every family reaches what it is built for -- exact ties, slewing clocks, decoded bits and messages,
the state machine's aborts -- so that tests/test_gpu_demod.py cannot pass on inputs that quietly became easy."""
import numpy as np
import pytest

import demod_inputs as di

N = 20000
ROWS = range(16 * len(di.FAMILIES))


def _rows():
    return [di.row(7, r, N) for r in ROWS]


@pytest.fixture(scope="module")
def rows(oracle):
    return [(x, m, oracle.run_oracle_900(x)) for x, m in _rows()]


@pytest.mark.parametrize("r", list(range(2 * len(di.FAMILIES))))
def test_900_hz_entry_is_the_unit_tap_chain(oracle, r):
    x, _ = di.row(3, r, 6000)
    a = oracle.run_oracle_900(x)
    iq = np.repeat(x, 280).view(np.float32)                   # every input sample of a 900 Hz sample holds its value
    b = oracle.run_oracle(iq, h1=[1.0], h2=[1.0], h3=[1.0], nco_hz=(0.0,), freq_tag=(518,))
    t = "518"
    assert np.array_equal(a.y3[t].view(np.uint64), x.astype(np.complex128).view(np.uint64))
    assert np.array_equal(b.y3[t].view(np.uint64), a.y3[t].view(np.uint64))
    assert a.bits[t] == b.bits[t] and len(a.bits[t]) > 500
    assert np.array_equal(a.bitpos[t], b.bitpos[t])
    assert np.array_equal(a.disc[t].view(np.uint32), b.disc[t].view(np.uint32))
    assert np.array_equal(a.pick_margins[t], b.pick_margins[t]) and len(a.pick_margins[t]) > 500
    assert a.events[t] == b.events[t]
    assert a.messages == b.messages


def test_lattice_rows_tie_exactly(rows):
    for x, m, o in rows:
        if m["family"] != "lattice":
            continue
        # a_n i^(k_n): both parts of every sample are exact zeros or +-a_n
        assert np.all((x.real == 0) | (x.imag == 0))
        assert not np.signbit(x.real[x.real == 0]).any() and not np.signbit(x.imag[x.imag == 0]).any()
        assert (o.pick_margins["518"][:, 1] == 0).sum() >= 3


def test_noise_rows_have_no_near_ties(rows):
    """what lets the GPU test hold noise rows to bit equality: no arg max pick within 1e-9 of a tie"""
    for x, m, o in rows:
        if m["family"] == "noise":
            assert o.pick_margins["518"][:, 1].min() > 1e-9


def test_fsk_rows_decode_the_intended_bits(rows):
    n9 = 0
    for x, m, o in rows:
        if "bits" not in m or m["spb"] != 9.0:
            continue
        want = di.decoded_span(m, o.bitpos["518"], N)
        assert len(want) > 300 and want in o.bits["518"], (m["family"], m.get("kind"))
        n9 += 1
    assert n9 >= 40


def test_drifting_rows_slew_one_way(rows):
    seen = set()
    for x, m, o in rows:
        if m["family"] == "fsk" and m["spb"] != 9.0:
            gaps = set(np.diff(o.bitpos["518"]).tolist())
            want = 8 if m["spb"] < 9 else 10
            assert want in gaps, (m["spb"], gaps)
            seen.add(want)
    assert seen == {8, 10}


def test_bulletins_and_torture_rows_show_what_they_are_built_for(rows):
    kinds = set()
    for x, m, o in rows:
        ev = o.events["518"]
        if "messages" in m:
            assert [b for _, b, _ in o.messages] == m["messages"], (m.get("kind"), o.messages)
        for e in m.get("events", ()):
            assert e in ev, (m["kind"], e, ev)
        if m["family"] == "bulletin" or m.get("kind") in ("no_nnnn", "extra_b", "shifts", "phasing_breaks"):
            assert di.eoe_aborts(ev) == 1, (m.get("kind"), ev)          # alpha alpha alpha in the DX slot
        if m.get("kind") == "garbage":
            assert di.eoe_aborts(ev) == 0
        kinds.add(m.get("kind"))
    assert kinds >= set(di.TORTURE)

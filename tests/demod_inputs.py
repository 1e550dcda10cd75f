"""Seeded 900 Hz complex rows for tests of the demodulator alone (bit sync, mark/space decision, SITOR-B state machine).

An engine with unit taps ([1], [1], [1]), one channel and a 0 Hz NCO passes its input through unchanged: a float32 sample
repeated over the 280 input samples of one 900 Hz sample comes out of the cascade as that y3 sample, bit for bit.  So these
rows reach the demodulator exactly as written, on the GPU and in the oracle (oracle_lib.run_oracle_900).

Families (row r gets FAMILIES[r % len(FAMILIES)], so neighbouring rows -- the lanes of one warp -- are in different states):
  lattice   a_n i^(k_n), a_n a float32 in [0.5, 2) or exactly 0: every delay-conjugate product lies on an axis, so atan2 returns
            one of its exact special values on every library, and the nine per-offset sums tie exactly wherever the angles do;
  noise     complex Gaussian, scale 1e-3 .. 1e3;
  fsk       phase-continuous +-85 Hz FSK written at 900 Hz ('Y' = -85 Hz as synth.fsk_iq), 9 samples per bit or a clock that
            keeps slewing one way (about 8.5 or 9.5), random bits, with silence before or after;
  bulletin  a NAVTEX bulletin (synth.random_message) as FSK;
  torture   SITOR-B strings that drive the byte state machine to its edges (TORTURE);
  silence   exact zeros, or zeros around a short burst.
Every sample is float32 and no zero is negative (-0 would become +0 in the cascade's mix)."""
from __future__ import annotations

import numpy as np

from navtex_b200 import synth

FS3 = 900
FAMILIES = ("lattice", "noise", "fsk", "bulletin", "torture", "silence")
TORTURE = ("garbage", "abort_then_phasing", "phasing_breaks", "extra_b", "second_phasing", "no_nnnn", "bad_rx", "shifts", "all_codes")
PHASING = "BBBBBBYYYYBBYYBBBBBBYYYYBBYYBB"          # the 30 bits the state machine matches (nav_b_sm.C:296-630)
_VALID = sorted(c for c in range(128) if c in synth._PRINTING) + [synth.SPACE]
_CONTROL = (synth.ALPHA, synth.RQ, synth.LTRS, synth.FIGS, synth.CR, synth.LF, 0x19, 0x5C)   # the other valid codes


def _f32(x) -> np.ndarray:
    """complex -> complex64 with every -0 turned into +0"""
    v = np.ascontiguousarray(np.asarray(x, dtype=np.complex64)).view(np.float32)
    v += np.float32(0.0)
    return v.view(np.complex64)


def lattice(rng, n) -> np.ndarray:
    amp = rng.uniform(0.5, 2.0, n).astype(np.float32)
    amp[rng.random(n) < 0.1] = 0.0
    if rng.random() < 0.5:
        k = rng.integers(0, 4, n)
    else:                                       # runs: constant phase gives zero angles, so zero correlations and nine-way ties
        runs = rng.geometric(1.0 / rng.choice([3, 12, 40]), n)
        k = np.repeat(rng.integers(0, 4, n), runs)[:n]
    for _ in range(rng.integers(0, 4)):         # silent stretches: atan2 of signed zeros, energy ties that decide 'Y'
        a = int(rng.integers(0, n))
        amp[a:a + int(rng.integers(5, 200))] = 0.0
    re = np.choose(k, [amp, 0 * amp, -amp, 0 * amp])
    im = np.choose(k, [0 * amp, amp, 0 * amp, -amp])
    return _f32(re + 1j * im)


def noise(rng, n) -> np.ndarray:
    s = 10.0 ** rng.uniform(-3, 3)
    return _f32(s * (rng.standard_normal(n) + 1j * rng.standard_normal(n)))


def fsk(rng, n, bits, spb=9.0, start=0, amp=None, sigma=None) -> np.ndarray:
    """bits (1 = 'Y') from sample `start` + a random fraction of a bit on, spb samples per bit, with noise of sigma x the
    amplitude while the signal is on (default 10^-3.5 .. 10^-1.5: clean FSK has per-offset sums that tie mathematically and
    differ only by rounding, which any atan2 difference can flip; the silence around it stays exact zeros)"""
    bits = np.asarray(bits, dtype=np.uint8)
    amp = 10.0 ** rng.uniform(-2, 2) if amp is None else amp
    t = np.arange(n) - start - rng.uniform(0, spb)
    k = np.floor(t / spb).astype(np.int64)
    on = (t >= 0) & (k < len(bits))
    f = np.where(bits[np.clip(k, 0, max(len(bits) - 1, 0))] == 1, -synth.FSK_SHIFT_HZ, synth.FSK_SHIFT_HZ) * on
    x = amp * np.exp(1j * (rng.uniform(0, 2 * np.pi) + 2 * np.pi * np.cumsum(f) / FS3)) * on
    sigma = 10.0 ** rng.uniform(-3.5, -1.5) if sigma is None else sigma
    x = x + sigma * amp * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) * on
    return _f32(x)


def _bits(s: str) -> np.ndarray:
    return np.frombuffer(s.encode(), np.uint8) == ord("Y")


def _fec(codes, n_phasing=10, n_tail=0):
    return synth.sitor_b_slots(list(codes), n_phasing, n_tail)


def torture(kind, rng):
    """(bits, what the oracle must show): SITOR-B strings for the state machine's edges"""
    text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=2)
    msg = synth.encode_text(text)
    if kind == "garbage":               # random codes after phasing: more than 12 invalid in 20 -> '*' and an abort
        slots = _fec(synth.encode_text("ZCZC AB01\n")) + list(rng.integers(0, 128, 60))
        return synth.slots_to_bits(slots), {"events": [b"*\x18"]}
    if kind == "abort_then_phasing":    # the byte that aborts ends in the first B of a phasing pattern, which only counts when the
        # state machine takes the byte before the phasing half of the same bit (nav_b_sm.C:266-634); then a bulletin without
        # another full pattern
        bad = [c for c in range(0, 128, 2) if c not in _VALID and c not in _CONTROL]
        aborting = synth.slots_to_bits([synth.RQ, synth.ALPHA] * 10 + [int(c) for c in rng.choice(bad, 13)])
        rest = synth.slots_to_bits([synth.ALPHA] + _fec(msg, n_phasing=0, n_tail=5))     # no RQ: "alpha RQ" would complete one
        return np.concatenate([aborting, _bits(PHASING[1:]), rest]), {"events": [b"*\x18"], "messages": [bbbb]}
    if kind == "phasing_breaks":        # the pattern broken at each of its 30 positions, then a bulletin
        pre = "".join(PHASING[:p] + ("Y" if PHASING[p] == "B" else "B") + "YYY" for p in range(30))
        return np.concatenate([_bits(pre), synth.slots_to_bits(_fec(msg, n_tail=5))]), {"messages": [bbbb]}
    if kind == "extra_b":               # extra B's after the first six: tolerated (nav_b_sm.C:363-372)
        b = synth.slots_to_bits(_fec(msg, n_tail=5))
        at = _bits(PHASING + "B").tobytes()
        k = b.astype(bool).tobytes().find(at) + 6
        return np.concatenate([b[:k], np.zeros(int(rng.integers(1, 5)), np.uint8), b[k:]]), {"messages": [bbbb]}
    if kind == "second_phasing":        # phasing again inside the 1100-bit hold-off: decoded as bytes, not matched
        cut = len(msg) // 2
        slots = _fec(msg[:cut]) + [synth.RQ, synth.ALPHA] * 8 + _fec(msg[cut:], n_phasing=0, n_tail=5)
        return synth.slots_to_bits(slots), {}
    if kind == "no_nnnn":               # the emission ends (alpha alpha alpha in the DX slot) inside the bulletin
        cut = synth.encode_text(text[: text.index("NNNN")])
        return synth.slots_to_bits(_fec(cut, n_tail=5)), {"events": [b"\x18"], "messages": [bbbb]}
    if kind == "bad_rx":                # RX copy invalid with a valid DX copy (DX wins), and both invalid ('*')
        slots = _fec(msg, n_tail=5)
        info = [k for k in range(2 * 10 + 4, len(slots) - 12, 2) if slots[k + 1] in _VALID]
        for k in info[1::3]:
            slots[k + 1] = 0x7F
        k = info[len(info) // 2]
        slots[k + 1] = 0x00
        slots[k - 4] = 0x01                 # its DX copy, two DX slots before
        return synth.slots_to_bits(slots), {"events": [b"*"]}
    if kind == "shifts":                # LTRS / FIGS runs
        codes = synth.encode_text("ZCZC XY12\nPOS 51-23.4N 002-45.6E 1A2B3C\nNNNN\n")
        return synth.slots_to_bits(_fec(codes, n_tail=5)), {"messages": ["XY12"]}
    if kind == "all_codes":             # every 7-bit code in both slots, three valid characters between them
        codes = []
        for c in range(128):
            codes += [c] + [int(x) for x in rng.choice(_VALID, 3)]
        return synth.slots_to_bits(_fec(codes, n_tail=5)), {}
    raise ValueError(kind)


def row(seed, r, n):
    """row r of a seeded set: (complex64 [n], meta).  meta: family, and for FSK rows spb, the intended bits, what must show."""
    rng = np.random.default_rng([seed, r])
    fam = FAMILIES[r % len(FAMILIES)]
    v = r // len(FAMILIES)
    meta = {"family": fam}
    if fam == "lattice":
        return lattice(rng, n), meta
    if fam == "noise":
        return noise(rng, n), meta
    if fam == "silence":
        x = np.zeros(n, np.complex64)
        if v % 2:
            a = int(rng.integers(0, n // 2))
            x[a:a + n // 4] = noise(rng, n // 4)[: n - a]
        return _f32(x), meta
    if fam == "fsk":
        spb = (9.0, 9.0, 8.5, 9.5)[v % 4] if v % 4 < 2 else rng.uniform(8.45, 8.55) if v % 4 == 2 else rng.uniform(9.45, 9.55)
        bits = rng.integers(0, 2, int(n / spb)).astype(np.uint8)
        start = int(rng.integers(0, n // 4)) if v % 3 == 1 else 0
        if v % 3 == 2:                      # the transmitter stops early
            bits = bits[: int(len(bits) * rng.uniform(0.4, 0.8))]
        sigma = 0.02 if v % 5 == 4 else None
        meta.update(spb=spb, bits=bits, start=start)
        return fsk(rng, n, bits, spb, start, sigma=sigma), meta
    if fam == "bulletin":
        text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=3)
        bits = synth.message_bits(text, n_phasing=10, n_tail=5)
        start = int(rng.integers(0, max(1, n - 9 * len(bits) - 20)))
        meta.update(spb=9.0, bits=bits, start=start, messages=[bbbb])
        return fsk(rng, n, bits, 9.0, start), meta
    kind = TORTURE[v % len(TORTURE)]
    bits, want = torture(kind, rng)
    start = int(rng.integers(0, max(1, n - 9 * len(bits) - 20)))
    meta.update(kind=kind, spb=9.0, bits=bits, start=start, **want)
    return fsk(rng, n, bits, 9.0, start), meta


def decoded_span(meta, bitpos, n):
    """the intended bits an oracle must have decoded, as 'B'/'Y' bytes: those of a 9-samples-per-bit row from 600 samples after
    the later of its start and its first decision (the bit sync needs a full ring of the signal) to two bits before its end"""
    want = bytes(np.where(meta["bits"] == 1, ord("Y"), ord("B")).astype(np.uint8))
    spb, st = meta["spb"], meta["start"]
    k0 = int((max(bitpos[0] if len(bitpos) else n, st + 600) - st) / spb) + 2
    k1 = min(len(want), int((n - st) / spb)) - 2
    return want[k0:k1]


def eoe_aborts(events: bytes) -> int:
    """aborts not caused by the error window ('*' then 0x18): end of emission"""
    return sum(1 for k, e in enumerate(events) if e == 0x18 and (k == 0 or events[k - 1] != ord("*")))

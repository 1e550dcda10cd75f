"""Synthetic NAVTEX (SITOR-B / CCIR 476) emissions in place of the SDRplay device.

The reference has no signal generator; captures come from the radio
(capt_sched.c:105-148).  This module builds what the radio would have
delivered: 252 kS/s zero-IF IQ with the tuner at 504 kHz (capt_sched.c:42), so
518 kHz sits at +14 kHz and 490 kHz at -14 kHz, carrying 100 baud +-85 Hz
continuous-phase FSK ('B' = +85 Hz, 'Y' = -85 Hz; decoder.C:115-131) of a
SITOR-B collective-FEC character stream (DX copy, RX copy five slots later;
nav_b_sm.C:150-232).  See SURVEY.md Appendix B for the recipe.

Host-side tooling only (tests, bench input); numpy, no GPU.
"""
from __future__ import annotations

import struct
import wave
from dataclasses import dataclass

import numpy as np

FS = 252_000            # capt_sched.c:29-34 (2.016 MS/s / 8)
BAUD = 100
SAMPLES_PER_BIT = FS // BAUD
FSK_SHIFT_HZ = 85.0     # decoder.h:13
ALPHA, RQ = 0x07, 0x4C  # phasing signals 1 / 2 (nav_b_sm.h:89-90)
LTRS, FIGS, CR, LF, SPACE = 0x52, 0x49, 0x70, 0x64, 0x62

# CCIR 476 code points (7 bits, MSB first, Y = 1) -> (letters case, figures case).
_PRINTING = {
    0x0B: ("J", None), 0x0D: ("W", "2"), 0x0E: ("A", "-"), 0x13: ("F", None), 0x15: ("Y", "6"),
    0x16: ("S", "'"), 0x1A: ("D", "%"), 0x1C: ("Z", "+"), 0x23: ("C", ":"), 0x25: ("P", "0"),
    0x26: ("I", "8"), 0x29: ("G", None), 0x2A: ("R", "4"), 0x2C: ("L", ")"), 0x31: ("M", "."),
    0x32: ("N", ","), 0x34: ("H", None), 0x38: ("O", "9"), 0x43: ("K", "("), 0x45: ("Q", "1"),
    0x46: ("U", "7"), 0x4A: ("E", "3"), 0x51: ("X", "/"), 0x58: ("B", "?"), 0x61: ("V", "="),
    0x68: ("T", "5"),
}
_LETTER_CODE = {l: c for c, (l, _) in _PRINTING.items()}
_FIGURE_CODE = {f: c for c, (_, f) in _PRINTING.items() if f is not None}


def encode_text(text: str) -> list[int]:
    """Text -> CCIR 476 codes with LTRS/FIGS shifts; '\\n' becomes CR LF."""
    codes: list[int] = []
    figures = False
    for ch in text.upper():
        if ch == "\n":
            codes += [CR, LF]
        elif ch == " ":
            codes.append(SPACE)
        elif ch in _LETTER_CODE:
            if figures:
                codes.append(LTRS)
                figures = False
            codes.append(_LETTER_CODE[ch])
        elif ch in _FIGURE_CODE:
            if not figures:
                codes.append(FIGS)
                figures = True
            codes.append(_FIGURE_CODE[ch])
        else:
            raise ValueError(f"no CCIR 476 code for {ch!r}")
    return codes


def sitor_b_slots(codes: list[int], n_phasing: int = 70, n_tail: int = 6) -> list[int]:
    """Interleave DX and RX copies: slot 2k = DX[k], slot 2k+1 = DX[k-2] (alpha while phasing)."""
    dx = [RQ] * n_phasing + list(codes) + [ALPHA] * n_tail
    info_lo, info_hi = n_phasing, n_phasing + len(codes)
    slots: list[int] = []
    for k, c in enumerate(dx):
        slots.append(c)
        j = k - 2
        slots.append(dx[j] if info_lo <= j < info_hi else ALPHA)
    return slots


def slots_to_bits(slots: list[int]) -> np.ndarray:
    """7 bits per slot, MSB first; 1 = 'Y' (nav_b_sm.C:271-276)."""
    arr = np.asarray(slots, dtype=np.uint8)
    return ((arr[:, None] >> np.arange(6, -1, -1)) & 1).astype(np.uint8).reshape(-1)


def message_bits(text: str, n_phasing: int = 70, n_tail: int = 6) -> np.ndarray:
    return slots_to_bits(sitor_b_slots(encode_text(text), n_phasing, n_tail))


@dataclass
class Emission:
    text: str
    offset_hz: float = 14_000.0      # +14 kHz = 518 kHz channel, -14 kHz = 490 kHz
    start_s: float = 0.5
    amplitude: float = 8000.0
    n_phasing: int = 70
    n_tail: int = 6
    stop_s: float | None = None   # transmitter drops out this many seconds after start_s


def fsk_iq(
    emissions: list[Emission],
    duration_s: float,
    snr_db: float | None = None,
    seed: int = 0,
    fading_hz: float = 0.0,
    idle_carrier: bool = False,
    rate: int = FS,
) -> np.ndarray:
    """Complex baseband capture (complex128, not yet quantised) of the given emissions, sampled at `rate` S/s (a multiple of
    100, so that a bit is a whole number of samples; the engine's own 252 kS/s by default, others for engines that resample).

    snr_db is the signal-to-noise ratio over the full sampled band relative to the
    first emission's amplitude (SURVEY.md 8d: the reference decodes at -20 dB).
    fading_hz > 0 applies a slow Rayleigh-like amplitude (two-pole filtered complex
    Gaussian, unit mean power) to every emission.
    """
    n = int(round(duration_s * rate))
    spb = rate // BAUD
    rng = np.random.default_rng(seed)
    x = np.zeros(n, dtype=np.complex128)
    for em in emissions:
        bits = message_bits(em.text, em.n_phasing, em.n_tail)
        start = int(round(em.start_s * rate))
        span = min(len(bits) * spb, max(0, n - start))
        if em.stop_s is not None:
            span = min(span, int(round(em.stop_s * rate)))
        if span <= 0:
            continue
        tone = np.where(bits == 1, -FSK_SHIFT_HZ, FSK_SHIFT_HZ)       # Y = -85 Hz, B = +85 Hz
        freq = np.repeat(tone, spb)[:span] + em.offset_hz
        phase = 2.0 * np.pi * np.cumsum(freq) / rate
        sig = em.amplitude * np.exp(1j * phase)
        if fading_hz > 0.0:
            g = rng.standard_normal(span) + 1j * rng.standard_normal(span)
            a = np.exp(-2.0 * np.pi * fading_hz / rate)
            env = np.empty(span, dtype=np.complex128)
            acc = 0.0 + 0.0j
            # one-pole IIR in blocks (vectorised via cumulative scaling is unstable for long spans)
            blk = 4096
            for s in range(0, span, blk):
                e = min(span, s + blk)
                w = a ** np.arange(1, e - s + 1)
                c = np.cumsum(g[s:e] / w) * w * (1 - a) + acc * w
                env[s:e] = c
                acc = c[-1]
            env /= np.sqrt(np.mean(np.abs(env) ** 2)) + 1e-30
            sig = sig * env
        x[start:start + span] += sig
        if idle_carrier and start > 0:
            x[:start] += em.amplitude * np.exp(2j * np.pi * (em.offset_hz + FSK_SHIFT_HZ) * np.arange(start) / rate)
    if snr_db is not None and emissions:
        sigma = emissions[0].amplitude / np.sqrt(2.0) * 10.0 ** (-snr_db / 20.0)
        x += sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x


def quantise_s16(x: np.ndarray) -> np.ndarray:
    """Complex capture -> interleaved int16 I,Q exactly as the SDRplay callback stores it (capt_sched.c:120-128)."""
    iq = np.empty(2 * len(x), dtype=np.int16)
    iq[0::2] = np.clip(np.rint(x.real), -32768, 32767).astype(np.int16)
    iq[1::2] = np.clip(np.rint(x.imag), -32768, 32767).astype(np.int16)
    return iq


def quantise_u8(x: np.ndarray) -> np.ndarray:
    """Complex capture -> interleaved unsigned 8-bit offset-binary I,Q (the RTL-SDR's format): rint, + 128, clipped to
    [0, 255].  The engine reads a byte u as u - 128."""
    iq = np.empty(2 * len(x), dtype=np.uint8)
    iq[0::2] = np.clip(np.rint(x.real) + 128, 0, 255).astype(np.uint8)
    iq[1::2] = np.clip(np.rint(x.imag) + 128, 0, 255).astype(np.uint8)
    return iq


def write_wav(path: str, iq_s16: np.ndarray) -> None:
    """Stereo s16 252 kHz WAV, I = left, Q = right: the format PrepWav would write (capt_sched.c:87-96)."""
    with wave.open(path, "wb") as w:
        w.setnchannels(2)
        w.setsampwidth(2)
        w.setframerate(FS)
        w.writeframes(np.ascontiguousarray(iq_s16, dtype="<i2").tobytes())


def read_wav(path: str) -> np.ndarray:
    with wave.open(path, "rb") as w:
        assert w.getnchannels() == 2 and w.getsampwidth() == 2
        return np.frombuffer(w.readframes(w.getnframes()), dtype="<i2").copy()


STATIONS = "ABCDEFGHIJKLMNOPQRSTUVWX"
SUBJECTS = "ABDEFGHIJKLTVWXYZ"
_WORDS = (
    "GALE WARNING NORTH SEA SOUTHWEST VEERING WEST FORCE 8 TO 9 EXPECTED SOON VISIBILITY MODERATE OR POOR "
    "NAVAREA ONE LIGHT BUOY UNLIT IN POSITION 51-23.4N 002-45.6E WIDE BERTH REQUESTED CANCEL THIS MSG "
    "DRIFTING CONTAINER REPORTED VESSELS KEEP SHARP LOOKOUT ICE REPORT NIL SAR EXERCISE AREA CLOSED"
).split()


def random_message(rng: np.random.Generator, n_lines: int = 3, words_per_line: int = 6) -> tuple[str, str]:
    """A plausible NAVTEX bulletin; returns (full text incl. ZCZC/NNNN framing, B1B2B3B4)."""
    bbbb = STATIONS[rng.integers(len(STATIONS))] + SUBJECTS[rng.integers(len(SUBJECTS))] + "%02d" % rng.integers(1, 100)
    lines = [" ".join(_WORDS[i] for i in rng.integers(len(_WORDS), size=words_per_line)) for _ in range(n_lines)]
    text = "ZCZC " + bbbb + "\n" + "\n".join(lines) + "\nNNNN\n"
    return text, bbbb


def pack_messages(records) -> bytes:
    """(stream, freq, bbbb, text) records -> a deterministic byte string, for multiset comparison across runs."""
    out = bytearray()
    for stream, freq, bbbb, text in sorted(records):
        t = text.encode("latin-1")
        out += struct.pack("<iiI", stream, freq, len(t)) + bbbb.encode("latin-1").ljust(8, b"\0") + t
    return bytes(out)

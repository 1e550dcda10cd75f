"""Comparison of one stream's GPU taps with the CPU reference / oracle taps: the numbers behind "1e-5 relative".

Test infrastructure (shared by tests/ and bench.py's same-run parity check); pure numpy, no GPU, no oracle import.

What north_star demands: decoded characters / headers / messages bit-exact; filtered samples and discriminator sums within a
stated FP32 relative tolerance (1e-5).  "Relative" needs a denominator, and this module reports all the sensible ones instead of
picking the most flattering:

  y3_rel_pair_peak   max |gpu - ref| over both channels / the larger channel peak of the stream (the FIR kernels are linear
                     maps of the SAME input, so their absolute rounding error scales with the input, i.e. with the strong
                     channel, whichever channel it lands in) -- the bar of every GPU test: <= 1e-5;
  y3_rel_own_rms     per OCCUPIED channel: max |gpu - ref| / that channel's own RMS -- the same bar, <= 1e-5 x a crest allowance
                     is not needed: measured ~1e-6;
  empty channel      (60+ dB below the occupied one: what is demodulated there is leakage comparable to FP32 rounding) the
                     error relative to its own RMS is reported, not bounded; its raw bit decisions are compared position by
                     position and every differing decision is reported with the reference's decision margin
                     |E_B - E_Y| / max(E_B, E_Y) (SURVEY.md 7.3-2: mismatches are confined to near-ties).  No character can come
                     out of such a channel without a 30-bit phasing match, and events / messages are exact on BOTH channels.
"""
from __future__ import annotations

import numpy as np

CHANNELS = ("518", "490")
REL_TOL = 1e-5


def decision_margin(disc_row) -> float:
    """|E_B - E_Y| / max(E_B, E_Y) of one mark/space decision from its four accumulators BR BI YR YI (decoder.C:121-125)."""
    br, bi, yr, yi = (float(v) for v in disc_row)
    eb, ey = br * br + bi * bi, yr * yr + yi * yi
    m = max(eb, ey)
    return abs(eb - ey) / m if m > 0 else 0.0


def compare_stream(y3_gpu, bits_gpu, disc_gpu, ref, occupied, channels=CHANNELS):
    """y3_gpu: [C, P] complex; bits_gpu / disc_gpu: per channel index bytes / (n, 4) float32 (disc may be None);
    ref: object with dicts y3 / bits / disc keyed by the tags of `channels`; occupied: tags that carry a signal;
    channels: the keys of channel indices 0 .. C-1 (oracle_lib.CHANNEL_KEYS[:C]; the pair peak is over all of them).
    Returns a dict of the figures described in the module docstring."""
    peak = max(np.abs(ref.y3[t]).max() if len(ref.y3[t]) else 0.0 for t in channels)
    peak = max(peak, 1e-30)
    out = {"y3_rel_pair_peak": 0.0, "y3_rel_own_rms": {}, "bit_mismatches": {}, "bit_len_diff": {}, "mismatch_margins": {},
           "disc_rel": {}, "empty_rel_own_rms": {}}
    for c, tag in enumerate(channels):
        r = ref.y3[tag]
        g = np.asarray(y3_gpu[c]).astype(np.complex128)
        assert g.shape == r.shape, (tag, g.shape, r.shape)
        err = np.abs(g - r).max() if len(r) else 0.0
        out["y3_rel_pair_peak"] = max(out["y3_rel_pair_peak"], err / peak)
        rms = float(np.sqrt(np.mean(np.abs(r) ** 2))) if len(r) else 0.0
        (out["y3_rel_own_rms"] if tag in occupied else out["empty_rel_own_rms"])[tag] = err / rms if rms > 0 else 0.0
        gb, rb = bits_gpu[c], ref.bits[tag]
        out["bit_len_diff"][tag] = len(gb) - len(rb)
        out.setdefault("bits_compared", {})[tag] = min(len(gb), len(rb))
        if len(gb) == len(rb):
            ga, ra = np.frombuffer(gb, dtype=np.uint8), np.frombuffer(rb, dtype=np.uint8)
            bad = np.nonzero(ga != ra)[0]
            out["bit_mismatches"][tag] = int(bad.size)
            out["mismatch_margins"][tag] = [decision_margin(ref.disc[tag][k]) for k in bad[:64]]
            # a RUN of differing decisions with healthy mark/space margins is a timing slip: one of the nine-way arg max
            # picks fell the other way at a near-tie and the slew-limited offset took a different path for a while.  With the
            # restated oracle's per-evaluation margins, report the tightest arg max in the 64 evaluations before the run.
            pm, bp = getattr(ref, "pick_margins", {}).get(tag), getattr(ref, "bitpos", {}).get(tag)
            if bad.size and pm is not None and len(pm) and bp is not None and len(bp) == len(rb):
                runs, start = [], int(bad[0])
                for a, b in zip(bad[:-1], bad[1:]):
                    if b - a > 16:
                        runs.append(start); start = int(b)
                runs.append(start)
                tight = []
                for k in runs:
                    at = np.searchsorted(pm[:, 0], bp[k])
                    tight.append(float(pm[max(0, at - 64):at + 1, 1].min()))
                out.setdefault("timing_slip_pick_margins", {})[tag] = tight
        else:
            out["bit_mismatches"][tag] = None
            out["mismatch_margins"][tag] = []
            # a different NUMBER of decisions is a timing slip that did not re-converge: attribute it like the runs above, from
            # the first decision where the two diverge (its bit, or its discriminator sums beyond 1e-3 of their peak)
            pm, bp = getattr(ref, "pick_margins", {}).get(tag), getattr(ref, "bitpos", {}).get(tag)
            m = min(len(gb), len(rb))
            if m and pm is not None and len(pm) and bp is not None and len(bp) == len(rb):
                diff = np.frombuffer(gb, dtype=np.uint8)[:m] != np.frombuffer(rb, dtype=np.uint8)[:m]
                if disc_gpu is not None and disc_gpu[c] is not None and len(disc_gpu[c]) == len(gb):
                    rs = np.asarray(ref.disc[tag][:m], dtype=np.float64)
                    dd = np.abs(np.asarray(disc_gpu[c][:m], dtype=np.float64) - rs).max(axis=1)
                    diff |= dd > 1e-3 * max(np.abs(rs).max(), 1e-30)
                k = int(np.argmax(diff)) if diff.any() else m - 1
                at = np.searchsorted(pm[:, 0], bp[k])
                out.setdefault("length_slip", {})[tag] = {"first_diverging_decision": k, "of": len(rb),
                                                          "pick_margin": float(pm[max(0, at - 64):at + 1, 1].min())}
        if disc_gpu is not None and disc_gpu[c] is not None and tag in occupied and len(rb) == len(gb) and len(rb):
            rs = np.asarray(ref.disc[tag], dtype=np.float64)
            out["disc_rel"][tag] = float(np.abs(np.asarray(disc_gpu[c], dtype=np.float64) - rs).max() / max(np.abs(rs).max(), 1e-30))
    return out


def assert_stream(cmp, occupied, where="", unbounded=(), near_tie=0.0):
    """The bar: pair-peak and own-RMS errors of occupied channels <= 1e-5, their bit decisions identical, discriminator sums
    within 5e-5 (five accumulated samples); empty channels: same number of decisions.  The channels are those compare_stream
    was given.  `unbounded`: empty channels tuned into the stage-1 stopband (>= 60 dB down), which hold nothing but residue at
    the level of FP32 rounding -- their samples are held to the pair-peak bar, their number of decisions is reported only.
    `near_tie` > 0: an empty channel may also end with a different number of decisions when the first decision where the two
    diverge follows an oracle arg max pick within that relative margin (a timing slip on noise that did not re-converge)."""
    assert cmp["y3_rel_pair_peak"] <= REL_TOL, (where, cmp["y3_rel_pair_peak"])
    for tag in occupied:
        assert cmp["y3_rel_own_rms"][tag] <= REL_TOL, (where, tag, cmp["y3_rel_own_rms"][tag])
        assert cmp["bit_mismatches"][tag] == 0, (where, tag, cmp["bit_mismatches"][tag], cmp["bit_len_diff"][tag])
        if tag in cmp["disc_rel"]:
            assert cmp["disc_rel"][tag] <= 5 * REL_TOL, (where, tag, cmp["disc_rel"][tag])
    for tag in cmp["bit_len_diff"]:
        if tag not in occupied and tag not in unbounded:
            slip = cmp.get("length_slip", {}).get(tag)
            if near_tie > 0 and slip is not None and slip["pick_margin"] <= near_tie:
                continue
            assert cmp["bit_len_diff"][tag] == 0, (where, tag, cmp["bit_len_diff"][tag], cmp.get("length_slip", {}).get(tag),
                                                   cmp["empty_rel_own_rms"].get(tag))


def summarise(cmps, occupied_of):
    """Aggregate a list of compare_stream() results (occupied_of[k] = occupied tags of stream k) into the bench's check record."""
    own = [v for c, occ in zip(cmps, occupied_of) for t, v in c["y3_rel_own_rms"].items() if t in occ]
    empty_mis = [c["bit_mismatches"][t] for c, occ in zip(cmps, occupied_of) for t in c["bit_len_diff"] if t not in occ]
    margins = [m for c, occ in zip(cmps, occupied_of) for t in c["bit_len_diff"] if t not in occ for m in c["mismatch_margins"][t]]
    disc = [v for c in cmps for v in c["disc_rel"].values()]
    return {
        "streams": len(cmps),
        "y3_max_rel_pair_peak": max(c["y3_rel_pair_peak"] for c in cmps),
        "y3_max_rel_own_rms_occupied": max(own) if own else None,
        "disc_max_rel_occupied": max(disc) if disc else None,
        "bit_mismatches_occupied": sum((c["bit_mismatches"][t] if c["bit_mismatches"][t] is not None else 10 ** 6)
                                       for c, occ in zip(cmps, occupied_of) for t in occ),
        "empty_channels": len(empty_mis),
        "empty_channel_bit_len_diffs": sum(1 for c, occ in zip(cmps, occupied_of) for t in c["bit_len_diff"] if t not in occ and c["bit_len_diff"][t] != 0),
        "empty_channel_bit_mismatches": sum(m for m in empty_mis if m is not None),
        "empty_channel_bits_compared": sum(c["bits_compared"][t] for c, occ in zip(cmps, occupied_of) for t in c["bit_len_diff"]
                                           if t not in occ and c["bit_mismatches"][t] is not None),
        "empty_channel_mismatch_margin_max": max(margins) if margins else None,
    }


REPORT = []      # (where, figures) of every stream compared during a test session; conftest.py writes it out at the end


def record(where, cmp, occupied):
    empty = [t for t in cmp["bit_len_diff"] if t not in occupied]
    REPORT.append({"where": where, "occupied": sorted(occupied), "y3_rel_pair_peak": cmp["y3_rel_pair_peak"],
                   "y3_rel_own_rms": cmp["y3_rel_own_rms"], "disc_rel": cmp["disc_rel"],
                   "empty_channels": {t: {"y3_rel_own_rms": cmp["empty_rel_own_rms"].get(t), "bit_len_diff": cmp["bit_len_diff"][t],
                                          "bit_mismatches": cmp["bit_mismatches"][t],
                                          "mismatch_margins": cmp["mismatch_margins"][t],
                                          "timing_slip_pick_margins": cmp.get("timing_slip_pick_margins", {}).get(t),
                                          "length_slip": cmp.get("length_slip", {}).get(t)} for t in empty}})

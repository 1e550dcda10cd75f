"""Per-stream lifecycle: one radio reconnects (nvx_engine_reset_streams), is retuned (nvx_engine_retune_stream) or drops out of
the capture front end (nvx_capture_detach / attach) while the other streams keep decoding.

The contract (navtex_b200.h): a reset that takes effect at input sample E restarts the stream at E0 = E - (E mod 158760), and
from then on the stream is bit for bit what a freshly created engine produces when fed Z = E - E0 zero samples followed by the
stream's input from E on.  Every check here compares against exactly that: a fresh one-stream engine fed Z zeros (one block)
and then the same blocks.  The other streams are compared with an engine that never reset.  Blocks are uneven multiples of
280, so that resets land on and off a 158 760-sample boundary.

Captures are at 8-bit scale (30 LSB, -3 dB full-band SNR), so the same values push as 8-bit pairs, int16 and float32."""
import functools

import numpy as np
import pytest

from navtex_b200 import engine, synth
from test_gpu_longtaps import designs

pytestmark = pytest.mark.gpu

FS = engine.FS
BLK = engine.BLOCK_ALIGN
RING = 158760                      # 567 x 280: the grid a reset restarts on
AMP = 30.0
MAX_BLOCK = 1800 * BLK
SECONDS = 25.0                     # a bulletin of random_message(1 line, 3 words) with 18 phasing slots lasts up to 10.7 s
N = int(SECONDS * FS)


def _bulletin(rng, offset, start):
    text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=3)
    return synth.Emission(text, offset, start_s=start, amplitude=AMP, n_phasing=18, n_tail=5), bbbb


def _capture_u8(emissions, seconds, seed):
    return synth.quantise_u8(synth.fsk_iq(emissions, seconds, snr_db=-3.0, seed=seed)).reshape(-1, 2)


def _as_fmt(u8, fmt):
    if fmt == "u8":
        return u8
    v = u8.astype(np.int16) - 128
    return v if fmt == "s16" else v.astype(np.float32)


def _silence(fmt, n):
    return np.full((n, 2), 128, np.uint8) if fmt == "u8" else np.zeros((n, 2), np.int16 if fmt == "s16" else np.float32)


def _plan(rng, total, cut):
    """uneven block lengths (multiples of 280) covering [0, total) with a block boundary at `cut`"""
    out = []
    for a, b in ((0, cut), (cut, total)):
        left = (b - a) // BLK
        while left:
            k = min(left, int(rng.integers(300, 1800)))
            out.append(k * BLK)
            left -= k
    return out


def _snapshot(eng, keep_bits):
    rec = {"y3": eng.read_y3().copy(), "ev": {}, "bits": {}}
    for s in range(eng.S):
        for c in range(eng.C):
            rec["ev"][s, c] = eng.read_events(s, c)
            if keep_bits:
                rec["bits"][s, c] = eng.read_bits(s, c)
    return rec


def _run(eng, x, blocks, keep_bits=True, at=None, action=None):
    """push x [S, n, 2] in `blocks`, calling action(eng) before block index `at`.  Returns the per-block records and the
    messages polled before the action and at the end."""
    recs, before, pos = [], [], 0
    for i, n in enumerate(blocks):
        if i == at:
            before = eng.poll_messages()
            action(eng)
        eng.push_host(np.ascontiguousarray(x[:, pos:pos + n]))
        pos += n
        recs.append(_snapshot(eng, keep_bits))
    return recs, before, eng.poll_messages()


def _fresh(make, x_row, blocks, at, E, fmt):
    """a fresh one-stream engine fed Z = E - E0 zeros (one block), then x_row's blocks from `at` on; the records of those blocks"""
    Z = E % RING
    xs = x_row[E:]
    eng = make()
    pre = [Z] if Z else []
    x = np.concatenate([_silence(fmt, Z), xs])[None] if Z else xs[None]
    recs, _, msgs = _run(eng, x, pre + blocks[at:], keep_bits=eng._keep_bits)
    eng.close()
    return recs[len(pre):], msgs


def _same(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _assert_equal_rows(got, s, want, s_want, C, bits=True, where=""):
    for k, (g, w) in enumerate(zip(got, want)):
        assert _same(g["y3"][s], w["y3"][s_want]), (where, "y3", k)
        for c in range(C):
            assert g["ev"][s, c] == w["ev"][s_want, c], (where, "events", k, c)
            if bits:
                gb, wb = g["bits"][s, c], w["bits"][s_want, c]
                assert gb[0] == wb[0] and _same(gb[1], wb[1]), (where, "bits", k, c)


class _Keep(engine.Engine):
    def __init__(self, *a, keep_bits=False, **kw):
        super().__init__(*a, keep_bits=keep_bits, **kw)
        self._keep_bits = keep_bits


@functools.lru_cache(maxsize=None)
def _scenario(seed, S, offsets, reset_stream=1):
    """S streams of SECONDS; the reset stream carries bulletin A (0.5 s, interrupted by the reset) and bulletin B (12 s), every
    other stream two bulletins, the first across the reset.  offsets[s] = the offset each stream's bulletins sit at."""
    rng = np.random.default_rng(seed)
    rows, want = [], {}
    for s in range(S):
        starts = (0.5, 12.0) if s == reset_stream else (0.3 + 0.3 * s, 12.5)
        (a, bbbb_a), (b, bbbb_b) = (_bulletin(rng, offsets[s], t) for t in starts)
        want[s] = (bbbb_a, bbbb_b)
        rows.append(_capture_u8([a, b], SECONDS, seed * 10 + s))
    return np.stack(rows), want


def _reset_points():
    return {"on_ring": 6 * RING, "off_ring": 6 * RING + 211 * BLK}


# ---- 1. fused path, reference NCO table ----------------------------------------------------------------------------------
@pytest.mark.parametrize("where", ["on_ring", "off_ring"])
@pytest.mark.parametrize("fmt", ["s16", "f32", "u8"])
def test_reset_one_stream_fused_reference_table(fmt, where):
    S = 4
    E = _reset_points()[where]
    u8, want = _scenario(11, S, (14000.0, 14000.0, -14000.0, 14000.0))
    x = np.stack([_as_fmt(r, fmt) for r in u8])
    blocks = _plan(np.random.default_rng(5), N, E)
    at = int(np.searchsorted(np.cumsum(blocks), E)) + 1
    assert sum(blocks[:at]) == E

    eng = _Keep(S, MAX_BLOCK, keep_bits=True)
    got, before, after = _run(eng, x, blocks, at=at, action=lambda e: e.reset_streams([1]))
    eng.close()
    ref = _Keep(S, MAX_BLOCK, keep_bits=True)
    base, _, base_msgs = _run(ref, x, blocks)
    ref.close()

    # streams 0, 2, 3: bit-identical to the engine that never reset, messages included
    for s in (0, 2, 3):
        _assert_equal_rows(got, s, base, s, 2, where=(fmt, where, s))
    assert sorted(m for m in before + after if m[0] != 1) == sorted(m for m in base_msgs if m[0] != 1)
    assert {m[2] for m in base_msgs if m[0] == 0} == set(want[0])

    # stream 1 from E on: a fresh engine fed Z zeros, then its input
    fresh, fresh_msgs = _fresh(lambda: _Keep(1, MAX_BLOCK, keep_bits=True, first_stream_id=1), x[1], blocks, at, E, fmt)
    _assert_equal_rows(got[at:], 1, fresh, 0, 2, where=(fmt, where, "fresh"))
    mine = [m for m in after if m[0] == 1]
    assert mine == fresh_msgs
    assert not [m for m in before if m[0] == 1]
    bbbb_a, bbbb_b = want[1]
    assert [m[2] for m in mine] == [bbbb_b], mine             # the interrupted bulletin is never delivered
    assert bbbb_a in {m[2] for m in base_msgs if m[0] == 1}    # (without the reset it would have been)


# ---- 2. general NCO, retune ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [3, 8])
def test_retune_one_stream_general_nco(C):
    S = 2
    old = np.array([-24000.0 + 47000 // (C - 1) * k + 0.5 * (k % 2) for k in range(C)])
    new = old + 2500.5
    old_tags, new_tags = np.arange(100, 100 + C), np.arange(200, 200 + C)
    nco = np.stack([old, old[::-1]])
    tags = np.stack([old_tags, old_tags + 50])
    E = 18 * RING + 97 * BLK                                   # 11.45 s
    rng = np.random.default_rng(23)
    b1, bbbb1 = _bulletin(rng, old[1], 0.3)                    # ends before the retune: old offset, old tag
    b2, bbbb2 = _bulletin(rng, new[C - 2], 12.0)               # after it: new offset, new tag
    b3, bbbb3 = _bulletin(rng, old[-1], 2.0)                   # stream 1, channel 0 (its offsets are reversed)
    x = np.stack([_capture_u8([b1, b2], SECONDS, 71), _capture_u8([b3], SECONDS, 72)])
    blocks = _plan(np.random.default_rng(6), N, E)
    at = int(np.searchsorted(np.cumsum(blocks), E)) + 1

    mk = lambda nc, tg, first=0, n=S: _Keep(n, MAX_BLOCK, keep_bits=True, nco_hz=nc, stream_freq_tag=tg, n_channels=C, first_stream_id=first)
    eng = mk(nco, tags)
    got, before, after = _run(eng, x, blocks, at=at, action=lambda e: e.retune_stream(0, new, new_tags))
    eng.close()
    ref = mk(nco, tags)
    base, _, base_msgs = _run(ref, x, blocks)
    ref.close()

    _assert_equal_rows(got, 1, base, 1, C, where=(C, "untouched"))
    assert [m for m in before + after if m[0] == 1] == [m for m in base_msgs if m[0] == 1]
    assert [(m[1], m[2]) for m in base_msgs if m[0] == 1] == [(int(tags[1][0]), bbbb3)]

    fresh, fresh_msgs = _fresh(lambda: mk(new[None], new_tags[None], 0, 1), x[0], blocks, at, E, "u8")
    _assert_equal_rows(got[at:], 0, fresh, 0, C, where=(C, "fresh"))
    assert [(m[1], m[2]) for m in before if m[0] == 0] == [(int(old_tags[1]), bbbb1)]      # completed before: old tag
    assert [m for m in after if m[0] == 0] == fresh_msgs
    assert [(m[1], m[2]) for m in fresh_msgs] == [(int(new_tags[C - 2]), bbbb2)]             # after: new tag


# ---- 3. long-tap path ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nco", [False, True], ids=["table", "nco"])
@pytest.mark.parametrize("tc", ["0", None], ids=["cuda_core", "tensor_core"])
def test_reset_one_stream_long_taps(monkeypatch, tc, nco):
    if tc is None:
        monkeypatch.delenv("NVX_LONG_TC", raising=False)
    else:
        monkeypatch.setenv("NVX_LONG_TC", tc)
    taps = designs()
    S = 3
    offs = [14000.5, -13999.5, 14000.5] if nco else [14000.0, -14000.0, 14000.0]
    nco_hz = np.array([[14000.5, -13999.5]] * S) if nco else None
    E = 6 * RING + 433 * BLK
    u8, want = _scenario(31, S, tuple(offs))
    x = np.stack([_as_fmt(r, "s16") for r in u8])
    blocks = _plan(np.random.default_rng(7), N, E)
    at = int(np.searchsorted(np.cumsum(blocks), E)) + 1
    exact = tc == "0"

    mk = lambda n=S, first=0: _Keep(n, MAX_BLOCK, keep_bits=exact, taps=taps, first_stream_id=first,
                                   nco_hz=None if nco_hz is None else nco_hz[:n])
    eng = mk()
    got, before, after = _run(eng, x, blocks, keep_bits=exact, at=at, action=lambda e: e.reset_streams([1]))
    eng.close()
    ref = mk()
    base, _, base_msgs = _run(ref, x, blocks, keep_bits=exact)
    ref.close()
    for s in (0, 2):        # same blocking: bit-identical on either kind of stage
        _assert_equal_rows(got, s, base, s, 2, bits=exact, where=(tc, nco, s))
    assert sorted(m for m in before + after if m[0] != 1) == sorted(m for m in base_msgs if m[0] != 1)

    fresh, fresh_msgs = _fresh(lambda: mk(1, 1), x[1], blocks, at, E, "s16")
    if exact:
        _assert_equal_rows(got[at:], 1, fresh, 0, 2, where=(tc, nco, "fresh"))
    else:                   # a different blocking on the tensor cores: equal to rounding (navtex_b200.h, n1 / n2 / n3)
        g = np.concatenate([r["y3"][1] for r in got[at:]], axis=-1)
        f = np.concatenate([r["y3"][0] for r in fresh], axis=-1)
        assert np.abs(g - f).max() <= 1e-5 * np.abs(f).max(), np.abs(g - f).max() / np.abs(f).max()
    mine = [m for m in after if m[0] == 1]
    assert mine == fresh_msgs and [m[2] for m in mine] == [want[1][1]], mine


# ---- 4. capture front end: detach / attach -------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["s16", "u8"])
def test_capture_detach_and_attach(fmt):
    S, blk, chunk = 3, 252000, 126000
    rng = np.random.default_rng(41)
    t_detach, t_attach, total = 3.0, 14.0, 28.0
    b0, bbbb0 = _bulletin(rng, 14000.0, 2.0)                 # runs across the detach of stream 1
    b2, bbbb2 = _bulletin(rng, -14000.0, 4.0)
    b1, bbbb1 = _bulletin(rng, 14000.0, 0.7)                 # stream 1 after it is attached again
    full = {0: _capture_u8([b0], total, 81), 2: _capture_u8([b2], total, 82)}
    early1 = _capture_u8([], t_detach, 83)                   # noise only before the radio drops out
    late1 = _capture_u8([b1], total - t_attach, 84)

    eng = engine.Engine(S, blk)
    cap = engine.Capture(eng, blk, 4 * blk, fmt=fmt)

    def write(s, u8):
        if fmt == "u8":
            return cap.write_u8(s, u8)
        v = u8.astype(np.int16) - 128
        return cap.write(s, v[:, 0], v[:, 1])

    t = 0
    while t * chunk < total * FS:
        a, b = t * chunk, (t + 1) * chunk
        sec = a / FS
        if sec == t_detach:
            cap.detach(1)
        if sec == t_attach:
            cap.attach(1)
        for s in (0, 2):
            assert write(s, full[s][a:b]) == 0
        if sec < t_detach:
            assert write(1, early1[a:b]) == 0
        elif sec < t_attach:
            assert write(1, early1[:chunk]) == -1            # NVX_ERR_ARG: the stream is detached
        else:
            a1 = a - int(t_attach * FS)
            assert write(1, late1[a1:a1 + chunk]) == 0
        while cap.pump() > 0:
            pass
        t += 1
    cap.stop()
    msgs = eng.poll_messages()
    for s in range(S):
        assert cap.dropped(s) == 0
    assert sorted((m[0], m[2]) for m in msgs) == sorted([(0, bbbb0), (1, bbbb1), (2, bbbb2)]), msgs
    cap.close()
    eng.close()


# ---- 5. errors and edge cases --------------------------------------------------------------------------------------------
def test_lifecycle_errors_and_reset_before_the_first_push():
    eng = engine.Engine(4, 28000)
    for bad in ([4], [-1], [0, 7]):
        with pytest.raises(engine.NvxError):
            eng.reset_streams(bad)
    with pytest.raises(engine.NvxError):                      # reference-table engines cannot be retuned
        eng.retune_stream(0, [14000.0, -14000.0])
    eng.close()
    g = engine.Engine(2, 28000, nco_hz=[[14000.0, -14000.0]] * 2)
    with pytest.raises(engine.NvxError):
        g.retune_stream(0, [14000.25, -14000.0])              # off the 0.5 Hz grid
    with pytest.raises(engine.NvxError):
        g.retune_stream(0, [40000.0, -14000.0])
    with pytest.raises(engine.NvxError):
        g.retune_stream(2, [14000.0, -14000.0])
    g.close()

    eng = engine.Engine(3, 28000)
    cap = engine.Capture(eng, 28000, 4 * 28000)
    for bad in (-1, 3):
        with pytest.raises(engine.NvxError):
            cap.detach(bad)
        with pytest.raises(engine.NvxError):
            cap.attach(bad)
    cap.detach(1)
    z = np.zeros(280, np.int16)
    assert cap.write(1, z, z) == -1
    assert cap.write(0, z, z) == 0
    cap.attach(1)
    assert cap.write(1, z, z) == 0
    cap.close()
    eng.close()

    # a reset before the first push changes nothing
    rng = np.random.default_rng(3)
    b, bbbb = _bulletin(rng, 14000.0, 0.3)
    x = np.stack([_capture_u8([b], 12.0, 5), _capture_u8([], 12.0, 6)]).astype(np.int16) - 128
    blocks = _plan(np.random.default_rng(8), x.shape[1] // BLK * BLK, 0)
    outs = []
    for first in (True, False):
        e = _Keep(2, MAX_BLOCK, keep_bits=True)
        if first:
            e.reset_streams([0, 1, 0])
        outs.append(_run(e, x, blocks))
        e.close()
    (r0, _, m0), (r1, _, m1) = outs
    for s in (0, 1):
        _assert_equal_rows(r0, s, r1, s, 2)
    assert m0 == m1 and [m[2] for m in m0] == [bbbb]

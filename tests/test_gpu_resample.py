"""Engines fed at the radio's own rate (nvx_config.input_rate_hz): the rational resampler on the GPU in front of both FIR paths.

The reference of every stream is the FP64 oracle fed the float64 scipy.signal.upfirdn(h, x, L, M) of the same quantised capture,
h being nvx_resampler_info's taps; the bar is the existing one (tests/parity.py)."""
import concurrent.futures as cf
import zlib

import numpy as np
import pytest
from scipy import signal

import oracle_lib as ol
import parity
from navtex_b200 import engine, synth

pytestmark = pytest.mark.gpu

AMP = {"f32": 8000.0, "s16": 8000.0, "u8": 30.0}
MEDIUM = (signal.firwin(61, 20000, window=("kaiser", 8.0), fs=252000), signal.firwin(75, 2000, window=("kaiser", 8.0), fs=63000),
          signal.firwin(111, 250, window=("kaiser", 7.0), fs=9000))
LONG = (signal.firwin(255, 20000, window=("kaiser", 8.0), fs=252000), signal.firwin(255, 2000, window=("kaiser", 8.0), fs=63000),
        signal.firwin(255, 250, window=("kaiser", 7.0), fs=9000))
SECONDS = 7.6
# a noise-only channel decides at an arg max near-tie now and then; a slip after a pick within this margin is reported, not
# failed, as in tests/test_gpu_rows.py (seen on a B200 at 912 kS/s: one empty channel of 33, pick margin 1.1e-7)
NEAR_TIE = 1e-3


def quantise(x, fmt):
    """complex capture -> [n, 2] array in the pushed format"""
    if fmt == "s16":
        return synth.quantise_s16(x).reshape(-1, 2)
    if fmt == "u8":
        return synth.quantise_u8(x).reshape(-1, 2)
    return np.stack([x.real, x.imag], axis=1).astype(np.float32)


def value(q):
    """the sample values the engine reads, as complex128"""
    v = q.astype(np.float64) - (128.0 if q.dtype == np.uint8 else 0.0)
    return v[:, 0] + 1j * v[:, 1]


def capture(rate, fmt, offset, seed, seconds=SECONDS, start_s=0.3):
    """one bulletin at `offset` Hz with noise, quantised to fmt; returns ([n, 2] array, (bbbb, text))"""
    rng = np.random.default_rng(seed)
    text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=1)
    em = synth.Emission(text, offset, start_s=start_s, n_phasing=18, n_tail=5, amplitude=AMP[fmt])
    return quantise(synth.fsk_iq([em], seconds, snr_db=3.0, seed=seed, rate=rate), fmt), (bbbb, text)


def resampled(q, info, n):
    """float64 interleaved I,Q of upfirdn(h, x, L, M) for the 252 kS/s samples of n input samples"""
    y = signal.upfirdn(info["taps"], value(q[:n]), info["up"], info["down"])[: n * info["up"] // info["down"]]
    iq = np.empty(2 * y.size)
    iq[0::2], iq[1::2] = y.real, y.imag
    return iq


def aligned(n, align):
    return n // align * align


def pmap(fn, items):
    ol.lib()
    fn(items[0])                                   # the oracle's lazily built tables, before threads share them
    with cf.ThreadPoolExecutor(8) as ex:
        return list(ex.map(fn, items))


CASES = [  # rate, format, streams, FIR variant
    (96_000, "f32", 33, "reference"), (192_000, "s16", 33, "reference"), (250_000, "s16", 33, "reference"),
    (256_000, "u8", 33, "reference"), (912_000, "f32", 33, "reference"), (2_048_000, "u8", 3, "reference"),
    (2_400_000, "u8", 3, "reference"), (3_200_000, "s16", 3, "reference"),
    (256_000, "s16", 33, "medium"), (192_000, "f32", 33, "long"), (96_000, "u8", 33, "nco4"),
    # many polyphase branches: L = 2520 (the tap table is read from global memory; align 961 is odd, and so are S and n, so the
    # float block's last 16-byte word is partial) and L = 840 at a high rate
    (96_100, "f32", 33, "reference"), (2_000_100, "s16", 3, "reference"),
]


@pytest.mark.parametrize("rate,fmt,S,variant", CASES)
def test_parity(rate, fmt, S, variant):
    """Each stream carries its own bulletin, at +-14 kHz (or, on the four-channel engine, at its own offset); the 900 Hz samples,
    bits, events and messages match the oracle on the upfirdn of the capture, and the messages are what was sent."""
    info = engine.resampler_info(rate)
    kw, offs = {}, None
    if variant == "medium":
        kw["taps"] = MEDIUM
    elif variant == "long":
        kw["taps"] = LONG
    elif variant == "nco4":
        offs = np.array([[14000.0, -14000.0, 7000.0 + 10.5 * s, -21000.0 - 20 * s] for s in range(S)])
        kw.update(n_channels=4, nco_hz=offs, stream_freq_tag=np.tile([518, 490, 1002, 1003], (S, 1)))
    C = kw.get("n_channels", 2)
    keys = ol.CHANNEL_KEYS[:C]
    occ = [s % C for s in range(S)]
    caps = [capture(rate, fmt, (offs[s, occ[s]] if offs is not None else (14000.0, -14000.0)[occ[s]]), zlib.crc32(repr((rate, fmt, variant, s)).encode()))
            for s in range(S)]
    n = aligned(min(c[0].shape[0] for c in caps), info["align"])
    if info["align"] % 2 and (n // info["align"]) % 2 == 0:
        n -= info["align"]                                    # an odd block length: S n samples end inside a 16-byte word
    x = np.ascontiguousarray(np.stack([c[0][:n] for c in caps]))
    eng = engine.Engine(S, n, keep_bits=True, input_rate_hz=rate, **kw)
    eng.push_host(x)
    msgs = eng.poll_messages()
    y3 = eng.read_y3()
    assert y3.shape[2] == n * info["up"] // info["down"] // 280

    def oracle(s):
        ok = {}
        if variant in ("medium", "long"):
            ok = dict(h1=kw["taps"][0], h2=kw["taps"][1], h3=kw["taps"][2])
        if offs is not None:
            ok.update(nco_hz=tuple(offs[s]), freq_tag=(518, 490, 1002, 1003))
        return ol.run_oracle(resampled(caps[s][0], info, n), **ok)

    refs = pmap(oracle, list(range(S)))
    tags = (518, 490, 1002, 1003)
    for s in range(S):
        bits, disc = {}, {}
        for c in range(C):
            bits[c], disc[c] = eng.read_bits(s, c)
        occupied = {keys[occ[s]]}
        cmp = parity.compare_stream(y3[s], bits, disc, refs[s], occupied, channels=keys)
        parity.assert_stream(cmp, occupied, where="%d S/s %s %s stream %d" % (rate, fmt, variant, s), near_tie=NEAR_TIE)
        parity.record("resampled %d S/s %s %s stream %d" % (rate, fmt, variant, s), cmp, sorted(occupied))
        assert eng.read_events(s, occ[s]) == refs[s].events[keys[occ[s]]]
        want = (tags[occ[s]],) + caps[s][1]
        assert refs[s].messages == [want]
        assert [m[1:] for m in msgs if m[0] == s] == [want]
    eng.close()


def _blocks(eng, x, cuts):
    ys, msgs = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        eng.push_host(np.ascontiguousarray(x[:, a:b]))
        ys.append(eng.read_y3())
        msgs += eng.poll_messages()
    return np.concatenate(ys, axis=2), msgs


@pytest.mark.parametrize("rate,fmt,variant", [(250_000, "s16", "reference"), (2_048_000, "u8", "reference"), (96_000, "f32", "nco4"),
                                              (256_000, "s16", "long")])
def test_blocking(rate, fmt, variant):
    """One block against uneven aligned blocks: y3 bitwise equal on the fused path; on the long-tap path, whose tensor-core
    stages depend on the blocking, equal to rounding."""
    info = engine.resampler_info(rate)
    align, S = info["align"], 5
    kw = {"taps": LONG} if variant == "long" else {"n_channels": 4, "nco_hz": np.tile([14000.0, -14000.0, 3000.5, -27000.0], (S, 1))} \
        if variant == "nco4" else {}
    rng = np.random.default_rng(rate)
    k = -(-rate * 3 // align)                                # about 3 s
    n = k * align
    x = np.ascontiguousarray(np.stack([quantise((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * AMP[fmt] / 3, fmt) for _ in range(S)]))
    one = engine.Engine(S, n, input_rate_hz=rate, **kw)
    y1, _ = _blocks(one, x, [0, n])
    one.close()
    cuts = sorted({0, n, align, 4 * align, (k // 2) * align, (k - 1) * align})
    many = engine.Engine(S, n, input_rate_hz=rate, **kw)
    y2, _ = _blocks(many, x, cuts)
    many.close()
    assert np.abs(y1).max() > 0
    if variant == "long":
        assert np.abs(y1 - y2).max() <= 1e-5 * np.abs(y1).max()
    else:
        assert np.array_equal(y1.view(np.uint64), y2.view(np.uint64))


def test_native_rate_unchanged():
    """input_rate_hz = 252000 is the default engine: bitwise the same y3, bits, events and messages, and the same launches."""
    caps = [capture(252_000, "s16", (14000.0, -14000.0)[s % 2], 900 + s) for s in range(3)]
    n = aligned(min(c[0].shape[0] for c in caps), 280)
    x = np.stack([c[0][:n] for c in caps])
    cuts = [0, 280 * 900, 280 * 2000, n]
    out = []
    for rate in (0, 252_000):
        eng = engine.Engine(3, n, keep_bits=True, input_rate_hz=rate)
        y, msgs = _blocks(eng, x, cuts)
        bits = [eng.read_bits(s, c) for s in range(3) for c in range(2)]
        ev = [eng.read_events(s, c) for s in range(3) for c in range(2)]
        st = eng.stats()
        out.append((y, msgs, bits, ev, st.aux_launches, st.samples))
        eng.close()
    (ya, ma, ba, ea, la, sa), (yb, mb, bb, eb, lb, sb) = out
    assert np.array_equal(ya.view(np.uint64), yb.view(np.uint64))
    assert ma == mb and len(ma) == 3 and ea == eb and (la, sa) == (lb, sb)
    assert all(p[0] == q[0] and np.array_equal(p[1].view(np.uint32), q[1].view(np.uint32)) for p, q in zip(ba, bb))


def test_reset_streams_is_fresh_engine_fed_zeros():
    """reset_streams at input sample E: from E on the stream is, bitwise, a fresh engine fed Z = E mod (0.63 r) input-rate zeros
    and then its input."""
    rate, fmt = 256_000, "u8"
    info = engine.resampler_info(rate)
    align, grid = info["align"], 161_280
    caps = [capture(rate, fmt, (14000.0, -14000.0)[s % 2], 950 + s, seconds=9.5, start_s=1.2) for s in range(3)]
    n = aligned(min(c[0].shape[0] for c in caps), align)
    x = np.stack([c[0][:n] for c in caps])
    E = 93 * align                                            # 0.93 s: before the bulletins start
    cuts = [0, 40 * align, E, E + 300 * align, n]
    eng = engine.Engine(3, n, input_rate_hz=rate)
    eng.push_host(np.ascontiguousarray(x[:, :40 * align]))
    eng.push_host(np.ascontiguousarray(x[:, 40 * align:E]))
    eng.reset_streams([1])
    ys, msgs = [], []
    for a, b in zip(cuts[2:-1], cuts[3:]):
        eng.push_host(np.ascontiguousarray(x[:, a:b]))
        ys.append(eng.read_y3())
        msgs += eng.poll_messages()
    eng.close()
    Z = E % grid
    fresh = engine.Engine(1, n, input_rate_hz=rate)
    if Z:
        fresh.push_host(np.full((1, Z, 2), 128, np.uint8))
    yf, mf = _blocks(fresh, x[1:2], [E, E + 300 * align, n])
    fresh.close()
    yr = np.concatenate(ys, axis=2)[1:2]
    assert np.array_equal(yr.view(np.uint64), yf.view(np.uint64))
    assert [m[1:] for m in msgs if m[0] == 1] == [m[1:] for m in mf] and len(mf) == 1


def test_save_load_and_refusals():
    """Save mid-bulletin at E and load into a fresh engine at the same rate: the streams continue bitwise and the bulletin in
    flight is delivered once.  Loading into a native engine or one at another rate fails with NVX_ERR_ARG and changes nothing."""
    rate, fmt = 2_400_000, "u8"
    info = engine.resampler_info(rate)
    align = info["align"]
    caps = [capture(rate, fmt, (14000.0, -14000.0)[s % 2], 970 + s) for s in range(2)]
    n = aligned(min(c[0].shape[0] for c in caps), align)
    x = np.stack([c[0][:n] for c in caps])
    E = aligned(n // 2, align)                                # mid-bulletin
    src = engine.Engine(2, n, input_rate_hz=rate, keep_bits=True)
    src.push_host(np.ascontiguousarray(x[:, :E]))
    before = src.poll_messages()
    state = src.save_streams([0, 1])
    assert engine.stream_state_info(state)["position"] == E
    src.push_host(np.ascontiguousarray(x[:, E:]))
    y_src, m_src = src.read_y3(), src.poll_messages()
    src.close()
    assert before == [] and len(m_src) == 2

    dst = engine.Engine(2, n, input_rate_hz=rate, keep_bits=True)
    dst.load_streams([0, 1], state)
    dst.push_host(np.ascontiguousarray(x[:, E:]))
    assert np.array_equal(dst.read_y3().view(np.uint64), y_src.view(np.uint64))
    assert sorted(dst.poll_messages()) == sorted(m_src)
    dst.close()

    for other in (0, 2_048_000):
        m = 280 * 100 if other == 0 else 8 * 20_480
        eng = engine.Engine(2, m, input_rate_hz=other)
        with pytest.raises(engine.NvxError, match="fed at"):
            eng.load_streams([0, 1], state)
        blk = np.full((2, m, 2), 128, np.uint8)
        eng.push_host(blk)                                    # nothing was queued: the engine runs as if the load never happened
        assert not np.any(eng.read_y3().view(np.uint64))
        eng.close()


def test_capture_front_end_u8_2400k():
    """An 8-bit capture at 2.4 MS/s written in odd-length rtlsdr-style chunks and pumped: the bulletins come out verbatim; a
    detached stream holds nothing back and an attached one restarts."""
    rate = 2_400_000
    align = engine.resampler_info(rate)["align"]
    caps = [capture(rate, "u8", (14000.0, -14000.0)[s % 2], 990 + s) for s in range(3)]
    n = min(c[0].shape[0] for c in caps)
    blk = 20 * align
    eng = engine.Engine(3, blk, input_rate_hz=rate)
    cap = engine.Capture(eng, blk, 3 * blk, fmt="u8")
    rng = np.random.default_rng(5)
    pos, pumped = [0, 0, 0], 0
    while min(pos) < n:
        for s in range(3):
            k = min(int(rng.integers(1, 8192)) | 1, n - pos[s])
            if k > 0 and pos[s] - pumped < 2 * blk:           # the ring (3 blk) never overflows
                assert cap.write_u8(s, caps[s][0][pos[s]:pos[s] + k]) == 0
                pos[s] += k
        while (p := cap.pump()) > 0:
            pumped += p
    msgs = eng.poll_messages()
    assert sorted(m[0:1] + m[2:] for m in msgs) == sorted((s,) + caps[s][1] for s in range(3))

    cap.detach(2)                                             # stream 2 stops: the others are pumped without it
    assert cap.write_u8(2, caps[2][0][:align]) == -1
    for s in range(2):
        assert cap.write_u8(s, caps[s][0][:blk]) == 0
    assert cap.pump() == blk
    cap.attach(2)
    for s in range(3):
        assert cap.write_u8(s, caps[s][0][:blk + 7]) == 0
    assert cap.pump() == blk                                  # a multiple of the engine's alignment, 7 samples stay behind
    cap.close()
    eng.close()


def test_more_than_2g_input_samples_in_one_block():
    """1024 streams x 10.24 s at 256 kS/s, 8-bit, in one device block (2.7 G input samples): stream s carries capture s mod 16
    and its own tag; every message arrives once, with the right stream id and tag."""
    import torch

    rate, S = 256_000, 1024
    n = 1024 * 2560
    caps = [capture(rate, "u8", (14000.0, -14000.0)[k % 2], 1100 + k, seconds=10.24) for k in range(16)]
    base = torch.from_numpy(np.stack([c[0][:n] for c in caps])).cuda()
    x = base[torch.arange(S) % 16].contiguous()
    del base
    assert x.numel() // 2 > 2 ** 31
    tags = np.stack([np.arange(S) + 10_000, np.arange(S) + 20_000], axis=1)
    eng = engine.Engine(S, n, input_rate_hz=rate, stream_freq_tag=tags)
    torch.cuda.synchronize()
    eng.push_device(x.data_ptr(), n, u8=True)
    msgs = eng.poll_messages()
    eng.close()
    assert len(msgs) == S
    got = sorted(msgs)
    want = sorted((s, int(tags[s, (s % 16) % 2]), caps[s % 16][1][0], caps[s % 16][1][1]) for s in range(S))
    assert got == want


def _launch_rates():
    """the accepted rates with the most branches and the longest windows, and a seeded sample of the rest"""
    from math import gcd
    worst = [r for r in range(3_200_000, 3_100_000, -100) if 2520 // gcd(2520, r // 100) == 2520][:3]
    rng = np.random.default_rng(2520)
    return [96_100, 96_700, 2_000_100] + worst + sorted(int(v) * 100 for v in rng.integers(960, 32_001, size=24))


def test_every_rate_launches():
    """Rates with up to 2520 branches and the widest windows create an engine and push blocks in all three formats (whose
    results do not depend on the format: the same values u - 128); the tap table that does not fit shared memory is read
    from global memory."""
    for rate in _launch_rates():
        info = engine.resampler_info(rate)
        n = 3 * info["align"]
        rng = np.random.default_rng(rate)
        u = rng.integers(0, 256, size=(3, 2 * n, 2), dtype=np.uint8)
        ys = []
        for x in (u, u.astype(np.int16) - 128, (u.astype(np.int16) - 128).astype(np.float32)):
            eng = engine.Engine(3, n, input_rate_hz=rate)
            y = []
            for a in (0, n):
                eng.push_host(np.ascontiguousarray(x[:, a:a + n]))
                y.append(eng.read_y3())
            eng.close()
            ys.append(np.concatenate(y, axis=2))
        assert ys[0].shape[2] == 2 * n * info["up"] // info["down"] // 280, rate
        assert np.all(np.isfinite(ys[0])) and np.abs(ys[0]).max() > 0, rate
        for y in ys[1:]:
            assert np.array_equal(ys[0].view(np.uint64), y.view(np.uint64)), rate


def test_argument_errors():
    for bad in (95_900, 3_200_100, 250_001, 252_001, -1):
        with pytest.raises(engine.NvxError, match="input_rate_hz"):
            engine.Engine(1, 2560 * 4, input_rate_hz=bad)
    with pytest.raises(engine.NvxError, match="max_block"):
        engine.Engine(1, 2800, input_rate_hz=256_000)          # a multiple of 280, not of 2560
    eng = engine.Engine(1, 2560 * 4, input_rate_hz=256_000)
    with pytest.raises(engine.NvxError, match="2560"):
        eng.push_host(np.full((1, 2800, 2), 128, np.uint8))
    with pytest.raises(engine.NvxError):
        engine.Capture(eng, 2800, 4 * 2800, fmt="u8")
    cap = engine.Capture(eng, 2560 * 2, 2560 * 4, fmt="u8")
    cap.close()
    eng.push_host(np.full((1, 2560, 2), 128, np.uint8))       # the failed push fixed nothing
    eng.close()

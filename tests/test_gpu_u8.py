"""8-bit unsigned I,Q input (the RTL-SDR's rtlsdr_read_async / rtl_tcp sample format) on the GPU.

A byte u is the sample value u - 128, exactly.  Those values are integers, so the same capture pushed as float or int16 must
give bit-identical 900 Hz samples, events and messages through every kernel variant -- the fused cascade's own 8-bit staging and
in-register conversion, and the long-tap path's widening to int16 -- and the oracles fed u - 128 as int16 are the parity bar."""
import threading
import zlib

import numpy as np
import pytest
from scipy import signal

import oracle_lib as ol
import parity
from navtex_b200 import engine, synth

pytestmark = pytest.mark.gpu

CLASS0 = (signal.firwin(33, 21000, window=("kaiser", 6.0), fs=252000), signal.firwin(45, 2200, window=("kaiser", 6.5), fs=63000),
          signal.firwin(69, 260, window=("kaiser", 5.0), fs=9000))
MEDIUM = (signal.firwin(61, 20000, window=("kaiser", 8.0), fs=252000), signal.firwin(75, 2000, window=("kaiser", 8.0), fs=63000),
          signal.firwin(111, 250, window=("kaiser", 7.0), fs=9000))
OFFSETS = [14000.0, -14000.0, 7000.0, -21000.0, 21000.5, -7000.5, 0.0, 28000.0]


def _engine_kwargs(variant, S):
    if variant == "reference":
        return {}
    if variant == "class0":
        return {"taps": CLASS0}
    if variant == "medium":
        return {"taps": MEDIUM}
    n_ch = int(variant[3:])                      # "ncoK": per-stream NCO with K channels
    return {"n_channels": n_ch, "nco_hz": np.tile(np.array(OFFSETS[:n_ch]), (S, 1))}


def _run(x, variant, blk, push, m):
    """Push x[:, :m] in blocks of blk as its dtype; returns (y3 of every block, events of the last block, messages)."""
    import torch

    S = x.shape[0]
    eng = engine.Engine(S, blk, **_engine_kwargs(variant, S))
    ys, msgs = [], []
    for a in range(0, m, blk):
        xb = np.ascontiguousarray(x[:, a:a + blk])
        if push == "host":
            eng.push_host(xb)
        else:
            d = torch.from_numpy(xb).cuda()
            torch.cuda.synchronize()
            eng.push_device(d.data_ptr(), blk, s16=xb.dtype == np.int16, u8=xb.dtype == np.uint8)
        ys.append(eng.read_y3())                 # (implies sync: the device block may go)
        msgs += eng.poll_messages()
    events = [eng.read_events(s, c) for s in range(S) for c in range(eng.C)]
    eng.close()
    return np.concatenate(ys, axis=2), events, msgs


@pytest.mark.parametrize("variant,S,blk,push", [
    ("reference", 33, 280 * 333, "host"), ("reference", 130, 2520 * 40, "device"), ("reference", 33, 280, "host"),
    ("class0", 130, 280 * 333, "device"), ("class0", 33, 280, "host"),
    ("medium", 33, 2520 * 40, "host"), ("medium", 130, 280 * 333, "device"), ("medium", 33, 280, "device"),
    ("nco1", 33, 280 * 333, "host"), ("nco2", 130, 2520 * 40, "device"), ("nco3", 33, 280 * 333, "device"),
    ("nco4", 130, 280 * 333, "host"), ("nco5", 33, 2520 * 40, "host"), ("nco8", 33, 280 * 333, "device"), ("nco8", 33, 280, "host"),
])
def test_u8_bit_identical_to_float_and_int16(variant, S, blk, push):
    """Random full-range bytes (0 and 255 included) pushed as 8-bit pairs, and the same values u - 128 as float32 and int16: the
    900 Hz samples of every block are bit-identical, and so are the events and messages.  Several blocks, so the carried 8-bit
    tail feeds the next block's warm-up."""
    rng = np.random.default_rng(zlib.crc32(repr((variant, S, blk, push)).encode()))
    n = 2520 * 40 * 3
    m = 280 * 200 if blk == 280 else n // blk * blk
    u = rng.integers(0, 256, size=(S, n, 2), dtype=np.uint8)
    u[0, :2] = [[0, 255], [255, 0]]
    v = u.astype(np.int16) - 128
    y8, ev8, msg8 = _run(u, variant, blk, push, m)
    assert np.abs(y8).max() > 0
    for other in (v.astype(np.float32), v):
        y, ev, msg = _run(other, variant, blk, push, m)
        assert np.array_equal(y8.view(np.uint64), y.view(np.uint64)), other.dtype
        assert ev8 == ev and sorted(msg8) == sorted(msg), other.dtype


def _designs(n1, n2, n3):
    return (signal.firwin(n1, 20000, window=("kaiser", 8.0), fs=252000), signal.firwin(n2, 2000, window=("kaiser", 8.0), fs=63000),
            signal.firwin(n3, 250, window=("kaiser", 7.0), fs=9000))


@pytest.mark.parametrize("tc", ["default", "0"])
@pytest.mark.parametrize("lengths", [(255, 255, 255), (516, 900, 71)])
def test_u8_long_taps_equal_int16(monkeypatch, tc, lengths):
    """Long-tap path: 8-bit blocks are widened to int16 (u - 128) in one small kernel, counted in aux_launches, in front of the
    unchanged int16 path -- bit-identical to pushing the same values as int16, on the tensor-core and the CUDA-core stages."""
    if tc != "default":
        monkeypatch.setenv("NVX_LONG_TC", tc)
    taps = _designs(*lengths)
    S, blk = 33, 2520 * 40
    rng = np.random.default_rng(sum(lengths))
    u = rng.integers(0, 256, size=(S, 2 * blk, 2), dtype=np.uint8)
    out = {}
    for name, x in (("u8", u), ("s16", u.astype(np.int16) - 128)):
        eng = engine.Engine(S, blk, taps=taps)
        ys = []
        for a in (0, blk):
            eng.push_host(np.ascontiguousarray(x[:, a:a + blk]))
            ys.append(eng.read_y3())
        out[name] = (np.concatenate(ys, axis=2), eng.stats())
        eng.close()
    (y8, st8), (y16, st16) = out["u8"], out["s16"]
    assert np.abs(y8).max() > 0
    assert np.array_equal(y8.view(np.uint64), y16.view(np.uint64))
    assert st8.long_tc_fallbacks == st16.long_tc_fallbacks
    assert st8.aux_launches == st16.aux_launches + 2


def _capture_u8(text, offset, seconds, snr, seed):
    """An 8-bit capture: the emission at 8-bit scale (30 LSB), AWGN, quantised as an RTL-SDR would."""
    em = synth.Emission(text, offset, start_s=0.3, n_phasing=18, n_tail=5, amplitude=30.0)
    return synth.quantise_u8(synth.fsk_iq([em], seconds, snr_db=snr, seed=seed))


@pytest.fixture(scope="module")
def captures():
    rng = np.random.default_rng(88)
    seconds = 11.0
    iqs, want = [], []
    for s in range(3):
        text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=3)
        occ = s % 2
        iqs.append(_capture_u8(text, 14000.0 if occ == 0 else -14000.0, seconds, snr=-3.0, seed=800 + s))
        want.append((518 if occ == 0 else 490, bbbb, text))
    return iqs, want


def _parity(captures, run):
    """900 Hz samples within tests/parity.py's 1e-5, bits, events and messages exact against `run` fed u - 128 as int16, and
    the messages what was transmitted."""
    iqs, want = captures
    x = np.stack([iq.reshape(-1, 2) for iq in iqs])
    assert 64 < np.abs(x.astype(int) - 128).max() <= 128                                    # really 8-bit scale
    n = x.shape[1]
    eng = engine.Engine(3, n, keep_bits=True)
    eng.push_host(np.ascontiguousarray(x))
    msgs = eng.poll_messages()
    y3 = eng.read_y3()
    for s, iq in enumerate(iqs):
        v = iq.astype(np.int16) - 128
        occ = ol.CHANNELS[s % 2]
        o = run(v)
        bits, disc = {}, {}
        for c in range(2):
            bits[c], disc[c] = eng.read_bits(s, c)
        cmp = parity.compare_stream(y3[s], bits, disc, o, {occ})
        parity.assert_stream(cmp, {occ}, where="8-bit stream %d" % s)
        parity.record("8-bit stream %d" % s, cmp, [occ])
        if o.events:                             # (the unmodified reference's run reports messages, not events)
            assert eng.read_events(s, s % 2) == o.events[occ]
        assert o.messages == [want[s]]
        assert [m[1:] for m in msgs if m[0] == s] == [want[s]]
    eng.close()


def test_u8_parity_with_restated_oracle(captures):
    _parity(captures, ol.run_oracle)


def test_u8_parity_with_unmodified_reference(captures):
    if not ol.have_ref():
        pytest.skip("oracle/_ref/ref_chain was not built (reference tree absent at build time)")
    _parity(captures, ol.run_ref)


def test_u8_format_lock_and_reset(captures):
    iqs, _ = captures
    n = iqs[0].size // 2
    u = np.ascontiguousarray(iqs[0].reshape(1, n, 2))
    v = u.astype(np.int16) - 128
    eng = engine.Engine(1, n)
    eng.push_host(u)
    first, y_first = eng.poll_messages(), eng.read_y3().copy()
    for other in (v.astype(np.float32), v):
        eng.reset()
        eng.push_host(other)
        with pytest.raises(engine.NvxError, match="format"):
            eng.push_host(u)                     # 8-bit after float / int16 without a reset
    eng.reset()
    eng.push_host(u)
    assert eng.poll_messages() == first and len(first) == 1
    assert np.array_equal(eng.read_y3().view(np.uint64), y_first.view(np.uint64))
    eng.close()


def test_u8_capture_front_end(captures):
    """Producer threads (one per stream) write uneven RTL-style buffers into 8-bit rings while the poller pumps: the messages
    equal one direct push_host_u8 of the same captures.  Overflow, wrong-format writes, and digital silence."""
    import time

    iqs, want = captures
    x = np.stack([iq.reshape(-1, 2) for iq in iqs])
    S, n = x.shape[0], x.shape[1]
    direct = engine.Engine(S, n)
    direct.push_host(np.ascontiguousarray(x))
    ref_msgs = direct.poll_messages()
    direct.close()
    assert sorted(m[1:] for m in ref_msgs) == sorted(want)

    blk = 280 * 90
    eng = engine.Engine(S, blk)
    cap = engine.Capture(eng, blk, n, fmt="u8")                    # a ring that holds the whole capture: no overflow here
    cap.start(poll_ms=5)
    rcs = [[] for _ in range(S)]

    def producer(s):
        rng = np.random.default_rng(s)
        pos = 0
        while pos < n:
            k = min(int(rng.integers(1, 16384)), n - pos)          # uneven buffers, up to librtlsdr's 16384 pairs
            rcs[s].append(cap.write_u8(s, x[s, pos:pos + k]))
            pos += k
            if rng.random() < 0.01:
                time.sleep(0.001)
    threads = [threading.Thread(target=producer, args=(s,)) for s in range(S)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    cap.stop()
    msgs = eng.poll_messages()
    assert all(rc == 0 for r in rcs for rc in r)
    assert sorted(msgs) == sorted(ref_msgs)
    assert all(cap.dropped(s) == 0 for s in range(S))
    cap.close()

    # overflow: the excess is dropped and counted; wrong-format writes are refused
    cap = engine.Capture(eng, blk, 2 * blk, fmt="u8")
    assert cap.write_u8(0, np.full((3 * blk, 2), 128, dtype=np.uint8)) == -4
    assert cap.dropped(0) == blk
    assert cap.write(0, np.zeros(280, np.int16), np.zeros(280, np.int16)) == -1
    cap.close()
    cap16 = engine.Capture(eng, blk, 2 * blk)
    assert cap16.write_u8(0, np.full((280, 2), 128, dtype=np.uint8)) == -1
    cap16.close()
    eng.close()

    # digital silence: every byte 128 is the value 0
    eng = engine.Engine(S, blk)
    cap = engine.Capture(eng, blk, 4 * blk, fmt="u8")
    for s in range(S):
        assert cap.write_u8(s, np.full((blk, 2), 128, dtype=np.uint8)) == 0
    assert cap.pump() == blk
    assert not np.any(eng.read_y3().view(np.uint64))
    assert eng.poll_messages() == []
    cap.close()
    eng.close()

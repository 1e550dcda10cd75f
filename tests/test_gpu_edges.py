"""GPU edge cases of the hot path against the CPU oracle: the config-1 WAV, digital silence, full-scale input, one very
long single-stream block (maximum time segmentation), reset, sample-format mixing, argument errors."""
import os

import numpy as np
import pytest

import cases
import oracle_lib as ol
import parity
from navtex_b200 import engine, synth

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REL_TOL = 1e-5


def _check_all(eng, k, o, exact_channels=("518", "490"), where=""):
    """tests/parity.py's bar for the channels that carry something to decide on; events exact there, decisions of the others
    counted and reported."""
    y3 = eng.read_y3()
    bits, disc = {}, {}
    for c in range(2):
        bits[c], disc[c] = eng.read_bits(k, c)
    cmp = parity.compare_stream(y3[k], bits, disc, o, set(exact_channels))
    parity.assert_stream(cmp, set(exact_channels), where=where)
    parity.record(where or "edge case", cmp, exact_channels)
    for c, tag in enumerate(ol.CHANNELS):
        if tag in exact_channels:
            assert eng.read_events(k, c) == o.events[tag], tag


def test_config1_wav_file(tmp_path):
    """BASELINE.json configs[0]: the single 518 kHz WAV (stereo s16, 252 kHz: the format wav.c / PrepWav writes,
    capt_sched.c:87-96) -> frames -> engine, against the golden add_message calls of the unmodified reference."""
    iq = cases.build("clean518")
    path = str(tmp_path / "navtex518.wav")
    synth.write_wav(path, iq)
    frames = synth.read_wav(path)                      # interleaved I,Q shorts, as wav_read hands them over
    n = frames.size // 2 // 280 * 280
    eng = engine.Engine(1, n, keep_bits=True)
    eng.push_host(np.ascontiguousarray(frames[: 2 * n].reshape(1, n, 2)))
    msgs = eng.poll_messages()
    g = np.load(os.path.join(GOLDEN, "clean518.npz"))
    gold = [(0, int(f), str(b), str(t)) for f, b, t in zip(g["msg_freq"], g["msg_bbbb"], g["msg_text"])]
    assert msgs == gold and len(gold) == 1
    _check_all(eng, 0, ol.run_oracle(frames[: 2 * n]), exact_channels=("518",), where="config-1 WAV")
    eng.close()


def test_digital_silence_and_full_scale():
    """All-zero input: every per-offset sum ties at 0 and the first maximum must win exactly as in the reference
    (free-running symbol clock, bits from the 'B' > 'Y' tie rule).  Full-scale square wave: no overflow, same bar."""
    n = 280 * 9 * 400
    zeros = np.zeros((n, 2), dtype=np.int16)
    t = np.arange(n)
    square = np.stack([np.where((t // 9) % 2 == 0, 32767, -32768), np.where((t // 7) % 2 == 0, -32768, 32767)], axis=1).astype(np.int16)
    x = np.stack([zeros, square])
    eng = engine.Engine(2, n, keep_bits=True)
    eng.push_host(np.ascontiguousarray(x))
    assert eng.poll_messages() == []
    o0 = ol.run_oracle(zeros.reshape(-1))
    _check_all(eng, 0, o0, where="digital silence")
    assert len(o0.bits["518"]) > 300 and set(o0.bits["518"]) == {ord("Y")}          # ties decide 'Y' (decoder.C:125)
    o1 = ol.run_oracle(square.reshape(-1))
    y3 = eng.read_y3()
    scale = max(np.abs(o1.y3["518"]).max(), np.abs(o1.y3["490"]).max())
    for c, tag in enumerate(ol.CHANNELS):
        assert np.abs(y3[1, c].astype(np.complex128) - o1.y3[tag]).max() <= REL_TOL * scale
    eng.close()


def test_one_stream_one_minute_single_block():
    """A single stream pushed as one 60 s block: the time axis is cut into the maximum number of segments (one group
    of 32 lanes, 31 of them TMA zero fill) and must still equal the oracle's sequential pass."""
    rng = np.random.default_rng(41)
    text, bbbb = synth.random_message(rng, n_lines=3, words_per_line=5)
    em = synth.Emission(text, 14000.0, start_s=2.0, n_phasing=40, n_tail=6)
    iq = synth.quantise_s16(synth.fsk_iq([em], 60.0, snr_db=-12.0, seed=42))
    n = iq.size // 2
    eng = engine.Engine(1, n, keep_bits=True)
    eng.push_host(np.ascontiguousarray(iq.reshape(1, n, 2)))
    msgs = eng.poll_messages()
    o = ol.run_oracle(iq)
    assert [m[1:] for m in msgs] == o.messages == [(518, bbbb, text)]
    _check_all(eng, 0, o, exact_channels=("518",), where="one stream, 60 s, single block")
    eng.close()


def test_reset_reproduces_and_formats_do_not_mix():
    iq = cases.build("noisy490")
    n = iq.size // 2 // 280 * 280
    x = np.ascontiguousarray(iq[: 2 * n].reshape(1, n, 2))
    eng = engine.Engine(1, n)
    eng.push_host(x)
    first, y_first = eng.poll_messages(), eng.read_y3().copy()
    with pytest.raises(engine.NvxError, match="format"):
        eng.push_host(x.astype(np.float32))              # int16 then float without a reset
    eng.reset()
    eng.push_host(x.astype(np.float32))                  # after a reset either format is fine
    assert eng.poll_messages() == first and len(first) == 1
    assert np.array_equal(eng.read_y3().view(np.uint64), y_first.view(np.uint64))
    eng.close()


def test_argument_errors():
    import torch

    eng = engine.Engine(2, 2800)
    with pytest.raises(engine.NvxError):
        eng.push_host(np.zeros((2, 281, 2), dtype=np.float32))       # not a multiple of 280
    with pytest.raises(engine.NvxError):
        eng.push_host(np.zeros((2, 5600, 2), dtype=np.float32))      # longer than max_block
    # a rejected device push does not fix the sample format: the next valid push may come in another one
    xf = torch.zeros((2, 2800, 2), dtype=torch.float32, device="cuda")
    xs = torch.zeros((2, 2800, 2), dtype=torch.int16, device="cuda")
    with pytest.raises(engine.NvxError):
        eng.push_device(xf.data_ptr(), 2790)
    eng.push_device(xs.data_ptr(), 2800, s16=True)
    eng.sync()
    eng.close()
    with pytest.raises(engine.NvxError):
        engine.Engine(0, 2800)
    with pytest.raises(engine.NvxError):
        engine.Engine(40000, 2800)                                   # more than one engine's worth of streams
    with pytest.raises(engine.NvxError):
        engine.Engine(1, 2800, taps=(np.ones(2000), np.ones(47), np.ones(71)))


def test_c_and_relinked_hosts(tmp_path):
    """The two example hosts -- plain C on the batched ABI, and a C++ host that only knows the reference's own names
    (init_fir_filter1 / sample_in_1 / init_fir2_wrapper / add_message, nav_sched.C-style wiring) -- print the golden
    messages of the unmodified reference."""
    import subprocess

    from test_abi import build_example

    iq = cases.build("clean518")
    g = np.load(os.path.join(GOLDEN, "clean518.npz"))
    want = "".join("%d|%s|%d\n%s\n" % (int(f), str(b), len(str(t)), str(t)) for f, b, t in zip(g["msg_freq"], g["msg_bbbb"], g["msg_text"]))
    wav, raw = str(tmp_path / "c.wav"), str(tmp_path / "c.s16")
    synth.write_wav(wav, iq)
    iq.tofile(raw)
    out = subprocess.run([build_example("wav_decode.c", tmp_path), wav], capture_output=True, text=True, check=True)
    assert out.stdout == want
    out = subprocess.run([build_example("relink_host.cpp", tmp_path), raw], capture_output=True, text=True, check=True)
    assert out.stdout == want


def test_reference_nav_sched_and_wav_c_host_on_the_gpu(tmp_path):
    """BASELINE.json configs[0] through the reference's own files: receiver/wav.c reads the WAV (wav_open / wav_read,
    wav.c:469, :494-528), the reference's unmodified nav_sched.C wires the object graph (compiled against include/compat/),
    sample_in_1 feeds libnavtex_compat.so -- and the host's add_message receives the golden call of the unmodified CPU chain.
    The binary is built where /root/reference is mounted (oracle/Makefile: compat_wav_host) and travels prebuilt."""
    import subprocess

    exe = os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "_ref", "compat_wav_host")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/compat_wav_host was not built (reference tree absent at build time)")
    g = np.load(os.path.join(GOLDEN, "clean518.npz"))
    want = "".join("%d|%s|%d\n%s\n" % (int(f), str(b), len(str(t)), str(t)) for f, b, t in zip(g["msg_freq"], g["msg_bbbb"], g["msg_text"]))
    wav = str(tmp_path / "navtex518.wav")
    synth.write_wav(wav, cases.build("clean518"))
    out = subprocess.run([exe, wav], capture_output=True, text=True, check=True)
    assert out.stdout == want and want.startswith("518|PA12|")


def test_two_engines_with_different_taps_on_one_device():
    """Tap sets are per engine (kernel parameter block), not per process: three engines alive on one device -- reference taps,
    a replacement class-0 set, and a long-tap set -- interleave their pushes and each equals its own oracle."""
    from scipy import signal

    iq = cases.build("clean518")
    n = iq.size // 2 // 280 * 280
    x = np.ascontiguousarray(iq[: 2 * n].reshape(1, n, 2))
    short = (signal.firwin(33, 21000, window=("kaiser", 6.0), fs=252000), signal.firwin(45, 2200, window=("kaiser", 6.5), fs=63000),
             signal.firwin(69, 260, window=("kaiser", 5.0), fs=9000))
    long_ = tuple(signal.firwin(129, fc, window=("kaiser", 8.0), fs=fs) for fc, fs in ((20000, 252000), (2000, 63000), (250, 9000)))
    sets = [None, short, long_]
    engs = [engine.Engine(1, n // 2, keep_bits=True, taps=t) for t in sets]          # all three alive before the first push
    oracles = [ol.run_oracle(iq[: 2 * n]) if t is None else ol.run_oracle(iq[: 2 * n], h1=t[0], h2=t[1], h3=t[2]) for t in sets]
    y3 = [[], [], []]
    for half in range(2):                                                             # interleaved: A, B, C, A, B, C
        for k, e in enumerate(engs):
            e.push_host(np.ascontiguousarray(x[:, half * (n // 2):(half + 1) * (n // 2)]))
            y3[k].append(e.read_y3()[0].copy())
    for k, (e, o) in enumerate(zip(engs, oracles)):
        got = np.concatenate(y3[k], axis=1)
        scale = max(np.abs(o.y3["518"]).max(), np.abs(o.y3["490"]).max())
        for c, tag in enumerate(ol.CHANNELS):
            assert np.abs(got[c].astype(np.complex128) - o.y3[tag]).max() <= REL_TOL * scale, (k, tag)
        assert [m[1:] for m in e.poll_messages()] == o.messages, k
    # the three filter sets really differ at the 900 Hz output
    assert np.abs(np.concatenate(y3[0], axis=1) - np.concatenate(y3[1], axis=1)).max() > 1e-3 * scale
    st = engs[2].stats()
    assert st.long_tc_fallbacks == 0
    for e in engs:
        e.close()


def test_long_tc_fallback_is_counted_and_explained(monkeypatch):
    """Stage 2 beyond 959 taps is not served by the tensor-core kernel: it runs on the CUDA-core one, and says so."""
    from scipy import signal

    taps = (signal.firwin(255, 20000, window=("kaiser", 8.0), fs=252000), signal.firwin(1001, 2000, window=("kaiser", 8.0), fs=63000),
            signal.firwin(71, 250, window=("kaiser", 7.0), fs=9000))
    n = 280 * 90
    eng = engine.Engine(2, n, taps=taps)
    assert "stage 2" in eng.L.nvx_last_error().decode() and "CUDA-core" in eng.L.nvx_last_error().decode()
    eng.push_host(np.zeros((2, n, 2), dtype=np.float32))
    eng.push_host(np.zeros((2, n, 2), dtype=np.float32))
    st = eng.stats()
    assert st.long_tc_fallbacks == 2
    eng.close()


def test_callbacks_arrive_while_the_capture_runs():
    """INTEGRATION.md's pattern: radio callbacks write the rings, the capture poller pumps, nvx_store_sink is the message
    callback -- rows must appear in the store while the capture is still running (the reference calls add_message the moment
    NNNN is seen, nav_b_sm.C:82-88), not only at nvx_capture_stop / sync."""
    import time

    iq = cases.build("clean518").reshape(-1, 2)
    blk = 280 * 90                                  # 0.1 s blocks
    eng = engine.Engine(1, blk)
    store = engine.Store()
    store.attach(eng)
    cap = engine.Capture(eng, blk, 8 * blk)
    cap.start(poll_ms=5)
    pos, seen_at = 0, None
    while pos < len(iq):                           # the "radio": 1008-sample callbacks, as fast as the ring takes them
        n = min(1008, len(iq) - pos)
        if cap.write(0, iq[pos:pos + n, 0], iq[pos:pos + n, 1]) == 0:
            pos += n
        else:
            time.sleep(0.002)
        if seen_at is None and len(store.rows()) > 0:
            seen_at = pos
    deadline = time.time() + 5.0                   # tail of the capture after the bulletin: the poller is still running
    while seen_at is None and time.time() < deadline:
        time.sleep(0.01)
        if len(store.rows()) > 0:
            seen_at = pos
    rows_before_stop = store.rows()
    cap.stop()
    assert rows_before_stop and rows_before_stop[0][2] == "PA12", "no message reached the store before nvx_capture_stop"
    assert store.rows() == rows_before_stop
    assert eng.stats().messages == 1
    cap.close(); store.close(); eng.close()


def test_two_engines_on_two_devices_in_one_process():
    """One process, one engine per GPU (INTEGRATION.md 3): function attributes and constant-bank tables are per device."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    iq = cases.build("clean518")
    n = iq.size // 2 // 280 * 280
    x = np.ascontiguousarray(iq[: 2 * n].reshape(1, n, 2))
    engs = [engine.Engine(1, n, device=d, first_stream_id=10 * d) for d in (0, 1)]
    for e in engs:
        e.push_host(x)
    got = [e.poll_messages() for e in engs]
    assert [m[1:] for m in got[0]] == [m[1:] for m in got[1]] and len(got[0]) == 1
    assert got[0][0][0] == 0 and got[1][0][0] == 10
    assert np.array_equal(engs[0].read_y3().view(np.uint64), engs[1].read_y3().view(np.uint64))
    for e in engs:
        e.close()


def test_pinned_host_pushes_fence_and_kernel_spans():
    """nvx_pinned_alloc buffers (the e2e arm's input) give the same bits as a pageable push; nvx_engine_fence orders the engine's
    main stream behind the demod stream; the per-launch kernel times are reported one per timed push."""
    import torch

    iq = cases.build("noisy490")
    n = iq.size // 2 // 280 * 280 // 2
    x = np.ascontiguousarray(iq[: 4 * n].reshape(1, 2 * n, 2))
    ref = engine.Engine(1, n)
    ys_ref = []
    for k in range(2):
        ref.push_host(np.ascontiguousarray(x[:, k * n:(k + 1) * n]))
        ys_ref.append(ref.read_y3().copy())
    msgs_ref = ref.poll_messages()
    ref.close()
    for wc in (False, True):
        pin = engine.PinnedBuffer((2, 1, n, 2), np.int16, write_combined=wc)
        pin.array[0], pin.array[1] = x[:, :n], x[:, n:]
        eng = engine.Engine(1, n)
        eng.enable_timing(1)
        eng.stats()
        es = torch.cuda.ExternalStream(eng.stream)
        for k in range(2):
            eng.push_host_ptr(pin.ptr + k * n * 4, n, s16=True)
            eng.fence()
            done = torch.cuda.Event()
            done.record(es)
            done.synchronize()                       # everything of block k, demod stream included, is over: its events are on the host
            assert np.array_equal(eng.read_y3().view(np.uint64), ys_ref[k].view(np.uint64))
        spans = eng.cascade_spans()
        st = eng.stats()
        assert len(spans) == 2 and abs(float(spans.sum()) - st.cascade_ms) < 1e-3 and st.cascade_ms_min <= st.cascade_ms_max
        assert eng.poll_messages() == msgs_ref and len(msgs_ref) == 1
        eng.close()
        pin.close()

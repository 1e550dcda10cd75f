"""Saved stream state: a stream survives an engine restart (nvx_engine_save_streams, then nvx_engine_load_streams into a fresh
engine) or moves into another running engine, and continues bit for bit as the uninterrupted stream would (navtex_b200.h).

Every check compares against a reference engine R fed all the input without interruption: y3, bits, discriminator sums and
events of every block after the save bit for bit, and the messages of the interrupted run (source before the save plus
destination after it) equal to R's, each bulletin once and with its full text.  The save points fall between ZCZC and NNNN on
some streams and inside the phasing signal on others, and off the 158 760-sample grid, so a restarted engine must adopt the
saved position."""
import numpy as np
import pytest

from navtex_b200 import engine
from test_gpu_longtaps import designs
from test_gpu_stream_lifecycle import BLK, FS, MAX_BLOCK, RING, _as_fmt, _assert_equal_rows, _bulletin, _capture_u8, _Keep, _plan, _run

pytestmark = pytest.mark.gpu

SECONDS = 20.0
N = int(SECONDS * FS)
CUT = 8 * FS                                 # the save point: 2 016 000 samples, not a multiple of 158 760
assert CUT % RING and CUT % BLK == 0
# bulletin starts relative to the save point: streams 0-2 are past their ZCZC line there, streams 3-5 still in their phasing
STARTS = (-6.0, -6.5, -7.0, -1.0, -0.5, -1.5)


def _scenario(seed, offsets):
    rng = np.random.default_rng(seed)
    rows, want = [], []
    for s, t in enumerate(STARTS):
        b, bbbb = _bulletin(rng, offsets[s], CUT / FS + t)
        rows.append(_capture_u8([b], SECONDS, seed * 10 + s))
        want.append(bbbb)
    return np.stack(rows), want


def _restart(mk, x, blocks, at, keep_bits=True):
    """engine A runs blocks [0, at), saves every stream and is destroyed; a fresh engine B loads the state and runs the rest"""
    a = mk()
    _, _, msgs_a = _run(a, x, blocks[:at], keep_bits=keep_bits)
    state = a.save_streams(np.arange(a.S))
    a.close()
    info = engine.stream_state_info(state)
    assert info["count"] == x.shape[0] and info["position"] == sum(blocks[:at])
    b = mk()
    b.load_streams(np.arange(b.S), state)
    recs, _, msgs_b = _run(b, np.ascontiguousarray(x[:, sum(blocks[:at]):]), blocks[at:], keep_bits=keep_bits)
    b.close()
    return recs, msgs_a, msgs_b


def _check_restart(mk, x, blocks, at, want, C, chans, keep_bits=True):
    """chans[s]: the channel stream s's bulletin is received on"""
    ref = mk()
    base, _, base_msgs = _run(ref, x, blocks, keep_bits=keep_bits)
    ref.close()
    for s in range(3):                                                        # the save falls after their ZCZC line
        assert b"ZC" in b"".join(r["ev"][s, chans[s]] for r in base[:at]), s
    got, msgs_a, msgs_b = _restart(mk, x, blocks, at, keep_bits)
    for s in range(x.shape[0]):
        _assert_equal_rows(got, s, base[at:], s, C, bits=keep_bits, where=("stream", s))
    assert sorted(msgs_a + msgs_b) == sorted(base_msgs)
    assert sorted(m[2] for m in base_msgs) == sorted(want), base_msgs       # every bulletin once, in R and so across the restart
    assert not msgs_a                                                         # all of them were in flight at the save
    return base_msgs


def _blocks(seed):
    blocks = _plan(np.random.default_rng(seed), N // BLK * BLK, CUT)
    at = int(np.searchsorted(np.cumsum(blocks), CUT)) + 1
    assert sum(blocks[:at]) == CUT
    return blocks, at


# ---- 1. restart, fused path ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt,nco", [("f32", False), ("s16", False), ("u8", False), ("u8", True)],
                         ids=["f32-table", "s16-table", "u8-table", "u8-nco4"])
def test_restart_fused_path(fmt, nco):
    S = len(STARTS)
    if nco:
        C = 4
        nco_hz = np.array([[-21000.5 + 1500 * s, -7000.0, 9000.5 - 500 * s, 14000.0 + 0.5 * s] for s in range(S)])
        offs = [nco_hz[s][s % C] for s in range(S)]
        tags = np.arange(S * C).reshape(S, C) + 700
        mk = lambda: _Keep(S, MAX_BLOCK, keep_bits=True, nco_hz=nco_hz, stream_freq_tag=tags, n_channels=C)
    else:
        C = 2
        offs = [14000.0, -14000.0] * 3
        mk = lambda: _Keep(S, MAX_BLOCK, keep_bits=True)
    u8, want = _scenario(17, offs)
    x = np.stack([_as_fmt(r, fmt) for r in u8])
    blocks, at = _blocks(9)
    msgs = _check_restart(mk, x, blocks, at, want, C, [s % C for s in range(S)])
    if nco:
        assert sorted((m[0], m[1]) for m in msgs) == sorted((s, int(tags[s][s % C])) for s in range(S))


# ---- 2. restart, long-tap path -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tc", ["0", None], ids=["cuda_core", "tensor_core"])
def test_restart_long_taps(monkeypatch, tc):
    if tc is None:
        monkeypatch.delenv("NVX_LONG_TC", raising=False)
    else:
        monkeypatch.setenv("NVX_LONG_TC", tc)
    taps = designs()
    S = len(STARTS)
    u8, want = _scenario(29, [14000.0, -14000.0] * 3)
    x = np.stack([_as_fmt(r, "s16") for r in u8])
    blocks, at = _blocks(10)
    _check_restart(lambda: _Keep(S, MAX_BLOCK, keep_bits=True, taps=taps), x, blocks, at, want, 2, [s % 2 for s in range(S)])


# ---- 3. move one stream into a running engine ----------------------------------------------------------------------------
def test_move_a_stream_into_a_running_engine():
    S = 3
    nco_a = np.array([[14000.0, -14000.0], [10000.5, -12000.0], [-3000.5, 6000.0]])
    nco_b = np.array([[12000.0, -9000.5], [14000.0, -14000.0], [5000.0, -5000.0]])
    tags_a, tags_b = np.array([[1, 2], [3, 4], [5, 6]]), np.array([[11, 12], [13, 14], [15, 16]])
    rng = np.random.default_rng(51)
    (b2, bbbb2), (b0, _), (b1, _) = (_bulletin(rng, f, t) for f, t in ((6000.0, CUT / FS - 5.0), (14000.0, 1.0), (-14000.0, 2.0)))
    xa = np.stack([_capture_u8([b0], SECONDS, 1), _capture_u8([], SECONDS, 2), _capture_u8([b2], SECONDS, 3)])
    xb = np.stack([_capture_u8([], SECONDS, 4), _capture_u8([b0], SECONDS, 5), _capture_u8([b1], SECONDS, 6)])
    blocks, at = _blocks(11)
    mk_a = lambda: _Keep(S, MAX_BLOCK, keep_bits=True, nco_hz=nco_a, stream_freq_tag=tags_a)
    mk_b = lambda: _Keep(S, MAX_BLOCK, keep_bits=True, nco_hz=nco_b, stream_freq_tag=tags_b, first_stream_id=100)

    # B's stream 0 takes A's stream 2's radio from the save on
    xb_moved = xb.copy()
    xb_moved[0, CUT:] = xa[2, CUT:]
    a, b = mk_a(), mk_b()
    rec_a, rec_b, pos = [], [], 0
    msgs_a, msgs_b = [], []
    for i, n in enumerate(blocks):
        if i == at:
            msgs_a += a.poll_messages()
            msgs_b += b.poll_messages()
            b.load_streams([0], a.save_streams([2]))
        a.push_host(np.ascontiguousarray(xa[:, pos:pos + n]))
        b.push_host(np.ascontiguousarray(xb_moved[:, pos:pos + n]))
        pos += n
        rec_a.append(_snap(a))
        rec_b.append(_snap(b))
    msgs_a += a.poll_messages()
    msgs_b += b.poll_messages()
    a.close()
    b.close()

    ref_a = mk_a()
    base_a, _, base_msgs_a = _run(ref_a, xa, blocks)
    ref_a.close()
    ref_b = mk_b()
    base_b, _, base_msgs_b = _run(ref_b, xb, blocks)
    ref_b.close()
    for s in range(S):                        # saving is read-only: A runs on exactly as R
        _assert_equal_rows(rec_a, s, base_a, s, 2, where=("A", s))
    assert msgs_a == base_msgs_a
    _assert_equal_rows(rec_b[at:], 0, rec_a[at:], 2, 2, where="moved")
    for s in (1, 2):
        _assert_equal_rows(rec_b, s, base_b, s, 2, where=("B", s))
    assert [m for m in msgs_b if m[0] != 100] == [m for m in base_msgs_b if m[0] != 100]
    moved = [m for m in msgs_b if m[0] == 100]
    assert moved == [(100, m[1], m[2], m[3]) for m in msgs_a if m[0] == 2] and [(m[1], m[2]) for m in moved] == [(6, bbbb2)], moved


def _snap(eng):
    rec = {"y3": eng.read_y3().copy(), "ev": {}, "bits": {}}
    for s in range(eng.S):
        for c in range(eng.C):
            rec["ev"][s, c] = eng.read_events(s, c)
            rec["bits"][s, c] = eng.read_bits(s, c)
    return rec


# ---- 4. rejected loads leave the destination untouched -------------------------------------------------------------------
def test_rejected_loads_change_nothing():
    S, C, n = 3, 2, 600 * BLK
    nco = np.array([[14000.0, -14000.0], [10000.5, -12000.0], [-3000.5, 6000.0]])
    rng = np.random.default_rng(61)
    b, _ = _bulletin(rng, 10000.5, 0.5)
    x = np.stack([_capture_u8([], 12.0, 7), _capture_u8([b], 12.0, 8), _capture_u8([], 12.0, 9)]).astype(np.float32) - 128
    blocks = [n] * (x.shape[1] // n)
    mk = lambda **kw: _Keep(S, MAX_BLOCK, keep_bits=True, **{"nco_hz": nco, **kw})

    def saved(eng, fmt=np.float32, blocks_=(n,), streams=(1,)):
        for k in blocks_:
            eng.push_host(np.zeros((eng.S, k, 2), fmt) + (128 if fmt == np.uint8 else 0))
        st = eng.save_streams(list(streams))
        eng.close()
        return st

    good = saved(mk())
    taps = [np.asarray(t) * 1.001 for t in engine_ref_taps()]
    bad = {
        "position": (saved(mk(), blocks_=(n + BLK,)), [1], "modulo"),
        "taps": (saved(mk(taps=taps)), [1], "tap set"),
        "n_channels": (saved(_Keep(S, MAX_BLOCK, nco_hz=np.tile([9000.0, 0.0, -9000.0], (S, 1)), n_channels=3)), [1], "channels"),
        "table": (saved(_Keep(S, MAX_BLOCK)), [1], "NCO"),
        "format": (saved(mk(), fmt=np.int16), [1], "format"),
        "count": (good, [0, 1], "holds"),
        "index": (good, [3], "outside"),
        "duplicate": (saved(mk(), streams=(0, 1)), [1, 1], "twice"),
        "corrupt": (good[:-40] + bytes([good[-40] ^ 4]) + good[-39:], [1], "checksum"),
        "truncated": (good[:-1], [1], "bytes"),
    }
    dest = mk()
    got = []
    for i, k in enumerate(blocks):
        dest.push_host(np.ascontiguousarray(x[:, i * k:(i + 1) * k]))
        got.append(_snap(dest))
        if i == 0:
            for name, (state, streams, words) in bad.items():
                with pytest.raises(engine.NvxError, match=words):
                    dest.load_streams(streams, state)
            # too small a buffer: NVX_ERR_OVERFLOW and the size needed
            L, size = dest.L, engine.C.c_size_t()
            lst = (engine.C.c_int * 1)(1)
            assert L.nvx_engine_save_streams(dest._h, lst, 1, None, 0, engine.C.byref(size)) == 0
            need = size.value
            buf = engine.C.create_string_buffer(need)
            assert L.nvx_engine_save_streams(dest._h, lst, 1, buf, need - 1, engine.C.byref(size)) == -4 and size.value == need
    msgs = dest.poll_messages()
    dest.close()
    ref = mk()
    base, _, base_msgs = _run(ref, x, blocks)
    ref.close()
    for s in range(S):
        _assert_equal_rows(got, s, base, s, C, where=("dest", s))
    assert msgs == base_msgs and len(msgs) == 1


def engine_ref_taps():
    from scipy import signal
    return (signal.firwin(37, 20000, fs=252000), signal.firwin(47, 2000, fs=63000), signal.firwin(71, 250, fs=9000))


# ---- 5. ordering with resets ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ["load_then_reset", "reset_then_load"])
def test_load_and_reset_before_one_push(order):
    S = 2
    u8, _ = _scenario(73, [14000.0, -14000.0] * 3)
    x = np.stack([_as_fmt(r, "s16") for r in u8[:S]])
    blocks, at = _blocks(12)
    mk = lambda: _Keep(S, MAX_BLOCK, keep_bits=True)
    src = mk()
    _run(src, x[::-1].copy(), blocks[:at])
    state = src.save_streams([0])
    src.close()

    def run(action):
        eng = mk()
        recs, before, after = _run(eng, x, blocks, at=at, action=action)
        eng.close()
        return recs, before + after

    def both(e):
        if order == "load_then_reset":
            e.load_streams([1], state)
            e.reset_streams([1])
        else:
            e.reset_streams([1])
            e.load_streams([1], state)

    got, msgs = run(both)
    want, want_msgs = run((lambda e: e.reset_streams([1])) if order == "load_then_reset" else (lambda e: e.load_streams([1], state)))
    for s in range(S):
        _assert_equal_rows(got, s, want, s, 2, where=(order, s))
    assert msgs == want_msgs

"""Every FIR kernel path with asymmetric tap sets whose outermost taps carry weight.

The reference taps and the firwin designs of the other GPU tests are symmetric, and their outermost taps are 1e-5 of the centre
tap or less: a kernel that reverses a stage's taps computes exactly the same samples, and one that drops its oldest taps stays
under the 1e-5 bar.  The oldest taps are also where the index arithmetic is most fragile: the MMA trimming and the padded
windows of the tensor-core kernels (fir_long_tc.cu), the zero padding of the fused kernel's tap classes (fir_cascade.cu), the
J padding of the CUDA-core kernel (fir_long.cu) and the carried history, which only the oldest taps reach into.  Three tap
families, each at the tap counts where those paths change:

  rand      i.i.d. normal taps scaled to sum |h| = 1: every tap weighs about 1 / T, nothing is symmetric, and a missing,
            duplicated, reversed or shifted tap moves y3 by about 1 / sqrt(T) of its peak.  y3 of every stream is compared with
            the float64 statement of the cascade (tests/test_fir_convention.py pins the oracle to the same statement) at the
            pair-peak bar of tests/parity.py (1e-5).
  impulse   a single 1.0 at tap j of one stage, the other stages also single taps: the cascade selects one input sample per
            output and rotates it by the NCO phasor.  Unit taps and integer samples are exact in FP32 and in the 3xTF32 split,
            so the input sample each output came from is read back from its magnitude (input n of stream s has magnitude
            ((n + 1000 s) mod 32000) + 1) and must be the one the convention names.
  edge      a firwin low-pass whose outermost 4 taps at each end are +-0.25 max with unequal signs: still a receiver, so bits,
            events and messages must equal the restated oracle's with the same taps.

Every case pushes three blocks of unequal length (2800 x 7, 11, 9 samples), so every path also runs on carried history.
The convention: h[0] weighs the newest sample, y[k] = sum_i h[i] x[D (k + 1) - 1 - i]."""
import concurrent.futures as cf
import os

import numpy as np
import pytest
from scipy import signal

import oracle_lib as ol
import parity
from navtex_b200 import engine, synth

pytestmark = pytest.mark.gpu

D1, D2, D3 = 4, 7, 10
BLOCKS = (2800 * 7, 2800 * 11, 2800 * 9)
N_IN = sum(BLOCKS)
CHUNK = {D1: 32, D2: 28}                  # samples per tensor-core chunk (fir_long_tc.cu chunk_samples)
POOL = min(16, os.cpu_count() or 1)


# ---- the float64 statement of the cascade -----------------------------------------------------------------------------------
def decimating_fir(x, h, D):
    """x: [R, n] complex128 -> y[R, k] = sum_i h[i] x[D (k + 1) - 1 - i], x zero before index 0."""
    full = signal.oaconvolve(x, np.asarray(h, dtype=np.float64)[None, :], axes=1)
    n = x.shape[1]
    return full[:, D - 1: D * (n // D): D]


def phasor(k, f):
    return np.exp(-2j * np.pi * np.mod(np.asarray(k, dtype=np.float64) * f, 63000.0) / 63000.0)


def cascade(x, taps, nco):
    """x: [S, n] complex128, nco: [S, C] Hz -> y3 [S, C, n // 280]."""
    y1 = decimating_fir(x, taps[0], D1)
    k = np.arange(y1.shape[1])
    out = []
    for c in range(nco.shape[1]):
        z = y1 * phasor(k[None, :], nco[:, c:c + 1])
        out.append(decimating_fir(decimating_fir(z, taps[1], D2), taps[2], D3))
    return np.stack(out, axis=1)


# ---- tap families -----------------------------------------------------------------------------------------------------------
def rand_taps(lengths, seed):
    rng = np.random.default_rng(seed)
    out = []
    for T in lengths:
        h = rng.normal(size=T)
        out.append(h / np.abs(h).sum())
    return tuple(out)


def impulse(T, j):
    h = np.zeros(T)
    h[j] = 1.0
    return h


def edge_taps(lengths):
    h1 = signal.firwin(lengths[0], 20000, window=("kaiser", 8.0), fs=252000)
    h2 = signal.firwin(lengths[1], 2000, window=("kaiser", 8.0), fs=63000)
    h3 = signal.firwin(lengths[2], 250, window=("kaiser", 7.0), fs=9000)
    out = []
    for h in (h1, h2, h3):
        h = h.copy()
        m = np.abs(h).max()
        h[:4] = 0.25 * m * np.array([1.0, -1.0, -1.0, -1.0])
        h[-4:] = 0.25 * m * np.array([1.0, 1.0, -1.0, 1.0])
        out.append(h)
    return tuple(out)


def row_offsets(S, C, seed):
    """[S, C] distinct offsets on the 0.5 Hz grid inside +-31 499.5 Hz (the largest accepted)."""
    rng = np.random.default_rng(seed)
    return rng.choice(np.arange(-62999, 63000), size=S * C, replace=False).reshape(S, C) / 2.0


def noise_input(S, seed, sigma, lim):
    rng = np.random.default_rng(seed)
    return np.clip(np.rint(rng.normal(0.0, sigma, size=(S, N_IN, 2))), -lim - 1, lim).astype(np.int16)


# ---- running the engine -----------------------------------------------------------------------------------------------------
def run(x, taps, nco=None, C=2, fmt="s16"):
    """x: [S, N_IN, 2] int16 pushed in BLOCKS as fmt; returns (y3 [S, C, N_IN / 280] complex64, stats)."""
    S = x.shape[0]
    eng = engine.Engine(S, max(BLOCKS), taps=taps, nco_hz=nco, n_channels=C)
    ys, a = [], 0
    for b in BLOCKS:
        blk = x[:, a:a + b]
        a += b
        if fmt == "f32":
            blk = blk.astype(np.float32)
        elif fmt == "u8":
            blk = (blk.astype(np.int32) + 128).astype(np.uint8)
        eng.push_host(np.ascontiguousarray(blk))
        ys.append(eng.read_y3())
    assert eng.L.nvx_engine_sync(eng._h) == 0, eng.L.nvx_last_error().decode()
    st = eng.stats()
    eng.close()
    return np.concatenate(ys, axis=2), st


def reference_offsets(S):
    return np.tile([14000.0, -14000.0], (S, 1))


def check_rand(where, y3, x, taps, nco):
    """Every stream's y3 against the float64 cascade: pair-peak error <= 1e-5 (tests/parity.py); records the worst stream."""
    xc = x[..., 0].astype(np.float64) + 1j * x[..., 1].astype(np.float64)
    want = cascade(xc, taps, nco)
    assert want.shape == y3.shape, (where, want.shape, y3.shape)
    err = np.abs(y3.astype(np.complex128) - want).max(axis=(1, 2)) / np.maximum(np.abs(want).max(axis=(1, 2)), 1e-30)
    s = int(np.argmax(err))
    cmp = {"y3_rel_pair_peak": float(err[s]), "y3_rel_own_rms": {}, "disc_rel": {}, "bit_len_diff": {}}
    parity.record("taps rand %s (worst of %d streams: %d)" % (where, len(err), s), cmp, set())
    parity.assert_stream(cmp, (), where="%s stream %d" % (where, s))
    return float(err[s])


# ---- rand: the fused kernel ------------------------------------------------------------------------------------------------
# class 0 (up to 37 / 47 / 71 taps): the reference lengths, zero-padded shorter sets, single taps, T = D and T = D + 1
CLASS0 = [(37, 47, 71), (33, 45, 69), (1, 1, 1), (4, 7, 10), (5, 8, 11)]


@pytest.mark.parametrize("C", [1, 3, 5])
@pytest.mark.parametrize("lengths", CLASS0, ids=["%d-%d-%d" % t for t in CLASS0])
def test_rand_fused_class0(lengths, C):
    """33 streams (a full 32-stream group + 1), per-row offsets; 8-bit, int16 and float input bit-identical.  Five channels
    take a second pass over the input (3 + 2)."""
    S = 33
    taps = rand_taps(lengths, seed=sum(lengths) + C)
    nco = row_offsets(S, C, seed=10 * sum(lengths) + C)
    x = noise_input(S, seed=sum(lengths) + 100 * C, sigma=40.0, lim=127)
    y3, st = run(x, taps, nco, C, "s16")
    for fmt in ("f32", "u8"):
        other, _ = run(x, taps, nco, C, fmt)
        assert np.array_equal(y3.view(np.uint64), other.view(np.uint64)), fmt
    assert st.aux_launches == len(BLOCKS) * (2 if C > 4 else 1)
    check_rand("fused class 0 %s C=%d" % (lengths, C), y3, x, taps, nco)


@pytest.mark.parametrize("lengths", [(37, 47, 71), (4, 7, 10)])
def test_rand_fused_class0_reference_offsets(lengths):
    """The reference offsets (+-14 kHz through the 9-entry table kernel) with replacement taps."""
    S = 33
    taps = rand_taps(lengths, seed=7 + sum(lengths))
    x = noise_input(S, seed=8, sigma=3000.0, lim=32767)
    y3, _ = run(x, taps)
    y3f, _ = run(x, taps, fmt="f32")
    assert np.array_equal(y3.view(np.uint64), y3f.view(np.uint64))
    check_rand("fused class 0 %s reference offsets" % (lengths,), y3, x, taps, reference_offsets(S))


# class 1 (up to 61 / 75 / 111 taps): just past class 0, the class lengths, and a set only one stage of which needs class 1
CLASS1 = [(38, 48, 72), (61, 75, 111), (37, 75, 72)]


@pytest.mark.parametrize("per_stream", [False, True])
@pytest.mark.parametrize("lengths", CLASS1, ids=["%d-%d-%d" % t for t in CLASS1])
def test_rand_fused_class1(lengths, per_stream):
    S = 33
    taps = rand_taps(lengths, seed=sum(lengths))
    nco = row_offsets(S, 2, seed=sum(lengths)) if per_stream else None
    x = noise_input(S, seed=sum(lengths) + 1, sigma=3000.0, lim=32767)
    y3, _ = run(x, taps, nco)
    y3f, _ = run(x, taps, nco, fmt="f32")
    assert np.array_equal(y3.view(np.uint64), y3f.view(np.uint64))
    check_rand("fused class 1 %s %s" % (lengths, "per-stream offsets" if per_stream else "reference offsets"), y3, x, taps,
               nco if per_stream else reference_offsets(S))


# ---- rand: the long-tap path -----------------------------------------------------------------------------------------------
# Stage 1 (D = 4): streaming tensor-core kernel up to 516 taps (two live tiles up to 260, three from 261), tile at a time with
# N = 128 at 517 .. 548 and N = 64 from 549.  Stage 2 (D = 7): streaming up to 903, tile at a time up to 959, CUDA-core kernel
# from 960 (a counted fallback).  Stage 3 (D = 10) always on the CUDA-core kernel, J = 8 ceil(ceil(T / 10) / 8): 112, 160 / 161
# and 1024 sit at the boundaries of the J padding.
LONG = [(1, 1, 112), (4, 7, 160), (5, 8, 161), (32, 28, 1024), (33, 29, 112), (62, 255, 160), (255, 903, 112), (256, 904, 161),
        (260, 959, 112), (261, 960, 112), (383, 1024, 160), (516, 255, 112), (517, 7, 161), (548, 28, 112), (549, 29, 1024),
        (1000, 903, 112), (1024, 904, 160)]
# With random taps the 3xTF32 rounding error grows about linearly with the tap count a tensor-core stage runs, and a stage 2 of
# 903 .. 959 taps on the tensor cores goes past the 1e-5 pair-peak bar.  Measured on one B200 (1000 W power limit), worst
# stream of 130: stage 2 alone at 903 taps 9.6e-6 (stage 1 on the CUDA cores), stage 1 alone at 1000 / 1024 taps 9.2e-6 /
# 9.9e-6; both stages on the tensor cores 1.1e-5 .. 1.2e-5 at 255 .. 260 + 903 .. 959 taps and 1.6e-5 .. 1.7e-5 at 1000 .. 1024
# + 903 .. 904.  Firwin low-pass designs at the same counts stay under the bar (tests/test_gpu_longtaps.py).  Strict: a more
# accurate tensor-core path makes these pass and must then drop the mark.  The index arithmetic at these counts is checked
# exactly by test_impulse_taps (540 / 904 and 1000 / 959 taps, streaming 516 / 900).
TF32_PAST_BAR = {(255, 903, 112), (256, 904, 161), (260, 959, 112), (1000, 903, 112), (1024, 904, 160)}


def long_case(monkeypatch, lengths, tc, per_stream, mix=None, S=130):
    """S = 130 streams: stage 1 sees two 128-row tiles (the last one ragged), stage 2 260 rows (three, the last ragged)."""
    for name, val in (("NVX_LONG_TC", tc), ("NVX_LONG_MIX", mix)):
        if val is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, val)
    taps = rand_taps(lengths, seed=sum(lengths))
    nco = row_offsets(S, 2, seed=3 * sum(lengths)) if per_stream else None
    x = noise_input(S, seed=sum(lengths) + 2, sigma=3000.0, lim=32767)
    y3, st = run(x, taps, nco, fmt="f32" if per_stream else "s16")
    mask = 3 if tc is None else int(tc)
    want_fallbacks = bool(mask & 2) and lengths[1] >= 960
    assert (st.long_tc_fallbacks > 0) == want_fallbacks, (lengths, tc, st.long_tc_fallbacks)
    return check_rand("long %s NVX_LONG_TC=%s%s %s" % (lengths, tc, "" if mix is None else " NVX_LONG_MIX=" + mix,
                                                       "per-stream offsets" if per_stream else "reference offsets"),
                      y3, x, taps, nco if per_stream else reference_offsets(S))


@pytest.mark.parametrize("per_stream", [False, True], ids=["ref", "nco"])
@pytest.mark.parametrize("lengths", [pytest.param(t, marks=pytest.mark.xfail(strict=True, reason="3xTF32 rounding past 1e-5 of the peak"))
                                     if t in TF32_PAST_BAR else t for t in LONG], ids=["%d-%d-%d" % t for t in LONG])
def test_rand_long_tensor_core(monkeypatch, lengths, per_stream):
    """The default NVX_LONG_TC=3.  Reference offsets: stage 2 mixes while it loads (streaming kernel); per-stream offsets (float
    input): the stage-1 epilogue mixes."""
    long_case(monkeypatch, lengths, None, per_stream)


@pytest.mark.parametrize("lengths", [(62, 255, 160), (32, 28, 1024)])
def test_rand_long_mix_in_stage1(monkeypatch, lengths):
    long_case(monkeypatch, lengths, None, False, mix="stage1")


# T = 8 D m and 8 D m + 1 on the CUDA-core kernel: J lands exactly on a multiple of kLongR, or one tap block beyond it
CUDA_CORE = [(256, 448, 160), (257, 449, 161), (62, 255, 160), (516, 255, 112), (1000, 903, 112), (1024, 1024, 1024)]


@pytest.mark.parametrize("tc", ["0", "1", "2"])
@pytest.mark.parametrize("lengths", CUDA_CORE, ids=["%d-%d-%d" % t for t in CUDA_CORE])
def test_rand_long_cuda_core(monkeypatch, lengths, tc):
    """NVX_LONG_TC=0: both stages on the CUDA-core kernel; 1: stage 1 on the tensor cores; 2: stage 2 on them."""
    long_case(monkeypatch, lengths, tc, lengths[0] % 2 == 1)


# ---- impulse: which input sample each output came from ---------------------------------------------------------------------
M_ENC = 32000


def impulse_input(S):
    n = np.arange(N_IN)[None, :] + 1000 * np.arange(S)[:, None]
    x = np.zeros((S, N_IN, 2), dtype=np.int16)
    x[..., 0] = (n % M_ENC) + 1
    return x


def check_impulse(where, y3, js, nco, S):
    """y3 of an all-impulse tap set (taps js) against the selected and rotated input sample."""
    P = y3.shape[2]
    k3 = np.arange(P)
    k2 = D3 * (k3 + 1) - 1 - js[2]
    k1 = D2 * (k2 + 1) - 1 - js[1]
    src = D1 * (k1 + 1) - 1 - js[0]
    live = (k2 >= 0) & (k1 >= 0) & (src >= 0)
    worst = 0.0
    for s in range(S):
        mag = np.where(live, ((np.maximum(src, 0) + 1000 * s) % M_ENC) + 1, 0).astype(np.float64)
        for c in range(y3.shape[1]):
            want = mag * np.where(live, phasor(np.maximum(k1, 0), nco[s, c]), 0)
            got = y3[s, c].astype(np.complex128)
            code = np.rint(np.abs(got)).astype(np.int64)
            dec = np.where(code == 0, -1, (code - 1 - 1000 * s) % M_ENC)
            exp = np.where(live, src % M_ENC, -1)
            bad = np.nonzero(dec != exp)[0]
            assert bad.size == 0, ("%s stream %d channel %d: y3[%d] came from input %d, expected %d (%d outputs wrong)"
                                   % (where, s, c, bad[0], dec[bad[0]], exp[bad[0]], bad.size))
            worst = max(worst, float(np.abs(got - want).max()) / M_ENC)
    cmp = {"y3_rel_pair_peak": worst, "y3_rel_own_rms": {}, "disc_rel": {}, "bit_len_diff": {}}
    parity.record("taps impulse %s" % where, cmp, set())
    parity.assert_stream(cmp, (), where=where)


def boundary_taps(T, Tp, step, new_end=False):
    """j in {0, 1, T - 2, T - 1} and both sides of the first two and last two window boundaries `step` apart, counted from
    the old end of the padded window Tp (tensor-core chunks) or from the new end (CUDA-core tap blocks)."""
    if new_end:
        cuts = [step * m for m in range(1, (T - 1) // step + 1)]
    else:
        cuts = [Tp - step * m for m in range(1, Tp // step + 1)]
    cuts = cuts[:2] + cuts[-2:]
    js = {0, 1, T - 2, T - 1} | {c for c in cuts} | {c - 1 for c in cuts}
    return sorted(j for j in js if 0 <= j < T)


def stage_kernels(lengths, tc):
    """(padded window, boundary step, counted from the new end) of each stage on the kernel the engine picks for it."""
    mask = 3 if tc is None else int(tc)
    out = []
    for k, (D, T) in enumerate(zip((D1, D2, D3), lengths)):
        on_tc = k < 2 and bool(mask & (1 << k)) and not (k == 1 and T >= 960)
        if on_tc:
            g, _, _ = engine.long_tc_band(D, np.ones(T))
            out.append((g["taps_padded"], CHUNK[D], False))
        else:
            out.append((T, 8 * D, True))                 # kLongR outputs per thread: tap blocks of 8 D inputs
    return out


IMPULSE = [("fused class 0", (37, 47, 71), None), ("fused class 1", (61, 75, 111), None),
           ("streaming", (255, 259, 112), None), ("streaming three tiles", (516, 900, 112), None),
           ("tile N=128 / tile", (540, 904, 112), None), ("tile N=64 / tile", (1000, 959, 160), None),
           ("cuda core", (257, 449, 161), "0"), ("stage-2 fallback", (1024, 1024, 1024), None)]


@pytest.mark.parametrize("stage", [0, 1, 2])
@pytest.mark.parametrize("name,lengths,tc", IMPULSE, ids=[c[0].replace(" ", "_") for c in IMPULSE])
def test_impulse_taps(monkeypatch, name, lengths, tc, stage):
    """Sweep the single tap of one stage over its ends and window boundaries, the other stages at tap 0 (and once at their
    last tap).  Fused cases: 33 streams with per-row offsets; long-tap cases: 3 streams, reference offsets (mix on load)."""
    if tc is None:
        monkeypatch.delenv("NVX_LONG_TC", raising=False)
    else:
        monkeypatch.setenv("NVX_LONG_TC", tc)
    monkeypatch.delenv("NVX_LONG_MIX", raising=False)
    fused = name.startswith("fused")
    S = 33 if fused else 3
    nco = row_offsets(S, 2, seed=sum(lengths)) if fused else None
    x = impulse_input(S)
    if fused:
        js_of = boundary_taps(lengths[stage], lengths[stage], 1 << 30)
    else:
        Tp, step, new_end = stage_kernels(lengths, tc)[stage]
        js_of = boundary_taps(lengths[stage], Tp, step, new_end)
    others = [(0, 0, 0), tuple(T - 1 for T in lengths)]
    for base in others:
        for j in js_of:
            js = list(base)
            js[stage] = j
            taps = tuple(impulse(T, jj) for T, jj in zip(lengths, js))
            y3, st = run(x, taps, nco)
            assert (st.long_tc_fallbacks > 0) == (not fused and tc is None and lengths[1] >= 960)
            check_impulse("%s %s stage %d taps %s" % (name, lengths, stage + 1, tuple(js)), y3, js,
                          nco if fused else reference_offsets(S), S)


# ---- edge: bits, events and messages ---------------------------------------------------------------------------------------
EDGE = [("fused class 0", (37, 47, 71)), ("fused class 1", (61, 75, 111)), ("streaming", (255, 259, 112)),
        ("tile at a time", (549, 259, 160))]


@pytest.mark.parametrize("name,lengths", EDGE, ids=[c[0].replace(" ", "_") for c in EDGE])
def test_edge_taps_decode_like_the_oracle(name, lengths):
    """Two streams, a bulletin on channel 518 / 490: y3 within the bar, bits, events and messages equal to the oracle's."""
    taps = edge_taps(lengths)
    seconds, blk = 12.0, 126000                                  # 0.5 s blocks
    n = int(seconds * 252000)
    rng = np.random.default_rng(sum(lengths))
    iqs, want = [], []
    for s in range(2):
        while True:                                              # (redrawn when the bulletin does not fit the capture)
            text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=3)
            if len(synth.message_bits(text, n_phasing=18, n_tail=5)) <= (seconds - 0.6) * 100:
                break
        em = synth.Emission(text, 14000.0 if s == 0 else -14000.0, start_s=0.3, n_phasing=18, n_tail=5)
        iqs.append(synth.quantise_s16(synth.fsk_iq([em], seconds, snr_db=0.0, seed=700 + s))[: 2 * n])
        want.append((518 if s == 0 else 490, bbbb, text))
    x = np.stack([iq.reshape(-1, 2) for iq in iqs])
    eng = engine.Engine(2, blk, taps=taps, keep_bits=True)
    y3 = []
    bits = {(s, c): b"" for s in range(2) for c in range(2)}
    disc = {(s, c): [] for s in range(2) for c in range(2)}
    events = dict.fromkeys(bits, b"")
    msgs = []
    for a in range(0, n, blk):
        eng.push_host(np.ascontiguousarray(x[:, a:a + blk]))
        assert eng.L.nvx_engine_sync(eng._h) == 0
        y3.append(eng.read_y3())
        for s in range(2):
            for c in range(2):
                b, d = eng.read_bits(s, c)
                bits[(s, c)] += b
                disc[(s, c)].append(d)
                events[(s, c)] += eng.read_events(s, c)
        msgs += eng.poll_messages()
    st = eng.stats()
    eng.close()
    assert st.long_tc_fallbacks == 0
    y3 = np.concatenate(y3, axis=2)
    with cf.ThreadPoolExecutor(POOL) as ex:
        orc = list(ex.map(lambda iq: ol.run_oracle(iq, h1=taps[0], h2=taps[1], h3=taps[2]), iqs))
    for s, o in enumerate(orc):
        occ = ol.CHANNELS[s]
        where = "taps edge %s %s stream %d" % (name, lengths, s)
        cmp = parity.compare_stream(y3[s], {c: bits[(s, c)] for c in range(2)}, {c: np.concatenate(disc[(s, c)]) for c in range(2)},
                                    o, {occ})
        parity.record(where, cmp, {occ})
        parity.assert_stream(cmp, {occ}, where=where)
        assert events[(s, s)] == o.events[occ], where
        assert o.messages == [want[s]], (where, o.messages)
        assert [m[1:] for m in msgs if m[0] == s] == [want[s]], where

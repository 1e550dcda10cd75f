"""Every (stream, channel) row with its own NCO offset, freq tag and signal, at stream counts where the row bookkeeping of the
kernels can go wrong: several 32-stream warp groups of the fused cascade, several 128-row tiles of the tensor-core stage 1, and
the engine's limits of 32 767 streams and 65 535 channel rows.

Each output row is one (stream, channel) pair and finds its NCO offset, freq tag, y3 row, demod row and message slot through
index arithmetic.  Here no two rows share an offset or a tag, and every stream carries its own bulletin (or FSK bits) on its own
channel, so a row that reads its neighbour's parameters or input shows up as a wrong sample, bit or message.  The bar is
tests/parity.py's: 900 Hz samples within 1e-5 of the stream's peak over all its channels and of an occupied channel's own RMS,
decisions / events / messages exact on the occupied channel, the same number of decisions on the empty ones -- against the
float64 restated oracle run with that row's own offsets, tags and taps.

The captures are synthesised on the device (synth.cu: counter-based, any block of any stream can be regenerated) at 8-bit scale,
30 LSB at -3 dB full-band SNR, rounded and clamped to [-128, 127]: the same values push as 8-bit pairs, int16 and float32."""
import concurrent.futures as cf
import os

import numpy as np
import pytest

import oracle_lib as ol
import parity
from navtex_b200 import engine, synth
from test_gpu_longtaps import designs
from test_gpu_u8 import CLASS0, MEDIUM

pytestmark = pytest.mark.gpu

FS = engine.FS
AMP = 30.0                                            # 8-bit scale
SIGMA = AMP / np.sqrt(2.0) * 10.0 ** (3.0 / 20.0)     # -3 dB full-band SNR (per-component sigma, as synth.fsk_iq)
# offsets every engine of this file gives to its first streams (one per stream, in the channel whose band holds it): the
# reference table's pair through the general kernel, DC and its neighbours, and the largest accepted offset (no emission there)
EDGES = (14000.0, -14000.0, 0.0, 0.5, -0.5, 31499.5, -31499.5)
TAPS = {"reference": None, "class0": CLASS0, "medium": MEDIUM}
# the long-tap designs (test_gpu_longtaps.designs: stage 1 cut at 20 kHz, -43 dB at 22 kHz with 255 taps) draw their offsets
# inside +-20 kHz: a receiver tunes its channels inside the band its stage 1 passes
LONG_BAND = 20000.0
# a noise-only channel decides at an arg max near-tie now and then; with thousands of them per run (3 132 in the long-tap cases)
# one such slip can leave it one decision short (seen on a B200: 1 of 3 132, pick margin 2e-4, its samples 1.1e-5 of own RMS).
# Its samples stay under the pair-peak bar; a slip after a pick within 1e-3 is reported, not failed (tests/parity.py).
NEAR_TIE = 1e-3
POOL = min(32, os.cpu_count() or 1)                   # oracle runs in threads: ctypes releases the GIL


def row_offsets(S, C, seed, band=25000.0):
    """[S, C] offsets in Hz, distinct over all rows, on the 0.5 Hz grid inside +-band (about half of them odd multiples of
    0.5 Hz).  Channel c draws from the c-th of C equal sub-bands, 1.5 kHz in from either edge, so the channels of a stream are
    at least 1.5 kHz apart; stream k < 7 then carries EDGES[k] in the channel whose sub-band holds it (clamped to the outer
    ones)."""
    rng = np.random.default_rng(seed)
    half = int(2 * band)                              # half-Hz units from here on
    width, margin = 2 * half // C, 3000
    edges2 = [int(2 * e) for e in EDGES]
    out = np.empty((S, C))
    for c in range(C):
        cand = np.arange(-half + c * width + margin, -half + (c + 1) * width - margin + 1)
        cand = cand[~np.isin(cand, edges2)]
        out[:, c] = rng.choice(cand, size=S, replace=False) / 2.0
    for k, e in enumerate(EDGES[:S]):
        out[k, min(max(int((2 * e + half) // width), 0), C - 1)] = e
    assert len(np.unique(out)) == out.size
    return out


def _reference_h1():
    with open(os.path.join(ol.ROOT, "include", "navtex_taps.h")) as f:
        src = f.read()
    body = src.split("#define NVX_H1_VALUES")[1].split("\n#define")[0]
    return np.array([float.fromhex(t) for t in body.replace("\\", " ").replace(",", " ").split()])


H1_REF = _reference_h1()


def stopband_keys(h1, offsets, occ):
    """Keys of the empty channels whose offset the stage-1 filter h1 attenuates by 60 dB or more: such a channel holds residue
    at the level of FP32 rounding, so its decisions are counted, not required equal (tests/parity.py: `unbounded`)."""
    h1 = H1_REF if h1 is None else np.asarray(h1)
    k = np.arange(len(h1))
    gain = lambda f: abs(np.sum(h1 * np.exp(-2j * np.pi * f * k / FS))) / abs(np.sum(h1))
    return {ol.CHANNEL_KEYS[c] for c, f in enumerate(offsets) if c != occ and gain(f) <= 1e-3}


def row_tags(S, C):
    return 1000 + 8 * np.arange(S)[:, None] + np.arange(C)[None, :]


def occupied_channel(nco, s):
    """Channel s % C carries stream s's signal; a stream whose channel sits at the +-31.5 kHz edge moves it to the next channel
    (with one channel it stays empty: None)."""
    C = nco.shape[1]
    c = s % C
    if abs(nco[s, c]) > 25000.0:
        c = (c + 1) % C if C > 1 else None
    return c


class Content:
    """Per stream: a random bulletin (or random FSK bits) at its occupied row's offset, its own start time, the 8-bit noise."""

    def __init__(self, nco, seconds, seed, bulletins=True, amp=AMP, sigma=SIGMA):
        S = nco.shape[0]
        rng = np.random.default_rng(seed)
        self.occ = [occupied_channel(nco, s) for s in range(S)]
        self.want, self.bits, self.offset, self.start = [], [], [], []
        for s in range(S):
            if bulletins:
                while True:                                          # (redrawn when the bulletin does not fit the capture)
                    text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=3)
                    b = synth.message_bits(text, n_phasing=18, n_tail=5)
                    if len(b) <= (seconds - 0.6) * 100:
                        break
                self.want.append((bbbb, text))
            else:
                b = rng.integers(0, 2, size=int(seconds * 80)).astype(np.uint8)
            room = seconds - 0.3 - len(b) / 100.0
            assert room > 0.15, (s, len(b))
            self.bits.append(b)
            self.start.append(0.05 + rng.uniform(0.0, room - 0.1))
            self.offset.append(nco[s, self.occ[s]] if self.occ[s] is not None else 0.0)
        self.amp = np.where([c is not None for c in self.occ], amp, 0.0)
        self.sigma = np.full(S, sigma)
        self.seed = int(seed)
        self.S = S

    def fill(self, buf, t0, lo=-128, hi=127):
        """buf: device float32 [S, n, 2] <- samples [t0, t0 + n) of every stream, rounded and clamped to [lo, hi]."""
        engine.synth_fill_device(0, buf.data_ptr(), self.S, t0, buf.shape[1], self.bits, self.offset, self.start, self.amp,
                                 self.sigma, self.seed)
        buf.clamp_(lo, hi)


def _sync0(eng):
    """nvx_engine_sync itself, not the binding's wrapper (which lets an event-buffer overflow pass): 0 or the test fails."""
    rc = eng.L.nvx_engine_sync(eng._h)
    assert rc == 0, (rc, eng.L.nvx_last_error().decode())


class Taps:
    """What one engine run produced for the rows it was asked to keep, gathered over every push."""

    def __init__(self, rows, C):
        self.rows, self.C = list(rows), C
        self.y3 = []
        self.bits = {(i, c): b"" for i in range(len(rows)) for c in range(C)}
        self.disc = {(i, c): [] for i in range(len(rows)) for c in range(C)}
        self.events = dict.fromkeys(self.bits, b"")
        self.msgs = []
        self.stats = None

    def collect(self, eng):
        _sync0(eng)
        self.y3.append(eng.read_y3()[self.rows])
        for i, s in enumerate(self.rows):              # read_bits / read_events hold the last block only
            for c in range(self.C):
                b, d = eng.read_bits(s, c)
                self.bits[(i, c)] += b
                self.disc[(i, c)].append(d)
                self.events[(i, c)] += eng.read_events(s, c)
        self.msgs += eng.poll_messages()

    def finish(self, eng):
        _sync0(eng)
        self.stats = eng.stats()
        self.y3 = np.concatenate(self.y3, axis=2)
        self.disc = {k: np.concatenate(v) for k, v in self.disc.items()}


def _oracle_parity(jobs, where):
    """jobs: (row index i in taps, stream s, int16 capture, oracle kwargs, occupied channel or None, Taps).  Runs the oracle of
    every job in a thread pool and applies the parity bar; returns {s: oracle messages}."""
    def one(job):
        i, s, iq, kw, occ, tp = job
        C = tp.C
        keys = ol.CHANNEL_KEYS[:C]
        o = ol.run_oracle(iq, **kw)
        occupied = {keys[occ]} if occ is not None else set()
        cmp = parity.compare_stream(tp.y3[i], {c: tp.bits[(i, c)] for c in range(C)}, {c: tp.disc[(i, c)] for c in range(C)},
                                    o, occupied, channels=keys)
        ev = o.events[keys[occ]] == tp.events[(i, occ)] if occ is not None else True
        return s, cmp, occupied, ev, o.messages, stopband_keys(kw.get("h1"), kw["nco_hz"], occ)

    with cf.ThreadPoolExecutor(POOL) as ex:
        res = list(ex.map(one, jobs))
    for s, cmp, occupied, ev, msgs, stop in res:
        parity.record("%s stream %d" % (where, s), cmp, occupied)
    for s, cmp, occupied, ev, msgs, stop in res:
        parity.assert_stream(cmp, occupied, where="%s stream %d" % (where, s), unbounded=stop, near_tie=NEAR_TIE)
        assert ev, ("%s stream %d: events differ from the oracle's" % (where, s))
    return {r[0]: r[4] for r in res}


def _wanted(content, tags, first=0):
    return sorted((first + s, int(tags[s, c]), *content.want[s]) for s, c in enumerate(content.occ) if c is not None)


# ---- A. the fused cascade: every instantiation the engine reaches, S = 67 (two full 32-stream groups + 3) ---------------------
A_CASES = [("reference", C, True) for C in range(1, 9)] + [("class0", C, True) for C in (1, 2, 7)] + [("medium", 2, True)] + \
          [(t, 2, False) for t in ("reference", "class0", "medium")]


@pytest.mark.parametrize("taps,C,gen", A_CASES, ids=["%s-%dch-%s" % (t, c, "nco" if g else "table") for t, c, g in A_CASES])
def test_fused_cascade_rows(taps, C, gen):
    """67 streams x C channels, 11 s pushed in four blocks as 8-bit pairs, int16 and float32 (bit-identical y3, bits, events and
    messages), every row against the oracle with its own offset and tag.  From five channels on, a second pass over the input
    (5 = 3 + 2, 6 = 3 + 3, 7 = 4 + 3, 8 = 4 + 4) is one more launch per push in aux_launches.  Without offsets (gen False) the
    reference table kernels run: distinct content per stream across the groups, distinct tags per row."""
    import torch

    S, blk, n_blk = 67, 280 * 2475, 4
    n = blk * n_blk                                                    # 11 s
    h = TAPS[taps]
    nco = row_offsets(S, C, 1000 + C) if gen else np.tile([14000.0, -14000.0], (S, 1))
    tags = row_tags(S, C)
    content = Content(nco, n / FS, seed=7000 + 100 * list(TAPS).index(taps) + 10 * C + gen)
    x = torch.empty((S, n, 2), dtype=torch.float32, device="cuda")
    content.fill(x, 0)
    kw = {"taps": h, "stream_freq_tag": tags, "n_channels": C, "keep_bits": True}
    if gen:
        kw["nco_hz"] = nco
    runs = {}
    for name, xv in (("u8", (x + 128).to(torch.uint8)), ("s16", x.to(torch.int16)), ("f32", x)):
        eng = engine.Engine(S, blk, **kw)
        tp = Taps(range(S), C)
        for a in range(0, n, blk):
            d = xv[:, a:a + blk].contiguous()
            torch.cuda.synchronize()
            eng.push_device(d.data_ptr(), blk, s16=name == "s16", u8=name == "u8")
            tp.collect(eng)
            del d
        tp.finish(eng)
        eng.close()
        runs[name] = tp
        del xv
    host = x.to(torch.int16).cpu().numpy()
    del x
    torch.cuda.empty_cache()

    ref = runs["u8"]
    for name in ("s16", "f32"):
        tp = runs[name]
        assert np.array_equal(ref.y3.view(np.uint64), tp.y3.view(np.uint64)), name
        assert ref.bits == tp.bits and ref.events == tp.events and sorted(ref.msgs) == sorted(tp.msgs), name
    for name, tp in runs.items():
        assert tp.stats.aux_launches == n_blk * (2 if C > 4 else 1), (name, tp.stats.aux_launches)

    okw = {"h1": h[0], "h2": h[1], "h3": h[2]} if h is not None else {}
    jobs = [(s, s, host[s].reshape(-1), dict(okw, nco_hz=tuple(nco[s]), freq_tag=tuple(int(t) for t in tags[s])),
             content.occ[s], ref) for s in range(S)]
    omsgs = _oracle_parity(jobs, "%s %d ch %s" % (taps, C, "nco" if gen else "table"))
    want = _wanted(content, tags)
    assert sorted((s, *m) for s, ms in omsgs.items() for m in ms) == want
    assert sorted(ref.msgs) == want
    assert {c for c in content.occ if c is not None} == set(range(C))     # every channel index decodes a bulletin somewhere


# ---- B. the long-tap path: per-stream offsets across tensor-core row blocks, S = 261 ---------------------------------------
@pytest.mark.parametrize("lengths", [(255, 255, 255), (255, 930, 71), (511, 511, 90)])
def test_long_taps_rows(monkeypatch, lengths):
    """261 streams (three 128-row stage-1 tiles, the last one ragged; 522 stage-2 rows): every 32-row epilogue quarter mixes
    rows of distinct offsets.  Random FSK bits at +10 dB on channel s % 2, 3 s in two pushes, with stage 1 / stage 2 on the
    tensor cores (default), both on the CUDA cores (NVX_LONG_TC=0), and each one alone on the tensor cores (1, 2)."""
    import torch

    S, C, blk = 261, 2, 280 * 1350
    n = 2 * blk                                                        # 3 s
    taps = designs(*lengths)
    nco = row_offsets(S, C, 2000 + lengths[1], band=LONG_BAND)
    tags = row_tags(S, C)
    content = Content(nco, n / FS, seed=3000 + lengths[0] + lengths[1], bulletins=False, amp=3000.0,
                      sigma=3000.0 / np.sqrt(2.0) * 10.0 ** (-10.0 / 20.0))
    x = torch.empty((S, n, 2), dtype=torch.float32, device="cuda")
    content.fill(x, 0, -32768, 32767)
    host = x.to(torch.int16).cpu().numpy()
    arms = {}
    for tc in (None, "0", "1", "2"):
        if tc is None:
            monkeypatch.delenv("NVX_LONG_TC", raising=False)
        else:
            monkeypatch.setenv("NVX_LONG_TC", tc)
        eng = engine.Engine(S, blk, taps=taps, nco_hz=nco, stream_freq_tag=tags, keep_bits=True)
        tp = Taps(range(S), C)
        for a in (0, blk):
            d = x[:, a:a + blk].contiguous()
            torch.cuda.synchronize()
            eng.push_device(d.data_ptr(), blk)
            tp.collect(eng)
            del d
        tp.finish(eng)
        eng.close()
        assert tp.stats.long_tc_fallbacks == 0, (tc, tp.stats.long_tc_fallbacks)
        arms[tc] = tp
    del x
    torch.cuda.empty_cache()

    okw = {"h1": taps[0], "h2": taps[1], "h3": taps[2]}
    decided = {}

    def run(s):
        return s, ol.run_oracle(host[s].reshape(-1), nco_hz=tuple(nco[s]), freq_tag=tuple(int(t) for t in tags[s]), **okw)

    keys = ol.CHANNEL_KEYS[:C]
    checks = []
    with cf.ThreadPoolExecutor(POOL) as ex:
        for s, o in ex.map(run, range(S)):
            occ = content.occ[s]
            for tc, tp in arms.items():
                where = "long %s NVX_LONG_TC=%s stream %d" % (lengths, tc, s)
                cmp = parity.compare_stream(tp.y3[s], {c: tp.bits[(s, c)] for c in range(C)},
                                            {c: tp.disc[(s, c)] for c in range(C)}, o, {keys[occ]}, channels=keys)
                parity.record(where, cmp, {keys[occ]})
                checks.append((where, cmp, {keys[occ]}, tp.events[(s, occ)] == o.events[keys[occ]], stopband_keys(taps[0], nco[s], occ)))
            decided[s] = len(o.bits[keys[occ]])
    for where, cmp, occupied, ev, stop in checks:
        parity.assert_stream(cmp, occupied, where=where, unbounded=stop, near_tie=NEAR_TIE)
        assert ev, where
    assert min(decided.values()) > 200                                   # every stream's occupied channel was decided


# ---- C. the engine's limits, a bulletin on every stream -----------------------------------------------------------------
def _limit_rows(S):
    return sorted({0, 31, 32, 63, S // 2, (S - 1) // 32 * 32, S - 1})


def _limit_case(S, C, taps, gen, first_stream_id=0):
    """11 s of S streams synthesised on the device in 0.1 s blocks (float32 pushes), messages of every stream checked, oracle
    parity on the streams of _limit_rows (their input rows copied out of each block before it is pushed)."""
    import torch

    blk, n_blk = 25200, 110
    n = blk * n_blk
    nco = row_offsets(S, C, 4000 + C, band=25000.0 if taps is None else LONG_BAND) if gen else np.tile([14000.0, -14000.0], (S, 1))
    tags = row_tags(S, C)
    content = Content(nco, n / FS, seed=5000 + S + C)
    rows = _limit_rows(S)
    kw = {"taps": taps, "stream_freq_tag": tags, "n_channels": C, "keep_bits": True, "first_stream_id": first_stream_id}
    if gen:
        kw["nco_hz"] = nco
    free0 = torch.cuda.mem_get_info()[0]
    eng = engine.Engine(S, blk, **kw)
    buf = torch.empty((S, blk, 2), dtype=torch.float32, device="cuda")
    idx = torch.tensor(rows, device="cuda")
    host = np.empty((len(rows), n, 2), dtype=np.int16)
    tp = Taps(rows, C)
    used = 0
    for k in range(n_blk):
        content.fill(buf, k * blk)
        host[:, k * blk:(k + 1) * blk] = buf.index_select(0, idx).to(torch.int16).cpu().numpy()
        torch.cuda.synchronize()
        eng.push_device(buf.data_ptr(), blk)
        tp.collect(eng)
        used = max(used, free0 - torch.cuda.mem_get_info()[0])       # engine buffers + the synthesised block
    tp.finish(eng)
    eng.close()
    del buf
    torch.cuda.empty_cache()

    where = "limit S=%d C=%d" % (S, C)
    okw = {"h1": taps[0], "h2": taps[1], "h3": taps[2]} if taps is not None else {}
    jobs = [(i, s, host[i].reshape(-1), dict(okw, nco_hz=tuple(nco[s]), freq_tag=tuple(int(t) for t in tags[s])), content.occ[s], tp)
            for i, s in enumerate(rows)]
    omsgs = _oracle_parity(jobs, where)
    for s in rows:
        assert sorted(omsgs[s]) == sorted(m[1:] for m in _wanted(content, tags) if m[0] == s), (where, s)
    want = _wanted(content, tags, first_stream_id)
    got = sorted(tp.msgs)
    print("%s: %d of %d streams' bulletins checked (%d messages); device memory of the case %.2f GB (float32 block %.2f GB)"
          % (where, len(want), S, len(got), used / 1e9, S * blk * 8 / 1e9))
    assert got == want, (where, len(got), len(want))
    assert len({m[0] for m in got}) == len(want)                       # once each


def test_limit_65535_rows_fused():
    """Exactly 65 535 channel rows: C = 3, S = 21 845, per-row offsets and tags, stream ids from 1 000 000."""
    _limit_case(21845, 3, None, True, first_stream_id=1_000_000)


def test_limit_32767_streams_table():
    """The stream limit on the reference table kernel: S = 32 767, C = 2 (65 534 rows)."""
    _limit_case(32767, 2, None, False)


def test_limit_32767_streams_long_taps():
    """The stream limit on the long-tap path (255 / 255 / 255 taps) with per-stream offsets."""
    _limit_case(32767, 2, designs(255, 255, 255), True)


def test_limit_rejections():
    with pytest.raises(engine.NvxError, match="exceeds 32767"):
        engine.Engine(32768, 2800, n_channels=1, nco_hz=np.zeros((32768, 1)))
    for C, S in ((4, 16384), (8, 8192)):
        with pytest.raises(engine.NvxError, match="65536 exceeds 65535 channel rows"):
            engine.Engine(S, 2800, n_channels=C, nco_hz=np.zeros((S, C)))

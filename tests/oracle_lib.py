"""ctypes bindings for the CPU oracle (oracle/libnavtex_oracle.so) and a runner for the
compiled reference (oracle/_ref/ref_chain).  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "libnavtex_oracle.so")
REF_CHAIN = os.path.join(ORACLE_DIR, "_ref", "ref_chain")
CHANNELS = ("518", "490")
CHANNEL_KEYS = ("518", "490", "ch2", "ch3", "ch4", "ch5", "ch6", "ch7")     # result keys of channels 0 .. 7


def build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "all"], check=True)


class Params(C.Structure):
    _fields_ = [
        ("h1", C.POINTER(C.c_double)), ("n1", C.c_int),
        ("h2", C.POINTER(C.c_double)), ("n2", C.c_int),
        ("h3", C.POINTER(C.c_double)), ("n3", C.c_int),
        ("nco_hz", C.c_double * 8),
        ("nco_period", C.c_int * 8),
        ("freq_tag", C.c_int * 8),
        ("record_taps", C.c_int),
        ("n_channels", C.c_int),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build_oracle()          # every time: make rebuilds a library older than its sources, and leaves a current one alone
        L = C.CDLL(ORACLE_SO)
        L.nvo_new.restype = C.c_void_p
        L.nvo_new.argtypes = [C.POINTER(Params)]
        L.nvo_free.argtypes = [C.c_void_p]
        L.nvo_default_params.argtypes = [C.POINTER(Params)]
        for name, t in (("nvo_push", C.c_double), ("nvo_push_f32", C.c_float), ("nvo_push_s16", C.c_int16)):
            getattr(L, name).argtypes = [C.c_void_p, C.POINTER(t), C.c_size_t]
        L.nvo_push_900.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.c_size_t]
        L.nvo_y1.restype = C.c_size_t
        L.nvo_y1.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_double))]
        for name, t in (("nvo_y2", C.c_double), ("nvo_y3", C.c_double), ("nvo_bits", C.c_char),
                        ("nvo_bitpos", C.c_int32), ("nvo_disc", C.c_float), ("nvo_events", C.c_char)):
            f = getattr(L, name)
            f.restype = C.c_size_t
            f.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.POINTER(t))]
        L.nvo_pick_margins.restype = C.c_size_t
        L.nvo_pick_margins.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.POINTER(C.c_double))]
        L.nvo_n_messages.restype = C.c_size_t
        L.nvo_n_messages.argtypes = [C.c_void_p]
        L.nvo_message.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p)]
        L.nvo_decoder_new.restype = C.c_void_p
        L.nvo_decoder_free.argtypes = [C.c_void_p]
        L.nvo_decoder_sample.restype = C.c_char
        L.nvo_decoder_sample.argtypes = [C.c_void_p, C.c_double, C.c_double, C.POINTER(C.c_float)]
        _lib = L
    return _lib


class Result:
    """Stage taps of one stream: y1, y2[ch], y3[ch] complex128; bits[ch] bytes; disc[ch] (n,4) float32; messages."""

    def __init__(self):
        self.y1 = None
        self.y2, self.y3, self.bits, self.bitpos, self.disc, self.events = {}, {}, {}, {}, {}, {}
        self.pick_margins = {}   # oracle only: (n, 2) [900 Hz sample count, (best - runner-up) / best] per bit-sync evaluation
        self.messages = []       # (freq, bbbb, text)
        self.timing = None


def _cplx(ptr, n):
    if n == 0:
        return np.zeros(0, dtype=np.complex128)
    a = np.ctypeslib.as_array(ptr, shape=(2 * n,)).copy()
    return a.view(np.complex128)


def run_oracle(iq, h1=None, h2=None, h3=None, nco_hz=(14000.0, -14000.0), nco_period=(0, 0),
               freq_tag=(518, 490), record_taps=True) -> Result:
    """iq: interleaved I,Q as int16 / float32 / float64 1-D array."""
    L = lib()
    p = Params()
    L.nvo_default_params(C.byref(p))
    keep = []
    for name, h in (("1", h1), ("2", h2), ("3", h3)):
        if h is not None:
            arr = np.ascontiguousarray(h, dtype=np.float64)
            keep.append(arr)
            setattr(p, "h" + name, arr.ctypes.data_as(C.POINTER(C.c_double)))
            setattr(p, "n" + name, len(arr))
    n_ch = len(nco_hz)
    for k in range(n_ch):
        p.nco_hz[k] = nco_hz[k]
        p.nco_period[k] = nco_period[k] if k < len(nco_period) else 0
        p.freq_tag[k] = freq_tag[k] if k < len(freq_tag) else 1000 + k
    p.n_channels = n_ch
    p.record_taps = int(record_taps)
    ch = L.nvo_new(C.byref(p))
    iq = np.ascontiguousarray(iq)
    n = iq.size // 2
    if iq.dtype == np.int16:
        L.nvo_push_s16(ch, iq.ctypes.data_as(C.POINTER(C.c_int16)), n)
    elif iq.dtype == np.float32:
        L.nvo_push_f32(ch, iq.ctypes.data_as(C.POINTER(C.c_float)), n)
    else:
        iq = iq.astype(np.float64)
        L.nvo_push(ch, iq.ctypes.data_as(C.POINTER(C.c_double)), n)
    return _collect(L, ch, n_ch)


def run_oracle_900(y3_row, freq_tag=518) -> Result:
    """One channel fed straight at 900 Hz (nvo_push_900): y3_row is a complex 1-D array, taken as FP64.  The Result holds that
    channel under key "518" (y3 = the input), its decisions, pick margins, events and messages."""
    L = lib()
    p = Params()
    L.nvo_default_params(C.byref(p))
    p.n_channels = 1
    p.freq_tag[0] = freq_tag
    p.record_taps = 1
    ch = L.nvo_new(C.byref(p))
    iq = np.ascontiguousarray(np.asarray(y3_row, dtype=np.complex128)).view(np.float64)
    L.nvo_push_900(ch, 0, iq.ctypes.data_as(C.POINTER(C.c_double)), iq.size // 2)
    return _collect(L, ch, 1)


def _collect(L, ch, n_ch) -> Result:
    """the taps, events and messages of chain `ch`, which is freed"""
    r = Result()
    pd = C.POINTER(C.c_double)()
    r.y1 = _cplx(pd, L.nvo_y1(ch, C.byref(pd)))
    for c, tag in enumerate(CHANNEL_KEYS[:n_ch]):
        pd = C.POINTER(C.c_double)()
        r.y2[tag] = _cplx(pd, L.nvo_y2(ch, c, C.byref(pd)))
        pd = C.POINTER(C.c_double)()
        r.y3[tag] = _cplx(pd, L.nvo_y3(ch, c, C.byref(pd)))
        pc = C.POINTER(C.c_char)()
        nb = L.nvo_bits(ch, c, C.byref(pc))
        r.bits[tag] = C.string_at(pc, nb) if nb else b""
        pi = C.POINTER(C.c_int32)()
        nb = L.nvo_bitpos(ch, c, C.byref(pi))
        r.bitpos[tag] = np.ctypeslib.as_array(pi, shape=(nb,)).copy() if nb else np.zeros(0, np.int32)
        pf = C.POINTER(C.c_float)()
        nb = L.nvo_disc(ch, c, C.byref(pf))
        r.disc[tag] = np.ctypeslib.as_array(pf, shape=(nb, 4)).copy() if nb else np.zeros((0, 4), np.float32)
        pm = C.POINTER(C.c_double)()
        nm = L.nvo_pick_margins(ch, c, C.byref(pm))
        r.pick_margins[tag] = np.ctypeslib.as_array(pm, shape=(nm, 2)).copy() if nm else np.zeros((0, 2))
        pc = C.POINTER(C.c_char)()
        ne = L.nvo_events(ch, c, C.byref(pc))
        r.events[tag] = C.string_at(pc, ne) if ne else b""
    for k in range(L.nvo_n_messages(ch)):
        f = C.c_int()
        b = C.c_char_p()
        t = C.c_char_p()
        L.nvo_message(ch, k, C.byref(f), C.byref(b), C.byref(t))
        r.messages.append((f.value, b.value.decode("latin-1"), t.value.decode("latin-1")))
    L.nvo_free(ch)
    return r


def have_ref() -> bool:
    return os.path.exists(REF_CHAIN)


def run_ref(iq=None, wav=None, passes=1, taps=True) -> Result:
    """Run the compiled, unmodified reference on one stream (one process: its state is global)."""
    with tempfile.TemporaryDirectory() as td:
        if wav is not None:
            args = ["--wav", wav]
        else:
            iq = np.ascontiguousarray(iq)
            kind = {np.dtype(np.int16): "--s16", np.dtype(np.float32): "--f32"}[iq.dtype]
            path = os.path.join(td, "in.raw")
            iq.tofile(path)
            args = [kind, path]
        prefix = os.path.join(td, "o")
        cmd = [REF_CHAIN] + args + ["--passes", str(passes)]
        if taps:
            cmd += ["--out", prefix]
        cp = subprocess.run(cmd, check=True, capture_output=True)
        r = Result()
        r.timing = json.loads(cp.stderr.decode().strip().splitlines()[-1])
        if not taps:
            return r
        r.y1 = np.fromfile(prefix + ".y1", dtype=np.complex128)
        for tag in CHANNELS:
            r.y2[tag] = np.fromfile(prefix + ".y2_" + tag, dtype=np.complex128)
            r.y3[tag] = np.fromfile(prefix + ".y3_" + tag, dtype=np.complex128)
            r.bits[tag] = open(prefix + ".bits_" + tag, "rb").read()
            r.bitpos[tag] = np.fromfile(prefix + ".bitpos_" + tag, dtype=np.int32)
            r.disc[tag] = np.fromfile(prefix + ".disc_" + tag, dtype=np.float32).reshape(-1, 4)
        raw = open(prefix + ".msgs", "rb").read()
        pos = 0
        while pos < len(raw):
            nl = raw.index(b"\n", pos)
            freq, bbbb, ln = raw[pos:nl].decode("latin-1").split("|")
            ln = int(ln)
            r.messages.append((int(freq), bbbb, raw[nl + 1: nl + 1 + ln].decode("latin-1")))
            pos = nl + 1 + ln + 1
        return r

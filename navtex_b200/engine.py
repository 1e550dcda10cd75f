"""ctypes binding of libnavtex_b200.so (include/navtex_b200.h).

Python is only the harness language here (tests, bench): the product is the C ABI.  There is no
CPU fallback: importing works anywhere, but creating an Engine needs the built library and a GPU.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NVX_LIB") or os.path.join(_HERE, "libnavtex_b200.so")   # NVX_LIB: tuning variants only
BLOCK_ALIGN = 280
FS = 252_000


class NvxError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("device", C.c_int), ("n_streams", C.c_int), ("max_block", C.c_longlong), ("freq_tag", C.c_int * 2),
        ("h1", C.POINTER(C.c_double)), ("h2", C.POINTER(C.c_double)), ("h3", C.POINTER(C.c_double)),
        ("keep_bits", C.c_int), ("first_stream_id", C.c_int),
        ("nco_hz", C.POINTER(C.c_double)), ("stream_freq_tag", C.POINTER(C.c_int)),
        ("n1", C.c_int), ("n2", C.c_int), ("n3", C.c_int), ("n_channels", C.c_int),
    ]


class Message(C.Structure):
    _fields_ = [("stream", C.c_int), ("freq", C.c_int), ("bbbb", C.c_char * 8), ("text", C.c_char_p), ("text_len", C.c_size_t)]


class Stats(C.Structure):
    _fields_ = [("cascade_ms", C.c_double), ("demod_ms", C.c_double), ("cascade_launches", C.c_longlong),
                ("demod_launches", C.c_longlong), ("aux_launches", C.c_longlong), ("samples", C.c_longlong),
                ("demod_stage_ms", C.c_double * 6), ("long_tc_fallbacks", C.c_longlong), ("messages", C.c_longlong),
                ("cascade_ms_min", C.c_double), ("cascade_ms_max", C.c_double)]


class SynthDesc(C.Structure):
    _fields_ = [("bits", C.POINTER(C.c_uint8)), ("bit_off", C.POINTER(C.c_longlong)), ("offset_hz", C.POINTER(C.c_float)),
                ("start_s", C.POINTER(C.c_float)), ("amplitude", C.POINTER(C.c_float)), ("noise_sigma", C.POINTER(C.c_float)),
                ("seed", C.c_ulonglong)]


EXPORTS = (
    "nvx_default_config", "nvx_last_error", "nvx_engine_create", "nvx_engine_destroy", "nvx_engine_reset",
    "nvx_engine_push_host_f32", "nvx_engine_push_host_s16", "nvx_engine_push_host_u8", "nvx_engine_push_device_f32",
    "nvx_engine_push_device_s16", "nvx_engine_push_device_u8",
    "nvx_engine_sync", "nvx_engine_wait_ingest", "nvx_engine_host_pushes", "nvx_engine_wait_ingest_of", "nvx_engine_poll_messages", "nvx_engine_try_poll_messages", "nvx_engine_set_message_callback", "nvx_engine_read_y3",
    "nvx_engine_read_bits", "nvx_engine_read_events", "nvx_engine_enable_timing", "nvx_engine_get_stats",
    "nvx_engine_stream", "nvx_engine_get_cascade_spans", "nvx_engine_fence", "nvx_pinned_alloc", "nvx_pinned_free", "nvx_synth_fill_device", "nvx_host_assemble", "nvx_debug_long_tc_band",
    "nvx_capture_create", "nvx_capture_create_u8", "nvx_capture_destroy", "nvx_capture_write", "nvx_capture_write_u8", "nvx_capture_pump",
    "nvx_capture_start", "nvx_capture_stop",
    "nvx_capture_dropped", "nvx_store_create", "nvx_store_destroy", "nvx_store_add", "nvx_store_add_at", "nvx_store_sink",
    "nvx_store_count", "nvx_store_get", "nvx_store_purge", "nvx_store_dump_csv",
)

MESSAGE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int)

_lib = None


def load_library():
    """dlopen the in-tree CUDA library; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NvxError(f"{LIB_PATH} is missing: run navtex_b200/build.sh (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.nvx_last_error.restype = C.c_char_p
    L.nvx_default_config.argtypes = [C.POINTER(Config)]
    L.nvx_engine_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    L.nvx_engine_destroy.argtypes = [C.c_void_p]
    L.nvx_engine_destroy.restype = None
    L.nvx_engine_reset.argtypes = [C.c_void_p]
    for name in ("nvx_engine_push_host_f32", "nvx_engine_push_host_s16", "nvx_engine_push_host_u8", "nvx_engine_push_device_f32",
                 "nvx_engine_push_device_s16", "nvx_engine_push_device_u8"):
        getattr(L, name).argtypes = [C.c_void_p, C.c_void_p, C.c_longlong]
    L.nvx_engine_sync.argtypes = [C.c_void_p]
    L.nvx_engine_poll_messages.argtypes = [C.c_void_p, C.POINTER(C.POINTER(Message)), C.POINTER(C.c_size_t)]
    L.nvx_engine_try_poll_messages.argtypes = [C.c_void_p, C.POINTER(C.POINTER(Message)), C.POINTER(C.c_size_t)]
    L.nvx_engine_wait_ingest.argtypes = [C.c_void_p]
    L.nvx_engine_host_pushes.argtypes = [C.c_void_p]
    L.nvx_engine_host_pushes.restype = C.c_longlong
    L.nvx_engine_wait_ingest_of.argtypes = [C.c_void_p, C.c_longlong]
    L.nvx_engine_read_y3.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.nvx_engine_read_bits.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.nvx_engine_read_events.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.nvx_engine_enable_timing.argtypes = [C.c_void_p, C.c_int]
    L.nvx_engine_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats), C.c_int]
    L.nvx_engine_stream.argtypes = [C.c_void_p]
    L.nvx_engine_get_cascade_spans.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.nvx_engine_fence.argtypes = [C.c_void_p]
    L.nvx_pinned_alloc.argtypes = [C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
    L.nvx_pinned_free.argtypes = [C.c_void_p]
    L.nvx_engine_stream.restype = C.c_void_p
    L.nvx_synth_fill_device.argtypes = [C.c_int, C.POINTER(SynthDesc), C.c_int, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p]
    L.nvx_host_assemble.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, MESSAGE_CB, C.c_void_p]
    L.nvx_engine_set_message_callback.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.nvx_capture_create.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.POINTER(C.c_void_p)]
    L.nvx_capture_create_u8.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.POINTER(C.c_void_p)]
    L.nvx_capture_destroy.argtypes = [C.c_void_p]
    L.nvx_capture_destroy.restype = None
    L.nvx_capture_write.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint]
    L.nvx_capture_write_u8.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint]
    for name in ("nvx_capture_pump", "nvx_capture_dropped"):
        getattr(L, name).restype = C.c_longlong
    L.nvx_capture_pump.argtypes = [C.c_void_p]
    L.nvx_capture_dropped.argtypes = [C.c_void_p, C.c_int]
    L.nvx_capture_start.argtypes = [C.c_void_p, C.c_int]
    L.nvx_capture_stop.argtypes = [C.c_void_p]
    L.nvx_store_create.restype = C.c_void_p
    L.nvx_store_destroy.argtypes = [C.c_void_p]
    L.nvx_store_destroy.restype = None
    L.nvx_store_add.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int]
    L.nvx_store_add_at.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int, C.c_longlong]
    L.nvx_store_count.argtypes = [C.c_void_p]
    L.nvx_store_count.restype = C.c_size_t
    L.nvx_store_get.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_char_p, C.POINTER(C.c_char_p)]
    L.nvx_store_purge.argtypes = [C.c_void_p, C.c_longlong, C.c_longlong]
    L.nvx_store_dump_csv.argtypes = [C.c_void_p, C.c_char_p]
    _lib = L
    return L


def host_assemble(events: bytes, stream: int = 0, freq: int = 518):
    """Host-side message assembly of one channel's event bytes -> [(stream, freq, bbbb, text)]."""
    out = []

    def cb(_user, strm, bbbb, text, f):
        out.append((strm, f, bbbb.decode("latin-1"), text.decode("latin-1")))
        return 0

    _check(min(0, load_library().nvx_host_assemble(events, len(events), stream, freq, MESSAGE_CB(cb), None)))
    return out


def long_tc_band(decimation: int, h):
    """The band-matrix operand of the tensor-core long-tap kernel for one stage (host only; tests): returns
    (geometry dict, g_hi, g_lo) with g_* shaped [copies][J][32], see nvx_debug_long_tc_band in navtex_b200.h."""
    L = load_library()
    L.nvx_debug_long_tc_band.argtypes = [C.c_int, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_float),
                                         C.POINTER(C.c_float), C.c_size_t]
    h = np.ascontiguousarray(h, dtype=np.float64)
    geo = (C.c_int * 5)()
    hp = h.ctypes.data_as(C.POINTER(C.c_double))
    n = L.nvx_debug_long_tc_band(decimation, hp, h.size, geo, None, None, 0)
    _check(min(0, n))
    hi, lo = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
    _check(min(0, L.nvx_debug_long_tc_band(decimation, hp, h.size, geo, hi.ctypes.data_as(C.POINTER(C.c_float)),
                                           lo.ctypes.data_as(C.POINTER(C.c_float)), n)))
    g = dict(zip(("taps_padded", "n_tile", "chunks", "band_rows", "copies"), list(geo)))
    shape = (g["copies"], g["band_rows"], 32)
    return g, hi.reshape(shape), lo.reshape(shape)


def _check(rc, allow_overflow=False):
    if rc == 0 or (allow_overflow and rc == -4):
        return rc
    raise NvxError(f"nvx error {rc}: {load_library().nvx_last_error().decode()}")


class Engine:
    """One GPU, S streams.  Mirrors the reference's init / per-sample push / add_message flow, batched."""

    def __init__(self, n_streams: int, max_block: int, device: int = 0, keep_bits: bool = False, taps=None,
                 first_stream_id: int = 0, nco_hz=None, stream_freq_tag=None, n_channels: int = 2):
        L = load_library()
        cfg = Config()
        L.nvx_default_config(C.byref(cfg))
        cfg.device, cfg.n_streams, cfg.max_block = device, n_streams, max_block
        cfg.keep_bits, cfg.first_stream_id = int(keep_bits), first_stream_id
        self._taps = None
        if taps is not None:
            self._taps = [np.ascontiguousarray(t, dtype=np.float64) for t in taps]
            cfg.h1, cfg.h2, cfg.h3 = (t.ctypes.data_as(C.POINTER(C.c_double)) for t in self._taps)
            # up to 37/47/71 and up to 61/75/111 taps: fused kernel (zero-padded); longer: the long-tap path
            cfg.n1, cfg.n2, cfg.n3 = (len(t) for t in self._taps)
        cfg.n_channels = n_channels
        if nco_hz is not None:           # [S, n_channels] per-stream channel offsets in Hz
            self._nco = np.ascontiguousarray(nco_hz, dtype=np.float64).reshape(n_streams, n_channels)
            cfg.nco_hz = self._nco.ctypes.data_as(C.POINTER(C.c_double))
        if stream_freq_tag is not None:
            self._tags = np.ascontiguousarray(stream_freq_tag, dtype=np.int32).reshape(n_streams, n_channels)
            cfg.stream_freq_tag = self._tags.ctypes.data_as(C.POINTER(C.c_int))
        self._h = C.c_void_p()
        _check(L.nvx_engine_create(C.byref(cfg), C.byref(self._h)))
        self.L, self.S, self.max_block, self.device = L, n_streams, max_block, device
        self.C = n_channels
        self.last_n = 0

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self.L.nvx_engine_destroy(h)
            h.value = None

    __del__ = close

    def reset(self):
        _check(self.L.nvx_engine_reset(self._h))

    def push_host(self, iq: np.ndarray):
        """iq: [S, n, 2] (or [S, 2n]) float32, int16 or uint8 (8-bit offset binary, value u - 128), C-contiguous."""
        iq = np.ascontiguousarray(iq)
        n = iq.size // (2 * self.S)
        fn = {np.dtype(np.float32): self.L.nvx_engine_push_host_f32, np.dtype(np.int16): self.L.nvx_engine_push_host_s16,
              np.dtype(np.uint8): self.L.nvx_engine_push_host_u8}[iq.dtype]
        _check(fn(self._h, iq.ctypes.data_as(C.c_void_p), n))
        self.last_n = n

    def push_host_ptr(self, ptr: int, n: int, s16: bool, u8: bool = False):
        fn = self.L.nvx_engine_push_host_u8 if u8 else self.L.nvx_engine_push_host_s16 if s16 else self.L.nvx_engine_push_host_f32
        _check(fn(self._h, C.c_void_p(ptr), n))
        self.last_n = n

    def push_device(self, ptr: int, n: int, s16: bool = False, u8: bool = False):
        fn = self.L.nvx_engine_push_device_u8 if u8 else self.L.nvx_engine_push_device_s16 if s16 else self.L.nvx_engine_push_device_f32
        _check(fn(self._h, C.c_void_p(ptr), n))
        self.last_n = n

    def sync(self):
        _check(self.L.nvx_engine_sync(self._h), allow_overflow=True)

    def wait_ingest(self):
        _check(self.L.nvx_engine_wait_ingest(self._h))

    def poll_messages(self, wait: bool = True):
        """Messages completed since the previous poll; wait=False does not sync (pipeline keeps running)."""
        msgs = C.POINTER(Message)()
        cnt = C.c_size_t()
        fn = self.L.nvx_engine_poll_messages if wait else self.L.nvx_engine_try_poll_messages
        _check(fn(self._h, C.byref(msgs), C.byref(cnt)), allow_overflow=True)
        return [(msgs[k].stream, msgs[k].freq, msgs[k].bbbb.decode("latin-1"), C.string_at(msgs[k].text, msgs[k].text_len).decode("latin-1"))
                for k in range(cnt.value)]

    def read_y3(self) -> np.ndarray:
        """[S, n_channels, P] complex64 of the last block."""
        P = self.last_n // BLOCK_ALIGN
        out = np.empty((self.S, self.C, P, 2), dtype=np.float32)
        got = C.c_size_t()
        _check(self.L.nvx_engine_read_y3(self._h, out.ctypes.data_as(C.c_void_p), out.size, C.byref(got)))
        assert got.value == P
        return out.view(np.complex64)[..., 0]

    def read_bits(self, stream: int, ch: int):
        cap = self.last_n // BLOCK_ALIGN // 8 + 4
        bits = np.empty(cap, dtype=np.uint8)
        sums = np.empty((cap, 4), dtype=np.float32)
        got = C.c_size_t()
        _check(self.L.nvx_engine_read_bits(self._h, stream, ch, bits.ctypes.data_as(C.c_void_p), sums.ctypes.data_as(C.c_void_p), cap, C.byref(got)))
        return bits[: got.value].tobytes(), sums[: got.value].copy()

    def read_events(self, stream: int, ch: int) -> bytes:
        cap = self.last_n // BLOCK_ALIGN // 30 + 64
        ev = np.empty(cap, dtype=np.uint8)
        got = C.c_size_t()
        _check(self.L.nvx_engine_read_events(self._h, stream, ch, ev.ctypes.data_as(C.c_void_p), cap, C.byref(got)))
        return ev[: got.value].tobytes()

    def enable_timing(self, level=2):
        """0/False off, 1 fused-FIR kernel only, 2/True every stage."""
        level = 2 if level is True else int(level)
        _check(self.L.nvx_engine_enable_timing(self._h, level), allow_overflow=True)

    def stats(self, reset: bool = True) -> Stats:
        st = Stats()
        _check(self.L.nvx_engine_get_stats(self._h, C.byref(st), int(reset)), allow_overflow=True)
        return st

    def cascade_spans(self) -> np.ndarray:
        """Per-launch times (ms) of the fused-FIR kernel since the last stats(reset=True)."""
        cnt = C.c_size_t()
        _check(self.L.nvx_engine_get_cascade_spans(self._h, None, 0, C.byref(cnt)), allow_overflow=True)
        out = np.zeros(cnt.value, dtype=np.float32)
        if cnt.value:
            _check(self.L.nvx_engine_get_cascade_spans(self._h, out.ctypes.data_as(C.c_void_p), out.size, C.byref(cnt)), allow_overflow=True)
        return out

    def fence(self):
        """Order the engine's main stream behind everything queued so far on its demod stream (device side, no host wait)."""
        _check(self.L.nvx_engine_fence(self._h))

    @property
    def stream(self) -> int:
        return self.L.nvx_engine_stream(self._h) or 0


class PinnedBuffer:
    """Page-locked host memory from nvx_pinned_alloc as a numpy array (int16 by default)."""

    def __init__(self, shape, dtype=np.int16, write_combined=False):
        self.L = load_library()
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self._p = C.c_void_p()
        _check(self.L.nvx_pinned_alloc(self.nbytes, int(write_combined), C.byref(self._p)))
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self._p.value)).view(self.dtype).reshape(self.shape)

    @property
    def ptr(self) -> int:
        return self._p.value

    def close(self):
        if getattr(self, "_p", None) is not None and self._p.value:
            self.array = None
            self.L.nvx_pinned_free(self._p)
            self._p = C.c_void_p()

    __del__ = close


class Store:
    """In-memory message store behind add_message (message_store.c:59-97): newest message per (stream, bbbb)."""

    def __init__(self):
        self.L = load_library()
        self._h = C.c_void_p(self.L.nvx_store_create())

    def close(self):
        if self._h and self._h.value:
            self.L.nvx_store_destroy(self._h)
            self._h = None

    __del__ = close

    def add(self, stream, bbbb, text, freq, when=None):
        if when is None:
            return self.L.nvx_store_add(self._h, stream, bbbb.encode("latin-1"), text.encode("latin-1"), freq)
        return self.L.nvx_store_add_at(self._h, stream, bbbb.encode("latin-1"), text.encode("latin-1"), freq, int(when))

    def attach(self, eng: "Engine"):
        """Route the engine's messages into this store (nvx_store_sink as the add_message-shaped callback)."""
        fn = C.cast(self.L.nvx_store_sink, C.c_void_p)
        _check(self.L.nvx_engine_set_message_callback(eng._h, fn, self._h))

    def rows(self):
        out = []
        for k in range(self.L.nvx_store_count(self._h)):
            stream, freq = C.c_int(), C.c_int()
            bbbb, stamp = C.create_string_buffer(8), C.create_string_buffer(20)
            text = C.c_char_p()
            _check(self.L.nvx_store_get(self._h, k, C.byref(stream), C.byref(freq), bbbb, stamp, C.byref(text)))
            out.append((stream.value, freq.value, bbbb.value.decode("latin-1"), stamp.value.decode(), text.value.decode("latin-1")))
        return out

    def purge(self, now, max_age_s=72 * 3600):
        return self.L.nvx_store_purge(self._h, int(now), int(max_age_s))

    def dump_csv(self, path):
        _check(self.L.nvx_store_dump_csv(self._h, path.encode()))


class Capture:
    """Radio front end: per-stream rings fed by radio callbacks, pumped into the engine in blocks.  fmt="s16": SDRplay-format
    int16 rings (write); fmt="u8": RTL-SDR 8-bit rings (write_u8)."""

    def __init__(self, eng: "Engine", max_block: int, ring_samples: int, fmt: str = "s16"):
        self.L, self.eng = eng.L, eng
        self._h = C.c_void_p()
        create = {"s16": self.L.nvx_capture_create, "u8": self.L.nvx_capture_create_u8}[fmt]
        _check(create(eng._h, eng.S, max_block, ring_samples, C.byref(self._h)))

    def write(self, stream: int, xi: np.ndarray, xq: np.ndarray) -> int:
        xi = np.ascontiguousarray(xi, dtype=np.int16)
        xq = np.ascontiguousarray(xq, dtype=np.int16)
        return self.L.nvx_capture_write(self._h, stream, xi.ctypes.data_as(C.c_void_p), xq.ctypes.data_as(C.c_void_p), len(xi))

    def write_u8(self, stream: int, iq: np.ndarray) -> int:
        """iq: interleaved I,Q bytes ([n, 2] or [2n] uint8), as the rtlsdr_read_async callback hands them over."""
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        return self.L.nvx_capture_write_u8(self._h, stream, iq.ctypes.data_as(C.c_void_p), iq.size // 2)

    def pump(self) -> int:
        n = self.L.nvx_capture_pump(self._h)
        if n < 0:
            _check(int(n))
        if n > 0:
            self.eng.last_n = int(n)             # read_y3 / read_events of the engine see this block
        return int(n)

    def start(self, poll_ms: int = 50):
        _check(self.L.nvx_capture_start(self._h, poll_ms))

    def stop(self):
        _check(self.L.nvx_capture_stop(self._h), allow_overflow=True)

    def dropped(self, stream: int) -> int:
        return int(self.L.nvx_capture_dropped(self._h, stream))

    def close(self):
        if self._h and self._h.value:
            self.L.nvx_capture_destroy(self._h)
            self._h = None

    __del__ = close


def synth_fill_device(device: int, d_ptr: int, n_streams: int, t0: int, n: int, bits_per_stream, offset_hz, start_s,
                      amplitude, noise_sigma, seed: int, cuda_stream: int = 0):
    """Fill a device float2 [S][n] block with samples [t0, t0+n) of S synthetic captures (see synth.cu)."""
    L = load_library()
    off = np.zeros(n_streams + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(b) for b in bits_per_stream])
    bits = np.concatenate([np.asarray(b, dtype=np.uint8) for b in bits_per_stream]) if off[-1] else np.zeros(1, np.uint8)
    arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in (offset_hz, start_s, amplitude, noise_sigma)]
    d = SynthDesc()
    d.bits = bits.ctypes.data_as(C.POINTER(C.c_uint8))
    d.bit_off = off.ctypes.data_as(C.POINTER(C.c_longlong))
    d.offset_hz, d.start_s, d.amplitude, d.noise_sigma = (a.ctypes.data_as(C.POINTER(C.c_float)) for a in arrs)
    d.seed = seed
    _check(L.nvx_synth_fill_device(device, C.byref(d), n_streams, t0, n, C.c_void_p(d_ptr), C.c_void_p(cuda_stream)))

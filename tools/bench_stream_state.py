"""Cost of saving and loading streams' receive state (nvx_engine_save_streams / nvx_engine_load_streams).

    python tools/bench_stream_state.py [--rounds R] [--out profiles/bench_stream_state_n1.json]

Two workloads on one GPU, float2 input:
  * bench.py's default shape: 1024 streams x bench.BLOCK samples, generated on the device by nvx_synth_fill_device from
    bench.make_bulletins;
  * the most streams an engine takes: 32 767 streams, 100 superblocks (28 000 samples) per push, silence.
Save: host clock around one nvx_engine_save_streams call of every stream into a preallocated buffer, on an engine that is idle
(the call's own sync finds nothing to wait for): the gather kernel, the one device-to-host copy, the message part and the
checksum.  Load: host clock around nvx_engine_load_streams (validation, checksum, the records copied into the engine) plus the
device time the next push spends on it: that push's time (CUDA events on the engine stream around the push and a sync) minus
the median of pushes without a load in the same run.  The state is loaded back into the engine that saved it (same position).
The GPU's name, power limit and clocks are read in the same run.  One JSON line goes to stdout and to --out."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (workload shape, bulletins)
from bench_u8 import gpu_info  # noqa: E402

# estimate from the sizes in the code, per stream of the fused reference class with float input and two channels:
# input tail 1960 x 8 B, and per channel 16 y3 (8 B) + 640 correlation values (8 B) + ClockState 24 B + FsmState 64 B + epoch 8 B
ESTIMATE_BYTES = 1960 * 8 + 2 * (16 * 8 + 640 * 8 + 24 + 64 + 8)


def measure(np, torch, eng, push, rounds):
    L, S = eng.L, eng.S
    streams = (C.c_int * S)(*range(S))
    size = C.c_size_t()
    push()
    eng.sync()
    assert L.nvx_engine_save_streams(eng._h, streams, S, None, 0, C.byref(size)) == 0
    buf = np.empty(size.value, dtype=np.uint8)
    ptr = C.c_void_p(buf.ctypes.data)
    es = torch.cuda.ExternalStream(eng.stream, device=torch.device("cuda", 0))

    def timed_push():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(es)
        push()
        eng.sync()
        e1.record(es)
        e1.synchronize()
        return e0.elapsed_time(e1)

    save, load_call, push_plain, push_loaded = [], [], [], []
    for _ in range(rounds):
        push_plain.append(timed_push())
        eng.sync()
        t0 = time.perf_counter()
        rc = L.nvx_engine_save_streams(eng._h, streams, S, ptr, size.value, C.byref(size))
        save.append((time.perf_counter() - t0) * 1e3)
        assert rc == 0, L.nvx_last_error()
        t0 = time.perf_counter()
        rc = L.nvx_engine_load_streams(eng._h, streams, S, ptr, size.value)
        load_call.append((time.perf_counter() - t0) * 1e3)
        assert rc == 0, L.nvx_last_error()
        push_loaded.append(timed_push())
        eng.poll_messages()
    base = statistics.median(push_plain)
    load = [c + p - base for c, p in zip(load_call, push_loaded)]

    def summary(v):
        return {"median": statistics.median(v), "min": min(v), "max": max(v), "rounds": v}

    return {
        "streams": S, "samples_per_push": eng.last_n, "state_bytes": size.value, "bytes_per_stream": size.value / S,
        "estimate_bytes_per_stream": ESTIMATE_BYTES,
        "save_ms": summary(save), "load_ms": summary(load), "load_call_ms": summary(load_call),
        "push_ms_without_load": summary(push_plain), "push_ms_with_load": summary(push_loaded),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_stream_state_n1.json"))
    args = ap.parse_args()

    import numpy as np
    import torch
    from navtex_b200 import engine, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench_stream_state.py: no CUDA device")
    dev = torch.device("cuda", 0)
    info_before = gpu_info()
    res = {}

    S, n = bench.STREAMS_PER_GPU, bench.BLOCK
    bits, off, start, amp, sigma, _ = bench.make_bulletins(np, synth, S, 0, 518490, n, 1, 3, 18, 5)
    x = torch.empty((S, n, 2), dtype=torch.float32, device=dev)
    engine.synth_fill_device(0, x.data_ptr(), S, 0, n, bits, off, start, amp, sigma, seed=518490)
    torch.cuda.synchronize()
    eng = engine.Engine(S, n)
    res["bench_1024"] = measure(np, torch, eng, lambda: eng.push_device(x.data_ptr(), n), args.rounds)
    eng.close()
    del x

    S, n = 32767, 100 * engine.BLOCK_ALIGN
    x = torch.zeros((S, n, 2), dtype=torch.float32, device=dev)
    eng = engine.Engine(S, n)
    res["max_32767"] = measure(np, torch, eng, lambda: eng.push_device(x.data_ptr(), n), args.rounds)
    eng.close()
    info_during = gpu_info()

    rec = {"what": "save / load of every stream's state (tools/bench_stream_state.py)", "gpu": info_before, "gpu_after_timing": info_during, **res}
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()

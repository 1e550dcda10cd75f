"""Engines fed at the radio's own rate: the rational resampler on the GPU in front of the fused cascade.

    python tools/bench_resample.py [--steps K] [--streams S] [--seconds T] [--out profiles/bench_resample_n1.json]

Workload per case: S = 1024 device-resident streams of about T = 10 s at the case's rate and format (256 kS/s 8-bit and int16,
192 kS/s int16, 2.048 and 2.4 MS/s 8-bit).  At 2.4 MS/s that is 24 G input samples, too many to synthesise per stream on the
host, so 32 distinct captures (one bulletin each, at +14 or -14 kHz, with noise; synth.fsk_iq at the case's rate) are tiled
over the streams, and every stream gets its own message tag: each of the S bulletins is verified, per stream, in every case.

Per case: the resampler kernel's time (the engine's CUDA events around its launch, nvx_stats.resample_ms, over K pushes), its
compulsory bytes (input bytes + 8 B per 252 kS/s output) over that time, against the device-to-device copy peak measured in
the same run (best of five 8 GB torch copies, read + write bytes over time); the whole step time (device events around K pushes and a sync);
and input Gsamples/s.  An e2e leg at 256 kS/s 8-bit pushes from page-locked memory beside a bare pinned cudaMemcpyAsync of the
same bytes (the ceiling), as tools/bench_u8.py does.  The GPU's name and power limit are read in the same run.  One JSON line
goes to stdout and to --out."""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [(256_000, "u8"), (256_000, "s16"), (192_000, "s16"), (2_048_000, "u8"), (2_400_000, "u8")]
AMP = {"s16": 8000.0, "u8": 30.0}
DISTINCT = 32


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {"error": "nvidia-smi unavailable"}


def copy_peak(torch):
    """device-to-device copy rate in GB/s (read + write bytes), best of 5 copies of 8 GB"""
    a = torch.empty(8 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * a.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def captures(rate, fmt, seconds):
    import numpy as np
    from navtex_b200 import synth

    def one(k):
        rng = np.random.default_rng(7000 + k)
        text, bbbb = synth.random_message(rng, n_lines=1, words_per_line=2)
        em = synth.Emission(text, (14000.0, -14000.0)[k % 2], start_s=0.3 + 0.05 * k, n_phasing=18, n_tail=5, amplitude=AMP[fmt])
        x = synth.fsk_iq([em], seconds, snr_db=6.0, seed=7000 + k, rate=rate)
        q = synth.quantise_u8(x) if fmt == "u8" else synth.quantise_s16(x)
        return q.reshape(-1, 2), (bbbb, text)

    with cf.ThreadPoolExecutor(8) as ex:
        return list(ex.map(one, range(DISTINCT)))


def run_case(torch, rate, fmt, S, seconds, steps):
    import numpy as np
    from navtex_b200 import engine

    info = engine.resampler_info(rate)
    n = int(seconds * rate) // info["align"] * info["align"]
    caps = captures(rate, fmt, n / rate + 0.01)
    base = torch.from_numpy(np.stack([c[0][:n] for c in caps])).cuda()
    x = base[torch.arange(S, device="cuda") % DISTINCT].contiguous()
    del base
    tags = np.stack([np.arange(S) + 100_000, np.arange(S) + 200_000], axis=1)
    eng = engine.Engine(S, n, input_rate_hz=rate, stream_freq_tag=tags)
    u8 = fmt == "u8"
    torch.cuda.synchronize()
    eng.push_device(x.data_ptr(), n, s16=not u8, u8=u8)          # the verified pass: one bulletin per stream
    msgs = eng.poll_messages()
    want = sorted((s, int(tags[s, (s % DISTINCT) % 2])) + caps[s % DISTINCT][1] for s in range(S))
    ok = sorted(msgs) == want
    eng.reset()
    eng.push_device(x.data_ptr(), n, s16=not u8, u8=u8)          # warm-up of the timed shape
    eng.sync()
    eng.enable_timing(1)                                         # CUDA events around the resampler (and the cascade) of every push
    eng.stats(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0 = torch.cuda.ExternalStream(eng.stream)
    e0.record(s0)
    t = time.perf_counter()
    for _ in range(steps):
        eng.push_device(x.data_ptr(), n, s16=not u8, u8=u8)
    eng.sync()
    e1.record(s0)
    e1.synchronize()
    wall = (time.perf_counter() - t) / steps
    step_ms = e0.elapsed_time(e1) / steps
    kern_ms = eng.stats(reset=True).resample_ms / steps
    eng.close()
    if not kern_ms > 0:
        raise SystemExit("bench_resample: no resampler kernel time was recorded at %d S/s %s" % (rate, fmt))
    del x
    torch.cuda.empty_cache()
    n_out = n * info["up"] // info["down"]
    bytes_ = S * n * (2 if u8 else 4) + S * n_out * 8
    return {"rate": rate, "format": fmt, "streams": S, "samples_per_stream": n, "seconds": n / rate, "bulletins_verified": ok,
            "messages": len(msgs), "resample_kernel_ms": kern_ms, "resample_bytes": bytes_,
            "resample_GBps": bytes_ / (kern_ms * 1e-3) / 1e9, "step_ms": step_ms, "step_wall_ms": wall * 1e3,
            "input_Gsamples_per_s": S * n / (step_ms * 1e-3) / 1e9, "taps_per_output": info["taps"].size // info["up"]}


def e2e_u8(torch, S, seconds, steps):
    """push_host_u8 from page-locked memory at 256 kS/s beside a bare pinned copy of the same bytes"""
    import numpy as np
    from navtex_b200 import engine

    rate = 256_000
    info = engine.resampler_info(rate)
    n = int(seconds * rate) // info["align"] * info["align"]
    caps = captures(rate, "u8", n / rate + 0.01)
    buf = engine.PinnedBuffer((S, n, 2), dtype=np.uint8)
    for s in range(S):
        buf.array[s] = caps[s % DISTINCT][0][:n]
    eng = engine.Engine(S, n, input_rate_hz=rate)
    eng.push_host_ptr(buf.ptr, n, s16=False, u8=True)
    eng.sync()
    t = time.perf_counter()
    for _ in range(steps):
        eng.push_host_ptr(buf.ptr, n, s16=False, u8=True)
    eng.sync()
    push_s = (time.perf_counter() - t) / steps
    msgs = eng.poll_messages()
    eng.close()
    d = torch.empty((S, n, 2), dtype=torch.uint8, device="cuda")
    src = torch.from_numpy(buf.array)
    d.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(steps):
        d.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    copy_s = (time.perf_counter() - t) / steps
    del d, src
    buf.close()
    return {"rate": rate, "format": "u8", "streams": S, "samples_per_stream": n, "push_host_ms": push_s * 1e3,
            "input_Gsamples_per_s": S * n / push_s / 1e9, "pinned_copy_ms": copy_s * 1e3, "pinned_copy_GBps": S * n * 2 / copy_s / 1e9,
            "messages_last_push": len(msgs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_resample_n1.json"))
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_resample: no CUDA device (this measurement has no CPU fallback)")
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "copy_peak_GBps": copy_peak(torch), "cases": []}
    for rate, fmt in CASES:
        c = run_case(torch, rate, fmt, a.streams, a.seconds, a.steps)
        c["resample_share_of_copy_peak"] = c["resample_GBps"] / res["copy_peak_GBps"]
        res["cases"].append(c)
        print(json.dumps(c), file=sys.stderr, flush=True)
    res["e2e"] = e2e_u8(torch, a.streams, a.seconds, a.steps)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()

"""8-bit (RTL-SDR) input on the default workload's shape: the same captures pushed as float2, int16 and unsigned 8-bit pairs.

    python tools/bench_u8.py [--rounds R] [--steps K] [--e2e-steps E] [--kernel-only] [--out profiles/bench_u8_n1.json]

Workload: 1024 streams x 2 590 000 samples (bench.py's default), generated on the device by nvx_synth_fill_device from
bench.make_bulletins; a per-stream gain brings each capture's total RMS to 30 LSB per component (a receiver's gain setting:
the SNR is unchanged), and the result is quantised to 8 bits on the device (rint, + 128, clipped to [0, 255]).  The float2
and int16 blocks carry the same values u - 128.

Kernel time per format comes from the engine's own CUDA-event spans around the fused kernel; the whole step (cascade, tail
carry, demod, event download, message assembly) from device events around K pushes and a sync.  The formats alternate, in a
rotating order, for R rounds, so that the spread of each figure is measured in the same run.  Checks: the three formats give
bit-identical y3 and the same messages, and the 8-bit push decodes every transmitted bulletin verbatim.

e2e: push_host_u8 from page-locked memory in consecutive 1.03 s blocks (bench.py's e2e leg, in 8-bit), beside a bare pinned
cudaMemcpyAsync of the same bytes (the ceiling).  The GPU's name, power limit and clocks are read in the same run.  One JSON
line goes to stdout and to --out."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload shape, bulletins, message check)

FMTS = ("f32", "s16", "u8")
RMS_LSB = 30.0


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {"error": "nvidia-smi unavailable"}


def build_inputs(torch, device):
    """[S][n][2] float32 / int16 / uint8 of the same 8-bit captures, and the bulletins they carry."""
    import numpy as np
    from navtex_b200 import engine, synth

    S, n = bench.STREAMS_PER_GPU, bench.BLOCK
    bits, off, start, amp, sigma, expect = bench.make_bulletins(np, synth, S, 0, 518490, n, 1, 3, 18, 5)
    x = torch.empty((S, n, 2), dtype=torch.float32, device=device)
    engine.synth_fill_device(device.index, x.data_ptr(), S, 0, n, bits, off, start, amp, sigma, seed=518490)
    u8 = torch.empty((S, n, 2), dtype=torch.uint8, device=device)
    s16 = torch.empty((S, n, 2), dtype=torch.int16, device=device)
    for a in range(0, S, 64):                              # in slices: no full-size float64 temporaries
        xs = x[a:a + 64]
        rms = xs.double().pow(2).mean(dim=(1, 2)).sqrt()   # total RMS per component, per stream
        g = (RMS_LSB / rms).float().view(-1, 1, 1)
        q = torch.clamp(torch.round(xs * g) + 128.0, 0.0, 255.0)
        u8[a:a + 64] = q.to(torch.uint8)
        xs.copy_(q - 128.0)                                # float2 of the 8-bit values, in place
        s16[a:a + 64] = (q - 128.0).to(torch.int16)
    torch.cuda.synchronize()
    return {"f32": x, "s16": s16, "u8": u8}, expect


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=4, help="pushes per format per round")
    ap.add_argument("--e2e-steps", type=int, default=40)
    ap.add_argument("--kernel-only", action="store_true", help="leave out the e2e leg")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_u8_n1.json"))
    args = ap.parse_args()

    import numpy as np
    import torch
    from navtex_b200 import engine

    if not torch.cuda.is_available():
        raise SystemExit("bench_u8.py: no CUDA device")
    dev = torch.device("cuda", 0)
    info_before = gpu_info()
    S, n = bench.STREAMS_PER_GPU, bench.BLOCK
    data, expect = build_inputs(torch, dev)
    engs = {f: engine.Engine(S, n) for f in FMTS}

    # ---- checks: one push per format from a fresh state
    y3, msgs = {}, {}
    for f in FMTS:
        engs[f].push_device(data[f].data_ptr(), n, s16=f == "s16", u8=f == "u8")
        msgs[f] = engs[f].poll_messages()
        y3[f] = engs[f].read_y3()
    identical = all(np.array_equal(y3["u8"].view(np.uint64), y3[f].view(np.uint64)) for f in ("f32", "s16"))
    same_msgs = all(sorted(msgs["u8"]) == sorted(msgs[f]) for f in ("f32", "s16"))
    exact, _ = bench.count_exact(msgs["u8"], expect)
    del y3

    # ---- timing: formats alternate, rotating order, R rounds
    per = {f: {"kernel_ms_median": [], "step_ms": []} for f in FMTS}
    for r in range(args.rounds):
        for f in FMTS[r % 3:] + FMTS[:r % 3]:
            eng = engs[f]
            eng.push_device(data[f].data_ptr(), n, s16=f == "s16", u8=f == "u8")      # warm
            eng.sync()
            eng.enable_timing(1)
            eng.stats()
            es = torch.cuda.ExternalStream(eng.stream, device=dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(es)
            for _ in range(args.steps):
                eng.push_device(data[f].data_ptr(), n, s16=f == "s16", u8=f == "u8")
            eng.sync()
            e1.record(es)
            e1.synchronize()
            spans = eng.cascade_spans()
            eng.stats()
            eng.poll_messages()
            eng.enable_timing(0)
            per[f]["kernel_ms_median"].append(float(statistics.median(map(float, spans))))
            per[f]["step_ms"].append(e0.elapsed_time(e1) / args.steps)
    info_during = gpu_info()
    for e in engs.values():
        e.close()

    def summary(v):
        return {"median": statistics.median(v), "min": min(v), "max": max(v), "rounds": v}

    kernel = {f: summary(per[f]["kernel_ms_median"]) for f in FMTS}
    step = {f: summary(per[f]["step_ms"]) for f in FMTS}
    # the 8-bit kernel is "not slower" when its median is within the larger of the two formats' round-to-round spreads
    spread = max(kernel["u8"]["max"] - kernel["u8"]["min"], kernel["s16"]["max"] - kernel["s16"]["min"])
    rec = {
        "what": "8-bit unsigned I,Q input vs int16 and float2 on the same captures (tools/bench_u8.py)",
        "gpu": info_before, "gpu_after_timing": info_during,
        "streams": S, "samples_per_stream": n, "rms_lsb_per_component": RMS_LSB,
        "kernel_ms": kernel, "step_ms": step,
        "kernel_gsamples_per_s": {f: S * n / kernel[f]["median"] / 1e6 for f in FMTS},
        "step_gsamples_per_s": {f: S * n / step[f]["median"] / 1e6 for f in FMTS},
        "u8_kernel_vs_s16": kernel["u8"]["median"] / kernel["s16"]["median"],
        "u8_not_slower_than_s16_beyond_spread": kernel["u8"]["median"] <= kernel["s16"]["median"] + spread,
        "check": {"y3_bit_identical_f32_s16_u8": bool(identical), "messages_equal": bool(same_msgs),
                  "bulletins_exact_u8": int(exact), "bulletins": len(expect)},
        "rounds": args.rounds, "steps_per_round": args.steps,
    }
    u8 = data.pop("u8")
    del data

    if not args.kernel_only:
        rec["e2e"] = leg_e2e(torch, dev, args.e2e_steps, expect, u8)
        rec["gpu_after_e2e"] = gpu_info()
    line = json.dumps(rec)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")


def leg_e2e(torch, dev, steps, expect, u8):
    """push_host_u8 from page-locked memory, consecutive 1.03 s blocks of the same captures; then a bare pinned copy of the same
    chunks (the ceiling)."""
    import numpy as np
    from navtex_b200 import engine

    S, ne, K = bench.STREAMS_PER_GPU, bench.E2E_BLOCK, bench.E2E_CHUNKS
    pinned = engine.PinnedBuffer((K, S, ne, 2), np.uint8)
    host = torch.from_numpy(pinned.array)
    for k in range(K):
        host[k].copy_(u8[:, k * ne:(k + 1) * ne])
    del u8
    torch.cuda.synchronize()
    chunk_ptr = [pinned.ptr + k * S * ne * 2 for k in range(K)]
    eng = engine.Engine(S, ne, device=dev.index)
    es = torch.cuda.ExternalStream(eng.stream, device=dev)
    for k in range(K):                                      # one whole capture untimed: step 0 starts a new one
        eng.push_host_ptr(chunk_ptr[k], ne, s16=False, u8=True)
        eng.poll_messages()
    torch.cuda.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    a0.record(es)
    msgs = []
    for k in range(steps):
        eng.push_host_ptr(chunk_ptr[k % K], ne, s16=False, u8=True)
        msgs += eng.poll_messages(wait=False)
    msgs += eng.poll_messages()
    a1.record(es)
    a1.synchronize()
    sec = max(a0.elapsed_time(a1) * 1e-3, time.time() - t0)
    eng.close()
    scratch = torch.empty((S, ne, 2), dtype=torch.uint8, device=dev)
    cs = torch.cuda.Stream(device=dev)
    n_copy = max(10, min(steps, 40))

    def copies(m):          # tensor.copy_ from page-locked memory = one cudaMemcpyAsync per chunk
        with torch.cuda.stream(cs):
            for k in range(m):
                scratch.copy_(host[k % K], non_blocking=True)
    copies(3)
    cs.synchronize()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record(cs)
    copies(n_copy)
    b1.record(cs)
    cs.synchronize()
    bytes_chunk = S * ne * 2
    ceiling = bytes_chunk * n_copy / (b0.elapsed_time(b1) * 1e-3) / 1e9
    del scratch, host
    pinned.close()
    gbs = bytes_chunk * steps / sec / 1e9
    expect_set = set(expect)
    return {"gsamples_per_s": S * ne * steps / sec / 1e9, "ms_per_step": sec * 1e3 / steps, "h2d_gbs": gbs,
            "h2d_ceiling_gbs": ceiling, "frac_of_ceiling": gbs / ceiling,
            "input": f"8-bit I,Q in page-locked host memory (nvx_pinned_alloc), [{S} streams][{ne} samples] per step",
            "ceiling": f"bare pinned cudaMemcpyAsync of the same chunks, {n_copy} copies",
            "steps": steps, "messages": len(msgs), "messages_exact": sum(1 for m in msgs if m in expect_set),
            "bulletins_completed_in_timed_steps": len(expect) * (steps // K)}


if __name__ == "__main__":
    main()

"""Cost of per-stream resets (nvx_engine_reset_streams) on the default workload's shape.

    python tools/bench_stream_reset.py [--rounds R] [--steps K] [--out profiles/bench_stream_reset_n1.json]

Workload: 1024 streams x bench.BLOCK samples of float2 (bench.py's default), generated on the device by nvx_synth_fill_device
from bench.make_bulletins.  One engine; each timed push is preceded by reset_streams() of 0, 1 or 1024 streams (a reset costs
one kernel on the engine stream, which first waits for the previous block's demod).  The step time is device events around K
pushes and a sync on the engine stream; the three cases alternate, in a rotating order, for R rounds, so the spread of each
figure is measured in the same run.  The GPU's name, power limit and clocks are read in the same run.  One JSON line goes to
stdout and to --out."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (workload shape, bulletins)
from bench_u8 import gpu_info  # noqa: E402

CASES = (0, 1, 1024)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=4, help="pushes per case per round")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_stream_reset_n1.json"))
    args = ap.parse_args()

    import numpy as np
    import torch
    from navtex_b200 import engine, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench_stream_reset.py: no CUDA device")
    dev = torch.device("cuda", 0)
    info_before = gpu_info()
    S, n = bench.STREAMS_PER_GPU, bench.BLOCK
    bits, off, start, amp, sigma, _ = bench.make_bulletins(np, synth, S, 0, 518490, n, 1, 3, 18, 5)
    x = torch.empty((S, n, 2), dtype=torch.float32, device=dev)
    engine.synth_fill_device(0, x.data_ptr(), S, 0, n, bits, off, start, amp, sigma, seed=518490)
    torch.cuda.synchronize()
    eng = engine.Engine(S, n)
    lists = {k: np.arange(0, S, S // k) if k else None for k in CASES}

    step = {k: [] for k in CASES}
    es = torch.cuda.ExternalStream(eng.stream, device=dev)
    for r in range(args.rounds):
        for k in CASES[r % 3:] + CASES[:r % 3]:
            eng.push_device(x.data_ptr(), n)        # warm
            eng.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(es)
            for _ in range(args.steps):
                if k:
                    eng.reset_streams(lists[k])
                eng.push_device(x.data_ptr(), n)
            eng.sync()
            e1.record(es)
            e1.synchronize()
            eng.poll_messages()
            step[k].append(e0.elapsed_time(e1) / args.steps)
    info_during = gpu_info()
    eng.close()

    def summary(v):
        return {"median": statistics.median(v), "min": min(v), "max": max(v), "rounds": v}

    rec = {
        "what": "push with 0 / 1 / 1024 streams reset before it (tools/bench_stream_reset.py)",
        "gpu": info_before, "gpu_after_timing": info_during,
        "streams": S, "samples_per_stream": n, "steps_per_round": args.steps,
        "step_ms": {str(k): summary(step[k]) for k in CASES},
    }
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
